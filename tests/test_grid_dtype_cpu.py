"""CPU-only checks of the grid dtype in the C ABI and the Python entries: the field sits at the end of the argument struct,
and every entry rejects an unsupported dtype before it touches a device."""
import ctypes

import pytest
import torch

EINVAL = -1


def _args():
    from mvxnet_makise_b200 import _lib
    a = _lib.PointPathArgs()
    a.grid = _lib.make_grid((0, -40, -3, 70.4, 40, 1), (0.2, 0.2, 0.4), (352, 400, 10), 35)
    a.B, a.cap, a.map_c = 2, 1024, 256
    for l, (h, w) in enumerate([(104, 336), (52, 168), (26, 84)]):
        a.map_h[l], a.map_w[l] = h, w
    return a


def test_grid_dtype_is_the_last_field_and_zero_means_fp32():
    from mvxnet_makise_b200 import _lib
    names = [n for n, _ in _lib.PointPathArgs._fields_]
    assert names[-1] == 'grid_dtype' and _lib.PointPathArgs.grid_dtype.offset + 4 <= ctypes.sizeof(_lib.PointPathArgs)
    assert _lib.PointPathArgs().grid_dtype == _lib.DTYPE_F32 == 0
    assert (_lib.DTYPE_F16, _lib.DTYPE_BF16) == (1, 2)
    assert [_lib.grid_dtype_code(d) for d in (torch.float32, torch.float16, torch.bfloat16)] == [0, 1, 2]
    for bad in (torch.float64, torch.int8, 'fp8', 1):
        with pytest.raises(ValueError):
            _lib.grid_dtype_code(bad)


def test_unsupported_grid_dtype_is_rejected_without_gpu():
    from mvxnet_makise_b200 import _lib
    lib = _lib.lib
    n = ctypes.c_size_t()
    for dt in (0, 1, 2):
        a = _args()
        a.grid_dtype = dt
        assert lib.mvx_pointpath_workspace_bytes(ctypes.byref(a), ctypes.byref(n)) == 0 and n.value > 0
    for dt in (-1, 3, 7):
        a = _args()
        a.grid_dtype = dt
        for fn in (lib.mvx_pointpath_forward, lib.mvx_pointpath_forward_train):
            assert fn(ctypes.byref(a)) == EINVAL, dt
            assert b'grid dtype must be' in lib.mvx_last_error()
        assert lib.mvx_pointpath_backward(ctypes.byref(a), None, None, None, 0, None, 0) == EINVAL
        assert b'grid dtype must be' in lib.mvx_last_error()


def test_typed_scatter_entries_reject_an_unsupported_dtype_without_gpu():
    from mvxnet_makise_b200 import _lib
    lib = _lib.lib
    fake = ctypes.c_void_p(256)
    for dt in (-1, 3):
        assert lib.mvx_scatter_dense_typed(fake, fake, 5, 128, 352, 400, 10, fake, dt, fake, None) == EINVAL
        assert b'grid dtype must be' in lib.mvx_last_error()
        assert lib.mvx_scatter_dense_backward_typed(fake, dt, fake, 5, 128, 352, 400, 10, fake, None) == EINVAL
        assert b'grid dtype must be' in lib.mvx_last_error()
    sb = lib.mvx_scatter_dense_backward_typed
    for dt in (0, 1, 2):
        assert sb(None, dt, None, 0, 128, 352, 400, 10, None, None) == 0          # nothing to gather
        assert sb(None, dt, fake, 5, 128, 352, 400, 10, fake, None) == EINVAL    # null d_grid
        assert lib.mvx_scatter_dense_typed(fake, fake, 5, 128, 352, 400, 10, None, dt, fake, None) == EINVAL   # null out


def test_python_entries_reject_an_unsupported_dtype_up_front():
    from mvxnet_makise_b200 import modules, pipeline, synth
    x = torch.zeros((2, 128))
    idx = torch.zeros((2, 4), dtype=torch.int64)
    with pytest.raises(ValueError):
        modules.reindex(x, idx, (8, 8, 4), dtype=torch.float64)
    with pytest.raises(ValueError):
        pipeline.PointPath(synth.make_weights(0), grid_dtype=torch.float64)
