"""CPU: the compact backward of the sparse CML.conv1 hand-off (tests/_cml_compact.py, the formulas csrc/sparse_conv.cu
implements) equals dense fp64 autograd of the reference ops (oracle.pointpath_oracle.cml_conv1, voxelnet/Pipe.py:31-43),
and the new C-ABI entries validate their arguments without a GPU."""
import ctypes

import numpy as np
import pytest
import torch

import _cml_compact as C
from oracle import pointpath_oracle as O

F64 = torch.float64


def _dense_autograd(vfeat, coords, shape, w, b, g, eps=1e-6):
    grid = C.dense_grid(vfeat.to(F64), coords, shape).requires_grad_(True)
    wd, bd = w.to(F64).clone().requires_grad_(True), b.to(F64).clone().requires_grad_(True)
    out = O.cml_conv1(grid, wd, bd, eps)
    (out[0] * g.to(F64)).sum().backward()
    d_vfeat = grid.grad[0][:, coords[:, 2], coords[:, 0], coords[:, 1]].t()
    return d_vfeat, wd.grad, bd.grad


def _rel(a, ref):
    return float((a - ref).abs().max() / ref.abs().max().clamp_min(1e-30)) if ref.numel() else float(a.abs().max() if a.numel() else 0)


def _case(coords, shape, seed, eps=1e-6):
    rng = np.random.default_rng(seed)
    coords = torch.as_tensor(np.asarray(coords, dtype=np.int64).reshape(-1, 3))
    n = coords.shape[0]
    vfeat = torch.from_numpy(rng.standard_normal((n, 128)))
    w = torch.from_numpy(rng.standard_normal((64, 128, 3, 3, 3)) / np.sqrt(128 * 27))
    b = torch.from_numpy(rng.standard_normal(64) * 0.1)
    b[:8] = torch.linspace(-0.3, 0.3, 8, dtype=F64)            # both signs for certain
    g = torch.from_numpy(rng.standard_normal((64, C.out_depth(shape[0]), shape[1], shape[2])))
    y, act = C.activations(vfeat, coords, shape, w, b)
    got = C.cml_conv1_backward(vfeat, coords, shape, w, b, g, y, act, eps)
    want = _dense_autograd(vfeat, coords, shape, w, b, g, eps)
    return got, want, act


def _check(got, want):
    for name, a, r in zip(('d_vfeat', 'd_w', 'd_b'), got, want):
        assert tuple(a.shape) == tuple(r.shape), name
        assert _rel(a, r) < 1e-9, (name, _rel(a, r))


def test_random_voxels_small_grid():
    shape = (6, 7, 5)                                            # (nz, nx, ny)
    rng = np.random.default_rng(0)
    cells = rng.choice(6 * 7 * 5, 20, replace=False)
    iz, rem = np.divmod(cells, 7 * 5)
    ix, iy = np.divmod(rem, 5)
    got, want, act = _case(np.stack([ix, iy, iz], 1), shape, 1)
    assert 0 < int(act.sum()) < act.numel()
    _check(got, want)


def test_voxels_on_every_face_and_both_z_parities():
    shape = (5, 6, 4)                                            # odd depth: the last output plane sees only iz = nz - 1
    coords = [(0, 2, 1), (5, 1, 2), (3, 0, 3), (2, 3, 2), (4, 2, 0), (1, 1, 4),      # faces x-, x+, y-, y+, z-, z+
              (0, 0, 0), (5, 3, 4), (2, 1, 1), (2, 1, 2), (3, 2, 3)]                 # corners, both z parities
    got, want, _ = _case(coords, shape, 2)
    _check(got, want)


def test_frame_without_voxels():
    shape = (4, 5, 3)
    got, want, act = _case(np.zeros((0, 3)), shape, 3)
    assert not bool(act.any())
    d_vfeat, d_w, d_b = got
    assert d_vfeat.shape == (0, 128) and float(d_w.abs().max()) == 0.0
    assert _rel(d_w, want[1]) == 0.0 and float((d_b - want[2]).abs().max()) < 1e-9 * max(1.0, float(want[2].abs().max()))


def test_frame_where_every_position_is_active():
    shape = (4, 3, 3)
    iz, ix, iy = np.meshgrid(np.arange(4), np.arange(3), np.arange(3), indexing='ij')
    got, want, act = _case(np.stack([ix.ravel(), iy.ravel(), iz.ravel()], 1), shape, 4)
    assert bool(act.all())
    _check(got, want)


def test_backward_abi_validates_without_gpu():
    from mvxnet_makise_b200 import _lib
    a = _lib.PointPathArgs()
    n = ctypes.c_size_t()
    assert _lib.lib.mvx_cml_conv1_backward_workspace_bytes(ctypes.byref(a), ctypes.byref(n)) == -1      # B = 0
    a.grid = _lib.make_grid((0, -4.8, -3, 8, 4.8, 1), (0.2, 0.2, 0.4), (40, 48, 10), 35)
    a.B, a.cap, a.map_c = 2, 1024, 256
    for l, (h, w) in enumerate([(13, 42), (7, 21), (4, 11)]):
        a.map_h[l], a.map_w[l] = h, w
    assert _lib.lib.mvx_cml_conv1_backward_workspace_bytes(ctypes.byref(a), None) == -1
    assert _lib.lib.mvx_cml_conv1_backward_workspace_bytes(ctypes.byref(a), ctypes.byref(n)) == 0
    go = 5 * 40 * 48
    assert n.value >= 2 * 1024 * 1792 * 4 + 2 * go * 64 * 4                         # D and the compact dOut rows
    fwd = ctypes.c_size_t()
    assert _lib.lib.mvx_cml_conv1_workspace_bytes(ctypes.byref(a), ctypes.byref(fwd)) == 0
    pw = ctypes.c_size_t()
    assert _lib.lib.mvx_pointpath_workspace_bytes(ctypes.byref(a), ctypes.byref(pw)) == 0
    p = ctypes.c_void_p(256)                                                         # never dereferenced: validation fails first
    fn = _lib.lib.mvx_cml_conv1_sparse_backward
    a.workspace, a.workspace_bytes, a.counts = p, pw.value, p
    args = [p, p, 1e-6, p, p, p, p, 0, p, fwd.value, p, n.value]
    for i in (0, 1, 3, 5, 6, 8, 10):                                                 # conv_w, conv_b, d_out, d_w, d_b, ws, bws
        bad = list(args)
        bad[i] = None
        assert fn(ctypes.byref(a), *bad) == -1, i
        assert b'null pointer' in _lib.lib.mvx_last_error()
    for i in (9, 11):                                                                # short forward / backward workspace
        bad = list(args)
        bad[i] -= 1
        assert fn(ctypes.byref(a), *bad) == -3, i
    a.workspace_bytes = pw.value - 1                                                  # short path workspace
    assert fn(ctypes.byref(a), *args) == -3
    a.workspace_bytes, a.counts = pw.value, None
    assert fn(ctypes.byref(a), *args) == -1
