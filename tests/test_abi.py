"""CPU-only checks of the drop-in boundary: the C-ABI library loads, exports every symbol include/mvx_b200.h
declares, validates arguments, and never computes without a GPU (no CPU fallback)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, 'include', 'mvx_b200.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(mvx_[a-z0-9_]+)\s*\(', text)))


def test_library_exports_every_declared_symbol():
    from mvxnet_makise_b200 import _lib
    syms = header_symbols()
    assert sorted(_lib.EXPORTS) == syms
    raw = ctypes.CDLL(_lib.LIB_PATH)
    for s in syms:
        assert hasattr(raw, s), f'{s} declared in include/mvx_b200.h but not exported'
    assert _lib.lib.mvx_version() >= 100


def test_struct_layout_matches_header():
    from mvxnet_makise_b200 import _lib
    assert ctypes.sizeof(_lib.Grid) == 3 * 8 + 3 * 8 + 3 * 4 + 4
    assert ctypes.sizeof(_lib.VoxelOut) == 7 * 8
    a = _lib.PointPathArgs()
    a.grid = _lib.make_grid((0, -40, -3, 70.4, 40, 1), (0.2, 0.2, 0.4), (352, 400, 10), 35)
    a.B, a.cap, a.map_c = 2, 1024, 256
    for l, (h, w) in enumerate([(104, 336), (52, 168), (26, 84)]):
        a.map_h[l], a.map_w[l] = h, w
    n = ctypes.c_size_t()
    assert _lib.lib.mvx_pointpath_workspace_bytes(ctypes.byref(a), ctypes.byref(n)) == 0
    offs = (ctypes.c_int64 * _lib.WS_REGIONS)()
    assert _lib.lib.mvx_pointpath_layout(ctypes.byref(a), offs) == 0
    names = [(_lib.lib.mvx_pointpath_layout_name(r) or b'').decode() for r in range(_lib.WS_REGIONS)]
    assert 'vfeat' in names and 'cell2vid' in names
    used = [offs[r] for r in range(_lib.WS_REGIONS) if names[r]]
    assert used == sorted(used) and names[len(used) - 1] == 'Y8' and used[-1] == n.value   # Y8: training-only tail region
    fwd, bwd = ctypes.c_size_t(), ctypes.c_size_t()
    assert _lib.lib.mvx_pointpath_train_workspace_bytes(ctypes.byref(a), ctypes.byref(fwd), ctypes.byref(bwd)) == 0
    assert fwd.value > n.value and bwd.value > 0 and _lib.lib.mvx_grad_floats() == 726_880
    # the dense cell->voxel map must be there for both frames
    assert n.value > 2 * 352 * 400 * 10 * 4


def test_argument_validation_without_gpu():
    from mvxnet_makise_b200 import _lib
    a = _lib.PointPathArgs()
    n = ctypes.c_size_t()
    assert _lib.lib.mvx_pointpath_workspace_bytes(ctypes.byref(a), ctypes.byref(n)) == -1     # B = 0
    assert b'B must be' in _lib.lib.mvx_last_error()
    assert _lib.lib.mvx_voxelize_workspace_bytes(1, 64, ctypes.byref(n)) == -1
    assert _lib.lib.mvx_voxelize_workspace_bytes(8, 120064, ctypes.byref(n)) == 0 and n.value > 0
    with pytest.raises(RuntimeError):
        _lib.check(-3, 'demo')


def test_mode_switches_accept_only_the_modes_that_exist():
    from mvxnet_makise_b200 import _lib
    einval = -1
    try:
        for m in (2, 3, 4, 7, 8, 11):
            assert _lib.lib.mvx_set_gemm_mode(m) == einval, m
            assert b'gemm mode must be' in _lib.lib.mvx_last_error()
        for m in (0, 1, 5, 6, 9, 10, 12):
            assert _lib.lib.mvx_set_gemm_mode(m) == 0, m
        assert _lib.lib.mvx_set_fold_mode(1) == einval
        assert b'fold mode must be' in _lib.lib.mvx_last_error()
        assert _lib.lib.mvx_set_fold_mode(2) == 0
    finally:
        assert _lib.lib.mvx_set_gemm_mode(1) == 0
        assert _lib.lib.mvx_set_fold_mode(0) == 0


@pytest.mark.skipif(torch.cuda.is_available(), reason='CPU-only behaviour')
def test_no_cpu_fallback():
    from mvxnet_makise_b200 import voxelize, modules, pipeline, synth
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        modules.lidar2Img(np.zeros((4, 4), np.float32), synth.kitti_calib(), True)
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        pipeline.PointPath(synth.make_weights(0))
    with pytest.raises((RuntimeError, AssertionError)):
        voxelize.cpp._group(np.zeros((4, 4), np.float32), np.zeros((4, 3), np.int32), 35)
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        voxelize.cpp.bboxOverlap(np.zeros((1, 4, 2), np.float32), np.zeros((1, 4, 2), np.float32))
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        voxelize.cpp._classifyAnchors(np.zeros((1, 4, 2), np.float32), np.zeros((2, 2, 2, 4, 2), np.float32), np.zeros(1, np.int64),
                                      np.zeros(1, np.int64), 0.45, 0.6)


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, 'mvxnet_makise_b200')
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r'^\s*(from|import)\s+oracle|oracle[./]|dlopen|_ref', text, flags=re.M), \
                    f'{f} reaches into the oracle'


def test_synth_frame_invariants():
    from mvxnet_makise_b200 import synth
    pts = synth.make_points(3, 5000)
    assert pts.shape == (5000, 4) and pts.dtype == np.float32
    r = synth.KITTI_VELORANGE
    assert np.all(pts[:, :3] >= np.array(r[:3])) and np.all(pts[:, :3] < np.array(r[3:]))
    assert np.array_equal(pts, synth.make_points(3, 5000))          # seeded
    sd = synth.make_weights(0)
    assert sum(v.size for v in sd.values()) == 726_880                # SURVEY.md §8b
    assert synth.fpn_shapes() == [(104, 336), (52, 168), (26, 84)]


def test_occupancy_helper_of_the_gpu_tests():
    """tests/_util.same_occupancy: cells where exactly one grid is zero may only hold rounding-level values."""
    import torch
    from _util import same_occupancy
    a = torch.zeros(4, 5)
    a[1, 2], a[3, 0] = 2.0, -1.5
    b = a.clone()
    assert same_occupancy(a, b)
    b[0, 0] = 1e-7              # an exactly-zero feature in one evaluation, rounding noise in the other
    assert same_occupancy(a, b)
    b[0, 0] = 1e-3              # a voxel that only one side has
    assert not same_occupancy(a, b)
    b[0, 0] = 0.0
    b[1, 2] = 0.0               # a voxel that only the other side has
    assert not same_occupancy(a, b)
