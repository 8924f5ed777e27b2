"""The gradient into the FPN maps, CPU side: the compact adjoint of the 4-corner gather (tests/_map_adjoint.py `map_adjoint`,
the formula csrc/map_backward.cu implements, applied to fcn1's dpre of the oracle's compact formulas) against fp64 autograd with
the maps as leaves of the dense reference chain featureMaping -> fusion -> VFE -> FCN -> max (`dense_backward`), and the
argument validation of the C entries mvx_pointpath_backward_maps(_workspace_bytes)."""
import ctypes
import os
import warnings

import numpy as np
import pytest
import torch

import _map_adjoint as MA
from mvxnet_makise_b200 import synth
from oracle import compact_backward as CB
from oracle import pointpath_oracle as O

G = synth.KITTI_GRID
SMALL_FPN = ((13, 42), (7, 21), (4, 11))
IMSIZE = synth.KITTI_IMSIZE_HW
W1 = 'head.fusion.fcn1.fc.weight'


def small_maps(seed):
    rng = np.random.default_rng(seed)
    return [rng.standard_normal((1, 256, h, w), dtype=np.float32) for (h, w) in SMALL_FPN]


def compact_vs_dense(voxels, maps, sd_np, seed):
    """max over the levels of |compact adjoint - dense fp64 autograd| / max |autograd|"""
    N = voxels.shape[0]
    d_vfeat = np.random.default_rng(seed).standard_normal((N, 128))
    dmaps = MA.dense_backward(voxels.clone(), maps, sd_np, IMSIZE, d_vfeat)
    v = voxels.clone()
    im768 = O.feature_mapping(v, [torch.from_numpy(m).double() for m in maps], torch.Tensor(list(IMSIZE)))
    cnt, rows, row_v = CB.compact_rows(v, G.T)
    K = len(rows)
    A1 = torch.cat([im768.reshape(-1, 768)[rows], torch.zeros(1, 768, dtype=torch.float64)], 0)
    vox7c = torch.cat([v[..., :7].double().reshape(-1, 7)[rows], torch.zeros(1, 7, dtype=torch.float64)], 0)
    proj = torch.cat([voxels[..., 7:9].reshape(-1, 2)[rows], torch.zeros(1, 2)], 0)
    real = torch.ones(K + 1, dtype=torch.bool)
    real[K] = False                                   # the frame's pad row samples nothing
    sd = {k: torch.from_numpy(np.asarray(x)) for k, x in sd_np.items()}
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        _, st, aux = CB.compact_forward(A1, vox7c, sd, cnt, row_v, G.T)
        dpre1 = MA.compact_dpre1(st, aux, d_vfeat, row_v)
    got = MA.map_adjoint(dpre1, sd[W1], proj, real, SMALL_FPN, IMSIZE)
    errs = []
    for g, ref in zip(got, dmaps):
        assert g.shape == ref.shape
        errs.append(float((g - ref).abs().max() / ref.abs().max()))
    return errs, dmaps


@pytest.mark.parametrize('tag', ['path_a', 'path_b'])
def test_compact_map_adjoint_equals_dense_autograd(golden_dir, tag):
    g = np.load(os.path.join(golden_dir, tag + '.npz'))
    maps = small_maps(int(g['map_seed']))
    sd_np = synth.make_weights(int(g['weight_seed']))
    voxels = torch.Tensor(O.group(O.points_with_proj(g['pcd4'], synth.kitti_calib()), G.velorange, G.voxelsize, G.T)[0])
    errs, dmaps = compact_vs_dense(voxels, maps, sd_np, 5)
    assert max(errs) < 1e-9, errs
    assert all(float(d.abs().max()) > 0 for d in dmaps)


def _hand_voxels():
    """six voxels whose points sit where the corner rules matter, per level l with regionSize rs_l = imsize / (H_l, W_l):
    exactly on pixel positions, in the last map row / column (corners on the zero pad), at projections 0 (q in (-1, 0):
    index 0 with a negative fraction), and one real point at the origin (treated as a pad slot, Pipe.py:53-59)"""
    rng = np.random.default_rng(3)
    (h0, w0), (h1, w1), _ = SMALL_FPN
    rs0 = (np.float32(IMSIZE[0]) / np.float32(h0), np.float32(IMSIZE[1]) / np.float32(w0))
    rs1 = (np.float32(IMSIZE[0]) / np.float32(h1), np.float32(IMSIZE[1]) / np.float32(w1))
    projs = [
        [(rs0[0] * 3, rs0[1] * 7), (rs0[0] * 5, rs0[1] * 11), (rs1[0] * 2, rs1[1] * 4)],           # on level-0 / level-1 pixels
        [((h0 - 0.25) * rs0[0], 17.0), (30.0, (w0 - 0.4) * rs0[1]), ((h0 - 0.5) * rs0[0], (w0 - 0.5) * rs0[1])],   # last row / column
        [(0.0, 0.0), (0.0, 250.0), (120.0, 0.0), (1e-7, 3e-6)],                                    # q in (-1, 0)
        [(IMSIZE[0] - 1e-3, IMSIZE[1] - 1e-3), (187.3, 611.9)],                                    # the image's last pixel
        [(100.5, 400.25), (101.0, 401.0), (99.75, 399.5)],                                         # three points, one cell
        [(55.0, 900.0), None],                                                                     # None: a real point at the origin
    ]
    v = np.zeros((len(projs), G.T, 9), np.float32)
    for i, ps in enumerate(projs):
        for s, p in enumerate(ps):
            if p is None:
                v[i, s, 6] = 0.7          # reflectance only: x = y = z = 0
                continue
            v[i, s, :3] = rng.uniform(1, 20, 3)
            v[i, s, 3:7] = rng.standard_normal(4)
            v[i, s, 7:9] = p
    return torch.from_numpy(v)


def test_compact_map_adjoint_on_hand_made_rows():
    voxels = _hand_voxels()
    errs, dmaps = compact_vs_dense(voxels, small_maps(7), synth.make_weights(2), 9)
    assert max(errs) < 1e-9, errs
    # the corners of the hand-made rows reach the first and last map row and column of level 0
    d0 = dmaps[0].abs().sum(0)
    assert float(d0[0].sum()) > 0 and float(d0[-1].sum()) > 0 and float(d0[:, 0].sum()) > 0 and float(d0[:, -1].sum()) > 0


def _args():
    from mvxnet_makise_b200 import _lib
    a = _lib.PointPathArgs()
    a.grid = _lib.make_grid(G.velorange, G.voxelsize, G.voxelshape, G.T)
    a.B, a.cap, a.map_c = 2, 1024, 256
    for l, (h, w) in enumerate(synth.fpn_shapes()):
        a.map_h[l], a.map_w[l] = h, w
    return a


def test_map_backward_argument_validation_without_gpu():
    from mvxnet_makise_b200 import _lib
    lib = _lib.lib
    a = _args()
    n = ctypes.c_size_t()
    assert lib.mvx_pointpath_backward_maps_workspace_bytes(ctypes.byref(a), None) == -1
    assert lib.mvx_pointpath_backward_maps_workspace_bytes(ctypes.byref(a), ctypes.byref(n)) == 0
    dz = 2 * sum(h * w for h, w in synth.fpn_shapes()) * 768 * 4
    assert n.value > dz                                       # the per-pixel dZ of both frames is part of it
    fwd, bwd = ctypes.c_size_t(), ctypes.c_size_t()
    assert lib.mvx_pointpath_train_workspace_bytes(ctypes.byref(a), ctypes.byref(fwd), ctypes.byref(bwd)) == 0
    fake = ctypes.c_void_p(1 << 40)                          # never dereferenced: every call below fails its checks first
    maps = (ctypes.c_void_p * 3)(fake, fake, fake)
    a.workspace, a.workspace_bytes, a.counts = fake, fwd.value, fake
    a.wt[0] = fake
    call = lambda bws, nb, m, ws, nw: lib.mvx_pointpath_backward_maps(ctypes.byref(a), bws, nb, m, ws, nw)
    assert call(fake, bwd.value, maps, fake, n.value - 1) == -3
    assert b'map backward workspace' in lib.mvx_last_error()
    assert call(fake, bwd.value - 1, maps, fake, n.value) == -3
    assert call(None, bwd.value, maps, fake, n.value) == -1
    assert call(fake, bwd.value, None, fake, n.value) == -1
    assert call(fake, bwd.value, (ctypes.c_void_p * 3)(fake, None, fake), fake, n.value) == -1
    assert call(fake, bwd.value, maps, None, n.value) == -1
    a.workspace_bytes = fwd.value - 1
    assert call(fake, bwd.value, maps, fake, n.value) == -3
    assert b'training workspace' in lib.mvx_last_error()
    a.B = 0
    assert call(fake, bwd.value, maps, fake, n.value) == -1
