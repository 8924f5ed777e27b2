"""Pins the oracle (oracle/pointpath_oracle.py + oracle/voxel_oracle.c) against the golden vectors the
UNMODIFIED reference produced (tests/golden/make_golden.py), and against the live reference where
/root/reference exists. CPU only."""
import hashlib
import os

import numpy as np
import pytest
import torch

from mvxnet_makise_b200 import synth
from oracle import pointpath_oracle as O
from oracle import refshim

G = synth.KITTI_GRID


def sha(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def rel_err(a, ref):
    a, ref = torch.as_tensor(a).double(), torch.as_tensor(ref).double()
    return float((a - ref).abs().max() / ref.abs().max())


def small_maps(seed, shapes=((13, 42), (7, 21), (4, 11))):
    rng = np.random.default_rng(seed)
    return [rng.standard_normal((1, 256, h, w), dtype=np.float32) for (h, w) in shapes]


@pytest.mark.parametrize('tag', ['vox_a', 'vox_b'])
def test_voxelizer_oracle_matches_reference_golden(golden_dir, tag):
    g = np.load(os.path.join(golden_dir, tag + '.npz'))
    pcd4 = g['pcd4']
    idx = O.cell_index(pcd4, G.velorange, G.voxelsize)
    assert np.array_equal(idx, g['idx'])                                  # fp64 index math, bit-exact
    assert np.array_equal(O.cell_index_numpy(pcd4, G.velorange, G.voxelsize), g['idx'])
    vox7, (x, y, z), cnt = O.cpp_group(pcd4, idx, G.T)
    assert vox7.dtype == np.float32 and np.array_equal(vox7, g['vox7'])
    assert np.array_equal(np.stack([x, y, z], 1), g['uidx7']) and np.array_equal(cnt, g['cnt7'])
    pcd6 = O.points_with_proj(pcd4, synth.kitti_calib())
    assert np.array_equal(pcd6[:, [5, 4]], g['proj_uv'])                  # lidar2Img, bit-exact on the same CPU libs
    vox9, uidx9 = O.group(pcd6, G.velorange, G.voxelsize, G.T)
    assert vox9.dtype == np.float64 and np.array_equal(uidx9, g['uidx9'])
    assert np.array_equal(vox9[..., [0, 1, 2, 6, 7, 8]], g['vox9'][..., [0, 1, 2, 6, 7, 8]])
    # centroid offsets: fp64, summation order may differ by an ulp of the fp64 sum
    np.testing.assert_allclose(vox9[..., 3:6], g['vox9'][..., 3:6], rtol=0, atol=1e-12)
    assert np.array_equal(vox9.astype(np.float32), g['vox9'].astype(np.float32))   # what reaches the GPU (train.py:125)


@pytest.mark.parametrize('tag', ['path_a', 'path_b'])
def test_path_oracle_matches_reference_golden(golden_dir, tag):
    g = np.load(os.path.join(golden_dir, tag + '.npz'))
    maps = small_maps(int(g['map_seed']))
    sd = synth.make_weights(int(g['weight_seed']))
    assert sha(*maps) == str(g['maps_sha']), 'numpy RNG stream changed: regenerate tests/golden'
    assert sha(*[sd[k] for k in sorted(sd)]) == str(g['weights_sha'])
    with torch.no_grad():
        r = O.forward_frame(g['pcd4'], synth.kitti_calib(), maps, sd, G, synth.KITTI_IMSIZE_HW)
    assert np.array_equal(r['voxels9'].numpy(), g['voxels9_after'])      # incl. in-place pad zeroing
    assert np.array_equal(r['idx'].numpy(), g['idx'])
    im768 = r['im768'].reshape(-1, 768)
    assert np.array_equal(im768[g['im768_rows']].numpy(), g['im768_sample'])
    np.testing.assert_allclose(im768.double().sum(0).numpy(), g['im768_colsum'], rtol=1e-12)
    # Tolerate accumulation-order noise only. The fp32 evaluation is bit-equal to the golden on the CPU that wrote it, but the
    # BLAS picks its kernels (and so its summation order) by CPU, and the batch-statistic BatchNorms amplify that: on another
    # x86 host the fp32 im16 / vfeat differ from the golden by up to 1.0e-4 / 4.6e-4 of max (fp32 vs fp64 there: 0.5-1.3e-4).
    # The fp64 evaluation is the same on every CPU. Both fp32 evaluations, the reference's and this CPU's, must lie within the
    # 5e-4 that bounds fp32 against fp32 in tests/test_gpu_parity.py (the golden: 1.1-3.5e-4; a 1 % change of any one bias: > 6e-4)
    with torch.no_grad():
        r64 = O.forward_frame(g['pcd4'], synth.kitti_calib(), maps, sd, G, synth.KITTI_IMSIZE_HW, dtype=torch.float64)
    for k in ('im16', 'vfeat'):
        assert rel_err(g[k], r64[k]) < 5e-4 and rel_err(r[k], r64[k]) < 5e-4, (k, rel_err(g[k], r64[k]), rel_err(r[k], r64[k]))
    if np.array_equal(r['im16'].numpy(), g['im16']):     # this CPU sums like the one that wrote the golden: exact from here on
        assert np.array_equal(r['vfeat'].numpy(), g['vfeat'])
    grid = r['grid'].numpy()
    assert tuple(grid.shape) == tuple(g['grid_shape'])
    assert int((grid != 0).sum()) == int(g['grid_nonzero'])
    if np.array_equal(r['vfeat'].numpy(), g['vfeat']):
        assert sha(grid) == str(g['grid_sha'])


@pytest.mark.skipif(not refshim.available(), reason='/root/reference absent (GPU box)')
def test_oracle_matches_live_reference():
    m = refshim.load()
    pcd4 = synth.make_points(21, 3000)
    idx = O.cell_index(pcd4, G.velorange, G.voxelsize)
    v_ref, u_ref, c_ref = m.cpp._group(pcd4, idx, G.T)
    v, u, c = O.cpp_group(pcd4, idx, G.T)
    assert np.array_equal(v, v_ref) and np.array_equal(c, c_ref)
    assert all(np.array_equal(a, b) for a, b in zip(u, u_ref))
    calib = {k: torch.Tensor(x) for k, x in synth.kitti_calib().items()}
    assert torch.equal(O.lidar2img(torch.Tensor(pcd4), calib), m.calib.lidar2Img(torch.Tensor(pcd4), calib, True))
    # one CRB block vs the reference FCN module
    torch.manual_seed(1)
    fcn = m.layers.FCN(24, 16)
    x = torch.randn(1, 50, 35, 24)
    with torch.no_grad():
        assert torch.allclose(fcn(x), O.crb(x, fcn.fc.weight, fcn.fc.bias), rtol=1e-6, atol=1e-6)


@pytest.mark.skipif(not refshim.available(), reason='/root/reference absent (GPU box)')
def test_merged_point_sets_follow_train_py():
    """train.py:29-42: scene through the torch branch of lidar2Img (`[:, [1, 0]]`), pasted objects through the numpy branch
    (`[:, ::-1]`), each with its own calibration; the two branches agree bit for bit, which is what lets the oracle (and the
    CUDA path) use one projection routine for every set."""
    m = refshim.load()
    base = synth.kitti_calib()
    other = {k: np.array(v, dtype=np.float32, copy=True) for k, v in base.items()}
    other['P2'][0, 0] += np.float32(11.5); other['P2'][0, 2] -= np.float32(3.25); other['Tr_velo_to_cam'][0, 3] += np.float32(0.031)
    scene, pasted = synth.make_points(31, 4000), synth.make_points(32, 700)
    pcd = torch.Tensor(scene)                                                       # train.py:31-35
    ct = {k: torch.Tensor(np.asarray(v)) for k, v in base.items()}
    ref_scene = torch.concat([pcd, m.calib.lidar2Img(pcd, ct, True)[:, [1, 0]]], dim=1).numpy()
    proj = m.calib.lidar2Img(pasted, other, True)[:, ::-1]                          # train.py:37-41 (numpy branch)
    ref = np.concatenate([ref_scene, np.concatenate([pasted, proj], axis=1)], axis=0)
    ours = O.merged_points_with_proj([scene, pasted], [base, other])
    assert ours.dtype == ref.dtype == np.float32 and np.array_equal(ours.view(np.uint32), ref.view(np.uint32))
    both = m.calib.lidar2Img(torch.Tensor(pasted), {k: torch.Tensor(v) for k, v in other.items()}, True).numpy()
    assert np.array_equal(both[:, ::-1].view(np.uint32), np.ascontiguousarray(proj).view(np.uint32))


def test_oracle_empty_and_single_point():
    idx = np.zeros((0, 3), dtype=np.int32)
    vox, (x, y, z), cnt = O.cpp_group(np.zeros((0, 4), np.float32), idx, 35)
    assert vox.shape == (0, 35, 7) and cnt.shape == (0,)
    p = np.array([[1.0, 2.0, -1.0, 0.5]], np.float32)
    vox, (x, y, z), cnt = O.cpp_group(p, O.cell_index(p, G.velorange, G.voxelsize), 35)
    assert vox.shape == (1, 35, 7) and cnt[0] == 1 and (x[0], y[0], z[0]) == (5, 210, 5)


def test_compact_backward_equals_dense_autograd():
    """Step (1) of the gradient parity chain (oracle/compact_backward.py): the compact training-mode formulas (weighted
    pad rows, first-argmax routing, batch-stat BatchNorm backward with multiplicities) reproduce autograd through the dense
    restatement of the reference chain, in fp64."""
    import warnings
    from mvxnet_makise_b200 import synth
    from oracle import compact_backward as CB
    G = synth.KITTI_GRID
    pts = synth.make_points(11, 700)
    maps = [np.random.default_rng(1).standard_normal((1, 256, h, w), dtype=np.float32) for (h, w) in ((13, 42), (7, 21), (4, 11))]
    sd_np = synth.make_weights(4)
    sd = {k: torch.from_numpy(v) for k, v in sd_np.items()}
    N = O.group_assign(O.cell_index(pts, G.velorange, G.voxelsize), G.T)[2].shape[0]
    Gw = np.random.default_rng(2).standard_normal((N, 128))
    vf, gref = O.backward_frame(pts, synth.kitti_calib(), maps, sd_np, G, synth.KITTI_IMSIZE_HW, Gw)
    voxels = torch.Tensor(O.group(O.points_with_proj(pts, synth.kitti_calib()), G.velorange, G.voxelsize, G.T)[0])
    im768 = O.feature_mapping(voxels, [torch.from_numpy(m) for m in maps], torch.Tensor(list(synth.KITTI_IMSIZE_HW))).double()
    cnt, rows, row_v = CB.compact_rows(voxels, G.T)
    A1 = torch.cat([im768.reshape(-1, 768)[rows], torch.zeros(1, 768, dtype=torch.float64)], 0)
    vox7c = torch.cat([voxels[..., :7].double().reshape(-1, 7)[rows], torch.zeros(1, 7, dtype=torch.float64)], 0)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        out, st, aux = CB.compact_forward(A1, vox7c, sd, cnt, row_v, G.T)
        grads = CB.compact_backward(st, aux, Gw, row_v)
    assert (out - vf).abs().max().item() < 1e-9
    assert set(grads) == set(gref)
    for k in gref:
        g = grads[k].reshape(gref[k].shape)
        assert ((g - gref[k]).abs().max() / gref[k].abs().max()).item() < 1e-9, k


@pytest.mark.parametrize('tag', ['a', 'b'])
def test_crop_oracle_matches_reference_golden(golden_dir, tag):
    """`crop` / `cropToSight` restatements vs the unmodified reference's selections (tests/golden/make_golden_crop.py)."""
    from mvxnet_makise_b200 import synth
    g = np.load(os.path.join(golden_dir, 'crop_a.npz'))
    raw = g[f'raw_{tag}']
    tagged = raw.copy()
    tagged[:, 3] = np.arange(raw.shape[0], dtype=np.float32)
    calib = synth.kitti_calib()
    wh = (synth.KITTI_IMSIZE_HW[1], synth.KITTI_IMSIZE_HW[0])
    c = O.crop(tagged, synth.KITTI_VELORANGE)
    assert np.array_equal(c[:, 3].astype(np.int32), g[f'crop_{tag}'])
    assert np.array_equal(O.crop_to_sight(tagged, calib, wh)[:, 3].astype(np.int32), g[f'sight_{tag}'])
    assert np.array_equal(O.crop_to_sight(c, calib, wh)[:, 3].astype(np.int32), g[f'both_{tag}'])
    # the dict as readCalib builds it (float64 matrices, Load.py:24-41): the numpy branch decides in fp64, and the fixture holds
    # border points on which the fp32 and fp64 evaluations disagree
    c64 = synth.kitti_calib_f64()
    assert np.array_equal(O.crop_to_sight(tagged, c64, wh)[:, 3].astype(np.int32), g[f'sight64_{tag}'])
    assert np.array_equal(O.crop_to_sight(c, c64, wh)[:, 3].astype(np.int32), g[f'both64_{tag}'])
    assert not np.array_equal(g[f'sight64_{tag}'], g[f'sight_{tag}'])


def _golden_other_calib(g):
    return {'P2': g['m_other_P2'], 'R0_rect': g['m_other_R0'], 'Tr_velo_to_cam': g['m_other_Tr']}


def test_merged_sets_with_float64_calibrations_match_reference_golden(golden_dir):
    """train.py:29-42 with readCalib-style float64 dicts: scene through the torch branch (fp32), pasted sets through the numpy
    branch (fp64), merged, rounded to fp32 by `torch.Tensor(voxel)`. Golden written by the UNMODIFIED lidar2Img."""
    from mvxnet_makise_b200 import synth
    g = np.load(os.path.join(golden_dir, 'crop_a.npz'))
    c64, other = synth.kitti_calib_f64(), _golden_other_calib(g)
    assert other['P2'].dtype == np.float64
    ours = O.merged_points_with_proj([g['m_scene'], g['m_p1'], g['m_p2']], [c64, c64, other])
    assert ours.dtype == np.float64
    assert np.array_equal(ours.astype(np.float32).view(np.uint32), g['m_merged32'].view(np.uint32))
    uv = O.lidar2img_numpy(g['m_p2'], other)
    assert uv.dtype == np.float64 and np.array_equal(uv, g['m_uv64_p2'])
    # and it matters: the fp32 evaluation of the same sets differs in the last bit for a good part of the points
    as32 = lambda c: {k: np.asarray(v, dtype=np.float32) for k, v in c.items()}
    o32 = O.merged_points_with_proj([g['m_scene'], g['m_p1'], g['m_p2']], [as32(c64), as32(c64), as32(other)])
    assert not np.array_equal(o32.astype(np.float32), g['m_merged32'])


def test_cml_oracle_matches_reference_golden(golden_dir):
    """The checker of the sparse hand-off (csrc/sparse_conv.cu) - `O.cml_conv1` / `O.crb3d` - against the UNMODIFIED reference's
    `CML` (voxelnet/Pipe.py:31-43, CRB3d of layers/Blocks.py:20-29) run on a small sparse grid (tests/golden/make_golden_cml.py)."""
    g = np.load(os.path.join(golden_dir, 'cml_a.npz'))
    nz, nx, ny = (int(v) for v in g['shape'])
    grid = torch.zeros((1, 128, nz, nx, ny))
    iz, rem = np.divmod(g['cells'], nx * ny)
    ix, iy = np.divmod(rem, ny)
    grid[0, :, iz, ix, iy] = torch.from_numpy(g['feats']).T
    ws = [torch.from_numpy(g[f'w{i}']) for i in (1, 2, 3)]
    bs = [torch.from_numpy(g[f'b{i}']) for i in (1, 2, 3)]
    with torch.no_grad():
        y1 = O.cml_conv1(grid, ws[0], bs[0])
        ys = O.cml(grid, ws, bs)
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max())
    assert tuple(y1.shape) == tuple(g['y1'].shape) and rel(y1, torch.from_numpy(g['y1'])) < 1e-6
    for y, k in zip(ys, ('y1', 'y2', 'y3')):
        assert tuple(y.shape) == tuple(g[k].shape) and rel(y, torch.from_numpy(g[k])) < 1e-5, k
    # the fp64 evaluation the GPU test compares against stays within fp32 rounding of the reference's own fp32 run
    with torch.no_grad():
        y1_64 = O.cml_conv1(grid.double(), ws[0].double(), bs[0].double())
    assert rel(y1_64, torch.from_numpy(g['y1']).double()) < 1e-4
