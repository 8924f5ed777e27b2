"""Parity of the CUDA path (through the C ABI) against the oracle and the reference-generated golden vectors.

Bars (BASELINE.json north_star): voxel coordinates, point->voxel assignment, slots and counts BIT-EXACT;
gather bit-exact for identical `proj`; layer-stack outputs within TOL = 1e-4 relative (fp32), measured per
tensor as max|a-ref| / max|ref|.

What "ref" is for the 8-layer chain: the fp32 reference is itself noisy at this level. 86 % of the N*T rows are
identical pad rows, so BatchNorm normalises real rows to tens of sigma and the fp32 rounding of the reference's
own GEMMs/statistics shows up as 1.2e-4 .. 3.5e-4 relative at the end of the chain (measured: the reference vs
the same algorithm evaluated in fp64, tools/diag_layers.py; DESIGN.md §parity). The end-to-end checks therefore
assert (i) CUDA vs the fp64 evaluation of the oracle < TOL (measured 5e-6 with the exact-fp32 SIMT layers,
~3e-5 with the 3xTF32 tensor-core layers), and (ii) CUDA vs the fp32 oracle / the reference's golden output
<= that reference's own distance to fp64 + TOL (what is left after the reference's rounding is within TOL),
capped at 5e-4. Single layers and the 5-layer fusion stack meet TOL against fp32 directly."""
import os

import numpy as np
import pytest
import torch

from _util import same_occupancy

from mvxnet_makise_b200 import synth
from oracle import pointpath_oracle as O

pytestmark = pytest.mark.gpu
G = synth.KITTI_GRID
TOL = 1e-4
SMALL_FPN = ((13, 42), (7, 21), (4, 11))


def small_maps(seed, shapes=SMALL_FPN, B=1):
    rng = np.random.default_rng(seed)
    return [rng.standard_normal((B, 256, h, w), dtype=np.float32) for (h, w) in shapes]


def rel_err(a, ref):
    a = torch.as_tensor(a).double().cpu()
    ref = torch.as_tensor(ref).double().cpu()
    return ((a - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()


@pytest.fixture(scope='module')
def mvx():
    import mvxnet_makise_b200.voxelize as V
    import mvxnet_makise_b200.modules as M
    import mvxnet_makise_b200.pipeline as P
    assert torch.cuda.is_available()
    return type('NS', (), dict(V=V, M=M, P=P))


# ------------------------------------------------------------------------------------------- before the path (§8f rank 1)
@pytest.mark.parametrize('tag', ['a', 'b'])
def test_crop_matches_reference_golden(mvx, golden_dir, tag):
    """On-GPU `crop` / `cropToSight` (Preprocessing.py:12-55): the same points, in the same order, as the unmodified
    reference selects - including points exactly on the range bounds and their fp32 neighbours."""
    g = np.load(os.path.join(golden_dir, 'crop_a.npz'))
    raw = g[f'raw_{tag}']
    tagged = raw.copy()
    tagged[:, 3] = np.arange(raw.shape[0], dtype=np.float32)
    calib = synth.kitti_calib()
    wh = (synth.KITTI_IMSIZE_HW[1], synth.KITTI_IMSIZE_HW[0])
    c = mvx.V.crop(tagged, synth.KITTI_VELORANGE)
    assert isinstance(c, np.ndarray) and c.dtype == np.float32 and np.array_equal(c[:, 3].astype(np.int32), g[f'crop_{tag}'])
    assert np.array_equal(c, tagged[g[f'crop_{tag}']])                        # whole rows, untouched
    s_ = mvx.V.cropToSight(tagged, calib, wh)
    assert np.array_equal(s_[:, 3].astype(np.int32), g[f'sight_{tag}'])
    both = mvx.V.cropFrame(tagged, synth.KITTI_VELORANGE, calib, wh)
    assert np.array_equal(both[:, 3].astype(np.int32), g[f'both_{tag}'])
    t = mvx.V.cropTensor(torch.from_numpy(tagged).cuda(), synth.KITTI_VELORANGE)  # torch in -> CUDA tensor out
    assert t.is_cuda and np.array_equal(t.cpu().numpy(), c)
    # float64 calibration dict (what readCalib returns, Load.py:24-41,73): the reference's numpy branch decides in fp64; the
    # fixture holds border points where the fp32 and fp64 evaluations disagree
    c64 = synth.kitti_calib_f64()
    s64 = mvx.V.cropToSight(tagged, c64, wh)
    assert np.array_equal(s64[:, 3].astype(np.int32), g[f'sight64_{tag}'])
    assert np.array_equal(mvx.V.cropFrame(tagged, synth.KITTI_VELORANGE, c64, wh)[:, 3].astype(np.int32), g[f'both64_{tag}'])
    assert not np.array_equal(g[f'sight64_{tag}'], g[f'sight_{tag}'])


def test_crop_batched_ragged_and_feeds_the_path(mvx):
    """Batched device entry with ragged frames (one empty), vs the oracle per frame; the cropped sweep is a valid input of
    the fused path (every point inside the grid and the image)."""
    from mvxnet_makise_b200.modules import pack_calib
    calib = synth.kitti_calib()
    wh = (synth.KITTI_IMSIZE_HW[1], synth.KITTI_IMSIZE_HW[0])
    frames = [synth.make_raw_sweep(80, 5000), np.zeros((0, 4), np.float32), synth.make_raw_sweep(81, 1), synth.make_raw_sweep(82, 33333)]
    offsets = np.concatenate([[0], np.cumsum([p.shape[0] for p in frames])]).tolist()
    pts = torch.from_numpy(np.concatenate(frames, 0)).cuda()
    c32 = torch.stack([pack_calib(calib) for _ in frames]).cuda()
    out, counts = mvx.V.crop_frames(pts, offsets, synth.KITTI_VELORANGE, c32, wh)
    counts = counts.cpu().numpy()
    kept = []
    for f, p in enumerate(frames):
        ref = O.crop_to_sight(O.crop(p, synth.KITTI_VELORANGE), calib, wh)
        got = out[offsets[f]:offsets[f] + counts[f]].cpu().numpy()
        assert counts[f] == ref.shape[0] and np.array_equal(got, ref), f
        kept.append(got)
    path = mvx.P.PointPath(synth.make_weights(1), G)
    maps = [torch.from_numpy(m) for m in small_maps(3, B=2)]
    _, cnt = path([kept[0], kept[3]], [calib, calib], maps, want_grid=False)
    cnt = cnt.cpu().numpy()
    assert (cnt[:, 2] == 0).all() and cnt[0, 1] <= kept[0].shape[0] and cnt[1, 0] > 0


# ------------------------------------------------------------------------------------------- stage 1
@pytest.mark.parametrize('tag', ['vox_a', 'vox_b'])
def test_group_matches_reference_golden(mvx, golden_dir, tag):
    g = np.load(os.path.join(golden_dir, tag + '.npz'))
    vox7, (x, y, z), cnt = mvx.V.cpp._group(g['pcd4'], g['idx'], G.T)
    assert vox7.dtype == np.float32 and np.array_equal(vox7, g['vox7'])
    assert x.dtype == np.int64 and np.array_equal(np.stack([x, y, z], 1), g['uidx7'])
    assert np.array_equal(cnt, g['cnt7'])
    # numba `group` layout, index math on the GPU in fp64
    pcd6 = np.concatenate([g['pcd4'], g['proj_uv'][:, [1, 0]]], axis=1).astype(np.float32)
    vox9, uidx9 = mvx.V.group(pcd6, list(G.velorange), list(G.voxelsize), G.T, shuffle=False)
    assert vox9.dtype == np.float64 and np.array_equal(uidx9, g['uidx9'])
    assert np.array_equal(vox9[..., [0, 1, 2, 6, 7, 8]], g['vox9'][..., [0, 1, 2, 6, 7, 8]])
    np.testing.assert_allclose(vox9[..., 3:6], g['vox9'][..., 3:6], rtol=0, atol=1e-12)
    assert np.array_equal(vox9.astype(np.float32), g['vox9'].astype(np.float32))
    # group_ (reference numpy glue around our _group)
    v7, u7 = mvx.V.group_(g['pcd4'].copy(), list(G.velorange), list(G.voxelsize), G.T, shuffle=False)
    v7o, u7o = O.group_(g['pcd4'], G.velorange, G.voxelsize, G.T)
    assert np.array_equal(v7, v7o) and np.array_equal(u7, u7o)


def test_group_edge_cases(mvx):
    T = 35
    # empty
    v, (x, y, z), c = mvx.V.cpp._group(np.zeros((0, 4), np.float32), np.zeros((0, 3), np.int32), T)
    assert v.shape == (0, T, 7) and c.shape == (0,)
    # single point, P not a multiple of 32, > T points in one voxel, duplicates, negative keys
    rng = np.random.default_rng(0)
    for P in (1, 33, 127, 1000):
        pcd = rng.standard_normal((P, 4)).astype(np.float32)
        idx = rng.integers(-3, 3, (P, 3)).astype(np.int32)
        if P == 1000:
            idx[:600] = (1, 1, 1)            # 600 points in one voxel
            pcd[10:20] = pcd[0]              # duplicate points
        a = mvx.V.cpp._group(pcd, idx, T)
        b = O.cpp_group(pcd, idx, T)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[2], b[2])
        assert all(np.array_equal(p, q) for p, q in zip(a[1], b[1]))
    # fp64 input is force-cast like pybind's array_t<float>
    pcd64 = rng.standard_normal((50, 5))
    idx64 = rng.integers(0, 4, (50, 3))
    a = mvx.V.cpp._group(pcd64, idx64, 4)
    b = O.cpp_group(pcd64, idx64, 4)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[2], b[2])
    with pytest.raises(ValueError):
        mvx.V.cpp._group(np.zeros((4,), np.float32), np.zeros((4, 3), np.int32), T)


def test_voxelize_whole_sweep_in_one_voxel(mvx):
    """Adversarial density: 120 000 points in ONE voxel (plus a few crowded and ordinary ones). The per-point rank loop would
    need 1.4e10 compares; crowded voxels are ranked by a CTA-wide selection of the T smallest point indices instead.
    Bit-exact against the C oracle, and fast (bounded below)."""
    import time
    T = 35
    rng = np.random.default_rng(3)
    P = 120_000
    pts = np.empty((P, 4), np.float32)
    pts[:, 0] = rng.uniform(10.0, 10.19, P)          # all inside cell (50, 200, 5) of the 0.2 x 0.2 x 0.4 grid
    pts[:, 1] = rng.uniform(0.0, 0.19, P)
    pts[:, 2] = rng.uniform(-1.0, -0.61, P)
    pts[:, 3] = rng.uniform(0, 1, P)
    idx_mid = rng.choice(P, 3000, replace=False)     # three voxels with ~300 / ~700 / ~2000 points, and 200 ordinary points
    pts[idx_mid[:300], 0] += 1.0
    pts[idx_mid[300:1000], 1] += 2.0
    pts[idx_mid[1000:], 2] += 0.8
    pts[rng.choice(P, 200, replace=False), :3] = synth.make_points(8, 200)[:, :3]
    idx = O.cell_index(pts, G.velorange, G.voxelsize)
    v_ref, (x_ref, y_ref, z_ref), cnt_ref = O.cpp_group(pts, idx, T)
    mvx.V.cpp._group(pts[:1000], idx[:1000], T)      # warm-up (context, allocations)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    vox7, (x, y, z), cnt = mvx.V.cpp._group(pts, idx, T)
    dt = time.perf_counter() - t0
    assert np.array_equal(vox7, v_ref) and np.array_equal(cnt, cnt_ref)
    assert np.array_equal(np.stack([x, y, z], 1), np.stack([x_ref, y_ref, z_ref], 1))
    assert int(cnt.max()) == T and dt < 0.5, f'crowded-voxel frame took {dt:.3f} s'
    # and through the fused path's voxelizer (raw points, fp64 index math on the GPU)
    from mvxnet_makise_b200 import _lib
    vb = mvx.V.voxelize(torch.from_numpy(pts).cuda(), [0, P], T, grid=_lib.make_grid(G.velorange, G.voxelsize, G.voxelshape, T))
    c = vb.counts[0].cpu().numpy()
    assert c[0] == cnt_ref.shape[0] and c[1] == cnt_ref.sum() and c[3] >= 100_000


def test_cell_index_boundary_floats(mvx):
    """fp64 subtract + TRUE division + truncation on fp32 neighbours of every cell boundary (trap 1)."""
    r, s = G.velorange, G.voxelsize
    pts = []
    for d, n in enumerate(G.voxelshape):
        b = (np.arange(1, n) * s[d] + r[d]).astype(np.float32)
        for w in (np.nextafter(b, np.float32(-1e9)), b, np.nextafter(b, np.float32(1e9))):
            p = np.tile(np.array([[1.0, 1.0, -1.0, 0.5]], np.float32), (len(w), 1))
            p[:, d] = w
            pts.append(p)
    pts = np.concatenate(pts)
    lo, hi = np.array(r[:3]), np.array(r[3:])
    pts = pts[np.all((pts[:, :3] >= lo) & (pts[:, :3] < hi), axis=1)]
    pcd6 = np.concatenate([pts, np.zeros((len(pts), 2), np.float32)], 1)
    _, uidx = mvx.V.group(pcd6, list(r), list(s), G.T, shuffle=False)
    _, uidx_o = O.group(pcd6, r, s, G.T)
    assert np.array_equal(uidx, uidx_o)


def test_voxelize_full_size_bit_exact(mvx):
    """BASELINE size (P = 120 000), against the C oracle (finishes in milliseconds)."""
    pcd = synth.make_points(0, 120_000)
    idx = O.cell_index(pcd, G.velorange, G.voxelsize)
    a = mvx.V.cpp._group(pcd, idx, G.T)
    b = O.cpp_group(pcd, idx, G.T)
    assert a[0].shape == b[0].shape and np.array_equal(a[0], b[0])
    assert np.array_equal(a[2], b[2]) and all(np.array_equal(p, q) for p, q in zip(a[1], b[1]))
    assert (a[2] == G.T).sum() > 0      # the case exercises the T cap


# ------------------------------------------------------------------------------------------- stage 2
@pytest.mark.parametrize('tag', ['vox_a', 'vox_b'])
def test_lidar2img_matches_reference_golden(mvx, golden_dir, tag):
    g = np.load(os.path.join(golden_dir, tag + '.npz'))
    uv = mvx.M.lidar2Img(g['pcd4'], synth.kitti_calib(), True)
    exact = (uv == g['proj_uv']).all(1).mean()
    np.testing.assert_allclose(uv, g['proj_uv'], rtol=2e-6, atol=1e-4)
    assert exact > 0.999, f'only {exact:.4f} of projections bit-exact'


@pytest.mark.parametrize('tag', ['path_a', 'path_b'])
def test_feature_mapping_bit_exact(mvx, golden_dir, tag):
    g = np.load(os.path.join(golden_dir, tag + '.npz'))
    maps = small_maps(int(g['map_seed']))
    pcd6 = O.points_with_proj(g['pcd4'], synth.kitti_calib())
    vox9, _ = O.group(pcd6, G.velorange, G.voxelsize, G.T)
    v_ref = torch.Tensor(vox9)
    v_gpu = v_ref.clone().cuda()[None]
    ref = O.feature_mapping(v_ref, [torch.from_numpy(m) for m in maps], torch.Tensor(list(synth.KITTI_IMSIZE_HW)))
    out = mvx.M.featureMaping(v_gpu, [torch.from_numpy(m).cuda() for m in maps], [None],
                              torch.Tensor(list(synth.KITTI_IMSIZE_HW)))[0]
    assert torch.equal(v_gpu[0].cpu(), v_ref), 'in-place pad zeroing differs'
    assert np.array_equal(v_gpu[0].cpu().numpy(), g['voxels9_after'])
    out = out.cpu()
    assert out.shape == ref.shape
    assert torch.equal(out, ref), f'gather not bit-exact: max diff {(out - ref).abs().max().item()}'
    assert np.array_equal(out.reshape(-1, 768)[g['im768_rows']].numpy(), g['im768_sample'])   # the reference itself


# ------------------------------------------------------------------------------------------- stage 3
def test_layer_modules_match_oracle(mvx):
    torch.manual_seed(0)
    N, T = 300, 35
    sd = {k: torch.from_numpy(v) for k, v in synth.make_weights(9).items()}
    x = torch.randn(1, N, T, 768)
    x[:, :, 20:] = 0          # pad-like rows
    fus = mvx.M.ImageFeatureFusion().cuda()
    fus.load_state_dict({k[len('head.fusion.'):]: v for k, v in sd.items() if k.startswith('head.fusion.')})
    with torch.no_grad():
        ref = O.fusion(x, sd)
        got = fus(x.cuda())
    assert got.shape == ref.shape and rel_err(got, ref) < TOL
    head = mvx.M.VoxelNetHead().cuda()
    head.load_state_dict({k[len('backbone.'):]: v for k, v in sd.items() if k.startswith('backbone.')})
    x23 = torch.randn(1, N, T, 23)
    x23[:, :, 25:] = 0
    with torch.no_grad():
        ref_v = O.voxel_features(x23, sd)
        got_v = head.voxel_features(x23.cuda())
        r1 = O.vfe(x23, sd['backbone.svfe.vfe1.fcn.fc.weight'], sd['backbone.svfe.vfe1.fcn.fc.bias'])
        g1 = head.svfe.vfe1(x23.cuda())
    assert g1.shape == r1.shape and rel_err(g1, r1) < TOL
    assert got_v.shape == ref_v.shape and rel_err(got_v, ref_v) < TOL


@pytest.mark.parametrize('R,cin,cout', [(1000, 768, 768), (5003, 768, 128), (777, 128, 128), (256, 768, 768)])
def test_tensor_core_layer_modes_are_fp32_accurate(mvx, R, cin, cout):
    """tcgen05 3xTF32 layer vs the exact-fp32 SIMT layer and vs an fp64 evaluation (ragged row counts)."""
    from mvxnet_makise_b200 import _lib
    torch.manual_seed(R)
    x = torch.randn(1, R, 1, cin, device='cuda')
    x[:, R // 2:] *= 0.01
    fcn = mvx.M.FCN(cin, cout).cuda()
    try:
        with torch.no_grad():
            _lib.set_gemm_mode(0)
            y_simt = fcn(x)
            _lib.set_gemm_mode(5)      # fp16 hi/lo operands (3xFP16), the default of the fused path's BatchNorm-ed layers
            y_f16 = fcn(x)
            _lib.set_gemm_mode(1)      # one 256 x BN tile per CTA (default), 3xTF32 for the dense API
            y_tc = fcn(x)
    finally:
        _lib.set_gemm_mode(1)
    y = torch.relu(x.double().reshape(-1, cin) @ fcn.fc.weight.double().t() + fcn.fc.bias.double())
    ref = (y - y.mean(0)) / torch.sqrt(y.var(0, unbiased=False) + 1e-6)
    assert rel_err(y_tc, y_simt) < 2e-5 and rel_err(y_f16, y_simt) < 2e-5
    assert rel_err(y_f16.reshape(-1, cout), ref) < 2e-5
    assert rel_err(y_tc.reshape(-1, cout), ref) < 2e-5 and rel_err(y_simt.reshape(-1, cout), ref) < 2e-5


def test_reindex_exact(mvx):
    rng = np.random.default_rng(1)
    N = 500
    cells = rng.choice(352 * 400 * 10, N, replace=False)
    iz, rem = np.divmod(cells, 352 * 400)
    ix, iy = np.divmod(rem, 400)
    idx = torch.from_numpy(np.stack([np.zeros(N, np.int64), ix, iy, iz], 1))
    x = torch.randn(N, 128)
    ref = O.reindex(x, idx, G.voxelshape)
    got = mvx.M.reindex(x.cuda(), idx.cuda(), G.voxelshape)
    assert got.shape == ref.shape and torch.equal(got.cpu(), ref)
    empty = mvx.M.reindex(torch.zeros(0, 128).cuda(), torch.zeros(0, 4, dtype=torch.int64).cuda(), G.voxelshape)
    assert float(empty.abs().max()) == 0.0


def test_reindex_exact_when_cells_are_not_a_multiple_of_32(mvx):
    """36 cells: a multiple of 4 but not of 32, so the cell-major fill runs instead of the plane-sequential one."""
    shape = (6, 2, 3)
    rng = np.random.default_rng(2)
    for N, C in ((20, 128), (36, 5)):
        cells = rng.choice(36, N, replace=False)
        iz, rem = np.divmod(cells, 12)
        ix, iy = np.divmod(rem, 2)
        idx = torch.from_numpy(np.stack([np.zeros(N, np.int64), ix, iy, iz], 1))
        x = torch.randn(N, C)
        ref = O.reindex(x, idx, shape)
        got = mvx.M.reindex(x.cuda(), idx.cuda(), shape)
        assert got.shape == ref.shape and torch.equal(got.cpu(), ref), (N, C)


# ------------------------------------------------------------------------------------------- fused path
def _check_close(got, ref32, ref64, what):
    e64 = rel_err(got, ref64)
    assert e64 < TOL, f'{what}: rel err vs fp64 evaluation {e64}'
    noise = rel_err(ref32, ref64)
    e32 = rel_err(got, ref32)
    assert e32 <= noise + TOL and e32 < 5e-4, f'{what}: rel err vs fp32 {e32}, fp32 reference noise {noise}'
    return e64, e32


def _check_frame(path, f, ref, ref64, counts, gold=None):
    n = ref['idx'].shape[0]
    assert counts[f, 0] == n and counts[f, 2] == 0
    vfeat, idx = path.voxel_features(f)
    assert np.array_equal(idx.cpu().numpy()[:, 1:], ref['idx'].numpy()[:, 1:])
    _check_close(vfeat, ref['vfeat'], ref64['vfeat'], 'voxel features')
    if gold is not None:      # the unmodified reference's own output
        _check_close(vfeat, gold['vfeat'], ref64['vfeat'], 'voxel features (reference golden)')


@pytest.fixture
def fusion_mode(request):
    """1 = pixel-first fcn1 (default), 0 = row-first (gather the (K,768) matrix, then the row GEMM)."""
    from mvxnet_makise_b200 import _lib
    _lib.set_fusion_mode(request.param)
    yield request.param
    _lib.set_fusion_mode(1)


@pytest.mark.parametrize('fusion_mode', [1, 0], indirect=True)
@pytest.mark.parametrize('tag', ['path_a', 'path_b'])
def test_fused_path_matches_reference_golden(mvx, golden_dir, tag, fusion_mode):
    g = np.load(os.path.join(golden_dir, tag + '.npz'))
    maps = small_maps(int(g['map_seed']))
    sd = synth.make_weights(int(g['weight_seed']))
    calib = synth.kitti_calib()
    path = mvx.P.PointPath(sd, G)
    grid, counts = path([g['pcd4']], [calib], [torch.from_numpy(m) for m in maps])
    torch.cuda.synchronize()
    counts = counts.cpu().numpy()
    with torch.no_grad():
        ref = O.forward_frame(g['pcd4'], calib, maps, sd, G, synth.KITTI_IMSIZE_HW)
        ref64 = O.forward_frame(g['pcd4'], calib, maps, sd, G, synth.KITTI_IMSIZE_HW, dtype=torch.float64)
    _check_frame(path, 0, ref, ref64, counts, g)
    # compact rows vs the dense reference tensors: voxel columns bit-exact, fused image features toleranced
    N, K = int(counts[0, 0]), int(counts[0, 1])
    cap = path.cap
    row0 = path.region('vox_row0', torch.int32, (1, cap + 1))[0, :N + 1].cpu().numpy()
    cnt = path.region('vox_cnt', torch.int32, (1, cap))[0, :N].cpu().numpy()
    assert row0[N] == K and np.array_equal(cnt, (ref['voxels9'][..., :3] != 0).any(-1).sum(1).numpy())
    # the concat [voxel columns | image features] of MVXNet.py:26: the default inference path builds it inside VFE1's loader
    # (fcn_layer_kernel<16, 1> in csrc/layers.cu); gemm mode 10 materialises it as X6 (prep_vfe1_kernel, what training uses), which is what is read here
    from mvxnet_makise_b200 import _lib
    try:
        _lib.set_gemm_mode(10)
        path([g['pcd4']], [calib], [torch.from_numpy(m) for m in maps])
        torch.cuda.synchronize()
    finally:
        _lib.set_gemm_mode(1)
    x6 = path.region('X6', torch.float32, (1, cap + 128, 32))[0, :K].cpu()
    vox8 = path.region('vox8', torch.float32, (1, cap + 128, 8))[0, :K].cpu()
    assert torch.equal(vox8[:, :7], x6[:, :7])      # the rows VFE1's fused loader reads
    dense_rows = np.concatenate([v * G.T + np.arange(c) for v, c in enumerate(cnt)])
    v9 = ref['voxels9'].reshape(-1, 9)[dense_rows]
    assert torch.equal(x6[:, :7], v9[:, :7]), 'voxel feature columns (x,y,z,dx,dy,dz,r) not bit-exact'
    im16 = ref['im16'].reshape(-1, 16)[dense_rows]
    im16_64 = ref64['im16'].reshape(-1, 16)[dense_rows]
    _check_close(x6[:, 7:23], im16, im16_64, 'fused image features')
    _check_close(x6[:, 7:23], torch.from_numpy(g['im16']).reshape(-1, 16)[dense_rows], im16_64, 'fused image features (golden)')
    # stage 4: exact placement (a copy) and exact zero elsewhere
    gcpu = grid[0].cpu()
    assert tuple(gcpu.shape) == tuple(g['grid_shape'][1:])
    assert same_occupancy(gcpu, ref['grid'][0])
    vfeat, idx = path.voxel_features(0)
    i = idx.cpu()
    assert torch.equal(gcpu[:, i[:, 3], i[:, 1], i[:, 2]].T, vfeat.cpu())
    assert rel_err(gcpu, ref64['grid'][0]) < TOL


def test_grid_fill_rewrites_every_cell(mvx):
    """The plane-sequential fill of the fused path writes every cell of the grid, zeros included: a second run into a
    NaN-filled grid gives the grid of the first run (voxels sharing a sector, sectors at frame / plane borders, an empty
    frame)."""
    sd = synth.make_weights(6)
    maps = [torch.from_numpy(np.concatenate([small_maps(70 + f)[l] for f in range(3)], axis=0)) for l in range(3)]
    frames = [synth.make_points(71, 6000), np.zeros((0, 4), np.float32), synth.make_points(73, 2500)]
    calib = synth.kitti_calib()
    path = mvx.P.PointPath(sd, G)
    ref, counts = path(frames, [calib] * 3, maps)
    ref, counts = ref.clone(), counts.clone()
    path.grid_out.fill_(float('nan'))      # every byte must be rewritten
    out, counts3 = path(frames, [calib] * 3, maps)
    torch.cuda.synchronize()
    assert torch.equal(counts, counts3)
    assert not torch.isnan(out).any() and int((out[1] != 0).sum()) == 0
    occ = (out[0] != 0).any(0)
    assert int(occ.sum()) == int(counts[0, 0])
    # bit-identical where both runs are deterministic (placement, zeros); features may differ in the last bits between two runs
    # (fp64 atomics of the statistics are unordered), so compare values with the run-to-run tolerance
    assert same_occupancy(out, ref)
    assert rel_err(out.cpu(), ref.cpu()) < 1e-5


def test_pixel_first_fcn1_equals_row_first(mvx):
    """fcn1 commutes with the (linear) 4-corner sample: relu(b + sum of 12 weighted rows of Z = F W1^T) must equal
    relu(A1 W1^T + b) on the gathered matrix A1. Compared on the raw fcn1 activations Y1, the BatchNorm sums and the
    final voxel features, for a batch with ragged frames (incl. points that sample the zero pad row/column)."""
    from mvxnet_makise_b200 import _lib
    sd = synth.make_weights(5)
    calib = synth.kitti_calib()
    frames = [synth.make_points(60 + f, P) for f, P in enumerate((1500, 700, 2300))]
    maps = [torch.from_numpy(m) for m in small_maps(9, B=3)]
    out = {}
    try:
        for mode in (0, 1):
            _lib.set_fusion_mode(mode)
            path = mvx.P.PointPath(sd, G)
            _, counts = path(frames, [calib] * 3, maps, want_grid=False)
            torch.cuda.synchronize()
            c = counts.cpu().numpy()
            capA = path.cap + 128
            y1 = path.region('Y1', torch.float32, (3, capA, 768))
            st = path.region('stats', torch.float64, (8, 3, 768, 2))[0]
            out[mode] = ([y1[f, :c[f, 1] + 1].clone() for f in range(3)], st.clone(),
                         [path.voxel_features(f)[0].clone() for f in range(3)])
    finally:
        _lib.set_fusion_mode(1)
    for f in range(3):
        assert rel_err(out[1][0][f], out[0][0][f]) < 1e-5, 'raw fcn1 activations'
        assert rel_err(out[1][2][f], out[0][2][f]) < TOL / 2, 'voxel features'
    assert rel_err(out[1][1], out[0][1]) < 1e-5, 'BatchNorm sums of fcn1'


@pytest.mark.parametrize('scale', [3e4, 1e-5])
@pytest.mark.parametrize('fusion_mode', [1, 0], indirect=True)
def test_fp16_operands_survive_extreme_feature_ranges(mvx, scale, fusion_mode):
    """The 3xFP16 tensor-core layers scale raw inputs by exact powers of two (per pixel row for the pixel GEMM, per gathered
    row for the row-first fcn1, per weight column): FPN features far outside fp16's range (values up to ~1e5, or ~1e-5)
    must give the same fp32-level agreement with the fp64 oracle as O(1) features."""
    sd = synth.make_weights(8)
    calib = synth.kitti_calib()
    pts = synth.make_points(90, 1800)
    maps = [m * np.float32(scale) for m in small_maps(13)]
    path = mvx.P.PointPath(sd, G)
    if fusion_mode == 0:
        from mvxnet_makise_b200.modules import pack_calib
        pd = torch.from_numpy(pts).cuda()
        path.forward_train(pd, [0, pts.shape[0]], pack_calib(calib)[None].cuda(), [torch.from_numpy(m).cuda() for m in maps],
                           want_grid=False, shuffle=False)       # row-first fcn1 in 3xFP16 (per-row scale from the gather)
    else:
        path([pts], [calib], [torch.from_numpy(m) for m in maps], want_grid=False)
    torch.cuda.synchronize()
    with torch.no_grad():
        ref64 = O.forward_frame(pts, calib, maps, sd, G, synth.KITTI_IMSIZE_HW, dtype=torch.float64, want_grid=False)
        ref32 = O.forward_frame(pts, calib, maps, sd, G, synth.KITTI_IMSIZE_HW, want_grid=False)
    vf, idx = path.voxel_features(0)
    assert np.array_equal(idx.cpu().numpy()[:, 1:], ref64['idx'].numpy()[:, 1:])
    # tiny features ride on an O(1e-2) bias: y = relu(b + delta) stored in fp32 keeps delta to ~1e-3 relative in ANY fp32
    # implementation, the reference included, so the bar is TOL on top of the fp32 oracle's own distance to fp64
    noise = rel_err(ref32['vfeat'], ref64['vfeat'])
    e = rel_err(vf, ref64['vfeat'])
    assert torch.isfinite(vf).all() and e < TOL + 2 * noise, (e, noise)
    if scale > 1:
        assert e < TOL


@pytest.mark.parametrize('case', ['path_a', 'path_b', 'shifted', 'large', 'tiny'])
def test_default_path_on_offset_and_extreme_features(mvx, golden_dir, case):
    """The default path meets the fp32 bar (voxel features within 1e-4 of the fp64 oracle) and places the voxels of the
    oracle's grid, also for features with a large common offset (|mean| >> sigma in every channel) and features far outside
    fp16's range."""
    g = np.load(os.path.join(golden_dir, ('path_b' if case == 'path_b' else 'path_a') + '.npz'))
    maps = small_maps(int(g['map_seed']))
    if case == 'shifted':
        maps = [m + np.float32(5.0) for m in maps]
    elif case == 'large':
        maps = [m * np.float32(3e4) for m in maps]
    elif case == 'tiny':
        maps = [m * np.float32(1e-5) for m in maps]
    sd = synth.make_weights(int(g['weight_seed']))
    calib = synth.kitti_calib()
    path = mvx.P.PointPath(sd, G)
    grid, counts = path([g['pcd4']], [calib], [torch.from_numpy(m) for m in maps])
    torch.cuda.synchronize()
    vf, idx = path.voxel_features(0)
    with torch.no_grad():
        ref64 = O.forward_frame(g['pcd4'], calib, maps, sd, G, synth.KITTI_IMSIZE_HW, dtype=torch.float64)
        ref32 = O.forward_frame(g['pcd4'], calib, maps, sd, G, synth.KITTI_IMSIZE_HW)
    noise = rel_err(ref32['vfeat'], ref64['vfeat'])
    e0 = rel_err(vf, ref64['vfeat'])
    print(f'{case}: voxel features vs fp64: {e0:.2e} (fp32 reference {noise:.2e})')
    assert np.array_equal(idx.cpu().numpy()[:, 1:], ref64['idx'].numpy()[:, 1:])
    assert torch.isfinite(vf).all()
    assert same_occupancy(grid[0], ref64['grid'][0])
    assert e0 < (TOL if case != 'tiny' else TOL + 2 * noise), (e0, noise)


def test_tma_fed_tmem_operand_layer_kernel_matches_one_tile_kernel(mvx, golden_dir):
    """Default mode 1: conv1, fcn2 and the last FCN through the persistent TMA-fed kernel (tc3_layer.cu): raw fp32 tiles
    by tensor copy, converter warps, A operand in tensor memory, double-buffered accumulators, tensor-store epilogue. Same
    3xFP16 arithmetic as the one-tile kernel: raw activations and BatchNorm sums agree with it to fp32 accumulation-order
    level, the voxel features meet the fp32 bar against the fp64 oracle; ragged batch with an empty frame, multi-tile frames."""
    from mvxnet_makise_b200 import _lib
    g = np.load(os.path.join(golden_dir, 'path_a.npz'))
    maps = small_maps(int(g['map_seed']))
    sd = synth.make_weights(int(g['weight_seed']))
    calib = synth.kitti_calib()
    frames = [g['pcd4'], synth.make_points(93, 5000), np.zeros((0, 4), np.float32), synth.make_points(94, 777)]
    fm = [torch.from_numpy(np.concatenate([m, small_maps(31)[l], small_maps(32)[l], small_maps(33)[l]], 0)) for l, m in enumerate(maps)]
    _lib.set_gemm_mode(9)                 # the one-tile kernel of tc_layer.cu as the comparison
    base = mvx.P.PointPath(sd, G)
    _, c0 = base(frames, [calib] * 4, fm, want_grid=False)
    _lib.set_gemm_mode(1)
    cap = base.cap
    keep = {n: base.region(n, torch.float32, (4, cap + 128, 128)).clone() for n in ('Y2', 'Y3')}
    st0 = base.region('stats', torch.float64, (8, 4 * 768 * 2)).clone()     # [layer][frame stride = 2 * Cout of the layer]
    vf0 = [base.voxel_features(f)[0].clone() for f in range(4)]
    try:
        _lib.set_gemm_mode(1)
        path = mvx.P.PointPath(sd, G)
        _, counts = path(frames, [calib] * 4, fm, want_grid=False)
        torch.cuda.synchronize()
        assert torch.equal(counts, c0)
        for f in (0, 1, 3):
            K = int(counts[f, 1])
            for n in ('Y2', 'Y3'):       # raw outputs of conv1 / fcn2 (rows 0..K: the kept points + the weighted pad row)
                got = path.region(n, torch.float32, (4, cap + 128, 128))[f, :K + 1]
                assert rel_err(got, keep[n][f, :K + 1]) < 2e-5, (f, n)
            assert rel_err(path.voxel_features(f)[0], vf0[f]) < 2e-5
        st = path.region('stats', torch.float64, (8, 4 * 768 * 2))
        for layer, cout in ((1, 128), (2, 128), (7, 128)):
            for f in (0, 1, 3):
                assert rel_err(st[layer, 2 * cout * f:2 * cout * (f + 1)], st0[layer, 2 * cout * f:2 * cout * (f + 1)]) < 1e-5, (layer, f)
        vf, _ = path.voxel_features(0)
        vf1, _ = path.voxel_features(1)
    finally:
        _lib.set_gemm_mode(1)
    with torch.no_grad():
        ref64 = O.forward_frame(g['pcd4'], calib, maps, sd, G, synth.KITTI_IMSIZE_HW, dtype=torch.float64, want_grid=False)
        ref64b = O.forward_frame(frames[1], calib, [m[1:2].numpy() for m in fm], sd, G, synth.KITTI_IMSIZE_HW, dtype=torch.float64,
                                 want_grid=False)
    assert rel_err(vf, ref64['vfeat']) < TOL and rel_err(vf1, ref64b['vfeat']) < TOL


BF16_TOL = 5e-2


@pytest.mark.parametrize('tag', ['path_a', 'path_b'])
def test_bf16_mode_tolerance(mvx, golden_dir, tag):
    """bf16 mode (mvx_set_gemm_mode(6)): the tensor-core layers of the fused path (pixel GEMM of fcn1, conv1, fcn2, last
    FCN) use ONE bf16 product per K-step instead of the fp32-accurate three-product split. Its tolerance is stated
    separately from the fp32 bar: voxel features within BF16_TOL = 5e-2 (max|a-ref| / max|ref|) of the fp64 evaluation
    (measured 0.6e-2 .. 1.2e-2: 8-bit operand mantissas through 8 BatchNorm-ed layers); voxelization, projection and
    grid placement stay bit-exact (integer / fp32 SIMT work is untouched)."""
    from mvxnet_makise_b200 import _lib
    g = np.load(os.path.join(golden_dir, tag + '.npz'))
    maps = small_maps(int(g['map_seed']))
    sd = synth.make_weights(int(g['weight_seed']))
    calib = synth.kitti_calib()
    try:
        _lib.set_gemm_mode(6)
        path = mvx.P.PointPath(sd, G)
        grid, counts = path([g['pcd4']], [calib], [torch.from_numpy(m) for m in maps])
        torch.cuda.synchronize()
        vf, idx = path.voxel_features(0)
        vf, idx = vf.clone(), idx.clone()
    finally:
        _lib.set_gemm_mode(1)
    with torch.no_grad():
        ref64 = O.forward_frame(g['pcd4'], calib, maps, sd, G, synth.KITTI_IMSIZE_HW, dtype=torch.float64)
    assert np.array_equal(idx.cpu().numpy()[:, 1:], ref64['idx'].numpy()[:, 1:])
    e = rel_err(vf, ref64['vfeat'])
    print(f'bf16 mode: voxel features vs fp64 {e:.3e}')
    assert TOL < e < BF16_TOL, e          # above the fp32 bar (it IS reduced precision), inside its own
    i = idx.cpu()
    assert torch.equal(grid[0].cpu()[:, i[:, 3], i[:, 1], i[:, 2]].T, vf.cpu())


def test_fused_batch_equals_single_frames(mvx):
    """Batch = independent frames with per-frame BatchNorm statistics (SURVEY.md §7 hard part 6)."""
    sd = synth.make_weights(2)
    calib = synth.kitti_calib()
    frames = [synth.make_points(30 + f, P) for f, P in enumerate((900, 2000, 1311))]
    maps = small_maps(77, B=3)
    path = mvx.P.PointPath(sd, G)
    _, counts = path(frames, [calib] * 3, [torch.from_numpy(m) for m in maps], want_grid=False)
    counts = counts.cpu().numpy()
    batch = [tuple(t.clone() for t in path.voxel_features(f)) for f in range(3)]
    for f in range(3):
        with torch.no_grad():
            kw = dict(want_grid=False)
            ref = O.forward_frame(frames[f], calib, [m[f:f + 1] for m in maps], sd, G, synth.KITTI_IMSIZE_HW, **kw)
            ref64 = O.forward_frame(frames[f], calib, [m[f:f + 1] for m in maps], sd, G, synth.KITTI_IMSIZE_HW,
                                    dtype=torch.float64, **kw)
        _check_frame(path, f, ref, ref64, counts)
    for f in range(3):
        single = mvx.P.PointPath(sd, G)
        single([frames[f]], [calib], [torch.from_numpy(m[f:f + 1]) for m in maps], want_grid=False)
        vf, idx = single.voxel_features(0)
        assert torch.equal(idx[:, 1:], batch[f][1][:, 1:])
        assert rel_err(vf, batch[f][0]) < 1e-5      # accumulation order (fp64 atomics, fp32 16-row runs in sorted-row order) is the only difference


@pytest.mark.parametrize('chunk', [1, 2, 8])
def test_host_entry_pipelined_equals_device_entry(mvx, chunk):
    """forward_host cuts the batch into sub-batches (H2D of chunk j+1 overlaps the kernels of chunk j): ragged last
    chunk, per-chunk workspaces, outputs written into slices of the batch outputs. Same results as one batched call."""
    from mvxnet_makise_b200.modules import pack_calib
    sd = synth.make_weights(3)
    calib = synth.kitti_calib()
    frames = [synth.make_points(50 + f, P) for f, P in enumerate((900, 2000, 1311, 640, 1500))]
    B = len(frames)
    maps = [torch.from_numpy(m) for m in small_maps(5, B=B)]
    ref_path = mvx.P.PointPath(sd, G)
    grid_ref, counts_ref = ref_path(frames, [calib] * B, maps)
    feats_ref = [tuple(t.clone() for t in ref_path.voxel_features(f)) for f in range(B)]
    grid_ref, counts_ref = grid_ref.clone(), counts_ref.cpu()
    offsets = np.concatenate([[0], np.cumsum([p.shape[0] for p in frames])]).tolist()
    points_h = torch.from_numpy(np.concatenate(frames, 0)).pin_memory()
    calib_h = torch.stack([pack_calib(calib) for _ in range(B)]).pin_memory()
    maps_h = [m.pin_memory() for m in maps]
    path = mvx.P.PointPath(sd, G)
    path.host_chunk = chunk
    for _ in range(2):                                    # second call reuses the buffers
        grid, counts_h, head = path.forward_host(points_h, offsets, calib_h, maps_h, head_rows=64)
    assert torch.equal(counts_h, counts_ref)
    for f in range(B):
        vf, idx = path.voxel_features(f)
        assert torch.equal(idx, feats_ref[f][1])
        assert rel_err(vf, feats_ref[f][0]) < 1e-5       # accumulation order is the only difference
    assert same_occupancy(grid, grid_ref) and rel_err(grid, grid_ref) < 1e-5
    assert rel_err(head, feats_ref[0][0][:64]) < 1e-5
    assert path.h2d_bytes == (points_h.numel() + calib_h.numel() + sum(m.numel() for m in maps_h)) * 4


def test_host_entry_async_steps_and_capacity_buckets(mvx):
    """forward_host(sync=False): calls are pipelined across steps on two buffer sets; frames whose point counts differ from
    call to call reuse the same contexts (capacity buckets, no re-allocation); a first sub-batch smaller than `head_rows`
    is clamped. Every call's host-visible results equal the synchronous device entry on the same inputs."""
    from mvxnet_makise_b200.modules import pack_calib
    sd = synth.make_weights(3)
    calib = synth.kitti_calib()
    B = 4
    maps = [torch.from_numpy(m) for m in small_maps(6, B=B)]
    maps_h = [m.pin_memory() for m in maps]
    calib_h = torch.stack([pack_calib(calib) for _ in range(B)]).pin_memory()
    path = mvx.P.PointPath(sd, G)
    path.host_chunk = 2
    ref_path = mvx.P.PointPath(sd, G)
    calls, handles = [], []
    for s_ in range(5):                                   # 5 calls on 2 slots: every slot is reused at least once
        frames = [synth.make_points(60 + 7 * s_ + f, 300 + 97 * ((s_ + f) % 4)) for f in range(B)]   # ragged, different every call
        offsets = np.concatenate([[0], np.cumsum([p.shape[0] for p in frames])]).tolist()
        pts_h = torch.from_numpy(np.concatenate(frames, 0)).pin_memory()
        calls.append((frames, offsets, pts_h))
        handles.append(path.forward_host(pts_h, offsets, calib_h, maps_h, head_rows=1024, sync=False))
        if s_ == 0:
            slots = [id(sl) for sl in path._slots]
        if s_ >= 1:                                       # consume the previous step while this one is in flight
            frames_p, _, _ = calls[s_ - 1]
            grid, counts_h, head = handles[s_ - 1].wait()
            g_ref, c_ref = ref_path(frames_p, [calib] * B, maps)
            assert torch.equal(counts_h, c_ref.cpu())
            n0 = int(c_ref[0, 0])
            vf0, _ = ref_path.voxel_features(0)
            assert head.shape[0] <= 1024 and rel_err(head[:min(n0, head.shape[0])], vf0[:head.shape[0]]) < 1e-5
            assert same_occupancy(grid, g_ref) and rel_err(grid, g_ref) < 1e-5
    assert [id(sl) for sl in path._slots] == slots, 'contexts were rebuilt although the capacity bucket did not change'
    handles[-1].wait()


def test_shuffle_option_matches_reference_group_semantics(mvx):
    """The reference shuffles inside `group` (Preprocessing.py:86): above the T cap the kept points are a random T-subset.
    shuffle=True permutes every frame on the device first; the result is bit-identical to the path run on the same
    permutation applied by the caller, the permutation is a per-frame permutation, and voxels above the cap keep a
    different point subset than the caller-order run (it is on by default in training mode, off in inference)."""
    from mvxnet_makise_b200.modules import pack_calib
    sd = synth.make_weights(2)
    calib = synth.kitti_calib()
    frames = [synth.make_points(70, 9000), synth.make_points(71, 5000)]
    frames[0][:600, :3] = frames[0][0, :3]              # one voxel far above the cap of 35
    offsets = [0, 9000, 14000]
    pts = torch.from_numpy(np.concatenate(frames, 0)).cuda()
    c32 = torch.stack([pack_calib(calib)] * 2).cuda()
    maps = [torch.from_numpy(m).cuda() for m in small_maps(4, B=2)]
    path = mvx.P.PointPath(sd, G)
    path.shuffle_generator = torch.Generator(device='cuda').manual_seed(5)
    _, c_sh = path.forward_device(pts, offsets, c32, maps, want_grid=False, shuffle=True)
    perm = path.last_perm.clone()
    assert sorted(perm[:9000].tolist()) == list(range(9000)) and sorted(perm[9000:].tolist()) == list(range(9000, 14000))
    assert not torch.equal(perm, torch.arange(14000, device='cuda'))
    feats_sh = [tuple(t.clone() for t in path.voxel_features(f)) for f in range(2)]
    rp_sh = path.region('row_point', torch.int32, (2, path.cap))[0, :int(c_sh[0, 1])].clone()
    other = mvx.P.PointPath(sd, G)
    _, c_pre = other.forward_device(pts[perm].contiguous(), offsets, c32, maps, want_grid=False, shuffle=False)
    assert other.last_perm is None and torch.equal(c_sh, c_pre)
    for f in range(2):
        vf, idx = other.voxel_features(f)
        assert torch.equal(idx, feats_sh[f][1]) and rel_err(vf, feats_sh[f][0]) < 1e-5   # accumulation order (atomics) is the only difference
    # the oracle on the same permutation: same voxel list, same kept points
    p0 = frames[0][perm[:9000].cpu().numpy()]
    vid, slot, coords, cnt = O.group_assign(O.cell_index(p0, G.velorange, G.voxelsize), G.T)
    assert np.array_equal(feats_sh[0][1][:, 1:].cpu().numpy(), coords) and int(c_sh[0, 1]) == int(cnt.sum())
    # caller order keeps points 0..34 of the crowded voxel; the shuffled run keeps another subset
    _, c_plain = other.forward_device(pts, offsets, c32, maps, want_grid=False)          # inference default: no shuffle
    rp_plain = other.region('row_point', torch.int32, (2, other.cap))[0, :int(c_plain[0, 1])]
    kept_plain = set(rp_plain[rp_plain < 600].tolist())
    kept_sh = set(perm[:9000][rp_sh.long()][perm[:9000][rp_sh.long()] < 600].tolist())
    assert kept_plain == set(range(35)) and 30 <= len(kept_sh) <= 35 and kept_sh != kept_plain   # (the voxel may also hold a few of the frame's own points)
    # training mode shuffles by default
    tr = mvx.P.PointPath(sd, G)
    tr.forward_train(pts, offsets, c32, maps, want_grid=False)
    assert tr.last_perm is not None
    tr.forward_train(pts, offsets, c32, maps, want_grid=False, shuffle=False)
    assert tr.last_perm is None


def test_fused_path_empty_and_tiny_frames(mvx):
    """Ragged batch with an empty frame and a one-point frame, and an all-empty batch: no NaNs, zero grid for empty frames,
    the one-point frame equals the oracle."""
    sd = synth.make_weights(1)
    calib = synth.kitti_calib()
    maps = small_maps(2, B=3)
    frames = [synth.make_points(1, 700), np.zeros((0, 4), np.float32), synth.make_points(2, 1)]
    path = mvx.P.PointPath(sd, G)
    grid, counts = path(frames, [calib] * 3, [torch.from_numpy(m) for m in maps])
    torch.cuda.synchronize()
    c = counts.cpu().numpy()
    assert c[:, 0].tolist() == [c[0, 0], 0, 1] and c[:, 1].tolist() == [700, 0, 1] and c[0, 0] > 0
    assert torch.isfinite(grid).all() and float(grid[1].abs().sum()) == 0.0
    for f in (0, 2):
        with torch.no_grad():
            ref64 = O.forward_frame(frames[f], calib, [m[f:f + 1] for m in maps], sd, G, synth.KITTI_IMSIZE_HW, dtype=torch.float64)
        vf, idx = path.voxel_features(f)
        assert np.array_equal(idx.cpu().numpy()[:, 1:], ref64['idx'].numpy()[:, 1:])
        assert rel_err(vf, ref64['vfeat']) < TOL and rel_err(grid[f], ref64['grid'][0]) < TOL
    assert path.voxel_features(1)[0].shape == (0, 128)
    empty = mvx.P.PointPath(sd, G)
    g2, c2 = empty([np.zeros((0, 4), np.float32)], [calib], [torch.from_numpy(m[:1]) for m in maps])
    torch.cuda.synchronize()
    assert c2.cpu().numpy().tolist() == [[0, 0, 0, 0]] and float(g2.abs().sum()) == 0.0


def test_sparse_cml_conv1_matches_dense_reference(mvx):
    """§8f rank 2: `CML.conv1` (Conv3d 128->64, k 3, stride (2,1,1), pad 1, + ReLU + batch-stat BatchNorm3d) computed
    sparsely from the voxel features equals the dense reference ops applied to the dense grid (small grid so the dense
    fp64 convolution runs in seconds on the CPU). Two frames with different occupancy, per-frame statistics."""
    small = synth.GridSpec((0.0, -4.8, -3.0, 8.0, 4.8, 1.0), (40, 48, 10), 35)
    sd = synth.make_weights(6)
    calib = synth.kitti_calib()
    frames = [synth.make_points(120 + f, P, grid=small) for f, P in enumerate((700, 350))]
    assert all(p.shape[0] > 100 for p in frames)
    maps = small_maps(14, B=2)
    rng = np.random.default_rng(3)
    w = (rng.standard_normal((64, 128, 3, 3, 3)) / np.sqrt(128 * 27)).astype(np.float32)
    b = (rng.standard_normal(64) * 0.1).astype(np.float32)
    path = mvx.P.PointPath(sd, small)
    grid, counts = path(frames, [calib] * 2, [torch.from_numpy(m) for m in maps])
    out = path.cml_conv1(torch.from_numpy(w), torch.from_numpy(b))
    torch.cuda.synchronize()
    assert tuple(out.shape) == (2, 64, 5, 40, 48) and torch.isfinite(out).all()
    for f in range(2):
        with torch.no_grad():
            ref = O.cml_conv1(grid[f:f + 1].double().cpu(), torch.from_numpy(w).double(), torch.from_numpy(b).double())
        assert rel_err(out[f], ref[0]) < TOL, f
    # the dense grid is not needed for it
    path2 = mvx.P.PointPath(sd, small)
    path2(frames, [calib] * 2, [torch.from_numpy(m) for m in maps], want_grid=False)
    assert rel_err(path2.cml_conv1(torch.from_numpy(w), torch.from_numpy(b)), out) < 1e-5


@pytest.mark.parametrize('n_split', [2, 3])
def test_device_split_equals_single_call(mvx, n_split):
    """forward_device_split: sub-batches on concurrent streams with their own workspaces give the batched call's results."""
    from mvxnet_makise_b200.modules import pack_calib
    sd = synth.make_weights(9)
    calib = synth.kitti_calib()
    frames = [synth.make_points(140 + f, P) for f, P in enumerate((800, 1200, 500, 1500, 950))]
    B = len(frames)
    offsets = np.concatenate([[0], np.cumsum([p.shape[0] for p in frames])]).tolist()
    pts = torch.from_numpy(np.concatenate(frames, 0)).cuda()
    c32 = torch.stack([pack_calib(calib) for _ in range(B)]).cuda()
    maps = [torch.from_numpy(m).cuda() for m in small_maps(15, B=B)]
    ref = mvx.P.PointPath(sd, G)
    g_ref, c_ref = ref.forward_device(pts, offsets, c32, maps)
    feats = [tuple(t.clone() for t in ref.voxel_features(f)) for f in range(B)]
    path = mvx.P.PointPath(sd, G)
    g, c = path.forward_device_split(pts, offsets, c32, maps, True, n_split)
    torch.cuda.synchronize()
    # values to rounding (the BatchNorm sums are fp64 atomics in launch-dependent order), occupancy through the voxel lists: a
    # feature that is EXACTLY 0.0 in one run (max == mean) may be 1e-7 in the other, so `g != 0` is not a stable occupancy test
    # (tools/split_stress.py: one such cell on this seed)
    assert torch.equal(c, c_ref) and rel_err(g, g_ref) < 1e-5
    for f in range(B):
        vf, idx = path.voxel_features(f)
        assert torch.equal(idx, feats[f][1]) and rel_err(vf, feats[f][0]) < 1e-5
        i = idx.long()
        occ = torch.zeros(g.shape[2:], dtype=torch.bool, device=g.device)
        occ[i[:, 3], i[:, 1], i[:, 2]] = True
        assert not (g[f][:, ~occ] != 0).any() and not (g_ref[f][:, ~occ] != 0).any()      # exact zero outside the occupied cells
        assert torch.equal(g[f][:, i[:, 3], i[:, 1], i[:, 2]].T, vf)                          # placement: a copy of the features


def test_load_state_dict_reaches_existing_sub_batch_contexts(mvx):
    """load_state_dict after forward_host / forward_device_split have built their sub-batch contexts: the next calls of both
    compute with the new weights, like a fresh PointPath of them."""
    from mvxnet_makise_b200.modules import pack_calib
    sd_a, sd_b = synth.make_weights(4), synth.make_weights(5)
    calib = synth.kitti_calib()
    frames = [synth.make_points(150 + f, P) for f, P in enumerate((700, 1100, 900, 500))]
    B = len(frames)
    offsets = np.concatenate([[0], np.cumsum([p.shape[0] for p in frames])]).tolist()
    pts_h = torch.from_numpy(np.concatenate(frames, 0)).pin_memory()
    c32_h = torch.stack([pack_calib(calib) for _ in range(B)]).pin_memory()
    maps_h = [torch.from_numpy(m).pin_memory() for m in small_maps(16, B=B)]
    pts, c32, maps = pts_h.cuda(), c32_h.cuda(), [m.cuda() for m in maps_h]
    ref = mvx.P.PointPath(sd_b, G)
    ref.forward_device(pts, offsets, c32, maps)
    want = [tuple(t.clone() for t in ref.voxel_features(f)) for f in range(B)]
    path = mvx.P.PointPath(sd_a, G)
    path.host_chunk = 2
    runs = {}
    for sd in ('a', 'b'):
        if sd == 'b':
            path.load_state_dict(sd_b)
        path.forward_host(pts_h, offsets, c32_h, maps_h)
        runs['host', sd] = [tuple(t.clone() for t in path.voxel_features(f)) for f in range(B)]
        path.forward_device_split(pts, offsets, c32, maps, True, n_split=2)
        runs['split', sd] = [tuple(t.clone() for t in path.voxel_features(f)) for f in range(B)]
    for entry in ('host', 'split'):
        assert rel_err(runs[entry, 'a'][0][0], want[0][0]) > 1e-2       # weights A and B give different features
        for f in range(B):
            vf, idx = runs[entry, 'b'][f]
            assert torch.equal(idx, want[f][1]) and rel_err(vf, want[f][0]) < 1e-5, (entry, f)


def test_fused_path_full_size_properties(mvx):
    """BASELINE-size frame (P = 120 000, real FPN shapes): size-independent properties."""
    sd = synth.make_weights(0)
    calib = synth.kitti_calib()
    pts = synth.make_points(0, 120_000)
    maps = [torch.from_numpy(m) for m in synth.make_fpn_maps(0)]
    path = mvx.P.PointPath(sd, G)
    grid, counts = path([pts], [calib], maps)
    torch.cuda.synchronize()
    c = counts.cpu().numpy()[0]
    idx = O.cell_index(pts, G.velorange, G.voxelsize)
    _, _, coords, cnt = O.group_assign(idx, G.T)
    assert c[0] == coords.shape[0] and c[1] == cnt.sum() and c[2] == 0
    vfeat, vidx = path.voxel_features(0)
    assert np.array_equal(vidx[:, 1:].cpu().numpy(), coords)
    assert torch.isfinite(vfeat).all()
    g0 = grid[0]
    assert int((g0 != 0).sum()) == int((vfeat != 0).sum())
    assert torch.equal(g0[:, vidx[:, 3], vidx[:, 1], vidx[:, 2]].T, vfeat)
    # BatchNorm property: over the N*T dense rows every channel of the last layer has mean 0 / var 1; the max over T
    # of such a channel is >= its mean, so every per-voxel max is >= the smallest normalised value (finite, bounded)
    assert float(vfeat.abs().max()) < 1e4


def test_dense_config5_frame(mvx):
    """BASELINE.json configs[4]: dense 128-beam-like frame (P = 250 000) on the larger 512x512x10 grid."""
    DG = synth.DENSE_GRID
    sd = synth.make_weights(0)
    calib = synth.kitti_calib()
    pts = synth.make_points(7, 250_000, grid=DG, beams=128)
    assert pts.shape[0] == 250_000
    maps = [torch.from_numpy(m) for m in synth.make_fpn_maps(7)]
    path = mvx.P.PointPath(sd, DG)
    grid, counts = path([pts], [calib], maps)
    torch.cuda.synchronize()
    c = counts.cpu().numpy()[0]
    idx = O.cell_index(pts, DG.velorange, DG.voxelsize)
    _, _, coords, cnt = O.group_assign(idx, DG.T)
    assert c[0] == coords.shape[0] and c[1] == cnt.sum() and c[2] == 0
    vfeat, vidx = path.voxel_features(0)
    assert np.array_equal(vidx[:, 1:].cpu().numpy(), coords) and torch.isfinite(vfeat).all()
    g0 = grid[0]
    assert tuple(g0.shape) == (128, 10, 512, 512)
    assert int((g0 != 0).sum()) == int((vfeat != 0).sum())
    assert torch.equal(g0[:, vidx[:, 3], vidx[:, 1], vidx[:, 2]].T, vfeat)


def _features_in_mode(mvx, frames, maps, sd, calib, gemm_mode=1, fold_mode=0):
    """Voxel features + raw fcn1 rows of a small batch under one kernel selection (restores the defaults afterwards)."""
    from mvxnet_makise_b200 import _lib
    try:
        _lib.set_gemm_mode(gemm_mode)
        _lib.set_fold_mode(fold_mode)
        path = mvx.P.PointPath(sd, G)
        path(frames, [calib] * len(frames), [torch.from_numpy(m) for m in maps], want_grid=False)
        torch.cuda.synchronize()
        counts = path.counts.cpu().numpy()
        feats = [path.voxel_features(f)[0].clone() for f in range(len(frames))]
        capA = path.cap + 128
        y1 = path.region('Y1', torch.float32, (len(frames), capA, 768)).clone()
        return feats, y1, counts
    finally:
        _lib.set_gemm_mode(1)
        _lib.set_fold_mode(0)


def test_run_structured_combine_equals_row_by_row_kernel(mvx):
    """The run-structured combine kernel (default: per-warp cp.async corner ring, branch-free runs) against the first-generation
    kernel (mvx_set_fold_mode(2)): the raw fcn1 rows Y1 are BIT-IDENTICAL (same arithmetic in the same order), the voxel features
    agree to rounding (the BatchNorm sums group their fp32 partial sums differently). Frames include an empty one, a tiny one
    (a single CTA with one run) and duplicates of one point (long runs in one cell)."""
    sd = synth.make_weights(12)
    calib = synth.kitti_calib()
    dup = np.repeat(synth.make_points(151, 40)[:3], 300, axis=0)      # 900 points in three cells: runs longer than 16 rows
    frames = [synth.make_points(150, 2600), np.zeros((0, 4), np.float32), synth.make_points(152, 37), dup]
    maps = small_maps(21, B=len(frames))
    new, y1_new, c_new = _features_in_mode(mvx, frames, maps, sd, calib, fold_mode=0)
    old, y1_old, c_old = _features_in_mode(mvx, frames, maps, sd, calib, fold_mode=2)
    assert np.array_equal(c_new, c_old)
    for f in range(len(frames)):
        K = int(c_new[f, 1])
        assert torch.equal(y1_new[f, :K + 1], y1_old[f, :K + 1]), f'frame {f}: raw fcn1 rows differ'
        if old[f].numel():
            # frames of a few dozen rows: batch statistics over so few rows amplify the regrouped fp32 partial sums (measured 9.5e-5)
            assert rel_err(new[f], old[f]) < (1e-5 if K > 2000 else 1e-3), f


def test_vfe_inputs_built_in_the_loader_equal_materialised_inputs(mvx):
    """Inference builds VFE1's [vox7 | norm5(Y5)] and VFE2's [norm6(Y6) | norm6(max6[v])] rows inside the layer kernel's tile
    loader; mvx_set_gemm_mode(10) materialises them with prep_vfe1 / prep_vfe2 as training does. Same arithmetic: the voxel
    features agree to rounding; voxels at the T cap (no pad row weight) and single-point voxels are in the mix."""
    sd = synth.make_weights(13)
    calib = synth.kitti_calib()
    crowd = synth.make_points(161, 30)
    crowd = np.concatenate([np.repeat(crowd[:1], 60, axis=0), crowd])     # one voxel beyond the cap of 35
    frames = [synth.make_points(160, 3100), crowd]
    maps = small_maps(22, B=len(frames))
    fused, _, c1 = _features_in_mode(mvx, frames, maps, sd, calib, gemm_mode=1)
    mat, _, c2 = _features_in_mode(mvx, frames, maps, sd, calib, gemm_mode=10)
    assert np.array_equal(c1, c2)
    for f in range(len(frames)):
        # same arithmetic; what differs is the order of the fp64 atomics of the statistics (amplified in a frame of a few dozen rows)
        assert rel_err(fused[f], mat[f]) < (1e-5 if c1[f, 1] > 2000 else 1e-3), f


def test_persistent_pixel_gemm_equals_one_tile_kernel(mvx):
    """The persistent per-pixel GEMM of fcn1 (default) against the one-tile kernel it replaced (mvx_set_gemm_mode(12)): same
    pre-packed operands, same sequence of tensor-core products per accumulator, same exact power-of-two rescale - the per-pixel
    products Z are BIT-IDENTICAL, including the partial last row tile of every level and a level smaller than one tile."""
    from mvxnet_makise_b200 import _lib
    sd = synth.make_weights(14)
    calib = synth.kitti_calib()
    frames = [synth.make_points(170, 1800), synth.make_points(171, 900), synth.make_points(172, 1200)]
    maps = small_maps(23, B=len(frames))
    npix = sum(m.shape[0] * m.shape[2] * m.shape[3] for m in maps)
    out = {}
    for mode in (1, 12):
        try:
            _lib.set_gemm_mode(mode)
            path = mvx.P.PointPath(sd, G)
            path(frames, [calib] * len(frames), [torch.from_numpy(m) for m in maps], want_grid=False)
            torch.cuda.synchronize()
            out[mode] = (path.region('Z', torch.float32, (npix, 768)).clone(), [path.voxel_features(f)[0].clone() for f in range(len(frames))])
        finally:
            _lib.set_gemm_mode(1)
    assert torch.isfinite(out[1][0]).all() and out[1][0].abs().max() > 0
    assert torch.equal(out[1][0], out[12][0]), 'per-pixel products differ between the two kernels'
    for a, b in zip(out[1][1], out[12][1]):
        assert rel_err(a, b) < 1e-4      # frames of ~1 000 rows: run-to-run order of the statistics' atomics
