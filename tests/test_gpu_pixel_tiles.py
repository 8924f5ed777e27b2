"""Active pixel tiles of the pixel-first fcn1: the per-pixel GEMM multiplies only the 256-row tiles of Z that some point's clamped
corners fall in (csrc/gather.cu tile_mark_kernel / tile_list_kernel) and writes zeros into the others.

Checks: (i) the device's tile list equals a numpy restatement of the mark on the benchmark batch and covers every corner the
kept rows sample; (ii) Z of inactive tiles is exactly zero and active tiles equal the one-tile kernel (gemm mode 12) bit for bit;
(iii) NaN poison: with Z filled with NaN between two calls on different frames, the features stay finite and within 1e-4 of the
fp64 oracle - a Z row read outside what the second call rewrote would turn the BatchNorm sums, and then every feature, into NaN."""
import numpy as np
import pytest
import torch

from mvxnet_makise_b200 import synth
from oracle import pointpath_oracle as O

pytestmark = pytest.mark.gpu
G = synth.KITTI_GRID
SMALL_FPN = ((13, 42), (7, 21), (4, 11))
TILE = 256


def maps_for(seed, shapes, B):
    rng = np.random.default_rng(seed)
    return [torch.from_numpy(rng.standard_normal((B, 256, h, w), dtype=np.float32)) for (h, w) in shapes]


def rel(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def tile_counts(B, shapes):
    return [-(-B * h * w // TILE) for h, w in shapes]


def device_tiles(path, shapes):
    """(active entries as (level, tile) tuples in list order, inactive entries, level starts, entries zeroed by this call) from
    the workspace region [bitmap | zero-state bitmap | list | meta]"""
    nt = tile_counts(path.B, shapes)
    words = sum(-(-n // 32) for n in nt)
    total = sum(nt)
    raw = path.region('tiles', torch.int32, (2 * words + total + 8,)).cpu().numpy()
    lst, meta = raw[2 * words:2 * words + total], raw[2 * words + total:]
    dec = [(int(e) >> 24, int(e) & 0xFFFFFF) for e in lst]
    return dec[:meta[3]], dec[meta[3]:], meta[:4].tolist(), dec[meta[3]:meta[4]]


def corner_tiles(proj_rc, f, shapes, eps=1e-6):
    """tiles of the clamped corners (gather.cuh corner_pos) of (row, col) projections of frame f, per level, fp32 index math"""
    H_img, W_img = synth.KITTI_IMSIZE_HW
    out = []
    for h, w in shapes:
        rs = np.array([np.float32(H_img) / np.float32(h), np.float32(W_img) / np.float32(w)], np.float32)
        q = (proj_rc.astype(np.float32) / rs) - np.float32(eps)
        i0, i1 = q[:, 0].astype(np.int64), q[:, 1].astype(np.int64)     # truncation toward zero, like (int)
        ys = [np.clip(i0, 0, h - 1), np.clip(i0 + 1, 0, h - 1)]
        xs = [np.clip(i1, 0, w - 1), np.clip(i1 + 1, 0, w - 1)]
        t = set()
        for y in ys:
            for x in xs:
                t.update(((f * h * w + y * w + x) // TILE).tolist())
        out.append(t)
    return out


def mark_numpy(frames, calib, shapes):
    """the mark restated: in-grid (fp64 cell index), not at the origin, oracle projection, clamped corners"""
    lo, size, shape = np.array(G.velorange[:3], np.float64), np.array(G.voxelsize, np.float64), np.array(G.voxelshape)
    act = [set() for _ in shapes]
    for f, pts in enumerate(frames):
        idx = np.trunc((pts[:, :3].astype(np.float64) - lo) / size).astype(np.int64)
        keep = np.all((idx >= 0) & (idx < shape), axis=1) & ~np.all(pts[:, :3] == 0, axis=1)
        proj = O.points_with_proj(pts[keep], calib)[:, 4:6]
        for l, t in enumerate(corner_tiles(proj, f, shapes)):
            act[l] |= t
    return sorted((l, t) for l in range(len(shapes)) for t in act[l])


def test_tile_list_matches_numpy_mark_on_bench_batch():
    from mvxnet_makise_b200.pipeline import PointPath
    shapes = synth.fpn_shapes()
    frames = [synth.make_points(g, 120_000) for g in range(8)]
    calib = synth.kitti_calib()
    path = PointPath(synth.make_weights(0), G)
    _, counts = path(frames, [calib] * 8, maps_for(1, shapes, 8), want_grid=False)
    torch.cuda.synchronize()
    active, inactive, starts, zeroed = device_tiles(path, shapes)
    assert zeroed == inactive      # a new workspace: every inactive tile is written
    want = mark_numpy(frames, calib, shapes)
    assert active == want, f'{len(active)} active tiles on the device, {len(want)} in the numpy mark'
    nt = tile_counts(8, shapes)
    assert sorted(active + inactive) == [(l, t) for l in range(3) for t in range(nt[l])] and inactive == sorted(inactive)
    assert starts == [sum(1 for e in active if e[0] < l) for l in range(4)]
    assert 0.5 * sum(nt) < len(active) < 0.8 * sum(nt), (len(active), sum(nt))   # the upper image is never sampled
    # invariant: every corner a kept row samples lies in an active tile
    counts = counts.cpu().numpy()
    proj = path.region('proj', torch.float32, (8, path.cap + 128, 2)).cpu().numpy()
    vox8 = path.region('vox8', torch.float32, (8, path.cap + 128, 8)).cpu().numpy()
    aset = set(active)
    for f in range(8):
        K = int(counts[f, 1])
        real = ~np.all(vox8[f, :K, :3] == 0, axis=1)
        for l, t in enumerate(corner_tiles(proj[f, :K][real], f, shapes)):
            assert {(l, x) for x in t} <= aset, f'frame {f} level {l}: a kept row samples an inactive tile'


def test_inactive_tiles_zero_and_active_tiles_equal_one_tile_kernel():
    from mvxnet_makise_b200 import _lib
    from mvxnet_makise_b200.pipeline import PointPath
    shapes = synth.fpn_shapes()
    frames = [synth.make_points(300 + f, 30_000) for f in range(3)]
    maps = maps_for(7, shapes, 3)
    npix = sum(3 * h * w for h, w in shapes)
    out = {}
    for mode in (1, 12):
        try:
            _lib.set_gemm_mode(mode)
            path = PointPath(synth.make_weights(5), G)
            path(frames, [synth.kitti_calib()] * 3, maps, want_grid=False)
            torch.cuda.synchronize()
            out[mode] = (path.region('Z', torch.float32, (npix, 768)).clone(), device_tiles(path, shapes))
        finally:
            _lib.set_gemm_mode(1)
    z, (active, inactive, _, _) = out[1]
    assert out[12][1][0] == active and len(inactive) > 0
    assert torch.isfinite(z).all() and torch.equal(z, out[12][0])
    base = np.cumsum([0] + [3 * h * w for h, w in shapes])
    zc = z.cpu()
    for l, t in inactive:
        r0, r1 = base[l] + t * TILE, min(base[l] + (t + 1) * TILE, base[l + 1])
        assert not zc[r0:r1].any(), f'level {l} tile {t} not zero'
    for l, t in active[:: max(1, len(active) // 50)]:
        assert zc[base[l] + t * TILE:min(base[l] + (t + 1) * TILE, base[l + 1])].any()


def _poisoned_run(first, second, calibs1, calibs2, shapes, B, seed=3):
    """run `first`, fill Z with NaN, run `second`; return the path and its maps"""
    from mvxnet_makise_b200.pipeline import PointPath
    sd = synth.make_weights(seed)
    path = PointPath(sd, G)
    path(first, calibs1, maps_for(seed + 10, shapes, B), want_grid=False)
    torch.cuda.synchronize()
    npix = sum(B * h * w for h, w in shapes)
    path.region('Z', torch.float32, (npix, 768)).fill_(float('nan'))
    maps = maps_for(seed + 20, shapes, B)
    _, counts = path(second, calibs2, maps, want_grid=False)
    torch.cuda.synchronize()
    return path, sd, [m.numpy() for m in maps], counts.cpu().numpy()


def _check_against_oracle(path, sd, maps, counts, frames, calibs, shapes):
    for f, (pts, cal) in enumerate(zip(frames, calibs)):
        with torch.no_grad():
            ref64 = O.forward_frame(pts, cal, [m[f:f + 1] for m in maps], sd, G, synth.KITTI_IMSIZE_HW, dtype=torch.float64,
                                    want_grid=False)
        assert counts[f, 0] == ref64['idx'].shape[0]
        vfeat, idx = path.voxel_features(f)
        assert torch.isfinite(vfeat).all(), f'frame {f}: NaN features (a Z row outside the rewritten set was read)'
        assert np.array_equal(idx.cpu().numpy()[:, 1:], ref64['idx'].numpy()[:, 1:])
        assert rel(vfeat, ref64['vfeat']) < 1e-4


def test_nan_poison_golden_frames(golden_dir):
    import os
    a, b = (np.load(os.path.join(golden_dir, t + '.npz'))['pcd4'] for t in ('path_a', 'path_b'))
    calib = synth.kitti_calib()
    for first, second in ((a, b), (b, a)):
        path, sd, maps, counts = _poisoned_run([first], [second], [calib], [calib], SMALL_FPN, 1)
        _check_against_oracle(path, sd, maps, counts, [second], [calib], SMALL_FPN)


def border_points(seed, n, calib, reach=50.0):
    """in-grid points that project onto the image border or up to `reach` pixels outside it (above / left of the image: the
    corner row / column -1 is the zero pad of Pipe.py:47-48; a point on the last pixel row / column has its second corner on
    the pad). The combine loads the clamped border pixels for the pad corners, with weight 0."""
    rng = np.random.default_rng(seed)
    lo, hi = np.array(G.velorange[:3], np.float32), np.array(G.velorange[3:], np.float32)
    H, W = synth.KITTI_IMSIZE_HW
    out = []
    while sum(len(o) for o in out) < n:
        p = np.concatenate([rng.uniform(lo, hi, (200_000, 3)).astype(np.float32), rng.uniform(0, 1, (200_000, 1)).astype(np.float32)], 1)
        rc = O.points_with_proj(p, calib)[:, 4:6]
        inside = (rc[:, 0] > -reach) & (rc[:, 0] < H) & (rc[:, 1] > -reach) & (rc[:, 1] < W)
        border = (rc[:, 0] < 0) | (rc[:, 1] < 0) | (rc[:, 0] >= H - 25) | (rc[:, 1] >= W - 25)
        out.append(p[inside & border])
    return np.concatenate(out)[:n]


def test_nan_poison_points_on_and_outside_the_image_border():
    calib = synth.kitti_calib()
    first = [synth.make_points(80 + f, 3000) for f in range(2)]
    second = [np.concatenate([synth.make_points(90 + f, 2000), border_points(f, 600, calib)]) for f in range(2)]
    H, W = synth.KITTI_IMSIZE_HW
    rc = O.points_with_proj(second[0], calib)[:, 4:6]
    assert (rc[:, 1] < 0).sum() > 20 and (rc[:, 0] >= H - 25).sum() > 20 and (rc[:, 1] >= W - 25).sum() > 20
    path, sd, maps, counts = _poisoned_run(first, second, [calib] * 2, [calib] * 2, SMALL_FPN, 2)
    _check_against_oracle(path, sd, maps, counts, second, [calib] * 2, SMALL_FPN)


def test_nan_poison_merged_sets_with_float64_calibration():
    """merged point sets, the scene and a pasted set projected in fp64 from float64 calibrations (point_calib / calib_f64)"""
    c64 = synth.kitti_calib_f64()
    c32 = synth.kitti_calib()
    scene = synth.make_points(70, 2500)
    near = synth.make_points(71, 20_000)
    near = O.crop_to_sight(near[(near[:, 0] > 8) & (near[:, 0] < 12)], c32, (synth.KITTI_IMSIZE_HW[1], synth.KITTI_IMSIZE_HW[0]))[:400]
    assert near.shape[0] > 50
    frames2 = [[scene, near]]
    cals2 = [[c64, c64]]
    path, sd, maps, counts = _poisoned_run([synth.make_points(72, 2000)], frames2, [c32], cals2, SMALL_FPN, 1)
    with torch.no_grad():
        ref64 = O.forward_frame([scene, near], [c64, c64], [m[0:1] for m in maps], sd, G, synth.KITTI_IMSIZE_HW,
                                dtype=torch.float64, want_grid=False)
    vfeat, idx = path.voxel_features(0)
    assert torch.isfinite(vfeat).all()
    assert np.array_equal(idx.cpu().numpy()[:, 1:], ref64['idx'].numpy()[:, 1:])
    assert rel(vfeat, ref64['vfeat']) < 1e-4


def test_nan_poison_frames_on_tile_boundaries():
    """level 1 has exactly 256 pixels per frame (every frame is one tile), level 2 has 128 (frames 0/1 share a tile, frame 2
    starts one): the clamped corners of border points land on the first and last row of a tile"""
    shapes = ((16, 64), (8, 32), (8, 16))
    calib = synth.kitti_calib()
    first = [synth.make_points(110 + f, 2500) for f in range(3)]
    second = [np.concatenate([synth.make_points(120 + f, 2000), border_points(10 + f, 400, calib, reach=20.0)]) for f in range(3)]
    path, sd, maps, counts = _poisoned_run(first, second, [calib] * 3, [calib] * 3, shapes, 3)
    active = device_tiles(path, shapes)[0]
    assert {(1, 0), (1, 1), (1, 2), (2, 0), (2, 1)} <= set(active)
    _check_against_oracle(path, sd, maps, counts, second, [calib] * 3, shapes)


def test_zero_state_across_calls_and_dtypes():
    """The workspace remembers which tiles of Z hold zeros: a repeated batch rewrites no zeros, a batch with other frames zeroes
    exactly the tiles that were active and no longer are, and switching Z to bf16 starts over. After every call Z equals what a
    new path computes on the same inputs, bit for bit (inactive tiles zero)."""
    from mvxnet_makise_b200 import _lib
    from mvxnet_makise_b200.pipeline import PointPath
    shapes = synth.fpn_shapes()
    calib = [synth.kitti_calib()] * 2
    fa = [synth.make_points(400 + f, 20_000) for f in range(2)]
    fb = [synth.make_points(410 + f, 20_000) for f in range(2)]
    fb[1] = fb[1][fb[1][:, 0] > 25]     # far points only: the near rows of frame 1 go inactive
    maps = maps_for(9, shapes, 2)
    sd = synth.make_weights(8)
    npix = sum(2 * h * w for h, w in shapes)

    def z_of(path, dtype=torch.float32):
        return path.region('Z', dtype, (npix, 768)).clone()

    path = PointPath(sd, G)
    path(fa, calib, maps, want_grid=False)
    act_a = set(device_tiles(path, shapes)[0])
    path(fa, calib, maps, want_grid=False)
    torch.cuda.synchronize()
    assert device_tiles(path, shapes)[3] == []          # the same batch again: nothing to zero
    path(fb, calib, maps, want_grid=False)
    torch.cuda.synchronize()
    act_b, _, _, zeroed = device_tiles(path, shapes)
    assert set(zeroed) == act_a - set(act_b) and len(zeroed) > 0
    fresh = PointPath(sd, G)
    fresh(fb, calib, maps, want_grid=False)
    torch.cuda.synchronize()
    assert torch.equal(z_of(path), z_of(fresh))
    try:
        _lib.set_gemm_mode(6)        # bf16 mode: Z holds bf16 elements, the zero state of the fp32 layout does not apply
        path(fb, calib, maps, want_grid=False)
        fresh2 = PointPath(sd, G)
        fresh2(fb, calib, maps, want_grid=False)
        torch.cuda.synchronize()
        assert device_tiles(path, shapes)[3] == device_tiles(path, shapes)[1]
        assert torch.equal(z_of(path, torch.int16), z_of(fresh2, torch.int16))
    finally:
        _lib.set_gemm_mode(1)
