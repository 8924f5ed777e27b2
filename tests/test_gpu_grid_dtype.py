"""The dense grid written in fp16 / bf16 (PointPath.grid_dtype, accelerate(grid_dtype=...), modules.reindex(dtype=...)).

Every element of a 16-bit grid is one fp32 voxel feature rounded once to nearest-even, so each grid is compared BIT FOR BIT with
a torch index_put_ of the voxel features of the same forward followed by `.to(dtype)` (two fp32 forwards are not bit-identical:
the BatchNorm sums use unordered fp64 atomics)."""
import copy
import os

import numpy as np
import pytest
import torch

from mvxnet_makise_b200 import synth
from mvxnet_makise_b200.modules import pack_calib, reindex
from mvxnet_makise_b200.pipeline import PointPath

pytestmark = pytest.mark.gpu
HALF = [torch.float16, torch.bfloat16]
SMALL_FPN = ((13, 42), (7, 21), (4, 11))
RAGGED = synth.GridSpec((0.0, -4.6, -3.0, 7.6, 4.6, 1.0), (38, 46, 10), 35)     # 17 480 cells: not a multiple of 32
ENTRIES = ['points', 'voxels', 'train', 'split', 'host']


@pytest.fixture(autouse=True)
def _restore_tf32_flags():
    flags = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = flags
    torch.cuda.empty_cache()


def bits(t):
    return t.contiguous().view(torch.int16)


def small_maps(seed, B=1):
    rng = np.random.default_rng(seed)
    return [torch.from_numpy(rng.standard_normal((B, 256, h, w), dtype=np.float32)).cuda() for h, w in SMALL_FPN]


class Batch:
    """point-entry inputs on the device (and the host copies forward_host reads)"""

    def __init__(self, frames, maps, sd, grid=synth.KITTI_GRID, voxels=None):
        self.frames, self.maps, self.sd, self.grid, self.voxels = frames, maps, sd, grid, voxels
        self.offsets = np.concatenate([[0], np.cumsum([p.shape[0] for p in frames])]).tolist()
        self.points_h = torch.from_numpy(np.concatenate(frames, 0)).pin_memory()
        self.points = self.points_h.cuda()
        self.calib_h = torch.stack([pack_calib(synth.kitti_calib()) for _ in frames]).pin_memory()
        self.calib = self.calib_h.cuda()


def golden(tag):
    g = np.load(os.path.join(os.path.dirname(__file__), 'golden', tag + '.npz'))
    idx = torch.from_numpy(g['idx']).to(torch.int64)
    if idx.shape[1] == 3:
        idx = torch.cat([torch.zeros((idx.shape[0], 1), dtype=torch.int64), idx], 1)
    vox = torch.from_numpy(g['voxels9_after']).float()
    return Batch([g['pcd4']], small_maps(int(g['map_seed'])), synth.make_weights(int(g['weight_seed'])), voxels=(vox, idx))


def bench_batch(B=8, voxels=False):
    """bench.py's forward inputs; voxels=True also builds each frame's (voxels, idx) for the dense-voxel entry the way train.py:44
    does (projection, then `group`), on the GPU"""
    frames = [synth.make_points(f, 120_000) for f in range(B)]
    maps = [torch.from_numpy(np.concatenate([synth.make_fpn_maps(f)[l] for f in range(B)], 0)).cuda() for l in range(3)]
    vox = None
    if voxels:
        from mvxnet_makise_b200.voxelize import group
        from oracle import pointpath_oracle as O
        g, vl, il = synth.KITTI_GRID, [], []
        for p in frames:
            v, i = group(np.ascontiguousarray(O.points_with_proj(p, synth.kitti_calib()), dtype=np.float32), g.velorange, g.voxelsize,
                         g.T, shuffle=False, voxelshape=g.voxelshape, device_out=True)
            vl.append(v)
            il.append(torch.cat([torch.zeros((i.shape[0], 1), dtype=torch.int64, device=i.device), i], 1))
        vox = (vl, il)
    return Batch(frames, maps, synth.make_weights(0), voxels=vox)


def run(path, entry, b):
    """one forward through `entry`; the returned grid was NaN-filled before a second identical forward, so every cell is rewritten"""
    def once():
        if entry == 'points':
            return path.forward_device(b.points, b.offsets, b.calib, b.maps)[0]
        if entry == 'voxels':
            vox, idx = b.voxels
            if isinstance(vox, list):      # one (voxels, idx) pair per frame
                return path.forward_voxels([v.clone() for v in vox], idx, b.maps)[0]
            return path.forward_voxels(vox.cuda(), idx.cuda(), b.maps)[0]
        if entry == 'train':
            return path.forward_train(b.points, b.offsets, b.calib, b.maps, shuffle=False)[0]
        if entry == 'split':
            return path.forward_device_split(b.points, b.offsets, b.calib, b.maps, n_split=2)[0]
        path.host_slots = 1
        return path.forward_host(b.points_h, b.offsets, b.calib_h, b.maps)[0]
    once().fill_(float('nan'))
    grid = once()
    torch.cuda.synchronize()
    return grid


def check_grid(path, grid, dtype, B):
    nz, nx, ny = path.grid.shape[2], path.grid.shape[0], path.grid.shape[1]
    assert grid.dtype == dtype and tuple(grid.shape) == (B, 128, nz, nx, ny)
    for f in range(B):
        vfeat, idx = path.voxel_features(f)
        ref = torch.zeros((nz, nx, ny, 128), dtype=torch.float32, device=grid.device)
        ref.index_put_((idx[:, 3], idx[:, 1], idx[:, 2]), vfeat)
        assert torch.equal(bits(grid[f]), bits(ref.permute(3, 0, 1, 2).to(dtype))), f'frame {f}'


def voxel_lists(path, B):
    return path.counts.cpu().clone(), [path.voxel_features(f)[1].cpu() for f in range(B)]


def check_entry(b, entry, dtype):
    B = len(b.frames)
    ref = PointPath(b.sd, b.grid)
    run(ref, entry, b)
    counts32, idx32 = voxel_lists(ref, B)
    del ref
    path = PointPath(b.sd, b.grid, grid_dtype=dtype)
    grid = run(path, entry, b)
    check_grid(path, grid, dtype, B)
    counts, idx = voxel_lists(path, B)
    assert torch.equal(counts, counts32) and all(torch.equal(a, c) for a, c in zip(idx, idx32))


@pytest.mark.parametrize('dtype', HALF)
@pytest.mark.parametrize('entry', ENTRIES)
@pytest.mark.parametrize('tag', ['path_a', 'path_b'])
def test_golden_frames_every_entry(tag, entry, dtype):
    check_entry(golden(tag), entry, dtype)


@pytest.fixture(scope='module')
def bench():
    return bench_batch(voxels=True)


@pytest.mark.parametrize('dtype', HALF)
@pytest.mark.parametrize('entry', ENTRIES)
def test_bench_batch_every_entry(bench, entry, dtype):
    check_entry(bench, entry, dtype)


@pytest.mark.parametrize('dtype', HALF)
def test_ragged_grid_empty_frame_and_dense_frame(dtype):
    # ragged kernel (G % 32 != 0)
    frames = [synth.make_points(80 + f, 2500, grid=RAGGED) for f in range(2)]
    b = Batch(frames, small_maps(3, B=2), synth.make_weights(1), grid=RAGGED)
    path = PointPath(b.sd, RAGGED, grid_dtype=dtype)
    check_grid(path, run(path, 'points', b), dtype, 2)
    # an empty frame between two others: its grid is all zero
    frames = [synth.make_points(71, 6000), np.zeros((0, 4), np.float32), synth.make_points(73, 2500)]
    b = Batch(frames, small_maps(4, B=3), synth.make_weights(6))
    path = PointPath(b.sd, grid_dtype=dtype)
    grid = run(path, 'points', b)
    check_grid(path, grid, dtype, 3)
    assert int(path.counts[1, 0]) == 0 and not bool(bits(grid[1]).any())
    # one frame of the dense configuration
    b = Batch([synth.make_points(5, 250_000, grid=synth.DENSE_GRID, beams=128)],
              [torch.from_numpy(m).cuda() for m in synth.make_fpn_maps(5)], synth.make_weights(0), grid=synth.DENSE_GRID)
    path = PointPath(b.sd, synth.DENSE_GRID, grid_dtype=dtype)
    check_grid(path, run(path, 'points', b), dtype, 1)


def test_backward_reads_the_half_gradient():
    b = bench_batch(2)
    path = PointPath(b.sd, grid_dtype=torch.float16)
    grid, counts = path.forward_train(b.points, b.offsets, b.calib, b.maps, shuffle=False)
    h = torch.randn(grid.shape, generator=torch.Generator(device='cuda').manual_seed(0), device='cuda').to(torch.float16)
    flat1 = path.backward(d_grid=h).clone()
    flat2 = path.backward(d_grid=h).clone()
    dv = torch.zeros((2, path.cap, 128), dtype=torch.float32, device='cuda')
    for f in range(2):
        vfeat, idx = path.voxel_features(f)
        dv[f, :idx.shape[0]] = h[f].float()[:, idx[:, 3], idx[:, 1], idx[:, 2]].t()
    flat3 = path.backward(d_vfeat=dv).clone()
    torch.cuda.synchronize()
    repeat = float((flat2 - flat1).abs().max())
    assert float((flat3 - flat1).abs().max()) <= 2 * repeat
    assert torch.isfinite(flat1).all() and float(flat1.abs().max()) > 0
    with pytest.raises(ValueError):
        path.backward(d_grid=h.float())
    with pytest.raises(ValueError):
        path.backward(d_grid=h.to(torch.bfloat16))


@pytest.mark.parametrize('dtype', HALF)
@pytest.mark.parametrize('shape', [(40, 48, 10), (38, 46, 10)])
def test_reindex_dropin(dtype, shape):
    nx, ny, nz = shape
    g = torch.Generator().manual_seed(7)
    cells = torch.randperm(nx * ny * nz, generator=g)[:900]
    idx = torch.stack([torch.zeros_like(cells), cells // nz // ny % nx, cells // nz % ny, cells % nz], 1).cuda()
    x = torch.randn((900, 128), generator=g).cuda().requires_grad_(True)
    out = reindex(x, idx, shape, dtype=dtype)
    ref = torch.zeros((nz, nx, ny, 128), device='cuda')
    ref.index_put_((idx[:, 3], idx[:, 1], idx[:, 2]), x.detach())
    assert out.dtype == dtype and torch.equal(bits(out[0]), bits(ref.permute(3, 0, 1, 2).to(dtype)))
    grad = torch.randn(out.shape, generator=g).cuda().to(dtype)
    out.backward(grad)
    want = grad[0].float()[:, idx[:, 3], idx[:, 1], idx[:, 2]].t()
    assert x.grad.dtype == x.dtype and torch.equal(x.grad, want)


# ---- accelerate on the stand-in module tree of test_gpu_map_backward ------------------------------------------------------
def _grid_seen(m):
    seen = []
    m.backbone.cml.register_forward_pre_hook(lambda mod, inp: seen.append(inp[0].detach().clone()))
    return seen


def _scaler_step(model, voxel, idx, init_scale=2.0 ** 16):
    from test_gpu_map_backward import _run
    opt = torch.optim.SGD(model.parameters(), lr=1e-2)
    scaler = torch.amp.GradScaler('cuda', init_scale=init_scale)
    with torch.autocast('cuda', torch.float16):
        out = _run(model, voxel, idx)             # the stand-in's RPN is one Conv2d: a single tensor
        loss = out.float().pow(2).mean()
    scaler.scale(loss).backward()
    scaler.step(opt)
    scaler.update()
    return scaler


def test_accelerate_autocast_grid():
    from mvxnet_makise_b200.dropin import accelerate, hot_parameters
    from test_gpu_map_backward import SMALL, _frame_inputs, _run, _standin
    torch.backends.cudnn.allow_tf32 = False
    voxel, idx = _frame_inputs(37, 1300)
    base, _ = _standin(7)
    m = accelerate(copy.deepcopy(base), grid=SMALL, grid_dtype='autocast')
    seen = _grid_seen(m)
    with torch.autocast('cuda', torch.float16):
        _run(m, voxel, idx)
    path = m._mvx_path
    vfeat, vidx = path.voxel_features(0)
    nz, (nx, ny) = SMALL.voxelshape[2], SMALL.voxelshape[:2]
    ref = torch.zeros((nz, nx, ny, 128), device='cuda')
    ref.index_put_((vidx[:, 3], vidx[:, 1], vidx[:, 2]), vfeat)
    assert seen[-1].dtype == torch.float16 and torch.equal(bits(seen[-1][0]), bits(ref.permute(3, 0, 1, 2).half()))
    with torch.no_grad():
        _run(m, voxel, idx)
    assert seen[-1].dtype == torch.float32
    # one GradScaler step (train.py:156-159): the hot parameters' gradients agree with the default (fp32-grid) model's
    grads = []
    for gd in ('autocast', torch.float32, torch.float32):
        mm = accelerate(copy.deepcopy(base), grid=SMALL, grid_dtype=gd)
        _scaler_step(mm, voxel, idx)
        grads.append(torch.cat([p.grad.flatten() for p in hot_parameters(mm)]))
    noise = float((grads[2] - grads[1]).abs().max())
    assert float((grads[0] - grads[1]).abs().max()) <= 2 * noise
    assert torch.isfinite(grads[0]).all() and float(grads[0].abs().max()) > 0
    # an overflowing fp16 gradient: the scaler skips the step and the parameters stay as they were
    mm = accelerate(copy.deepcopy(base), grid=SMALL, grid_dtype='autocast')
    before = [p.detach().clone() for p in mm.parameters()]
    scaler = _scaler_step(mm, voxel, idx, init_scale=2.0 ** 100)
    assert scaler.get_scale() < 2.0 ** 100
    assert all(torch.equal(a, p.detach()) for a, p in zip(before, mm.parameters()))


def test_accelerate_rejects_other_grid_dtypes():
    from mvxnet_makise_b200.dropin import accelerate
    from test_gpu_map_backward import SMALL, _standin
    base, _ = _standin(8)
    for bad in (torch.float64, 'fp8'):
        with pytest.raises(ValueError):
            accelerate(copy.deepcopy(base), grid=SMALL, grid_dtype=bad)
