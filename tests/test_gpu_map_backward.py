"""The gradient into the FPN maps (csrc/map_backward.cu, mvx_pointpath_backward_maps): CUDA against the fp64 adjoint of
the 4-corner gather evaluated on the CUDA run's own saved dpre1 and projections (tests/_map_adjoint.py `map_adjoint`;
same decisions, so 1e-4 of max|ref| per level), end to end against dense fp64 autograd with the maps as leaves, determinism,
no side effect on the parameter gradients or the launches of a frozen-backbone step, and the drop-in with a trainable
`head.extractor` on both routes of `dropin.accelerate`."""
import copy

import numpy as np
import pytest
import torch

import _map_adjoint as MA
from mvxnet_makise_b200 import synth
from oracle import pointpath_oracle as O

pytestmark = pytest.mark.gpu
G = synth.KITTI_GRID
TOL = 1e-4
SMALL = synth.GridSpec((0.0, -4.8, -3.0, 8.0, 4.8, 1.0), (40, 48, 10), 35)
SMALL_FPN = ((13, 42), (7, 21), (4, 11))
W1 = 'head.fusion.fcn1.fc.weight'


@pytest.fixture(autouse=True)
def _restore_tf32_flags():
    flags = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = flags
    torch.cuda.empty_cache()


def rel_err(a, ref):
    a, ref = torch.as_tensor(a).double().cpu(), torch.as_tensor(ref).double().cpu()
    return float((a - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def cosine(a, b):
    a, b = torch.as_tensor(a).double().cpu().flatten(), torch.as_tensor(b).double().cpu().flatten()
    return float((a * b).sum() / (a.norm() * b.norm()).clamp_min(1e-300))


def small_maps(seed, B):
    rng = np.random.default_rng(seed)
    return [torch.from_numpy(rng.standard_normal((B, 256, h, w), dtype=np.float32)).cuda() for (h, w) in SMALL_FPN]


def map_buffers(maps):
    return [torch.full(m.shape, float('nan'), dtype=torch.float32, device='cuda') for m in maps]   # NaN: every element must be written


def adjoint_on_saved(path, sd, f):
    """the fp64 adjoint on what the CUDA forward / backward saved for frame f: [(256, H_l, W_l)]"""
    K = int(path.counts[f, 1])
    capA = path.cap + 128
    dpre1 = path.backward_saved()['dpre1'][f, :K].double().cpu()
    proj = path.region('proj', torch.float32, (path.B, capA, 2))[f, :K].cpu()
    xyz = path.region('vox8', torch.float32, (path.B, capA, 8))[f, :K, :3].cpu()
    real = (xyz != 0).any(1)
    hw = [tuple(m.shape[-2:]) for m in path._record.maps]
    return MA.map_adjoint(dpre1, torch.from_numpy(np.asarray(sd[W1])), proj, real, hw, path.imsize_hw, path.eps)


def map_entry(path, d_maps):
    """mvx_pointpath_backward_maps alone, on the state the last PointPath.backward(d_maps=...) left"""
    import ctypes
    from mvxnet_makise_b200 import _lib
    a = path._record.args
    out = (ctypes.c_void_p * 3)(*[t.data_ptr() for t in d_maps])
    _lib.check(_lib.lib.mvx_pointpath_backward_maps(ctypes.byref(a), path._bws.data_ptr(), path._bws.numel(), out,
                                                    path._map_bws.data_ptr(), path._map_bws.numel()), 'backward_maps')


def check_against_saved(path, sd, d_maps):
    for f in range(path.B):
        ref = adjoint_on_saved(path, sd, f)
        for l in range(3):
            got = d_maps[l][f]
            assert torch.isfinite(got).all()
            if float(ref[l].abs().max()) == 0:       # a frame without points
                assert float(got.abs().max()) == 0
            else:
                assert rel_err(got, ref[l]) < TOL, (f, l, rel_err(got, ref[l]))


def points_train(path, frames, maps, calibs=None, point_calib=None):
    from mvxnet_makise_b200.modules import pack_calib
    offsets = np.concatenate([[0], np.cumsum([p.shape[0] for p in frames])]).tolist()
    points = torch.from_numpy(np.concatenate(frames, 0)).cuda()
    calib32 = torch.stack([pack_calib(c) for c in (calibs or [synth.kitti_calib()] * len(frames))]).cuda()
    return path.forward_device(points, offsets, calib32, maps, train=True, shuffle=False, point_calib=point_calib)


def test_points_entry_with_an_empty_frame():
    from mvxnet_makise_b200.pipeline import PointPath
    sd = synth.make_weights(5)
    path = PointPath(sd, G)
    frames = [synth.make_points(40, 2200), np.zeros((0, 4), np.float32), synth.make_points(41, 1500)]
    maps = small_maps(6, 3)
    points_train(path, frames, maps)
    dv = torch.randn((3, path.cap, 128), device='cuda', generator=torch.Generator(device='cuda').manual_seed(2))
    d_maps = map_buffers(maps)
    path.backward(d_vfeat=dv, d_maps=d_maps)
    torch.cuda.synchronize()
    check_against_saved(path, sd, d_maps)
    assert all(float(d[1].abs().max()) == 0 for d in d_maps) and all(float(d[0].abs().max()) > 0 for d in d_maps)


def test_dense_voxel_entry():
    from mvxnet_makise_b200.pipeline import PointPath
    sd = synth.make_weights(8)
    path = PointPath(sd, G)
    vs, ids = [], []
    for f, seed in enumerate((50, 51)):
        voxel, idx = O.group(O.points_with_proj(synth.make_points(seed, 1800), synth.kitti_calib()), G.velorange, G.voxelsize, G.T)
        vs.append(torch.as_tensor(np.asarray(voxel), dtype=torch.float32).cuda())
        ids.append(torch.as_tensor(np.concatenate([np.full((idx.shape[0], 1), f), idx], 1), dtype=torch.int64).cuda())
    maps = small_maps(9, 2)
    path.forward_voxels(vs, ids, maps, want_grid=False, train=True)
    dv = torch.randn((2, path.cap, 128), device='cuda', generator=torch.Generator(device='cuda').manual_seed(3))
    d_maps = map_buffers(maps)
    path.backward(d_vfeat=dv, d_maps=d_maps)
    torch.cuda.synchronize()
    check_against_saved(path, sd, d_maps)


def test_merged_point_sets():
    """GT-paste (train.py:29-42): the pasted objects project through their own calibration"""
    from mvxnet_makise_b200.pipeline import PointPath
    sd = synth.make_weights(10)
    path = PointPath(sd, G)
    base = synth.kitti_calib()
    other = {k: np.array(v, dtype=np.float32, copy=True) for k, v in base.items()}
    other['P2'][0, 0] += np.float32(11.5)
    other['P2'][0, 2] -= np.float32(3.25)
    scene, pasted = synth.make_points(60, 2000), synth.make_points(61, 600)
    pc = torch.from_numpy(np.concatenate([np.zeros(len(scene), np.int32), np.ones(len(pasted), np.int32)])).cuda()
    maps = small_maps(11, 1)
    points_train(path, [np.concatenate([scene, pasted])], maps, calibs=[base, other], point_calib=pc)
    dv = torch.randn((1, path.cap, 128), device='cuda', generator=torch.Generator(device='cuda').manual_seed(4))
    d_maps = map_buffers(maps)
    path.backward(d_vfeat=dv, d_maps=d_maps)
    torch.cuda.synchronize()
    check_against_saved(path, sd, d_maps)


def test_end_to_end_against_dense_autograd_determinism_and_parameter_gradients():
    from mvxnet_makise_b200.pipeline import PointPath
    seed, P = 12, 2500
    sd = synth.make_weights(seed)
    pts = synth.make_points(seed, P)
    maps = small_maps(seed, 1)
    path = PointPath(sd, G)
    _, counts = points_train(path, [pts], maps)
    N = int(counts[0, 0])
    d_vfeat = np.random.default_rng(seed + 100).standard_normal((N, 128)).astype(np.float32)
    dv = torch.zeros((1, path.cap, 128), dtype=torch.float32, device='cuda')
    dv[0, :N] = torch.from_numpy(d_vfeat).cuda()
    flat0 = path.backward(d_vfeat=dv).clone()
    d1, d2 = map_buffers(maps), map_buffers(maps)
    flat1 = path.backward(d_vfeat=dv, d_maps=d1)
    # the parameter backward sums with fp32 atomics (its reruns agree to rounding); the map backward runs after it and only
    # reads: on ONE saved state, a second and a third call of the map entry leave the parameter gradients bit-identical and
    # reproduce d_maps bit for bit
    kept = flat1.clone()
    map_entry(path, d2)
    map_entry(path, d1)
    torch.cuda.synchronize()
    assert rel_err(flat1, flat0) < 1e-6
    assert torch.equal(flat1, kept), 'the map backward changed the parameter gradients'
    assert all(torch.equal(a, b) for a, b in zip(d1, d2)), 'two map backward calls differ'
    check_against_saved(path, sd, d1)
    np_maps = [m.cpu().numpy() for m in maps]
    calib = synth.kitti_calib()
    ref64 = MA.dense_backward_frame(pts, calib, np_maps, sd, G, synth.KITTI_IMSIZE_HW, d_vfeat)
    ref32 = MA.dense_backward_frame(pts, calib, np_maps, sd, G, synth.KITTI_IMSIZE_HW, d_vfeat, dtype=torch.float32)
    ours = max(rel_err(d1[l][0], ref64[l]) for l in range(3))
    noise = max(rel_err(ref32[l], ref64[l]) for l in range(3))
    cos = [cosine(d1[l][0], ref64[l]) for l in range(3)]
    print(f'map gradients vs fp64 autograd: ours {ours:.3e}, fp32 reference {noise:.3e}, cosines {cos}')
    assert ours <= 2 * noise + TOL and min(cos) > 0.999


# ---- drop-in: a stand-in module tree with the reference's attribute names and a TRAINABLE head.extractor ---------------
class _CRB3d(torch.nn.Module):
    def __init__(self, cin, cout, stride, pad):
        super().__init__()
        self.conv = torch.nn.Conv3d(cin, cout, 3, stride, pad)
        self.bn = torch.nn.BatchNorm3d(cout, affine=False, track_running_stats=False)

    def forward(self, x):
        return self.bn(torch.relu(self.conv(x)))


class _CML(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.conv1 = _CRB3d(128, 64, (2, 1, 1), (1, 1, 1))
        self.conv2 = _CRB3d(64, 64, 1, (0, 1, 1))
        self.conv3 = _CRB3d(64, 64, (2, 1, 1), 1)

    def forward(self, x):
        return self.conv3(self.conv2(self.conv1(x)))


class _Probe(torch.nn.Module):
    """a fixed linear functional of its input: every route receives the same upstream gradient"""

    def __init__(self, weight):
        super().__init__()
        self.register_buffer('w', weight)

    def forward(self, x):
        return (x * self.w).sum(), x.new_zeros(())


class _TrainableMaps(torch.nn.Module):
    """stands in for the image backbone: its FPN maps are its parameters, so their .grad is what the backbone receives"""

    def __init__(self, seed):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.maps = torch.nn.ParameterList([torch.nn.Parameter(torch.randn((1, 256, h, w), generator=g)) for h, w in SMALL_FPN])

    def forward(self, x):
        return list(self.maps)


def _standin(seed):
    """MVXNet's attribute tree (head.fusion.*, backbone.svfe.*, backbone.fcn, backbone.cml, backbone.rpn, head.extractor)"""
    torch.manual_seed(seed)
    sd = synth.make_weights(seed)
    root = torch.nn.Module()
    for name, cin, cout, is_conv in synth.HOT_LAYERS:
        parent = root
        parts = name.split('.')
        for p in parts[:-1]:
            if not hasattr(parent, p):
                parent.add_module(p, torch.nn.Module())
            parent = getattr(parent, p)
        layer = torch.nn.Conv2d(cin, cout, 1) if is_conv else torch.nn.Linear(cin, cout)
        with torch.no_grad():
            layer.weight.copy_(torch.as_tensor(np.asarray(sd[name + '.weight'])).reshape(layer.weight.shape))
            layer.bias.copy_(torch.as_tensor(np.asarray(sd[name + '.bias'])))
        parent.add_module(parts[-1], layer)
    root.head.add_module('extractor', _TrainableMaps(seed))
    root.backbone.add_module('cml', _CML())
    root.backbone.add_module('rpn', torch.nn.Conv2d(128, 2, 1))
    return root.cuda(), sd


def _frame_inputs(seed, P, grid=SMALL):
    pts = synth.make_points(seed, P, grid=grid)
    voxel, idx = O.group(O.points_with_proj(pts, synth.kitti_calib()), grid.velorange, grid.voxelsize, grid.T)
    voxel = torch.as_tensor(np.asarray(voxel), dtype=torch.float32)[None].cuda()
    idx = torch.as_tensor(np.concatenate([np.zeros((idx.shape[0], 1)), idx], 1), dtype=torch.int64).cuda()
    return voxel, idx


def _run(model, voxel, idx):
    img = torch.zeros((1, 3, 8, 8), device='cuda')
    imsize = torch.tensor(synth.KITTI_IMSIZE_HW, dtype=torch.float32, device='cuda')
    return model(voxel.clone(), img, idx, None, imsize)


def _probed(base, sparse, w_grid, w_conv1):
    """probe on the grid (dense route: the CML is skipped) or on conv1's output (sparse route: conv2 / conv3 skipped)"""
    from mvxnet_makise_b200.dropin import accelerate
    m = copy.deepcopy(base)
    if sparse:
        m.backbone.cml.conv2, m.backbone.cml.conv3, m.backbone.rpn = torch.nn.Identity(), torch.nn.Identity(), _Probe(w_conv1)
    else:
        m.backbone.cml, m.backbone.rpn = torch.nn.Identity(), _Probe(w_grid)
    return accelerate(m, grid=SMALL, sparse_cml_conv1=sparse)


def _extractor_grads(m):
    return [None if p.grad is None else p.grad.detach()[0].double().cpu().clone() for p in m.head.extractor.maps]


def test_dropin_trains_the_extractor_on_both_routes():
    from mvxnet_makise_b200.dropin import hot_parameters
    torch.backends.cudnn.allow_tf32 = False
    voxel, idx = _frame_inputs(35, 1400)
    base, sd = _standin(4)
    nz, (nx, ny) = SMALL.voxelshape[2], SMALL.voxelshape[:2]
    gen = torch.Generator().manual_seed(1)
    w_grid = (torch.randn((1, 128 * nz, nx, ny), generator=gen) * 1e-3).cuda()
    w_conv1 = (torch.randn((1, 64 * 5, nx, ny), generator=gen) * 1e-3).cuda()
    # the oracle under the grid probe: d vfeat[v] = d grid[:, iz, ix, iy] of the voxel's cell, maps as leaves of the dense chain
    dg = w_grid.reshape(128, nz, nx, ny).cpu()
    d_vfeat = dg[:, idx[:, 3].cpu(), idx[:, 1].cpu(), idx[:, 2].cpu()].t().numpy()
    maps_np = [p.detach().cpu().numpy() for p in base.head.extractor.maps]
    ref64 = MA.dense_backward(voxel[0].cpu().clone(), maps_np, sd, synth.KITTI_IMSIZE_HW, d_vfeat)
    ref32 = MA.dense_backward(voxel[0].cpu().clone(), maps_np, sd, synth.KITTI_IMSIZE_HW, d_vfeat, dtype=torch.float32)
    res = {}
    for sparse in (False, True):
        m = _probed(base, sparse, w_grid, w_conv1)
        score, _ = _run(m, voxel, idx)
        score.backward()
        res[sparse] = _extractor_grads(m)
        assert all(g is not None and torch.isfinite(g).all() and float(g.abs().max()) > 0 for g in res[sparse])
        assert all(p.grad is not None for p in hot_parameters(m))
    ours = max(rel_err(g, r) for g, r in zip(res[False], ref64))
    noise = max(rel_err(r32, r) for r32, r in zip(ref32, ref64))
    print(f'extractor gradient (grid probe) vs fp64 autograd: {ours:.3e}, fp32 reference {noise:.3e}')
    assert ours <= 2 * noise + TOL and min(cosine(g, r) for g, r in zip(res[False], ref64)) > 0.999
    # the sparse route: the same probe on conv1's output through the dense route (conv1 the stock module on the grid)
    from mvxnet_makise_b200.dropin import accelerate
    m = copy.deepcopy(base)
    m.backbone.cml.conv2, m.backbone.cml.conv3, m.backbone.rpn = torch.nn.Identity(), torch.nn.Identity(), _Probe(w_conv1)
    m = accelerate(m, grid=SMALL, sparse_cml_conv1=False)
    _run(m, voxel, idx)[0].backward()
    dense_conv1 = _extractor_grads(m)
    errs = [rel_err(a, b) for a, b in zip(res[True], dense_conv1)]
    print('extractor gradient, sparse vs dense route:', [f'{e:.1e}' for e in errs])
    assert max(errs) < 1e-3 and min(cosine(a, b) for a, b in zip(res[True], dense_conv1)) > 0.999


def test_dropin_adamw_step_and_maps_only_training():
    from mvxnet_makise_b200.dropin import accelerate, hot_parameters
    torch.backends.cudnn.allow_tf32 = False
    voxel, idx = _frame_inputs(36, 1200)
    base, _ = _standin(5)
    for sparse in (False, True):
        fast = accelerate(copy.deepcopy(base), grid=SMALL, sparse_cml_conv1=sparse)
        score = _run(fast, voxel, idx)
        loss = (score ** 2).mean()
        loss.backward()
        opt = torch.optim.AdamW(fast.parameters(), lr=1e-3)
        before = [p.detach().clone() for p in fast.head.extractor.maps]
        opt.step()
        assert all(not torch.equal(a, p) for a, p in zip(before, fast.head.extractor.maps)), 'AdamW did not move the extractor'
        # maps-only training: the hot path still runs its backward (dpre1), the 16 hot parameters get no .grad
        m = accelerate(copy.deepcopy(base), grid=SMALL, sparse_cml_conv1=sparse)
        for p in hot_parameters(m):
            p.requires_grad_(False)
        (_run(m, voxel, idx) ** 2).mean().backward()
        assert all(p.grad is None for p in hot_parameters(m))
        assert all(g is not None and float(g.abs().max()) > 0 for g in _extractor_grads(m))


def test_frozen_maps_step_never_reaches_the_map_backward():
    """a drop-in step with a frozen extractor launches exactly the kernels of the same step driven through
    PointPath.backward(d_maps=None)"""
    from mvxnet_makise_b200 import _lib
    from mvxnet_makise_b200.dropin import accelerate
    voxel, idx = _frame_inputs(37, 1300)
    base, _ = _standin(6)
    base.head.extractor.requires_grad_(False)
    m = accelerate(base, grid=SMALL)
    m.backbone.cml = torch.nn.Identity()
    w = torch.randn((1, 128 * SMALL.voxelshape[2], *SMALL.voxelshape[:2]), generator=torch.Generator().manual_seed(2)).cuda() * 1e-3
    m.backbone.rpn = _Probe(w)
    _run(m, voxel, idx)[0].backward()                     # warm-up: workspaces allocated, parameters pushed
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    _run(m, voxel, idx)[0].backward()
    torch.cuda.synchronize()
    n_dropin = _lib.launch_count() - n0
    path = m._mvx_path
    maps = [p.detach() for p in m.head.extractor.maps]
    n0 = _lib.launch_count()
    grid, _ = path.forward_voxels(voxel.clone(), idx, maps, want_grid=True, train=True)
    path.backward(d_grid=w.reshape(grid.shape).contiguous(), d_maps=None)
    torch.cuda.synchronize()
    assert n_dropin == _lib.launch_count() - n0 > 0


def test_dropin_on_the_reference_mvxnet():
    from oracle import refshim
    if not refshim.available():
        pytest.skip('no staged reference tree')
    from mvxnet_makise_b200.dropin import accelerate
    ref = refshim.load(device='cuda')
    torch.manual_seed(4)
    model = ref.MVXNet()
    model.head.extractor = _TrainableMaps(4)
    voxel, idx = _frame_inputs(33, 2500, grid=synth.KITTI_GRID)
    base = model.cuda()
    res = {}
    torch.backends.cudnn.allow_tf32 = False
    w = torch.randn((1, 64 * 5, 352, 400), generator=torch.Generator().manual_seed(1)).cuda() * 1e-3
    for sparse in (False, True):
        m = accelerate(copy.deepcopy(base), sparse_cml_conv1=sparse)
        m.backbone.cml.conv2, m.backbone.cml.conv3, m.backbone.rpn = torch.nn.Identity(), torch.nn.Identity(), _Probe(w)
        _run(m, voxel, idx)[0].backward()
        res[sparse] = _extractor_grads(m)
    assert all(float(g.abs().max()) > 0 for g in res[False])
    assert max(rel_err(a, b) for a, b in zip(res[True], res[False])) < 1e-3


def test_full_size_batch():
    """8 x 120 000-point KITTI frames: forward, backward and the map backward finite; frame 0 against the fp64 adjoint on its
    saved activations"""
    from mvxnet_makise_b200.pipeline import PointPath
    B = 8
    frames = [synth.make_points(f, 120_000) for f in range(B)]
    gen = torch.Generator(device='cuda').manual_seed(1)
    maps = [torch.randn((B, 256, h, w), generator=gen, device='cuda') for (h, w) in synth.fpn_shapes()]
    sd = synth.make_weights(0)
    path = PointPath(sd, G)
    points_train(path, frames, maps)
    dv = torch.randn((B, path.cap, 128), generator=gen, device='cuda')
    d_maps = map_buffers(maps)
    flat = path.backward(d_vfeat=dv, d_maps=d_maps)
    torch.cuda.synchronize()
    assert torch.isfinite(flat).all() and all(torch.isfinite(d).all() for d in d_maps)
    ref = adjoint_on_saved(path, sd, 0)
    for l in range(3):
        assert rel_err(d_maps[l][0], ref[l]) < TOL, (l, rel_err(d_maps[l][0], ref[l]))
