"""Training through the sparse CML.conv1 hand-off (csrc/sparse_conv.cu, mvx_cml_conv1_sparse_backward): the CUDA backward
against the compact fp64 formulas on the CUDA forward's own saved activations (same ReLU decisions, tests/_cml_compact.py),
against dense fp64 autograd of the reference ops, the two routes into the hot-path backward, and the opt-in route of
`dropin.accelerate(..., sparse_cml_conv1=True)` on a stand-in module tree with the reference's attribute names."""
import copy

import numpy as np
import pytest
import torch

import _cml_compact as C
from mvxnet_makise_b200 import synth
from oracle import pointpath_oracle as O

pytestmark = pytest.mark.gpu
TOL = 1e-4
SMALL = synth.GridSpec((0.0, -4.8, -3.0, 8.0, 4.8, 1.0), (40, 48, 10), 35)
SMALL_FPN = ((13, 42), (7, 21), (4, 11))
F64 = torch.float64


@pytest.fixture(autouse=True)
def _restore_tf32_flags():
    """the dense routes compared here run with TF32 off; later tests get the flags back, and the multi-GB buffers of the
    full-size test go back to the device"""
    flags = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = flags
    torch.cuda.empty_cache()


def rel_err(a, ref):
    a, ref = torch.as_tensor(a).double().cpu(), torch.as_tensor(ref).double().cpu()
    return float((a - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


def small_maps(seed, B):
    rng = np.random.default_rng(seed)
    return [torch.from_numpy(rng.standard_normal((B, 256, h, w), dtype=np.float32)).cuda() for (h, w) in SMALL_FPN]


def conv1_params(seed=3):
    rng = np.random.default_rng(seed)
    w = torch.from_numpy((rng.standard_normal((64, 128, 3, 3, 3)) / np.sqrt(128 * 27)).astype(np.float32)).cuda()
    b = torch.from_numpy((rng.standard_normal(64) * 0.1).astype(np.float32)).cuda()
    return w, b


def train_forward(path, frames, maps, want_grid=True, cap=None):
    from mvxnet_makise_b200.modules import pack_calib
    offsets = np.concatenate([[0], np.cumsum([p.shape[0] for p in frames])]).tolist()
    points = torch.from_numpy(np.concatenate(frames, 0)).cuda()
    calib32 = torch.stack([pack_calib(synth.kitti_calib()) for _ in frames]).cuda()
    return path.forward_train(points, offsets, calib32, maps, want_grid=want_grid, cap=cap, shuffle=False)


def grid_shape(path):
    return (path.grid.shape[2], path.grid.shape[0], path.grid.shape[1])


def compact_on_saved(path, f, w, b, g):
    """the fp64 formulas on what the CUDA forward saved for frame f: (d_vfeat (N,128), d_w, d_b)"""
    vfeat, idx = path.voxel_features(f)
    saved = path.cml_saved()
    shape = grid_shape(path)
    oz = C.out_depth(shape[0])
    ai = saved['act_idx'][f].long()
    act = ai >= 0
    y = torch.zeros((64, act.numel()), dtype=F64, device=ai.device)
    y[:, act] = saved['Yact'][f][ai[act]].double().t()
    assert int(act.sum()) == int(saved['act_count'][f])
    return C.cml_conv1_backward(vfeat.double().cpu(), idx[:, 1:].cpu(), shape, w.cpu(), b.cpu(), g.cpu(),
                                y.cpu().reshape(64, oz, shape[1], shape[2]), act.cpu().reshape(oz, shape[1], shape[2]), path.eps)


def test_backward_matches_formulas_and_dense_autograd():
    from mvxnet_makise_b200.pipeline import PointPath
    sd = synth.make_weights(6)
    frames = [synth.make_points(120 + f, P, grid=SMALL) for f, P in enumerate((700, 350))]
    maps = small_maps(14, 2)
    w, b = conv1_params()
    path = PointPath(sd, SMALL)
    grid, counts = train_forward(path, frames, maps)
    out = path.cml_conv1(w, b)
    g = torch.randn(out.shape, generator=torch.Generator(device='cuda').manual_seed(7), device='cuda')
    d_vfeat, d_w, d_b = path.cml_conv1_backward(g, w, b)
    torch.cuda.synchronize()
    assert d_vfeat.shape == (2, path.cap, 128) and d_w.shape == (64, 128, 3, 3, 3) and d_b.shape == (64,)
    # (1) the kernels against the compact formulas on the SAME saved activations
    ref_w, ref_b = 0, 0
    for f in range(2):
        n = int(counts[f, 0])
        rv, rw, rb = compact_on_saved(path, f, w, b, g[f])
        assert rel_err(d_vfeat[f, :n], rv) < TOL, f
        assert float(d_vfeat[f, n:].abs().max()) == 0.0
        ref_w, ref_b = ref_w + rw, ref_b + rb
    assert rel_err(d_w, ref_w) < TOL and rel_err(d_b, ref_b) < TOL, (rel_err(d_w, ref_w), rel_err(d_b, ref_b))
    # (2) against dense autograd of the reference ops on the CUDA grid: fp64, bounded by the fp32 route's own distance to it
    res = {}
    for dt in (F64, torch.float32):
        gw, gb, gv = 0, 0, []
        for f in range(2):
            gr = grid[f:f + 1].detach().cpu().to(dt).requires_grad_(True)
            wd, bd = w.cpu().to(dt).requires_grad_(True), b.cpu().to(dt).requires_grad_(True)
            (O.cml_conv1(gr, wd, bd) * g[f:f + 1].cpu().to(dt)).sum().backward()
            _, idx = path.voxel_features(f)
            idx = idx.cpu()
            gv.append(gr.grad[0][:, idx[:, 3], idx[:, 1], idx[:, 2]].t())
            gw, gb = gw + wd.grad, gb + bd.grad
        res[dt] = (gv, gw, gb)
    ours = max([rel_err(d_vfeat[f, :int(counts[f, 0])], res[F64][0][f]) for f in range(2)] +
               [rel_err(d_w, res[F64][1]), rel_err(d_b, res[F64][2])])
    noise = max([rel_err(res[torch.float32][0][f], res[F64][0][f]) for f in range(2)] +
                [rel_err(res[torch.float32][1], res[F64][1]), rel_err(res[torch.float32][2], res[F64][2])])
    print(f'sparse conv1 backward vs dense fp64 autograd {ours:.3e}; fp32 dense route {noise:.3e}')
    assert ours <= 2 * noise + TOL
    # accumulate doubles; want_d_vfeat=False gives the same parameter gradients
    acc = (d_w.clone(), d_b.clone())
    path.cml_conv1_backward(g, w, b, grads=acc)
    assert rel_err(acc[0], 2 * d_w) < 1e-6 and rel_err(acc[1], 2 * d_b) < 1e-6
    none, d_w2, d_b2 = path.cml_conv1_backward(g, w, b, want_d_vfeat=False)
    assert none is None and rel_err(d_w2, d_w) < 1e-6 and rel_err(d_b2, d_b) < 1e-6
    # the gradient of the batch is the sum of the per-frame gradients
    tw, tb = 0, 0
    for f in range(2):
        single = PointPath(sd, SMALL)
        train_forward(single, frames[f:f + 1], [m[f:f + 1].contiguous() for m in maps], want_grid=False, cap=path.cap)
        single.cml_conv1(w, b)
        v1, w1, b1 = single.cml_conv1_backward(g[f:f + 1].contiguous(), w, b)
        n = int(counts[f, 0])
        assert rel_err(v1[0, :n], d_vfeat[f, :n]) < 1e-5
        tw, tb = tw + w1, tb + b1
    assert rel_err(d_w, tw) < 1e-5 and rel_err(d_b, tb) < 1e-5
    # a later forward invalidates the saved state
    train_forward(path, frames, maps)
    with pytest.raises(RuntimeError, match='cml_conv1'):
        path.cml_conv1_backward(g, w, b)


def _two_routes(path, w, b, g):
    """(a) fp64 autograd of the dense conv1 on the grid -> path.backward(d_grid); (b) sparse forward + backward ->
    path.backward(d_vfeat). Returns both (bucket, d_w, d_b)."""
    grid = path.grid_out
    gr = grid.detach().double().requires_grad_(True)
    wd, bd = w.double().requires_grad_(True), b.double().requires_grad_(True)
    for f in range(grid.shape[0]):
        (O.cml_conv1(gr[f:f + 1], wd, bd) * g[f:f + 1].double()).sum().backward()
    flat_a = path.backward(d_grid=gr.grad.float().contiguous()).clone()
    path.cml_conv1(w, b)
    d_vfeat, d_w, d_b = path.cml_conv1_backward(g, w, b)
    flat_b = path.backward(d_vfeat=d_vfeat).clone()
    return (flat_a, wd.grad, bd.grad), (flat_b, d_w, d_b)


def test_two_routes_into_the_hot_path_backward():
    from mvxnet_makise_b200.pipeline import PointPath
    sd = synth.make_weights(8)
    frames = [synth.make_points(130 + f, P, grid=SMALL) for f, P in enumerate((600, 900))]
    path = PointPath(sd, SMALL)
    train_forward(path, frames, small_maps(15, 2))
    w, b = conv1_params(4)
    g = torch.randn((2, 64, 5, 40, 48), generator=torch.Generator(device='cuda').manual_seed(2), device='cuda')
    a, s = _two_routes(path, w, b, g)
    torch.cuda.synchronize()
    assert a[0].numel() == 726_880
    errs = [rel_err(x, y) for x, y in zip(s, a)]
    print('two routes (bucket, d_w, d_b):', errs)
    assert max(errs) < TOL, errs


def _voxel_frame(coords, T, rng):
    """hand-made dense-voxel input: one to three points per voxel at its cell, projection inside the image"""
    n = len(coords)
    vox = torch.zeros((n, T, 9))
    vs, lo = SMALL.voxelsize, SMALL.velorange
    for v, (ix, iy, iz) in enumerate(coords):
        k = int(rng.integers(1, 4))
        c = np.array([lo[0] + (ix + 0.5) * vs[0], lo[1] + (iy + 0.5) * vs[1], lo[2] + (iz + 0.5) * vs[2]])
        pts = c + (rng.random((k, 3)) - 0.5) * np.array(vs) * 0.9
        vox[v, :k, :3] = torch.from_numpy(pts).float()
        vox[v, :k, 3:6] = torch.from_numpy(pts - pts.mean(0)).float()
        vox[v, :k, 6] = torch.from_numpy(rng.random(k)).float()
        vox[v, :k, 7] = torch.from_numpy(rng.random(k) * 360).float()
        vox[v, :k, 8] = torch.from_numpy(rng.random(k) * 1200).float()
    idx = torch.cat([torch.zeros((n, 1), dtype=torch.int64), torch.as_tensor(np.asarray(coords, np.int64).reshape(n, 3))], 1)
    return vox.cuda(), idx.cuda()


def test_two_routes_on_corner_edge_and_empty_frames():
    from mvxnet_makise_b200.pipeline import PointPath
    nx, ny, nz = SMALL.voxelshape
    rng = np.random.default_rng(11)
    corners = [(x, y, z) for x in (0, nx - 1) for y in (0, ny - 1) for z in (0, nz - 1)]
    edges = [(x, 5 + x % 7, 0) for x in range(0, nx, 3)] + [(0, y, nz - 1) for y in range(1, ny, 4)] + [(nx - 1, 7, z) for z in range(nz)]
    frames = [_voxel_frame(corners, SMALL.T, rng), _voxel_frame([], SMALL.T, rng), _voxel_frame(edges, SMALL.T, rng)]
    path = PointPath(synth.make_weights(2), SMALL)
    path.forward_voxels([v for v, _ in frames], [i for _, i in frames], small_maps(16, 3), want_grid=True, train=True)
    assert path.counts[:, 0].tolist() == [len(corners), 0, len(edges)]
    w, b = conv1_params(5)
    g = torch.randn((3, 64, 5, nx, ny), generator=torch.Generator(device='cuda').manual_seed(3), device='cuda')
    # what each route hands to the hot-path backward (dLoss/d voxel features) and the conv1 gradients
    gr = path.grid_out.detach().double().requires_grad_(True)
    wd, bd = w.double().requires_grad_(True), b.double().requires_grad_(True)
    for f in range(3):
        (O.cml_conv1(gr[f:f + 1], wd, bd) * g[f:f + 1].double()).sum().backward()
    path.cml_conv1(w, b)
    d_vfeat, d_w, d_b = path.cml_conv1_backward(g, w, b)
    errs = [rel_err(d_w, wd.grad), rel_err(d_b, bd.grad)]
    for f in (0, 2):
        _, idx = path.voxel_features(f)
        errs.append(rel_err(d_vfeat[f, :idx.shape[0]], gr.grad[f][:, idx[:, 3], idx[:, 1], idx[:, 2]].t()))
    print('hand-made frames, two routes (d_w, d_b, d_vfeat of the corner and edge frames):', errs)
    assert max(errs) < TOL, errs
    assert float(d_vfeat[1].abs().max()) == 0.0


# ---- drop-in: a stand-in module tree with the reference's attribute names -------------------------------------------
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
    """a fixed linear functional of the CML output: both routes receive the same upstream gradient"""

    def __init__(self, weight):
        super().__init__()
        self.register_buffer('w', weight)

    def forward(self, x):
        return (x * self.w).sum(), x.new_zeros(())


class _SmallRPN(torch.nn.Module):
    def __init__(self, cin):
        super().__init__()
        self.score, self.reg = torch.nn.Conv2d(cin, 2, 1), torch.nn.Conv2d(cin, 14, 1)

    def forward(self, x):
        return self.score(x), self.reg(x)


class _Maps(torch.nn.Module):
    def __init__(self, seed):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.maps = [torch.randn((1, 256, h, w), generator=g) for h, w in SMALL_FPN]

    def forward(self, x):
        return [m.to(x.device) for m in self.maps]


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
    root.head.add_module('extractor', _Maps(seed))
    root.backbone.add_module('cml', _CML())
    root.backbone.add_module('rpn', _SmallRPN(128))
    return root.cuda()


def _frame_inputs(seed, P, grid=SMALL):
    pts = synth.make_points(seed, P, grid=grid)
    calib = synth.kitti_calib()
    pcd6 = O.points_with_proj(pts, calib)
    voxel, idx = O.group(pcd6, grid.velorange, grid.voxelsize, grid.T)
    voxel = torch.as_tensor(np.asarray(voxel), dtype=torch.float32)[None].cuda()
    idx = torch.as_tensor(np.concatenate([np.zeros((idx.shape[0], 1)), idx], 1), dtype=torch.int64).cuda()
    return voxel, idx


def _run(model, voxel, idx):
    img = torch.zeros((1, 3, 8, 8), device='cuda')
    imsize = torch.tensor(synth.KITTI_IMSIZE_HW, dtype=torch.float32, device='cuda')
    return model(voxel.clone(), img, idx, None, imsize)


def _grads(model):
    from mvxnet_makise_b200.dropin import hot_parameters
    c = model.backbone.cml.conv1.conv
    return [None if p.grad is None else p.grad.detach().double().cpu().clone() for p in hot_parameters(model) + [c.weight, c.bias]]


def _probe_comparison(base, voxel, idx, nx, ny):
    from mvxnet_makise_b200.dropin import accelerate
    torch.backends.cudnn.allow_tf32 = False
    w = torch.randn((1, 64 * 5, nx, ny), generator=torch.Generator().manual_seed(1)).cuda() * 1e-3
    res = {}
    for sparse in (False, True):
        m = copy.deepcopy(base)
        m.backbone.cml.conv2, m.backbone.cml.conv3, m.backbone.rpn = torch.nn.Identity(), torch.nn.Identity(), _Probe(w)
        m = accelerate(m, grid=SMALL, sparse_cml_conv1=sparse)
        score, _ = _run(m, voxel, idx)
        score.backward()
        res[sparse] = (score.detach(), _grads(m))
    assert rel_err(res[True][0], res[False][0]) < TOL
    errs = [rel_err(a, b) for a, b in zip(res[True][1], res[False][1])]
    print('drop-in, sparse vs dense route, 18 gradients:', [f'{e:.1e}' for e in errs])
    assert len(errs) == 18 and max(errs) < TOL, errs


def test_dropin_sparse_route_matches_dense_route():
    voxel, idx = _frame_inputs(31, 900)
    _probe_comparison(_standin(1), voxel, idx, SMALL.voxelshape[0], SMALL.voxelshape[1])


def test_dropin_full_cml_train_step_and_cml_only_finetuning():
    from mvxnet_makise_b200.dropin import accelerate, hot_parameters
    torch.backends.cudnn.allow_tf32 = False
    voxel, idx = _frame_inputs(32, 1100)
    base = _standin(2)
    res = {}
    for sparse in (False, True):
        m = accelerate(copy.deepcopy(base), grid=SMALL, sparse_cml_conv1=sparse)
        score, reg = _run(m, voxel, idx)
        loss = (score ** 2).mean() + (reg ** 2).mean()
        assert torch.isfinite(loss)
        loss.backward()
        res[sparse] = (m, _grads(m))
    cos = [float((a * b).sum() / (a.norm() * b.norm()).clamp_min(1e-300)) for a, b in zip(res[True][1], res[False][1])]
    print('full CML, gradient cosines sparse vs dense:', [f'{c:.6f}' for c in cos])
    assert min(cos) > 0.999, cos
    fast = res[True][0]
    opt = torch.optim.AdamW(fast.parameters(), lr=1e-3)
    conv = fast.backbone.cml.conv1.conv
    before = [p.detach().clone() for p in hot_parameters(fast) + [conv.weight, conv.bias]]
    with torch.no_grad():
        s0 = _run(fast, voxel, idx)[0].clone()
    opt.step()
    assert all(not torch.equal(a, p) for a, p in zip(before, hot_parameters(fast) + [conv.weight, conv.bias]))
    with torch.no_grad():
        s1 = _run(fast, voxel, idx)[0]
    assert not torch.equal(s0, s1), 'the optimiser step did not reach the sparse route'
    # fine-tuning the CML alone: no hot-path gradient, the conv1 gradient still equals the dense route's
    for sparse in (False, True):
        m = accelerate(copy.deepcopy(base), grid=SMALL, sparse_cml_conv1=sparse)
        for p in hot_parameters(m):
            p.requires_grad_(False)
        score, reg = _run(m, voxel, idx)
        ((score ** 2).mean() + (reg ** 2).mean()).backward()
        res[sparse] = _grads(m)
    assert all(g is None for g in res[True][:16])
    cos = [float((a * b).sum() / (a.norm() * b.norm())) for a, b in zip(res[True][16:], res[False][16:])]
    assert min(cos) > 0.999, cos


@pytest.mark.parametrize('sparse,freeze_hot', [(False, False), (True, False), (True, True)])
def test_dropin_backward_after_another_forward_raises(sparse, freeze_hot):
    """HotPathFunction / SparseConv1Function (also with the hot path frozen: CML-only fine-tuning): another forward of the
    model, training or inference, before the backward of the first overwrites what that backward reads, so it raises."""
    from mvxnet_makise_b200.dropin import accelerate, hot_parameters
    voxel, idx = _frame_inputs(34, 700)
    m = accelerate(_standin(4), grid=SMALL, sparse_cml_conv1=sparse)
    for p in hot_parameters(m):
        p.requires_grad_(not freeze_hot)
    for second in ('training', 'inference'):
        score, _ = _run(m, voxel, idx)
        with torch.set_grad_enabled(second == 'training'):
            _run(m, voxel, idx)
        with pytest.raises(RuntimeError, match='another forward'):
            score.sum().backward()
    score, _ = _run(m, voxel, idx)
    score.sum().backward()                  # the latest forward's backward runs


def test_dropin_rejects_non_stock_conv1():
    from mvxnet_makise_b200.dropin import accelerate
    m = _standin(3)
    m.backbone.cml.conv1.conv = torch.nn.Conv3d(128, 64, 3, 1, 1).cuda()
    with pytest.raises(ValueError, match='stock'):
        accelerate(m, grid=SMALL, sparse_cml_conv1=True)
    m = _standin(3)
    m.backbone.cml.conv1.bn = torch.nn.BatchNorm3d(64, affine=True, track_running_stats=False).cuda()
    with pytest.raises(ValueError, match='stock'):
        accelerate(m, grid=SMALL, sparse_cml_conv1=True)
    m = _standin(3)
    m.backbone.cml.conv1.bn.eps = 1e-3
    assert accelerate(m, grid=SMALL, sparse_cml_conv1=True)._mvx_conv1_eps == 1e-3


def test_full_size_batch_forward_backward():
    """8 x 120 000-point KITTI frames through the sparse conv1 forward + backward and the hot-path backward; frame 0 against
    the formulas on its saved activations"""
    from mvxnet_makise_b200.pipeline import PointPath
    from mvxnet_makise_b200.modules import pack_calib
    G = synth.KITTI_GRID
    B = 8
    frames = [synth.make_points(f, 120_000) for f in range(B)]
    gen = torch.Generator(device='cuda').manual_seed(1)
    maps = [torch.randn((B, 256, h, w), generator=gen, device='cuda') for (h, w) in synth.fpn_shapes()]
    w, b = conv1_params(6)
    path = PointPath(synth.make_weights(0), G)
    offsets = np.concatenate([[0], np.cumsum([p.shape[0] for p in frames])]).tolist()
    points = torch.from_numpy(np.concatenate(frames, 0)).cuda()
    calib32 = torch.stack([pack_calib(synth.kitti_calib()) for _ in frames]).cuda()
    _, counts = path.forward_train(points, offsets, calib32, maps, want_grid=False, shuffle=False)
    out = path.cml_conv1(w, b)
    g = torch.randn(out.shape, generator=gen, device='cuda')
    d_vfeat, d_w, d_b = path.cml_conv1_backward(g, w, b)
    flat = path.backward(d_vfeat=d_vfeat)
    torch.cuda.synchronize()
    assert all(torch.isfinite(t).all() for t in (out, d_vfeat, d_w, d_b, flat)) and float(flat.abs().max()) > 0
    n = int(counts[0, 0])
    rv, _, _ = compact_on_saved(path, 0, w, b, g[0])
    assert rel_err(d_vfeat[0, :n], rv) < TOL
    single = PointPath(synth.make_weights(0), G)
    _, c1 = single.forward_train(points[:offsets[1]], offsets[:2], calib32[:1], [m[:1].contiguous() for m in maps], want_grid=False,
                                 cap=path.cap, shuffle=False)
    single.cml_conv1(w, b)
    v1, w1, b1 = single.cml_conv1_backward(g[:1].contiguous(), w, b)
    rv1, rw1, rb1 = compact_on_saved(single, 0, w, b, g[0])
    assert rel_err(v1[0, :n], rv1) < TOL and rel_err(w1, rw1) < TOL and rel_err(b1, rb1) < TOL


def test_dropin_on_the_reference_mvxnet():
    from oracle import refshim
    if not refshim.available():
        pytest.skip('no staged reference tree')
    ref = refshim.load(device='cuda')
    torch.manual_seed(4)
    model = ref.MVXNet()
    model.head.extractor = _Maps(4)
    voxel, idx = _frame_inputs(33, 2500, grid=synth.KITTI_GRID)
    from mvxnet_makise_b200.dropin import accelerate
    base = model.cuda()
    res = {}
    torch.backends.cudnn.allow_tf32 = False
    w = torch.randn((1, 64 * 5, 352, 400), generator=torch.Generator().manual_seed(1)).cuda() * 1e-3
    for sparse in (False, True):
        m = accelerate(copy.deepcopy(base), sparse_cml_conv1=sparse)
        m.backbone.cml.conv2, m.backbone.cml.conv3, m.backbone.rpn = torch.nn.Identity(), torch.nn.Identity(), _Probe(w)
        score, _ = _run(m, voxel, idx)
        score.backward()
        res[sparse] = (score.detach(), _grads(m))
    assert rel_err(res[True][0], res[False][0]) < TOL
    assert max(rel_err(a, b) for a, b in zip(res[True][1], res[False][1])) < TOL
