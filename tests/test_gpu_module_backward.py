"""Training through the per-module drop-ins (mvxnet_makise_b200/modules.py) on the GPU: the CUDA layer backward against the fp64
formulas of tests/_module_adjoint.py on the CUDA forward's own raw outputs and BatchNorm sums, the module chains against fp64
autograd of the oracle, the featureMaping and reindex adjoints, unchanged no-grad behaviour, a training step and a full-size frame."""
import ctypes

import numpy as np
import pytest
import torch

import _module_adjoint as MAD
from mvxnet_makise_b200 import _lib, synth
from oracle import pointpath_oracle as O
from test_module_backward_cpu import SMALL_FPN, _hand_voxels

pytestmark = pytest.mark.gpu

G = synth.KITTI_GRID
IMSIZE = synth.KITTI_IMSIZE_HW
F64 = torch.float64


def rel(a, ref):
    a, ref = torch.as_tensor(a).double().cpu(), torch.as_tensor(ref).double().cpu()
    return float((a - ref).abs().max() / ref.abs().max().clamp_min(1e-30))


@pytest.fixture(scope='module')
def M():
    import mvxnet_makise_b200.modules as modules
    assert torch.cuda.is_available()
    return modules


def golden_voxels(golden_dir, tag='path_a'):
    g = np.load(f'{golden_dir}/{tag}.npz')
    v = torch.Tensor(O.group(O.points_with_proj(g['pcd4'], synth.kitti_calib()), G.velorange, G.voxelsize, G.T)[0])
    return v, int(g['map_seed']), int(g['weight_seed'])


LAYERS = [(1015, 768, 768, 'fcn'), (1015, 768, 128, 'fcn'), (1015, 128, 128, 'fcn'), (1015, 128, 16, 'fcn'), (1015, 16, 16, 'fcn'),
          (1015, 23, 16, 'vfe'), (1015, 32, 64, 'vfe'), (1015, 128, 128, 'fcn_max'),
          (1000, 768, 768, 'fcn'), (5003, 768, 128, 'fcn'), (777, 128, 128, 'fcn'), (256, 768, 768, 'fcn')]


@pytest.mark.parametrize('mode', [1, 0])
@pytest.mark.parametrize('R,cin,cout,kind', LAYERS)
def test_layer_backward_matches_fp64_formulas(M, R, cin, cout, kind, mode):
    T = 35 if kind != 'fcn' else 1
    torch.manual_seed(R + cin + cout)
    x = torch.randn(1, R // max(T, 1), T, cin, device='cuda')
    x[:, x.shape[1] // 2:] *= 0.01
    x[:, 3] = 0.5                                              # identical rows of one voxel: tied maxima
    x.requires_grad_(True)
    w = (torch.randn(cout, cin, device='cuda') / cin ** 0.5).requires_grad_(True)
    b = (torch.randn(cout, device='cuda') * 0.1).requires_grad_(True)
    try:
        _lib.set_gemm_mode(mode)
        out = M._layer_forward(kind, x, w, b, M.EPS, T)
        _, _, y_raw, stats = out.grad_fn.saved_tensors       # the CUDA forward's raw output and BatchNorm sums (freed by backward)
        dy = torch.randn_like(out)
        out.backward(dy)
        torch.cuda.synchronize()
    finally:
        _lib.set_gemm_mode(1)
    st = stats[:cout * 16].view(torch.float64).reshape(cout, 2).cpu()
    dx, dw, db = MAD.layer_backward(kind, x.detach().reshape(R, cin).cpu(), w.detach().cpu(), y_raw.cpu(),
                                    dy.reshape(-1, dy.shape[-1]).cpu(), T, M.EPS, st)
    errs = (rel(x.grad.reshape(R, cin), dx), rel(w.grad, dw), rel(b.grad, db))
    assert max(errs) < 1e-4, errs


def test_no_grad_path_is_the_forward_entry_and_recorded_outputs_are_bit_identical(M):
    torch.manual_seed(0)
    x = torch.randn(1, 40, 35, 32, device='cuda')
    x23, x128 = x[..., :23], x.repeat(1, 1, 1, 4)
    fcn, vfe, head = M.FCN(32, 768).cuda(), M.VFE(23, 16, 35).cuda(), M.VoxelNetHead().cuda()
    calls = [lambda: fcn(x), lambda: vfe(x23), lambda: M._layer_forward('fcn_max', x128, head.fcn.fc.weight, head.fcn.fc.bias, M.EPS, 35)]
    with torch.no_grad():
        ref = [c() for c in calls]
        assert all(r.grad_fn is None for r in ref)
        n0 = _lib.launch_count()
        fcn(x)
        n1 = _lib.launch_count()
        # what the module ran before it could train: the forward-only C entry, called directly
        x2, wt = x.reshape(-1, 32).contiguous(), M._wt(fcn.fc.weight)
        nbytes = ctypes.c_size_t()
        _lib.check(_lib.lib.mvx_layer_workspace_bytes(32, 768, ctypes.byref(nbytes)))
        ws = torch.empty(nbytes.value, dtype=torch.uint8, device='cuda')
        y = torch.empty(x2.shape[0], 768, device='cuda')
        n2 = _lib.launch_count()
        _lib.check(_lib.lib.mvx_fcn_forward(_lib.ptr(x2), x2.shape[0], 32, _lib.ptr(wt), _lib.ptr(fcn.fc.bias), 768, M.EPS, _lib.ptr(y),
                                            _lib.ptr(ws), _lib.stream_ptr()))
        n3 = _lib.launch_count()
    assert n1 - n0 == n3 - n2 and torch.equal(ref[0].reshape(-1, 768), y)
    got = [c() for c in calls]
    for g, r in zip(got, ref):
        assert g.grad_fn is not None and torch.equal(g.detach(), r)


def fusion_head(M, sd_np):
    fusion, head = M.ImageFeatureFusion().cuda(), M.VoxelNetHead().cuda()
    sd = {k: torch.from_numpy(np.asarray(v)) for k, v in sd_np.items()}
    fusion.load_state_dict({k[len('head.fusion.'):]: v for k, v in sd.items() if k.startswith('head.fusion.')})
    head.load_state_dict({k[len('backbone.'):]: v for k, v in sd.items() if k.startswith('backbone.')})
    return fusion, head


def oracle_grads(im768, vox7, sd_np, d_vfeat, dtype):
    params = {k: torch.from_numpy(np.asarray(v)).to(dtype).requires_grad_(True) for k, v in sd_np.items()}
    im16 = O.fusion(im768[None].to(dtype), params)
    vfeat = O.voxel_features(torch.concat([vox7[None].to(dtype), im16], dim=-1), params)
    (vfeat * d_vfeat.to(dtype)).sum().backward()
    return {k: p.grad for k, p in params.items()}


def test_fusion_and_voxel_feature_chains_match_fp64_autograd(M, golden_dir):
    v, map_seed, weight_seed = golden_voxels(golden_dir)
    sd_np = synth.make_weights(weight_seed)
    rng = np.random.default_rng(map_seed)
    maps = [torch.from_numpy(rng.standard_normal((1, 256, h, w), dtype=np.float32)) for h, w in SMALL_FPN]
    with torch.no_grad():
        im768 = O.feature_mapping(v, maps, torch.Tensor(list(IMSIZE)))
    d_vfeat = torch.from_numpy(np.random.default_rng(2).standard_normal((v.shape[0], 128)))
    ref = oracle_grads(im768, v[..., :7], sd_np, d_vfeat, F64)
    f32 = oracle_grads(im768, v[..., :7], sd_np, d_vfeat, torch.float32)
    fusion, head = fusion_head(M, sd_np)
    im16 = fusion(im768[None].cuda())
    vfeat = head.voxel_features(torch.cat([v[None][..., :7].cuda(), im16], dim=-1))
    (vfeat * d_vfeat.float().cuda()).sum().backward()
    got = {'head.fusion.' + k: p.grad for k, p in fusion.named_parameters()}
    got.update({'backbone.' + k: p.grad for k, p in head.named_parameters()})
    assert sorted(got) == sorted(ref)
    # The gradient is only piecewise continuous in the activations (ReLU masks, argmax of the max over T): any two fp32
    # evaluations take a few near-tie decisions differently, each moving one O(1) entry, and BatchNorm over 86 % identical pad
    # rows amplifies their rounding. The fp32 oracle is subject to the same effect, so its own distance to fp64 autograd is the
    # noise floor. Two independent fp32 evaluations land within a factor of two of each other, the bound of
    # tests/test_gpu_backward.py (one B200 run: 4.53e-2 against the fp32 oracle's 4.62e-2 over the chain, while fcn3's weight
    # alone gave 2.32e-2 against 2.14e-2). The tight bar is the per-layer test above: the CUDA backward within 1e-4 of the fp64
    # formulas on its own forward.
    ours = max(rel(got[k], ref[k]) for k in ref)
    noise = max(rel(f32[k], ref[k]) for k in ref)
    print(f'module chain gradients vs fp64 autograd: ours {ours:.3e}, fp32 oracle {noise:.3e}')
    assert ours <= 2 * noise + 1e-4, (ours, noise)


def test_feature_mapping_map_gradients(M, golden_dir):
    gv, _, _ = golden_voxels(golden_dir)
    voxels = torch.cat([_hand_voxels(), gv[:200]], 0)          # pad slots, border corners, tied slots, real rows
    rng = np.random.default_rng(5)
    maps = [torch.from_numpy(rng.standard_normal((1, 256, h, w), dtype=np.float32)) for h, w in SMALL_FPN]
    d_out = torch.from_numpy(np.random.default_rng(6).standard_normal((voxels.shape[0], G.T, 768)).astype(np.float32))
    leaves = [m.double().requires_grad_(True) for m in maps]
    out = O.feature_mapping(voxels.clone(), leaves, torch.Tensor(list(IMSIZE)))
    (out * d_out.double()).sum().backward()
    grads = []
    for _ in range(2):
        cm = [m.cuda().requires_grad_(True) for m in maps]
        vc = voxels.clone().cuda()
        o = M.featureMaping([vc], cm, None, torch.Tensor(list(IMSIZE)))[0]
        o.backward(d_out.cuda())
        grads.append([m.grad.clone() for m in cm])
        with torch.no_grad():
            o_ng = M.featureMaping([voxels.clone().cuda()], [m.cuda() for m in maps], None, torch.Tensor(list(IMSIZE)))[0]
        assert torch.equal(o.detach(), o_ng)
    for l in range(3):
        assert torch.equal(grads[0][l], grads[1][l]), 'reruns differ'
        assert rel(grads[0][l][0], leaves[l].grad[0]) < 1e-5, l
    g0 = grads[0][0][0].abs().sum(0)
    assert float(g0[-1].sum()) > 0 and float(g0[:, -1].sum()) > 0


@pytest.mark.parametrize('N', [0, 1, 300])
def test_reindex_backward_is_an_exact_gather(M, N):
    rng = np.random.default_rng(N)
    nx, ny, nz = G.voxelshape
    cells = rng.choice(nx * ny * nz, max(N, 1), replace=False)[:N]
    if N > 2:
        cells[1] = cells[0]                                     # duplicate cell: both rows receive its gradient
    iz, rem = np.divmod(cells, nx * ny)
    ix, iy = np.divmod(rem, ny)
    idx = torch.from_numpy(np.stack([np.zeros(N, np.int64), ix, iy, iz], 1)).cuda()
    x = torch.randn(N, 128, device='cuda', requires_grad=True)
    grid = M.reindex(x, idx)
    with torch.no_grad():
        assert torch.equal(grid.detach(), M.reindex(x.detach(), idx))
    dg = torch.randn_like(grid)
    grid.backward(dg)
    assert x.grad.shape == (N, 128)
    assert torch.equal(x.grad, dg[0, :, idx[:, 3], idx[:, 1], idx[:, 2]].t())


def test_training_step_through_the_drop_ins(M, golden_dir):
    v, map_seed, weight_seed = golden_voxels(golden_dir)
    fusion, head = fusion_head(M, synth.make_weights(weight_seed))
    rng = np.random.default_rng(map_seed)
    maps = [torch.nn.Parameter(torch.from_numpy(rng.standard_normal((1, 256, h, w), dtype=np.float32)).cuda()) for h, w in SMALL_FPN]
    idx = torch.from_numpy(np.load(f'{golden_dir}/path_a.npz')['idx']).cuda()
    params = list(fusion.parameters()) + list(head.parameters()) + maps
    opt = torch.optim.AdamW(params, lr=1e-3)

    def loss_fn():
        vc = v.clone().cuda()
        im768 = M.featureMaping([vc], maps, None, torch.Tensor(list(IMSIZE)))[0]
        im16 = fusion(im768[None])
        grid = head(torch.cat([vc[None][..., :7], im16], dim=-1), idx)
        return (grid * torch.linspace(-1, 1, grid.shape[1], device='cuda')[None, :, None, None, None]).square().sum()

    loss = loss_fn()
    loss.backward()
    assert all(p.grad is not None and bool(torch.isfinite(p.grad).all()) for p in params)
    first = [p.grad.clone() for p in params]
    loss_fn().backward()
    assert all(torch.allclose(p.grad, 2 * g, rtol=1e-3, atol=1e-6 * float(g.abs().max())) for p, g in zip(params, first))
    opt.step()
    with torch.no_grad():
        assert float(loss_fn()) != float(loss)


def test_full_size_frame_forward_and_backward(M):
    pcd6 = O.points_with_proj(synth.make_points(7), synth.kitti_calib())
    v = torch.Tensor(O.group(pcd6, G.velorange, G.voxelsize, G.T)[0]).cuda()
    assert v.shape[0] * G.T > 600_000
    maps = [torch.nn.Parameter(torch.randn(1, 256, h, w, device='cuda')) for h, w in synth.fpn_shapes()]
    fusion, head = fusion_head(M, synth.make_weights(1))
    im768 = M.featureMaping([v], maps, None, torch.Tensor(list(IMSIZE)))[0]
    vfeat = head.voxel_features(torch.cat([v[None][..., :7], fusion(im768[None])], dim=-1))
    (vfeat * torch.randn_like(vfeat)).sum().backward()
    torch.cuda.synchronize()
    for p in list(fusion.parameters()) + list(head.parameters()) + maps:
        assert p.grad is not None and bool(torch.isfinite(p.grad).all()) and float(p.grad.abs().max()) > 0
