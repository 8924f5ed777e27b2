"""The per-module backward, CPU side: the dense fp64 formulas of tests/_module_adjoint.py (what csrc/module_backward.cu and the
gather adjoint of csrc/map_backward.cu implement) against fp64 autograd through the oracle's reference modules, and the argument
validation of the new C entries."""
import ctypes
import os

import numpy as np
import pytest
import torch

import _module_adjoint as M
from mvxnet_makise_b200 import synth
from oracle import pointpath_oracle as O

G = synth.KITTI_GRID
SMALL_FPN = ((13, 42), (7, 21), (4, 11))
IMSIZE = synth.KITTI_IMSIZE_HW
FUSION = ['head.fusion.fcn1.fc', 'head.fusion.conv1.conv', 'head.fusion.fcn2.fc', 'head.fusion.conv2.conv', 'head.fusion.fcn3.fc']
VOXEL = ['backbone.svfe.vfe1.fcn.fc', 'backbone.svfe.vfe2.fcn.fc', 'backbone.fcn.fc']
F64 = torch.float64


def rel(a, b):
    return float((a.double() - b.double()).abs().max() / max(float(b.double().abs().max()), 1e-300))


def autograd_chain(voxels, maps, sd_np, d_vfeat):
    """fp64 autograd of featureMaping -> ImageFeatureFusion -> concat -> SVFE / FCN / max with the maps and the 16 parameters as
    leaves: {name: gradient}, [map gradients]"""
    params = {k: torch.from_numpy(np.asarray(v)).to(F64).requires_grad_(True) for k, v in sd_np.items()}
    feats = [torch.from_numpy(m).to(F64).requires_grad_(True) for m in maps]
    im768 = O.feature_mapping(voxels, feats, torch.Tensor(list(IMSIZE)))
    im16 = O.fusion(im768[None].to(F64), params)
    x23 = torch.concat([voxels[None][..., :7].to(F64), im16], dim=-1)
    vfeat = O.voxel_features(x23, params)
    (vfeat * d_vfeat).sum().backward()
    return {k: p.grad for k, p in params.items()}, [f.grad[0] for f in feats]


def formula_chain(voxels, maps, sd_np, d_vfeat):
    """the same gradients from the dense formulas, layer by layer (the order the modules' autograd nodes run in)"""
    sd = {k: torch.from_numpy(np.asarray(v)).to(F64) for k, v in sd_np.items()}
    N, T = voxels.shape[:2]
    R = N * T
    with torch.no_grad():
        im768 = O.feature_mapping(voxels, [torch.from_numpy(m).to(F64) for m in maps], torch.Tensor(list(IMSIZE)))
    xs, ys = [], []
    x = im768.reshape(R, -1).to(F64)
    for name in FUSION:
        xs.append(x)
        x, y = M.layer_forward('fcn', x, sd[name + '.weight'], sd[name + '.bias'])
        ys.append(y)
    x = torch.cat([voxels.reshape(R, 9)[:, :7].to(F64), x], 1)
    for name, kind in zip(VOXEL, ('vfe', 'vfe', 'fcn_max')):
        xs.append(x)
        x, y = M.layer_forward(kind, x, sd[name + '.weight'], sd[name + '.bias'], T)
        ys.append(y)
    grads = {}
    d = torch.as_tensor(d_vfeat).to(F64)
    for i, (name, kind) in reversed(list(enumerate(zip(FUSION + VOXEL, ['fcn'] * 5 + ['vfe', 'vfe', 'fcn_max'])))):
        d, dw, db = M.layer_backward(kind, xs[i], sd[name + '.weight'], ys[i], d, T)
        grads[name + '.weight'], grads[name + '.bias'] = dw.reshape(sd[name + '.weight'].shape), db
        if i == 5:
            d = d[:, 7:]          # the image-feature columns of VFE1's input (MVXNet.py:26)
    return grads, M.gather_adjoint(voxels, d, SMALL_FPN, IMSIZE)


def small_maps(seed):
    rng = np.random.default_rng(seed)
    return [rng.standard_normal((1, 256, h, w), dtype=np.float32) for (h, w) in SMALL_FPN]


def check_chain(voxels, maps, sd_np, seed):
    d_vfeat = torch.from_numpy(np.random.default_rng(seed).standard_normal((voxels.shape[0], 128)))
    ref, ref_maps = autograd_chain(voxels.clone(), maps, sd_np, d_vfeat)
    got, got_maps = formula_chain(voxels.clone(), maps, sd_np, d_vfeat)
    errs = {k: rel(got[k], ref[k]) for k in ref}
    errs.update({f'map{l}': rel(g, r) for l, (g, r) in enumerate(zip(got_maps, ref_maps))})
    assert max(errs.values()) < 1e-9, errs
    return ref, ref_maps


@pytest.mark.parametrize('tag', ['path_a', 'path_b'])
def test_dense_formulas_equal_autograd_on_golden_frames(golden_dir, tag):
    g = np.load(os.path.join(golden_dir, tag + '.npz'))
    voxels = torch.Tensor(O.group(O.points_with_proj(g['pcd4'], synth.kitti_calib()), G.velorange, G.voxelsize, G.T)[0])
    ref, ref_maps = check_chain(voxels, small_maps(int(g['map_seed'])), synth.make_weights(int(g['weight_seed'])), 3)
    assert all(float(v.abs().max()) > 0 for v in ref.values()) and all(float(m.abs().max()) > 0 for m in ref_maps)


def _hand_voxels():
    """an all-pad voxel, a voxel of identical points (tied maxima in every column), points whose corners sit on the last map row and
    column of every level, a point at the origin (a pad slot) and points at projection 0"""
    rng = np.random.default_rng(11)
    T = G.T
    v = np.zeros((5, T, 9), np.float32)
    row = np.concatenate([rng.uniform(1, 20, 3), rng.standard_normal(4), [100.0, 300.0]]).astype(np.float32)
    v[1, :6] = row                                             # six identical points: ties among them and among the pad slots
    for s, (h, w) in enumerate(SMALL_FPN):                      # the last row / column of each level
        rs = (np.float32(IMSIZE[0]) / np.float32(h), np.float32(IMSIZE[1]) / np.float32(w))
        v[2, s, :7] = np.concatenate([rng.uniform(1, 20, 3), rng.standard_normal(4)])
        v[2, s, 7:9] = ((h - 0.3) * rs[0], (w - 0.6) * rs[1])
        v[2, 3 + s, :7] = np.concatenate([rng.uniform(1, 20, 3), rng.standard_normal(4)])
        v[2, 3 + s, 7:9] = ((h - 1.0) * rs[0], 40.0 * (s + 1))
    v[3, 0, 6] = 0.7                                           # a real point at the origin: a pad slot
    v[3, 1, :7] = np.concatenate([rng.uniform(1, 20, 3), rng.standard_normal(4)])
    v[3, 1, 7:9] = (0.0, 0.0)
    v[4, :T, :7] = np.concatenate([rng.uniform(1, 20, (T, 3)), rng.standard_normal((T, 4))], 1)   # a full voxel
    v[4, :T, 7:9] = rng.uniform(0, 1, (T, 2)) * np.array(IMSIZE, np.float32)
    return torch.from_numpy(v)


def test_dense_formulas_equal_autograd_on_hand_made_voxels():
    voxels = _hand_voxels()
    ref, ref_maps = check_chain(voxels, small_maps(4), synth.make_weights(6), 8)
    d0 = ref_maps[0].abs().sum(0)
    assert float(d0[-1].sum()) > 0 and float(d0[:, -1].sum()) > 0   # corners on the last row and column were reached


def test_route_max_takes_the_first_of_tied_slots():
    y = torch.tensor([[[1.0, 2.0], [3.0, 2.0], [3.0, 0.5]]], dtype=F64)   # (V=1, T=3, C=2)
    r = M.route_max(y, torch.tensor([[10.0, 20.0]], dtype=F64))
    assert r[0, :, 0].tolist() == [0.0, 10.0, 0.0] and r[0, :, 1].tolist() == [20.0, 0.0, 0.0]


@pytest.mark.parametrize('cin,cout,kind', [(16, 16, 'fcn'), (23, 16, 'vfe'), (32, 64, 'vfe'), (128, 128, 'fcn_max'), (40, 16, 'fcn')])
def test_layer_formulas_equal_autograd_of_one_layer(cin, cout, kind):
    torch.manual_seed(cin + cout)
    N, T = 7, 5
    x = torch.randn(1, N, T, cin, dtype=F64)
    x[0, 2] = 0                                                  # identical rows: tied maxima
    x.requires_grad_(True)
    w = (torch.randn(cout, cin, dtype=F64) * 0.3).requires_grad_(True)
    b = (torch.randn(cout, dtype=F64) * 0.1).requires_grad_(True)
    if kind == 'fcn':
        out = O.crb(x, w, b)
    elif kind == 'vfe':
        out = O.vfe(x, w, b)
    else:
        out = torch.max(O.crb(x, w, b), dim=2)[0][0]
    dy = torch.randn_like(out)
    (out * dy).sum().backward()
    R = N * T
    y_raw = torch.relu(x.detach().reshape(R, cin) @ w.detach().t() + b.detach())
    dx, dw, db = M.layer_backward(kind, x.detach().reshape(R, cin), w.detach(), y_raw, dy.reshape(-1, dy.shape[-1]), T)
    assert rel(dx, x.grad.reshape(R, cin)) < 1e-9 and rel(dw, w.grad) < 1e-9 and rel(db, b.grad) < 1e-9


def test_reindex_backward_is_a_gather():
    N, C, shape = 6, 5, (4, 3, 2)
    x = torch.randn(N, C, dtype=F64, requires_grad=True)
    idx = torch.tensor([[0, 1, 2, 0], [0, 3, 0, 1], [0, 0, 0, 0], [0, 2, 1, 1], [0, 3, 2, 1], [0, 1, 1, 0]])
    grid = O.reindex(x, idx, shape)
    dg = torch.randn_like(grid)
    (grid * dg).sum().backward()
    assert torch.equal(x.grad, dg[0, :, idx[:, 3], idx[:, 1], idx[:, 2]].t())


def test_module_backward_argument_validation_without_gpu():
    from mvxnet_makise_b200 import _lib
    lib = _lib.lib
    n = ctypes.c_size_t()
    fake = ctypes.c_void_p(1 << 40)                              # never dereferenced: every call below fails its checks first
    R, T = 35 * 4, 35
    shapes = [(768, 768), (768, 128), (128, 128), (128, 16), (16, 16), (32, 16), (32, 64)]
    for cin, cout in shapes:
        assert lib.mvx_fcn_backward_workspace_bytes(R, cin, cout, ctypes.byref(n)) == 0 and n.value >= R * cout * 4
        assert lib.mvx_vfe_backward_workspace_bytes(R, T, cin, cout, ctypes.byref(n)) == 0
        assert lib.mvx_fcn_max_backward_workspace_bytes(R, T, cin, cout, ctypes.byref(n)) == 0
    assert lib.mvx_fcn_backward_workspace_bytes(R, 768, 768, None) == -1
    assert lib.mvx_fcn_backward_workspace_bytes(R, 784, 128, ctypes.byref(n)) == -1
    assert b'Cin' in lib.mvx_last_error()
    assert lib.mvx_fcn_backward_workspace_bytes(R, 23, 16, ctypes.byref(n)) == -1           # Cin is the padded width
    assert lib.mvx_fcn_backward_workspace_bytes(0, 16, 16, ctypes.byref(n)) == -1
    assert lib.mvx_vfe_backward_workspace_bytes(R + 1, T, 32, 16, ctypes.byref(n)) == -1
    assert b'multiple of T' in lib.mvx_last_error()
    assert lib.mvx_fcn_backward_workspace_bytes(R, 32, 48, ctypes.byref(n)) == -1           # no dW kernel for this shape
    assert lib.mvx_vfe_backward_workspace_bytes(R, T, 32, 16, ctypes.byref(n)) == 0
    need = n.value
    args = lambda **k: dict(dict(x=fake, wt=fake, y=fake, st=fake, dy=fake, dx=fake, dw=fake, db=fake, ws=fake, nb=need), **k)

    def vfe(a, R=R, T=T, cin=32):
        return lib.mvx_vfe_backward(a['x'], R, T, cin, a['wt'], 16, a['y'], a['st'], 1e-6, a['dy'], a['dx'], a['dw'], a['db'], 0,
                                    a['ws'], a['nb'], None)
    assert vfe(args(nb=need - 1)) == -3
    assert b'workspace' in lib.mvx_last_error()
    for k in ('x', 'wt', 'y', 'st', 'dy', 'dw', 'db', 'ws'):
        assert vfe(args(**{k: None})) == -1, k
    assert vfe(args(), R=R + 1) == -1
    assert vfe(args(), cin=784) == -1
    assert lib.mvx_fcn_max_backward(fake, R, 0, 32, fake, 16, fake, fake, 1e-6, fake, fake, fake, fake, 0, fake, need, None) == -1
    assert lib.mvx_fcn_backward(None, R, 32, fake, 16, fake, fake, 1e-6, fake, fake, fake, fake, 0, fake, need, None) == -1
    # training forward entries
    assert lib.mvx_fcn_forward_train(fake, R, 32, fake, fake, 16, 1e-6, fake, None, fake, None) == -1
    assert lib.mvx_vfe_forward_train(fake, R + 1, T, 32, fake, fake, 16, 1e-6, fake, fake, fake, fake, None) == -1
    assert lib.mvx_fcn_max_forward_train(fake, R, T, 32, fake, fake, 16, 1e-6, fake, None, fake, fake, None) == -1
    # gather adjoint
    mh = (ctypes.c_int32 * 3)(*[h for h, _ in SMALL_FPN])
    mw = (ctypes.c_int32 * 3)(*[w for _, w in SMALL_FPN])
    assert lib.mvx_feature_mapping_backward_workspace_bytes(R, mh, mw, ctypes.byref(n)) == 0 and n.value >= 3 * R * 24
    assert lib.mvx_feature_mapping_backward_workspace_bytes(R, None, mw, ctypes.byref(n)) == -1
    assert lib.mvx_feature_mapping_backward_workspace_bytes(-1, mh, mw, ctypes.byref(n)) == -1
    maps = (ctypes.c_void_p * 3)(fake, fake, fake)
    fm = lambda v, d, m, C, ws, nb: lib.mvx_feature_mapping_backward(v, R, d, mh, mw, C, 370.0, 1224.0, 1e-6, m, ws, nb, None)
    assert fm(fake, fake, maps, 256, fake, n.value - 1) == -3
    assert fm(None, fake, maps, 256, fake, n.value) == -1
    assert fm(fake, None, maps, 256, fake, n.value) == -1
    assert fm(fake, fake, (ctypes.c_void_p * 3)(fake, None, fake), 256, fake, n.value) == -1
    assert fm(fake, fake, maps, 254, fake, n.value) == -1
    assert fm(fake, fake, maps, 256, None, n.value) == -1
    # scatter adjoint
    sb = lib.mvx_scatter_dense_backward
    assert sb(None, None, 0, 128, 352, 400, 10, None, None) == 0                          # nothing to gather
    assert sb(None, fake, 5, 128, 352, 400, 10, fake, None) == -1
    assert sb(fake, fake, 5, 0, 352, 400, 10, fake, None) == -1
    assert sb(fake, fake, -1, 128, 352, 400, 10, fake, None) == -1
