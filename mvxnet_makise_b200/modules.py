"""Host-side mirror of the reference's nn.Module surface for the hot path (SURVEY.md §8b seam 3).

Same class names, constructor arguments, parameter names/shapes (checkpoint compatible) and forward
signatures as the reference; the arithmetic runs in the sm_100a kernels behind the C ABI.
They train like the reference's modules: when grad mode is on and an input, weight, bias or FPN map requires a gradient, the
call records an autograd node whose backward runs the CUDA backward entries (dLoss/d x, weight, bias; dLoss/d maps for
featureMaping; dLoss/d x for reindex). Otherwise the forward-only entries run, and no node is recorded.

  lidar2Img            modules/utils/Calib.py:47-70
  featureMaping        modules/imhead/Pipe.py:23-82
  FCN, CRB2d           modules/layers/Blocks.py:5-18, 31-40
  ImageFeatureFusion   modules/imhead/Pipe.py:84-104
  VFE, SVFE            modules/voxelnet/Pipe.py:5-29
  VoxelNetHead         modules/voxelnet/VoxelNet.py:16-34 (svfe, fcn, max over T, reindex)
"""
from __future__ import annotations

import ctypes
from typing import Dict, List, Sequence

import numpy as np
import torch
from torch import nn

from . import _lib
from ._lib import lib, check, ptr, stream_ptr

EPS = 1e-6          # cfg.eps with half: False (modules/config/Config.py:11-13)
SAMPLENUM = 35      # cfg.samplenum (config.yml:21)
VOXELSHAPE = (352, 400, 10)


def pack_calib(calib: Dict[str, torch.Tensor]) -> torch.Tensor:
    """[R0_rect @ Tr_velo_to_cam | P2] as 32 fp32 values. The 4x4 product is formed on the host in fp32 exactly as
    the reference forms it (Calib.py:65: `calib['R0_rect'] @ calib['Tr_velo_to_cam'] @ points` associates left)."""
    r0 = torch.as_tensor(calib['R0_rect'], dtype=torch.float32).cpu()
    tr = torch.as_tensor(calib['Tr_velo_to_cam'], dtype=torch.float32).cpu()
    p2 = torch.as_tensor(calib['P2'], dtype=torch.float32).cpu()
    return torch.cat([(r0 @ tr).reshape(-1), p2.reshape(-1)]).contiguous()


def calib_is_f64(calib: Dict) -> bool:
    """True when the calibration holds float64 matrices - what `readCalib` returns (Load.py:24-41: `np.zeros((4, 4))` and
    `np.concatenate([float32 block, [[0, 0, 0, 1]]])` are float64). The reference's numpy branches then evaluate the whole
    projection in fp64 (cropToSight at Load.py:73; lidar2Img of the pasted ground-truth sets, train.py:36-39); its torch
    branches see `torch.Tensor(calib[k])`, i.e. fp32 (Load.py:75-76, train.py:113-115)."""
    return any((isinstance(v, np.ndarray) and v.dtype == np.float64) or (isinstance(v, torch.Tensor) and v.dtype == torch.float64)
               for v in (calib['R0_rect'], calib['Tr_velo_to_cam'], calib['P2']))


def pack_calib64(calib: Dict) -> torch.Tensor:
    """[R0_rect @ Tr_velo_to_cam | P2] as 32 fp64 values, the 4x4 product formed by numpy in fp64 like Calib.py:65 does."""
    r0, tr, p2 = (np.asarray(calib[k].cpu() if isinstance(calib[k], torch.Tensor) else calib[k], dtype=np.float64)
                  for k in ('R0_rect', 'Tr_velo_to_cam', 'P2'))
    return torch.from_numpy(np.concatenate([(r0 @ tr).reshape(-1), p2.reshape(-1)])).contiguous()


def lidar2Img(pcd, calib: dict, uncheck: bool = False):
    """Project points to the image; returns (N,2) in (width, height) order like the reference.
    Accepts numpy or torch input and returns the same kind (torch results stay on the GPU). numpy points with a float64
    calibration (readCalib's dicts) follow the reference's numpy branch: fp64 arithmetic, float64 result."""
    _lib.require_cuda()
    assert pcd.ndim == 2, 'Point cloud should be in (N, 3 + C)'
    as_numpy = isinstance(pcd, np.ndarray)
    pts = torch.from_numpy(np.ascontiguousarray(pcd, dtype=np.float32)).cuda() if as_numpy \
        else pcd.to(device='cuda', dtype=torch.float32).contiguous()
    if as_numpy and calib_is_f64(calib):
        c64 = pack_calib64(calib).cuda()
        out = torch.empty((pts.shape[0], 2), dtype=torch.float64, device=pts.device)
        check(lib.mvx_lidar2img_f64(ptr(pts), pts.shape[1], pts.shape[0], ptr(c64), ptr(out), stream_ptr()), 'lidar2img_f64')
        if not uncheck:
            m = c64[:16].reshape(4, 4)
            depth = pts[:, :3].double() @ m[2, :3] + m[2, 3]
            out = out[depth > 0]
        return out.cpu().numpy()
    c32 = pack_calib(calib).cuda()
    out = torch.empty((pts.shape[0], 2), dtype=torch.float32, device=pts.device)
    check(lib.mvx_lidar2img(ptr(pts), pts.shape[1], pts.shape[0], ptr(c32), ptr(out), stream_ptr()), 'lidar2img')
    if not uncheck:   # Calib.py:66-67: drop points behind the camera (depth = row 2 of (R0@Tr)@p)
        m = c32[:16].reshape(4, 4)
        depth = pts[:, :3] @ m[2, :3] + m[2, 3]
        out = out[depth > 0]
    return out.cpu().numpy() if as_numpy else out


def _records(*tensors) -> bool:
    """Record an autograd node only when the result can carry a gradient back to one of these tensors."""
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors)


def _map_extents(features):
    hw = [(int(f.shape[-2]), int(f.shape[-1])) for f in features]
    return (ctypes.c_int32 * 3)(*[h for h, _ in hw]), (ctypes.c_int32 * 3)(*[w for _, w in hw])


def _feature_mapping_frame(v: torch.Tensor, maps, C: int, imsize, eps: float):
    """mvx_feature_mapping for one frame; returns (out, the contiguous voxel tensor the kernel read and zeroed)."""
    assert v.is_cuda and v.dtype == torch.float32 and v.shape[-1] == 9
    mh, mw = _map_extents(maps)
    nbytes = ctypes.c_size_t()
    check(lib.mvx_maps_nhwc_bytes(mh, mw, C, ctypes.byref(nbytes)), 'maps_nhwc_bytes')
    vc = v if v.is_contiguous() else v.contiguous()
    R = vc.numel() // 9
    maps = [m.detach().contiguous() for m in maps]
    ws = torch.empty(nbytes.value, dtype=torch.uint8, device=v.device)
    out = torch.empty(tuple(v.shape[:-1]) + (3 * C,), dtype=torch.float32, device=v.device)
    mp = (ctypes.c_void_p * 3)(*[m.data_ptr() for m in maps])
    check(lib.mvx_feature_mapping(ptr(vc), R, mp, mh, mw, C, float(imsize[0]), float(imsize[1]), float(eps), ptr(out), ptr(ws),
                                  nbytes.value, stream_ptr()), 'feature_mapping')
    if vc is not v:
        v.copy_(vc)
    return out, vc


class _FeatureMappingFunction(torch.autograd.Function):
    """featureMaping of one frame with the frame's three maps as inputs; backward = mvx_feature_mapping_backward (the adjoint of
    the 4-corner sample). The voxel tensor is data (no gradient), passed inside a list so that autograd does not track it."""

    @staticmethod
    def forward(ctx, vbox, imsize, eps, m0, m1, m2):
        out, vc = _feature_mapping_frame(vbox[0], [m0, m1, m2], int(m0.shape[0]), imsize, eps)
        ctx.save_for_backward(vc)
        ctx.imsize, ctx.eps = imsize, eps
        ctx.map_meta = [(m.shape, m.dtype) for m in (m0, m1, m2)]
        return out

    @staticmethod
    def backward(ctx, d_out):
        vc, = ctx.saved_tensors
        shapes = [shp for shp, _ in ctx.map_meta]
        C = int(shapes[0][0])
        R = vc.numel() // 9
        mh = (ctypes.c_int32 * 3)(*[int(shp[-2]) for shp in shapes])
        mw = (ctypes.c_int32 * 3)(*[int(shp[-1]) for shp in shapes])
        nbytes = ctypes.c_size_t()
        check(lib.mvx_feature_mapping_backward_workspace_bytes(R, mh, mw, ctypes.byref(nbytes)), 'feature_mapping_backward_workspace_bytes')
        d_out = d_out.to(torch.float32).contiguous()
        ws = torch.empty(nbytes.value, dtype=torch.uint8, device=vc.device)
        d_maps = [torch.empty(tuple(shp), dtype=torch.float32, device=vc.device) for shp in shapes]
        dp = (ctypes.c_void_p * 3)(*[d.data_ptr() for d in d_maps])
        check(lib.mvx_feature_mapping_backward(ptr(vc), R, ptr(d_out), mh, mw, C, float(ctx.imsize[0]), float(ctx.imsize[1]),
                                               float(ctx.eps), dp, ptr(ws), nbytes.value, stream_ptr()), 'feature_mapping_backward')
        grads = [d.to(dt) if need else None for d, (_, dt), need in zip(d_maps, ctx.map_meta, ctx.needs_input_grad[3:])]
        return (None, None, None, *grads)


def featureMaping(voxels, features: List[torch.Tensor], calibs, imsize: torch.Tensor, eps: float = EPS):
    """Drop-in for ``featureMaping`` (Pipe.py:23-82). voxels: batch * (N,T,C>=9 is NOT required: exactly the
    reference layout (N,T,9)); features: 3 maps (batch,256,Hf,Wf); returns batch * (N,T,768).
    Side effects kept: pad slots (x==y==z==0) of ``voxels`` are zeroed in place (Pipe.py:53-59).
    Unlike the reference the ``features`` list is not replaced by padded copies (the pad is a bounds predicate).
    Maps that require a gradient receive dLoss/d map through the adjoint of the 4-corner sample (no gradient reaches voxels)."""
    _lib.require_cuda()
    res = []
    C = int(features[0].shape[1])
    ims = (float(imsize[0]), float(imsize[1]))
    for i, v in enumerate(voxels):
        maps = [f[i] for f in features]
        if _records(*maps):
            res.append(_FeatureMappingFunction.apply([v], ims, float(eps), *maps))
        else:
            res.append(_feature_mapping_frame(v, maps, C, ims, eps)[0])
    return res


def _pad_cols(x2d: torch.Tensor, mult: int = 16) -> torch.Tensor:
    cin = x2d.shape[1]
    pad = (-cin) % mult
    if pad == 0:
        return x2d.contiguous()
    return torch.cat([x2d, x2d.new_zeros((x2d.shape[0], pad))], dim=1).contiguous()


def _wt(weight: torch.Tensor, mult: int = 16) -> torch.Tensor:
    """(Cout, Cin[,1,1]) -> W^T (Cin_pad, Cout) fp32 contiguous, zero rows for the padded inputs."""
    w = weight.detach().reshape(weight.shape[0], -1).to(torch.float32)
    wt = w.t().contiguous()
    pad = (-wt.shape[0]) % mult
    if pad:
        wt = torch.cat([wt, wt.new_zeros((pad, wt.shape[1]))], dim=0).contiguous()
    return wt


_FORWARD = {'fcn': 'fcn_forward', 'vfe': 'vfe_forward', 'fcn_max': 'fcn_max_forward'}


def _layer_call(kind: str, x: torch.Tensor, weight, bias, eps: float, T: int, train: bool):
    """One dense layer entry. Returns (y, y_raw, stats workspace); train selects the *_forward_train entry, which also keeps
    the raw post-ReLU output y_raw (R, Cout) and leaves the fp64 sums of the layer in the stats workspace."""
    _lib.require_cuda()
    lead = x.shape[:-1]
    cout = weight.shape[0]
    x2 = _pad_cols(x.detach().reshape(-1, x.shape[-1]).to(torch.float32))
    wt = _wt(weight)
    b = bias.detach().to(torch.float32).contiguous()
    R, cin = x2.shape
    nbytes = ctypes.c_size_t()
    check(lib.mvx_layer_workspace_bytes(cin, cout, ctypes.byref(nbytes)), 'layer_workspace_bytes')
    stats = torch.empty(nbytes.value, dtype=torch.uint8, device=x.device)
    y_raw = torch.empty((R, cout), dtype=torch.float32, device=x.device) if train else None
    raw = (ptr(y_raw),) if train else ()
    name = _FORWARD[kind] + ('_train' if train else '')
    fn = getattr(lib, 'mvx_' + name)
    if kind == 'fcn':
        y = torch.empty((R, cout), dtype=torch.float32, device=x.device)
        check(fn(ptr(x2), R, cin, ptr(wt), ptr(b), cout, float(eps), ptr(y), *raw, ptr(stats), stream_ptr()), name)
        return y.reshape(lead + (cout,)), y_raw, stats
    vmax = torch.empty((R // T, cout), dtype=torch.int32, device=x.device)
    if kind == 'vfe':
        y = torch.empty((R, 2 * cout), dtype=torch.float32, device=x.device)
        check(fn(ptr(x2), R, T, cin, ptr(wt), ptr(b), cout, float(eps), ptr(y), *raw, ptr(stats), ptr(vmax), stream_ptr()), name)
        return y.reshape(lead + (2 * cout,)), y_raw, stats
    y = torch.empty((R // T, cout), dtype=torch.float32, device=x.device)
    check(fn(ptr(x2), R, T, cin, ptr(wt), ptr(b), cout, float(eps), ptr(y), *raw, ptr(stats), ptr(vmax), stream_ptr()), name)
    return y, y_raw, stats


class _LayerFunction(torch.autograd.Function):
    """FCN / CRB2d (kind 'fcn'), VFE ('vfe') and the last FCN + max over T ('fcn_max') with x, weight and bias as inputs; backward =
    mvx_{kind}_backward on the training forward's raw output and BatchNorm sums."""

    @staticmethod
    def forward(ctx, x, weight, bias, kind, eps, T):
        y, y_raw, stats = _layer_call(kind, x, weight, bias, eps, T, train=True)
        ctx.save_for_backward(x, weight, y_raw, stats)
        ctx.kind, ctx.eps, ctx.T, ctx.bias_dtype = kind, eps, T, bias.dtype
        return y

    @staticmethod
    def backward(ctx, dy):
        x, weight, y_raw, stats = ctx.saved_tensors
        kind, T = ctx.kind, ctx.T
        need_x, need_w, need_b = ctx.needs_input_grad[:3]
        cin_true, cout = x.shape[-1], weight.shape[0]
        x2 = _pad_cols(x.detach().reshape(-1, cin_true).to(torch.float32))
        wt = _wt(weight)
        R, cin = x2.shape
        dy = dy.to(torch.float32).contiguous()
        dx = torch.empty((R, cin), dtype=torch.float32, device=x.device) if need_x else None
        dW = torch.empty((cout, cin), dtype=torch.float32, device=x.device)
        db = torch.empty((cout,), dtype=torch.float32, device=x.device)
        nbytes = ctypes.c_size_t()
        lead = (R,) if kind == 'fcn' else (R, T)
        check(getattr(lib, f'mvx_{kind}_backward_workspace_bytes')(*lead, cin, cout, ctypes.byref(nbytes)), f'{kind}_backward_workspace_bytes')
        ws = torch.empty(nbytes.value, dtype=torch.uint8, device=x.device)
        check(getattr(lib, f'mvx_{kind}_backward')(ptr(x2), *lead, cin, ptr(wt), cout, ptr(y_raw), ptr(stats), float(ctx.eps), ptr(dy),
                                                    ptr(dx), ptr(dW), ptr(db), 0, ptr(ws), nbytes.value, stream_ptr()), f'{kind}_backward')
        gx = dx[:, :cin_true].reshape(x.shape).to(x.dtype) if need_x else None
        gw = dW[:, :cin_true].reshape(weight.shape).to(weight.dtype) if need_w else None
        gb = db.to(ctx.bias_dtype) if need_b else None
        return gx, gw, gb, None, None, None


def _layer_forward(kind: str, x: torch.Tensor, weight, bias, eps: float, T: int = 1):
    """x (..., Cin) CUDA fp32 -> BN(relu(x W^T + b)) with batch statistics over all leading dims."""
    if _records(x, weight, bias):
        return _LayerFunction.apply(x, weight, bias, kind, eps, T)
    return _layer_call(kind, x, weight, bias, eps, T, train=False)[0]


class FCN(nn.Module):
    """Blocks.py:5-18: relu(Linear) -> BatchNorm2d(affine=False, track_running_stats=False). Input (batch,h,w,c)."""

    def __init__(self, cin, cout, eps: float = EPS):
        super().__init__()
        self.fc = nn.Linear(cin, cout)
        self.eps = eps

    def forward(self, x):
        return _layer_forward('fcn', x, self.fc.weight, self.fc.bias, self.eps)


class CRB2d(nn.Module):
    """Blocks.py:31-40 for the 1x1/stride-1/no-pad case the path uses (Pipe.py:89,91). Input (batch,c,h,w)."""

    def __init__(self, cin, cout, k, s, p, eps: float = EPS):
        super().__init__()
        if (k, s, p) != (1, 1, 0):
            raise NotImplementedError('only the 1x1 CRB2d of the fusion stack is on the hot path')
        self.conv = nn.Conv2d(cin, cout, k, s, p)
        self.eps = eps

    def forward(self, x):
        y = _layer_forward('fcn', x.permute(0, 2, 3, 1), self.conv.weight, self.conv.bias, self.eps)
        return y.permute(0, 3, 1, 2)


class ImageFeatureFusion(nn.Module):
    """Pipe.py:84-104: 768 -> 768 -> 128 -> 128 -> 16 -> 16."""

    def __init__(self):
        super().__init__()
        self.fcn1 = FCN(768, 768)
        self.conv1 = CRB2d(768, 128, 1, 1, 0)
        self.fcn2 = FCN(128, 128)
        self.conv2 = CRB2d(128, 16, 1, 1, 0)
        self.fcn3 = FCN(16, 16)

    def forward(self, x):
        x = self.fcn1(x)
        x = self.conv1(x.permute(0, 3, 1, 2)).permute(0, 2, 3, 1)
        x = self.fcn2(x)
        x = self.conv2(x.permute(0, 3, 1, 2)).permute(0, 2, 3, 1)
        return self.fcn3(x)


class VFE(nn.Module):
    """voxelnet/Pipe.py:5-18: FCN -> max over T -> tile -> concat. Input (batch,N,T,cin) -> (batch,N,T,2*cout)."""

    def __init__(self, cin, cout, sampleNum):
        super().__init__()
        self.fcn = FCN(cin, cout)
        self.sampleNum = sampleNum

    def forward(self, x):
        assert x.shape[2] == self.sampleNum
        return _layer_forward('vfe', x, self.fcn.fc.weight, self.fcn.fc.bias, self.fcn.eps, T=self.sampleNum)


class SVFE(nn.Module):
    """voxelnet/Pipe.py:20-29."""

    def __init__(self, sampleNum=SAMPLENUM):
        super().__init__()
        self.vfe1 = VFE(7 + 16, 16, sampleNum)
        self.vfe2 = VFE(32, 64, sampleNum)

    def forward(self, x):
        return self.vfe2(self.vfe1(x))


def _reindex_call(x: torch.Tensor, idx: torch.Tensor, voxelshape: Sequence[int]) -> torch.Tensor:
    _lib.require_cuda()
    nx, ny, nz = (int(s) for s in voxelshape)
    x = x.detach().to(torch.float32).contiguous()
    N, C = x.shape
    out = torch.empty((1, C, nz, nx, ny), dtype=torch.float32, device=x.device)
    G = nx * ny * nz
    mapws = torch.empty(G + G // 32 + 1, dtype=torch.int32, device=x.device)
    check(lib.mvx_scatter_dense(ptr(x), ptr(idx), N, C, nx, ny, nz, ptr(out), ptr(mapws), stream_ptr()), 'scatter_dense')
    return out


class _ReindexFunction(torch.autograd.Function):
    """reindex with x as input; backward = mvx_scatter_dense_backward (a gather of the grid gradient at every voxel's cell)."""

    @staticmethod
    def forward(ctx, x, idx, voxelshape):
        ctx.save_for_backward(idx)
        ctx.voxelshape, ctx.x_dtype = voxelshape, x.dtype
        return _reindex_call(x, idx, voxelshape)

    @staticmethod
    def backward(ctx, d_grid):
        idx, = ctx.saved_tensors
        nx, ny, nz = (int(s) for s in ctx.voxelshape)
        d_grid = d_grid.to(torch.float32).contiguous()
        N, C = idx.shape[0], d_grid.shape[1]
        dx = torch.empty((N, C), dtype=torch.float32, device=d_grid.device)
        check(lib.mvx_scatter_dense_backward(ptr(d_grid), ptr(idx), N, C, nx, ny, nz, ptr(dx), stream_ptr()), 'scatter_dense_backward')
        return dx.to(ctx.x_dtype), None, None


def reindex(x: torch.Tensor, idx: torch.Tensor, voxelshape: Sequence[int] = VOXELSHAPE) -> torch.Tensor:
    """Drop-in for ``VoxelNet.reindex`` (VoxelNet.py:16-22): (N,C) + idx (N,4) int64 -> (1,C,nz,nx,ny)."""
    idx = idx.to(torch.int64).contiguous()
    if _records(x):
        return _ReindexFunction.apply(x, idx, tuple(voxelshape))
    return _reindex_call(x, idx, voxelshape)


class VoxelNetHead(nn.Module):
    """The hot-path part of ``VoxelNet`` (VoxelNet.py:9-34): svfe, fcn, max over T, reindex. ``cml``/``rpn`` stay the
    reference's stock modules and consume the returned grid. Parameter names match ``backbone.svfe.*``/``backbone.fcn.*``."""

    def __init__(self, sampleNum=SAMPLENUM, voxelshape=VOXELSHAPE):
        super().__init__()
        self.svfe = SVFE(sampleNum)
        self.fcn = FCN(128, 128)
        self.sampleNum = sampleNum
        self.voxelshape = tuple(voxelshape)

    reindex = staticmethod(reindex)

    def voxel_features(self, x):
        x = self.svfe(x)
        return _layer_forward('fcn_max', x, self.fcn.fc.weight, self.fcn.fc.bias, self.fcn.eps, T=self.sampleNum)

    def forward(self, x, idx):
        return reindex(self.voxel_features(x), idx, self.voxelshape)
