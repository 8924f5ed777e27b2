"""Drop-in for the reference's own objects: the unmodified `MVXNet` model and `train.py` loop keep working, the hot path
underneath them runs on the sm_100a kernels.

    from MVXNet import MVXNet                       # the reference's class, untouched
    from mvxnet_makise_b200.dropin import accelerate, install_extension
    install_extension()                             # modules/Extension.py seam: cpp._group / _classifyAnchors / bboxOverlap / bboxIntersection
    model = accelerate(MVXNet().to(device))         # same parameters, same state_dict, same forward signature
    score, reg = model(voxel, img, idx, [calib], imsize)     # train.py:131, unchanged
    loss.backward(); opt.step()                     # train.py:161-162, unchanged: gradients reach head.fusion.* / backbone.svfe.* / backbone.fcn.*

What `accelerate` replaces is the body of `MVXNet.forward` (MVXNet.py:21-27) between the image backbone and the CML:
`featureMaping` -> `ImageFeatureFusion` -> concat -> `SVFE` -> `FCN` -> max over T -> `reindex` become one call of the fused
path on the dense-voxel entry (`PointPath.forward_voxels`), wrapped in a `torch.autograd.Function` whose backward is the CUDA
backward of the eight layers (`mvx_pointpath_backward`) and, when the FPN maps want a gradient, of the 4-corner gather
(`mvx_pointpath_backward_maps`). `head.extractor` (the torchvision backbone: frozen by Head.py:9-11, trained like any module
after `model.head.extractor.requires_grad_(True)`), `backbone.cml` and `backbone.rpn` stay the reference's own modules. The model's `nn.Parameter`s remain the single source of truth: they are read
on every forward (an optimiser step is picked up through the tensors' version counters) and receive `.grad` like any other
parameter, so `model.parameters()`, `AdamW`, `state_dict()` / `load_state_dict()` and checkpoints are unaffected.
"""
from __future__ import annotations

import sys
import types
from typing import List, Sequence

import torch

from . import synth
from .modules import _records
from .pipeline import PointPath

_HOT = [name for name, *_ in synth.HOT_LAYERS]


def _get(module, dotted: str):
    for part in dotted.split('.'):
        module = getattr(module, part)
    return module


def hot_parameters(model) -> List[torch.nn.Parameter]:
    """The 16 tensors of the eight hot-path layers, checkpoint order (SURVEY.md §8b): weight, bias per layer."""
    out = []
    for name in _HOT:
        out += [_get(model, name + '.weight'), _get(model, name + '.bias')]
    return out


def _path_inputs(path: PointPath, params: Sequence[torch.Tensor], maps) -> List[torch.Tensor]:
    """Pushes the parameters into the path's W^T / bias tensors (skipped while their version counters stand still) and
    returns the maps as the fp32 contiguous tensors the path reads."""
    versions = tuple((p.data_ptr(), p._version) for p in params)
    if path._param_versions != versions:
        with torch.no_grad():
            path.load_parameters(params)
        path._param_versions = versions
    return [m.detach().to(torch.float32).contiguous() for m in maps]


def _check_record(ctx):
    if ctx.path._record is not ctx.record:
        raise RuntimeError('the hot path ran another forward before this backward: its saved activations are gone '
                           '(one forward/backward at a time per accelerated model)')


def _path_backward(ctx, wanted_maps, wanted_params, d_vfeat=None, d_grid=None):
    """The path backward of a node: (16 parameter gradients, 3 map gradients in the maps' own dtypes), None where not wanted"""
    path = ctx.path
    d_maps = None
    if any(wanted_maps):       # the map backward runs only when a map wants a gradient
        d_maps = [torch.empty(m.shape, dtype=torch.float32, device=path.device) for m in ctx.record.maps]
    flat = path.backward(d_vfeat=d_vfeat, d_grid=d_grid, d_maps=d_maps)
    grads = list(path.grads(flat).values()) if any(wanted_params) else [None] * (2 * len(_HOT))
    if d_maps is None:
        return grads, [None] * 3
    return grads, [d.to(dt) if w else None for d, w, dt in zip(d_maps, wanted_maps, ctx.map_dtypes)]


class HotPathFunction(torch.autograd.Function):
    """grid = hot_path(voxels, idx, fpn maps 0..2; 16 parameters). Differentiable with respect to the parameters and the three
    FPN maps (the image backbone trains when `head.extractor` is unfrozen); the voxel tensor is data. Map gradients are
    computed only where `needs_input_grad` asks for them, in each map's own dtype."""

    @staticmethod
    def forward(ctx, path: PointPath, voxels, idx, m0, m1, m2, *params):
        maps = _path_inputs(path, params, (m0, m1, m2))
        nz, nx, ny = path.grid.shape[2], path.grid.shape[0], path.grid.shape[1]
        B = len(voxels) if isinstance(voxels, (list, tuple)) else 1
        grid = torch.empty((B, 128, nz, nx, ny), dtype=torch.float32, device=path.device)   # a fresh tensor: the CML saves it for ITS backward
        path.forward_voxels(voxels, idx, maps, want_grid=True, train=True, grid_out=grid)
        ctx.path, ctx.record = path, path._record
        ctx.map_dtypes = [m.dtype for m in (m0, m1, m2)]
        return grid

    @staticmethod
    def backward(ctx, d_grid):
        _check_record(ctx)
        grads, map_grads = _path_backward(ctx, ctx.needs_input_grad[3:6], ctx.needs_input_grad[6:], d_grid=d_grid.contiguous())
        return (None, None, None, *map_grads, *grads)


def hot_path(path: PointPath, voxels, idx, maps, params: Sequence[torch.Tensor]) -> torch.Tensor:
    """The dense grid (B,128,nz,nx,ny) for the reference's (voxels, idx) arguments. Records an autograd node when gradients are
    enabled and a parameter or an FPN map wants one; otherwise takes the inference route (pixel-first fcn1, no saved
    activations)."""
    maps = list(maps)
    if _records(*params, *maps):
        return HotPathFunction.apply(path, voxels, idx, *maps, *params)
    grid, _ = path.forward_voxels(voxels, idx, _path_inputs(path, params, maps), want_grid=True, train=False)
    return grid


class SparseConv1Function(torch.autograd.Function):
    """y1 = backbone.cml.conv1(hot_path(voxels, idx, fpn maps 0..2; 16 parameters)) without the dense grid: the sparse hand-off
    (`PointPath.cml_conv1`) reads the voxel features directly. Differentiable with respect to the 16 hot-path parameters, the
    three FPN maps and the conv1 weight / bias. `train` says whether a hot parameter or a map wants a gradient: without one
    the path forward runs in inference mode and the backward skips d_vfeat and the path backward (fine-tuning of the CML
    alone)."""

    @staticmethod
    def forward(ctx, path: PointPath, eps: float, train: bool, voxels, idx, m0, m1, m2, *params):
        hot, weight, bias = params[:-2], params[-2], params[-1]
        path.forward_voxels(voxels, idx, _path_inputs(path, hot, (m0, m1, m2)), want_grid=False, train=train)
        y1 = path.cml_conv1(weight, bias, eps)
        ctx.path, ctx.record, ctx.eps, ctx.train = path, path._record, eps, train
        ctx.map_dtypes = [m.dtype for m in (m0, m1, m2)]
        ctx.save_for_backward(weight, bias)
        return y1

    @staticmethod
    def backward(ctx, d_y1):
        _check_record(ctx)
        weight, bias = ctx.saved_tensors
        d_vfeat, d_w, d_b = ctx.path.cml_conv1_backward(d_y1.contiguous(), weight, bias, ctx.eps, want_d_vfeat=ctx.train)
        grads, map_grads = [None] * (2 * len(_HOT)), [None] * 3
        if ctx.train:
            grads, map_grads = _path_backward(ctx, ctx.needs_input_grad[5:8], ctx.needs_input_grad[8:8 + 2 * len(_HOT)], d_vfeat=d_vfeat)
        return (None, None, None, None, None, *map_grads, *grads, d_w, d_b)


def sparse_conv1(path: PointPath, voxels, idx, maps, params: Sequence[torch.Tensor], weight, bias, eps: float) -> torch.Tensor:
    """`backbone.cml.conv1` of the grid `hot_path` would return, (B, 64, (nz+1)//2, nx, ny), computed without that grid. Records an
    autograd node when gradients are enabled and any of the 18 tensors or an FPN map wants one."""
    maps = list(maps)
    train = _records(*params, *maps)
    if train or _records(weight, bias):
        return SparseConv1Function.apply(path, eps, train, voxels, idx, *maps, *params, weight, bias)
    path.forward_voxels(voxels, idx, _path_inputs(path, params, maps), want_grid=False, train=False)
    return path.cml_conv1(weight, bias, eps)


def _stock_conv1_eps(cml) -> float:
    """`cml.conv1` must be the stock CRB3d(128, 64, 3, (2,1,1), (1,1,1)) (voxelnet/Pipe.py:31-43, Blocks.py CRB3d): Conv3d with
    bias, ReLU, BatchNorm3d(affine=False, track_running_stats=False). Returns that BatchNorm's eps; raises otherwise."""
    block = cml.conv1
    conv = getattr(block, 'conv', None)
    bns = [m for m in block.modules() if isinstance(m, torch.nn.modules.batchnorm._BatchNorm)]
    ok = (isinstance(conv, torch.nn.Conv3d) and conv.in_channels == 128 and conv.out_channels == 64 and conv.kernel_size == (3, 3, 3)
          and conv.stride == (2, 1, 1) and conv.padding == (1, 1, 1) and conv.dilation == (1, 1, 1) and conv.groups == 1
          and conv.bias is not None and conv.padding_mode == 'zeros'
          and len(bns) == 1 and isinstance(bns[0], torch.nn.BatchNorm3d) and not bns[0].affine and not bns[0].track_running_stats
          and sum(1 for m in block.modules() if isinstance(m, torch.nn.Conv3d)) == 1)
    if not ok:
        raise ValueError('sparse_cml_conv1=True needs the stock backbone.cml.conv1: CRB3d(128, 64, 3, (2,1,1), (1,1,1)) = Conv3d with '
                         'bias, ReLU, BatchNorm3d(affine=False, track_running_stats=False)')
    return float(bns[0].eps)


def _forward(self, voxels, imgs, idx, calibs, imsize):
    """`MVXNet.forward(voxels, imgs, idx, calibs, imsize)` (MVXNet.py:21-27): same arguments, same (score, reg) result.
    `calibs` is accepted and unused, as in the reference's featureMaping (the projection already sits in voxels[..., 7:9])."""
    path = self._mvx_path
    hw = self._mvx_imsize.get(id(imsize))
    if hw is None:                                   # cfg.imsize travels as a tensor (train.py:69): read it once, not per step
        hw = (float(imsize[0]), float(imsize[1]))
        self._mvx_imsize[id(imsize)] = hw
    path.imsize_hw = hw
    feats = self.head.extractor(imgs)                # FPN levels '0','1','2' (Pipe.py:17-21); trains when unfrozen
    nx, ny = path.grid.shape[0], path.grid.shape[1]
    if self._mvx_sparse_conv1:                       # CML.forward (voxelnet/Pipe.py:31-43) with conv1 taken from the voxel features
        cml = self.backbone.cml
        y1 = sparse_conv1(path, voxels, idx.to(torch.int64), feats, hot_parameters(self), cml.conv1.conv.weight, cml.conv1.conv.bias,
                          self._mvx_conv1_eps)
        outs = [self.backbone.rpn(cml.conv3(cml.conv2(y1[b:b + 1])).reshape((1, -1, nx, ny))) for b in range(y1.shape[0])]
        return outs[0] if len(outs) == 1 else outs
    grid = hot_path(path, voxels, idx.to(torch.int64), feats, hot_parameters(self))
    outs = []
    for b in range(grid.shape[0]):                   # CML / RPN are batch-1 in the reference (VoxelNet.py:35-37)
        x = self.backbone.cml(grid[b:b + 1])
        outs.append(self.backbone.rpn(x.reshape((1, -1, nx, ny))))
    return outs[0] if len(outs) == 1 else outs


def accelerate(model, grid: synth.GridSpec = synth.KITTI_GRID, imsize_hw: Sequence[int] = synth.KITTI_IMSIZE_HW, eps: float = 1e-6,
               sparse_cml_conv1: bool = False):
    """Swap the hot path of a reference `MVXNet` instance (already on its CUDA device) for the fused sm_100a path, in place.
    `grid` / `eps` mirror config.yml (velorange, voxelshape, samplenum; eps 1e-6 with half: False). Returns the model.

    sparse_cml_conv1=True also computes `backbone.cml.conv1` sparsely from the voxel features, forward and backward, so the
    dense (B,128,nz,nx,ny) grid is never written; conv2 / conv3 and the RPN remain the model's own modules. Opt-in because a
    caller can tell the difference: `backbone.cml` and `cml.conv1` are not called as modules (their hooks do not fire) and
    no grid tensor exists. conv1 must be the stock block (ValueError otherwise)."""
    params = hot_parameters(model)                   # raises AttributeError if this is not the reference's module tree
    conv1_eps = _stock_conv1_eps(model.backbone.cml) if sparse_cml_conv1 else None
    dev = params[0].device
    if dev.type != 'cuda':
        raise RuntimeError('accelerate() needs the model on a CUDA device; mvxnet_makise_b200 has no CPU fallback')
    sd = {name + suffix: _get(model, name + suffix).detach() for name in _HOT for suffix in ('.weight', '.bias')}
    model._mvx_path = PointPath(sd, grid, imsize_hw, eps, device=dev)
    model._mvx_imsize = {}
    model._mvx_sparse_conv1, model._mvx_conv1_eps = bool(sparse_cml_conv1), conv1_eps
    model.forward = types.MethodType(_forward, model)
    return model


def install_extension():
    """The `modules/Extension.py` seam (Extension.py:1-3): point every already-imported user of the reference's `cpp` object
    (modules/data/Preprocessing.py:3, modules/Calc.py:4, modules/augment/Augment.py:6) at the CUDA implementation. Returns
    the names of the modules that were patched. A maintainer editing the reference writes instead, in modules/Extension.py:
    `from mvxnet_makise_b200.voxelize import cpp`."""
    from .voxelize import cpp
    patched = []
    for name in ('modules.Extension', 'modules.data.Preprocessing', 'modules.Calc', 'modules.augment.Augment'):
        mod = sys.modules.get(name)
        if mod is not None and hasattr(mod, 'cpp'):
            mod.cpp = cpp
            patched.append(name)
    return patched
