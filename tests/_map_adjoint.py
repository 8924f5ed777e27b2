"""TEST INFRASTRUCTURE: the checker side of the gradient into the FPN maps (csrc/map_backward.cu), in plain torch on the CPU,
built on the oracle's restatement of the reference chain (oracle/pointpath_oracle.py) and its compact training formulas
(oracle/compact_backward.py), which it uses unchanged.
  * `map_adjoint`: the compact adjoint of featureMaping's 4-corner gather (Pipe.py:62-75), dLoss/d maps from fcn1's dpre;
  * `compact_dpre1`: fcn1's dpre from the compact formulas;
  * `dense_backward`: fp64 (or fp32) autograd through the dense chain featureMaping -> fusion -> VFE -> FCN -> max with the
    maps as leaves (an unfrozen image backbone), from a point cloud (`frame`) or a dense (N, T, 9) voxel tensor."""
from __future__ import annotations

import numpy as np
import torch

from oracle import compact_backward as CB
from oracle import pointpath_oracle as O

F64 = torch.float64
FCN1 = CB.LAYERS[0]


def compact_dpre1(st, aux, dOut, row_v):
    """fcn1's dpre (K+1, 768) of the compact formulas. `compact_backward` returns fcn1's weight gradient dpre1ᵀ·x; evaluated with
    x = I (the only use of st[0]['x']) that gradient is dpre1ᵀ itself."""
    n = st[0]['x'].shape[0]
    st1 = dict(st)
    st1[0] = dict(st[0], x=torch.eye(n, dtype=F64))
    return CB.compact_backward(st1, aux, dOut, row_v)[FCN1 + '.weight'].t()


def map_adjoint(dpre1, W1, proj, real, map_hw, imsize_hw, eps: float = 1e-6):
    """dLoss/d FPN maps of ONE frame: the adjoint of featureMaping's 4-corner gather applied to dA1 = dpre1 W1.
    dpre1 (R,768) fcn1's dpre of the compact rows; W1 (768,768) fcn1's weight; proj (R,2) fp32 (row, col) projections; real (R,)
    bool: rows that sample the maps (kept points away from the origin; False for the frame's pad row). The corner indices and
    the fractional parts a, b, 1-a, 1-b are evaluated in fp32 as the forward does; the weights a*b, (1-a)*b, a*(1-b), (1-a)*(1-b)
    are then multiplied in fp64, as autograd multiplies them into fp64 maps. Corners outside the H x W map (the zero pad row /
    column of Pipe.py:47-48) receive nothing. Returns [(256, H_l, W_l)] fp64."""
    dA1 = torch.as_tensor(dpre1).to(F64) @ torch.as_tensor(W1).to(F64).reshape(768, 768)
    proj = torch.as_tensor(proj).to(torch.float32)[real]
    dA1 = dA1[real]
    out = []
    for l, (H, W) in enumerate(map_hw):
        rs = torch.tensor(list(imsize_hw), dtype=torch.float32) / torch.tensor([float(H), float(W)], dtype=torch.float32)
        q = proj / rs - eps
        i = q.long()
        a, b = q[:, 0] - i[:, 0], q[:, 1] - i[:, 1]
        a_, b_ = (1 - a).to(F64), (1 - b).to(F64)
        a, b = a.to(F64), b.to(F64)
        g = torch.zeros(H * W, 256, dtype=F64)
        dA = dA1[:, 256 * l:256 * (l + 1)]
        for dy, dx, w in ((0, 0, a * b), (1, 0, a_ * b), (0, 1, a * b_), (1, 1, a_ * b_)):
            y, x = i[:, 0] + dy, i[:, 1] + dx
            ok = (y >= 0) & (y < H) & (x >= 0) & (x < W)
            g.index_add_(0, (y * W + x)[ok], dA[ok] * w[ok, None])
        out.append(g.t().reshape(256, H, W))
    return out


def dense_backward(voxels: torch.Tensor, fpn_maps, sd_np, imsize_hw, d_vfeat, eps: float = 1e-6, dtype: torch.dtype = F64):
    """What `loss.backward()` leaves in the FPN maps' .grad for ONE frame when the gradient arriving at the voxel features is
    d_vfeat (N,128): autograd through O.feature_mapping -> O.fusion -> concat -> O.voxel_features with the maps (and the 16
    parameters) as leaves in `dtype`. voxels: the dense (N,T,9) fp32 tensor of `group` + train.py:125 (mutated like featureMaping
    does). Returns [(256, H_l, W_l)]."""
    params = {k: torch.from_numpy(np.asarray(v)).to(dtype).requires_grad_(True) for k, v in sd_np.items()}
    feats = [torch.from_numpy(np.asarray(m)).to(dtype).requires_grad_(True) for m in fpn_maps]
    im768 = O.feature_mapping(voxels, feats, torch.Tensor(list(imsize_hw)), eps)
    im16 = O.fusion(im768[None].to(dtype), params, eps)
    x23 = torch.concat([voxels[None][..., :7].to(dtype), im16], dim=-1)
    vfeat = O.voxel_features(x23, params, eps)
    (vfeat * torch.from_numpy(np.asarray(d_vfeat)).to(dtype)).sum().backward()
    return [f.grad[0] for f in feats]


def dense_backward_frame(pcd4, calib_np, fpn_maps, sd_np, grid, imsize_hw, d_vfeat, eps: float = 1e-6, dtype: torch.dtype = F64):
    """`dense_backward` from a raw (P,4) cloud: projection and `group` as in O.backward_frame"""
    voxel9, _ = O.group(O.points_with_proj(pcd4, calib_np), grid.velorange, grid.voxelsize, grid.T)
    return dense_backward(torch.Tensor(voxel9), fpn_maps, sd_np, imsize_hw, d_vfeat, eps, dtype)
