"""TEST INFRASTRUCTURE: the checker side of the per-module backward (csrc/module_backward.cu, the gather adjoint of
csrc/map_backward.cu), in plain torch fp64 on the CPU. These are the dense formulas the CUDA entries implement, written out so
that the tests can pin them to torch autograd through the oracle's restatement of the reference modules
(oracle/pointpath_oracle.py: crb, vfe, voxel_features, feature_mapping, reindex) and evaluate them on the CUDA forward's own
raw outputs and BatchNorm sums.
  * `bn_relu_backward`: batch-statistic BatchNorm + ReLU backward over all R rows (multiplicity 1);
  * `route_max`: the max over T routes its gradient to the FIRST slot that attains the maximum;
  * `layer_backward`: one FCN / VFE / last-FCN-max layer, dx, dW, db from dy in the forward's output layout;
  * `gather_adjoint`: dLoss/d maps of featureMaping's 4-corner sample from dLoss/d out."""
from __future__ import annotations

import torch

F64 = torch.float64


def bn_relu_backward(y_raw, dz, eps: float = 1e-6, stats=None):
    """dpre = rstd (dz - S1/R - z S2/R) [y > 0] with S1 = sum dz, S2 = sum dz z, z = (y - mean) rstd; y_raw, dz (R, C).
    stats: optional (C, 2) sums (sum y, sum y^2) the mean and variance come from (the CUDA forward's fp64 sums); default: y_raw's."""
    y = torch.as_tensor(y_raw).to(F64)
    dz = torch.as_tensor(dz).to(F64)
    R = y.shape[0]
    if stats is None:
        stats = torch.stack([y.sum(0), (y * y).sum(0)], 1)
    stats = torch.as_tensor(stats).to(F64)
    mean = stats[:, 0] / R
    var = (stats[:, 1] / R - mean * mean).clamp_min(0)
    rstd = 1.0 / torch.sqrt(var + eps)
    z = (y - mean) * rstd
    s1, s2 = dz.sum(0), (dz * z).sum(0)
    return rstd * (dz - s1 / R - z * s2 / R) * (y > 0)


def route_max(y_raw, d_max):
    """y_raw (V, T, C), d_max (V, C) -> (V, T, C): d_max at the first slot attaining max_t y_raw[v, t, c], 0 elsewhere."""
    y = torch.as_tensor(y_raw)
    V, T, C = y.shape
    first = (y == y.max(dim=1, keepdim=True)[0]).to(torch.int64).argmax(dim=1)   # argmax of a 0/1 tensor: the first 1
    out = torch.zeros((V, T, C), dtype=F64)
    out.scatter_(1, first[:, None, :], torch.as_tensor(d_max).to(F64)[:, None, :])
    return out


def layer_backward(kind: str, x, w, y_raw, dy, T: int = 1, eps: float = 1e-6, stats=None):
    """dx (R, Cin), dW (Cout, Cin), db (Cout) of one layer. x (R, Cin), w (Cout, Cin), y_raw (R, Cout) = relu(x W^T + b) of the
    forward, dy in the forward's output layout: (R, Cout) 'fcn', (R, 2 Cout) 'vfe' = [pointwise | max tiled over T], (R/T, Cout)
    'fcn_max'."""
    x = torch.as_tensor(x).to(F64)
    w = torch.as_tensor(w).to(F64).reshape(w.shape[0], -1)
    y = torch.as_tensor(y_raw)
    dy = torch.as_tensor(dy).to(F64)
    R, C = y.shape
    if kind == 'fcn':
        dz = dy
    elif kind == 'vfe':
        d_max = dy[:, C:].reshape(R // T, T, C).sum(1)
        dz = dy[:, :C] + route_max(y.reshape(R // T, T, C), d_max).reshape(R, C)
    else:
        dz = route_max(y.reshape(R // T, T, C), dy).reshape(R, C)
    dpre = bn_relu_backward(y, dz, eps, stats)
    return dpre @ w, dpre.t() @ x, dpre.sum(0)


def layer_forward(kind: str, x, w, b, T: int = 1, eps: float = 1e-6):
    """fp64 forward of the same layer on (R, Cin) rows: (output in the layout above, y_raw)"""
    x = torch.as_tensor(x).to(F64)
    y = torch.relu(x @ torch.as_tensor(w).to(F64).reshape(w.shape[0], -1).t() + torch.as_tensor(b).to(F64))
    R, C = y.shape
    z = (y - y.mean(0)) / torch.sqrt(y.var(0, unbiased=False) + eps)
    if kind == 'fcn':
        return z, y
    m = z.reshape(R // T, T, C).max(1)[0]
    if kind == 'vfe':
        return torch.cat([z, m.repeat_interleave(T, 0)], 1), y
    return m, y


def gather_adjoint(voxels9, d_out, map_hw, imsize_hw, eps: float = 1e-6):
    """dLoss/d maps [(C, H_l, W_l)] fp64 of featureMaping for ONE frame: voxels9 (..., 9) fp32 as the forward left them, d_out
    (..., 3C). Corner indices and fractions in fp32 like the forward, weights multiplied in fp64; pad slots (x == y == z == 0) and
    corners outside the H x W map (the zero pad row / column of Pipe.py:47-48) contribute nothing."""
    v = torch.as_tensor(voxels9).reshape(-1, 9)
    d = torch.as_tensor(d_out).to(F64).reshape(v.shape[0], -1)
    C = d.shape[1] // 3
    real = ~torch.all(v[:, :3] == 0, dim=1)
    proj, d = v[real][:, 7:9].to(torch.float32), d[real]
    out = []
    for l, (H, W) in enumerate(map_hw):
        rs = torch.tensor(list(imsize_hw), dtype=torch.float32) / torch.tensor([float(H), float(W)], dtype=torch.float32)
        q = proj / rs - eps
        i = q.long()
        a, b = (q[:, 0] - i[:, 0]).to(F64), (q[:, 1] - i[:, 1]).to(F64)
        a_, b_ = (1 - (q[:, 0] - i[:, 0])).to(F64), (1 - (q[:, 1] - i[:, 1])).to(F64)
        g = torch.zeros(H * W, C, dtype=F64)
        dl = d[:, C * l:C * (l + 1)]
        for dy, dx, wgt in ((0, 0, a * b), (1, 0, a_ * b), (0, 1, a * b_), (1, 1, a_ * b_)):
            y, x = i[:, 0] + dy, i[:, 1] + dx
            ok = (y >= 0) & (y < H) & (x >= 0) & (x < W)
            g.index_add_(0, (y * W + x)[ok], dl[ok] * wgt[ok, None])
        out.append(g.t().reshape(C, H, W))
    return out
