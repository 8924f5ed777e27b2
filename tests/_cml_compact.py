"""fp64 restatement of the compact backward of `CML.conv1` = CRB3d(128, 64, 3, (2,1,1), (1,1,1)) (voxelnet/Pipe.py:31-43,
Blocks.py CRB3d; oracle.pointpath_oracle.cml_conv1) that csrc/sparse_conv.cu implements, in plain torch on the CPU.

Per frame, with R output positions, the active set A (positions with a non-empty neighbour), background y = relu(b), the
batch-statistic mean m / rstd r over all R positions and g = dLoss/d out:
    S1 = sum_all g, A1 = sum_A g, A2 = sum_A g y,  S2 = r (A2 + relu(b) (S1 - A1) - m S1)
    dpre_p = r (g_p - S1/R - z_p S2/R) [y_p > 0] on A;  db = sum_A dpre + [b > 0] r ((S1 - A1) - n_bg S1/R - z_bg n_bg S2/R)
    D[v][t][o] = dpre[pos(v, t)][o];  d_vfeat = sum_t D[:, t] W_t,  dW_t = D[:, t]^T vfeat
tests/test_oracle_cml_backward.py pins these against dense fp64 autograd of the reference ops; the GPU tests evaluate them
on the CUDA forward's own saved activations (same ReLU decisions)."""
from __future__ import annotations

import torch
import torch.nn.functional as F

F64 = torch.float64


def out_depth(nz: int) -> int:
    return (nz + 2 - 3) // 2 + 1


def dense_grid(vfeat, coords, grid_shape):
    """(1, 128, nz, nx, ny) grid of VoxelNet.reindex: coords (N, 3) [ix, iy, iz]"""
    nz, nx, ny = grid_shape
    g = torch.zeros((1, vfeat.shape[1], nz, nx, ny), dtype=vfeat.dtype)
    g[0][:, coords[:, 2], coords[:, 0], coords[:, 1]] = vfeat.t()
    return g


def activations(vfeat, coords, grid_shape, w, b):
    """relu(conv) (64, oz, nx, ny) and the active mask (oz, nx, ny) of the dense route, in fp64"""
    grid = dense_grid(vfeat.to(F64), coords, grid_shape)
    y = F.relu(F.conv3d(grid, w.to(F64), b.to(F64), stride=(2, 1, 1), padding=(1, 1, 1)))[0]
    occ = torch.zeros((1, 1) + tuple(grid_shape), dtype=F64)
    occ[0, 0, coords[:, 2], coords[:, 0], coords[:, 1]] = 1.0
    act = F.conv3d(occ, torch.ones((1, 1, 3, 3, 3), dtype=F64), stride=(2, 1, 1), padding=(1, 1, 1))[0, 0] > 0
    return y, act


def tap_positions(coords, grid_shape):
    """(N, 27) flat output position each voxel reaches through each tap (t = (kz * 3 + kx) * 3 + ky), -1 where none"""
    nz, nx, ny = grid_shape
    oz = out_depth(nz)
    ix, iy, iz = coords[:, 0:1], coords[:, 1:2], coords[:, 2:3]
    t = torch.arange(27)
    kz, kx, ky = t // 9, (t // 3) % 3, t % 3
    oz2, ox, oy = iz + 1 - kz, ix + 1 - kx, iy + 1 - ky
    ok = (oz2 >= 0) & (oz2 % 2 == 0) & (oz2 // 2 < oz) & (ox >= 0) & (ox < nx) & (oy >= 0) & (oy < ny)
    pos = ((oz2 // 2) * nx + ox) * ny + oy
    return torch.where(ok, pos, torch.full_like(pos, -1))


def cml_conv1_backward(vfeat, coords, grid_shape, w, b, g, y, act, eps=1e-6):
    """vfeat (N, 128), coords (N, 3) long [ix, iy, iz], w (64, 128, 3, 3, 3), b (64), g (64, oz, nx, ny) = dLoss/d out;
    y (64, oz, nx, ny) relu(conv), read on the active positions only; act (oz, nx, ny) bool.
    Returns (d_vfeat (N, 128), d_w (64, 128, 3, 3, 3), d_b (64)) in fp64."""
    vfeat, w, b = vfeat.to(F64), w.to(F64), b.to(F64)
    g = g.to(F64).reshape(64, -1)
    R = g.shape[1]
    a = act.reshape(-1)
    ya = y.to(F64).reshape(64, -1)[:, a]
    ga = g[:, a]
    n_bg = R - int(a.sum())
    bg = b.clamp_min(0)
    m = (ya.sum(1) + n_bg * bg) / R
    var = ((ya * ya).sum(1) + n_bg * bg * bg) / R - m * m
    r = 1.0 / torch.sqrt(var.clamp_min(0) + eps)
    S1, A1, A2 = g.sum(1), ga.sum(1), (ga * ya).sum(1)
    S2 = r * (A2 + bg * (S1 - A1) - m * S1)
    z = (ya - m[:, None]) * r[:, None]
    dpre = r[:, None] * (ga - (S1 / R)[:, None] - z * (S2 / R)[:, None]) * (ya > 0)
    z_bg = (bg - m) * r
    d_b = dpre.sum(1) + (b > 0) * r * ((S1 - A1) - n_bg * S1 / R - z_bg * n_bg * S2 / R)
    full = torch.zeros((R + 1, 64), dtype=F64)          # last row: "no position"
    full[torch.nonzero(a)[:, 0]] = dpre.t()
    pos = tap_positions(coords, grid_shape)
    D = full[torch.where(pos >= 0, pos, torch.full_like(pos, R))]          # (N, 27, 64)
    Wt = w.reshape(64, 128, 27)
    d_vfeat = torch.einsum('nto,oct->nc', D, Wt)
    d_w = torch.einsum('nto,nc->oct', D, vfeat).reshape(64, 128, 3, 3, 3)
    return d_vfeat, d_w, d_b
