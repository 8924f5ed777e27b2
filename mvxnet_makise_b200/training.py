"""Training-mode step of the hot path (BASELINE.json configs[3]): forward_train -> backward -> ONE all-reduce of the flat
gradient bucket over the frame-sharded ranks -> AdamW on the flat parameter vector.

What it stands in for in the reference (train.py:60-66, 130-166): `AdamW(lr=1e-3, eps=1e-6)` over the model parameters and
`loss.backward()`; here only the 726 880 parameters of the 8 hot-path layers (SURVEY.md §8b) are owned - the CML / RPN /
loss that produce dLoss/d(voxel features) are outside the path, so the caller passes that gradient in
(`d_vfeat` (B, cap, 128) or `d_grid` (B,128,nz,nx,ny)).

The flat vector has the checkpoint layout ([weight (Cout,Cin) | bias (Cout)] per layer, `PointPath.grad_layout()`), so
gradients come out of the CUDA backward already packed: no per-parameter pack/unpack, one NCCL message of 2.9 MB."""
from __future__ import annotations

from typing import Dict, Sequence

import numpy as np
import torch
import torch.distributed as dist

from . import synth


class FlatAdamW:
    """AdamW (train.py:64: lr 1e-3, eps 1e-6, torch defaults otherwise) on ONE flat fp32 parameter vector whose gradient
    arrives as one flat bucket; `reduce_and_step` sums the bucket over the ranks (one collective), divides by the global
    number of frames and applies the update. Device-agnostic (NCCL on the GPUs, gloo in the CPU tests)."""

    def __init__(self, params: torch.Tensor, lr: float = 1e-3, eps: float = 1e-6, betas: Sequence[float] = (0.9, 0.999),
                 weight_decay: float = 1e-2):
        self.params = params
        self.m = torch.zeros_like(params)
        self.v = torch.zeros_like(params)
        self.lr, self.eps, self.betas, self.weight_decay = lr, eps, tuple(betas), weight_decay
        self.t = 0

    def reduce_and_step(self, grad: torch.Tensor, local_frames: int, global_frames: int | None = None):
        """`grad` is this rank's bucket with ONE spare element at the end (`numel() == params.numel() + 1`) or exactly the
        parameter count. With the spare element the number of frames travels in the same message, so ragged shards (5 frames
        on 2 ranks = 3 + 2) divide by the same global count on every rank; without it `global_frames` is mandatory when
        world > 1 (a per-rank guess `local_frames * world` would make the replicas diverge silently)."""
        world = dist.get_world_size() if dist.is_initialized() else 1
        n = self.params.numel()
        carries_count = grad.numel() == n + 1
        assert carries_count or grad.numel() == n
        if world > 1 and not carries_count and global_frames is None:
            raise ValueError('global_frames is required when the bucket has no frame-count slot (ragged shards would diverge)')
        if carries_count:
            grad[n] = float(local_frames)
        if world > 1:
            dist.all_reduce(grad, op=dist.ReduceOp.SUM)          # NCCL over NVLink: the path's only collective
        if global_frames is None:
            # the count rides in the bucket; the division stays on the device (no host read-back in the step)
            denom = grad[n:n + 1] if carries_count else torch.full((1,), float(local_frames), device=grad.device)
        else:
            denom = torch.full((1,), float(global_frames), device=grad.device)
        grad = grad[:n]
        grad.div_(denom)                                         # the reference optimises a per-frame loss
        b1, b2 = self.betas
        self.t += 1
        self.params.mul_(1.0 - self.lr * self.weight_decay)
        self.m.mul_(b1).add_(grad, alpha=1.0 - b1)
        self.v.mul_(b2).addcmul_(grad, grad, value=1.0 - b2)
        bc1, bc2 = 1.0 - b1 ** self.t, 1.0 - b2 ** self.t
        denom = (self.v / bc2).sqrt_().add_(self.eps)
        self.params.addcdiv_(self.m, denom, value=-self.lr / bc1)


class HotPathTrainer:
    def __init__(self, state_dict: Dict, grid: synth.GridSpec = synth.KITTI_GRID, lr: float = 1e-3, eps: float = 1e-6,
                 betas: Sequence[float] = (0.9, 0.999), weight_decay: float = 1e-2, device='cuda'):
        from ._lib import lib                 # needs the CUDA library; FlatAdamW above does not
        from .pipeline import PointPath
        self.path = PointPath(state_dict, grid, device=device)
        dev = self.path.device
        n = int(lib.mvx_grad_floats())
        self.params = torch.empty(n, dtype=torch.float32, device=dev)
        views = self.path.grads(self.params)
        for name, v in views.items():
            t = torch.as_tensor(np.asarray(state_dict[name])) if not isinstance(state_dict[name], torch.Tensor) else state_dict[name]
            v.copy_(t.detach().reshape(v.shape))
        self._param_views = list(views.values())      # checkpoint order: what PointPath.load_parameters takes
        self.bucket = torch.zeros(n + 1, dtype=torch.float32, device=dev)   # gradients + one slot for the frame count
        self.grad = self.bucket[:n]                                          # what the CUDA backward fills
        self.opt = FlatAdamW(self.params, lr, eps, betas, weight_decay)

    def state_dict(self) -> Dict[str, torch.Tensor]:
        return {name: v.clone() for name, v in self.path.grads(self.params).items()}

    def _push_weights(self):
        """flat parameters -> the W^T (Cin_pad, Cout) / bias tensors the kernels read (in place: pointers stay valid)"""
        self.path.load_parameters(self._param_views)

    def step(self, points, offsets, calib32, maps, d_vfeat=None, d_grid=None, global_frames: int | None = None,
             want_grid: bool = True):
        """One optimisation step on this rank's frames. Returns (grid, counts) of the forward."""
        grid, counts = self.path.forward_train(points, offsets, calib32, maps, want_grid)
        self.path.backward(d_vfeat=d_vfeat, d_grid=d_grid, grad_flat=self.grad, accumulate=False)
        self.opt.reduce_and_step(self.bucket, len(offsets) - 1, global_frames)
        self._push_weights()
        return grid, counts
