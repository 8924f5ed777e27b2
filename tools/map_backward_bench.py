"""Dev tool (GPU): cost of the gradient into the FPN maps (mvx_pointpath_backward_maps, csrc/map_backward.cu) at the headline
size, 8 x 120 000-point KITTI frames with the KITTI FPN shapes, through the dense-voxel entry the drop-in uses:
  * the map backward alone and with the path backward it follows, in CUDA events;
  * its parts (pixel CSR, dZ, GEMM): device times of each kernel from torch.profiler, in a run of their own;
  * bytes: the compulsory ones of the dZ pass (dpre1 read once, dZ written once) and the GEMM's FLOPs;
  * like for like on the same GPU: torch-eager fp32 autograd of the oracle's feature_mapping (Pipe.py:23-82) into the maps,
    per frame on the reference's dense (N, T, 768) tensor, from a given gradient of its output.
Prints the card name and its power limit."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mvxnet_makise_b200 import _lib, synth
from mvxnet_makise_b200.pipeline import PointPath
from oracle import pointpath_oracle as O

B, P = 8, 120_000
dev = torch.device('cuda')
G = synth.KITTI_GRID
card = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True,
                      text=True).stdout.strip().splitlines()[0]
vs, ids = [], []
for f in range(B):
    voxel, idx = O.group(O.points_with_proj(synth.make_points(f, P), synth.kitti_calib()), G.velorange, G.voxelsize, G.T)
    vs.append(torch.as_tensor(np.asarray(voxel), dtype=torch.float32).to(dev))
    ids.append(torch.as_tensor(np.concatenate([np.full((idx.shape[0], 1), f), idx], 1), dtype=torch.int64).to(dev))
g = torch.Generator(device=dev).manual_seed(1)
maps = [torch.randn((B, 256, h, w), generator=g, device=dev) for (h, w) in synth.fpn_shapes()]
path = PointPath(synth.make_weights(0), G, device=dev)
path.forward_voxels(vs, ids, maps, want_grid=False, train=True)
dv = torch.randn((B, path.cap, 128), generator=g, device=dev)
d_maps = [torch.empty_like(m) for m in maps]
path.backward(d_vfeat=dv, d_maps=d_maps)
counts = path.counts.cpu()
K = int(counts[:, 1].sum())
px = sum(h * w for h, w in synth.fpn_shapes())


def entry():
    a = path._record.args
    out = (ctypes.c_void_p * 3)(*[t.data_ptr() for t in d_maps])
    _lib.check(_lib.lib.mvx_pointpath_backward_maps(ctypes.byref(a), path._bws.data_ptr(), path._bws.numel(), out,
                                                    path._map_bws.data_ptr(), path._map_bws.numel()), 'backward_maps')


def timed(fn, n=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


t_entry = timed(entry)
t_bwd = timed(lambda: path.backward(d_vfeat=dv))
t_both = timed(lambda: path.backward(d_vfeat=dv, d_maps=d_maps))
print(f'{card} | batch {B} x {P} points, {K} kept rows, {B * px} map pixels')
print(f'map backward (mvx_pointpath_backward_maps) {t_entry:.3f} ms | path backward (mvx_pointpath_backward) {t_bwd:.3f} ms | '
      f'both through PointPath.backward(d_maps=...) {t_both:.3f} ms')

# parts: device time of every kernel of the entry, torch.profiler in a run of its own
from torch.profiler import profile, ProfilerActivity
reps = 5
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(reps):
        entry()
    torch.cuda.synchronize()
parts = {'CSR': ('mb_hist', 'mb_scan', 'mb_scatter', 'mb_rank', 'Memset'), 'dZ': ('mb_dz',),
         'GEMM': ('transpose_w', 'pack_weights', 'tc_layer_kernel')}
rows, total = {}, {k: 0.0 for k in parts}
for e in prof.key_averages():
    t = getattr(e, 'self_device_time_total', None) or getattr(e, 'self_cuda_time_total', 0)
    if t <= 0:
        continue
    ms = t / reps / 1000.0
    rows[e.key] = ms
    for k, names in parts.items():
        if any(n in e.key for n in names):
            total[k] += ms
compulsory = K * 768 * 4 + B * px * 768 * 4          # dpre1 read once + dZ written once
flop = 2.0 * B * px * 768 * 256
print(f'parts (profiler device time): CSR {total["CSR"]:.3f} ms | dZ {total["dZ"]:.3f} ms '
      f'({compulsory / 1e9:.2f} GB compulsory -> {compulsory / (total["dZ"] * 1e-3) / 1e12:.2f} TB/s effective) | '
      f'GEMM {total["GEMM"]:.3f} ms ({flop / 1e9:.1f} GFLOP 3xTF32 -> {flop / (total["GEMM"] * 1e-3) / 1e12:.1f} TFLOP/s effective)')
for name, ms in sorted(rows.items(), key=lambda kv: -kv[1]):
    print(f'  {ms:8.3f} ms  {name[:120]}')

# like for like: torch-eager fp32 autograd of feature_mapping into the maps, per frame (the reference runs batch 1)
imsize = torch.tensor(synth.KITTI_IMSIZE_HW, dtype=torch.float32, device=dev)
t_torch, rows_dense = 0.0, 0
for f in range(B):
    leaves = [m[f:f + 1].detach().clone().requires_grad_(True) for m in maps]
    im = O.feature_mapping(vs[f].clone(), leaves, imsize)
    dA = torch.randn(im.shape, generator=g, device=dev)
    rows_dense += im.shape[0] * im.shape[1]
    t_torch += timed(lambda: torch.autograd.grad(im, leaves, dA, retain_graph=True), n=3)
    del im, dA, leaves
    torch.cuda.empty_cache()
print(f'torch eager fp32 autograd of feature_mapping into the maps, {B} frames one at a time ({rows_dense} dense rows, '
      f'from d feature_mapping output): {t_torch:.3f} ms | ours from dpre1 (incl. the W1 product) {t_entry:.3f} ms')
