"""Dev tool (GPU): cost of the sparse CML.conv1 hand-off (SURVEY.md §8f rank 2) at the headline size, next to the dense route
(grid fill + torch/cuDNN Conv3d + BatchNorm3d on the dense grid, what the reference does after the path)."""
import os, sys
import numpy as np, torch
import torch.nn.functional as F
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mvxnet_makise_b200 import synth
from mvxnet_makise_b200.pipeline import PointPath
from mvxnet_makise_b200.modules import pack_calib

B, P = 8, 120_000
dev = torch.device('cuda')
frames = [synth.make_points(f, P) for f in range(B)]
offsets = np.concatenate([[0], np.cumsum([p.shape[0] for p in frames])]).tolist()
points = torch.from_numpy(np.concatenate(frames, 0)).to(dev)
calib = torch.stack([pack_calib(synth.kitti_calib()) for _ in range(B)]).to(dev)
g = torch.Generator(device=dev).manual_seed(1)
maps = [torch.randn((B, 256, h, w), generator=g, device=dev) for (h, w) in synth.fpn_shapes()]
w = torch.randn((64, 128, 3, 3, 3), generator=g, device=dev) / (128 * 27) ** 0.5
b = torch.randn(64, generator=g, device=dev) * 0.1
path = PointPath(synth.make_weights(0), synth.KITTI_GRID, device=dev)


def timed(fn, n=10):
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


t_path_grid = timed(lambda: path.forward_device(points, offsets, calib, maps, True))
t_path_nogrid = timed(lambda: path.forward_device(points, offsets, calib, maps, False))
t_sparse = timed(lambda: (path.forward_device(points, offsets, calib, maps, False), path.cml_conv1(w, b)))
grid, _ = path.forward_device(points, offsets, calib, maps, True)


def dense_conv1():
    outs = []
    for f in range(B):                                   # the reference runs CML per frame (batch 1)
        y = F.relu(F.conv3d(grid[f:f + 1], w, b, stride=(2, 1, 1), padding=(1, 1, 1)))
        outs.append(F.batch_norm(y, None, None, None, None, True, 0.0, 1e-6))
    return outs


torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False
t_dense = timed(dense_conv1, 3)
out = path.cml_conv1(w, b)
ref = torch.cat(dense_conv1())
err = ((out - ref).abs().max() / ref.abs().max()).item()
print(f'path with dense grid {t_path_grid:.3f} ms | path without grid {t_path_nogrid:.3f} ms | path + sparse conv1 {t_sparse:.3f} ms '
      f'(sparse conv1 alone {t_sparse - t_path_nogrid:.3f} ms) | dense route: grid fill {t_path_grid - t_path_nogrid:.3f} ms + torch Conv3d/BN3d fp32 '
      f'{t_dense:.3f} ms | sparse vs torch dense rel diff {err:.2e}  (batch {B})')


# ---- training leg: forward + backward of the hot path and conv1, dense route vs sparse route ------------------------------
import subprocess
card = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True).stdout.strip()
go = out.shape[2] * out.shape[3] * out.shape[4]
d_out = torch.randn(out.shape, generator=g, device=dev)


def dense_train():
    grid_t, _ = path.forward_train(points, offsets, calib, maps, want_grid=True, shuffle=False)
    gr = grid_t.detach().requires_grad_(True)
    wd, bd = w.detach().requires_grad_(True), b.detach().requires_grad_(True)
    for f in range(B):
        y = F.relu(F.conv3d(gr[f:f + 1], wd, bd, stride=(2, 1, 1), padding=(1, 1, 1)))
        (F.batch_norm(y, None, None, None, None, True, 0.0, 1e-6) * d_out[f:f + 1]).sum().backward()
    path.backward(d_grid=gr.grad)


def sparse_train():
    path.forward_train(points, offsets, calib, maps, want_grid=False, shuffle=False)
    path.cml_conv1(w, b)
    d_vfeat, _, _ = path.cml_conv1_backward(d_out, w, b)
    path.backward(d_vfeat=d_vfeat)


def sparse_train_fwd():
    path.forward_train(points, offsets, calib, maps, want_grid=False, shuffle=False)
    path.cml_conv1(w, b)


t_dense_train = {}
for tf32 in (False, True):
    torch.backends.cudnn.allow_tf32 = tf32
    torch.backends.cuda.matmul.allow_tf32 = tf32
    t_dense_train[tf32] = timed(dense_train, 3)
t_sparse_train = timed(sparse_train)
t_sparse_fwd = timed(sparse_train_fwd)
t_conv1_bwd = timed(lambda: path.cml_conv1_backward(d_out, w, b))
t_conv1_bwd_nodv = timed(lambda: path.cml_conv1_backward(d_out, w, b, want_d_vfeat=False))
n_vox = path.counts[:, 0].sum().item()
n_act = path.cml_saved()['act_count'].sum().item()
print(f'training, batch {B} x {P} points, {card}: dense route (forward_train with grid, torch Conv3d/BN3d forward + backward, '
      f'path.backward(d_grid)) {t_dense_train[False]:.3f} ms TF32 off / {t_dense_train[True]:.3f} ms TF32 on | sparse route '
      f'(forward_train without grid, sparse conv1 forward + backward, path.backward(d_vfeat)) {t_sparse_train:.3f} ms | '
      f'sparse conv1 backward alone {t_conv1_bwd:.3f} ms ({t_conv1_bwd_nodv:.3f} ms without d_vfeat) | voxels {n_vox}, active positions {n_act}')

# each kernel of the sparse backward alone: device times from torch.profiler (a run of its own), bytes from shapes
from torch.profiler import profile, ProfilerActivity
for _ in range(2):
    path.cml_conv1_backward(d_out, w, b)
torch.cuda.synchronize()
reps = 5
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(reps):
        path.cml_conv1_backward(d_out, w, b)
    torch.cuda.synchronize()
cap = path.cap
compulsory = {   # bytes each kernel must move at least (reads + writes), from the shapes of this batch
    'scb_reduce_kernel': B * 64 * go * 4 + 2 * n_act * 64 * 4 + B * go * 4,
    'scb_dpre_kernel': 3 * n_act * 64 * 4,
    'scb_tap_gather_kernel': n_vox * 1792 * 4 + n_vox * 16 + n_act * 64 * 4,
    'dw_tc_kernel': n_vox * (1792 + 128) * 4,
    'tc_layer_kernel': n_vox * (1792 + 128) * 4,
}
rows = {}
for e in prof.key_averages():
    if e.device_type.name == 'CUDA' or getattr(e, 'self_device_time_total', 0) > 0:
        t = getattr(e, 'self_device_time_total', None) or getattr(e, 'self_cuda_time_total', 0)
        rows[e.key] = rows.get(e.key, 0) + t / reps / 1000.0
for name, ms in sorted(rows.items(), key=lambda kv: -kv[1]):
    key = next((k for k in compulsory if k in name), None)
    bw = f' | {compulsory[key] / (ms * 1e-3) / 1e9:.0f} GB/s of compulsory bytes' if key and ms > 0 else ''
    print(f'  {ms:8.3f} ms  {name[:110]}{bw}')
