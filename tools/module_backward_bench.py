"""Dev tool (GPU): forward + backward of the per-module drop-ins (mvxnet_makise_b200/modules.py) on ONE full-size synthetic KITTI
frame (120 000 points, about 21 k voxels, R = N x 35 dense rows, KITTI FPN shapes), in CUDA events, against torch-eager fp32
autograd of the oracle's reference modules (oracle/pointpath_oracle.py) on the same GPU and the same inputs:
  * featureMaping (gradient into the three maps), ImageFeatureFusion, SVFE, the last FCN + max over T, reindex;
  * every input that can take a gradient requires one (x, the 16 parameters, the maps), so each backward computes dx too;
  * FLOPs (2 R Cin Cout per layer forward, twice that backward: dW and dx) and compulsory bytes (each layer's input, output and
    raw output once forward; dy, raw output, input and dx once backward) come from the shapes below.
Prints the card name and its power limit from the same run; writes the report to the path given as the first argument."""
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mvxnet_makise_b200 import modules as M, synth
from oracle import pointpath_oracle as O

dev = torch.device('cuda')
G = synth.KITTI_GRID
IMSIZE = torch.Tensor(list(synth.KITTI_IMSIZE_HW))
card = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True,
                      text=True).stdout.strip().splitlines()[0]
voxel, uidx = O.group(O.points_with_proj(synth.make_points(0, 120_000), synth.kitti_calib()), G.velorange, G.voxelsize, G.T)
vox = torch.as_tensor(np.asarray(voxel), dtype=torch.float32).to(dev)
idx = torch.as_tensor(np.concatenate([np.zeros((uidx.shape[0], 1)), uidx], 1), dtype=torch.int64).to(dev)
N, T = vox.shape[:2]
R = N * T
g = torch.Generator(device=dev).manual_seed(1)
maps = [torch.randn((1, 256, h, w), generator=g, device=dev) for (h, w) in synth.fpn_shapes()]
sd_np = synth.make_weights(0)
sd = {k: torch.from_numpy(np.asarray(v)).to(dev) for k, v in sd_np.items()}

fusion, head = M.ImageFeatureFusion().to(dev), M.VoxelNetHead().to(dev)
fusion.load_state_dict({k[len('head.fusion.'):]: v for k, v in sd.items() if k.startswith('head.fusion.')})
head.load_state_dict({k[len('backbone.'):]: v for k, v in sd.items() if k.startswith('backbone.')})
params = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
with torch.no_grad():
    vox_after = vox.clone()
    im768 = M.featureMaping([vox_after], maps, None, IMSIZE)[0]
    im16 = fusion(im768[None])
    x23 = torch.cat([vox_after[None][..., :7], im16], -1)
    x128 = head.svfe(x23)
    vfeat = head.voxel_features(x23)


def leaf(t):
    return t.detach().clone().requires_grad_(True)


def run_ours(name):
    if name == 'featureMaping':
        ms = [leaf(m) for m in maps]
        out = M.featureMaping([vox.clone()], ms, None, IMSIZE)[0]
    elif name == 'ImageFeatureFusion':
        out = fusion(leaf(im768[None]))
    elif name == 'SVFE':
        out = head.svfe(leaf(x23))
    elif name == 'FCN + max':
        out = M._layer_forward('fcn_max', leaf(x128), head.fcn.fc.weight, head.fcn.fc.bias, M.EPS, T)
    else:
        out = M.reindex(leaf(vfeat), idx)
    out.backward(torch.ones_like(out))


def run_torch(name):
    if name == 'featureMaping':
        ms = [leaf(m) for m in maps]
        out = O.feature_mapping(vox.clone(), ms, IMSIZE.to(dev))
    elif name == 'ImageFeatureFusion':
        out = O.fusion(leaf(im768[None]), params)
    elif name == 'SVFE':
        x = O.vfe(leaf(x23), params['backbone.svfe.vfe1.fcn.fc.weight'], params['backbone.svfe.vfe1.fcn.fc.bias'])
        out = O.vfe(x, params['backbone.svfe.vfe2.fcn.fc.weight'], params['backbone.svfe.vfe2.fcn.fc.bias'])
    elif name == 'FCN + max':
        out = torch.max(O.crb(leaf(x128), params['backbone.fcn.fc.weight'], params['backbone.fcn.fc.bias']), dim=2)[0]
    else:
        out = O.reindex(leaf(vfeat), idx, G.voxelshape)
    out.backward(torch.ones_like(out))


def timed(fn, n):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


LAYERS = {'ImageFeatureFusion': [(768, 768), (768, 128), (128, 128), (128, 16), (16, 16)], 'SVFE': [(23, 16), (32, 64)],
          'FCN + max': [(128, 128)], 'featureMaping': [], 'reindex': []}


def cost(name):
    """(GFLOP, compulsory GB) of forward + backward from the shapes"""
    if name == 'featureMaping':    # out (R, 768) written, d_out read, three maps read and their gradients written
        px = sum(h * w for h, w in synth.fpn_shapes()) * 256
        return 0.0, (2 * R * 768 + 2 * px + R * 9) * 4 / 1e9
    if name == 'reindex':          # the grid written and its gradient read, N x 128 features read and written
        cells = G.voxelshape[0] * G.voxelshape[1] * G.voxelshape[2] * 128
        return 0.0, (2 * cells + 2 * N * 128) * 4 / 1e9
    fl = sum(6 * R * ci * co for ci, co in LAYERS[name]) / 1e9
    by = sum((R * ci + 2 * R * co) + (2 * R * co + 2 * R * ci) for ci, co in LAYERS[name]) * 4 / 1e9
    return fl, by


lines = [f'{card} | one frame: 120000 points, N = {N} voxels, T = {T}, R = {R} dense rows | forward + backward, CUDA events, '
         'every input requires a gradient']
for name in ['featureMaping', 'ImageFeatureFusion', 'SVFE', 'FCN + max', 'reindex']:
    ours = timed(lambda: run_ours(name), 10)
    ref = timed(lambda: run_torch(name), 3)
    fl, by = cost(name)
    rate = f'{fl / ours:.1f} TFLOP/s, ' if fl else ''
    lines.append(f'{name:20s} ours {ours:9.3f} ms ({fl:7.1f} GFLOP, {by:6.2f} GB compulsory -> {rate}{by / ours:.2f} TB/s effective) | '
                 f'torch eager fp32 autograd {ref:9.3f} ms | {ref / ours:6.1f}x')
report = '\n'.join(lines)
print(report)
if len(sys.argv) > 1:
    os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
    with open(sys.argv[1], 'w') as fh:
        fh.write(report + '\n')
