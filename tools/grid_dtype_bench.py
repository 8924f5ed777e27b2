"""Grid dtype A/B on bench.py's forward inputs (8 frames of synth.make_points(g, 120 000), make_fpn_maps(g), make_weights(0),
kitti_calib()): the grid_fill segment and its write rate, the forward step with an fp32 / fp16 / bf16 grid, the step an
autocast consumer pays with an fp32 grid (+ grid.to(fp16)), and one training leg (forward_train + backward(d_grid)) with an
fp16 grid against fp32 + cast + cast-back. The grid_fill segment is also timed on a batch of 8 empty frames: that fill is the
pure streaming write of the zero grid, and the difference to the full batch is the cost of gathering the voxel features
into the occupied cells. Variants alternate inside every round. Prints one JSON line (and writes it to --out)."""
import argparse
import json
import subprocess
import sys
import os

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mvxnet_makise_b200 import _lib, synth  # noqa: E402
from mvxnet_makise_b200.modules import pack_calib  # noqa: E402
from mvxnet_makise_b200.pipeline import PointPath  # noqa: E402

DT = {'fp32': torch.float32, 'fp16': torch.float16, 'bf16': torch.bfloat16}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--frames', type=int, default=8)
    ap.add_argument('--rounds', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--out', default=None, help='also write the JSON line to this file')
    a = ap.parse_args()
    _lib.require_cuda()
    # name and power limit of the device this process runs on (by UUID: immune to CUDA_VISIBLE_DEVICES renumbering)
    uuid = f'GPU-{torch.cuda.get_device_properties(torch.cuda.current_device()).uuid}'
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,uuid', '--format=csv,noheader', '-i', uuid],
                         capture_output=True, text=True).stdout.strip()
    B = a.frames
    frames = [synth.make_points(g, 120_000) for g in range(B)]
    offsets = np.concatenate([[0], np.cumsum([p.shape[0] for p in frames])]).tolist()
    points = torch.from_numpy(np.concatenate(frames, 0)).cuda()
    calib = torch.stack([pack_calib(synth.kitti_calib()) for _ in range(B)]).cuda()
    maps = [torch.from_numpy(np.concatenate([synth.make_fpn_maps(g)[l] for g in range(B)], 0)).cuda() for l in range(3)]
    paths = {k: PointPath(synth.make_weights(0), grid_dtype=d) for k, d in DT.items()}
    G = int(np.prod(synth.KITTI_GRID.voxelshape))
    names = [(_lib.lib.mvx_timing_segment_name(i) or b'').decode() for i in range(_lib.NUM_SEGMENTS)]
    seg = names.index('grid_fill')

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1)

    fwd = {k: (lambda p=p: p.forward_device(points, offsets, calib, maps)) for k, p in paths.items()}
    empty = {k: PointPath(synth.make_weights(0), grid_dtype=d) for k, d in DT.items()}
    no_points = torch.zeros((0, 4), dtype=torch.float32, device='cuda')
    fwd_empty = {k: (lambda p=p: p.forward_device(no_points, [0] * (B + 1), calib, maps)) for k, p in empty.items()}
    fwd['fp32+cast'] = lambda: paths['fp32'].forward_device(points, offsets, calib, maps)[0].to(torch.float16)
    tr16 = PointPath(synth.make_weights(0), grid_dtype=torch.float16)
    tr32 = PointPath(synth.make_weights(0))
    h = {}

    def train16():
        grid, _ = tr16.forward_train(points, offsets, calib, maps, shuffle=False)
        if 'g16' not in h:
            h['g16'] = torch.randn(grid.shape, device='cuda', dtype=torch.float16)
        tr16.backward(d_grid=h['g16'])

    def train32_cast():
        grid, _ = tr32.forward_train(points, offsets, calib, maps, shuffle=False)
        grid.to(torch.float16)                         # what the CML's autocast does to the fp32 grid
        tr32.backward(d_grid=h['g16'].to(torch.float32))   # the cast's backward hands the path an fp32 d_grid

    legs = dict(fwd, **{'train fp16': train16, 'train fp32+cast': train32_cast})
    legs.update({'empty ' + k: fn for k, fn in fwd_empty.items()})
    for _ in range(a.warmup):
        for fn in legs.values():
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in legs}
    fill = {k: [] for k in DT}
    fill_empty = {k: [] for k in DT}
    buf = (_lib.c_float * _lib.NUM_SEGMENTS)()
    for _ in range(a.rounds):
        for k, fn in legs.items():
            times[k].append(timed(fn))
        for k in DT:                                   # the stage timing leg: one forward with segment events
            _lib.check(_lib.lib.mvx_timing_enable(1), 'timing_enable')
            fwd[k]()
            _lib.check(_lib.lib.mvx_timing_read(0, buf), 'timing_read')
            fill[k].append(buf[seg])
            _lib.check(_lib.lib.mvx_timing_enable(1), 'timing_enable')
            fwd_empty[k]()
            _lib.check(_lib.lib.mvx_timing_read(0, buf), 'timing_read')
            fill_empty[k].append(buf[seg])
    _lib.lib.mvx_timing_enable(0)
    res = dict(gpu=gpu, frames=B, rounds=a.rounds, warmup=a.warmup, grid_cells=G,
               note='median ms over rounds; variants alternate within each round; grid_fill GB/s = grid bytes written / segment time')
    res['step_ms'] = {k: float(np.median(v)) for k, v in times.items()}
    res['grid_fill_ms'] = {k: float(np.median(v)) for k, v in fill.items()}
    res['grid_fill_GBps'] = {k: B * 128 * G * DT[k].itemsize / (res['grid_fill_ms'][k] * 1e-3) / 1e9 for k in DT}
    res['grid_fill_empty_ms'] = {k: float(np.median(v)) for k, v in fill_empty.items()}
    res['grid_fill_empty_GBps'] = {k: B * 128 * G * DT[k].itemsize / (res['grid_fill_empty_ms'][k] * 1e-3) / 1e9 for k in DT}
    res['gather_ms'] = {k: res['grid_fill_ms'][k] - res['grid_fill_empty_ms'][k] for k in DT}
    res['fill_rate_vs_fp32'] = {k: res['grid_fill_GBps'][k] / res['grid_fill_GBps']['fp32'] for k in DT}
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == '__main__':
    main()
