"""bench.py — frames/s of the point-side hot path (voxelize + fuse + VFE + scatter) on N B200s of one node.

    python bench.py --gpus 1 --steps 10 --warmup 3                       # ours (CUDA, through the C ABI)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W                           # N ranks, frame-sharded, no collective
    python bench.py --impl reference --steps K --warmup W                # the reference algorithm on the host cores
    python bench.py --steps K --warmup W --dump-outputs DIR              # + what the last timed step returned, as DIR/*.npy

A step = one pass of the hot path over one batch of 8 synthetic KITTI-shaped frames per GPU (BASELINE.json
configs[1]): P = 120 000 points, FPN maps (256,104,336)/(256,52,168)/(256,26,84), grid 352x400x10, T = 35.
Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FRAMES_PER_GPU = 8
POINTS = 120_000
METRIC = 'frames/sec voxelize+fuse+VFE+scatter'
WORKLOAD = ('configs[1]: batch-8 synthetic KITTI-shaped frames per GPU (P=120000 pts/frame, FPN maps '
            '256x{104x336,52x168,26x84} fp32, grid 352x400x10, T=35): voxelize + project + 4-corner gather + '
            '8-layer fusion/VFE stack (fp32) + dense (128,10,352,400) grid')
# --dump-outputs budget (< 64 MB): 16 MB of uniformly sampled grid values (98 % of the cells are empty: this catches writes
# outside the voxels) + up to 8 frames x 8192 voxel rows x (128 features + 4 coordinates) = 36 MB from the occupied cells
DUMP_GRID_SAMPLES = 1 << 22
DUMP_VOXEL_ROWS = 8192


def grid_sample_index(numel: int) -> np.ndarray:
    """Flat indices into the (B,128,nz,nx,ny) grid whose values --dump-outputs writes (sorted, drawn with replacement). They
    depend on the seed and the grid size only, so two builds of the project are compared at the same elements."""
    return np.sort(np.random.default_rng(0).integers(0, numel, min(DUMP_GRID_SAMPLES, numel), dtype=np.int64))


def voxel_sample_rows(f: int, n: int) -> np.ndarray:
    """Rows of frame f's (n,128) voxel features that --dump-outputs writes: all of them up to DUMP_VOXEL_ROWS, else a sorted
    sample drawn from a seed that depends on f only (builds with equal voxel counts are compared at the same voxels)."""
    if n <= DUMP_VOXEL_ROWS:
        return np.arange(n)
    return np.sort(np.random.default_rng(f).choice(n, DUMP_VOXEL_ROWS, replace=False))


def dump_outputs(out_dir: str, path, grid, counts):
    """Writes what one step of the timed path returned, for output-for-output comparison of two builds:
    counts.npy         (B,4) float64, the int32 per-frame counts (voxels, kept rows, invalid points, max points in one voxel)
    grid_sample.npy    (n,) float32, the grid at the flat indices of grid_sample_index(grid.numel())
    voxel_features.npy (m,128) float32, rows voxel_sample_rows(f, N_f) of path.voxel_features(f), frame after frame
    voxel_index.npy    (m,4) float64, their [frame, ix, iy, iz]"""
    import torch
    idx = torch.from_numpy(grid_sample_index(grid.numel())).to(grid.device)
    feats, coords = [], []
    for f in range(counts.shape[0]):
        vfeat, vidx = path.voxel_features(f)
        rows = torch.from_numpy(voxel_sample_rows(f, vfeat.shape[0])).to(vfeat.device)
        feats.append(vfeat[rows].cpu())
        coords.append(vidx[rows].cpu())
    arrays = dict(counts=counts.cpu().numpy().astype(np.float64), grid_sample=grid.reshape(-1)[idx].cpu().numpy(),
                  voxel_features=torch.cat(feats).numpy(), voxel_index=torch.cat(coords).numpy().astype(np.float64))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def static_config(world: int, dense: bool = False):
    """The `config` object of the JSON line: identical for both arms (`--impl ours` / `--impl reference`) of one workload."""
    B = FRAMES_PER_GPU
    G = (512 * 512 * 10) if dense else (352 * 400 * 10)
    return dict(workload=(WORKLOAD if not dense else
                          'configs[4]: batch-8 dense 128-beam-like synthetic frames per GPU (P=250000 pts/frame, velorange [0,-51.2,-3,102.4,51.2,1], '
                          'grid 512x512x10 = 1.34 GB dense output per frame, same FPN maps / layers): NOT the headline configuration'),
                frames_per_gpu=B, points_per_frame=250_000 if dense else POINTS,
                inputs='frame id g (global, rank r owns g = r, r + world, ...): synth.make_points(g, P), synth.make_fpn_maps(g), synth.make_weights(0), synth.kitti_calib()',
                l2=f'no flush: per step the inputs (376 MB FPN maps) and outputs ({B * 128 * G * 4 / 1e9:.1f} GB grid) exceed the 126 MB L2',
                parallelism=f'frame-sharded x{world}, no forward collective')


def refuse_debug_env():
    """The release library reads no environment switch (work-skipping MVX_DBG & co. exist only in -DMVX_DEVTOOLS builds);
    a bench run with one of them set is refused so that no number can come from a kernel with work removed."""
    bad = sorted(k for k in os.environ if k.startswith('MVX_'))
    if bad:
        print(f'bench.py: refusing to run with {bad} set (debug switches; unset them)', file=sys.stderr)
        sys.exit(2)


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d['hbm_gbs'], tensor=d.get('bf16_tflops_sustained', d['bf16_tflops']), src='measured (MEASURED_PEAKS.json)')
    return dict(hbm=6650.0, tensor=1400.0, src='fallback (B200_PROFILING.md)')


class ClockSampler:
    """nvidia-smi sampled every 20 ms from before the warm-up; only rows inside the timed window are used."""
    Q = ('timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index: int):
        self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
        self.p = None
        self.t0 = self.t1 = None
        try:
            self.p = subprocess.Popen(['nvidia-smi', '-i', str(gpu_index), f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                       '-lms', '20'], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            pass

    def begin(self):
        self.t0 = time.time()

    def end(self):
        self.t1 = time.time()

    def stop(self):
        import datetime
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        if self.p is None:
            return out
        time.sleep(0.05)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(', ') for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons, allsm = [], [], set(), []
        for r in rows:
            try:
                ts = datetime.datetime.strptime(r[0], '%Y/%m/%d %H:%M:%S.%f').timestamp()
                clk, cmax = float(r[1]), float(r[2])
            except (ValueError, IndexError):
                continue
            allsm.append(clk)
            mx.append(cmax)
            if self.t0 is not None and not (self.t0 - 0.02 <= ts <= self.t1 + 0.02):
                continue
            sm.append(clk)
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[4:8]):
                if v.strip().lower() == 'active':
                    reasons.add(name)
        if not sm and allsm:          # window shorter than the sampling period: fall back to the whole run
            sm = allsm
        if sm:
            out = dict(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


def bind_near_gpu(local: int):
    """Run this rank, and first-touch its pinned host buffers, on the NUMA node its GPU hangs off: eight ranks whose pinned
    buffers all sit on one socket pull 3 GB of FPN maps per step through one memory controller and the socket interconnect
    (round 1: 23 GB/s per GPU at 8 GPUs against 45 GB/s at 1). Best effort - every failure leaves the process as it was."""
    info = dict(node=None, cpus=None, mempolicy=None)
    try:
        import ctypes
        import torch
        pr = torch.cuda.get_device_properties(local)
        bdf = f'{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0'
        base = f'/sys/bus/pci/devices/{bdf}'
        node = int(open(f'{base}/numa_node').read().strip())
        info['pci'] = bdf
        if node < 0:
            return info
        info['node'] = node
        cpus = set()
        for part in open(f'/sys/devices/system/node/node{node}/cpulist').read().strip().split(','):
            lo, _, hi = part.partition('-')
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0)
        use = cpus & allowed
        if use:
            os.sched_setaffinity(0, use)
            info['cpus'] = len(use)
        mask = ctypes.c_ulong(1 << node)
        rc = ctypes.CDLL(None, use_errno=True).syscall(238, 1, ctypes.byref(mask), 65)   # set_mempolicy(MPOL_PREFERRED, {node})
        info['mempolicy'] = 'preferred' if rc == 0 else f'errno {ctypes.get_errno()}'
    except Exception as exc:
        info['error'] = f'{type(exc).__name__}: {exc}'[:120]
    return info


# ------------------------------------------------------------------------------------------------ reference arm
def cpu_reference_frame(frame_id: int, threads: int, dtype=None, keep: bool = False):
    """One full-size frame through the oracle port of the reference path on the host cores; returns seconds + stages
    (+ the oracle's voxel features / idx when `keep`: the parity check of the bench line uses them, outside any timed region)."""
    import torch
    from mvxnet_makise_b200 import synth
    from oracle import pointpath_oracle as O
    torch.set_num_threads(threads)
    pts = synth.make_points(frame_id, POINTS)
    maps = synth.make_fpn_maps(frame_id)
    sd = synth.make_weights(0)
    stages = {}
    t0 = time.perf_counter()
    with torch.no_grad():
        out = O.forward_frame(pts, synth.kitti_calib(), maps, sd, synth.KITTI_GRID, synth.KITTI_IMSIZE_HW, stages=stages,
                              **({'dtype': dtype} if dtype is not None else {}))
    t = time.perf_counter() - t0
    if keep:
        return t, stages, dict(vfeat=out['vfeat'], idx=out['idx'])
    return t, stages


def gpu_eager_reference_frame(frame_id: int, device):
    """Second comparison line of SURVEY.md §8d: the reference's GPU half (featureMaping -> ImageFeatureFusion -> concat ->
    SVFE/FCN/max -> reindex, MVXNet.py:21-27 on cfg.device='cuda') as torch-eager ops on THIS GPU, through the oracle port;
    the CPU half (lidar2Img + group, train.py:26-49) is timed separately on the host like the reference runs it."""
    import torch
    from mvxnet_makise_b200 import synth
    from oracle import pointpath_oracle as O
    pts = synth.make_points(frame_id, POINTS)
    maps = synth.make_fpn_maps(frame_id)
    sd = {k: torch.from_numpy(np.asarray(v)).to(device) for k, v in synth.make_weights(0).items()}
    t0 = time.perf_counter()
    pcd6 = O.points_with_proj(pts, synth.kitti_calib())
    voxel9, uidx = O.group(pcd6, synth.KITTI_GRID.velorange, synth.KITTI_GRID.voxelsize, synth.KITTI_GRID.T)
    t_cpu = time.perf_counter() - t0
    feats = [torch.from_numpy(m).to(device) for m in maps]
    imsize = torch.Tensor(list(synth.KITTI_IMSIZE_HW)).to(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    with torch.no_grad():
        for it in range(4):
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            voxels = torch.Tensor(voxel9).to(device)                              # train.py:125-128 (H2D of the dense tensor)
            idx = torch.LongTensor(np.concatenate([np.zeros((uidx.shape[0], 1)), uidx], axis=1)).to(device)
            e0.record()
            im768 = O.feature_mapping(voxels, feats, imsize, 1e-6)
            im16 = O.fusion(im768[None], sd, 1e-6)
            x23 = torch.concat([voxels[None][..., :7], im16], dim=-1)
            vfeat = O.voxel_features(x23, sd, 1e-6)
            grid = O.reindex(vfeat, idx, synth.KITTI_GRID.voxelshape)
            e1.record()
            torch.cuda.synchronize()
            if it:
                times.append((e0.elapsed_time(e1) * 1e-3, time.perf_counter() - t1))
            del im768, im16, x23, vfeat, grid
    gpu_s = sum(t[0] for t in times) / len(times)
    wall_s = sum(t[1] for t in times) / len(times)
    return dict(gpu_half_ms=round(gpu_s * 1e3, 2), gpu_half_with_h2d_ms=round(wall_s * 1e3, 2), cpu_half_ms=round(t_cpu * 1e3, 2),
                value=round(1.0 / (wall_s + t_cpu), 3), unit='frames/s', kind='port',
                sample=f'1 full-size frame (P={POINTS}), dense (N,T,.) formulation like the reference: CPU lidar2Img+group on the host, '
                       'then featureMaping .. reindex as torch-eager CUDA ops (oracle/pointpath_oracle.py); 3 timed repeats after 1 warm-up')


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import torch
    from oracle import pointpath_oracle as O
    O.build_c_oracle() if not os.path.exists(os.path.join(ROOT, 'oracle', '_build', 'libvoxel_oracle.so')) else None
    threads = os.cpu_count() or 1
    steps = args.steps
    for w in range(args.warmup):
        cpu_reference_frame(w, threads)
    times, stages_acc = [], {}
    for s in range(steps):
        t, st = cpu_reference_frame(100 + s, threads)
        times.append(t)
        for k, v in st.items():
            stages_acc[k] = stages_acc.get(k, 0.0) + v / steps
    total = sum(times)
    fps = steps / total
    sample = (f'each step = ONE full-size frame (1 of the 8 frames of the batch, P={POINTS}) through the numpy/torch-CPU port of '
              f'the reference path (oracle/pointpath_oracle.py), {threads} torch threads')
    line = dict(impl='reference', metric=METRIC, value=fps, unit='frames/s', n_gpus=args.gpus, steps=steps, warmup=args.warmup,
                ms_per_step=1e3 * total / steps, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32',
                data='synthetic', config=static_config(int(os.environ.get('WORLD_SIZE', str(args.gpus)))),
                cpu_baseline=dict(value=fps, unit='frames/s', cores=threads, kind='port', sample=sample,
                                  stages_s={k: round(v, 4) for k, v in stages_acc.items()}),
                e2e=dict(value=fps, unit='frames/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ our arm
def algorithmic_work(seg: str, N, K, B, G, npts=POINTS):
    """(bound, work per launch) for a timed segment: bytes for HBM-bound kernels, flops for the GEMM layers
    (SURVEY.md §8d minimal figures: kept rows + weighted pad rows only)."""
    sumK, sumN = float(sum(K)), float(sum(N))
    rowsA, rowsB = sumK + B, sumK + sumN
    maps_b = 4.0 * 256 * (104 * 336 + 52 * 168 + 26 * 84)
    gemm = dict(fcn1=(768, 768, rowsA), conv1=(768, 128, rowsA), fcn2=(128, 128, rowsA), conv2=(128, 16, rowsA),
                fcn3=(16, 16, rowsA), vfe1=(23, 16, rowsA), vfe2=(32, 64, rowsB), fcn=(128, 128, rowsB))
    pixels = 104 * 336 + 52 * 168 + 26 * 84
    if seg == 'pixel_gemm':      # pixel-first fcn1, tensor half: Z_l = F_l W1_l^T over every map pixel (3 launches)
        return 'tensor', 2.0 * 256 * 768 * B * pixels
    if seg == 'fcn1_combine':    # pixel-first fcn1, memory half: read Z once, 12-corner combine, write raw Y1 rows
        return 'hbm', B * pixels * 768 * 4.0 + rowsA * (3072 + 16)
    if seg in gemm:
        cin, cout, rows = gemm[seg]
        return 'tensor', 2.0 * cin * cout * rows
    if seg == 'grid_fill':
        return 'hbm', B * (128.0 * G * 4 + G * 4) + sumN * 512
    if seg == 'gather':
        return 'hbm', B * maps_b + rowsA * (3072 + 40)
    if seg == 'maps_nhwc':
        return 'hbm', 2 * B * maps_b
    if seg == 'voxelize':
        return 'hbm', B * npts * 16.0 + sumK * 8 + sumN * 32 + B * G * 4
    return 'hbm', 0.0


def run_ours(args):
    import torch
    import torch.distributed as dist
    from mvxnet_makise_b200 import synth, _lib, dist as mdist
    from mvxnet_makise_b200.pipeline import PointPath
    from mvxnet_makise_b200.modules import pack_calib

    rank, world, local = mdist.env_rank_world()
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    numa = bind_near_gpu(local)            # before any pinned allocation: first touch decides where the host pages live
    mdist.init('nccl')
    dense = args.workload == 'dense'       # BASELINE.json configs[4]: 128-beam-like frames on the larger 512x512x10 grid
    grid_spec = synth.DENSE_GRID if dense else synth.KITTI_GRID
    npts = 250_000 if dense else POINTS
    B, G = FRAMES_PER_GPU, grid_spec.cells

    # ---- synthetic inputs for THIS rank's frames: global frame ids, sharded round-robin (weak scaling: B frames per GPU)
    frame_ids = mdist.shard_frames(world * B, rank, world)
    frames = [synth.make_points(g_, npts, grid=grid_spec, beams=128 if dense else 64) for g_ in frame_ids]
    offsets = np.concatenate([[0], np.cumsum([p.shape[0] for p in frames])]).tolist()
    points_h = torch.from_numpy(np.concatenate(frames, 0)).pin_memory()
    calib_h = torch.stack([pack_calib(synth.kitti_calib()) for _ in range(B)]).pin_memory()
    per_frame_maps = [synth.make_fpn_maps(g_) for g_ in frame_ids]
    maps_h = [torch.from_numpy(np.concatenate([m[l] for m in per_frame_maps], 0)).pin_memory() for l in range(3)]
    del per_frame_maps
    points_d, calib_d = points_h.to(dev), calib_h.to(dev)
    maps_d = [m.to(dev) for m in maps_h]
    _lib.set_fusion_mode(args.fusion_mode)
    if args.dtype == 'bf16':
        _lib.set_gemm_mode(6)
    path = PointPath(synth.make_weights(0), grid_spec, device=dev)
    path.host_chunk, path.host_streams = args.host_chunk, args.host_streams

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize()

    # ---- device-resident leg (`value`) ----------------------------------------------------------------
    sampler = ClockSampler(local) if rank == 0 else None
    def step():
        if args.device_split > 1:
            return path.forward_device_split(points_d, offsets, calib_d, maps_d, True, args.device_split)
        return path.forward_device(points_d, offsets, calib_d, maps_d)

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    launches0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if sampler:
        sampler.begin()
    e0.record()
    for _ in range(args.steps):
        out = step()
    e1.record()
    barrier()
    if sampler:
        sampler.end()
    ms_total = e0.elapsed_time(e1)
    launches = _lib.launch_count() - launches0
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:     # before the passes below overwrite the outputs of the last timed step
        dump_outputs(args.dump_outputs, path, *out)
    # per-stage pass (outside the timed region): CUDA events around every stage on the stream it runs on, with the map
    # branch serialised behind the point branch (fusion mode 2) so that a stage's time is its own and not the time it
    # spent sharing the SMs with the other branch; `value` above is the default, overlapped schedule
    n_stage = min(args.steps, 10)
    _lib.set_fusion_mode(2 if args.fusion_mode == 1 else args.fusion_mode)
    path.forward_device(points_d, offsets, calib_d, maps_d)
    _lib.check(_lib.lib.mvx_timing_enable(n_stage), 'timing_enable')
    es0, es1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    es0.record()
    for _ in range(n_stage):
        path.forward_device(points_d, offsets, calib_d, maps_d)
    es1.record()
    torch.cuda.synchronize()
    ms_serial = es0.elapsed_time(es1) / n_stage
    seg_ms = np.zeros(_lib.NUM_SEGMENTS)
    buf = (_lib.c_float * _lib.NUM_SEGMENTS)()
    for c in range(n_stage):
        _lib.check(_lib.lib.mvx_timing_read(c, buf), 'timing_read')
        seg_ms += np.array(buf[:]) / n_stage
    _lib.lib.mvx_timing_enable(0)
    _lib.set_fusion_mode(args.fusion_mode)
    counts = path.counts.cpu().numpy()
    if world > 1:
        t = torch.tensor([ms_total], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())

    # ---- context leg (SURVEY.md §8f rank 2): the path WITHOUT the dense grid + the sparse hand-off to the CML's first CRB3d ------
    # (voxelnet/Pipe.py:35): what a consumer that takes the sparse hand-off pays instead of grid fill + dense Conv3d. Rank 0, N = 1
    # shape of the question only; outside the timed region of `value`.
    handoff = None
    if rank == 0 and not dense and args.fusion_mode == 1 and args.dtype != 'bf16':
        gw = torch.Generator().manual_seed(11)
        cw = (torch.randn((64, 128, 3, 3, 3), generator=gw) * 0.02).to(dev)
        cb = (torch.randn((64,), generator=gw) * 0.1).to(dev)
        for _ in range(2):
            path.forward_device(points_d, offsets, calib_d, maps_d, want_grid=False)
            c1 = path.cml_conv1(cw, cb)
        n_h = min(args.steps, 5)
        eh0, eh1, eh2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        ms_nogrid = ms_conv = 0.0
        for _ in range(n_h):
            eh0.record()
            path.forward_device(points_d, offsets, calib_d, maps_d, want_grid=False)
            eh1.record()
            c1 = path.cml_conv1(cw, cb)
            eh2.record()
            torch.cuda.synchronize()
            ms_nogrid += eh0.elapsed_time(eh1) / n_h
            ms_conv += eh1.elapsed_time(eh2) / n_h
        handoff = dict(path_without_grid_ms=round(ms_nogrid, 4), sparse_cml_conv1_ms=round(ms_conv, 4),
                       frames_per_s=round(B / ((ms_nogrid + ms_conv) * 1e-3), 1), out_shape=list(c1.shape),
                       note='context, not the headline: PointPath.forward_device(want_grid=False) + PointPath.cml_conv1 (mvx_cml_conv1_sparse: '
                            'Conv3d(128,64,3,(2,1,1),(1,1,1)) + ReLU + batch-stat BatchNorm3d from the voxel features, no dense grid), one GPU, '
                            f'{B} frames per step; the dense alternative is the grid_fill stage above plus a dense Conv3d over 180 M cells per frame')
        del c1, cw, cb
        path.forward_device(points_d, offsets, calib_d, maps_d)    # back to the grid-producing context

    # ---- host-buffer leg (`e2e`): pinned H2D of every input + path + D2H of the result, every step -------
    # Steps are pipelined across calls (two buffer sets): step s+1's copies run while step s computes. Every step still
    # copies ITS inputs host->device and its result device->host inside the timed region; the host consumes the result of
    # step s-1 (waits for it) before it submits step s+1, like a data loader running one batch ahead.
    for _ in range(3):
        path.forward_host(points_h, offsets, calib_h, maps_h)
    barrier()
    e0.record()
    prev, checksum = None, 0
    for _ in range(args.steps):
        step_h = path.forward_host(points_h, offsets, calib_h, maps_h, sync=False)
        if prev is not None:
            checksum += int(prev.wait()[1][:, 0].sum())
        prev = step_h
    checksum += int(prev.wait()[1][:, 0].sum())
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1)
    assert checksum == args.steps * int(counts[:, 0].sum()), 'e2e leg: host-visible voxel counts differ from the device leg'
    # context leg: the reference's own data flow - the FPN maps are produced ON the GPU by the frozen backbone (Head.py:14-22) and
    # never cross PCIe; only the raw points and the calibration do (train.py:125-128 ships the voxel tensor instead)
    for _ in range(3):
        path.forward_host(points_h, offsets, calib_h, maps_d)
    barrier()
    e0.record()
    prev = None
    for _ in range(args.steps):
        step_h = path.forward_host(points_h, offsets, calib_h, maps_d, sync=False)
        if prev is not None:
            prev.wait()
        prev = step_h
    prev.wait()
    e1.record()
    barrier()
    ms_e2e_res = e0.elapsed_time(e1)
    h2d_res = int(path.h2d_bytes)
    if world > 1:
        t = torch.tensor([ms_e2e_res], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e2e_res = float(t.item())
    path.forward_host(points_h, offsets, calib_h, maps_h)      # back to the host-maps contexts (h2d_bytes of the headline leg)
    if world > 1:
        t = torch.tensor([ms_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e2e = float(t.item())

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk = peaks()
    names = [(_lib.lib.mvx_timing_segment_name(i) or b'').decode() for i in range(_lib.NUM_SEGMENTS)]
    stages = {n: round(float(ms), 4) for n, ms in zip(names, seg_ms) if n}
    dom = max(stages, key=stages.get)
    bound, work = algorithmic_work(dom, counts[:, 0], counts[:, 1], B, G, npts)
    dur_s = stages[dom] * 1e-3
    if bound == 'tensor':
        achieved, peak, unit = work / dur_s / 1e12, pk['tensor'], 'TFLOP/s'
    else:
        achieved, peak, unit = work / dur_s / 1e9, pk['hbm'], 'GB/s'
    traffic = None
    tpath = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(tpath) and not dense:      # the ncu capture was taken on the headline (KITTI) configuration
        traffic = json.load(open(tpath)).get(dom)
    # whole path against the HBM bound of SURVEY.md §8(d)'s MINIMAL bytes: points + FPN maps + grid + coords per frame, weights once
    min_bytes = B * (npts * 16.0 + 4.0 * 256 * sum(h * w for h, w in synth.fpn_shapes()) + 128.0 * G * 4) + float(counts[:, 0].sum()) * 32 + 726_880 * 4
    step_s = ms_total / args.steps * 1e-3
    whole = dict(algorithmic_bytes_per_frame=round(min_bytes / B), achieved_gbs=round(min_bytes / step_s / 1e9, 1), peak_gbs=pk['hbm'],
                 frac=round(min_bytes / step_s / 1e9 / pk['hbm'], 4),
                 note='minimal HBM bytes of the fused path (SURVEY.md §8d: 93 % of them the dense grid write) / measured step time; the fp32 layer stack between the reads and the grid write is tensor-bound, see stage_rooflines')
    roofline = dict(kernel=dom, bound=bound, achieved=round(achieved, 3), peak=peak, unit=unit, frac=round(achieved / peak, 4),
                    traffic=traffic, peak_source=pk['src'], ms_per_launch=stages[dom], share_of_step=round(stages[dom] / ms_serial, 4),
                    whole_path=whole)
    # every memory-bound stage against the HBM roofline (the north star's per-stage report)
    per_stage = {}
    for n in ('voxelize', 'maps_nhwc', 'gather', 'fcn1_combine', 'grid_fill'):
        b, w = algorithmic_work(n, counts[:, 0], counts[:, 1], B, G, npts)
        if stages.get(n, 0) > 0:
            per_stage[n] = dict(gbs=round(w / (stages[n] * 1e-3) / 1e9, 1), frac_hbm=round(w / (stages[n] * 1e-3) / 1e9 / pk['hbm'], 4))
    for n in ('fcn1', 'pixel_gemm', 'conv1'):
        if stages.get(n, 0) <= 0:
            continue
        b, w = algorithmic_work(n, counts[:, 0], counts[:, 1], B, G)
        per_stage[n] = dict(tflops=round(w / (stages[n] * 1e-3) / 1e12, 2), frac_tensor=round(w / (stages[n] * 1e-3) / 1e12 / pk['tensor'], 4))

    line = dict(metric=METRIC, value=world * B * args.steps / (ms_total * 1e-3), unit='frames/s', n_gpus=world, steps=args.steps,
                warmup=max(args.warmup, 3), ms_per_step=ms_total / args.steps, higher_is_better=True, scaling='weak',
                vs_baseline=None, dtype='bf16' if args.dtype == 'bf16' else 'f32', data='synthetic',
                config=static_config(world, dense),
                workload_stats=dict(voxels_per_frame=int(counts[:, 0].mean()), kept_points_per_frame=int(counts[:, 1].mean()), frame_ids=frame_ids),
                host_numa=numa, clocks=clocks,
                e2e=dict(value=world * B * args.steps / (ms_e2e * 1e-3), unit='frames/s', h2d_bytes_per_step=int(path.h2d_bytes),
                         d2h_bytes_per_step=int(path.d2h_bytes), ms_per_step=ms_e2e / args.steps,
                         note=f'PointPath.forward_host(sync=False): pinned-host points+calib+FPN maps -> H2D -> fused path -> D2H counts + feature head, every step; sub-batches of {args.host_chunk} frame(s) (H2D of sub-batch j+1 overlaps the kernels of sub-batch j) and two buffer sets (the copies of step s+1 overlap the kernels of step s); the host waits for the result of step s-1 before it submits step s+1. The FPN maps (376 of the 391 MB) are shipped from the host although the reference produces them on the GPU: the conservative reading of "host inputs"'),
                e2e_maps_resident=dict(value=world * B * args.steps / (ms_e2e_res * 1e-3), unit='frames/s', h2d_bytes_per_step=h2d_res, ms_per_step=ms_e2e_res / args.steps,
                                       note='context, not the headline: the same host entry with the FPN maps already on the GPU, where the reference produces them (Head.py:14-22); only points + calibration cross PCIe'),
                sparse_handoff=handoff,
                gpu_launches=int(launches), roofline=roofline, stages_ms=stages, stage_rooflines=per_stage,
                stages_note=f'per-stage CUDA events from a separate pass of {n_stage} steps with the map branch serialised (fusion mode 2, {ms_serial:.3f} ms/step); the timed region runs it on a side stream concurrently with the point branch')
    if world == 1 and not args.no_cpu_baseline and not dense:
        # the checker, outside every timed region: frame 0 of the timed batch through the oracle (fp32 = the reference's own
        # arithmetic, timed as the CPU baseline; fp64 = its rounding-free value) against what the timed kernels produced
        path.forward_device(points_d, offsets, calib_d, maps_d)
        got_v, got_i = (t_.cpu() for t_ in path.voxel_features(0))
        t, st, ref32 = cpu_reference_frame(frame_ids[0], os.cpu_count() or 1, keep=True)
        line['cpu_baseline'] = dict(value=1.0 / t, unit='frames/s', cores=os.cpu_count() or 1, kind='port',
                                    sample=f'1 full-size frame (P={POINTS}) of the batch through oracle/pointpath_oracle.py (numpy + torch CPU fp32)',
                                    stages_s={k: round(v, 3) for k, v in st.items()})
        _, _, ref64 = cpu_reference_frame(frame_ids[0], os.cpu_count() or 1, dtype=torch.float64, keep=True)

        def rel(a_, b_):
            return float((a_.double() - b_.double()).abs().max() / b_.double().abs().max().clamp_min(1e-30))
        line['parity'] = dict(checked_frames=1, frame_id=frame_ids[0], voxel_coords_bit_exact=bool(torch.equal(got_i[:, 1:], ref32['idx'][:, 1:])),
                              rel_err_fp64=rel(got_v, ref64['vfeat']), rel_err_fp32=rel(got_v, ref32['vfeat']),
                              fp32_reference_noise=rel(ref32['vfeat'], ref64['vfeat']),
                              tolerance=5e-2 if args.dtype == 'bf16' else 1e-4,
                              note='max|a-ref|/max|ref| over the (N,128) voxel features of frame 0 of the timed batch vs oracle.forward_frame evaluated in fp64 / fp32; all 8 frames: tests/test_gpu_fullsize.py')
        del ref32, ref64
        if not args.no_gpu_eager_baseline:
            try:
                del path
                torch.cuda.empty_cache()
                line['gpu_eager_baseline'] = gpu_eager_reference_frame(0, dev)
            except Exception as exc:   # a context line only: never let it take the bench line down
                line['gpu_eager_baseline'] = dict(error=f'{type(exc).__name__}: {exc}'[:200])
        ge = line.get('gpu_eager_baseline', {}).get('value')
        # two denominators, equal prominence: the whole path ported to the host cores (the contract's CPU baseline) and the
        # reference AS DEPLOYED (CPU lidar2Img + group, then its GPU half as torch-eager ops on this same B200)
        line['speedup_e2e'] = dict(vs_cpu_port=round(line['e2e']['value'] / line['cpu_baseline']['value'], 1),
                                   vs_reference_as_deployed_gpu_eager=round(line['e2e']['value'] / ge, 1) if ge else None)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ training workload
def run_train(args):
    """BASELINE.json configs[3]: training step through the fused VFE/fusion layers, 16 frames per GPU - forward_train,
    CUDA backward into one flat gradient bucket, NCCL all-reduce of the bucket, AdamW. Not the headline metric (that is
    the forward path above); run with `--workload train`."""
    import torch
    import torch.distributed as dist
    from mvxnet_makise_b200 import synth, _lib, dist as mdist
    from mvxnet_makise_b200.training import HotPathTrainer
    from mvxnet_makise_b200.modules import pack_calib

    rank, world, local = mdist.env_rank_world()
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    mdist.init('nccl')
    B = args.train_frames
    frames = [synth.make_points(g_, POINTS) for g_ in mdist.shard_frames(world * B, rank, world)]
    offsets = np.concatenate([[0], np.cumsum([p.shape[0] for p in frames])]).tolist()
    points = torch.from_numpy(np.concatenate(frames, 0)).to(dev)
    calib = torch.stack([pack_calib(synth.kitti_calib()) for _ in range(B)]).to(dev)
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    maps = [torch.randn((B, 256, h, w), generator=g, device=dev) for (h, w) in synth.fpn_shapes()]
    tr = HotPathTrainer(synth.make_weights(0), synth.KITTI_GRID, device=dev)
    cap = max(128, (POINTS + 127) // 128 * 128)
    d_vfeat = torch.randn((B, cap, 128), generator=g, device=dev) * 1e-3      # stand-in for dLoss/d(voxel features) from CML/RPN

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize()

    sampler = ClockSampler(local) if rank == 0 else None
    for _ in range(max(args.warmup, 3)):
        tr.step(points, offsets, calib, maps, d_vfeat=d_vfeat)
    barrier()
    launches0 = _lib.launch_count()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(args.steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if sampler:
        sampler.begin()
    e0.record()
    for s_ in range(args.steps):
        ev[s_][0].record()
        tr.path.forward_train(points, offsets, calib, maps, True)
        ev[s_][1].record()
        tr.path.backward(d_vfeat=d_vfeat, grad_flat=tr.grad)
        ev[s_][2].record()
        tr.opt.reduce_and_step(tr.bucket, B)
        tr._push_weights()
        ev[s_][3].record()
    e1.record()
    barrier()
    if sampler:
        sampler.end()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler else None
    phases = [sum(ev[s_][i].elapsed_time(ev[s_][i + 1]) for s_ in range(args.steps)) / args.steps for i in range(3)]
    launches = _lib.launch_count() - launches0
    counts = tr.path.counts.cpu().numpy()
    if world > 1:
        t = torch.tensor([ms_total], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    if rank == 0:
        K = float(counts[:, 1].sum())
        flops_fwd = 2.0 * 706816 * (K + B) + 2.0 * 18800 * (K + B + float(counts[:, 0].sum()))
        line = dict(metric='frames/sec training step (forward + backward of the fused VFE/fusion layers, gradient all-reduce, AdamW)',
                    value=world * B * args.steps / (ms_total * 1e-3), unit='frames/s', n_gpus=world, steps=args.steps,
                    warmup=max(args.warmup, 3), ms_per_step=ms_total / args.steps, higher_is_better=True, scaling='weak',
                    vs_baseline=None, dtype='f32', data='synthetic',
                    config=dict(workload=f'configs[3]: training step, {B} synthetic KITTI-shaped frames per GPU (P={POINTS}), forward_train '
                                         '(row-first fcn1, activations kept) + backward of the 8 hot-path layers into one flat fp32 bucket '
                                         '(726 880 floats) + NCCL all-reduce of the bucket + AdamW; upstream gradient dLoss/d(voxel features) synthetic',
                                frames_per_gpu=B, points_per_frame=POINTS, parallelism=f'frame-sharded x{world}; one all-reduce of 2.9 MB per step',
                                l2='no flush: activations (A1/Y1: 5.9 GB each at 16 frames) exceed the 126 MB L2'),
                    clocks=clocks, gpu_launches=int(launches),
                    phases_ms=dict(forward_train=round(phases[0], 3), backward=round(phases[1], 3), allreduce_adamw=round(phases[2], 3)),
                    algorithmic_tflops=dict(forward=round(flops_fwd / (phases[0] * 1e-3) / 1e12, 2),
                                            backward=round((2.0 * flops_fwd - 2.0 * 768 * 768 * (K + B)) / (phases[1] * 1e-3) / 1e12, 2)))
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-gpu-eager-baseline', action='store_true', help='skip the torch-eager-on-this-GPU context line')
    ap.add_argument('--host-streams', type=int, default=2, help='compute streams the sub-batches of the e2e leg alternate between')
    ap.add_argument('--fusion-mode', type=int, default=1, help='1 = pixel-first fcn1 (default), 0 = row-first (gather + row GEMM)')
    ap.add_argument('--workload', default='forward', choices=['forward', 'train', 'dense'],
                    help="'train' = BASELINE configs[3], 'dense' = configs[4] (128-beam-like frames, 512x512x10 grid); neither is the headline metric")
    ap.add_argument('--train-frames', type=int, default=16)
    ap.add_argument('--device-split', type=int, default=1, help='run the device-resident leg as this many concurrent sub-batches (streams)')
    ap.add_argument('--host-chunk', type=int, default=2, help='frames per sub-batch of the host-buffer (e2e) leg')
    ap.add_argument('--dtype', default='f32', choices=['f32', 'bf16'],
                    help="'bf16' = reduced-precision mode of the layer stack (tolerance stated separately: tests/test_gpu_parity.py); not the headline line")
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one returned as DIR/*.npy: the counts, and fixed, seeded '
                         'samples of the grid and of the voxel features (see dump_outputs); forward and dense workloads of --impl ours')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs and (args.impl != 'ours' or args.workload == 'train'):
        ap.error('--dump-outputs applies to the forward and dense workloads of --impl ours')
    refuse_debug_env()
    if args.impl == 'reference':
        run_reference(args)
    elif args.workload == 'train':
        run_train(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
