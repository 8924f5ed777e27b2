"""The fused batched point path (stages 1-4) behind one call — what ``MVXNet.forward`` does between the image
backbone and ``VoxelNet.cml`` (MVXNet.py:21-27; Head.py:14-22; VoxelNet.py:24-34), with the CPU half of
train.py:26-49 (projection + voxelization) moved onto the GPU.

    path = PointPath(state_dict)                      # reference parameter names (SURVEY.md §8b)
    grid, counts = path(points_list, calibs, fpn_maps)   # (B,128,nz,nx,ny) fp32 on the GPU, counts (B,4) int32

Frames are independent (per-frame BatchNorm statistics, as in the batch-1 reference), so multi-GPU use is pure
frame sharding: see ``mvxnet_makise_b200.dist``.
"""
from __future__ import annotations

import ctypes
from typing import Dict, List, Sequence

import numpy as np
import torch

from . import _lib, synth
from ._lib import lib, check, ptr, stream_ptr
from .modules import pack_calib, pack_calib64, calib_is_f64

LAYER_NAMES = [name for name, *_ in synth.HOT_LAYERS]


class _Forward:
    """The record of one forward: everything a later call on its results (backward, cml_conv1, voxel_features, the drop-in's
    autograd nodes) reads. Every forward makes a new one, so a stale holder can tell by identity."""

    def __init__(self, args=None, keep=(), maps=None, train=False, subs=None):
        self.args = args            # the PointPathArgs of the launch (workspace pointers, B, cap)
        self.keep = keep            # host arrays and tensors the pointers in `args` refer to, kept alive with it
        self.maps = maps            # the fp32 FPN maps it read (the shapes of dLoss/d maps)
        self.train = train          # forward_train: the workspace holds the activations backward() needs
        self.subs = subs            # None: results live in this path; else the _Sub list of forward_host / forward_device_split
        self.cml_done = False       # cml_conv1 ran on it: the CML workspace holds what cml_conv1_backward reads


class _Sub:
    """Frames [f0, f1) of a batch run by forward_host / forward_device_split on their own PointPath context `path`."""

    def __init__(self, path, f0: int, f1: int, stream=None):
        self.path, self.f0, self.f1, self.stream = path, f0, f1, stream
        # forward_host only: device input buffers, the event that marks them copied, this call's offsets and point count
        self.in_points = self.in_calib = self.in_maps = self.ev = self.offsets = None
        self.n_points = 0


class _HostSlot:
    """One complete set of host-entry buffers (sub-batch input buffers + workspaces, device outputs, pinned results)."""

    def __init__(self):
        self.subs, self.used = [], False
        self.grid_out = self.counts = self.out_counts = self.out_head = self.done = None


class HostStep:
    """Handle of one asynchronous `PointPath.forward_host(..., sync=False)` call."""

    def __init__(self, slot: _HostSlot):
        self._slot = slot
        self.event = slot.done

    def wait(self):
        """Blocks until this call's results are in host memory; returns (grid on device, counts on host, head block on host)."""
        self.event.synchronize()
        return self._slot.grid_out, self._slot.out_counts, self._slot.out_head


class PointPath:
    def __init__(self, state_dict: Dict[str, torch.Tensor], grid: synth.GridSpec = synth.KITTI_GRID,
                 imsize_hw: Sequence[int] = synth.KITTI_IMSIZE_HW, eps: float = 1e-6, device='cuda'):
        _lib.require_cuda()
        dev = torch.device(device)
        # the parameter format the kernels read: W^T (Cin_pad16, Cout) with zero pad rows, and the bias, per layer; allocated
        # once and only ever written in place (load_parameters), so sub-batch contexts and earlier launches see every update
        wt = [torch.zeros((cin + (-cin) % 16, cout), dtype=torch.float32, device=dev) for _, cin, cout, _ in synth.HOT_LAYERS]
        bias = [torch.empty(cout, dtype=torch.float32, device=dev) for _, _, cout, _ in synth.HOT_LAYERS]
        self._init(dev, grid, (float(imsize_hw[0]), float(imsize_hw[1])), float(eps), wt, bias)
        self.load_state_dict(state_dict)

    def _init(self, device, grid_spec: synth.GridSpec, imsize_hw, eps: float, wt, bias):
        """Declares every attribute; `__init__` and `_sub_context` call it."""
        self.device = device
        self.grid_spec = grid_spec
        self.grid = _lib.make_grid(grid_spec.velorange, grid_spec.voxelsize, grid_spec.voxelshape, grid_spec.T)
        self.imsize_hw = imsize_hw
        self.eps = eps
        self.wt, self.bias = wt, bias
        self.host_chunk = 1        # frames per sub-batch of forward_host: H2D of chunk j+1 overlaps compute of chunk j
        self.host_streams = 2      # sub-batches alternate between this many compute streams (their kernels may overlap)
        self.host_taper = True     # split the last sub-batch in two: less compute left after the last copy has landed
        self.host_slots = 2        # complete buffer sets of forward_host, used alternately: call s+1's copies overlap call s's kernels
        # The reference shuffles the points INSIDE group / group_ (Preprocessing.py:66,86), so "the first T points of a voxel"
        # is a random T-subset, redrawn every epoch. None: shuffle in training mode (forward_train), keep the caller's order in
        # inference; True / False force it. `shuffle_generator` seeds it (torch.Generator on the device); the permutation
        # applied by the last call is kept in `last_perm` (global row indices into the call's point array).
        self.shuffle = None
        self.shuffle_generator = None
        self.last_perm = None
        self.B = self.cap = 0
        self.grid_out = self.counts = None
        self.layout = {}           # workspace region name -> byte offset (region())
        self._ws = self._bws = None                # forward workspace; backward scratch of a training forward
        self._ws_key = None
        self._cml_ws = self._cml_bws = self._map_bws = None   # grown on demand (_scratch)
        self._record = None        # _Forward of the last forward
        self._param_versions = None                # (data_ptr, _version) of the parameters dropin last copied in
        self._split, self._split_key = [], None    # forward_device_split's sub-batch contexts
        self._slots, self._in_key = [], None       # forward_host's buffer sets
        self._copy_stream, self._compute_streams, self._host_calls = None, [], 0
        self._h2d_bytes = self._d2h_bytes = 0

    def _sub_context(self, f0: int, f1: int, stream=None) -> _Sub:
        """A context for frames [f0, f1) with its own workspace and outputs, sharing the grid, eps, shuffle settings and
        parameter tensors."""
        c = PointPath.__new__(PointPath)
        c._init(self.device, self.grid_spec, self.imsize_hw, self.eps, self.wt, self.bias)
        c.shuffle, c.shuffle_generator = self.shuffle, self.shuffle_generator
        return _Sub(c, f0, f1, stream)

    def load_state_dict(self, sd):
        self.load_parameters([torch.as_tensor(np.asarray(v)) if not isinstance(v, torch.Tensor) else v.detach()
                              for v in (sd[name + suffix] for name in LAYER_NAMES for suffix in ('.weight', '.bias'))])

    def load_parameters(self, params: Sequence[torch.Tensor]):
        """Copies the 16 tensors of the eight layers, checkpoint order (weight, bias per layer), into the W^T / bias tensors
        the kernels read, in place: one copy per tensor. Call under torch.no_grad() when a tensor requires grad."""
        for l, (_, cin, cout, _) in enumerate(synth.HOT_LAYERS):
            self.wt[l][:cin].copy_(params[2 * l].reshape(cout, cin).t())
            self.bias[l].copy_(params[2 * l + 1])

    def _scratch(self, buf, bytes_fn):
        """`buf`, or a new uint8 device buffer when it is missing or smaller than `bytes_fn` (a *_workspace_bytes entry of
        the library) asks for on the last forward's arguments."""
        nbytes = ctypes.c_size_t()
        check(bytes_fn(ctypes.byref(self._record.args), ctypes.byref(nbytes)), bytes_fn.__name__)
        if buf is None or buf.numel() < nbytes.value:
            buf = torch.empty(nbytes.value, dtype=torch.uint8, device=self.device)
        return buf

    # ------------------------------------------------------------------------------------------------
    def _prepare(self, B: int, cap: int, map_hw, own_outputs: bool = True, train: bool = False):
        key = (B, cap, tuple(map_hw), own_outputs, train)
        self.cap, self.B = cap, B
        if self._ws_key == key:
            return
        a = _lib.PointPathArgs()
        a.grid = self.grid
        a.B, a.cap = B, cap
        for l, (h, w) in enumerate(map_hw):
            a.map_h[l], a.map_w[l] = h, w
        a.map_c = 256
        nbytes = ctypes.c_size_t()
        check(lib.mvx_pointpath_workspace_bytes(ctypes.byref(a), ctypes.byref(nbytes)), 'pointpath_workspace_bytes')
        offs = (ctypes.c_int64 * _lib.WS_REGIONS)()
        check(lib.mvx_pointpath_layout(ctypes.byref(a), offs), 'pointpath_layout')
        self.layout = {}
        for r in range(_lib.WS_REGIONS):
            n = lib.mvx_pointpath_layout_name(r)
            if n:
                self.layout[n.decode()] = int(offs[r])
        self._bws = None
        if train:     # training workspace: + the raw output of the last FCN; backward scratch (gradient buffers)
            fwd_b, bwd_b = ctypes.c_size_t(), ctypes.c_size_t()
            check(lib.mvx_pointpath_train_workspace_bytes(ctypes.byref(a), ctypes.byref(fwd_b), ctypes.byref(bwd_b)),
                  'pointpath_train_workspace_bytes')
            nbytes = fwd_b
            self._bws = torch.empty(bwd_b.value, dtype=torch.uint8, device=self.device)
        self._ws = torch.empty(nbytes.value, dtype=torch.uint8, device=self.device)
        self._ws_key = key
        if own_outputs:
            self._alloc_outputs(B)

    def _alloc_outputs(self, B: int):
        nz, nx, ny = self.grid.shape[2], self.grid.shape[0], self.grid.shape[1]
        if self.grid_out is None or self.grid_out.shape[0] != B:
            self.grid_out = torch.empty((B, 128, nz, nx, ny), dtype=torch.float32, device=self.device)
            self.counts = torch.empty((B, 4), dtype=torch.int32, device=self.device)

    def region(self, name: str, dtype, shape):
        """Typed view into a named workspace region (tests / diagnostics)."""
        n = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
        off = self.layout[name]
        return self._ws[off:off + n].view(dtype).view(*shape)

    # ------------------------------------------------------------------------------------------------
    def forward_device(self, points: torch.Tensor, offsets: Sequence[int], calib32: torch.Tensor,
                       maps: List[torch.Tensor], want_grid: bool = True, cap: int | None = None,
                       grid_out: torch.Tensor | None = None, counts: torch.Tensor | None = None, train: bool = False,
                       point_calib: torch.Tensor | None = None, shuffle: bool | None = None,
                       calib64: torch.Tensor | None = None, calib_f64: torch.Tensor | None = None):
        """points (sum P, stride>=4) fp32 CUDA, offsets host [B+1], calib32 (B,32) CUDA, maps 3 x (B,256,Hf,Wf) CUDA.
        grid_out / counts: optional caller-owned outputs ((B,128,nz,nx,ny) fp32, (B,4) int32, contiguous).
        train=True keeps every activation for `backward` (row-first fcn1; mvx_pointpath_forward_train).
        point_calib: optional (sum P) int32 CUDA — merged point sets (GT-paste, train.py:29-42): calibration set of every
        point; calib32 is then the (n_sets, 32) table it indexes.
        calib64 (n_sets, 32) float64 CUDA + calib_f64 (n_sets) int32 CUDA: calibration sets flagged 1 are projected in fp64
        (the reference's numpy lidar2Img with readCalib's float64 matrices, train.py:36-39) and rounded to fp32 once.
        shuffle: permute every frame's points on the device first, like the in-function shuffle of the reference's `group`
        (None: `self.shuffle`, which defaults to training mode only)."""
        B = len(offsets) - 1
        if shuffle is None:
            shuffle = self.shuffle
        if shuffle is None:
            shuffle = train
        self.last_perm = None
        if shuffle and points.shape[0] > 0:
            gen = self.shuffle_generator
            perm = torch.cat([torch.randperm(int(offsets[f + 1]) - int(offsets[f]), device=points.device, generator=gen) + int(offsets[f])
                              for f in range(B)])
            points = points.index_select(0, perm)
            if point_calib is not None:
                point_calib = point_calib.index_select(0, perm).contiguous()
            self.last_perm = perm
        maxp = max(offsets[i + 1] - offsets[i] for i in range(B))
        cap = cap or max(128, (maxp + 127) // 128 * 128)
        map_hw = [(int(m.shape[-2]), int(m.shape[-1])) for m in maps]
        self._prepare(B, cap, map_hw, own_outputs=counts is None, train=train)
        if counts is not None:
            assert counts.is_contiguous() and counts.shape == (B, 4) and (grid_out is None or grid_out.is_contiguous())
            self.grid_out, self.counts = grid_out, counts
        a = _lib.PointPathArgs()
        if points.shape[0] == 0:     # all-empty batch: the kernels read no point, but the ABI wants a valid pointer
            points = torch.zeros((1, max(4, points.shape[1])), dtype=torch.float32, device=self.device)
        a.points, a.point_stride = points.data_ptr(), points.shape[1]
        off = (ctypes.c_int32 * (B + 1))(*[int(o) for o in offsets])
        a.pt_off_host = off
        a.calib32 = calib32.data_ptr()
        if point_calib is not None:
            assert point_calib.is_cuda and point_calib.dtype == torch.int32 and point_calib.is_contiguous()
            assert point_calib.numel() == offsets[-1] and calib32.dim() == 2 and calib32.shape[1] == 32
            a.point_calib = point_calib.data_ptr()
        if calib64 is not None:
            assert calib64.is_cuda and calib64.dtype == torch.float64 and calib64.is_contiguous() and calib64.shape == calib32.shape
            assert calib_f64 is not None and calib_f64.is_cuda and calib_f64.dtype == torch.int32 and calib_f64.numel() == calib32.shape[0]
            a.calib64, a.calib_f64 = calib64.data_ptr(), calib_f64.data_ptr()
        self._launch(a, (off, points, calib32, point_calib, calib64, calib_f64), maps, map_hw, want_grid, train)
        return (self.grid_out if want_grid else None), self.counts

    def _launch(self, a, keep, maps: List[torch.Tensor], map_hw, want_grid: bool, train: bool):
        """Fills the fields both entries share, runs the fused path (training variant with `train`) and records the forward."""
        a.grid = self.grid
        a.B, a.cap = self.B, self.cap
        for l in range(3):
            assert maps[l].is_cuda and maps[l].is_contiguous() and maps[l].shape[0] == self.B and maps[l].shape[1] == 256
            a.maps[l] = maps[l].data_ptr()
            a.map_h[l], a.map_w[l] = map_hw[l]
        a.map_c = 256
        a.imsize_h, a.imsize_w = self.imsize_hw
        a.gather_eps, a.bn_eps = self.eps, self.eps
        for l in range(8):
            a.wt[l] = self.wt[l].data_ptr()
            a.bias[l] = self.bias[l].data_ptr()
        a.grid_out = self.grid_out.data_ptr() if want_grid else None
        a.counts = self.counts.data_ptr()
        a.workspace, a.workspace_bytes = self._ws.data_ptr(), self._ws.numel()
        a.stream = torch.cuda.current_stream().cuda_stream
        if train:
            check(lib.mvx_pointpath_forward_train(ctypes.byref(a)), 'pointpath_forward_train')
        else:
            check(lib.mvx_pointpath_forward(ctypes.byref(a)), 'pointpath_forward')
        self._record = _Forward(a, keep, maps, train)

    # ---- the reference's own arguments: MVXNet.forward(voxels, imgs, idx, calibs, imsize) (MVXNet.py:21-27) ----------------
    def forward_voxels(self, voxels, idx, maps: List[torch.Tensor], want_grid: bool = True, train: bool = False,
                       grid_out: torch.Tensor | None = None):
        """Dense-voxel entry: `voxels` = the (1, N, T, 9) / (N, T, 9) fp32 CUDA tensor [x,y,z,dx,dy,dz,r,row,col] that
        `pre.group` + train.py:118-128 produce, `idx` = (N, 4) int64 [batch, ix, iy, iz]; or lists of B such pairs (one per
        frame, per-frame BatchNorm statistics like the batch-1 reference). maps: 3 x (B,256,Hf,Wf) CUDA.
        Stage 1 and the projection are the caller's (the reference runs them on the CPU); stages 2b-4 run here. Pad slots
        (x == y == z == 0, Pipe.py:53-54) are zeroed IN PLACE in `voxels` like featureMaping does (Pipe.py:58-59).
        Costs one device->host read of the per-frame real-slot counts (the reference's featureMaping synchronises three
        times, Pipe.py:71). Returns (grid (B,128,nz,nx,ny), counts (B,4))."""
        orig = list(voxels) if isinstance(voxels, (list, tuple)) else [voxels]
        il = list(idx) if isinstance(idx, (list, tuple)) else [idx]
        assert len(orig) == len(il)
        T = int(self.grid.T)
        vl = [v.reshape(-1, T, 9) for v in orig]              # a view when the caller's tensor is contiguous
        for v, i in zip(vl, il):
            assert v.is_cuda and v.dtype == torch.float32 and i.is_cuda and i.dtype == torch.int64 and i.shape == (v.shape[0], 4)
        B = len(vl)
        single_inplace = B == 1 and vl[0].is_contiguous() and vl[0].data_ptr() == orig[0].data_ptr()
        vcat = vl[0] if single_inplace else torch.cat(vl, dim=0).contiguous()
        icat = il[0].contiguous() if B == 1 else torch.cat(il, dim=0).contiguous()
        voff = np.concatenate([[0], np.cumsum([v.shape[0] for v in vl])]).astype(np.int64).tolist()
        voff_c = (ctypes.c_int32 * (B + 1))(*[int(o) for o in voff])
        cnt = torch.empty((B, 4), dtype=torch.int32, device=self.device)
        check(lib.mvx_dense_voxel_counts(ptr(vcat), voff_c, B, T, ptr(cnt), stream_ptr()), 'dense_voxel_counts')
        c = cnt.cpu()
        need = max(int(c[:, 1].max()), int(c[:, 0].max()), 1)
        cap = (need + 4095) // 4096 * 4096                     # capacity bucket: no re-allocation for every new frame size
        map_hw = [(int(m.shape[-2]), int(m.shape[-1])) for m in maps]
        self._prepare(B, cap, map_hw, own_outputs=grid_out is None, train=train)
        if grid_out is not None:
            assert grid_out.is_contiguous() and grid_out.dtype == torch.float32
            self.grid_out = grid_out
            if self.counts is None or self.counts.shape[0] != B:
                self.counts = torch.empty((B, 4), dtype=torch.int32, device=self.device)
        a = _lib.PointPathArgs()
        a.voxels_dense, a.voxel_idx, a.vox_off_host = vcat.data_ptr(), icat.data_ptr(), voff_c
        self._launch(a, (voff_c, vcat, icat), maps, map_hw, want_grid, train)
        if not single_inplace:                                 # the in-place side effect, for callers that handed in views / lists
            for f, v in enumerate(orig):
                v.copy_(vcat[voff[f]:voff[f + 1]].reshape(v.shape))
        return (self.grid_out if want_grid else None), self.counts

    # ---- after the path: sparse hand-off to CML.conv1 (SURVEY.md §8f rank 2) -------------------------------------
    def cml_conv1(self, weight: torch.Tensor, bias: torch.Tensor, eps: float | None = None) -> torch.Tensor:
        """`backbone.cml.conv1` = CRB3d(128, 64, 3, (2,1,1), (1,1,1)) (voxelnet/Pipe.py:31-43) of the dense grid of the LAST
        forward, computed sparsely from the voxel features (the forward may have run with want_grid=False).
        weight (64,128,3,3,3), bias (64) as in the reference checkpoint (`backbone.cml.conv1.conv.*`).
        Returns (B, 64, (nz+1)//2, nx, ny) fp32 on the GPU, per-frame BatchNorm statistics like the batch-1 reference."""
        rec = self._record
        if rec is None or rec.subs is not None:
            raise RuntimeError('cml_conv1() needs a preceding forward (device entry) on this PointPath')
        a = rec.args
        w = weight.detach().to(self.device, torch.float32).contiguous()
        b = bias.detach().to(self.device, torch.float32).contiguous()
        assert tuple(w.shape) == (64, 128, 3, 3, 3) and tuple(b.shape) == (64,)
        nz, nx, ny = self.grid.shape[2], self.grid.shape[0], self.grid.shape[1]
        self._cml_ws = self._scratch(self._cml_ws, lib.mvx_cml_conv1_workspace_bytes)
        out = torch.empty((self.B, 64, (nz + 2 - 3) // 2 + 1, nx, ny), dtype=torch.float32, device=self.device)
        a.stream = torch.cuda.current_stream().cuda_stream
        check(lib.mvx_cml_conv1_sparse(ctypes.byref(a), ptr(w), ptr(b), float(self.eps if eps is None else eps), ptr(out),
                                       ptr(self._cml_ws), self._cml_ws.numel()), 'cml_conv1_sparse')
        rec.cml_done = True
        return out

    def cml_conv1_backward(self, d_out: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, eps: float | None = None,
                           want_d_vfeat: bool = True, grads=None):
        """Backward of the last `cml_conv1` (same weight, bias, eps): d_out = dLoss/d its output (B,64,(nz+1)//2,nx,ny).
        Returns (d_vfeat, d_w, d_b): d_vfeat (B, cap, 128) = dLoss/d voxel features for `backward(d_vfeat=...)` (rows past
        each frame's voxel count are zero), or None with want_d_vfeat=False; d_w (64,128,3,3,3) and d_b (64) summed over the
        frames. grads=(d_w, d_b): add into these tensors instead of returning new ones."""
        if self._record is None or not self._record.cml_done:
            raise RuntimeError('cml_conv1_backward() needs the cml_conv1() of the latest forward on this PointPath')
        a = self._record.args
        w = weight.detach().to(self.device, torch.float32).contiguous()
        b = bias.detach().to(self.device, torch.float32).contiguous()
        nz, nx, ny = self.grid.shape[2], self.grid.shape[0], self.grid.shape[1]
        assert tuple(d_out.shape) == (self.B, 64, (nz + 2 - 3) // 2 + 1, nx, ny) and d_out.dtype == torch.float32 and d_out.is_cuda
        d_out = d_out.contiguous()
        self._cml_bws = self._scratch(self._cml_bws, lib.mvx_cml_conv1_backward_workspace_bytes)
        if grads is None:
            d_w = torch.empty((64, 128, 3, 3, 3), dtype=torch.float32, device=self.device)
            d_b = torch.empty(64, dtype=torch.float32, device=self.device)
        else:
            d_w, d_b = grads
            assert d_w.is_contiguous() and d_w.dtype == torch.float32 and tuple(d_w.shape) == (64, 128, 3, 3, 3)
            assert d_b.is_contiguous() and d_b.dtype == torch.float32 and tuple(d_b.shape) == (64,)
        d_vfeat = torch.zeros((self.B, self.cap, 128), dtype=torch.float32, device=self.device) if want_d_vfeat else None
        a.stream = torch.cuda.current_stream().cuda_stream
        check(lib.mvx_cml_conv1_sparse_backward(ctypes.byref(a), ptr(w), ptr(b), float(self.eps if eps is None else eps), ptr(d_out),
                                                ptr(d_vfeat), ptr(d_w), ptr(d_b), int(grads is not None),
                                                ptr(self._cml_ws), self._cml_ws.numel(), ptr(self._cml_bws), self._cml_bws.numel()),
              'cml_conv1_sparse_backward')
        return d_vfeat, d_w, d_b

    def cml_saved(self):
        """Read-only views of what the last `cml_conv1` saved for its backward (tests / diagnostics): act_count (B,) active
        output positions per frame, act_idx (B, Go) compact row of each position (-1: background), Yact (B, Go, 64) relu(conv)
        of the active rows (rows >= act_count unused). Mirrors the workspace layout of sparse_conv.cu (sc_layout)."""
        nz, nx, ny = self.grid.shape[2], self.grid.shape[0], self.grid.shape[1]
        B, go = self.B, ((nz + 2 - 3) // 2 + 1) * nx * ny
        sizes = [('wt', 128 * 1792 * 4), ('wpack', 2 * 128 * 1792 * 4), ('P', B * self.cap * 1792 * 4), ('act_count', B * 4),
                 ('act_idx', B * go * 4), ('yact', B * go * 64 * 4), ('stats', B * 64 * 2 * 8)]
        off, o = {}, 0
        for name, n in sizes:
            off[name] = o
            o += (n + 255) // 256 * 256
        nbytes = ctypes.c_size_t()
        check(lib.mvx_cml_conv1_workspace_bytes(ctypes.byref(self._record.args), ctypes.byref(nbytes)), 'cml_conv1_workspace_bytes')
        assert o == nbytes.value, 'cml_saved() is out of step with sc_layout'
        view = lambda name, dtype, shape: self._cml_ws[off[name]:off[name] + int(np.prod(shape)) * 4].view(dtype).view(*shape)
        return dict(act_count=view('act_count', torch.int32, (B,)), act_idx=view('act_idx', torch.int32, (B, go)),
                    Yact=view('yact', torch.float32, (B, go, 64)))

    # ---- training mode -------------------------------------------------------------------------------------
    def forward_train(self, points, offsets, calib32, maps, want_grid: bool = True, cap: int | None = None,
                      shuffle: bool | None = None):
        """Forward that keeps the activations the backward needs (BASELINE.json configs[3]). Shuffles every frame's points
        first unless `shuffle=False` / `self.shuffle = False` (the reference's `group` does, Preprocessing.py:86)."""
        return self.forward_device(points, offsets, calib32, maps, want_grid, cap, train=True, shuffle=shuffle)

    @staticmethod
    def grad_layout():
        """(name, offset, shape) of every parameter gradient inside the flat bucket: checkpoint names/order (SURVEY.md §8b)."""
        out, o = [], 0
        for name, cin, cout, is_conv in synth.HOT_LAYERS:
            out.append((name + '.weight', o, (cout, cin, 1, 1) if is_conv else (cout, cin)))
            o += cout * cin
            out.append((name + '.bias', o, (cout,)))
            o += cout
        return out

    def backward(self, d_vfeat: torch.Tensor | None = None, d_grid: torch.Tensor | None = None,
                 grad_flat: torch.Tensor | None = None, accumulate: bool = False,
                 d_maps: Sequence[torch.Tensor] | None = None) -> torch.Tensor:
        """Gradients of the 8 hot-path layers for the last forward_train call, summed over its frames, as ONE flat fp32
        bucket (the message of the NCCL all-reduce; `grad_layout()` names its slices). Give dLoss/d voxel features
        (B, cap, 128) or dLoss/d dense grid (B,128,nz,nx,ny).
        d_maps: three contiguous fp32 CUDA tensors shaped like the forward's FPN maps (B,256,H_l,W_l): they are overwritten
        with dLoss/d maps (the gradient an unfrozen image backbone receives; mvx_pointpath_backward_maps). None: no map
        gradient, and nothing beyond the parameter backward runs."""
        rec = self._record
        if rec is None or not rec.train:
            raise RuntimeError('backward() needs a preceding forward_train() on this PointPath')
        a = rec.args
        n = int(lib.mvx_grad_floats())
        if grad_flat is None:
            grad_flat = torch.empty(n, dtype=torch.float32, device=self.device)
            accumulate = False
        assert grad_flat.is_contiguous() and grad_flat.numel() == n and grad_flat.dtype == torch.float32
        for t, shape in ((d_vfeat, (self.B, self.cap, 128)), (d_grid, tuple(self.grid_out.shape) if self.grid_out is not None else None)):
            if t is not None:
                assert t.is_cuda and t.is_contiguous() and t.dtype == torch.float32 and tuple(t.shape) == shape, (tuple(t.shape), shape)
        a.stream = torch.cuda.current_stream().cuda_stream
        check(lib.mvx_pointpath_backward(ctypes.byref(a), ptr(d_vfeat), ptr(d_grid), grad_flat.data_ptr(), int(bool(accumulate)),
                                         self._bws.data_ptr(), self._bws.numel()), 'pointpath_backward')
        if d_maps is not None:
            assert len(d_maps) == len(rec.maps) == _lib.NUM_LEVELS
            for t, m in zip(d_maps, rec.maps):
                assert t.is_cuda and t.is_contiguous() and t.dtype == torch.float32 and t.shape == m.shape, (tuple(t.shape), tuple(m.shape))
            self._map_bws = self._scratch(self._map_bws, lib.mvx_pointpath_backward_maps_workspace_bytes)
            out = (ctypes.c_void_p * _lib.NUM_LEVELS)(*[t.data_ptr() for t in d_maps])
            check(lib.mvx_pointpath_backward_maps(ctypes.byref(a), self._bws.data_ptr(), self._bws.numel(), out, self._map_bws.data_ptr(),
                                                  self._map_bws.numel()), 'pointpath_backward_maps')
        return grad_flat

    def backward_saved(self):
        """Read-only view of what the last `backward` left for the map gradient (tests / diagnostics): dpre1 (B, capA, 768),
        dLoss/d fcn1's pre-activation of every compact row. Mirrors make_blayout of backward.cu (its first region)."""
        capA = self.cap + 128
        return dict(dpre1=self._bws[:self.B * capA * 768 * 4].view(torch.float32).view(self.B, capA, 768))

    def grads(self, grad_flat: torch.Tensor) -> Dict[str, torch.Tensor]:
        """Named views into a flat gradient bucket (reference state-dict names)."""
        return {name: grad_flat[o:o + int(np.prod(shape))].view(*shape) for name, o, shape in self.grad_layout()}

    def forward_device_split(self, points: torch.Tensor, offsets: Sequence[int], calib32: torch.Tensor,
                             maps: List[torch.Tensor], want_grid: bool = True, n_split: int = 2):
        """Same inputs/outputs as forward_device, but the batch is cut into `n_split` sub-batches that run CONCURRENTLY on
        their own streams and workspaces (frames are independent): the memory-bound kernels of one sub-batch (grid fill,
        combine) overlap the tensor-core kernels of the other. Joins back into the current stream."""
        B = len(offsets) - 1
        n_split = max(1, min(int(n_split), B))
        if n_split == 1:
            return self.forward_device(points, offsets, calib32, maps, want_grid)
        key = (B, n_split)
        if self._split_key != key:
            bounds = [round(i * B / n_split) for i in range(n_split + 1)]
            self._split = [self._sub_context(bounds[i], bounds[i + 1], torch.cuda.Stream(device=self.device)) for i in range(n_split)]
            self._split_key = key
        self._alloc_outputs(B)
        self.B = B
        cur = torch.cuda.current_stream()
        for s in self._split:
            p0, p1 = int(offsets[s.f0]), int(offsets[s.f1])
            s.stream.wait_stream(cur)
            with torch.cuda.stream(s.stream):
                s.path.forward_device(points[p0:p1], [int(o) - p0 for o in offsets[s.f0:s.f1 + 1]], calib32[s.f0:s.f1],
                                      [m[s.f0:s.f1] for m in maps], want_grid,
                                      grid_out=self.grid_out[s.f0:s.f1] if want_grid else None, counts=self.counts[s.f0:s.f1])
        for s in self._split:
            cur.wait_stream(s.stream)
        self._record = _Forward(subs=self._split)
        return (self.grid_out if want_grid else None), self.counts

    def __call__(self, points_list: List, calibs: List[dict], fpn_maps: List, want_grid: bool = True,
                 shuffle: bool | None = None):
        """points_list: B arrays/tensors (P_f, >=4) [x,y,z,r]; calibs: B dicts of 4x4 matrices (Load.py:24-41);
        fpn_maps: 3 tensors (B,256,Hf,Wf) (FPN levels '0','1','2').
        A frame may also be a LIST of point sets with a LIST of calibration dicts, one per set — the scene followed by the
        pasted ground-truth objects of the GT-paste augmentation, each projected through its own calibration and then
        merged in that order (train.py:29-42)."""
        def as_t(p):
            return torch.as_tensor(np.asarray(p, dtype=np.float32)) if not isinstance(p, torch.Tensor) else p
        merged = any(isinstance(c, (list, tuple)) for c in calibs)
        pts, table, pc, table64, is64 = [], [], [], [], []
        for p, c in zip(points_list, calibs):
            sets, cals = (list(p), list(c)) if isinstance(c, (list, tuple)) else ([p], [c])
            assert len(sets) == len(cals), 'one calibration per point set'
            sets = [as_t(q) for q in sets]
            pts.append(torch.cat([q[:, :4].to(torch.float32) for q in sets], dim=0))
            if merged:
                for k, (q, cal) in enumerate(zip(sets, cals)):
                    pc.append(np.full(q.shape[0], len(table), dtype=np.int32))
                    table.append(pack_calib(cal))
                    table64.append(pack_calib64(cal))
                    # train.py:31-33 projects the scene (set 0) with torch in fp32 whatever the dict holds; the pasted sets go
                    # through the numpy branch (train.py:36-39), which is fp64 when their dicts are readCalib's float64 ones
                    is64.append(1 if (k > 0 and calib_is_f64(cal)) else 0)
            else:
                table.append(pack_calib(cals[0]))
        offsets = np.concatenate([[0], np.cumsum([p.shape[0] for p in pts])]).tolist()
        points = torch.cat(pts, dim=0).contiguous().to(self.device, non_blocking=True)
        calib32 = torch.stack(table).to(self.device, non_blocking=True)
        point_calib = torch.from_numpy(np.concatenate(pc)).to(self.device, non_blocking=True) if merged else None
        c64 = f64 = None
        if merged and any(is64):
            c64 = torch.stack(table64).to(self.device)
            f64 = torch.tensor(is64, dtype=torch.int32, device=self.device)
        maps = [torch.as_tensor(m).to(self.device, torch.float32).contiguous() for m in fpn_maps]
        return self.forward_device(points, offsets, calib32, maps, want_grid, point_calib=point_calib, shuffle=shuffle,
                                   calib64=c64, calib_f64=f64)

    # ---- host-buffer entry: H2D of this batch's inputs, the fused path, D2H of the counts ---------------
    def forward_host(self, points_host: torch.Tensor, offsets: Sequence[int], calib32_host: torch.Tensor,
                     maps_host: List[torch.Tensor], want_grid: bool = True, head_rows: int = 1024, sync: bool = True):
        """Inputs in (ideally pinned) HOST memory: points (sum P, 4) fp32, calib32 (B,32), maps 3 x (B,256,Hf,Wf). The maps may
        also be CUDA tensors (the reference produces them on the GPU, Head.py:14-22): then only points + calib cross PCIe.
        Frames are independent, so the batch is cut into sub-batches of `self.host_chunk` frames: the H2D copy of
        sub-batch j+1 (copy stream) overlaps the kernels of sub-batch j (compute streams); each sub-batch has its own
        input buffers and workspace and writes its slice of the batch outputs. Reads back the per-frame counts and
        the first `head_rows` voxel feature rows of frame 0 (the host-visible result).

        Steps are pipelined ACROSS calls as well: there are `self.host_slots` (2) complete sets of input buffers,
        workspaces and outputs, used alternately, and the copies of call s+1 wait only for the kernels that last read
        the same slot (call s-1), not for call s - so while call s computes, the copy engine already moves call s+1's
        inputs. sync=True (default) waits for this call's results and returns (grid on device, counts on host, head block
        on host); sync=False returns a `HostStep` handle at once: `.wait()` blocks until the results of THAT call are in
        its pinned buffers and returns the same triple (valid until the slot is reused two calls later)."""
        dev = self.device
        B = len(offsets) - 1
        # sub-batch schedule: `host_chunk` frames per sub-batch, or an explicit list of sizes; the default tapers the tail
        # (..., 1, 1): the step ends one sub-batch of compute after the LAST copy lands, so the last sub-batch should be small
        if isinstance(self.host_chunk, (list, tuple)):
            sizes = [int(c) for c in self.host_chunk]
        else:
            chunk = max(1, min(int(self.host_chunk) or B, B))
            sizes = [chunk] * (B // chunk) + ([B % chunk] if B % chunk else [])
            if self.host_taper and chunk > 1 and len(sizes) >= 2 and sizes[-1] == chunk:
                sizes = sizes[:-1] + [chunk - chunk // 2, chunk // 2] if chunk > 2 else sizes[:-1] + [1, 1]
        assert sum(sizes) == B and all(c > 0 for c in sizes), sizes
        bounds = [0]
        for c in sizes:
            bounds.append(bounds[-1] + c)
        # contexts are keyed on capacity BUCKETS, not on the exact per-frame point counts: real sweeps differ in size from
        # call to call, and rebuilding the sub-batch contexts would re-allocate multi-GB workspaces and pinned buffers
        maxp = max([int(offsets[i + 1]) - int(offsets[i]) for i in range(B)] + [1])
        cap = (maxp + 4095) // 4096 * 4096
        stride = int(points_host.shape[1])
        n_slots = max(1, int(self.host_slots))
        key = (B, cap, stride, tuple(tuple(m.shape[1:]) + (m.is_cuda,) for m in maps_host), tuple(sizes), int(head_rows), n_slots)
        if self._in_key != key:
            self._slots = []
            for _ in range(n_slots):
                slot = _HostSlot()
                for f0, f1 in zip(bounds[:-1], bounds[1:]):
                    s = self._sub_context(f0, f1)
                    s.in_points = torch.empty(((f1 - f0) * cap, stride), dtype=torch.float32, device=dev)
                    s.in_calib = torch.empty((f1 - f0, 32), dtype=torch.float32, device=dev)
                    s.in_maps = [None if m.is_cuda else torch.empty((f1 - f0,) + tuple(m.shape[1:]), dtype=torch.float32, device=dev) for m in maps_host]
                    s.ev = torch.cuda.Event()
                    slot.subs.append(s)
                nz, nx, ny = self.grid.shape[2], self.grid.shape[0], self.grid.shape[1]
                slot.grid_out = torch.empty((B, 128, nz, nx, ny), dtype=torch.float32, device=dev) if want_grid else None
                slot.counts = torch.empty((B, 4), dtype=torch.int32, device=dev)
                slot.out_counts = torch.empty((B, 4), dtype=torch.int32).pin_memory()
                slot.out_head = torch.empty((min(int(head_rows), cap), 128), dtype=torch.float32).pin_memory()
                slot.done = torch.cuda.Event()
                self._slots.append(slot)
            self._copy_stream = torch.cuda.Stream(device=dev)
            ns = max(1, min(int(self.host_streams), len(sizes)))
            self._compute_streams = [torch.cuda.Stream(device=dev) for _ in range(ns)]
            self._host_calls = 0
            self._in_key = key
        slot = self._slots[self._host_calls % len(self._slots)]
        self._host_calls += 1
        if want_grid and slot.grid_out is None:
            nz, nx, ny = self.grid.shape[2], self.grid.shape[0], self.grid.shape[1]
            slot.grid_out = torch.empty((B, 128, nz, nx, ny), dtype=torch.float32, device=dev)
        self._h2d_bytes = (points_host.numel() + calib32_host.numel() + sum(m.numel() for m in maps_host if not m.is_cuda)) * 4
        self.B, self.grid_out, self.counts = B, slot.grid_out, slot.counts
        cur = torch.cuda.current_stream()
        cs = self._copy_stream
        ns = len(self._compute_streams)
        if slot.used:
            cs.wait_event(slot.done)             # the kernels of the call that last used this slot have read its inputs
        with torch.cuda.stream(cs):              # every copy is queued up front: the copy engine never waits for the CPU
            for s in slot.subs:
                p0, p1 = int(offsets[s.f0]), int(offsets[s.f1])
                s.offsets = [int(o) - p0 for o in offsets[s.f0:s.f1 + 1]]
                s.n_points = p1 - p0
                if p1 > p0:
                    s.in_points[:p1 - p0].copy_(points_host[p0:p1], non_blocking=True)
                s.in_calib.copy_(calib32_host[s.f0:s.f1], non_blocking=True)
                for d, h in zip(s.in_maps, maps_host):
                    if d is not None:
                        d.copy_(h[s.f0:s.f1], non_blocking=True)
                s.ev.record(cs)
        for j, s in enumerate(slot.subs):
            ks = self._compute_streams[j % ns]
            if j < ns:
                ks.wait_stream(cur)              # work the caller queued before this call (weight updates ...) is ordered first
            with torch.cuda.stream(ks):
                ks.wait_event(s.ev)
                sub_maps = [d if d is not None else h[s.f0:s.f1] for d, h in zip(s.in_maps, maps_host)]   # device-resident maps: a view
                s.path.forward_device(s.in_points[:s.n_points], s.offsets, s.in_calib, sub_maps, want_grid, cap=cap,
                                      grid_out=slot.grid_out[s.f0:s.f1] if want_grid else None, counts=slot.counts[s.f0:s.f1])
        k0 = self._compute_streams[0]
        for s_ in self._compute_streams[1:]:
            k0.wait_stream(s_)
        with torch.cuda.stream(k0):              # device -> host read of the step's result
            slot.out_counts.copy_(slot.counts, non_blocking=True)
            c0 = slot.subs[0].path
            n_head = slot.out_head.shape[0]
            slot.out_head.copy_(c0.region('vfeat', torch.float32, (c0.B, c0.cap, 128))[0, :n_head], non_blocking=True)
            slot.done.record(k0)
        slot.used = True
        cur.wait_event(slot.done)                # later work on the caller's stream sees this call's device outputs
        self._record = _Forward(subs=slot.subs)
        self._d2h_bytes = slot.out_counts.numel() * 4 + slot.out_head.numel() * 4
        step = HostStep(slot)
        return step.wait() if sync else step

    @property
    def h2d_bytes(self):
        return self._h2d_bytes

    @property
    def d2h_bytes(self):
        return self._d2h_bytes

    # ---- compact outputs (reference voxel order), for callers that do not want the dense grid -----------
    def voxel_features(self, f: int):
        """(N_f,128) fp32 features and (N_f,4) int64 idx [batch, ix, iy, iz] of frame f (after a forward)."""
        n = int(self.counts[f, 0].item())
        src, fl = self, f
        if self._record.subs is not None:          # the last forward ran in sub-batches: frame f lives in one of them
            s = next(s for s in self._record.subs if s.f0 <= f < s.f1)
            src, fl = s.path, f - s.f0
        vfeat = src.region('vfeat', torch.float32, (src.B, src.cap, 128))[fl, :n]
        coord = src.region('vox_coord', torch.int32, (src.B, src.cap, 4))[fl, :n, :3].to(torch.int64)
        idx = torch.cat([torch.full((n, 1), f, dtype=torch.int64, device=coord.device), coord], dim=1)
        return vfeat, idx
