"""ctypes binding of the C-ABI library ``libmvx_b200.so`` (include/mvx_b200.h).

PyTorch is used only for device memory and streams; every compute call goes through the C ABI with raw
pointers. There is no CPU fallback: if the library is missing the import of this module raises, and every
compute entry point returns MVX_ECUDA without a CUDA device.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import sys
from ctypes import POINTER, c_char_p, c_double, c_float, c_int32, c_int64, c_size_t, c_void_p

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
LIB_PATH = os.environ.get('MVX_B200_LIB') or os.path.join(_PKG, 'libmvx_b200.so')   # the override serves A/B builds in tools/; bench.py refuses MVX_* variables

NUM_LAYERS = 8
NUM_LEVELS = 3
WS_REGIONS = 64
NUM_SEGMENTS = 20
DTYPE_F32, DTYPE_F16, DTYPE_BF16 = 0, 1, 2     # MVX_DTYPE_*: element types of a dense grid

# every symbol include/mvx_b200.h declares (tests check that the .so exports all of them)
EXPORTS = [
    'mvx_last_error', 'mvx_version', 'mvx_launch_count',
    'mvx_voxelize_workspace_bytes', 'mvx_voxelize', 'mvx_group_emit7', 'mvx_group_emit9',
    'mvx_crop_workspace_bytes', 'mvx_crop_points', 'mvx_crop_points_f64',
    'mvx_lidar2img', 'mvx_lidar2img_f64', 'mvx_dense_voxel_counts', 'mvx_maps_nhwc_bytes', 'mvx_feature_mapping',
    'mvx_set_gemm_mode', 'mvx_layer_workspace_bytes', 'mvx_fcn_forward', 'mvx_vfe_forward', 'mvx_fcn_max_forward', 'mvx_scatter_dense',
    'mvx_scatter_dense_typed', 'mvx_scatter_dense_backward_typed',
    'mvx_feature_mapping_backward_workspace_bytes', 'mvx_feature_mapping_backward', 'mvx_fcn_forward_train', 'mvx_vfe_forward_train',
    'mvx_fcn_max_forward_train', 'mvx_fcn_backward_workspace_bytes', 'mvx_vfe_backward_workspace_bytes',
    'mvx_fcn_max_backward_workspace_bytes', 'mvx_fcn_backward', 'mvx_vfe_backward', 'mvx_fcn_max_backward', 'mvx_scatter_dense_backward',
    'mvx_pointpath_workspace_bytes', 'mvx_pointpath_layout', 'mvx_pointpath_layout_name', 'mvx_pointpath_forward',
    'mvx_set_fusion_mode', 'mvx_set_fold_mode', 'mvx_pointpath_train_workspace_bytes', 'mvx_pointpath_forward_train', 'mvx_grad_floats',
    'mvx_pointpath_backward', 'mvx_pointpath_backward_maps_workspace_bytes', 'mvx_pointpath_backward_maps', 'mvx_cml_conv1_workspace_bytes', 'mvx_cml_conv1_sparse',
    'mvx_cml_conv1_backward_workspace_bytes', 'mvx_cml_conv1_sparse_backward',
    'mvx_bbox_pairwise', 'mvx_classify_anchors_workspace_bytes', 'mvx_classify_anchors',
    'mvx_timing_enable', 'mvx_timing_read', 'mvx_timing_segment_name',
]


class Grid(ctypes.Structure):
    _fields_ = [('range_lo', c_double * 3), ('voxel_size', c_double * 3), ('shape', c_int32 * 3), ('T', c_int32)]


class VoxelOut(ctypes.Structure):
    _fields_ = [('counts', c_void_p), ('vox_coord', c_void_p), ('vox_cnt', c_void_p), ('vox_row0', c_void_p),
                ('row_point', c_void_p), ('row_vox', c_void_p), ('cell2vid', c_void_p)]


class PointPathArgs(ctypes.Structure):
    _fields_ = [('grid', Grid), ('B', c_int32), ('cap', c_int32), ('points', c_void_p), ('point_stride', c_int32),
                ('pt_off_host', POINTER(c_int32)), ('calib32', c_void_p), ('maps', c_void_p * NUM_LEVELS),
                ('map_h', c_int32 * NUM_LEVELS), ('map_w', c_int32 * NUM_LEVELS), ('map_c', c_int32),
                ('imsize_h', c_float), ('imsize_w', c_float), ('gather_eps', c_float), ('bn_eps', c_double),
                ('wt', c_void_p * NUM_LAYERS), ('bias', c_void_p * NUM_LAYERS), ('grid_out', c_void_p),
                ('counts', c_void_p), ('workspace', c_void_p), ('workspace_bytes', c_size_t), ('stream', c_void_p),
                ('point_calib', c_void_p), ('calib64', c_void_p), ('calib_f64', c_void_p),
                ('voxels_dense', c_void_p), ('voxel_idx', c_void_p), ('vox_off_host', POINTER(c_int32)), ('grid_dtype', c_int32)]


def make_grid(velorange, voxelsize, voxelshape, T) -> Grid:
    g = Grid()
    for i in range(3):
        g.range_lo[i] = float(velorange[i])
        g.voxel_size[i] = float(voxelsize[i])
        g.shape[i] = int(voxelshape[i])
    g.T = int(T)
    return g


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f'{LIB_PATH} is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` '
            '(nvcc, sm_100a). mvxnet_makise_b200 has no CPU fallback.')
    lib = ctypes.CDLL(LIB_PATH)
    vp, i32, i64 = c_void_p, c_int32, c_int64
    lib.mvx_last_error.restype = c_char_p
    lib.mvx_version.restype = i32
    lib.mvx_launch_count.restype = i64
    lib.mvx_voxelize_workspace_bytes.argtypes = [i32, i32, POINTER(c_size_t)]
    lib.mvx_voxelize.argtypes = [POINTER(Grid), i32, i32, vp, i32, POINTER(i32), vp, i32, POINTER(VoxelOut), vp, c_size_t, vp]
    lib.mvx_group_emit7.argtypes = [vp, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.mvx_group_emit9.argtypes = [vp, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.mvx_crop_workspace_bytes.argtypes = [i32, i64, i64, POINTER(c_size_t)]
    lib.mvx_crop_points.argtypes = [vp, i32, i32, POINTER(i32), POINTER(c_double), vp, c_double, c_double, vp, vp, vp, c_size_t, vp]
    lib.mvx_lidar2img.argtypes = [vp, i32, i64, vp, vp, vp]
    lib.mvx_lidar2img_f64.argtypes = [vp, i32, i64, vp, vp, vp]
    lib.mvx_crop_points_f64.argtypes = [vp, i32, i32, POINTER(i32), POINTER(c_double), vp, c_double, c_double, vp, vp, vp, c_size_t, vp]
    lib.mvx_dense_voxel_counts.argtypes = [vp, POINTER(i32), i32, i32, vp, vp]
    lib.mvx_maps_nhwc_bytes.argtypes = [POINTER(i32), POINTER(i32), i32, POINTER(c_size_t)]
    lib.mvx_feature_mapping.argtypes = [vp, i64, POINTER(vp), POINTER(i32), POINTER(i32), i32, c_float, c_float, c_float,
                                        vp, vp, c_size_t, vp]
    lib.mvx_set_gemm_mode.argtypes = [i32]
    lib.mvx_layer_workspace_bytes.argtypes = [i32, i32, POINTER(c_size_t)]
    lib.mvx_fcn_forward.argtypes = [vp, i64, i32, vp, vp, i32, c_double, vp, vp, vp]
    lib.mvx_vfe_forward.argtypes = [vp, i64, i32, i32, vp, vp, i32, c_double, vp, vp, vp, vp]
    lib.mvx_fcn_max_forward.argtypes = [vp, i64, i32, i32, vp, vp, i32, c_double, vp, vp, vp, vp]
    lib.mvx_scatter_dense.argtypes = [vp, vp, i64, i32, i32, i32, i32, vp, vp, vp]
    lib.mvx_scatter_dense_typed.argtypes = [vp, vp, i64, i32, i32, i32, i32, vp, i32, vp, vp]
    lib.mvx_feature_mapping_backward_workspace_bytes.argtypes = [i64, POINTER(i32), POINTER(i32), POINTER(c_size_t)]
    lib.mvx_feature_mapping_backward.argtypes = [vp, i64, vp, POINTER(i32), POINTER(i32), i32, c_float, c_float, c_float, POINTER(vp),
                                                 vp, c_size_t, vp]
    lib.mvx_fcn_forward_train.argtypes = [vp, i64, i32, vp, vp, i32, c_double, vp, vp, vp, vp]
    lib.mvx_vfe_forward_train.argtypes = [vp, i64, i32, i32, vp, vp, i32, c_double, vp, vp, vp, vp, vp]
    lib.mvx_fcn_max_forward_train.argtypes = [vp, i64, i32, i32, vp, vp, i32, c_double, vp, vp, vp, vp, vp]
    lib.mvx_fcn_backward_workspace_bytes.argtypes = [i64, i32, i32, POINTER(c_size_t)]
    lib.mvx_vfe_backward_workspace_bytes.argtypes = [i64, i32, i32, i32, POINTER(c_size_t)]
    lib.mvx_fcn_max_backward_workspace_bytes.argtypes = [i64, i32, i32, i32, POINTER(c_size_t)]
    lib.mvx_fcn_backward.argtypes = [vp, i64, i32, vp, i32, vp, vp, c_double, vp, vp, vp, vp, i32, vp, c_size_t, vp]
    lib.mvx_vfe_backward.argtypes = [vp, i64, i32, i32, vp, i32, vp, vp, c_double, vp, vp, vp, vp, i32, vp, c_size_t, vp]
    lib.mvx_fcn_max_backward.argtypes = [vp, i64, i32, i32, vp, i32, vp, vp, c_double, vp, vp, vp, vp, i32, vp, c_size_t, vp]
    lib.mvx_scatter_dense_backward.argtypes = [vp, vp, i64, i32, i32, i32, i32, vp, vp]
    lib.mvx_scatter_dense_backward_typed.argtypes = [vp, i32, vp, i64, i32, i32, i32, i32, vp, vp]
    lib.mvx_pointpath_workspace_bytes.argtypes = [POINTER(PointPathArgs), POINTER(c_size_t)]
    lib.mvx_pointpath_layout.argtypes = [POINTER(PointPathArgs), POINTER(i64)]
    lib.mvx_pointpath_layout_name.argtypes = [i32]
    lib.mvx_pointpath_layout_name.restype = c_char_p
    lib.mvx_pointpath_forward.argtypes = [POINTER(PointPathArgs)]
    lib.mvx_set_fusion_mode.argtypes = [i32]
    lib.mvx_set_fold_mode.argtypes = [i32]
    lib.mvx_pointpath_train_workspace_bytes.argtypes = [POINTER(PointPathArgs), POINTER(c_size_t), POINTER(c_size_t)]
    lib.mvx_pointpath_forward_train.argtypes = [POINTER(PointPathArgs)]
    lib.mvx_grad_floats.restype = i64
    lib.mvx_cml_conv1_workspace_bytes.argtypes = [POINTER(PointPathArgs), POINTER(c_size_t)]
    lib.mvx_cml_conv1_sparse.argtypes = [POINTER(PointPathArgs), vp, vp, c_double, vp, vp, c_size_t]
    lib.mvx_cml_conv1_backward_workspace_bytes.argtypes = [POINTER(PointPathArgs), POINTER(c_size_t)]
    lib.mvx_cml_conv1_sparse_backward.argtypes = [POINTER(PointPathArgs), vp, vp, c_double, vp, vp, vp, vp, i32, vp, c_size_t, vp, c_size_t]
    lib.mvx_pointpath_backward.argtypes = [POINTER(PointPathArgs), vp, vp, vp, i32, vp, c_size_t]
    lib.mvx_pointpath_backward_maps_workspace_bytes.argtypes = [POINTER(PointPathArgs), POINTER(c_size_t)]
    lib.mvx_pointpath_backward_maps.argtypes = [POINTER(PointPathArgs), vp, c_size_t, POINTER(vp), vp, c_size_t]
    lib.mvx_bbox_pairwise.argtypes = [vp, i64, vp, i64, i32, vp, vp]
    lib.mvx_classify_anchors_workspace_bytes.argtypes = [i64, i64, i64, i32, POINTER(c_size_t)]
    lib.mvx_classify_anchors.argtypes = [vp, i64, vp, i64, i64, i32, vp, vp, c_float, c_float, vp, vp, vp, i64, vp, vp, c_size_t, vp]
    lib.mvx_timing_enable.argtypes = [i32]
    lib.mvx_timing_read.argtypes = [i32, POINTER(c_float)]
    lib.mvx_timing_segment_name.argtypes = [i32]
    lib.mvx_timing_segment_name.restype = c_char_p
    for name in EXPORTS:
        fn = getattr(lib, name)
        if fn.restype is ctypes.c_int:   # default restype: the int status code
            fn.restype = i32
    return lib


lib = _load()

ERRORS = {-1: 'MVX_EINVAL', -2: 'MVX_ECUDA', -3: 'MVX_ESPACE', -4: 'MVX_ERANGE'}


def check(rc: int, what: str = ''):
    if rc != 0:
        msg = lib.mvx_last_error().decode('utf-8', 'replace')
        raise RuntimeError(f'mvx_b200 {what} failed: {ERRORS.get(rc, rc)}: {msg}')


def grid_dtype_code(dtype) -> int:
    """MVX_DTYPE_* of a dense grid's torch dtype: torch.float32, torch.float16 or torch.bfloat16; ValueError otherwise."""
    import torch
    codes = {torch.float32: DTYPE_F32, torch.float16: DTYPE_F16, torch.bfloat16: DTYPE_BF16}
    if not isinstance(dtype, torch.dtype) or dtype not in codes:
        raise ValueError(f'grid dtype must be torch.float32, torch.float16 or torch.bfloat16, not {dtype!r}')
    return codes[dtype]


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError('mvxnet_makise_b200 needs a CUDA device (sm_100a); there is no CPU fallback')


def stream_ptr():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t) -> c_void_p:
    return c_void_p(t.data_ptr()) if t is not None else c_void_p(0)


c_float = c_float  # re-export for callers building timing buffers


def set_gemm_mode(mode: int):
    """0 = exact-fp32 SIMT layers everywhere, 1 = tcgen05 layers (default): 3xFP16 operands for the fused path's BatchNorm-ed /
    row-scaled inputs, 3xTF32 for the dense layer API, conv1 / fcn2 / last FCN in the TMA-fed A-from-TMEM persistent kernel
    (tc3_layer.cu), 5 = like 1 with the one-tile kernel for those layers, and the dense layer API also uses fp16 operands (inputs
    must be O(1)), 6 = bf16 mode (single-pass bf16 operands for the layers mode 1 runs in 3xFP16; reduced precision), 9 = like 1
    with the one-tile kernel of tc_layer.cu for conv1 / fcn2 / last FCN (A/B timing), 10 = like 1 with the VFE inputs materialised
    by prep_vfe1 / prep_vfe2 as in training, 12 = like 1 with the one-tile kernel for the per-pixel GEMM of fcn1 instead of the
    persistent one (A/B timing). Any other number raises: 2, 3, 4, 7 and 8 selected variants that have been removed."""
    check(lib.mvx_set_gemm_mode(int(mode)), 'set_gemm_mode')


def set_fold_mode(mode: int):
    """0 = the run-structured combine kernel (default), 2 = its first, row-by-row version (A/B runs)."""
    check(lib.mvx_set_fold_mode(int(mode)), 'set_fold_mode')


def set_fusion_mode(mode: int):
    """1 = pixel-first fcn1 (per-pixel tensor-core GEMM + 12-corner combine; default), 0 = row-first (gather the
    (K,768) matrix, then fcn1 over the point rows)."""
    check(lib.mvx_set_fusion_mode(int(mode)), 'set_fusion_mode')


def launch_count() -> int:
    return int(lib.mvx_launch_count())
