"""ctypes binding of libd3d_b200.so (C ABI declared in include/d3d_b200.h).

This is the only place the shared library is loaded.  There is deliberately no fallback: if the
extension has not been built (`python -c "import __graft_entry__ as g; g.build()"` or
`make -C d3d_b200/csrc`) the import fails.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("D3D_B200_LIB") or os.path.join(_HERE, "libd3d_b200.so")   # override: A/B builds while tuning
if not os.path.exists(LIB_PATH):
    raise ImportError(f"{LIB_PATH} not found: build the CUDA extension first (make -C d3d_b200/csrc). "
                      "d3d_b200 has no CPU fallback.")
lib = C.CDLL(LIB_PATH)

F32, F64 = 0, 1
OK, ERR_INVALID, ERR_CUDA, ERR_WORKSPACE, ERR_UNSUPPORTED, ERR_RANGE = range(6)

_vp, _i64, _i32, _f, _sz = C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_size_t


class VoxelParams(C.Structure):
    """struct d3d_voxel_params"""
    _fields_ = [("size", C.c_float * 3), ("vlo", C.c_int64 * 3), ("vhi", C.c_int64 * 3), ("offset", C.c_int32 * 3),
                ("min_points", C.c_int32), ("max_points", C.c_int32), ("max_voxels", C.c_int32),
                ("max_points_filter", C.c_int32), ("max_voxels_filter", C.c_int32), ("bound", C.c_float * 6),
                ("shape", C.c_int32 * 3), ("reduction", C.c_int32), ("algo", C.c_int32), ("max_frame_points", C.c_int64)]


def _sig(name, restype, argtypes):
    f = getattr(lib, name)
    f.restype, f.argtypes = restype, argtypes
    return f


abi_version = _sig("d3d_abi_version", C.c_int, [])
error_string = _sig("d3d_error_string", C.c_char_p, [C.c_int])
last_cuda_error = _sig("d3d_last_cuda_error", C.c_char_p, [])
launch_count = _sig("d3d_launch_count", _i64, [])
_tuning_set = _sig("d3d_tuning_set", C.c_int, [C.c_char_p, C.c_int, C.c_int])


def tuning_set(name, value=None):
    """override (value) or clear (None) a tuning knob of the library, e.g. tuning_set("D3D_B200_NMS_PATH", 2)"""
    if _tuning_set(name.encode(), 0 if value is None else int(value), 0 if value is None else 1) != 0:
        raise ValueError(f"unknown tuning knob {name}")
iou_workspace_bytes = _sig("d3d_iou_workspace_bytes", _sz, [_i64, _i64, C.c_int])
_iou_sig = [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _sz, _vp]
iou2dr = {F32: _sig("d3d_iou2dr_f32", C.c_int, _iou_sig), F64: _sig("d3d_iou2dr_f64", C.c_int, _iou_sig)}
iou2d = {F32: _sig("d3d_iou2d_f32", C.c_int, _iou_sig), F64: _sig("d3d_iou2d_f64", C.c_int, _iou_sig)}
iou3d_distance_workspace_bytes = _sig("d3d_iou3d_distance_workspace_bytes", _sz, [_i64, _i64])
iou3d_distance = _sig("d3d_iou3d_distance_f32", C.c_int, [_vp, _i64, _vp, _i64, C.c_int, _vp, _i64, _vp, _sz, _vp])
iou3d_distance_batch_workspace_bytes = _sig("d3d_iou3d_distance_batch_workspace_bytes", _sz, [_i64, _i64, _i64])
iou3d_distance_batch = _sig("d3d_iou3d_distance_batch_f32", C.c_int, [_vp, _i64, _vp, _vp, _i64, _vp, _i64, _i64, _i64, C.c_int, _vp, _vp, _vp, _sz, _vp])
crop_workspace_bytes = _sig("d3d_crop2dr_workspace_bytes", _sz, [_i64, _i64, C.c_int])
_crop_sig = [_vp, _i64, _vp, _i64, _vp, _vp, _sz, _vp]
crop2dr = {F32: _sig("d3d_crop2dr_f32", C.c_int, _crop_sig), F64: _sig("d3d_crop2dr_f64", C.c_int, _crop_sig)}
_pd_sig = [_vp, _i64, _vp, _i64, _vp, _vp, _vp]
pdist2dr = {F32: _sig("d3d_pdist2dr_f32", C.c_int, _pd_sig), F64: _sig("d3d_pdist2dr_f64", C.c_int, _pd_sig)}
_pdb_sig = [_vp, _i64, _vp, _i64, _vp, _vp, _vp, _vp]
pdist2dr_backward = {F32: _sig("d3d_pdist2dr_backward_f32", C.c_int, _pdb_sig), F64: _sig("d3d_pdist2dr_backward_f64", C.c_int, _pdb_sig)}
crop_grid_min_pairs = _sig("d3d_crop2dr_grid_min_pairs", _i64, [])
crop_batch_workspace_bytes = _sig("d3d_crop2dr_batch_workspace_bytes", _sz, [_i64, C.c_int])
_pbb_sig = [_vp, _i64, _vp, _vp, _i64, _vp, _i64, _i64, _i64, C.c_int, _vp]   # packed points / boxes, offsets, bounds, axis, out offsets
crop2dr_batch = {k: _sig(f"d3d_crop2dr_batch_{s}", C.c_int, _pbb_sig + [_vp, _vp, _sz, _vp]) for k, s in ((F32, "f32"), (F64, "f64"))}
pdist2dr_batch = {k: _sig(f"d3d_pdist2dr_batch_{s}", C.c_int, _pbb_sig + [_vp, _vp]) for k, s in ((F32, "f32"), (F64, "f64"))}
pdist2dr_batch_backward = {k: _sig(f"d3d_pdist2dr_batch_backward_{s}", C.c_int, _pbb_sig + [_vp, _vp, _vp, _vp]) for k, s in ((F32, "f32"), (F64, "f64"))}
_iex_sig = [_vp, _i64, _vp, _i64, _vp, _i64, _vp]
giou2dr = {F32: _sig("d3d_giou2dr_f32", C.c_int, _iex_sig), F64: _sig("d3d_giou2dr_f64", C.c_int, _iex_sig)}
diou2dr = {F32: _sig("d3d_diou2dr_f32", C.c_int, _iex_sig), F64: _sig("d3d_diou2dr_f64", C.c_int, _iex_sig)}
_ibw_sig = [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _vp, _vp]
iou_backward = {name: {F32: _sig(f"d3d_{name}_backward_f32", C.c_int, _ibw_sig), F64: _sig(f"d3d_{name}_backward_f64", C.c_int, _ibw_sig)}
                for name in ("iou2d", "iou2dr", "giou2dr", "diou2dr")}
match_greedy = _sig("d3d_match_greedy_f32", C.c_int, [_vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp])
match_greedy_batch = _sig("d3d_match_greedy_batch_f32", C.c_int, [_vp, _vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp])
iou_count_candidates = _sig("d3d_iou_count_candidates", C.c_int, [_vp, _i64, _vp, _i64, C.c_int, _vp, _vp, _sz, _vp])
nms_workspace_bytes = _sig("d3d_nms2d_workspace_bytes", _sz, [_i64, C.c_int])
_nms_sig = [_vp, _vp, _i64, C.c_int, C.c_int, _f, _f, _f, _vp, _vp, _sz, _vp]
nms2d = {F32: _sig("d3d_nms2d_f32", C.c_int, _nms_sig), F64: _sig("d3d_nms2d_f64", C.c_int, _nms_sig)}
nms_batch_workspace_bytes = _sig("d3d_nms2d_batch_workspace_bytes", _sz, [_i64, _i64, _i64, C.c_int])
_nmsb_sig = [_vp, _vp, _i64, _vp, _i64, _i64, C.c_int, C.c_int, _f, _f, _vp, _vp, _sz, _vp]
nms2d_batch = {F32: _sig("d3d_nms2d_batch_f32", C.c_int, _nmsb_sig), F64: _sig("d3d_nms2d_batch_f64", C.c_int, _nmsb_sig)}
nms_batch_soft_workspace_bytes = _sig("d3d_nms2d_batch_soft_workspace_bytes", _sz, [_i64, _i64, _i64, C.c_int])
_nmsbs_sig = [_vp, _vp, _i64, _vp, _i64, _i64, C.c_int, C.c_int, _f, _f, _f, _vp, _vp, _sz, _vp]
nms2d_batch_soft = {F32: _sig("d3d_nms2d_batch_soft_f32", C.c_int, _nmsbs_sig), F64: _sig("d3d_nms2d_batch_soft_f64", C.c_int, _nmsbs_sig)}
voxelize_workspace_bytes = _sig("d3d_voxelize_workspace_bytes", _sz, [_i64, _i64, _i64])
voxelize_sparse = _sig("d3d_voxelize_sparse_f32", C.c_int,
                       [_vp, _i64, _i32, _vp, _i64, C.POINTER(VoxelParams), _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp])
voxelize_dense = _sig("d3d_voxelize_dense_f32", C.c_int,
                      [_vp, _i64, _i32, _vp, _i64, C.POINTER(VoxelParams), _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp])
_sc_sig = [_vp, _i64, _i32, _vp, _i64, _i64, C.POINTER(C.c_int64), C.c_int, C.c_int, _vp, _vp]
scatter_forward = _sig("d3d_aligned_scatter_forward", C.c_int, _sc_sig)
scatter_backward = _sig("d3d_aligned_scatter_backward", C.c_int, _sc_sig)
_scw_sig = _sc_sig[:-1] + [_vp, _sz, C.c_int, _vp]
scatter_workspace_bytes = _sig("d3d_aligned_scatter_workspace_bytes", _sz, [_i64, _i32, _i64, C.POINTER(C.c_int64)])
scatter_forward_ws = _sig("d3d_aligned_scatter_forward_ws", C.c_int, _scw_sig)
scatter_backward_ws = _sig("d3d_aligned_scatter_backward_ws", C.c_int, _scw_sig)
fma_peak_probe = _sig("d3d_fma_peak_probe", C.c_int, [C.c_int, _i64, _vp, C.POINTER(C.c_double), _vp])

if abi_version() != 5:
    raise ImportError("libd3d_b200.so ABI version mismatch")


def check(status, what):
    """Map a d3d_status to the Python exception the reference raises for the same problem."""
    if status == OK:
        return
    msg = f"{what}: {error_string(status).decode()}"
    if status == ERR_CUDA:
        raise RuntimeError(msg + f" ({last_cuda_error().decode()})")
    if status == ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    if status in (ERR_INVALID, ERR_RANGE):
        raise ValueError(msg)
    raise RuntimeError(msg)


def require_cuda():
    if not torch.cuda.is_available():
        raise RuntimeError("d3d_b200 needs a CUDA device (sm_100a); there is no CPU fallback")


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def workspace(nbytes, device):
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


def dtype_code(dt):
    if dt == torch.float32:
        return F32
    if dt == torch.float64:
        return F64
    raise RuntimeError(f"expected a float32 or float64 tensor, got {dt}")  # ATen accessor error in the reference


def to_device(t):
    """Inputs may live on the host (the reference voxelizer is CPU-only): stage them on the current
    CUDA device; outputs are returned on the device the inputs came from."""
    require_cuda()
    if t.is_cuda:
        return t.contiguous()
    return t.contiguous().to("cuda", non_blocking=True)
