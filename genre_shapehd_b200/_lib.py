"""ctypes binding of libgenre_b200.so (the C ABI in include/genre_b200.h).

This module is the only place that knows the ABI.  Loading fails loudly: there is no fallback path.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libgenre_b200.so")

FLAG_SHIFT_TDF = 1

_i64 = ctypes.c_int64
_int = ctypes.c_int
_uint = ctypes.c_uint
_ptr = ctypes.c_void_p
_size = ctypes.c_size_t
_f32 = ctypes.c_float

# name -> argument types, in include/genre_b200.h order
_SIGNATURES = {
    "genre_b200_cam_bp_forward": [_ptr] + [_i64] * 8 + [_ptr, _i64, _i64, _ptr, _i64, _i64, _ptr, _ptr, _int, _uint,
                                                       _ptr, _size, _ptr],
    "genre_b200_cam_bp_backward": [_ptr] + [_i64] * 8 + [_ptr, _i64, _i64, _ptr, _i64, _i64, _ptr, _ptr, _int, _ptr,
                                                        _ptr, _ptr, _ptr],
    "genre_b200_surface_mask": [_ptr] + [_i64] * 8 + [_ptr, _i64, _i64, _ptr, _i64, _i64, _ptr, _ptr, _int, _ptr],
    "genre_b200_sph_bp_forward": [_ptr] + [_i64] * 8 + [_ptr] + [_i64] * 5 + [_ptr, _ptr, _int, _ptr, _size, _ptr],
    "genre_b200_sph_bp_backward": [_ptr] + [_i64] * 8 + [_ptr] + [_i64] * 5 + [_ptr, _ptr, _int, _ptr, _ptr],
    "genre_b200_calc_prob_forward": [_ptr, _ptr, _i64, _i64, _ptr],
    "genre_b200_calc_prob_backward": [_ptr, _ptr, _ptr, _i64, _i64, _ptr],
    "genre_b200_render_spherical_forward": [_ptr, _i64, _int, _ptr, _int, _int, _ptr, _ptr, _ptr],
    "genre_b200_render_spherical_backward": [_ptr, _i64, _int, _ptr, _int, _int, _ptr, _ptr, _ptr, _ptr],
    "genre_b200_nnd_forward": [_ptr, _ptr, _i64, _i64, _i64, _ptr, _ptr, _ptr, _ptr, _ptr],
    "genre_b200_nnd_backward": [_ptr, _ptr, _i64, _i64, _i64, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr],
    "genre_b200_convt3d_s2_forward": [_ptr, _int, _ptr, _int, _i64, _i64, _i64, _i64, _ptr, _int, _int, _int, _ptr, _ptr,
                                      _f32, _ptr, _int, _ptr],
    "genre_b200_conv3d_taps_forward": [_ptr, _int, _ptr, _int, _i64, _i64, _i64, _i64, _ptr, _int, _int, _int, _int, _ptr,
                                       _ptr, _f32, _ptr, _int, _ptr],
    "genre_b200_convt_c1_forward": [_ptr, _int, _ptr, _int, _i64, _i64, _i64, _i64, _ptr, _f32, _int, _ptr, _ptr],
    "genre_b200_conv3d_k4s2_forward": [_ptr, _int, _int, _i64, _i64, _i64, _i64, _ptr, _int, _int, _ptr, _ptr, _f32, _ptr, _int,
                                       _ptr],
    "genre_b200_blocked_split3": [_ptr, _int, _i64, _i64, _i64, _ptr, _ptr],
    "genre_b200_convt3d_s2_merged_forward": [_ptr, _int, _ptr, _int, _i64, _i64, _i64, _i64, _ptr, _int, _int, _int, _ptr,
                                             _ptr, _f32, _ptr, _int, _ptr],
    "genre_b200_conv3d_k8s2_s4d_forward": [_ptr, _int, _i64, _i64, _i64, _i64, _ptr, _int, _int, _ptr, _ptr, _f32, _ptr,
                                           _int, _ptr],
    "genre_b200_convt_c1_tc_forward": [_ptr, _int, _ptr, _int, _i64, _i64, _i64, _i64, _ptr, _int, _ptr, _int, _ptr, _ptr],
    "genre_b200_blocked_f32_to_f16": [_ptr, _int, _i64, _i64, _i64, _ptr, _ptr],
    "genre_b200_blocked_split2_f16": [_ptr, _int, _i64, _i64, _i64, _ptr, _ptr],
    "genre_b200_voxel_surface": [_ptr, _i64, _int, _int, _int, _ptr, _ptr, _size, _ptr],
    "genre_b200_convt_c1_col2im_forward": [_ptr, _int, _ptr, _int, _i64, _i64, _i64, _i64, _ptr, _int, _ptr, _ptr, _ptr],
    "genre_b200_skinny_gemm": [_ptr, _ptr, _i64, _i64, _i64, _int, _int, _ptr, _ptr, _f32, _ptr, _ptr, _size, _ptr],
    "genre_b200_convflat_pack": [_ptr, _int, _i64, _int, _int, _int, _int, _ptr, _int, _int, _int, _int, _ptr],
    "genre_b200_convflat_forward": [_ptr, _int, _i64, _int, _int, _int, _int, _ptr, _int, _int, _ptr, _ptr, _f32, _ptr, _int, _ptr],
    "genre_b200_render_spherical_forward_pre": [_ptr, _i64, _int, _ptr, _int, _int, _ptr, _f32, _f32, _f32, _ptr, _ptr],
    "genre_b200_render_spherical_forward_skip": [_ptr, _i64, _int, _ptr, _int, _int, _ptr, _int, _f32, _f32, _f32, _ptr, _ptr, _size,
                                                 _ptr],
    "genre_b200_sph_bp_forward_fused": [_ptr] + [_i64] * 8 + [_ptr] + [_i64] * 5 + [_f32, _f32, _ptr, _i64, _int, _ptr,
                                                                                       _size, _ptr],
    "genre_b200_scale_clamp_strided": [_ptr, _i64, _i64, _f32, _f32, _f32, _ptr, _i64, _ptr],
    "genre_b200_convt_c1_wgrad": [_ptr, _ptr, _i64, _i64, _i64, _i64, _i64, _ptr, _ptr, _size, _ptr],
    "genre_b200_convt_c1_dgrad": [_ptr, _ptr, _i64, _i64, _i64, _i64, _i64, _ptr, _ptr],
    "genre_b200_conv_k8s2_wgrad": [_ptr, _ptr, _i64, _i64, _i64, _i64, _i64, _i64, _ptr, _ptr, _size, _ptr],
    "genre_b200_bn_act_train_forward": [_ptr, _i64, _i64, _i64, _ptr, _ptr, _ptr, _ptr, _f32, _f32, _f32, _ptr, _ptr, _ptr, _ptr,
                                        _size, _ptr],
    "genre_b200_bn_act_train_backward": [_ptr, _ptr, _i64, _i64, _i64, _ptr, _ptr, _ptr, _ptr, _f32, _ptr, _ptr, _ptr, _ptr,
                                         _size, _ptr],
    "genre_b200_ncdhw_to_blocked": [_ptr, _i64, _i64, _i64, _i64, _i64, _int, _int, _int, _ptr, _ptr],
    "genre_b200_blocked_to_ncdhw": [_ptr, _int, _i64, _i64, _i64, _i64, _i64, _ptr, _ptr],
    "genre_b200_cam_bp_stage_project": [_ptr] + [_i64] * 8 + [_ptr, _i64, _i64, _ptr, _i64, _i64, _int, _ptr, _size,
                                                             _ptr],
    "genre_b200_voxelize_stage_splat": [_i64, _i64, _int, _ptr, _ptr, _f32, _f32, _f32, _ptr, _size, _ptr],
    "genre_b200_iso_surface_count": [_ptr, _i64, _int, _int, _int, _f32, _ptr, _size, _ptr, _ptr],
    "genre_b200_iso_surface_emit": [_ptr, _i64, _int, _int, _int, _f32] + [_f32] * 6 + [_ptr, _ptr, _ptr, _ptr, _ptr, _size,
                                                                                         _ptr],
}

# every symbol include/genre_b200.h declares (tests check the library exports all of them)
EXPORTED_SYMBOLS = sorted(list(_SIGNATURES) + [
    "genre_b200_last_error", "genre_b200_version", "genre_b200_voxelize_workspace_bytes",
    "genre_b200_convt_c1_wgrad_workspace_bytes", "genre_b200_conv_k8s2_wgrad_workspace_bytes",
    "genre_b200_bn_workspace_bytes", "genre_b200_render_spherical_workspace_bytes",
    "genre_b200_voxel_surface_workspace_bytes", "genre_b200_convflat_positions", "genre_b200_skinny_gemm_workspace_bytes",
    "genre_b200_iso_surface_workspace_bytes"])

_lib = None
launch_count = 0  # kernels of this library enqueued through the binding (bench.py reports it as gpu_launches)

# how many of this library's KERNELS one call of each entry point launches (memset nodes not counted)
_LAUNCHES = {
    "genre_b200_cam_bp_forward": 2, "genre_b200_cam_bp_backward": 1, "genre_b200_surface_mask": 1,
    "genre_b200_sph_bp_forward": 2, "genre_b200_sph_bp_backward": 1, "genre_b200_calc_prob_forward": 1,
    "genre_b200_calc_prob_backward": 1, "genre_b200_render_spherical_forward": 1,
    "genre_b200_render_spherical_backward": 1, "genre_b200_nnd_forward": 1, "genre_b200_nnd_backward": 1,
    "genre_b200_cam_bp_stage_project": 1, "genre_b200_voxelize_stage_splat": 1,
    "genre_b200_convt3d_s2_forward": 1, "genre_b200_conv3d_taps_forward": 1,
    "genre_b200_convt_c1_forward": 1, "genre_b200_conv3d_k4s2_forward": 1,
    "genre_b200_render_spherical_forward_pre": 1, "genre_b200_render_spherical_forward_skip": 2, "genre_b200_sph_bp_forward_fused": 2, "genre_b200_scale_clamp_strided": 1,
    "genre_b200_bn_act_train_forward": 3, "genre_b200_bn_act_train_backward": 2, "genre_b200_conv_k8s2_wgrad": 2, "genre_b200_convt_c1_wgrad": 2, "genre_b200_convt_c1_dgrad": 1,
    "genre_b200_blocked_split3": 1, "genre_b200_blocked_split2_f16": 1, "genre_b200_voxel_surface": 2, "genre_b200_convt_c1_col2im_forward": 1, "genre_b200_skinny_gemm": 2, "genre_b200_convflat_pack": 1, "genre_b200_convflat_forward": 1, "genre_b200_convt_c1_tc_forward": 1, "genre_b200_blocked_f32_to_f16": 1,
    "genre_b200_convt3d_s2_merged_forward": 1, "genre_b200_conv3d_k8s2_s4d_forward": 1, "genre_b200_ncdhw_to_blocked": 1, "genre_b200_blocked_to_ncdhw": 1,
    "genre_b200_iso_surface_count": 3, "genre_b200_iso_surface_emit": 1,
}


def load():
    """Load the shared library once; raise (never fall back) if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libgenre_b200.so not found at %s: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C genre_shapehd_b200/csrc`. There is no CPU or PyTorch fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, argtypes in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = _int
    lib.genre_b200_last_error.restype = ctypes.c_char_p
    lib.genre_b200_last_error.argtypes = []
    lib.genre_b200_version.restype = _int
    lib.genre_b200_voxelize_workspace_bytes.restype = _size
    lib.genre_b200_voxelize_workspace_bytes.argtypes = [_i64, _i64, _int]
    lib.genre_b200_convt_c1_wgrad_workspace_bytes.restype = _size
    lib.genre_b200_convt_c1_wgrad_workspace_bytes.argtypes = [_int]
    lib.genre_b200_conv_k8s2_wgrad_workspace_bytes.restype = _size
    lib.genre_b200_conv_k8s2_wgrad_workspace_bytes.argtypes = []
    lib.genre_b200_bn_workspace_bytes.restype = _size
    lib.genre_b200_bn_workspace_bytes.argtypes = [_i64]
    lib.genre_b200_render_spherical_workspace_bytes.restype = _size
    lib.genre_b200_render_spherical_workspace_bytes.argtypes = [_i64, _int]
    lib.genre_b200_skinny_gemm_workspace_bytes.restype = _size
    lib.genre_b200_skinny_gemm_workspace_bytes.argtypes = [_i64, _i64, _i64, _int]
    lib.genre_b200_convflat_positions.restype = _i64
    lib.genre_b200_convflat_positions.argtypes = [_i64, _int, _int, _int, ctypes.POINTER(ctypes.c_int)]
    lib.genre_b200_voxel_surface_workspace_bytes.restype = _size
    lib.genre_b200_voxel_surface_workspace_bytes.argtypes = [_i64, _int]
    lib.genre_b200_iso_surface_workspace_bytes.restype = _size
    lib.genre_b200_iso_surface_workspace_bytes.argtypes = [_i64, _int, _int, _int]
    _lib = lib
    return lib


def call(name, *args):
    """Invoke an entry point; non-zero status -> RuntimeError (the reference's THError("aborting"))."""
    global launch_count
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        msg = lib.genre_b200_last_error()
        raise RuntimeError("%s failed (status %d): %s" % (name, rc, msg.decode() if msg else "?"))
    launch_count += _LAUNCHES.get(name, 0)


def stream_ptr(t):
    """the current stream of the tensor's device; the kernels launch on the CURRENT device, so it must be the tensor's"""
    if t.device.index != torch.cuda.current_device():
        raise RuntimeError("genre_shapehd_b200: tensor on %s but the current CUDA device is %d; wrap the call in "
                           "`with torch.cuda.device(tensor.device):`" % (t.device, torch.cuda.current_device()))
    return torch.cuda.current_stream(t.device).cuda_stream


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("genre_shapehd_b200 ops are CUDA-only (sm_100a); got a %s tensor. "
                               "There is no CPU fallback." % t.device)


def require_f32(*tensors):
    for t in tensors:
        if t is not None and t.dtype != torch.float32:
            raise TypeError("expected float32 tensor, got %s" % t.dtype)


def workspace_for(n_maps, pixels, res, device):
    nbytes = load().genre_b200_voxelize_workspace_bytes(n_maps, pixels, res)
    return torch.empty(nbytes, dtype=torch.uint8, device=device), nbytes
