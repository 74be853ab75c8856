"""Mirror of the reference's cffi module ``cam_bp._ext.cam_bp_lib``.

Same five function names, argument orders and in-place-output convention as
toolbox/cam_bp/cam_bp/src/back_projection.h:1-5 (the caller allocates every output), but bound to
libgenre_b200.so through its C ABI instead of THCudaTensor*.  Failure raises RuntimeError (the
reference: THError("aborting"), back_projection.c:11-16).  Returns 1 like the reference.
"""
import torch

from genre_shapehd_b200 import _lib


def _dense(t, name):
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % name)
    return t


def _check_maps(depth, fl, camdist):
    _lib.require_cuda(depth, fl, camdist)
    _lib.require_f32(depth, fl, camdist)
    if depth.dim() != 4:
        raise ValueError("4D input tensor expected but got: %s" % (tuple(depth.shape),))
    n, c = depth.shape[:2]
    for t, nm in ((fl, "fl"), (camdist, "camdist")):
        if t.dim() != 2 or t.shape[0] != n or t.shape[1] != c:
            raise ValueError("Need %s of shape [%d, %d] but got %s" % (nm, n, c, tuple(t.shape)))


def _check_vol(vol, depth, name):
    if vol.dim() != 5 or vol.shape[0] != depth.shape[0] or vol.shape[1] != depth.shape[1] or \
            not (vol.shape[2] == vol.shape[3] == vol.shape[4]):
        raise ValueError("Need %s of shape [N, C, R, R, R] but got %s" % (name, tuple(vol.shape)))
    _lib.require_cuda(vol)
    _lib.require_f32(vol)
    return _dense(vol, name)


def back_projection_forward(depth, camdist, fl, voxel, cnt, shift=False):
    """back_projection.h:1.  ``voxel`` is fully overwritten (the reference needs it pre-filled with
    1/res and accumulates into it; the values coming out are the same).  ``cnt`` may be None when the
    count volume is not needed (inference), ``shift`` fuses Camera_back_projection_layer.shift_tdf."""
    _check_maps(depth, fl, camdist)
    _check_vol(voxel, depth, "voxel")
    if cnt is not None:
        _check_vol(cnt, depth, "cnt")
    n, c, h, w = depth.shape
    res = voxel.shape[2]
    ws, nbytes = _lib.workspace_for(n * c, h * w, res, depth.device)
    _lib.call("genre_b200_cam_bp_forward", depth.data_ptr(), n, c, h, w, *depth.stride(),
              fl.data_ptr(), *fl.stride(), camdist.data_ptr(), *camdist.stride(),
              voxel.data_ptr(), cnt.data_ptr() if cnt is not None else None, res,
              _lib.FLAG_SHIFT_TDF if shift else 0, ws.data_ptr(), nbytes, _lib.stream_ptr(depth))
    return 1


def back_projection_backward(depth, fl, camdist, cnt, grad_in, grad_depth, grad_camdist, grad_fl):
    """back_projection.h:2 (note the (…, grad_camdist, grad_fl) order)."""
    _check_maps(depth, fl, camdist)
    _check_vol(cnt, depth, "cnt")
    _check_vol(grad_in, depth, "grad_in")
    n, c, h, w = depth.shape
    _lib.require_cuda(grad_depth, grad_camdist, grad_fl)
    if tuple(grad_depth.shape) != (n, c, h, w) or tuple(grad_fl.shape) != (n, c) or tuple(grad_camdist.shape) != (n, c):
        raise ValueError("gradient buffers have the wrong shape")
    _dense(grad_depth, "grad_depth"), _dense(grad_fl, "grad_fl"), _dense(grad_camdist, "grad_camdist")
    _lib.call("genre_b200_cam_bp_backward", depth.data_ptr(), n, c, h, w, *depth.stride(),
              fl.data_ptr(), *fl.stride(), camdist.data_ptr(), *camdist.stride(),
              cnt.data_ptr(), grad_in.data_ptr(), cnt.shape[2],
              grad_depth.data_ptr(), grad_fl.data_ptr(), grad_camdist.data_ptr(), _lib.stream_ptr(depth))
    return 1


def get_surface_mask(depth, camdist, fl, cnt, mask):
    """back_projection.h:3."""
    _check_maps(depth, fl, camdist)
    _check_vol(cnt, depth, "cnt")
    _check_vol(mask, depth, "mask")
    n, c, h, w = depth.shape
    _lib.call("genre_b200_surface_mask", depth.data_ptr(), n, c, h, w, *depth.stride(),
              fl.data_ptr(), *fl.stride(), camdist.data_ptr(), *camdist.stride(),
              cnt.data_ptr(), mask.data_ptr(), cnt.shape[2], _lib.stream_ptr(depth))
    return 1


def _check_sph(depth, grid_in):
    _lib.require_cuda(depth, grid_in)
    _lib.require_f32(depth, grid_in)
    if depth.dim() != 4:
        raise ValueError("4D input tensor expected but got: %s" % (tuple(depth.shape),))
    if grid_in.dim() != 5 or tuple(grid_in.shape) != tuple(depth.shape) + (3,):
        raise ValueError("Need grid of shape %s but got %s" % (tuple(depth.shape) + (3,), tuple(grid_in.shape)))


def spherical_back_proj_forward(depth, grid_in, voxel, cnt):
    """back_projection.h:4.  ``voxel`` and ``cnt`` are fully overwritten."""
    _check_sph(depth, grid_in)
    _check_vol(voxel, depth, "voxel")
    _check_vol(cnt, depth, "cnt")
    n, c, h, w = depth.shape
    res = voxel.shape[2]
    ws, nbytes = _lib.workspace_for(n * c, h * w, res, depth.device)
    _lib.call("genre_b200_sph_bp_forward", depth.data_ptr(), n, c, h, w, *depth.stride(),
              grid_in.data_ptr(), *grid_in.stride(), voxel.data_ptr(), cnt.data_ptr(), res,
              ws.data_ptr(), nbytes, _lib.stream_ptr(depth))
    return 1


def spherical_back_proj_backward(depth, grid_in, cnt, grad_in, grad_depth):
    """back_projection.h:5."""
    _check_sph(depth, grid_in)
    _check_vol(cnt, depth, "cnt")
    _check_vol(grad_in, depth, "grad_in")
    n, c, h, w = depth.shape
    if tuple(grad_depth.shape) != (n, c, h, w):
        raise ValueError("grad_depth has the wrong shape")
    _dense(grad_depth, "grad_depth")
    _lib.call("genre_b200_sph_bp_backward", depth.data_ptr(), n, c, h, w, *depth.stride(),
              grid_in.data_ptr(), *grid_in.stride(), cnt.data_ptr(), grad_in.data_ptr(), cnt.shape[2],
              grad_depth.data_ptr(), _lib.stream_ptr(depth))
    return 1
