"""numpy front end of the marching-cubes checker (libmc_oracle.so, built from mc_oracle.c by this directory's Makefile or
__graft_entry__.build()).  TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and
profiles/microbench_mesh.py; never by the product package."""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "libmc_oracle.so")

_c = ctypes
_f = np.float32
_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB):
            raise RuntimeError("oracle_mesh/libmc_oracle.so missing: run `make -C oracle_mesh` (or __graft_entry__.build())")
        _lib = ctypes.CDLL(LIB)
    return _lib


def _p(a):
    return a.ctypes.data_as(_c.c_void_p)


def iso_surface(volume, level, spacing=(1.0, 1.0, 1.0), offset=(0.0, 0.0, 0.0), values=False):
    """one [D,H,W] volume -> (verts [V,3] fp32, faces [F,3] int32[, values [V] fp32]) in the order and rounding of
    genre_b200_iso_surface_emit (single-threaded per-cell loop)."""
    vol = np.ascontiguousarray(volume, dtype=_f)
    d, h, w = vol.shape
    nv, nf = _c.c_long(), _c.c_long()
    lib().oracle_iso_surface_count(_p(vol), _c.c_long(d), _c.c_long(h), _c.c_long(w), _c.c_float(level), _c.byref(nv),
                                   _c.byref(nf))
    verts = np.empty((nv.value, 3), _f)
    faces = np.empty((nf.value, 3), np.int32)
    vals = np.empty(nv.value, _f) if values else None
    idx = np.empty(d * h * w * 3, np.int32)
    sp = np.ascontiguousarray(np.broadcast_to(np.asarray(spacing, _f), (3,)))
    of = np.ascontiguousarray(np.broadcast_to(np.asarray(offset, _f), (3,)))
    lib().oracle_iso_surface(_p(vol), _c.c_long(d), _c.c_long(h), _c.c_long(w), _c.c_float(level), _p(sp), _p(of), _p(verts),
                             _p(faces), _p(vals) if values else None, _p(idx))
    return (verts, faces, vals) if values else (verts, faces)
