"""The C-ABI library loads on a CPU-only box and exports every symbol include/genre_b200.h declares
(no compute calls here)."""
import ctypes
import os
import re

import pytest

from conftest import REPO
from genre_shapehd_b200 import _lib

HEADER = os.path.join(REPO, "include", "genre_b200.h")


def declared_symbols():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(genre_b200_\w+)\s*\(", text)))


def test_header_declares_what_binding_binds():
    assert declared_symbols() == _lib.EXPORTED_SYMBOLS


def test_library_exports_every_declared_symbol():
    assert os.path.exists(_lib.LIB_PATH), "build the library first (__graft_entry__.build())"
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared_symbols():
        assert hasattr(lib, name), "missing export: " + name


def test_version_and_error_string():
    lib = _lib.load()
    assert lib.genre_b200_version() >= 2000
    # argument errors are reported without touching the device
    rc = lib.genre_b200_nnd_forward(None, None, 1, 1, 1, None, None, None, None, None)
    assert rc == -1
    assert b"null" in lib.genre_b200_last_error()
    assert lib.genre_b200_voxelize_workspace_bytes(32, 256 * 256, 128) > 32 * 256 * 256 * 20


def test_workspace_too_small_is_rejected():
    lib = _lib.load()
    dummy = ctypes.c_void_p(256)  # never dereferenced: the size check comes first
    rc = lib.genre_b200_cam_bp_forward(dummy, 1, 1, 16, 16, 256, 256, 16, 1, dummy, 1, 1, dummy, 1, 1, dummy, None, 16,
                                       0, dummy, 16, None)
    assert rc == -2


def test_cpu_tensors_are_refused():
    import torch
    from nndistance.functions.nnd import nndistance
    from toolbox.cam_bp.cam_bp.modules.camera_backprojection_module import Camera_back_projection_layer
    with pytest.raises((RuntimeError, AssertionError)):
        nndistance(torch.zeros(1, 4, 3), torch.zeros(1, 5, 3))
    with pytest.raises((RuntimeError, AssertionError)):
        Camera_back_projection_layer()(torch.zeros(1, 1, 8, 8))


def _d(v=4096):
    """a fake, 16-byte aligned device address: argument checks come before any launch and never dereference it"""
    return ctypes.c_void_p(v)


@pytest.mark.parametrize("call,code,needle", [
    # convolution entry points: shape support is part of the contract (include/genre_b200.h)
    (lambda L: L.genre_b200_convt3d_s2_forward(_d(), 2, None, 0, 1, 2, 16, 24, _d(), 8, 32, 1, _d(), _d(), 1.0, _d(), 5, None),
     -1, b"width"),
    (lambda L: L.genre_b200_convt3d_s2_forward(_d(), 3, None, 0, 1, 2, 16, 16, _d(), 8, 32, 1, _d(), _d(), 1.0, _d(), 5, None),
     -1, b"even"),
    (lambda L: L.genre_b200_convt3d_s2_forward(_d(), 2, None, 0, 1, 2, 16, 16, _d(), 6, 32, 1, _d(), _d(), 1.0, _d(), 5, None),
     -1, b"kernel size"),
    (lambda L: L.genre_b200_convt3d_s2_forward(_d(4100), 2, None, 0, 1, 2, 16, 16, _d(), 8, 32, 1, _d(), _d(), 1.0, _d(), 5, None),
     -3, b"aligned"),
    (lambda L: L.genre_b200_convt3d_s2_merged_forward(_d(), 2, None, 0, 1, 2, 16, 16, _d(), 8, 64, 1, _d(), _d(), 1.0, _d(), 5, None),
     -1, b"npad"),
    (lambda L: L.genre_b200_conv3d_k8s2_s4d_forward(_d(), 2, 1, 2, 16, 24, _d(), 160, 1, _d(), _d(), 1.0, _d(), 5, None),
     -1, b"extent"),
    (lambda L: L.genre_b200_conv3d_k4s2_forward(_d(), 3, 1, 1, 2, 16, 16, _d(), 64, 1, _d(), _d(), 1.0, _d(), 16, None),
     -1, b"even"),
    (lambda L: L.genre_b200_convt_c1_tc_forward(_d(), 2, None, 0, 1, 2, 16, 48, _d(), 1, _d(), 0, _d(), None), -1, b"width"),
    (lambda L: L.genre_b200_convt_c1_forward(_d(), 2, None, 0, 1, 2, 16, 18, _d(), 0.0, 0, _d(), None), -1, b"extent"),
    # layout converters
    (lambda L: L.genre_b200_ncdhw_to_blocked(_d(), 1, 6, 2, 4, 4, 0, 4, 0, _d(), None), -1, b"multiple"),
    (lambda L: L.genre_b200_ncdhw_to_blocked(_d(), 1, 4, 2, 4, 4, 0, 5, 0, _d(), None), -1, b"group"),
    (lambda L: L.genre_b200_ncdhw_to_blocked(_d(), 1, 2, 3, 4, 4, 1, 4, 0, _d(), None), -1, b"odd"),
    (lambda L: L.genre_b200_blocked_to_ncdhw(_d(), 2, 1, 9, 2, 4, 4, _d(), None), -1, b"shape"),
    (lambda L: L.genre_b200_scale_clamp_strided(_d(), 2, 6, 1.0, 0.0, 1.0, _d(), 8, None), -1, b"multiples of 4"),
    # training kernels
    (lambda L: L.genre_b200_convt_c1_wgrad(_d(), _d(), 1, 80, 2, 8, 8, _d(), _d(), 1 << 30, None), -1, b"Cin"),
    (lambda L: L.genre_b200_convt_c1_wgrad(_d(), _d(), 1, 40, 2, 8, 8, _d(), _d(), 16, None), -2, b"workspace"),
    (lambda L: L.genre_b200_conv_k8s2_wgrad(_d(), _d(), 1, 3, 20, 2, 16, 16, _d(), _d(), 1 << 30, None), -1, b"Cin"),
    # fused glue
    (lambda L: L.genre_b200_render_spherical_forward_pre(_d(), 1, 16, _d(), 8, 16, _d(), 50.0, 1.0, 0.0, _d(), None), -1, b"clamp"),
    # projection flags: only GENRE_B200_FLAG_SHIFT_TDF is defined, any other bit is refused rather than ignored
    (lambda L: L.genre_b200_cam_bp_forward(_d(), 1, 1, 16, 16, 256, 256, 16, 1, _d(), 1, 1, _d(), 1, 1, _d(), None, 16, 2, _d(),
                                           1 << 30, None), -1, b"flag"),
])
def test_conv_and_layout_entry_points_validate_before_launching(call, code, needle):
    """every unsupported shape / misaligned buffer is an argument error with a message, reported without touching a GPU"""
    lib = _lib.load()
    rc = call(lib)
    msg = lib.genre_b200_last_error()
    assert rc == code, (rc, msg)
    assert needle.lower() in msg.lower(), msg
