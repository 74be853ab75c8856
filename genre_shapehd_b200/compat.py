"""Harness that lets the reference's FROZEN caller files (models/*.py, util/*.py ...) import and run on a current
PyTorch on top of this package, without editing or copying them (SURVEY.md §7.1 step 0, Appendix B).

    import genre_shapehd_b200.compat as compat
    compat.bootstrap("/path/to/GenRe-ShapeHD")     # then: from models.genre_full_model import Net

What it does:
  * genre_shapehd_b200.install(reference_root): toolbox / nndistance / networks.networks resolve HERE, everything
    else (models, util, loggers, visualize, datasets, options, networks.uresnet/revresnet) in the reference checkout;
  * stubs the optional third-party modules the frozen files import at module level but never use on the
    differentiable path (skimage, trimesh; visualize/visualizer.py:8, util/util_sph.py:1-3); the stub
    skimage.measure.marching_cubes(_lewiner) is a working mesher on the GPU (``marching_cubes`` below), so the
    visualiser writes its .obj files;
  * makes torchvision's resnet18(pretrained=True) build offline (random init) — there is no network here.
"""
import os
import sys
import types

import genre_shapehd_b200


def _stub(name, **attrs):
    if name in sys.modules:
        return sys.modules[name]
    try:
        return __import__(name)
    except Exception:
        pass
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    m.__genre_b200_stub__ = True
    sys.modules[name] = m
    return m


def _unavailable(what):
    def f(*a, **k):
        raise RuntimeError("%s is not available in this environment (stubbed by genre_shapehd_b200.compat)" % what)
    return f


_NO_CUDA_HINT = ("run the visualiser in the main process (--vis_workers 0), or export meshes for a whole batch with "
                 "genre_shapehd_b200.postprocess.export_obj")


def marching_cubes(volume, level=None, spacing=(1.0, 1.0, 1.0), gradient_direction="descent", step_size=1,
                   allow_degenerate=True, method="lewiner", mask=None, use_classic=False):
    """Stand-in for skimage.measure.marching_cubes / marching_cubes_lewiner when skimage is not installed.

    Returns numpy ``(verts, faces, normals, values)`` like skimage.  The mesh comes from
    ``postprocess.iso_surface`` on the current CUDA device (its case table does no MC33 interior disambiguation, so in
    ambiguous cells the triangles can differ from Lewiner's).  ``normals`` are NOT skimage's gradient normals: they are
    area-weighted face normals accumulated per vertex and normalised, pointing from the > level side to the <= level side
    (outward for an occupancy volume).  ``values`` are max(f(p), f(p + e_a)) of each vertex's grid edge.  Arguments this
    stand-in does not implement raise NotImplementedError instead of being ignored."""
    import numpy as np
    import torch
    if method != "lewiner":
        raise NotImplementedError("marching_cubes stand-in: method=%r (only 'lewiner' is accepted)" % (method,))
    if step_size != 1:
        raise NotImplementedError("marching_cubes stand-in: step_size=%r (only 1)" % (step_size,))
    if mask is not None:
        raise NotImplementedError("marching_cubes stand-in: mask is not supported")
    if gradient_direction != "descent":
        raise NotImplementedError("marching_cubes stand-in: gradient_direction=%r (only 'descent')" % (gradient_direction,))
    if not allow_degenerate:
        raise NotImplementedError("marching_cubes stand-in: allow_degenerate=False is not supported")
    if use_classic:
        raise NotImplementedError("marching_cubes stand-in: use_classic=True is not supported")
    if torch.cuda._is_in_bad_fork():
        raise RuntimeError("marching_cubes stand-in: CUDA cannot be used in a process forked after the parent initialised "
                           "CUDA (a multiprocessing Pool worker); " + _NO_CUDA_HINT)
    if not torch.cuda.is_available():
        raise RuntimeError("marching_cubes stand-in: no CUDA device (the mesher runs on the GPU); " + _NO_CUDA_HINT)
    from . import postprocess
    vol = np.ascontiguousarray(volume, dtype=np.float32)
    if vol.ndim != 3:
        raise ValueError("marching_cubes stand-in: expected a 3-D volume, got shape %s" % (vol.shape,))
    if level is None:
        level = float(vol.min() + vol.max()) / 2
    if not (vol.min() <= level <= vol.max()):
        raise ValueError("Surface level must be within volume data range.")
    dev = torch.device("cuda", torch.cuda.current_device())
    t = torch.from_numpy(vol).to(dev)
    verts, faces, values = postprocess.iso_surface(t, level, spacing=tuple(spacing), values=True)[0]
    fl = faces.long()
    v0, v1, v2 = verts[fl[:, 0]], verts[fl[:, 1]], verts[fl[:, 2]]
    fn = torch.cross(v1 - v0, v2 - v0, dim=1)                # |fn| = twice the area: area-weighted
    normals = torch.zeros_like(verts)
    for c in range(3):
        normals.index_add_(0, fl[:, c], fn)
    normals = torch.nn.functional.normalize(normals, dim=1)
    return (verts.cpu().numpy(), faces.cpu().numpy(), normals.cpu().numpy(), values.cpu().numpy())


def marching_cubes_lewiner(volume, level=None, spacing=(1.0, 1.0, 1.0), gradient_direction="descent", step_size=1,
                           allow_degenerate=True, use_classic=False, mask=None):
    """skimage.measure.marching_cubes_lewiner's signature on top of ``marching_cubes``"""
    return marching_cubes(volume, level, spacing, gradient_direction, step_size, allow_degenerate, "lewiner", mask,
                          use_classic)


def find_reference():
    """a checkout of the original GenRe-ShapeHD project named by $GENRE_REF, or None"""
    root = os.environ.get("GENRE_REF")
    return root if root and os.path.isdir(os.path.join(root, "models")) else None


def bootstrap(reference_root=None, offline_resnet=True):
    root = reference_root or find_reference()
    if root is None or not os.path.isdir(os.path.join(root, "models")):
        raise FileNotFoundError("no GenRe-ShapeHD checkout at %r: pass its path or set $GENRE_REF" % root)
    os.environ["GENRE_REF"] = root
    genre_shapehd_b200.install(root)
    stub_optional_modules(offline_resnet)
    return root


def stub_optional_modules(offline_resnet=True):
    """stand-ins for skimage / trimesh (imported at module level by the frozen files, unused on the differentiable path; the
    skimage.measure marching cubes is a working GPU mesher) and an offline torchvision resnet18.  A real skimage, where
    installed, is left alone."""
    sk = _stub("skimage")
    if getattr(sk, "__genre_b200_stub__", False):
        measure = _stub("skimage.measure", marching_cubes_lewiner=marching_cubes_lewiner, marching_cubes=marching_cubes)
        sk.measure = measure
        _stub("skimage.io", imread=_unavailable("skimage.io.imread"), imsave=_unavailable("skimage.io.imsave"))
        _stub("skimage.transform", resize=_unavailable("skimage.transform.resize"))
    tm = _stub("trimesh")
    if getattr(tm, "__genre_b200_stub__", False):
        tm.Trimesh = _unavailable("trimesh.Trimesh")
        tm.load = _unavailable("trimesh.load")
    if offline_resnet:
        import torchvision.models as tvm
        if not getattr(tvm.resnet18, "__genre_b200_offline__", False):
            orig = tvm.resnet18

            def resnet18(pretrained=False, **kw):  # the frozen files pass pretrained=True (uresnet.py:16,87)
                kw.pop("weights", None)
                return orig(weights=None, **kw)
            resnet18.__genre_b200_offline__ = True
            tvm.resnet18 = resnet18
            try:
                import torchvision.models.resnet as tvr
                tvr.resnet18 = resnet18
            except Exception:
                pass


def fold_batchnorm2d_eval(root):
    """Deployment-side cheap win for the reference's 2D U-ResNets (SURVEY 8f-2; their code stays the reference's): fold every
    eval-mode ``BatchNorm2d`` that directly follows a ``Conv2d`` / ``ConvTranspose2d`` into that convolution, in place, on THIS
    module instance (the BatchNorm becomes ``nn.Identity``).  Patterns: the (conv_k, bn_k) / (deconv_k, bn_k) attribute pairs of
    torchvision's BasicBlock and networks/revresnet.py's RevBasicBlock / RevBottleneck, and adjacent pairs inside ``nn.Sequential``
    (stems, down/up-sample branches, the decoders' heads).  Mathematically identical, rounding differs at the 1e-6 level.
    Returns the number of BatchNorms folded.  Inference only: call after ``.eval()``; state_dict keys of the folded layers change."""
    import torch.nn as nn
    from torch.nn.utils.fusion import fuse_conv_bn_eval
    folded = 0

    def fuse(conv, bn):
        return fuse_conv_bn_eval(conv, bn, transpose=isinstance(conv, nn.ConvTranspose2d))

    def ok(conv, bn):
        return (isinstance(conv, (nn.Conv2d, nn.ConvTranspose2d)) and isinstance(bn, nn.BatchNorm2d) and not bn.training
                and not conv.training and bn.track_running_stats and conv.out_channels == bn.num_features)
    for mod in list(root.modules()):
        if isinstance(mod, nn.Sequential):
            names = list(mod._modules.keys())
            for a, b in zip(names, names[1:]):
                if ok(mod._modules[a], mod._modules[b]):
                    mod._modules[a] = fuse(mod._modules[a], mod._modules[b])
                    mod._modules[b] = nn.Identity()
                    folded += 1
            continue
        for k in ("1", "2", "3"):
            bn = mod._modules.get("bn" + k)
            for cname in ("conv" + k, "deconv" + k):
                conv = mod._modules.get(cname)
                if conv is not None and bn is not None and ok(conv, bn):
                    mod._modules[cname] = fuse(conv, bn)
                    mod._modules["bn" + k] = nn.Identity()
                    folded += 1
                    break
    return folded
