"""Harness that lets the reference's FROZEN caller files (models/*.py, util/*.py ...) import and run on a current
PyTorch on top of this package, without editing or copying them (SURVEY.md §7.1 step 0, Appendix B).

    import genre_shapehd_b200.compat as compat
    compat.bootstrap("/path/to/GenRe-ShapeHD")     # then: from models.genre_full_model import Net

What it does:
  * genre_shapehd_b200.install(reference_root): toolbox / nndistance / networks.networks resolve HERE, everything
    else (models, util, loggers, visualize, datasets, options, networks.uresnet/revresnet) in the reference checkout;
  * stubs the optional third-party modules the frozen files import at module level but never use on the
    differentiable path (skimage, trimesh; visualize/visualizer.py:8, util/util_sph.py:1-3);
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
    """stand-ins for skimage / trimesh (imported at module level by the frozen files, unused on the differentiable path) and
    an offline torchvision resnet18"""
    sk = _stub("skimage")
    if getattr(sk, "__genre_b200_stub__", False):
        measure = _stub("skimage.measure", marching_cubes_lewiner=_unavailable("skimage.measure.marching_cubes"),
                        marching_cubes=_unavailable("skimage.measure.marching_cubes"))
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
