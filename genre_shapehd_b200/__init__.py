"""genre_shapehd_b200 — B200-native (sm_100a) hot path of GenRe / ShapeHD.

The product is ``lib/libgenre_b200.so`` (hand-written CUDA behind a C ABI, ``include/genre_b200.h``)
plus thin Python packages that mirror the reference's import surface, so that the reference's own
``models/*.py`` run on top of them unchanged, and the GenRe / ShapeHD model classes built on them
(``genre_models.py``):

    toolbox.cam_bp.cam_bp.{functions,modules}      toolbox/cam_bp/cam_bp/      in the reference
    toolbox.calc_prob.calc_prob.functions.calc_prob toolbox/calc_prob/
    toolbox.spherical_proj                          toolbox/spherical_proj.py
    nndistance.{functions,modules}                  toolbox/nndistance/
    networks.networks                               networks/networks.py (3D voxel nets)

``install()`` puts those packages first on ``sys.path`` (and, given a checkout of the reference, that checkout
after them and its ``networks`` directory on ``networks.__path__``, so ``models``, ``util``, ``networks.uresnet`` ...
resolve there).

There is no CPU fallback anywhere: every op raises if the CUDA library is missing or a tensor is
not on a CUDA device.
"""
import os
import sys

__version__ = "0.1.0"

PACKAGE_DIR = os.path.dirname(os.path.abspath(__file__))
REPO_ROOT = os.path.dirname(PACKAGE_DIR)


def install(reference_root=None):
    """Make ``toolbox``, ``nndistance`` and ``networks`` resolve to this package.

    reference_root: optional path of a GenRe-ShapeHD checkout (default: $GENRE_REF); appended AFTER this package
    so that everything outside the hot path (models/, util/, loggers/, networks/uresnet.py ...) comes from it.
    """
    for p in (os.path.join(PACKAGE_DIR, "toolbox"), PACKAGE_DIR):
        if p in sys.path:
            sys.path.remove(p)
        sys.path.insert(0, p)
    if REPO_ROOT not in sys.path:
        sys.path.append(REPO_ROOT)
    if reference_root is None:
        reference_root = os.environ.get("GENRE_REF")
    if reference_root and os.path.isdir(reference_root) and reference_root not in sys.path:
        sys.path.append(reference_root)
    for name in ("toolbox", "nndistance", "networks"):
        mod = sys.modules.get(name)
        if mod is not None and not getattr(mod, "__file__", "").startswith(PACKAGE_DIR):
            raise ImportError(
                "%s was already imported from %s; call genre_shapehd_b200.install() first" % (name, mod.__file__))
    ref_networks = os.path.join(reference_root, "networks") if reference_root else None
    if ref_networks and os.path.isdir(ref_networks):
        import networks                          # this package's: the checkout's 2D nets resolve as networks.<name>
        if ref_networks not in networks.__path__:
            networks.__path__.append(ref_networks)
    return PACKAGE_DIR
