"""Drop-in for the reference's ``networks`` package: ``networks.networks`` holds the 3D voxel nets (on the hot
path).  The 2D U-ResNet-18s of GenRe are in genre_shapehd_b200/genre_models.py; genre_shapehd_b200.install() given a
checkout of the reference appends its ``networks`` directory to this package's ``__path__``, so that the reference's
own ``networks.uresnet`` / ``networks.revresnet`` resolve there (nothing is copied)."""
import os
import sys

_REPO_ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if _REPO_ROOT not in sys.path:
    sys.path.append(_REPO_ROOT)
