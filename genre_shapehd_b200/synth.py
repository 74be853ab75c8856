"""Synthetic inputs for the benchmark configs (SURVEY.md §8d): numpy only, no oracle, no GPU."""
import numpy as np


def sphere_depth(h=256, w=256, fl=418.3, cam_dist=2.2, radius=0.4, background=0.0):
    """Analytic ray depth of a sphere at the origin seen from (-cam_dist, 0, 0); fp32 [h, w].
    Ray of pixel (h~, w~): (fl, -w~, -h~)/norm, the convention of back_projection_kernel.cu:239-242."""
    hh = np.arange(h, dtype=np.float64)[:, None] - (h - 1) / 2.0
    ww = np.arange(w, dtype=np.float64)[None, :] - (w - 1) / 2.0
    norm = np.sqrt(hh * hh + ww * ww + fl * fl)
    dx = fl / norm
    bq = -cam_dist * dx
    disc = bq * bq - (cam_dist * cam_dist - radius * radius)
    t = -bq - np.sqrt(np.maximum(disc, 0.0))
    return np.where(disc > 0, t, background).astype(np.float32)


def uniform_depth(seed, h=256, w=256, lo=1.7, hi=2.7, fg=0.6, background=0.0):
    """d ~ U(lo, hi) on a random `fg` fraction of the pixels, `background` elsewhere."""
    rng = np.random.RandomState(seed)
    d = rng.uniform(lo, hi, size=(h, w))
    m = rng.uniform(size=(h, w)) < fg
    return np.where(m, d, background).astype(np.float32)


def bench_depth_batch(n, h=256, w=256):
    """BASELINE.json configs[1] input: [n,1,h,w]; even samples are spheres, odd ones U(1.7,2.7) on a 60 % mask;
    the generator seed is the sample index."""
    out = np.empty((n, 1, h, w), np.float32)
    for i in range(n):
        out[i, 0] = sphere_depth(h, w, radius=0.3 + 0.01 * (i % 16)) if i % 2 == 0 else uniform_depth(i, h, w)
    return out


def iso_field(kind, shape, center=None, scale=None):
    """Analytic signed fields for the marching-cubes tests and microbenchmark: fp32 [D,H,W], > 0 inside, level 0.
    Coordinates are in voxels; the default centre is the middle of the volume shifted by a small irrational offset, so no
    sample is exactly 0.  ``scale`` defaults to the smallest extent.  Returns (field, analytic enclosed volume in voxels^3).
        sphere       radius 0.3 s
        torus        major radius 0.28 s, minor radius 0.1 s, axis along array axis 0
        two_spheres  radius 0.17 s, centres at -/+ 0.23 s along array axis 2
        shell        hollow ball between radii 0.22 s and 0.42 s"""
    shape = tuple(int(n) for n in shape)
    s = float(min(shape) if scale is None else scale)
    c = [(n - 1) / 2.0 + 0.1234567 * (a + 1) for a, n in enumerate(shape)] if center is None else list(center)
    x, y, z = np.meshgrid(*[np.arange(n, dtype=np.float64) - c[a] for a, n in enumerate(shape)], indexing="ij")
    if kind == "sphere":
        r = 0.3 * s
        f = r - np.sqrt(x * x + y * y + z * z)
        vol = 4.0 / 3.0 * np.pi * r ** 3
    elif kind == "torus":
        big, small = 0.28 * s, 0.1 * s
        f = small - np.sqrt((np.sqrt(y * y + z * z) - big) ** 2 + x * x)
        vol = 2.0 * np.pi ** 2 * big * small ** 2
    elif kind == "two_spheres":
        r, d = 0.17 * s, 0.23 * s
        f = np.maximum(r - np.sqrt(x * x + y * y + (z - d) ** 2), r - np.sqrt(x * x + y * y + (z + d) ** 2))
        vol = 2 * 4.0 / 3.0 * np.pi * r ** 3
    elif kind == "shell":
        r0, r1 = 0.22 * s, 0.42 * s
        dist = np.sqrt(x * x + y * y + z * z)
        f = np.minimum(r1 - dist, dist - r0)
        vol = 4.0 / 3.0 * np.pi * (r1 ** 3 - r0 ** 3)
    else:
        raise ValueError(kind)
    return f.astype(np.float32), vol
