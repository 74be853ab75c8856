#!/usr/bin/env python
"""Golden outputs of the REFERENCE's own kernels at full size, for the "vs reference kernel" tests of
tests/test_gpu_toolbox.py and tests/test_oracle_cpu.py.

The reference's CUDA and CPU sources are compiled unmodified into oracle/_ref/ by oracle/Makefile (given a checkout of
the original project); this script runs them on a B200 on the tests' own seeded inputs and stores what the tests
compare against, small enough to keep in git:
  * outputs compared bit for bit (voxel counts, surface mask, Chamfer distances and indices) as the sha256 of their bytes;
  * outputs compared within a tolerance at a fixed subset of their elements (every SAMPLE-th hit voxel of a
    back-projection, every STRIDE-th element of a dense output), plus their float64 sum and largest magnitude;
  * small outputs whole.

    python tests/golden/make_golden_fullsize.py OUT_DIR        # then copy OUT_DIR/*.npz into tests/golden/
"""
import hashlib
import os
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, REPO)
import genre_shapehd_b200  # noqa: E402

genre_shapehd_b200.install()
from oracle import oracle, ref_gpu  # noqa: E402
from toolbox.spherical_proj import gen_sph_grid  # noqa: E402

DEV = "cuda:0"
SAMPLE = 32          # every SAMPLE-th hit voxel of a back-projection
STRIDE = 14          # every STRIDE-th element of a dense gradient
CALC_PROB_STRIDE = 512


def sha(t):
    return hashlib.sha256(t.detach().contiguous().cpu().numpy().tobytes()).hexdigest()


def sparse(cnt, tdf):
    """hit voxels of a back-projection: the counts bit for bit, the distances at every SAMPLE-th hit"""
    c = cnt.reshape(-1).cpu().numpy()
    idx = np.flatnonzero(c)[::SAMPLE]
    t = tdf.reshape(-1).cpu().numpy()
    return {"cnt_sha256": sha(cnt), "n_hits": int((c != 0).sum()), "idx": idx.astype(np.int32), "tdf": t[idx],
            "tdf_sum_f64": float(tdf.double().sum())}


def strided(name, t, stride=STRIDE):
    return {name: t.detach().reshape(-1).cpu().numpy()[::stride], name + "_absmax": float(t.abs().max()),
            name + "_sum_f64": float(t.double().sum())}


def save(out_dir, name, **arrays):
    np.savez_compressed(os.path.join(out_dir, name + ".npz"), **arrays)


def main(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    n_ = lambda x: x.detach().cpu().numpy()  # noqa: E731
    # camera back-projection forward, bench depth maps
    for n in (1, 4):
        d = torch.from_numpy(oracle.bench_depth_batch(n)).to(DEV)
        tdf, cnt = ref_gpu.cam_bp_forward(d, torch.full((n, 1), 418.3, device=DEV), torch.full((n, 1), 2.2, device=DEV), 128)
        save(out_dir, "ref_cam_bp_forward_n%d" % n, **sparse(cnt, tdf))
    # camera back-projection backward, one map (the reference kernel reads cam_dist out of bounds for n >= 1)
    d = torch.from_numpy(oracle.bench_depth_batch(2)[1:2]).to(DEV)
    fl, cd = torch.full((1, 1), 418.3, device=DEV), torch.full((1, 1), 2.2, device=DEV)
    tdf, cnt = ref_gpu.cam_bp_forward(d, fl, cd, 128)
    g = torch.randn(1, 1, 128, 128, 128, device=DEV, generator=torch.Generator(DEV).manual_seed(0))
    gd, gfl, gcd = ref_gpu.cam_bp_backward(d, fl, cd, cnt, g)
    save(out_dir, "ref_cam_bp_backward", **sparse(cnt, tdf), **strided("grad_depth", gd), grad_fl=n_(gfl), grad_camdist=n_(gcd))
    # surface mask, background marked -1
    d = oracle.bench_depth_batch(2)
    d[d == 0] = -1.0
    d = torch.from_numpy(d).to(DEV)
    fl, cd = torch.full((2, 1), 418.3, device=DEV), torch.full((2, 1), 2.2, device=DEV)
    tdf, cnt = ref_gpu.cam_bp_forward(d, fl, cd, 128)
    mask = ref_gpu.surface_mask(d, fl, cd, cnt)
    save(out_dir, "ref_surface_mask", cnt_sha256=sha(cnt), mask_sha256=sha(mask),
         mask_zero_frac=float((mask == 0).float().mean()))
    # spherical back-projection, forward and backward
    n = 3
    rng = np.random.RandomState(5)
    sph = rng.uniform(0.02, 0.7, size=(n, 1, 128, 128)).astype(np.float32)
    sph[0, 0, :16] = -0.5
    sph = torch.from_numpy(sph).to(DEV)
    grid = gen_sph_grid().to(DEV).expand(n, -1, -1, -1, -1)
    tdf, cnt = ref_gpu.sph_bp_forward(sph, grid, 128)
    g = torch.randn(tdf.shape, device=DEV, generator=torch.Generator(DEV).manual_seed(1))
    gs = ref_gpu.sph_bp_backward(sph, grid, cnt, g)
    save(out_dir, "ref_sph_bp", **sparse(cnt, tdf), **strided("grad_sph", gs))
    # stop probability, forward and backward
    gen = torch.Generator(DEV).manual_seed(0)
    p = torch.rand(2, 1, 128, 128, 256, device=DEV, generator=gen).clamp_(1e-5, 1 - 1e-5)
    p = torch.where(torch.rand(p.shape, device=DEV, generator=gen) < 0.9, torch.full_like(p, 1e-5), p)
    s = ref_gpu.calc_prob_forward(p)
    g = torch.randn(p.shape, device=DEV, generator=gen)
    gr = ref_gpu.calc_prob_backward(p, s * g)
    save(out_dir, "ref_calc_prob", stride=CALC_PROB_STRIDE, **strided("stop", s, CALC_PROB_STRIDE),
         **strided("grad_prob", gr, CALC_PROB_STRIDE))
    # Chamfer, GPU kernels
    for b, n, m in ((4, 4096, 4096), (2, 3000, 5000)):
        gen = torch.Generator(DEV).manual_seed(n)
        x1 = torch.rand(b, n, 3, device=DEV, generator=gen) - 0.5
        x2 = torch.rand(b, m, 3, device=DEV, generator=gen) - 0.5
        d1, d2, i1, i2 = ref_gpu.nnd_forward(x1, x2)
        g1, g2 = torch.rand(b, n, device=DEV, generator=gen), torch.rand(b, m, device=DEV, generator=gen)
        o1, o2 = ref_gpu.nnd_backward(x1, x2, g1, g2, i1, i2)
        save(out_dir, "ref_nnd_%d_%d_%d" % (b, n, m), dist1_sha256=sha(d1), dist2_sha256=sha(d2), idx1_sha256=sha(i1),
             idx2_sha256=sha(i2), **strided("grad_xyz1", o1), **strided("grad_xyz2", o2))
    # Chamfer, the reference's CPU code
    cpu = {}
    for b, n, m, seed in ((1, 50, 50, 0), (2, 257, 129, 1), (3, 64, 700, 2)):
        rng = np.random.RandomState(seed)
        p1 = (rng.rand(b, n, 3) * 20).astype(np.float32)
        p2 = (rng.rand(b, m, 3) * 20).astype(np.float32)
        dist, idx = oracle.ref_nnsearch_cpu(p1, p2)
        cpu["dist_%d" % seed], cpu["idx_%d" % seed] = dist, idx
    save(out_dir, "ref_nnd_cpu", **cpu)
    print("golden vectors written to", out_dir, sorted(os.listdir(out_dir)))


if __name__ == "__main__":
    main(sys.argv[1])
