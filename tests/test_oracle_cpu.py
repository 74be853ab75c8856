"""CPU-only checks of the oracle (oracle/genre_oracle.c): against the reference's own CPU code where it has
any (nndistance, my_lib.c: its outputs stored in tests/golden/ref_nnd_cpu.npz), against independent float64 restatements, against the
torch-CPU composition the reference's render_spherical is written in, and the C1 plumbing config
(depth -> voxel -> spherical on one 256x256 map, SURVEY.md §8d)."""
import os

import numpy as np
import pytest
import torch

from toolbox.spherical_proj import gen_sph_grid, render_spherical


# --------------------------------------------------------------------------------------------------
# nndistance: the only op with a CPU implementation in the reference
# --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("b,n,m,seed", [(1, 50, 50, 0), (2, 257, 129, 1), (3, 64, 700, 2)])
def test_nnd_oracle_matches_reference_cpu_code(oracle, golden_dir, b, n, m, seed):
    rng = np.random.RandomState(seed)
    p1 = (rng.rand(b, n, 3) * 20).astype(np.float32)  # the reference demo's scale (nndistance/test.py:11-12)
    p2 = (rng.rand(b, m, 3) * 20).astype(np.float32)
    ref = np.load(os.path.join(golden_dir, "ref_nnd_cpu.npz"))     # tests/golden/make_golden_fullsize.py
    d_ref, i_ref = ref["dist_%d" % seed], ref["idx_%d" % seed]
    d, i = oracle.nnsearch(p1, p2, fused=False)
    assert np.array_equal(i, i_ref)
    assert np.array_equal(d, d_ref)
    # the GPU rounding (FMA-contracted) differs from the CPU code by at most an ulp or two
    d_f, i_f = oracle.nnsearch(p1, p2, fused=True)
    np.testing.assert_allclose(d_f, d_ref, rtol=5e-7)


def test_nnd_oracle_ties_pick_lowest_index(oracle):
    p1 = np.zeros((1, 4, 3), np.float32)
    p2 = np.array([[[1, 0, 0], [0, 1, 0], [0, 0, 1], [-1, 0, 0], [0.5, 0, 0], [0, 0.5, 0]]], np.float32)
    for fused in (False, True):
        d, i = oracle.nnsearch(p1, p2, fused=fused)
        assert (i == 4).all() and np.allclose(d, 0.25)
    if oracle.ref_available("libref_nnd_cpu.so"):
        d, i = oracle.ref_nnsearch_cpu(p1, p2)
        assert (i == 4).all()


def test_nnd_oracle_backward_matches_autograd(oracle):
    rng = np.random.RandomState(3)
    p1 = rng.rand(2, 40, 3).astype(np.float32)
    p2 = rng.rand(2, 33, 3).astype(np.float32)
    d1, d2, i1, i2 = oracle.nnd_forward(p1, p2)
    g1 = rng.rand(2, 40).astype(np.float32)
    g2 = rng.rand(2, 33).astype(np.float32)
    o1, o2 = oracle.nnd_backward(p1, p2, g1, g2, i1, i2)
    t1 = torch.tensor(p1, dtype=torch.float64, requires_grad=True)
    t2 = torch.tensor(p2, dtype=torch.float64, requires_grad=True)
    dd = ((t1[:, :, None, :] - t2[:, None, :, :]) ** 2).sum(-1)
    loss = (dd.min(2).values * torch.tensor(g1, dtype=torch.float64)).sum() + \
        (dd.min(1).values * torch.tensor(g2, dtype=torch.float64)).sum()
    loss.backward()
    np.testing.assert_allclose(o1, t1.grad.numpy(), atol=1e-5)
    np.testing.assert_allclose(o2, t2.grad.numpy(), atol=1e-5)


# --------------------------------------------------------------------------------------------------
# cam_bp: independent float64 restatement of the geometry
# --------------------------------------------------------------------------------------------------
def _cam_points64(depth, fl, cd):
    h, w = depth.shape
    hh = np.arange(h, dtype=np.float64)[:, None] - (h - 1) / 2.0
    ww = np.arange(w, dtype=np.float64)[None, :] - (w - 1) / 2.0
    z = depth.astype(np.float64) * fl / np.sqrt(hh * hh + ww * ww + fl * fl)
    return z - cd, -z * ww / fl, -z * hh / fl


@pytest.mark.parametrize("res,hw", [(128, 256), (32, 64), (20, 48)])
def test_cam_bp_oracle_vs_float64_geometry(oracle, res, hw):
    fl, cd = 418.3 * hw / 256, 2.2
    depth = oracle.uniform_depth(5, hw, hw)
    depth[::7, ::5] = -1.0  # exercise the d < 0 skip (back_projection_kernel.cu:225)
    vidx = oracle.cam_bp_voxel_index(depth[None, None], fl, cd, res)[0, 0]
    gx, gy, gz = _cam_points64(depth, np.float32(fl).astype(np.float64), np.float32(cd).astype(np.float64))
    f = [(g + 0.5) * res for g in (gx, gy, gz)]
    idx = [np.floor(a).astype(np.int64) for a in f]
    inb = np.ones_like(depth, bool)
    for a in idx:
        inb &= (a >= 0) & (a < res)
    inb &= ~(depth < 0)
    lin = np.where(inb, (idx[0] * res + idx[1]) * res + idx[2], -1)
    # away from voxel faces the fp32 sequence and float64 must agree exactly
    safe = np.ones_like(depth, bool)
    for a in f:
        safe &= np.abs(a - np.round(a)) > 1e-3
    safe |= depth <= 0  # background (0) and skipped (<0) pixels are unambiguous
    assert safe.mean() > 0.98
    assert np.array_equal(vidx[safe], lin[safe])
    # TDF: mean distance to the voxel centre
    tdf, cnt = oracle.cam_bp_forward(depth[None, None], fl, cd, res)
    assert cnt.sum() == (vidx >= 0).sum()
    hit = cnt[0, 0] > 0
    assert np.all(tdf[0, 0][~hit] == np.float32(1.0 / res))
    assert tdf[0, 0][hit].max() <= np.sqrt(3) / (2 * res) * (1 + 1e-5)
    # shifted output: empty voxels exactly 0 for power-of-two res, hit voxels in (0.134, 1]
    sh, _ = oracle.cam_bp_forward(depth[None, None], fl, cd, res, shift=True)
    if res & (res - 1) == 0:
        assert np.all(sh[0, 0][~hit] == 0.0)
    assert sh[0, 0][hit].min() > 0.13 and sh[0, 0][hit].max() <= 1.0


def test_cam_bp_oracle_strides_and_channels(oracle):
    rng = np.random.RandomState(0)
    base = rng.uniform(1.7, 2.7, size=(2, 3, 40, 40)).astype(np.float32)
    fl = np.array([[100.0, 110.0, 90.0], [95.0, 105.0, 100.0]], np.float32) * 0.65
    cd = np.array([[2.2, 2.1, 2.3], [2.0, 2.2, 2.4]], np.float32)
    a = oracle.cam_bp_voxel_index(base, fl, cd, 32)
    # transposed + flipped view with the same logical content (GenRe feeds such a view,
    # depth_pred_with_sph_inpaint.py:140-141)
    view = np.ascontiguousarray(base.transpose(0, 1, 3, 2)[:, :, ::-1]).transpose(0, 1, 3, 2)[:, :, :, ::-1]
    assert np.array_equal(np.asarray(view), base) and not view.flags.c_contiguous
    b = oracle.cam_bp_voxel_index(view, fl, cd, 32)
    assert np.array_equal(a, b)


def test_cam_bp_oracle_backward_is_directional_derivative(oracle):
    """grad_depth = -g * cos(ray, point - centre) / cnt is d(mean distance)/d(depth) for a single-point voxel."""
    res, hw = 32, 64
    fl, cd = 104.0, 2.2
    depth = oracle.uniform_depth(9, hw, hw, fg=0.3)
    tdf, cnt = oracle.cam_bp_forward(depth[None, None], fl, cd, res)
    g = np.ones_like(tdf)
    gd, gfl, gcd = oracle.cam_bp_backward(depth[None, None], fl, cd, cnt, g, res)
    vidx = oracle.cam_bp_voxel_index(depth[None, None], fl, cd, res)[0, 0]
    single = (vidx >= 0) & (cnt[0, 0].reshape(-1)[np.maximum(vidx, 0)] == 1)
    ys, xs = np.nonzero(single)
    eps = 1e-4
    checked = 0
    for y, x in list(zip(ys, xs))[:40]:
        v = vidx[y, x]
        vals = []
        for sgn in (+1, -1):
            d2 = depth.copy()
            d2[y, x] += sgn * eps
            if oracle.cam_bp_voxel_index(d2[None, None], fl, cd, res)[0, 0, y, x] != v:
                break
            vals.append(oracle.cam_bp_forward(d2[None, None], fl, cd, res)[0].reshape(-1)[v])
        if len(vals) < 2:
            continue
        num = (vals[0] - vals[1]) / (2 * eps)
        # back_projection_kernel.cu:448-455: -g*cos(-ray, point-centre)/cnt == +d(dist)/d(depth) * g / cnt
        assert abs(num - gd[0, 0, y, x]) < 3e-3
        checked += 1
    assert checked >= 10
    assert np.isfinite(gfl).all() and np.isfinite(gcd).all()


def test_surface_mask_oracle_carves_behind_the_surface(oracle):
    res, hw = 32, 64
    fl, cd = 418.3 * hw / 256, 2.2
    depth = oracle.sphere_depth(hw, hw, fl=fl, radius=0.35, background=-1.0)
    _, cnt = oracle.cam_bp_forward(depth[None, None], fl, cd, res)
    mask = oracle.surface_mask(depth[None, None], fl, cd, cnt, res)
    assert set(np.unique(mask)) <= {0.0, 1.0}
    c = (np.arange(res) + 0.5) / res - 0.5
    X, Y, Z = np.meshgrid(c, c, c, indexing="ij")
    r = np.sqrt(X * X + Y * Y + Z * Z)
    m = mask[0, 0]
    assert m[cnt[0, 0] > 0].min() == 1.0               # surface voxels are never carved
    # well inside the sphere (behind the observed surface): carved.  Outside the silhouette cone: kept.
    assert (m[r < 0.25] == 0).mean() > 0.99
    assert (m[(np.abs(Y) > 0.45) & (np.abs(Z) > 0.45)] == 1).all()


# --------------------------------------------------------------------------------------------------
# spherical back-projection
# --------------------------------------------------------------------------------------------------
def test_sph_bp_oracle_vs_float64(oracle):
    res = 32
    grid = gen_sph_grid(32).numpy()  # [1,1,32,32,3]
    rng = np.random.RandomState(2)
    sph = rng.uniform(0.05, 0.6, size=(2, 1, 32, 32)).astype(np.float32)
    sph[0, 0, :4] = -1.0
    tdf, cnt = oracle.sph_bp_forward(sph, grid, res)
    p = grid[0, 0].astype(np.float64)[None] * sph[:, 0, :, :, None].astype(np.float64)
    f = (p + 0.5) * res
    idx = np.floor(f).astype(np.int64)
    inb = ((idx >= 0) & (idx < res)).all(-1) & ~(sph[:, 0] < 0)
    safe = (np.abs(f - np.round(f)) > 1e-3).all(-1)
    cnt64 = np.zeros((2, res, res, res))
    for n in range(2):
        for (a, b, c) in idx[n][inb[n]]:
            cnt64[n, a, b, c] += 1
    if safe[inb].all():
        assert np.array_equal(cnt64, cnt[:, 0])
    assert cnt.sum() == inb.sum()
    assert np.all(tdf[cnt == 0] == 0.0)
    # backward: g * (r - dir.centre) / (cnt * dist) is d(dist)/dr averaged
    gsph = oracle.sph_bp_backward(sph, grid, cnt, np.ones_like(tdf), res)
    assert gsph.shape == sph.shape and np.isfinite(gsph).all()
    assert np.all(gsph[0, 0, :4] == 0)


# --------------------------------------------------------------------------------------------------
# calc_prob
# --------------------------------------------------------------------------------------------------
def test_calc_prob_oracle_closed_form_and_gradient(oracle):
    rng = np.random.RandomState(4)
    p = np.clip(rng.rand(3, 1, 4, 5, 64), 1e-5, 1 - 1e-5).astype(np.float32)
    s = oracle.calc_prob_forward(p)
    p64 = p.astype(np.float64)
    closed = p64 * np.concatenate([np.ones_like(p64[..., :1]), np.cumprod(1 - p64, -1)[..., :-1]], -1)
    np.testing.assert_allclose(s, closed, rtol=2e-5, atol=1e-30)
    g = rng.randn(*p.shape).astype(np.float32)
    grad = oracle.calc_prob_backward(p, s * g)  # CalcStopProb.backward, calc_prob.py:23-29
    t = torch.tensor(p64, requires_grad=True)
    cp = torch.cat([torch.ones_like(t[..., :1]), torch.cumprod(1 - t, -1)[..., :-1]], -1)
    (t * cp * torch.tensor(g, dtype=torch.float64)).sum().backward()
    np.testing.assert_allclose(grad, t.grad.numpy(), rtol=1e-3, atol=1e-4)


# --------------------------------------------------------------------------------------------------
# render_spherical: the oracle against the torch-CPU composition the reference is written in
# --------------------------------------------------------------------------------------------------
def _torch_render(module, vox):
    """spherical_proj.py:62-72 on CPU tensors with the oracle's stop-probability (align_corners=True)."""
    from oracle import oracle as o
    grid = module.grid.expand(vox.shape[0], -1, -1, -1, -1)
    v = vox.permute(0, 1, 4, 3, 2)
    prob = torch.nn.functional.grid_sample(v, grid, mode="bilinear", padding_mode="zeros", align_corners=True)
    prob = torch.clamp(prob, 1e-5, 1 - 1e-5)
    stop = torch.from_numpy(o.calc_prob_forward(prob.numpy()))
    return torch.matmul(stop, module.depth_weight) + torch.prod(1.0 - prob, dim=4), prob


def test_render_spherical_oracle_vs_torch_composition(oracle):
    torch.manual_seed(0)
    m = render_spherical(sph_res=16, z_res=64)
    vox = torch.rand(2, 1, 24, 24, 24)
    vox[:, :, 8:14, 8:14, 8:14] = 1 - 1e-5
    ref, prob_ref = _torch_render(m, vox)
    out, prob = oracle.render_spherical(vox.numpy(), m.grid.numpy(), m.depth_weight.numpy(), return_prob=True)
    np.testing.assert_allclose(prob.reshape(prob_ref.shape), prob_ref.numpy(), atol=2e-6)
    np.testing.assert_allclose(out, ref.numpy(), atol=1e-5)


def test_config1_depth_to_voxel_to_spherical_on_one_map(oracle):
    """BASELINE.json configs[0]: one 256x256 depth map, CPU only.  A sphere of radius 0.4 seen from
    (-2.2,0,0) must render spherical depth ~0.6 on the camera-facing hemisphere and ~1 elsewhere."""
    depth = oracle.sphere_depth(256, 256, radius=0.4)
    proj, _ = oracle.cam_bp_forward(depth[None, None], 418.3, 2.2, 128, shift=True)
    vox = np.clip(proj * 50, 1e-5, 1 - 1e-5)  # depth_pred_with_sph_inpaint.py:124
    m = render_spherical()
    # render a 32x32 subset of the 128x128 rays to keep the CPU suite short
    sub = m.grid[::4, ::4].contiguous()
    sph = oracle.render_spherical(vox, sub.numpy(), m.depth_weight.numpy())[0, 0]
    dirs = gen_sph_grid()[0, 0, ::4, ::4].numpy()
    facing = dirs[..., 0] < -0.8      # rays towards the camera hit the densely sampled front cap
    away = dirs[..., 0] > 0.2         # the far side of the sphere is not in a single depth map
    # the shell is one voxel thick and sampled trilinearly at half-voxel steps, so part of each ray
    # leaks through: expected depth sits slightly above the geometric 0.6
    assert 0.58 < np.median(sph[facing]) < 0.66
    assert sph[facing].min() > 0.57 and sph[facing].max() < 0.8
    assert sph[away].min() > 0.95
    again = oracle.render_spherical(vox, sub.numpy(), m.depth_weight.numpy())[0, 0]
    assert np.array_equal(sph, again)


def test_render_skip_brick_rule_never_hides_an_occupied_tap():
    """The empty-space-skipping renderer (csrc/render_sph.cu) may only call a sample empty when none of its VALID trilinear taps
    is occupied.  Emulates its marking rule (occupied voxel v marks bricks floor((v-2)/4) .. floor((v+1)/4), clipped to the
    volume; a marked boundary brick 0 also marks the outside brick -1) and its lookup (brick floor(f_est / 4), f_est an fp32
    estimate within 1e-4 of the exact coordinate f) in one dimension -- the 3-D rule is the product of three such tests --
    over every voxel position and a dense sweep of sample coordinates, boundary cases included."""
    R, BR = 128, 4
    rng = np.random.RandomState(0)
    for v in list(range(0, 20)) + list(range(100, 128)) + [63, 64, 65]:
        marked = set(range(max(v - 2, 0) // BR, min(v + 1, R - 1) // BR + 1))
        if 0 in marked:
            marked.add(-1)
        f = np.concatenate([np.linspace(-2.0, 130.0, 26401), v + rng.uniform(-1.2, 1.2, 2000)])
        t0 = np.floor(f).astype(int)
        touches = ((t0 == v) & (t0 >= 0) & (t0 < R)) | ((t0 + 1 == v) & (t0 + 1 >= 0) & (t0 + 1 < R))
        for err in (-1e-4, 0.0, 1e-4):
            brick = np.floor((f + err) / BR).astype(int)
            hidden = touches & ~np.isin(brick, list(marked))
            # a tap may only be "hidden" when its interpolation weight is below the estimate's error
            w = np.where(t0 == v, 1.0 - (f - t0), f - t0)
            assert not (hidden & (w > 2e-4)).any(), (v, err, f[hidden & (w > 2e-4)][:5])
