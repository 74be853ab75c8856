"""GPU parity tests: the CUDA path, called through the C ABI (via the Python mirror of the reference's
toolbox packages), against
  (1) the CPU oracle (oracle/genre_oracle.c) on seeded inputs small enough to finish in seconds,
  (2) the reference's OWN kernels at BASELINE sizes, through golden outputs recorded from them
      (tests/golden/ref_*.npz, written by tests/golden/make_golden_fullsize.py),
  (3) size-independent properties (point conservation, determinism, idempotence).
Bars (BASELINE.json north_star): voxel / neighbour indices bit-exact, values within 1e-4 (most are far tighter).
"""
import hashlib
import os

import numpy as np
import pytest
import torch

from genre_shapehd_b200 import _lib
from genre_shapehd_b200.synth import sphere_depth, uniform_depth
from nndistance.functions.nnd import NNDFunction, nndistance, nndistance_score
from toolbox.calc_prob.calc_prob.functions.calc_prob import CalcStopProb
from toolbox.cam_bp.cam_bp._ext import cam_bp_lib
from toolbox.cam_bp.cam_bp.functions import CameraBackProjection, SphericalBackProjection, get_surface_mask
from toolbox.cam_bp.cam_bp.modules.camera_backprojection_module import Camera_back_projection_layer
from toolbox.spherical_proj import gen_sph_grid, render_spherical, sph_pad

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden(name):
    """outputs of the reference's own kernels on the test's inputs (see tests/golden/make_golden_fullsize.py)"""
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def sha(t):
    return hashlib.sha256(t.detach().contiguous().cpu().numpy().tobytes()).hexdigest()


def assert_sampled(got, r, name, tol, stride):
    """|got - reference| <= tol at the stored every-stride-th elements, and over the whole tensor on average"""
    flat = got.detach().reshape(-1)
    assert (flat[::stride].cpu() - torch.from_numpy(r[name])).abs().max().item() <= tol, name
    assert abs(flat.double().sum().item() - float(r[name + "_sum_f64"])) <= tol * flat.numel(), name


def assert_hits(tdf, cnt, r, tol):
    """a back-projection against the reference's: counts bit for bit, distances at every stored hit voxel"""
    assert sha(cnt) == str(r["cnt_sha256"]), "counts differ from the reference kernel"
    idx = torch.from_numpy(r["idx"].astype(np.int64)).to(tdf.device)
    assert (tdf.reshape(-1)[idx].cpu() - torch.from_numpy(r["tdf"])).abs().max().item() < tol
    assert abs(tdf.double().sum().item() - float(r["tdf_sum_f64"])) <= tol * tdf.numel()


def dev(a, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).to(DEV)


def test_native_library_is_loaded_and_there_is_no_fallback():
    _lib.load()
    assert _lib.LIB_PATH.endswith("libgenre_b200.so")
    with pytest.raises((RuntimeError, AssertionError)):
        nndistance(torch.zeros(1, 4, 3), torch.zeros(1, 4, 3))


# --------------------------------------------------------------------------------------------------
# camera back-projection
# --------------------------------------------------------------------------------------------------
def _cam_inputs(oracle, n, c, hw, seed=0, bg=0.0):
    rng = np.random.RandomState(seed)
    d = np.stack([np.stack([oracle.uniform_depth(seed * 100 + i * c + j, hw, hw, background=bg) for j in range(c)])
                  for i in range(n)])
    fl = (418.3 * hw / 256 * rng.uniform(0.9, 1.1, size=(n, c))).astype(np.float32)
    cd = rng.uniform(2.0, 2.4, size=(n, c)).astype(np.float32)
    return d, fl, cd


@pytest.mark.parametrize("res,hw,n,c", [(32, 64, 2, 2), (16, 40, 3, 1), (21, 48, 2, 1), (128, 256, 2, 1)])
@pytest.mark.parametrize("shift", [False, True])
def test_cam_bp_forward_vs_oracle(oracle, res, hw, n, c, shift):
    d, fl, cd = _cam_inputs(oracle, n, c, hw, seed=res)
    d[0, 0, ::5, ::3] = -1.0
    tdf_o, cnt_o = oracle.cam_bp_forward(d, fl, cd, res, shift=shift)
    tdf = torch.empty((n, c, res, res, res), device=DEV)
    cnt = torch.empty_like(tdf)
    cam_bp_lib.back_projection_forward(dev(d), dev(cd), dev(fl), tdf, cnt, shift=shift)
    assert np.array_equal(cnt.cpu().numpy(), cnt_o), "voxel indices / counts must be bit-exact"
    np.testing.assert_allclose(tdf.cpu().numpy(), tdf_o, atol=2e-6 if shift else 2e-8, rtol=0)
    # without the count volume (inference contract) the TDF is the same
    tdf2 = torch.empty_like(tdf)
    cam_bp_lib.back_projection_forward(dev(d), dev(cd), dev(fl), tdf2, None, shift=shift)
    assert torch.equal(tdf, tdf2)


def test_cam_bp_forward_strided_and_rectangular_input(oracle):
    n, c, h, w, res = 2, 2, 48, 80, 32
    rng = np.random.RandomState(1)
    d = rng.uniform(1.8, 2.6, size=(n, c, h, w)).astype(np.float32)
    fl = np.full((n, c), 130.0, np.float32)
    cd = np.full((n, c), 2.2, np.float32)
    _, cnt_o = oracle.cam_bp_forward(d, fl, cd, res)
    base = dev(d)
    # the view GenRe feeds: permute(0,1,3,2) then flip (depth_pred_with_sph_inpaint.py:140-141); here built so that
    # the logical content is unchanged but the memory order is h-fastest
    view = base.permute(0, 1, 3, 2).contiguous().permute(0, 1, 3, 2)
    assert not view.is_contiguous() and torch.equal(view, base)
    for inp in (base, view, base[:, :, :, :].expand(n, c, h, w)):
        tdf = torch.empty((n, c, res, res, res), device=DEV)
        cnt = torch.empty_like(tdf)
        cam_bp_lib.back_projection_forward(inp, dev(cd), dev(fl), tdf, cnt)
        assert np.array_equal(cnt.cpu().numpy(), cnt_o)


@pytest.mark.parametrize("case", ["all_background_zero", "all_negative", "single_pixel", "everything_one_voxel"])
def test_cam_bp_forward_edge_cases(oracle, case):
    res, hw = 32, (64 if case == "everything_one_voxel" else 32)
    d = np.zeros((1, 1, hw, hw), np.float32)
    fl, cd = 52.0, 2.2
    if case == "all_negative":
        d[:] = -1.0
    elif case == "single_pixel":
        d[0, 0, 17, 9] = 2.25
    elif case == "everything_one_voxel":
        fl = 1.0e6  # telephoto: every ray is (almost) the optical axis -> 4096 pixels land in 4 voxels, 1024 each,
        # which makes the 32-bit partial sums of the splat kernel carry
        d[:] = 2.2 + 0.25 / res
    tdf_o, cnt_o = oracle.cam_bp_forward(d, fl, cd, res)
    out = CameraBackProjection.apply(dev(d), dev(np.full((1, 1), fl)), dev(np.full((1, 1), cd)), res)
    np.testing.assert_allclose(out.cpu().numpy(), tdf_o, atol=2e-8, rtol=0)
    if case == "everything_one_voxel":
        assert cnt_o.max() >= 1024
        cnt = torch.empty_like(out)
        cam_bp_lib.back_projection_forward(dev(d), dev(np.full((1, 1), cd)), dev(np.full((1, 1), fl)),
                                           torch.empty_like(out), cnt)
        assert np.array_equal(cnt.cpu().numpy(), cnt_o)


def test_cam_bp_forward_bucket_overflow_wall(oracle):
    """A fronto-parallel wall puts ~all 65536 pixels into a few 4096-voxel tiles: every tile bucket (1024 records)
    spills into the per-map overflow list, which the splat CTAs then have to pick apart."""
    hw = 256
    hh = np.arange(hw, dtype=np.float64)[:, None] - (hw - 1) / 2.0
    ww = np.arange(hw, dtype=np.float64)[None, :] - (hw - 1) / 2.0
    norm = np.sqrt(hh * hh + ww * ww + 418.3 ** 2)
    wall = ((2.2 + 0.1037) * norm / 418.3).astype(np.float32)  # plane depth 2.3037 -> constant x
    d = np.stack([wall, wall * 0.97])[:, None]
    tdf_o, cnt_o = oracle.cam_bp_forward(d, 418.3, 2.2, 128, shift=True)
    assert cnt_o.sum() > 30000
    tdf = torch.empty((2, 1, 128, 128, 128), device=DEV)
    cnt = torch.empty_like(tdf)
    fl, cd = torch.full((2, 1), 418.3, device=DEV), torch.full((2, 1), 2.2, device=DEV)
    cam_bp_lib.back_projection_forward(dev(d), cd, fl, tdf, cnt, shift=True)
    assert np.array_equal(cnt.cpu().numpy(), cnt_o)
    np.testing.assert_allclose(tdf.cpu().numpy(), tdf_o, atol=2e-6, rtol=0)
    # at least one tile really overflowed its bucket
    per_tile = cnt_o.reshape(2, -1, 4096).sum(-1)
    assert per_tile.max() > 1024


@pytest.mark.parametrize("n", [1, 4])
def test_cam_bp_forward_vs_reference_kernel_at_full_size(oracle, n):
    r = golden("ref_cam_bp_forward_n%d" % n)
    d = oracle.bench_depth_batch(n)
    depth = dev(d)
    fl = torch.full((n, 1), 418.3, device=DEV)
    cd = torch.full((n, 1), 2.2, device=DEV)
    tdf = torch.empty((n, 1, 128, 128, 128), device=DEV)
    cnt = torch.empty_like(tdf)
    cam_bp_lib.back_projection_forward(depth, cd, fl, tdf, cnt)
    assert_hits(tdf, cnt, r, 1e-7)
    assert (cnt.sum().item()) > 10000 * n and int((cnt != 0).sum()) == int(r["n_hits"])
    # module path with fused shift == reference module path (shift_tdf as two dense torch ops)
    out = Camera_back_projection_layer()(depth)
    idx = torch.from_numpy(r["idx"].astype(np.int64)).to(DEV)
    assert (out.reshape(-1)[idx].cpu() - (1 - 128 * torch.from_numpy(r["tdf"]))).abs().max().item() < 1e-5
    assert (out - (1 - 128 * tdf)).abs().max().item() < 1e-5
    assert torch.equal(out == 0, cnt == 0)


def test_cam_bp_forward_is_bitwise_deterministic(oracle):
    d = dev(oracle.bench_depth_batch(4))
    layer = Camera_back_projection_layer()
    a = layer(d)
    for _ in range(3):
        assert torch.equal(a, layer(d))


def test_cam_bp_point_conservation_at_bench_size(oracle):
    """every in-bounds foreground pixel lands in exactly one voxel: sum(cnt) == #valid pixels (oracle index)"""
    d = oracle.bench_depth_batch(8)
    vidx = oracle.cam_bp_voxel_index(d, 418.3, 2.2, 128)
    import importlib
    get_vox_surface_cnt = importlib.import_module("toolbox.cam_bp.cam_bp.functions.get_surface_mask").get_vox_surface_cnt
    cnt = get_vox_surface_cnt(dev(d), torch.full((8, 1), 418.3, device=DEV), torch.full((8, 1), 2.2, device=DEV), 128)
    per_map = cnt.sum(dim=(1, 2, 3, 4)).cpu().numpy()
    assert np.array_equal(per_map, (vidx >= 0).sum(axis=(1, 2, 3)).astype(np.float32))
    # and the histogram of voxel ids is identical
    for i in (0, 1, 7):
        expect = np.bincount(vidx[i][vidx[i] >= 0], minlength=128 ** 3).astype(np.float32)
        assert np.array_equal(cnt[i, 0].reshape(-1).cpu().numpy(), expect)


@pytest.mark.parametrize("res,hw,n,c", [(32, 64, 2, 2), (128, 256, 1, 1)])
def test_cam_bp_backward_vs_oracle(oracle, res, hw, n, c):
    d, fl, cd = _cam_inputs(oracle, n, c, hw, seed=7)
    _, cnt_o = oracle.cam_bp_forward(d, fl, cd, res)
    g = np.random.RandomState(3).randn(n, c, res, res, res).astype(np.float32)
    gd_o, gfl_o, gcd_o = oracle.cam_bp_backward(d, fl, cd, cnt_o, g, res)
    depth = dev(d).requires_grad_(True)
    flt, cdt = dev(fl).requires_grad_(True), dev(cd).requires_grad_(True)
    out = CameraBackProjection.apply(depth, flt, cdt, res)
    out.backward(dev(g))
    np.testing.assert_allclose(depth.grad.cpu().numpy(), gd_o, atol=1e-5, rtol=1e-5)
    np.testing.assert_allclose(flt.grad.cpu().numpy(), gfl_o, rtol=2e-4, atol=1e-5)
    np.testing.assert_allclose(cdt.grad.cpu().numpy(), gcd_o, rtol=2e-4, atol=1e-4)
    if res == 128:  # the fused-shift module differentiates to -res * the same thing
        depth2 = dev(d).requires_grad_(True)
        Camera_back_projection_layer()(depth2, float(fl[0, 0]), float(cd[0, 0])).backward(dev(g))
        np.testing.assert_allclose(depth2.grad.cpu().numpy(), -128 * gd_o, atol=2e-3, rtol=1e-4)


def test_cam_bp_backward_vs_reference_kernel_single_sample(oracle):
    """N == 1 only: the reference kernel reads cam_dist out of bounds for n >= 1 (back_projection_kernel.cu:401)."""
    r = golden("ref_cam_bp_backward")
    d = dev(oracle.bench_depth_batch(2)[1:2])
    fl = torch.full((1, 1), 418.3, device=DEV)
    cd = torch.full((1, 1), 2.2, device=DEV)
    tdf = torch.empty((1, 1, 128, 128, 128), device=DEV)
    cnt = torch.empty_like(tdf)
    cam_bp_lib.back_projection_forward(d, cd, fl, tdf, cnt)
    assert_hits(tdf, cnt, r, 1e-7)
    g = torch.randn(1, 1, 128, 128, 128, device=DEV, generator=torch.Generator(DEV).manual_seed(0))
    gfl_r, gcd_r = float(r["grad_fl"].reshape(-1)[0]), float(r["grad_camdist"].reshape(-1)[0])
    gd = torch.empty_like(d)
    gfl = torch.empty(r["grad_fl"].shape, device=DEV)
    gcd = torch.empty(r["grad_camdist"].shape, device=DEV)
    cam_bp_lib.back_projection_backward(d, fl, cd, cnt, g, gd, gcd, gfl)
    assert_sampled(gd, r, "grad_depth", 1e-5, 14)
    assert abs(gfl.item() - gfl_r) <= 2e-4 * max(1.0, abs(gfl_r))
    assert abs(gcd.item() - gcd_r) <= 2e-4 * max(1.0, abs(gcd_r))


@pytest.mark.parametrize("res,hw", [(32, 64), (21, 40)])
def test_surface_mask_vs_oracle(oracle, res, hw):
    fl, cd = 418.3 * hw / 256, 2.2
    d = np.stack([oracle.sphere_depth(hw, hw, fl=fl, radius=0.35, background=-1.0),
                  oracle.uniform_depth(3, hw, hw, background=-1.0)])[:, None]
    _, cnt_o = oracle.cam_bp_forward(d, fl, cd, res)
    mask_o = oracle.surface_mask(d, fl, cd, cnt_o, res)
    surf, mask = get_surface_mask(dev(d), float(fl), 2.2, res)
    assert np.array_equal(mask.cpu().numpy(), mask_o)
    assert np.array_equal(surf.cpu().numpy(), np.clip(cnt_o, 0, 1))


def test_surface_mask_vs_reference_kernel(oracle):
    r = golden("ref_surface_mask")
    d = oracle.bench_depth_batch(2)
    d[d == 0] = -1.0
    depth = dev(d)
    fl = torch.full((2, 1), 418.3, device=DEV)
    cd = torch.full((2, 1), 2.2, device=DEV)
    tdf = torch.empty((2, 1, 128, 128, 128), device=DEV)
    cnt = torch.empty_like(tdf)
    cam_bp_lib.back_projection_forward(depth, cd, fl, tdf, cnt)
    assert sha(cnt) == str(r["cnt_sha256"])
    mask = torch.empty_like(cnt)
    cam_bp_lib.get_surface_mask(depth, cd, fl, cnt, mask)
    assert sha(mask) == str(r["mask_sha256"]), "surface mask differs from the reference kernel"
    assert 0.05 < (mask == 0).float().mean().item() < 0.9


# --------------------------------------------------------------------------------------------------
# spherical back-projection
# --------------------------------------------------------------------------------------------------
def _sph_inputs(n, s, seed):
    rng = np.random.RandomState(seed)
    sph = rng.uniform(0.02, 0.7, size=(n, 1, s, s)).astype(np.float32)
    sph[0, 0, : s // 8] = -0.5
    return sph


@pytest.mark.parametrize("res,s,n", [(32, 32, 2), (20, 24, 3), (128, 128, 2)])
def test_sph_bp_forward_backward_vs_oracle(oracle, res, s, n):
    sph = _sph_inputs(n, s, res)
    grid1 = gen_sph_grid(s)
    tdf_o, cnt_o = oracle.sph_bp_forward(sph, grid1.numpy(), res)
    g = np.random.RandomState(1).randn(n, 1, res, res, res).astype(np.float32)
    gs_o = oracle.sph_bp_backward(sph, grid1.numpy(), cnt_o, g, res)
    grid = grid1.to(DEV).expand(n, -1, -1, -1, -1)  # batch stride 0, as genre_full_model.py:136-137
    assert grid.stride(0) == 0
    x = dev(sph).requires_grad_(True)
    tdf, cnt = SphericalBackProjection.apply(x, grid, res)
    assert np.array_equal(cnt.cpu().numpy(), cnt_o)
    np.testing.assert_allclose(tdf.detach().cpu().numpy(), tdf_o, atol=2e-8, rtol=0)
    tdf.backward(dev(g))
    # (r - dir.centre) / (cnt * dist) is ill-conditioned for points near their voxel centre; FMA contraction of the
    # dot products differs between nvcc and the oracle build
    np.testing.assert_allclose(x.grad.cpu().numpy(), gs_o, atol=2e-4 * max(1.0, np.abs(gs_o).max()), rtol=2e-3)


def test_sph_bp_vs_reference_kernels_full_size():
    r = golden("ref_sph_bp")
    n = 3
    sph = dev(_sph_inputs(n, 128, 5))
    grid = gen_sph_grid().to(DEV).expand(n, -1, -1, -1, -1)
    tdf = torch.empty((n, 1, 128, 128, 128), device=DEV)
    cnt = torch.empty_like(tdf)
    cam_bp_lib.spherical_back_proj_forward(sph, grid, tdf, cnt)
    assert_hits(tdf, cnt, r, 1e-7)
    g = torch.randn(tdf.shape, device=DEV, generator=torch.Generator(DEV).manual_seed(1))
    gs = torch.empty_like(sph)
    cam_bp_lib.spherical_back_proj_backward(sph, grid, cnt, g, gs)
    assert_sampled(gs, r, "grad_sph", 1e-4 * max(1.0, float(r["grad_sph_absmax"])), 14)


def test_genre_backproject_spherical_glue_runs_on_the_new_op():
    """Net.backproject_spherical, models/genre_full_model.py:134-143, verbatim on top of the new op."""
    n, margin = 2, 16
    sph = torch.rand(n, 1, 160, 160, device=DEV) * 0.5 + 0.3
    grid = gen_sph_grid().to(DEV).expand(1, -1, -1, -1, -1)[0].expand(n, -1, -1, -1, -1)
    crop = sph[:, :, margin:160 - margin, margin:160 - margin]
    proj_df, cnt = SphericalBackProjection().apply(1 - crop, grid, 128)
    mask = torch.clamp(cnt.detach(), 0, 1)
    out = (-proj_df + 1 / 128) * 128 * mask
    assert out.shape == (n, 1, 128, 128, 128) and torch.isfinite(out).all()
    assert out.max().item() <= 1.0 and (out[mask == 0] == 0).all()


# --------------------------------------------------------------------------------------------------
# stop probability
# --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(2, 1, 8, 8, 256), (1, 1, 5, 3, 64), (1, 2, 3, 3, 37), (1, 1, 2, 2, 300)])
def test_calc_prob_vs_oracle(oracle, shape):
    rng = np.random.RandomState(sum(shape))
    p = np.clip(rng.rand(*shape), 1e-5, 1 - 1e-5).astype(np.float32)
    p[0, 0, 0, 0, 3:9] = 1 - 1e-5  # a solid run drives the transmittance to the denormal range
    s_o = oracle.calc_prob_forward(p)
    x = dev(p).requires_grad_(True)
    s = CalcStopProb.apply(x)
    np.testing.assert_allclose(s.detach().cpu().numpy(), s_o, rtol=1e-4, atol=1e-7)
    g = rng.randn(*shape).astype(np.float32)
    s.backward(dev(g))
    grad_o = oracle.calc_prob_backward(p, s_o * g)
    scale = np.abs(grad_o).max()
    np.testing.assert_allclose(x.grad.cpu().numpy(), grad_o, rtol=1e-3, atol=1e-5 * scale)


def test_calc_prob_backward_is_finite_when_the_last_sample_is_certain():
    """ADVICE r1: p[Z-1] == 1 made the last sample's gradient 0/0; the reference special-cases it as w/p (calc_prob_kernel.cu:169-172)"""
    p = torch.rand(3, 1, 4, 4, 64, device=DEV).clamp_(0.05, 0.95)
    p[..., -1] = 1.0
    p.requires_grad_(True)
    s = CalcStopProb.apply(p)
    g = torch.rand_like(s)
    (gp,) = torch.autograd.grad(s, p, g)
    assert torch.isfinite(gp).all()
    # last sample: d s_last / d p_last = prod_{k<last}(1 - p_k), nothing follows it
    trans = torch.cumprod(1 - p.detach(), dim=-1)[..., -2]
    assert torch.allclose(gp[..., -1], g[..., -1] * trans, rtol=1e-4, atol=1e-7)


def test_calc_prob_vs_reference_kernels_full_size(oracle):
    """every element against the CPU oracle (the reference's loop order, one rounding per fp32 op), and a fixed subset of
    the elements against the reference's own kernels"""
    gen = torch.Generator(DEV).manual_seed(0)
    p = torch.rand(2, 1, 128, 128, 256, device=DEV, generator=gen).clamp_(1e-5, 1 - 1e-5)
    p = torch.where(torch.rand(p.shape, device=DEV, generator=gen) < 0.9, torch.full_like(p, 1e-5), p)
    r = golden("ref_calc_prob")
    k = int(r["stride"])
    s = CalcStopProb.apply(p)
    s_o = torch.from_numpy(oracle.calc_prob_forward(p.cpu().numpy()))
    assert (s.cpu() - s_o).abs().max().item() < 1e-5
    torch.testing.assert_close(s.cpu(), s_o, rtol=1e-4, atol=1e-7)
    assert_sampled(s, r, "stop", 1e-5, k)
    torch.testing.assert_close(s.reshape(-1)[::k].cpu(), torch.from_numpy(r["stop"]), rtol=1e-4, atol=1e-7)
    g = torch.randn(p.shape, device=DEV, generator=gen)
    from toolbox.calc_prob.calc_prob._ext import calc_prob_lib
    gr = torch.empty_like(p)
    calc_prob_lib.calc_prob_backward(p, (s * g).contiguous(), gr)
    gr_o = torch.from_numpy(oracle.calc_prob_backward(p.cpu().numpy(), (s * g).cpu().numpy()))
    assert (gr.cpu() - gr_o).abs().max().item() <= 1e-4 * gr_o.abs().max().item()
    assert_sampled(gr, r, "grad_prob", 1e-4 * float(r["grad_prob_absmax"]), k)


# --------------------------------------------------------------------------------------------------
# fused spherical renderer
# --------------------------------------------------------------------------------------------------
def _occupancy(n, res, seed):
    gen = torch.Generator(DEV).manual_seed(seed)
    v = torch.full((n, 1, res, res, res), 1e-5, device=DEV)
    c = (torch.arange(res, device=DEV) + 0.5) / res - 0.5
    X, Y, Z = torch.meshgrid(c, c, c, indexing="ij")
    for i in range(n):
        r = torch.sqrt((X - 0.05 * i) ** 2 + Y ** 2 + (Z + 0.03 * i) ** 2)
        shell = (r - 0.3).abs() < 1.2 / res
        v[i, 0][shell] = 1 - 1e-5
    soft = torch.rand(v.shape, device=DEV, generator=gen) * 0.05
    return torch.clamp(v + soft * (torch.rand(v.shape, device=DEV, generator=gen) < 0.02), 1e-5, 1 - 1e-5)


@pytest.mark.parametrize("res,s,z", [(24, 16, 64), (32, 8, 50), (128, 128, 256), (40, 24, 100)])
def test_render_spherical_fused_vs_oracle_and_unfused(oracle, res, s, z):
    """the renderer (empty-space skipping included: res % 4 == 0 in every case) against the INDEPENDENT CPU oracle at every
    size, full GenRe size (128^3, 128x128 rays, 256 samples) included, and against the op-by-op torch composition"""
    m = render_spherical(sph_res=s, z_res=z).to(DEV)
    n = 2
    vox = _occupancy(n, res, 1) if res >= 32 else torch.rand(n, 1, res, res, res, device=DEV)
    out = m(vox)
    assert out.shape == (n, 1, s, s)
    ref = m.forward_unfused(vox)  # grid_sample(align_corners=True) + clamp + CalcStopProb + matmul + prod
    assert (out - ref).abs().max().item() < 1e-4
    o = oracle.render_spherical(vox.cpu().numpy(), m.grid.cpu().numpy(), m.depth_weight.cpu().numpy())
    np.testing.assert_allclose(out.cpu().numpy(), o, atol=2e-5)


@pytest.mark.parametrize("kind", ["empty", "shell", "dense", "genre", "corner_voxel", "zeros_and_negatives"])
def test_render_spherical_skipping_equals_the_plain_kernel(kind):
    """genre_b200_render_spherical_forward_skip against genre_b200_render_spherical_forward (no skipping) on inputs that
    stress the occupancy logic: nothing occupied, a thin shell, everything occupied, GenRe's own clamp(cam_bp * 50) volume,
    single voxels at brick / volume corners, and raw volumes with exact zeros and negative values"""
    from genre_shapehd_b200 import _lib
    from toolbox.spherical_proj import render_forward
    res, s, z, n = 128, 128, 256, 2
    m = render_spherical(sph_res=s, z_res=z).to(DEV)
    if kind == "empty":
        vox = torch.full((n, 1, res, res, res), 1e-5, device=DEV)
    elif kind == "shell":
        vox = _occupancy(n, res, 3)
    elif kind == "dense":
        vox = torch.rand(n, 1, res, res, res, device=DEV)
    elif kind == "genre":
        d = torch.from_numpy(np.stack([sphere_depth(radius=0.35), uniform_depth(1)])[:, None]).to(DEV)
        vox = torch.clamp(Camera_back_projection_layer()(d) * 50, 1e-5, 1 - 1e-5)
    elif kind == "corner_voxel":
        vox = torch.full((n, 1, res, res, res), 1e-5, device=DEV)
        for (x, y, zz) in [(0, 0, 0), (127, 127, 127), (7, 8, 63), (64, 64, 64), (8, 7, 120), (127, 0, 64)]:
            vox[0, 0, x, y, zz] = 0.9
        vox[1, 0, 56:72, 63, 64] = 0.5
    else:
        vox = torch.zeros(n, 1, res, res, res, device=DEV)
        vox[0, 0, 40:50, 40:50, 40:50] = -3.0
        vox[1, 0, 60:70, 60:70, 60:70] = 0.3
    out = m(vox)
    plain = torch.empty_like(out)
    _lib.call("genre_b200_render_spherical_forward", vox.data_ptr(), n, res, m._dirs_on(vox.device).data_ptr(), s, z,
              m.depth_weight.data_ptr(), plain.data_ptr(), _lib.stream_ptr(vox))
    assert (out - plain).abs().max().item() <= 1e-5     # closed-form q^n against the sample-by-sample fp32 product chain
    # the pre-transform form: clamp(v * 50, 1e-5, 1 - 1e-5) applied on the fly, skipping decided on the transformed values
    raw = vox / 50
    a, b = torch.empty_like(out), torch.empty_like(out)
    render_forward(raw, n, res, m._dirs_on(vox.device), s, z, m.depth_weight, a, pre=(50.0, 1e-5, 1 - 1e-5))
    _lib.call("genre_b200_render_spherical_forward_pre", raw.data_ptr(), n, res, m._dirs_on(vox.device).data_ptr(), s, z,
              m.depth_weight.data_ptr(), 50.0, 1e-5, 1 - 1e-5, b.data_ptr(), _lib.stream_ptr(vox))
    assert (a - b).abs().max().item() <= 1e-5


def test_render_spherical_backward_vs_autograd_of_the_composition():
    m = render_spherical(sph_res=16, z_res=64).to(DEV)
    vox = (torch.rand(2, 1, 24, 24, 24, device=DEV) * 0.5 + 0.05)
    vox[:, :, 9:13, 9:13, 9:13] = 0.97
    g = torch.randn(2, 1, 16, 16, device=DEV)
    a = vox.clone().requires_grad_(True)
    m(a).backward(g)
    b = vox.clone().requires_grad_(True)
    m.forward_unfused(b).backward(g)
    scale = b.grad.abs().max().item()
    assert (a.grad - b.grad).abs().max().item() <= 2e-4 * scale


@pytest.mark.parametrize("batch", [1, 3])
def test_fused_genre_glue_matches_the_callers_op_by_op_lines(oracle, batch):
    """genre_shapehd_b200/fused.py against the frozen callers' glue (depth_pred_with_sph_inpaint.py:120-126,
    genre_full_model.py:120-143) run on the drop-in ops; differences are rounding only"""
    from genre_shapehd_b200.fused import GenRe3DGlue
    from genre_shapehd_b200.synth import bench_depth_batch
    glue = GenRe3DGlue().to(DEV)
    depth = dev(bench_depth_batch(batch))
    with torch.no_grad():
        proj, sph_in = glue.project_and_render(depth)
        # the callers' lines
        proj_ref = Camera_back_projection_layer()(depth)
        sph_ref = sph_pad(glue.render(torch.clamp(proj_ref * 50, 1e-5, 1 - 1e-5)), 16)
        assert torch.equal(proj, proj_ref)
        assert (sph_in - sph_ref).abs().max().item() <= 1e-6
        # a stand-in for the inpainting net's output: the padded partial map, perturbed
        g = torch.Generator(device=DEV).manual_seed(3)
        pred_sph = (sph_ref + 0.01 * torch.rand(sph_ref.shape, device=DEV, generator=g)).clamp(0, 1)
        refine = glue.refine_input(proj, pred_sph)
        grid = glue.grid.expand(batch, -1, -1, -1, -1)
        crop = pred_sph[:, :, 16:144, 16:144]
        df, cnt = SphericalBackProjection.apply(1 - crop, grid, 128)
        ps = (-df + 1 / 128) * 128 * torch.clamp(cnt, 0, 1)
        pd = torch.clamp((proj_ref * 50) / 50, 1e-5, 1 - 1e-5)
        ref = torch.cat((ps, pd), dim=1)
    assert refine.shape == ref.shape
    assert torch.equal(refine[:, 0] != 0, ps[:, 0] != 0)                      # same hit voxels
    assert (refine - ref).abs().max().item() <= 1e-5


def test_sph_pad_and_grid_buffers_match_reference_layout():
    m = render_spherical()
    assert tuple(m.grid.shape) == (128, 128, 256, 3) and tuple(m.depth_weight.shape) == (256,)
    assert set(dict(m.named_buffers())) == {"grid", "depth_weight"}
    x = torch.arange(128 * 128, dtype=torch.float32, device=DEV).reshape(1, 1, 128, 128)
    p = sph_pad(x, 16)
    assert p.shape == (1, 1, 160, 160)
    assert torch.equal(p[0, 0, 16:144, 16:144], x[0, 0])
    assert torch.equal(p[0, 0, 16:144, :16], x[0, 0, :, 112:128])   # horizontal wrap of the azimuth
    assert torch.equal(p[0, 0, 16:144, 144:], x[0, 0, :, :16])


# --------------------------------------------------------------------------------------------------
# Chamfer nearest neighbour
# --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("b,n,m", [(1, 50, 50), (2, 257, 1300), (4, 1024, 777), (1, 1, 5), (3, 5, 1)])
def test_nnd_forward_backward_vs_oracle(oracle, b, n, m):
    rng = np.random.RandomState(n + m)
    p1 = (rng.rand(b, n, 3) - 0.5).astype(np.float32)
    p2 = (rng.rand(b, m, 3) - 0.5).astype(np.float32)
    p2[:, m // 2] = p2[:, 0]  # exact duplicate candidates: ties must resolve to the lower index
    d1o, d2o, i1o, i2o = oracle.nnd_forward(p1, p2, fused=True)
    x1, x2 = dev(p1).requires_grad_(True), dev(p2).requires_grad_(True)
    d1, d2, i1, i2 = NNDFunction.apply(x1, x2)
    assert np.array_equal(i1.cpu().numpy(), i1o) and np.array_equal(i2.cpu().numpy(), i2o)
    assert np.array_equal(d1.detach().cpu().numpy(), d1o) and np.array_equal(d2.detach().cpu().numpy(), d2o)
    g1, g2 = rng.rand(b, n).astype(np.float32), rng.rand(b, m).astype(np.float32)
    (d1 * dev(g1)).sum().backward(retain_graph=True)
    (d2 * dev(g2)).sum().backward()
    o1, o2 = oracle.nnd_backward(p1, p2, g1, g2, i1o, i2o)
    np.testing.assert_allclose(x1.grad.cpu().numpy(), o1, atol=1e-5)
    np.testing.assert_allclose(x2.grad.cpu().numpy(), o2, atol=1e-5)


@pytest.mark.parametrize("b,n,m", [(4, 4096, 4096), (2, 3000, 5000)])
def test_nnd_vs_reference_kernels(b, n, m):
    r = golden("ref_nnd_%d_%d_%d" % (b, n, m))
    gen = torch.Generator(DEV).manual_seed(n)
    x1 = torch.rand(b, n, 3, device=DEV, generator=gen) - 0.5
    x2 = torch.rand(b, m, 3, device=DEV, generator=gen) - 0.5
    d1, d2, i1, i2 = NNDFunction.apply(x1, x2)
    assert sha(i1) == str(r["idx1_sha256"]) and sha(i2) == str(r["idx2_sha256"])
    assert sha(d1) == str(r["dist1_sha256"]) and sha(d2) == str(r["dist2_sha256"])
    g1, g2 = torch.rand(b, n, device=DEV, generator=gen), torch.rand(b, m, device=DEV, generator=gen)
    from nndistance._ext import my_lib
    o1, o2 = torch.empty_like(x1), torch.empty_like(x2)
    my_lib.nnd_backward_cuda(x1, x2, o1, o2, g1, g2, i1, i2)
    assert_sampled(o1, r, "grad_xyz1", 1e-5, 14)
    assert_sampled(o2, r, "grad_xyz2", 1e-5, 14)


def test_nnd_score_and_layouts():
    x1 = torch.rand(2, 3, 100, device=DEV)  # [B,3,N] is transposed by nndistance(), nnd.py:73-76
    x2 = torch.rand(2, 80, 3, device=DEV)
    s = nndistance_score(x1, x2)
    assert s.shape == (2,) and torch.isfinite(s).all()
    d1, d2 = nndistance(x1, x2)
    brute = torch.cdist(x1.transpose(1, 2), x2) ** 2
    assert (d1 - brute.min(2).values).abs().max().item() < 1e-5
    assert (d2 - brute.min(1).values).abs().max().item() < 1e-5


# --------------------------------------------------------------------------------------------------
# error behaviour through the C ABI
# --------------------------------------------------------------------------------------------------
def test_bad_arguments_raise_runtime_error():
    d = torch.zeros(1, 1, 8, 8, device=DEV)
    with pytest.raises((RuntimeError, ValueError)):
        cam_bp_lib.back_projection_forward(d, torch.zeros(2, 1, device=DEV), torch.zeros(1, 1, device=DEV),
                                           torch.empty(1, 1, 8, 8, 8, device=DEV), None)
    with pytest.raises(RuntimeError):
        _lib.call("genre_b200_cam_bp_forward", d.data_ptr(), 1, 1, 8, 8, 64, 64, 8, 1, d.data_ptr(), 1, 1,
                  d.data_ptr(), 1, 1, d.data_ptr(), None, 8, 0, d.data_ptr(), 16, None)


# --------------------------------------------------------------------------------------------------
# ground-truth surface voxels (SURVEY 8f-3): Model.preprocess of genre_full_model.py:86-96 on the GPU
# --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("res,iters,xform", [(128, 2, True), (64, 2, True), (32, 1, False), (96, 3, True), (128, 2, False)])
def test_voxel_surface_equals_scipy_binary_erosion(res, iters, xform):
    """bit-exact against the reference's own call: val - binary_erosion(val, ones((3,3,3)), iterations) after the transpose + flip"""
    from scipy.ndimage import binary_erosion
    from genre_shapehd_b200.postprocess import voxel_surface
    rng = np.random.RandomState(res + iters)
    c = (np.arange(res) + 0.5) / res - 0.5
    X, Y, Z = np.meshgrid(c, c, c, indexing="ij")
    vols = []
    for i in range(3):
        solid = ((X - 0.05 * i) ** 2 / 0.16 + Y ** 2 / 0.09 + (Z + 0.1 * i) ** 2 / 0.2) < 1.0           # an ellipsoid ...
        solid |= (np.abs(X) < 0.45) & (np.abs(Y + 0.3) < 0.06) & (np.abs(Z) < 0.49)                     # ... a slab touching the border
        solid &= rng.rand(res, res, res) > 0.002                                                       # ... with pin holes
        vols.append(solid.astype(np.float32))
    vols[2][0, :, :] = 1.0                                                                             # a face of the volume
    v = np.stack(vols)[:, None]
    out = voxel_surface(torch.from_numpy(v).to(DEV), iterations=iters, transpose_flip=xform).cpu().numpy()
    for i in range(3):
        val = v[i, 0]
        if xform:
            val = np.flip(np.transpose(val, (0, 2, 1)), 2)
        want = np.clip(val - binary_erosion(val, structure=np.ones((3, 3, 3)), iterations=iters).astype(float), 0, 1)
        assert np.array_equal(out[i, 0], want.astype(np.float32)), i


# --------------------------------------------------------------------------------------------------
# BASELINE full sizes: size-independent properties (the oracle runs in seconds only at small sizes)
# --------------------------------------------------------------------------------------------------
def test_cam_bp_full_batch32_checksums_and_batch_equivariance(oracle):
    """BASELINE configs[1] size (32 x 256x256 -> 128^3): per-map hit count = number of in-bounds foreground pixels (the oracle's
    bit-exact voxel indices), background voxels exactly 0, hit voxels in (0.13, 1], and permuting the batch permutes the
    output bit for bit (integer accumulation: no run-to-run or placement dependence)"""
    from genre_shapehd_b200.synth import bench_depth_batch
    d = bench_depth_batch(32)
    x = torch.from_numpy(d).to(DEV)
    layer = Camera_back_projection_layer()
    out = layer(x)
    idx = oracle.cam_bp_voxel_index(d, 418.3, 2.2, 128)              # [32,1,256,256] int32, -1 = skipped / out of bounds
    for n in (0, 1, 17, 31):
        hit = np.unique(idx[n][idx[n] >= 0])
        got = torch.nonzero(out[n].reshape(-1)).reshape(-1).cpu().numpy()
        assert np.array_equal(got, hit)
    hitv = out[out != 0]
    assert hitv.min().item() > 0.13 and hitv.max().item() <= 1.0
    perm = torch.randperm(32, device=DEV)
    assert torch.equal(layer(x[perm]), out[perm])
    assert torch.equal(layer(x), out)                                 # and run to run


def test_calc_prob_full_size_conserves_probability():
    """[16,1,128,128,256] (the GenRe size): sum_z stop_prob + prod_z (1 - p) == 1 for every ray"""
    gen = torch.Generator(DEV).manual_seed(4)
    p = torch.rand(16, 1, 128, 128, 256, device=DEV, generator=gen).pow_(6).clamp_(1e-5, 1 - 1e-5)
    s = CalcStopProb.apply(p)
    total = s.sum(-1, dtype=torch.float64) + torch.prod(1 - p.double(), dim=-1)
    assert (total - 1).abs().max().item() < 2e-5
    assert (s >= 0).all()


def test_render_and_sph_bp_batch_equivariance_full_size():
    """B=16 at GenRe sizes: the renderer (per-volume brick masks, strided ray groups) and the spherical back-projection give
    bit-identical per-sample results whatever the sample's position in the batch"""
    d = np.stack([sphere_depth(radius=0.3 + 0.008 * i) for i in range(16)])[:, None]
    vox = torch.clamp(Camera_back_projection_layer()(torch.from_numpy(d).to(DEV)) * 50, 1e-5, 1 - 1e-5)
    m = render_spherical().to(DEV)
    sph = m(vox)
    perm = torch.randperm(16, device=DEV)
    assert torch.equal(m(vox[perm]), sph[perm])
    assert torch.equal(m(vox[3:4]), sph[3:4])                         # batch 1: a different CTA count per volume
    grid = gen_sph_grid().to(DEV).expand(16, -1, -1, -1, -1)
    tdf, cnt = SphericalBackProjection.apply(1 - sph, grid, 128)
    tdf_p, cnt_p = SphericalBackProjection.apply((1 - sph)[perm].contiguous(), grid, 128)
    assert torch.equal(tdf_p, tdf[perm]) and torch.equal(cnt_p, cnt[perm])
    assert int(cnt.sum().item()) <= 16 * 128 * 128 and cnt.max().item() >= 1


def test_nnd_full_size_symmetry_and_minimality():
    """[4,16384,3] (BASELINE configs[4]): direction 1 of (a, b) is direction 2 of (b, a) bit for bit, every reported distance is
    the distance to the reported index, and no sampled candidate is closer"""
    gen = torch.Generator(DEV).manual_seed(9)
    a = torch.rand(4, 16384, 3, device=DEV, generator=gen) - 0.5
    b = torch.rand(4, 16384, 3, device=DEV, generator=gen) - 0.5
    d1, d2, i1, i2 = NNDFunction.apply(a, b)
    e1, e2, j1, j2 = NNDFunction.apply(b, a)
    assert torch.equal(d1, e2) and torch.equal(d2, e1) and torch.equal(i1, j2) and torch.equal(i2, j1)
    nb = torch.gather(b, 1, i1.long().unsqueeze(-1).expand(-1, -1, 3))
    diff = nb - a
    recomputed = torch.addcmul(torch.addcmul(diff[..., 1] * diff[..., 1], diff[..., 0], diff[..., 0]), diff[..., 2], diff[..., 2])
    assert (recomputed - d1).abs().max().item() <= 1e-9
    probe = b[:, torch.randint(0, 16384, (256,), device=DEV, generator=gen)]          # [4,256,3]
    dp = ((a.unsqueeze(2) - probe.unsqueeze(1)) ** 2).sum(-1).min(-1).values
    assert (d1 <= dp + 1e-7).all()
