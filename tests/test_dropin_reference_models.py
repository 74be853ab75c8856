"""GenRe and ShapeHD model classes (genre_shapehd_b200/genre_models.py) against the published GenRe-ShapeHD models.

The CPU tests rebuild the models under fixed seeds and compare their state_dict layout, parameter bytes and the 2D
U-ResNets' outputs with digests recorded from the original project (tests/golden/models_digest.json, written by
tests/golden/make_golden_models.py).  The GPU tests (``-m gpu``) run ``GenReNet.forward`` (BASELINE configs[2]) and one
ShapeHD training step on CUDA and check every hot-path tensor against the CPU oracle / torch fp32.
"""
import hashlib
import json
import os
import sys
import types

import numpy as np
import pytest
import torch

from genre_shapehd_b200 import compat
from genre_shapehd_b200 import genre_models as gm

DIGEST = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "models_digest.json")))["cases"]


def _mine(obj):
    from conftest import REPO
    mod = sys.modules[obj.__module__]
    return os.path.abspath(mod.__file__).startswith(os.path.join(REPO, "genre_shapehd_b200"))


def _layout(net):
    """(keys and shapes of the state_dict, sha256 of the parameter bytes), as tests/golden/make_golden_models.py records them"""
    sd = net.state_dict()
    h = hashlib.sha256()
    for k, v in sd.items():
        h.update(k.encode())
        h.update(np.ascontiguousarray(v.numpy()).tobytes())
    return [[k, list(v.shape)] for k, v in sd.items()], h.hexdigest()


def _assert_layout(keys, case):
    assert len(keys) == case["n_keys"]
    assert hashlib.sha256(json.dumps(keys).encode()).hexdigest() == case["state_dict_sha256"], "state_dict keys / shapes differ"


def _genre_net(joint_train=False):
    from genre_shapehd_b200.synth_genre import init_genre_net_for_bench
    torch.manual_seed(0)
    return init_genre_net_for_bench(gm.GenReNet(joint_train=joint_train))


def test_models_are_built_on_this_package():
    assert _mine(gm.Camera_back_projection_layer) and _mine(gm.SphericalBackProjection) and _mine(gm.Unet_3D)
    assert gm.gen_sph_grid.__module__ == "toolbox.spherical_proj" and _mine(gm.gen_sph_grid)
    assert _mine(gm.render_spherical)
    assert _mine(gm.VoxelGenerator) and _mine(gm.VoxelDiscriminator) and _mine(gm.VoxelDecoder) and _mine(gm.ImageEncoder)


def test_bootstrap_resolves_a_checkouts_own_modules(tmp_path, monkeypatch):
    """the zero-edit route (INTEGRATION.md §1): given a GenRe-ShapeHD checkout, its models/*.py and its 2D nets
    (networks/uresnet.py ...) import on top of this package's toolbox / networks.networks"""
    import networks
    (tmp_path / "models").mkdir()
    (tmp_path / "models" / "__init__.py").write_text("")
    (tmp_path / "models" / "probe_model.py").write_text(
        "from networks.networks import Unet_3D\nfrom networks.probe_uresnet import TAG\n"
        "from toolbox.cam_bp.cam_bp.functions import SphericalBackProjection\n")
    (tmp_path / "networks").mkdir()
    (tmp_path / "networks" / "probe_uresnet.py").write_text("TAG = 'checkout'\n")
    monkeypatch.setattr(sys, "path", list(sys.path))
    monkeypatch.setattr(networks, "__path__", list(networks.__path__))
    monkeypatch.delenv("GENRE_REF", raising=False)
    assert "models" not in sys.modules
    try:
        assert compat.bootstrap(str(tmp_path), offline_resnet=False) == str(tmp_path)
        import models.probe_model as probe
        assert probe.TAG == "checkout"
        assert os.path.abspath(probe.__file__).startswith(str(tmp_path))
        assert _mine(probe.Unet_3D) and _mine(probe.SphericalBackProjection)
    finally:
        for name in ("models", "models.probe_model", "networks.probe_uresnet"):
            sys.modules.pop(name, None)


def test_genre_net_builds_with_reference_constructor():
    """same state_dict keys, shapes and seeded parameters as the published Net (seed 0, then the bench's head init)"""
    net = _genre_net()
    assert _mine(type(net.refine_net)) and _mine(type(net.proj_depth))
    keys, sha = _layout(net)
    _assert_layout(keys, DIGEST["GenReNet"])
    assert sha == DIGEST["GenReNet"]["params_sha256"], "same seed must give the reference's parameters (creation order)"
    assert "grid" in dict(keys) and any(k.startswith("depth_and_inpaint.render_spherical.") for k, _ in keys)


@pytest.mark.parametrize("name,cls", [("ShapeHDNet", gm.ShapeHDNet), ("WganCritic", gm.WganCritic)])
def test_shapehd_models_match_the_reference_digests(name, cls):
    case = DIGEST[name]
    torch.manual_seed(case["seed"])
    keys, sha = _layout(cls())
    _assert_layout(keys, case)
    assert sha == case["params_sha256"]


def test_2d_nets_match_the_reference_on_cpu():
    """net1 (depth, normal, silhouette, min/max heads) and net2 (spherical inpainting) in eval mode, on seeded inputs"""
    case = DIGEST["GenReNet"]
    net = _genre_net().eval()
    torch.manual_seed(case["inputs_seed"])
    rgb, sph = torch.randn(1, 3, 256, 256), torch.rand(1, 1, 160, 160)
    with torch.no_grad():
        outs = {"net1": net.depth_and_inpaint.net1(types.SimpleNamespace(rgb=rgb)), "net2": net.depth_and_inpaint.net2(sph)}
    for which, out in outs.items():
        assert sorted(out) == sorted(case[which])
        for k, want in case[which].items():
            flat = out[k].reshape(-1).double()
            idx = torch.linspace(0, flat.numel() - 1, len(want["samples"])).long()
            scale = max(1.0, abs(want["abs_sum"]) / flat.numel())
            assert list(out[k].shape) == want["shape"], (which, k)
            np.testing.assert_allclose(flat[idx].numpy(), want["samples"], rtol=1e-4, atol=1e-5 * scale, err_msg=k)
            assert abs(float(flat.sum()) - want["sum"]) <= 1e-4 * max(1.0, want["abs_sum"]), (which, k)


def test_genre_forward_matches_the_reference_on_cpu():
    """the whole GenReNet.forward (2D nets, the glue between them and Unet_3D) against the original Net.forward on the CPU,
    both with the toolbox ops of oracle/cpu_toolbox (oracle/cpu_genre.py; its own process: another `toolbox`).  A depth
    that moves by one rounding can move a point into the next voxel, hence the sums' relative bound of 1e-3."""
    import subprocess
    from conftest import REPO
    p = subprocess.run([sys.executable, os.path.join(REPO, "oracle", "cpu_genre.py")], stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True, timeout=600, cwd=REPO)
    assert p.returncode == 0, p.stderr[-2000:]
    got = json.loads(p.stdout.strip().splitlines()[-1])
    want = DIGEST["GenReNet"]["forward_cpu"]
    assert sorted(got) == sorted(want)
    for k, w in want.items():
        g = got[k]
        assert g["shape"] == w["shape"], k
        assert abs(g["sum"] - w["sum"]) <= 1e-3 * max(1.0, w["abs_sum"]), k
        assert abs(g["abs_sum"] - w["abs_sum"]) <= 1e-3 * max(1.0, w["abs_sum"]), k
        scale = max(1.0, max(abs(v) for v in w["samples"]))
        np.testing.assert_allclose(g["samples"], w["samples"], rtol=0, atol=1e-4 * scale, err_msg=k)
    assert want["proj_depth"]["abs_sum"] > 0 and want["pred_proj_sph_full"]["abs_sum"] > 0   # the voxel path is exercised


def test_fold_batchnorm2d_eval_keeps_the_2d_nets_outputs():
    """compat.fold_batchnorm2d_eval (the 2D nets' cheap win used by bench.py): every BatchNorm2d of the U-ResNets
    disappears into its convolution and the outputs move only at rounding level"""
    net = _genre_net()
    net.eval()
    dn = net.depth_and_inpaint
    x = types.SimpleNamespace(rgb=torch.randn(1, 3, 256, 256))      # the min/max head needs the 8x8 encoder output of a 256^2 image
    s = torch.rand(1, 1, 160, 160)
    with torch.no_grad():
        a1, a2 = dn.net1(x), dn.net2(s)
        n = compat.fold_batchnorm2d_eval(dn.net1) + compat.fold_batchnorm2d_eval(dn.net2)
        b1, b2 = dn.net1(x), dn.net2(s)
    assert n == 124 and not any(isinstance(m, torch.nn.BatchNorm2d) for m in list(dn.net1.modules()) + list(dn.net2.modules()))
    for a, b in ((a1, b1), (a2, b2)):
        for k in a:
            assert (a[k] - b[k]).abs().max().item() <= 1e-5 * max(1.0, a[k].abs().max().item()), k
    assert compat.fold_batchnorm2d_eval(dn.net1) == 0            # idempotent


# ---- on the GPU: the models RUN on this package's kernels ---------------------------------------------------------------
def genre_inputs(batch, device, seed=0):
    """C3 inputs (SURVEY 8d): rgb ~ N(0,1), silhou = 100 * disc mask (scale_25d, marrnetbase.py:17)"""
    g = torch.Generator().manual_seed(seed)
    rgb = torch.randn(batch, 3, 256, 256, generator=g)
    yy, xx = torch.meshgrid(torch.arange(256.0), torch.arange(256.0), indexing="ij")
    sil = torch.stack([(((yy - 127.5) ** 2 + (xx - 127.5) ** 2) < (70.0 + 6 * i) ** 2).float() for i in range(batch)])[:, None] * 100
    return types.SimpleNamespace(rgb=rgb.to(device), silhou=sil.to(device))


@pytest.mark.gpu
def test_genre_full_model_forward_runs_on_cuda_and_matches_the_oracle(oracle):
    """GenReNet.forward (models/genre_full_model.py:116-132), B=2, eval, random init, on CUDA through the drop-in ops; every
    hot-path tensor it returns is recomputed from ITS OWN inputs by the CPU oracle (toolbox ops) / fp32 cuDNN (Unet_3D)."""
    from genre_shapehd_b200 import _lib, ops_conv
    dev = torch.device("cuda:0")
    net = _genre_net().to(dev).eval()
    captured = {}
    net.depth_and_inpaint.proj_depth.register_forward_pre_hook(lambda m, a: captured.__setitem__("depth", a[0].detach().clone()))
    n0 = _lib.launch_count
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False          # fp32 semantics of the reference: the conv kernels run their fp32-accurate mode
    try:
        with torch.no_grad():
            out = net(genre_inputs(2, dev))
            torch.cuda.synchronize()
            assert _lib.launch_count - n0 >= 10, "GenReNet did not run on this library's kernels"
            depth = captured["depth"]
            assert depth.shape == (2, 1, 256, 256) and not depth.is_contiguous()     # permuted + flipped view (depth_pred...:140-141)
            # cam_bp (a1, a3)
            tdf_o, cnt_o = oracle.cam_bp_forward(depth.cpu().numpy(), 418.3, 2.2, 128, shift=True)
            assert (cnt_o > 0).sum() > 2000, "the synthetic depth must hit the voxel grid (bench init of the minmax head)"
            proj = (out["proj_depth"] / 50).cpu().numpy()
            assert np.array_equal(proj != 0, cnt_o > 0)
            assert np.abs(proj - tdf_o).max() < 1e-5
            # render_spherical + sph_pad (a9, a10), full size, against the independent oracle
            rs = net.depth_and_inpaint.render_spherical
            vox = np.clip(tdf_o * np.float32(50), np.float32(1e-5), np.float32(1 - 1e-5))
            sph_o = oracle.render_spherical(vox, rs.grid.cpu().numpy(), rs.depth_weight.cpu().numpy())
            from toolbox.spherical_proj import sph_pad
            sph_o = sph_pad(torch.from_numpy(sph_o), 16).numpy()
            assert np.abs(out["pred_sph_partial"].cpu().numpy() - sph_o).max() < 1e-4
            # spherical back-projection glue (a4, a6)
            full = out["pred_sph_full"]
            crop = (1 - full[:, :, 16:144, 16:144]).cpu().numpy()
            from toolbox.spherical_proj import gen_sph_grid
            tdf_s, cnt_s = oracle.sph_bp_forward(crop, gen_sph_grid().numpy()[0], 128)
            want = (-tdf_s + np.float32(1 / 128)) * np.float32(128) * np.clip(cnt_s, 0, 1)
            got = out["pred_proj_sph_full"].cpu().numpy()
            assert np.array_equal(got != 0, want != 0) or np.abs(got - want).max() < 1e-4
            assert np.abs(got - want).max() < 1e-4
            # Unet_3D (a12): same module, same input, custom kernels off -> cuDNN fp32
            refine_in = torch.cat((out["pred_proj_sph_full"], out["pred_proj_depth"]), dim=1)
            enabled = ops_conv.ENABLED
            ops_conv.ENABLED = False
            try:
                ref = net.refine_net(refine_in)
            finally:
                ops_conv.ENABLED = enabled
            pv = out["pred_voxel"]
            assert pv.shape == (2, 1, 128, 128, 128) and torch.isfinite(pv).all()
            err = (pv - ref).abs().max().item()
            assert err <= 1e-4 * max(1.0, ref.abs().max().item()), "Unet_3D logits differ from cuDNN fp32 by %g" % err
            occ = (torch.sigmoid(pv) - torch.sigmoid(ref)).abs().max().item()
            assert occ <= 1e-4, "occupancies differ by %g" % occ
    finally:
        torch.backends.cudnn.allow_tf32 = tf32


@pytest.mark.gpu
def test_shapehd_training_step_runs_on_cuda():
    """ShapeHDNet.forward (models/shapehd.py:113-118) + the loss of :67-79 + backward + Adam step (BASELINE configs[3], B=2), on CUDA
    through the drop-in 3D nets; loss and the decoder's gradients are compared with the same step on cuDNN fp32."""
    from genre_shapehd_b200 import ops_conv
    dev = torch.device("cuda:0")
    torch.manual_seed(1)
    net = gm.ShapeHDNet().to(dev)
    net.train()
    g = torch.Generator().manual_seed(2)
    B = 2

    def batch():
        sil = (torch.rand(B, 1, 256, 256, generator=g) > 0.4).float()
        return types.SimpleNamespace(depth=torch.rand(B, 1, 256, 256, generator=g).to(dev), normal=torch.rand(B, 3, 256, 256, generator=g).to(dev),
                                     silhou=sil.to(dev))
    gt = (torch.rand(B, 1, 128, 128, 128, generator=g) < 0.05).float().to(dev)
    crit = torch.nn.BCEWithLogitsLoss()
    state = {k: v.clone() for k, v in net.state_dict().items()}
    inp = batch()

    def step(custom):
        net.load_state_dict(state)
        enabled = ops_conv.ENABLED
        ops_conv.ENABLED = custom
        tf32 = torch.backends.cudnn.allow_tf32
        torch.backends.cudnn.allow_tf32 = False
        try:
            opt = torch.optim.Adam(net.marrnet2.parameters(), lr=1e-3)
            opt.zero_grad()
            x = types.SimpleNamespace(depth=inp.depth.clone(), normal=inp.normal.clone(), silhou=inp.silhou.clone())
            pred = net(x)
            loss = crit(pred["voxel"], gt) + 1e-3 * (-pred["is_real"].mean())
            loss.backward()
            grads = {n: p.grad.detach().clone() for n, p in net.marrnet2.decoder.named_parameters() if p.grad is not None}
            opt.step()
            torch.cuda.synchronize()
            return loss.item(), grads
        finally:
            ops_conv.ENABLED = enabled
            torch.backends.cudnn.allow_tf32 = tf32
    loss_c, g_c = step(True)
    loss_r, g_r = step(False)
    assert np.isfinite(loss_c) and abs(loss_c - loss_r) <= 1e-4 * max(1.0, abs(loss_r))
    assert g_c.keys() == g_r.keys() and len(g_c) >= 10
    overall = max(v.abs().max().item() for v in g_r.values())
    for name in g_c:
        scale = g_r[name].abs().max().item()
        # two fp32 implementations with different summation orders, through training-mode BatchNorm at batch 2 and the BCE's
        # cancellation: weight gradients agree to a few 1e-3 of their scale.  The bias of a convolution that feeds a
        # training-mode BatchNorm has an exactly-zero gradient (the mean is subtracted): both sides hold rounding noise there,
        # hence the absolute floor.
        assert (g_c[name] - g_r[name]).abs().max().item() <= 1e-2 * scale + 1e-6 * overall, name
    for p in net.d.parameters():
        assert p.grad is None            # D stays frozen (shapehd.py:104-105)


@pytest.mark.gpu
def test_fused_batched_forward_equals_the_frozen_forward():
    """genre_shapehd_b200.fused.genre_forward_fused (SURVEY 8f-1 / 8f-4: the batched, mesh-free stand-in for
    forward_with_trimesh) returns the tensors of GenReNet.forward"""
    from genre_shapehd_b200.fused import genre_forward_fused
    dev = torch.device("cuda:0")
    net = _genre_net().to(dev).eval()
    x = genre_inputs(3, dev, seed=4)
    # The back-projections bin points into voxels: a 1e-7 change of a depth value can move a point across a voxel boundary.
    # cuDNN does not promise bitwise-identical results between two calls of the 2D nets, so both forwards are fed the SAME
    # 2D-net outputs (computed once, replayed): what is compared is the 3D path.
    dn = net.depth_and_inpaint
    cache = {}

    def replay(name, mod):
        orig = mod.forward

        def fwd(inp):
            if name not in cache:
                cache[name] = {k: v.clone() for k, v in orig(inp).items()}
            return {k: v.clone() for k, v in cache[name].items()}
        mod.forward = fwd
    replay("net1", dn.net1)
    replay("net2", dn.net2)
    with torch.no_grad():
        a = net(types.SimpleNamespace(rgb=x.rgb.clone(), silhou=x.silhou.clone()))
        b = genre_forward_fused(net, types.SimpleNamespace(rgb=x.rgb.clone(), silhou=x.silhou.clone()))
    for key in ("proj_depth", "pred_sph_partial", "pred_sph_full", "pred_proj_sph_full", "pred_proj_depth", "pred_voxel"):
        assert a[key].shape == b[key].shape, key
        scale = max(1.0, a[key].abs().max().item())
        assert (a[key] - b[key]).abs().max().item() <= 2e-4 * scale, key
    assert (a["pred_voxel"] - b["pred_voxel"]).abs().max().item() <= 1e-4 * max(1.0, a["pred_voxel"].abs().max().item())
