#!/usr/bin/env python
"""BASELINE configs[3] and [4] (ShapeHD fine-tune step and 3D-WGAN-GP critic step, batch 8 per GPU; GenRe end-to-end fine-tune
with the Chamfer op, batch 4 per GPU; DDP over NCCL) on the
networks drop-in, driven through genre_shapehd_b200.genre_models (the published model classes):
  shapehd step : models/shapehd.py Net (:82-118: two marrnet2 = ImageEncoder -> VoxelDecoder, frozen D) + the loss of
                 :67-79 (BCE-with-logits + w * -mean(D(sigmoid(voxel)))) + Adam on marrnet2 (:42-47)
  wgangp D step: models/wgangp.py:77-112,144-164 restated on its own D / G classes (:193-214): D(real), D(G(z)) and the
                 gradient penalty (double backward through D), accumulated under no_sync() so that the three backward()
                 calls cost ONE all-reduce (SURVEY.md 8e)
run() is imported by bench.py (the `secondary_ddp` block of every --gpus N line); stand-alone:
    torchrun --nproc-per-node N profiles/bench_train_ddp.py [--steps K]          # one JSON line from rank 0
Reports per step: ms (max over ranks), shapes/s, and the all-reduce time that backward does NOT hide = step time with
gradient sync minus the same step under no_sync() (no collective issued).
NCU=shapehd|wgan: run one warm step of that kind between cudaProfilerStart/Stop (for `ncu --profile-from-start off`).
"""
import argparse
import contextlib
import json
import os
import sys
import types

import torch
import torch.nn.functional as F

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)


def run(dev, world, rank, local, batch=8, steps=6, warmup=3, which=("shapehd", "wgan", "genre"), genre_batch=4):
    import genre_shapehd_b200
    genre_shapehd_b200.install()
    from genre_shapehd_b200 import dist_util, genre_models, ops_conv
    from torch.nn.parallel import DistributedDataParallel as DDP

    torch.manual_seed(1 + rank)
    B = batch
    res = {"n_gpus": world, "batch_per_gpu": B, "steps": steps, "conv_mode": ops_conv.describe_mode(),
           "bn_train_custom": ops_conv.BN_TRAIN, "tc_backward": ops_conv.TC_BACKWARD,
           "workload": "BASELINE configs[3]: ShapeHDNet (models/shapehd.py Net) + loss, and the models/wgangp.py critic step, DDP over NCCL"}

    def wrap(m):
        return DDP(m, device_ids=[local], gradient_as_bucket_view=True) if world > 1 else m

    def timed(fn):
        for _ in range(warmup):
            fn()
        dist_util.barrier(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        last = None
        for _ in range(steps):
            last = fn()
        e1.record()
        dist_util.barrier(dev)
        return dist_util.max_over_ranks(e0.elapsed_time(e1), dev) / steps, float(last)

    target = (torch.rand(B, 1, 128, 128, 128, device=dev) < 0.05).float()

    # ---- ShapeHD fine-tune step ---------------------------------------------------------------------------------------
    if "shapehd" in which:
        net = genre_models.ShapeHDNet().to(dev)
        net.train()
        ddp = wrap(net)
        opt = torch.optim.Adam(net.marrnet2.parameters(), lr=1e-3)
        depth, normal = torch.rand(B, 1, 256, 256, device=dev), torch.rand(B, 3, 256, 256, device=dev)
        silhou = (torch.rand(B, 1, 256, 256, device=dev) > 0.4).float()

        def shapehd_step(sync=True):
            opt.zero_grad(set_to_none=True)
            ctx = contextlib.nullcontext() if (sync or world == 1) else ddp.no_sync()
            with ctx:
                pred = ddp(types.SimpleNamespace(depth=depth.clone(), normal=normal.clone(), silhou=silhou))
                loss = F.binary_cross_entropy_with_logits(pred["voxel"], target) + 1e-3 * (-pred["is_real"].mean())
                loss.backward()
            opt.step()
            return loss.detach()
        if os.environ.get("NCU") == "shapehd":
            return _ncu(shapehd_step)
        ms, loss = timed(shapehd_step)
        res["shapehd"] = {"step_ms": ms, "shapes_per_s": world * B / ms * 1e3, "loss_finite": bool(loss == loss)}
        if world > 1:
            ms_ns, _ = timed(lambda: shapehd_step(sync=False))
            res["shapehd"].update({"step_ms_no_sync": ms_ns, "exposed_allreduce_ms": max(0.0, ms - ms_ns),
                                   "exposed_allreduce_frac": max(0.0, ms - ms_ns) / ms,
                                   "allreduce_bytes": 4 * sum(p.numel() for p in net.marrnet2.parameters())})
        del net, ddp, opt

    # ---- WGAN-GP critic step ---------------------------------------------------------------------------------------------
    if "wgan" in which:
        G = genre_models.WganGenerator(200).to(dev)
        Dn = genre_models.WganCritic().to(dev)
        for p in G.parameters():
            p.requires_grad = False
        ddp_d = wrap(Dn)
        opt_d = torch.optim.Adam(Dn.parameters(), lr=1e-4, betas=(0.5, 0.9))
        real = target
        lam, norm = 10.0, 1.0

        def wgan_d_step(sync=True):
            opt_d.zero_grad(set_to_none=True)
            nosync = ddp_d.no_sync if world > 1 else contextlib.nullcontext
            with nosync():
                ddp_d(real).mean().backward(torch.tensor(-1.0, device=dev))          # wgangp.py:94-95
                with torch.no_grad():
                    _, fake = G(B)
                ddp_d(fake).mean().backward(torch.tensor(1.0, device=dev))           # :100-103
            with (nosync() if not sync else contextlib.nullcontext()):
                alpha = torch.rand(B, 1, 1, 1, 1, device=dev)                         # :144-164
                inter = (alpha * real + (1 - alpha) * fake).requires_grad_(True)
                out = ddp_d(inter)
                grads, = torch.autograd.grad(outputs=out, inputs=inter, grad_outputs=torch.ones_like(out), create_graph=True,
                                             retain_graph=True, only_inputs=True)
                gp = (((grads.view(B, -1) + 1e-16).norm(2, dim=1) - norm) ** 2).mean() * lam
                gp.backward()
            opt_d.step()
            return gp.detach()
        if os.environ.get("NCU") == "wgan":
            return _ncu(wgan_d_step)
        ms, gp = timed(wgan_d_step)
        res["wgangp_critic"] = {"step_ms": ms, "shapes_per_s": world * B / ms * 1e3, "gp_finite": bool(gp == gp)}
        if world > 1:
            ms_ns, _ = timed(lambda: wgan_d_step(sync=False))
            res["wgangp_critic"].update({"step_ms_no_sync": ms_ns, "exposed_allreduce_ms": max(0.0, ms - ms_ns),
                                         "exposed_allreduce_frac": max(0.0, ms - ms_ns) / ms,
                                         "allreduce_bytes": 4 * sum(p.numel() for p in Dn.parameters())})
    # ---- GenRe end-to-end fine-tune step + Chamfer (BASELINE configs[4], batch 4 per GPU) ---------------------------------
    if "genre" in which:
        from genre_shapehd_b200.synth_genre import genre_inputs, init_genre_net_for_bench
        from nndistance.functions.nnd import nndistance
        Bg = genre_batch
        gnet = genre_models.GenReNet(joint_train=True)                # joint_train: gradients reach net1 / net2
        init_genre_net_for_bench(gnet)                                # through cam_bp / render_spherical / spherical bp backward
        gnet = gnet.to(dev).train()
        gddp = wrap(gnet)
        gopt = torch.optim.Adam(gnet.parameters(), lr=1e-4)
        gin = genre_inputs(Bg, dev, seed=5 + rank)
        gvox = (torch.rand(Bg, 1, 128, 128, 128, device=dev) < 0.05).float()
        npts = 4096
        gen = torch.Generator(dev).manual_seed(3 + rank)
        xyz2 = torch.rand(Bg, npts, 3, device=dev, generator=gen) - 0.5
        xyz1 = (torch.rand(Bg, npts, 3, device=dev, generator=gen) - 0.5).requires_grad_(True)

        def genre_step(sync=True):
            gopt.zero_grad(set_to_none=True)
            xyz1.grad = None
            ctx = contextlib.nullcontext() if (sync or world == 1) else gddp.no_sync()
            with ctx:
                pred = gddp(types.SimpleNamespace(rgb=gin.rgb, silhou=gin.silhou))
                voxel_loss = F.binary_cross_entropy_with_logits(pred["pred_voxel"], gvox)           # genre_full_model.py:64
                surface_loss = F.binary_cross_entropy(torch.sigmoid(pred["pred_voxel"]) * gvox, gvox)  # :65-66
                d1, d2 = nndistance(xyz1, xyz2)                        # the shipped-but-unwired Chamfer op, timed in the step (SURVEY 8d)
                # the reference's joint loss also supervises net1's normal / silhouette / min-max heads (marrnet1.py:120-136; the 3D path
                # reads depth_minmax detached, depth_pred_with_sph_inpaint.py:135): keep them in
                # the graph (weight 0) so that every parameter receives a gradient, as DDP's reducer expects
                loss = voxel_loss + surface_loss + (d1.mean() + d2.mean()) + 0.0 * (pred["normal"].mean() + pred["silhou"].mean() +
                                                                                    pred["depth_minmax"].mean())
                loss.backward()
            gopt.step()
            return loss.detach()
        if os.environ.get("NCU") == "genre":
            return _ncu(genre_step)
        ms, loss = timed(genre_step)
        res["genre_finetune"] = {"batch_per_gpu": Bg, "step_ms": ms, "shapes_per_s": world * Bg / ms * 1e3, "loss_finite": bool(loss == loss),
                                 "chamfer_points": npts,
                                 "workload": "BASELINE configs[4]: GenReNet, joint_train, voxel + surface loss, "
                                             "backward through every toolbox op, + nndistance fwd/bwd on [B,4096,3] clouds"}
        if world > 1:
            ms_ns, _ = timed(lambda: genre_step(sync=False))
            res["genre_finetune"].update({"step_ms_no_sync": ms_ns, "exposed_allreduce_ms": max(0.0, ms - ms_ns),
                                          "exposed_allreduce_frac": max(0.0, ms - ms_ns) / ms,
                                          "allreduce_bytes": 4 * sum(p.numel() for p in gnet.parameters() if p.requires_grad)})
    return res


def _ncu(fn):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    torch.cuda.profiler.start()
    fn()
    torch.cuda.synchronize()
    torch.cuda.profiler.stop()
    return None


def main():
    import genre_shapehd_b200
    genre_shapehd_b200.install()
    from genre_shapehd_b200 import dist_util
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--which", default="shapehd,wgan,genre")
    args = ap.parse_args()
    world, rank, local = dist_util.env_world()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist_util.init("nccl", dev)
    res = run(dev, world, rank, local, args.batch, args.steps, args.warmup, tuple(args.which.split(",")))
    if rank == 0 and res is not None:
        print(json.dumps(res), flush=True)
    dist_util.finalize()


if __name__ == "__main__":
    main()
