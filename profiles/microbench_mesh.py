#!/usr/bin/env python
"""Batched marching cubes (postprocess.iso_surface) at B = 16, 128^3, level 0.25, on two inputs:
  genre  : sigmoid(pred_voxel) of a seeded GenReNet.forward (the visualiser's pred_voxel meshes); the seeded, untrained
           refiner may stay below 0.25 everywhere (an empty mesh: pack + count + scan only), so it is also meshed at the
           median of its values (a dense, noisy surface),
  shells : hollow balls (iso_field("shell")) of 16 sizes, a surface-heavy volume.
Prints one JSON line:
  device_us  count + scan + emit (the 4 kernels, bases precomputed), CUDA events, mean of `reps` back-to-back calls; the
             16 x 8 MiB volumes (128 MiB) about fill the 126 MB L2, so successive calls partly hit L2;
  wall_us    the whole postprocess.iso_surface call (allocation + the one host sync + slicing), host clock;
  bytes      compulsory HBM traffic from shapes and mesh sizes: volume read, bit plane written and read back, row counts
             and bases written and read, mesh written;  hbm_frac = bytes / device time / 7.7 TB/s;
  tris_per_s triangles / device time;
  oracle_ms_per_volume  the single-threaded C checker (oracle_mesh/mc_oracle.c) on the host, per volume, for context: it is
             NOT skimage, which is not available here.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import genre_shapehd_b200  # noqa: E402
genre_shapehd_b200.install()
from genre_shapehd_b200 import _lib, postprocess  # noqa: E402
from genre_shapehd_b200.synth import iso_field  # noqa: E402
import oracle_mesh  # noqa: E402

HBM_BPS = 7.7e12
LEVEL = 0.25


def genre_volumes(B, dev):
    from genre_shapehd_b200.genre_models import GenReNet
    from genre_shapehd_b200.synth_genre import genre_inputs, init_genre_net_for_bench
    torch.manual_seed(0)
    net = init_genre_net_for_bench(GenReNet()).to(dev).eval()
    with torch.no_grad():
        v = torch.sigmoid(net(genre_inputs(B, dev, seed=0))["pred_voxel"][:, 0]).contiguous()
    del net
    torch.cuda.empty_cache()
    return v


def shell_volumes(B, dev, R=128):
    # field in voxels (> 0 inside the shell wall) -> an occupancy-like volume around the 0.25 level
    vols = [1 / (1 + np.exp(-(iso_field("shell", (R, R, R), scale=R * (0.7 + 0.3 * i / (B - 1)))[0] / 2) - np.log(3)))
            for i in range(B)]
    return torch.from_numpy(np.stack(vols).astype(np.float32)).to(dev)


def measure(v, reps, level=LEVEL):
    n, d, h, w = v.shape
    lib = _lib.load()
    st = _lib.stream_ptr(v)
    nbytes = lib.genre_b200_iso_surface_workspace_bytes(n, d, h, w)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=v.device)
    totals = torch.empty((n, 2), dtype=torch.int64, device=v.device)
    _lib.call("genre_b200_iso_surface_count", v.data_ptr(), n, d, h, w, level, ws.data_ptr(), nbytes, totals.data_ptr(), st)
    bases = torch.cumsum(totals, 0) - totals
    nv, nf = (int(x) for x in totals.sum(0).tolist())
    verts = torch.empty((max(nv, 1), 3), device=v.device)
    faces = torch.empty((max(nf, 1), 3), dtype=torch.int32, device=v.device)

    def run():
        _lib.call("genre_b200_iso_surface_count", v.data_ptr(), n, d, h, w, level, ws.data_ptr(), nbytes, totals.data_ptr(), st)
        _lib.call("genre_b200_iso_surface_emit", v.data_ptr(), n, d, h, w, level, 1 / 128, 1 / 128, 1 / 128, -0.5, -0.5, -0.5,
                  bases.data_ptr(), verts.data_ptr(), faces.data_ptr(), None, ws.data_ptr(), nbytes, st)
    for _ in range(3):
        run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        run()
    e1.record()
    torch.cuda.synchronize()
    dev_s = e0.elapsed_time(e1) / reps / 1e3

    for _ in range(2):
        postprocess.iso_surface(v, level, 1 / 128, -0.5)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        meshes = postprocess.iso_surface(v, level, 1 / 128, -0.5)
    torch.cuda.synchronize()
    wall_s = (time.perf_counter() - t0) / reps

    # one sample against the oracle, and the oracle's single-thread time
    x = v[0].cpu().numpy()
    t0 = time.perf_counter()
    ov, of = oracle_mesh.iso_surface(x, level, 1 / 128, -0.5)
    oracle_s = time.perf_counter() - t0
    exact = bool(np.array_equal(meshes[0][0].cpu().numpy(), ov) and np.array_equal(meshes[0][1].cpu().numpy(), of))

    rows = n * d * h
    plane = rows * ((w + 31) // 32) * 4
    nbytes_moved = n * d * h * w * 4 + 2 * plane + 2 * rows * 16 + nv * 12 + nf * 12
    return {"level": level, "B": n, "shape": [d, h, w], "verts": nv, "faces": nf, "device_us": dev_s * 1e6, "wall_us": wall_s * 1e6,
            "bytes": nbytes_moved, "hbm_frac": nbytes_moved / dev_s / HBM_BPS, "tris_per_s": nf / dev_s,
            "oracle_ms_per_volume": oracle_s * 1e3, "sample0_equals_oracle": exact}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("microbench_mesh.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True).stdout.strip()
    except OSError:
        smi = "nvidia-smi unavailable"
    res = {"bench": "microbench_mesh", "device": torch.cuda.get_device_name(dev), "nvidia_smi": smi, "level": LEVEL,
           "timing": "device_us: CUDA events over count+emit (4 kernels); wall_us: iso_surface incl. host sync"}
    g = genre_volumes(args.batch, dev)
    res["genre_pred_voxel"] = measure(g, args.reps)
    res["genre_pred_voxel_median_level"] = measure(g, args.reps, float(g.median()))
    del g
    res["shells"] = measure(shell_volumes(args.batch, dev), args.reps)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
