#!/usr/bin/env python
"""bench.py — BASELINE.json metric: "GenRe shapes/sec @128^3 voxel, 1/2/4/8 GPU; cam_bp HBM GB/s vs peak".

    python bench.py [--gpus N] [--steps K] [--warmup W]            this repo (one rank per GPU, torchrun for N > 1)
    python bench.py --impl reference [...]                         the reference's CPU path (rank 0 only)
    python bench.py --dump-outputs DIR [...]                       also write the last timed step's outputs as DIR/<name>.npy

Workload = BASELINE configs[2]: GenRe full_model inference, batch 16 per GPU, through
``genre_shapehd_b200.genre_models.GenReNet.forward`` (the published models/genre_full_model.py:116-132 Net.forward) on this
package's toolbox / networks: net1 (2D U-ResNet18 on cuDNN) -> cam_bp -> render_spherical -> sph_pad ->
net2 (2D inpainting U-ResNet18) -> spherical back-projection -> Unet_3D refiner.  Random-init weights (no checkpoints
offline; genre_shapehd_b200/synth_genre.py), synthetic rgb / silhouette inputs.  A "step" is one forward over a batch.

One JSON line on stdout (rank 0):
  value        whole-job shapes/s, inputs resident in HBM, device-timed, max over ranks
  e2e          the same through predict()+pack_output()'s data flow (netinterface.py:340-350, genre_full_model.py:188-200):
               pinned host rgb+silhou -> H2D -> Net.forward -> D2H of pred_voxel, every step, double-buffered over streams
  roofline     the metric's second clause, cam_bp: algorithmic bytes B*(4*H*W + 4*R^3) / whole-op time (project + splat)
               against the measured HBM peak; `clauses` adds the splat kernel alone, render_spherical, spherical
               back-projection (HBM) and the Unet_3D refiner (tensor pipe: useful FLOP/s against the measured dense peak)
  cpu_baseline the reference arm (below) on a bounded sample, run as a sub-process on rank 0 at N = 1
  secondary    BASELINE configs[1] (cam_bp batch 32) and the same GenRe step with single-pass fp16 conv operands
  secondary_ddp  BASELINE configs[3] and [4]: ShapeHD fine-tune step and WGAN-GP critic step (batch 8 per GPU), GenRe end-to-end
               fine-tune + Chamfer (batch 4 per GPU), genre_shapehd_b200.genre_models classes, DDP over NCCL for N > 1 with the exposed all-reduce time

--impl reference: the same GenReNet.forward on the host CPU: toolbox ops = the CPU oracle port (the reference's ops are
CUDA-only), networks on torch CPU, every host thread.
The oracle is only executed by that arm (and therefore by the cpu_baseline sub-process).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# the contract is ONE JSON line on stdout: keep NCCL's "NCCL version ..." banner (NCCL_DEBUG=VERSION) off it
if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

H = W = 256
RES = 128
FL, CAM_DIST = 418.3, 2.2
METRIC = "GenRe shapes/sec @128^3 voxel (full_model inference); cam_bp HBM GB/s vs peak"
UNIT = "shapes/s"
UNET3D_GFLOP = 78.0          # per shape, forward (SURVEY 8a a12 / Appendix A)
DUMP_BYTES = 60 << 20        # --dump-outputs: float32 payload of all arrays together (under 64 MB with the .npy headers)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=16, help="shapes per GPU per step (BASELINE configs[2]: 16)")
    ap.add_argument("--no-graph", action="store_true", help="launch steps from Python instead of replaying a CUDA graph")
    ap.add_argument("--cpu-seconds", type=float, default=25.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--cpu-budget", type=float, default=150.0, help="--impl reference: wall-clock budget of the whole run (s)")
    ap.add_argument("--skip", default=os.environ.get("GENRE_B200_BENCH_SKIP", ""),
                    help="comma list of legs to skip: e2e,roofline,cpu,secondary,ddp")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (rank 0) as DIR/<name>.npy, float32, %d MiB in all: an "
                         "output larger than its share of that as a fixed seeded sample" % (DUMP_BYTES >> 20))
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


def config(args, n_gpus, extra=None):
    c = {"workload": "GenRe full_model inference (depth + sph-inpaint + voxel refine), batch=%d per GPU (BASELINE configs[2]), "
                     "GenReNet.forward (models/genre_full_model.py Net) on this package's toolbox/networks" % args.batch,
         "batch_per_gpu": args.batch, "global_batch": args.batch * n_gpus, "rgb_hw": [H, W], "voxel_res": RES,
         "weights": "random init (PyTorch defaults; min/max-depth head biased to the dataset depth range so cam_bp hits the grid)",
         "parallelism": "replicas x%d (batch-sharded, no collective)" % n_gpus,
         "l2": "no explicit flush: one step streams > 1 GB of activations (Unet_3D enc1 output alone is 336 MB at batch 16) "
               "through the 126 MB L2; inputs rotate over 2 buffers"}
    if extra:
        c.update(extra)
    return c


# ----------------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for t, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                clk, mxc = float(f[1]), float(f[2])
            except ValueError:
                continue
            mx = mxc
            if t0 - 0.05 <= t <= t1 + 0.05:
                sm.append(clk)
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        if not sm:  # region shorter than the sampling period: fall back to every sample taken
            sm = [float(l.split(",")[1]) for _, l in self.rows if len(l.split(",")) > 2 and l.split(",")[1].strip().replace(".", "").isdigit()]
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------
# reference arm: GenReNet.forward on the host CPU (toolbox = oracle port, networks on torch CPU)
# ----------------------------------------------------------------------------------------------------
def _numa_node_cpus():
    """CPU sets of the host's NUMA nodes (within this process's affinity mask)"""
    allowed = os.sched_getaffinity(0)
    nodes = []
    try:
        base = "/sys/devices/system/node"
        for d in sorted(os.listdir(base)):
            if d.startswith("node") and d[4:].isdigit():
                cpus = set()
                for part in open(os.path.join(base, d, "cpulist")).read().strip().split(","):
                    if part:
                        a, _, b = part.partition("-")
                        cpus.update(range(int(a), int(b or a) + 1))
                cpus &= allowed
                if cpus:
                    nodes.append(cpus)
    except OSError:
        pass
    return nodes


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # idle OpenMP workers must sleep, not spin: torch's pool and the oracle's thread pool take turns on the same cores
    os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")
    os.environ.setdefault("KMP_BLOCKTIME", "0")
    os.environ.pop("OMP_NUM_THREADS", None)            # torchrun sets it to 1; this arm is the only process using the host
    import torch
    all_cpus = os.sched_getaffinity(0)
    from oracle.cpu_genre import build_cpu_genre_net
    from genre_shapehd_b200.synth_genre import genre_inputs
    t_build = time.time()
    net = build_cpu_genre_net()
    steps, warmup = args.steps, args.warmup

    def forward(x):
        with torch.no_grad():
            return net(x)["pred_voxel"]

    def use(cpus):
        os.sched_setaffinity(0, cpus)
        torch.set_num_threads(len(cpus))
        os.environ["GENRE_ORACLE_THREADS"] = str(len(cpus))

    # give the CPU arm its best footing: every host thread, or one NUMA node's threads (torch's CPU convolutions often run
    # faster inside one socket than across two) -- whichever a 2-shape probe finds faster
    probe = genre_inputs(2, seed=0)
    candidates = [("all %d host threads" % len(all_cpus), all_cpus)]
    nodes = _numa_node_cpus()
    if len(nodes) > 1:
        big = max(nodes, key=len)
        candidates.append(("the %d threads of one NUMA node (of %d nodes)" % (len(big), len(nodes)), big))
    best = None
    for name, cpus in candidates:
        use(cpus)
        import toolbox._pool as tp
        tp._pool = None                               # rebuild the oracle's pool at this width
        forward(probe)                                # page in, build thread pools
        t = time.time()
        forward(probe)
        dt = (time.time() - t) / 2
        if best is None or dt < best[0]:
            best = (dt, name, cpus)
    per_shape, thread_desc, cpus = best
    use(cpus)
    import toolbox._pool as tp
    tp._pool = None
    cores = len(cpus)
    # each step = a bounded sample of the batch, sized so that warmup + steps fit the budget
    budget = max(10.0, args.cpu_budget - (time.time() - t_build))
    sample = int(max(1, min(args.batch, budget / (per_shape * (steps + warmup)))))
    x = genre_inputs(sample, seed=0)
    for _ in range(warmup):
        forward(x)
    t0 = time.time()
    for _ in range(steps):
        out = forward(x)
    dt = time.time() - t0
    value = sample * steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config(args, args.gpus),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": "%d of the %d shapes of a batch per step; GenReNet.forward on CPU: toolbox ops = oracle/genre_oracle.c "
                                       "over a thread pool (the reference's ops are CUDA-only), 2D/3D networks on torch CPU; threads: %s (the faster of %d placements probed; host has %d logical CPUs)"
                                       % (sample, args.batch, thread_desc, len(candidates), os.cpu_count() or 0)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "result_checksum": float(out.double().abs().sum())}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------
# helpers of our arm
# ----------------------------------------------------------------------------------------------------
def measured_peaks():
    hbm, tens, src = 6650.0, 1500.0, "fallback (B200_PROFILING.md)"
    pk = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        try:
            d = json.load(open(pk))
            hbm, tens, src = float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return hbm, tens, src


def bind_to_gpu_numa_node(local):
    """Pin this rank's host threads (and therefore the first-touch placement of its pinned buffers) to the CPUs next to
    its GPU: with 8 ranks streaming results to the host, remote-socket pinned memory halves the D2H rate."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=20).stdout.strip()
        dom, rest = bus.split(":", 1)
        path = "/sys/bus/pci/devices/%s:%s/local_cpulist" % (dom[-4:].lower(), rest.lower())
        cpus = set()
        for part in open(path).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"pci": bus, "cpus": len(cpus)}
    except Exception as e:
        return {"error": repr(e)[:120]}
    return None


def time_cuda(torch, fn, reps, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def graph_of(torch, fn, warm=2):
    """CUDA graph of fn() (warm-up on a side stream first); returns (replay, result)"""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(warm):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = fn()
    return g.replay, out


# ----------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch

    import genre_shapehd_b200
    genre_shapehd_b200.install()
    from genre_shapehd_b200 import _lib, compat, dist_util, ops_conv
    from genre_shapehd_b200.genre_models import GenReNet
    from genre_shapehd_b200.synth_genre import genre_inputs, init_genre_net_for_bench

    skip = set(x for x in args.skip.split(",") if x)
    world, rank, local = dist_util.env_world()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this benchmark has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local)
    dist_util.init("nccl", dev)
    _lib.load()

    B, K, Wm = args.batch, args.steps, max(args.warmup, 3)
    torch.manual_seed(0)
    net = GenReNet()
    init_genre_net_for_bench(net)
    net = net.to(dev).eval()
    # the two 2D U-ResNet18 nets run on cuDNN (outside the hot path, SURVEY 8f-2); their one cheap win here is the
    # memory format of the module instances
    nets2d = os.environ.get("GENRE_B200_BENCH_2D_FORMAT", "channels_last")
    if nets2d == "channels_last":
        net.depth_and_inpaint.net1.to(memory_format=torch.channels_last)
        net.depth_and_inpaint.net2.to(memory_format=torch.channels_last)
    folded = 0
    if os.environ.get("GENRE_B200_BENCH_2D_FOLD_BN", "1") != "0":     # eval-mode BatchNorm2d folded into the preceding (transposed) conv
        folded = compat.fold_batchnorm2d_eval(net.depth_and_inpaint.net1) + compat.fold_batchnorm2d_eval(net.depth_and_inpaint.net2)
    nets2d += ", %d eval BatchNorm2d folded into their convolutions" % folded
    conv_mode = ops_conv.describe_mode()

    def barrier():
        dist_util.barrier(dev)

    def max_over_ranks(ms):
        return dist_util.max_over_ranks(ms, dev)

    # ---- leg 1: inputs resident in HBM --------------------------------------------------------------
    n_in = 2
    inputs = [genre_inputs(B, dev, seed=10 * rank + i) for i in range(n_in)]

    def forward(x):
        with torch.no_grad():
            return net(x)["pred_voxel"]

    def forward_all(x):
        with torch.no_grad():
            return net(x)

    # launches of THIS library per step (eager, counted by the binding); cuDNN / aten kernels of the 2D nets are not ours
    forward(inputs[0])
    torch.cuda.synchronize()
    n0 = _lib.launch_count
    forward(inputs[0])
    torch.cuda.synchronize()
    own_per_step = _lib.launch_count - n0

    use_graph = not args.no_graph and os.environ.get("GENRE_B200_BENCH_GRAPH", "1") != "0"
    replays, graph_note = [], None
    if use_graph:
        try:
            for x in inputs:
                replays.append(graph_of(torch, lambda x=x: forward_all(x)))
        except Exception as e:       # e.g. an op of the 2D nets that cannot be captured: launch from Python instead
            graph_note = "capture failed: " + repr(e)[:160]
            use_graph, replays = False, []
            torch.cuda.synchronize()

    def step(i):
        """one forward; returns the dict it computed (for a graph: the graph's output tensors, valid until its next replay)"""
        if use_graph:
            replay, out = replays[i % n_in]
            replay()
            return out
        return forward_all(inputs[i % n_in])

    for i in range(Wm):
        step(i)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    prof_range = os.environ.get("GENRE_B200_BENCH_PROFILE_RANGE") == "1"    # `ncu --profile-from-start off`: the timed steps only
    if prof_range:
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
    t_wall0 = time.time()
    e0.record()
    for i in range(K):
        last = step(i)
    e1.record()
    barrier()
    t_wall1 = time.time()
    if prof_range:
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    t_load1 = t_wall1
    try:    # keep the same step running (untimed) so that nvidia-smi's 100 ms samples describe this kernel mix under load
        n_load = min(2000, max(K, int(0.6 / max(ms_total / K * 1e-3, 1e-6))))
        for i in range(n_load):
            step(i)
        torch.cuda.synchronize()
        t_load1 = time.time()
    except Exception:
        pass
    clocks = sampler.stop(t_wall0, t_load1) if rank == 0 else None
    if clocks is not None:
        clocks["window"] = "timed region + %.2f s untimed replay of the same step" % (t_load1 - t_wall1)
    value = world * B * K / (ms_total * 1e-3)

    # ---- leg 2: end to end with host buffers, double-buffered over three streams ----------------------
    e2e = None
    if "e2e" not in skip:
        e2e = e2e_leg(torch, net, dev, B, K, rank, world, barrier, max_over_ranks, use_graph, genre_inputs)
        if e2e is not None and numa is not None:
            e2e["host_affinity"] = numa

    # ---- leg 3: rooflines of the hot-path ops at this batch (rank 0) -----------------------------------
    roofline = None
    if rank == 0 and "roofline" not in skip:
        try:
            roofline = roofline_leg(torch, net, dev, B, inputs[0])
        except Exception as e:
            roofline = {"error": repr(e)[:300]}

    # ---- leg 4: CPU baseline (rank 0, N = 1): the reference arm on a bounded sample, own process --------
    cpu = None
    if rank == 0 and world == 1 and "cpu" not in skip:
        cpu = cpu_baseline_leg(args)

    # ---- secondary: configs[1] and the fast conv mode (rank 0, N = 1) ----------------------------------
    secondary = None
    if rank == 0 and world == 1 and "secondary" not in skip:
        try:
            secondary = secondary_leg(torch, net, dev, B, forward, inputs)
        except Exception as e:
            secondary = {"error": repr(e)[:300]}

    # ---- secondary_ddp: configs[3] training steps under DDP (every N) ----------------------------------
    ddp = None
    if "ddp" not in skip:
        try:
            sys.path.insert(0, os.path.join(REPO, "profiles"))
            import bench_train_ddp
            ddp = {}
            for which in ("shapehd", "wgan", "genre"):      # one at a time: a failing workload must not hide the others
                try:
                    ddp.update(bench_train_ddp.run(dev, world, rank, local, batch=8, steps=6, warmup=3, which=(which,)))
                except Exception as e:
                    ddp[which + "_error"] = repr(e)[:300]
                torch.cuda.empty_cache()
        except Exception as e:
            ddp = {"error": repr(e)[:300]}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
                "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": config(args, world, {"conv_mode": conv_mode, "nets2d": "U-ResNet18 modules on cuDNN (TF32 allowed, PyTorch default), %s" % nets2d}),
                "e2e": e2e, "gpu_launches": own_per_step * K,
                "launch_mode": "cuda_graph" if use_graph else "python" + ("; " + graph_note if graph_note else ""),
                "own_kernel_launches_per_step": own_per_step,
                "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks, "secondary": secondary, "secondary_ddp": ddp}
        print(json.dumps(line), flush=True)
    dist_util.finalize()


def dump_outputs(out_dir, out):
    """out: the dict of one GenReNet.forward.  Each tensor gets an equal share of DUMP_BYTES and is written as <name>.npy in
    float32: whole when it fits its share, else the elements at that many sorted flat indices drawn from a generator
    seeded with 0 (the same indices for the same shape in every run)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    cap = DUMP_BYTES // (4 * len(out))
    for name, t in sorted(out.items()):
        a = t.detach().float().reshape(-1).cpu().numpy()
        if a.size > cap:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a if a.size != t.numel() else a.reshape(tuple(t.shape)))


def e2e_leg(torch, net, dev, B, K, rank, world, barrier, max_over_ranks, use_graph, genre_inputs):
    """pinned rgb+silhou -> H2D -> Net.forward -> D2H(pred_voxel), every step; two slots so that step i's result copy and step
    i+1's input copy overlap compute.  Mirrors NetInterface.predict + Model.pack_output of the reference."""
    import types
    Ke = max(4, min(K, 20))
    s_in, s_cmp, s_out = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
    slots = []
    for s in range(2):
        host = genre_inputs(B, None, seed=100 + 10 * rank + s, pin=True)
        d_in = types.SimpleNamespace(rgb=torch.empty((B, 3, H, W), device=dev), silhou=torch.empty((B, 1, H, W), device=dev))
        slots.append({"host": host, "dev": d_in, "pin_out": torch.empty((B, 1, RES, RES, RES), dtype=torch.float32).pin_memory(),
                      "in_done": torch.cuda.Event(), "cmp_done": torch.cuda.Event(), "out_done": torch.cuda.Event(), "run": None,
                      "out": None})

    def fwd(slot):
        with torch.no_grad():
            return net(slot["dev"])["pred_voxel"]

    torch.cuda.synchronize()
    for slot in slots:
        slot["dev"].rgb.copy_(slot["host"].rgb)
        slot["dev"].silhou.copy_(slot["host"].silhou)
        if use_graph:
            try:
                replay, out = graph_of(torch, lambda slot=slot: fwd(slot))
                slot["run"], slot["out"] = replay, out
            except Exception:
                use_graph = False
                torch.cuda.synchronize()
    for slot in slots:       # first use: nothing to wait for
        slot["out_done"].record(torch.cuda.current_stream())
        slot["cmp_done"].record(torch.cuda.current_stream())
    torch.cuda.synchronize()

    def e2e_step(i):
        slot = slots[i % 2]
        with torch.cuda.stream(s_in):
            s_in.wait_event(slot["cmp_done"])                 # the previous forward of this slot has consumed its inputs
            slot["dev"].rgb.copy_(slot["host"].rgb, non_blocking=True)
            slot["dev"].silhou.copy_(slot["host"].silhou, non_blocking=True)
            slot["in_done"].record(s_in)
        with torch.cuda.stream(s_cmp):
            s_cmp.wait_event(slot["in_done"])
            s_cmp.wait_event(slot["out_done"])                # the previous result of this slot has left the device
            if slot["run"] is not None:
                slot["run"]()
                out = slot["out"]
            else:
                out = fwd(slot)
                out.record_stream(s_out)
            slot["cmp_done"].record(s_cmp)
        with torch.cuda.stream(s_out):
            s_out.wait_event(slot["cmp_done"])
            slot["pin_out"].copy_(out, non_blocking=True)
            slot["out_done"].record(s_out)

    for i in range(4):
        e2e_step(i)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cur = torch.cuda.current_stream()
    e0.record(cur)
    for st in (s_in, s_cmp, s_out):
        st.wait_event(e0)
    for i in range(Ke):
        e2e_step(i)
    for st in (s_in, s_cmp, s_out):
        cur.wait_stream(st)
    e1.record(cur)
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    bytes_in, bytes_out = B * 4 * H * W * 4, B * RES ** 3 * 4
    return {"value": world * B * Ke / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": bytes_in, "d2h_bytes_per_step": bytes_out,
            "steps": Ke, "ms_per_step": ms / Ke, "result_checksum": float(slots[0]["pin_out"].double().abs().sum()),
            "d2h_GBps_per_rank_if_serial": bytes_out / (ms / Ke * 1e-3) / 1e9,
            "pipeline": "2 slots x 3 streams (H2D | Net.forward%s | D2H)" % (" as a CUDA graph" if slots[0]["run"] is not None else "")}


def roofline_leg(torch, net, dev, B, x):
    """Each hot-path op of the step, alone, at the step's batch and ON THE STEP'S OWN TENSORS (one real forward is run first and
    its intermediates captured): CUDA events around a CUDA-graph replay of the public call (so that launch gaps are not billed
    to the kernels), algorithmic bytes / flops from SURVEY 8(d)."""
    from genre_shapehd_b200 import _lib, ops_conv
    from toolbox.cam_bp.cam_bp.functions import SphericalBackProjection
    from toolbox.spherical_proj import gen_sph_grid
    hbm, tens, src = measured_peaks()
    layer = net.proj_depth
    cap = {}
    h1 = net.depth_and_inpaint.proj_depth.register_forward_pre_hook(lambda m, a: cap.__setitem__("depth", a[0].detach().clone()))
    h2 = net.depth_and_inpaint.render_spherical.register_forward_pre_hook(lambda m, a: cap.__setitem__("vox", a[0].detach().clone()))
    h3 = net.refine_net.register_forward_pre_hook(lambda m, a: cap.__setitem__("refine_in", a[0].detach().clone()))
    with torch.no_grad():
        out = net(x)
    for h in (h1, h2, h3):
        h.remove()
    depth, vox, refine_in = cap["depth"], cap["vox"], cap["refine_in"]     # depth: the permuted + flipped view the caller passes
    reps = 30
    with torch.no_grad():
        # cam_bp whole op (memset node + project + splat)
        run, proj = graph_of(torch, lambda: layer(depth))
        ms_cam = time_cuda(torch, run, reps)
        cam_bytes = B * (4 * H * W + 4 * RES ** 3)
        # splat kernel alone (the HBM-bound kernel of the op)
        ws, nbytes = _lib.workspace_for(B, H * W, RES, dev)
        tdf = torch.empty((B, 1, RES, RES, RES), device=dev)
        st = _lib.stream_ptr(depth)
        fl = torch.full((1, 1), FL, device=dev).expand(B, 1)
        cd = torch.full((1, 1), CAM_DIST, device=dev).expand(B, 1)
        _lib.call("genre_b200_cam_bp_stage_project", depth.data_ptr(), B, 1, H, W, *depth.stride(), fl.data_ptr(), *fl.stride(),
                  cd.data_ptr(), *cd.stride(), RES, ws.data_ptr(), nbytes, st)
        ms_splat = time_cuda(torch, lambda: _lib.call("genre_b200_voxelize_stage_splat", B, H * W, RES, tdf.data_ptr(), None, 1.0,
                                                      -1.0 / 16777216.0, 0.0, ws.data_ptr(), nbytes, st), reps)
        # render_spherical on the volume the caller hands it: clamp(proj * 50, 1e-5, 1 - 1e-5) (depth_pred_with_sph_inpaint.py:124)
        rend = net.depth_and_inpaint.render_spherical
        run, sph = graph_of(torch, lambda: rend(vox))
        ms_rend = time_cuda(torch, run, reps)
        rend_bytes = B * (4 * RES ** 3 + 4 * 128 * 128)
        # spherical back-projection (tdf + cnt out) of the inpainted map (genre_full_model.py:134-143)
        grid = gen_sph_grid().to(dev).expand(B, -1, -1, -1, -1)
        sph_in = (1 - out["pred_sph_full"][:, :, 16:144, 16:144]).contiguous()
        run, _ = graph_of(torch, lambda: SphericalBackProjection.apply(sph_in, grid, RES))
        ms_sbp = time_cuda(torch, run, reps)
        sbp_bytes = B * (4 * 128 * 128 + 8 * RES ** 3)
        # the refiner on its real input
        run, _ = graph_of(torch, lambda: net.refine_net(refine_in))
        ms_unet = time_cuda(torch, run, 10)
    tf_useful = UNET3D_GFLOP * 1e9 * B / (ms_unet * 1e-3) / 1e12
    ncu = None
    f = os.path.join(REPO, "profiles", "r02_tensor_pipe.json")
    if os.path.exists(f):
        try:
            ncu = json.load(open(f))
        except Exception:
            pass
    traffic = None
    f = os.path.join(REPO, "profiles", "splat_traffic.json")
    if os.path.exists(f):
        try:
            traffic = json.load(open(f))
        except Exception:
            pass
    gbs = lambda nbytes, ms: nbytes / (ms * 1e-3) / 1e9
    occ_frac = float((vox > 1e-5).float().mean())
    return {"bound": "hbm", "kernel": "cam_bp whole op: cam_project_kernel + vox_splat_kernel (+ counter memset), batch %d, the step's own depth maps" % B,
            "achieved": gbs(cam_bytes, ms_cam), "peak": hbm, "unit": "GB/s", "frac": gbs(cam_bytes, ms_cam) / hbm,
            "traffic": (traffic or {}).get("dram_bytes_per_launch_b16"), "traffic_source": "ncu --set full capture, profiles/splat_traffic.json (static: needs a profiler)",
            "peak_source": src, "algorithmic_bytes_per_launch": cam_bytes, "op_us": ms_cam * 1e3,
            "clauses": {
                "vox_splat_kernel": {"bound": "hbm", "us": ms_splat * 1e3, "achieved": gbs(cam_bytes, ms_splat), "frac": gbs(cam_bytes, ms_splat) / hbm,
                                     "algorithmic_bytes": cam_bytes},
                "render_spherical": {"bound": "hbm", "us": ms_rend * 1e3, "achieved": gbs(rend_bytes, ms_rend), "frac": gbs(rend_bytes, ms_rend) / hbm,
                                     "algorithmic_bytes": rend_bytes, "kernels": "render_occupancy128_kernel + render_spherical_forward_skip_kernel",
                                     "occupied_voxel_fraction_of_the_input": occ_frac},
                "spherical_back_projection": {"bound": "hbm", "us": ms_sbp * 1e3, "achieved": gbs(sbp_bytes, ms_sbp), "frac": gbs(sbp_bytes, ms_sbp) / hbm,
                                              "algorithmic_bytes": sbp_bytes},
                "unet3d_refiner": {"bound": "tensor", "ms": ms_unet, "achieved": tf_useful, "peak": tens, "unit": "TFLOP/s (useful: 78.0 GFLOP/shape)",
                                   "frac": tf_useful / tens, "conv_mode": ops_conv.describe_mode(),
                                   "note": "useful flops of the reference layers; the hi/lo-split mode issues 2 MMAs per useful one and merged-parity "
                                           "layers carry structural zeros, so this understates tensor-pipe activity",
                                   "ncu_tensor_pipe": ncu}}}


def cpu_baseline_leg(args):
    cmd = [sys.executable, os.path.join(REPO, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
           "--batch", str(args.batch), "--cpu-budget", str(args.cpu_seconds)]
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        env.pop(k, None)
    try:
        p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600, env=env, cwd=REPO)
        line = [l for l in p.stdout.splitlines() if l.startswith("{")][-1]
        d = json.loads(line)
        cb = d["cpu_baseline"]
        cb["ms_per_step"] = d["ms_per_step"]
        cb["host_cpus"] = os.cpu_count()
        return cb
    except Exception as e:
        return {"error": repr(e)[:300]}


def secondary_leg(torch, net, dev, B, forward, inputs):
    from genre_shapehd_b200 import ops_conv
    from genre_shapehd_b200.synth import bench_depth_batch
    hbm, _, _ = measured_peaks()
    out = {}
    with torch.no_grad():
        # BASELINE configs[1]: cam_bp 256x256 -> 128^3, batch 32
        depth = torch.from_numpy(bench_depth_batch(32)).to(dev)
        run, _ = graph_of(torch, lambda: net.proj_depth(depth))
        ms = time_cuda(torch, run, 50)
        nbytes = 32 * (4 * H * W + 4 * RES ** 3)
        out["cam_bp_b32"] = {"workload": "BASELINE configs[1]: cam_bp 256x256 depth -> 128^3, batch 32", "us": ms * 1e3,
                             "shapes_per_s": 32 / ms * 1e3, "whole_op_GBps": nbytes / (ms * 1e-3) / 1e9,
                             "whole_op_frac": nbytes / (ms * 1e-3) / 1e9 / hbm}
        # the same GenRe step with single-pass fp16 operands in the 3D convolutions (10-bit mantissa, tested at 4e-3 per layer)
        with ops_conv.precision("f16"):
            ms_fast = time_cuda(torch, lambda: forward(inputs[0]), 5)
        out["genre_fast_conv_mode"] = {"conv_mode": "f16 single pass (10-bit operand mantissa; NOT the 1e-4 parity mode)",
                                       "ms_per_step_python_launch": ms_fast, "shapes_per_s": B / ms_fast * 1e3}
        ms_exact = time_cuda(torch, lambda: forward(inputs[0]), 5)
        out["genre_default_mode_python_launch"] = {"conv_mode": ops_conv.describe_mode(), "ms_per_step": ms_exact,
                                                   "shapes_per_s": B / ms_exact * 1e3}
        # the 3D hot path alone (2D nets excluded), fused glue (genre_shapehd_b200/fused.py)
        from genre_shapehd_b200.fused import GenRe3DGlue
        glue = GenRe3DGlue().to(dev)
        d16 = depth[:B]
        sph_full = torch.rand(B, 1, 160, 160, device=dev) * 0.4 + 0.3

        def path3d():
            pd, sph = glue.project_and_render(d16)
            return net.refine_net(glue.refine_input(pd, sph_full))
        ms3 = time_cuda(torch, path3d, 5)
        out["genre_3d_path_fused_glue"] = {"ms_per_batch": ms3, "shapes_per_s": B / ms3 * 1e3, "conv_mode": ops_conv.describe_mode()}
    return out


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
