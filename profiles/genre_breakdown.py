#!/usr/bin/env python
"""Where the GenRe full-model forward (BASELINE configs[2], batch 16, GenReNet.forward) spends its time:
CUDA events around the sub-modules (forward hooks, eager launches), and the effect of the 2D nets' "cheap wins"
(channels_last; bf16 autocast) on the whole step.  One JSON line."""
import json, os, sys
import torch
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
import genre_shapehd_b200
genre_shapehd_b200.install()
from genre_shapehd_b200 import ops_conv
from genre_shapehd_b200.genre_models import GenReNet
from genre_shapehd_b200.synth_genre import genre_inputs, init_genre_net_for_bench
dev = torch.device("cuda:0"); torch.cuda.set_device(dev)
B = int(os.environ.get("B", 16))
torch.manual_seed(0)
net = GenReNet(); init_genre_net_for_bench(net); net = net.to(dev).eval()
x = genre_inputs(B, dev, seed=0)

def timeit(fn, reps=10, warm=3):
    for _ in range(warm): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps

def fwd():
    with torch.no_grad():
        return net(x)["pred_voxel"]

out = {"B": B, "conv_mode": ops_conv.describe_mode(), "step_ms_eager": timeit(fwd)}
# per-module times (hooks add sync points only through events: negligible)
mods = {"net1 (2D U-ResNet18, 3 decoders + minmax)": net.depth_and_inpaint.net1, "cam_bp": net.depth_and_inpaint.proj_depth,
        "render_spherical": net.depth_and_inpaint.render_spherical, "net2 (2D inpaint U-ResNet18)": net.depth_and_inpaint.net2,
        "Unet_3D refiner": net.refine_net}
ev = {k: [] for k in mods}
hooks = []
for k, m in mods.items():
    def pre(mod, a, k=k):
        e = torch.cuda.Event(enable_timing=True); e.record(); ev[k].append([e, None])
    def post(mod, a, o, k=k):
        e = torch.cuda.Event(enable_timing=True); e.record(); ev[k][-1][1] = e
    hooks += [m.register_forward_pre_hook(pre), m.register_forward_hook(post)]
for _ in range(3): fwd()
for k in ev: ev[k].clear()
reps = 10
for _ in range(reps): fwd()
torch.cuda.synchronize()
per = {k: sum(a.elapsed_time(b) for a, b in v) / reps for k, v in ev.items()}
for h in hooks: h.remove()
per["everything else (glue of the frozen callers: elementwise torch ops, sph_pad, spherical back-projection, cat)"] = out["step_ms_eager"] - sum(per.values())
out["per_module_ms"] = per
# cheap wins on the 2D nets (out of the hot-path scope, SURVEY 8f-2): memory format and autocast, whole-step effect
n1, n2 = net.depth_and_inpaint.net1, net.depth_and_inpaint.net2
n1.to(memory_format=torch.channels_last); n2.to(memory_format=torch.channels_last)
out["step_ms_eager_2d_channels_last"] = timeit(fwd)
ref = fwd().clone()
def fwd_bf16():
    # autocast only around the 2D nets: hooks that cast their outputs back would need caller changes, so this is whole-forward
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        return net(x)["pred_voxel"]
try:
    out["step_ms_eager_autocast_bf16_whole_forward"] = timeit(fwd_bf16)
    out["autocast_max_abs_diff_logits"] = float((fwd_bf16().float() - ref).abs().max())
except Exception as e:
    out["autocast_error"] = repr(e)[:200]
print(json.dumps(out))
