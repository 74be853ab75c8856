#!/usr/bin/env python
"""Golden digests of the published GenRe-ShapeHD model classes (models/genre_full_model.py Net, models/shapehd.py Net,
models/wgangp.py D), recorded from a checkout of the original project on torch CPU fp32.  Each model is built under a
fixed seed; the sha256 of its state_dict layout (keys and shapes) and of its parameter bytes are recorded, and for
GenRe also sampled signatures of the two 2D U-ResNet-18s' outputs on seeded inputs and of every output of the whole
Net.forward on the CPU (toolbox ops through oracle/cpu_toolbox, as oracle/cpu_genre.py runs GenReNet; own process).
tests/test_dropin_reference_models.py rebuilds the models from
genre_shapehd_b200/genre_models.py under the same seeds and must reproduce all of it.

    python tests/golden/make_golden_models.py /path/to/GenRe-ShapeHD      # writes tests/golden/models_digest.json
"""
import hashlib
import json
import os
import subprocess
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)
from genre_shapehd_b200 import compat  # noqa: E402
from genre_shapehd_b200.synth_genre import genre_opt, init_genre_net_for_bench  # noqa: E402


def signature(t, n=64):
    flat = t.detach().reshape(-1).double()
    idx = torch.linspace(0, flat.numel() - 1, n).long()
    return {"shape": list(t.shape), "sum": float(flat.sum()), "abs_sum": float(flat.abs().sum()),
            "samples": [float(v) for v in flat[idx]]}


def layout(net):
    sd = net.state_dict()
    h = hashlib.sha256()
    for k, v in sd.items():
        h.update(k.encode())
        h.update(np.ascontiguousarray(v.numpy()).tobytes())
    keys = json.dumps([[k, list(v.shape)] for k, v in sd.items()])
    return {"n_keys": len(sd), "state_dict_sha256": hashlib.sha256(keys.encode()).hexdigest(), "params_sha256": h.hexdigest()}


def original_forward_on_cpu(ref):
    """the original Net.forward on the CPU, networks from the checkout, toolbox ops from oracle/cpu_toolbox"""
    sys.path.insert(0, ref)
    sys.path.insert(0, os.path.join(REPO, "oracle", "cpu_toolbox"))
    compat.stub_optional_modules()
    import models.genre_full_model as gfm
    from oracle.cpu_genre import forward_signatures
    torch.manual_seed(0)
    net = gfm.Net(genre_opt(), gfm.Model)
    init_genre_net_for_bench(net)
    print(json.dumps(forward_signatures(net.eval())))


def main(ref):
    compat.bootstrap(ref)
    import models.genre_full_model as gfm
    import models.shapehd as shd
    import models.wgangp as wg

    out = {"torch": torch.__version__, "source": "GenRe-ShapeHD models/*.py on torch CPU fp32", "cases": {}}
    torch.manual_seed(0)
    net = gfm.Net(genre_opt(), gfm.Model)
    init_genre_net_for_bench(net)
    case = {"seed": 0, "bench_init": True, **layout(net)}
    net.eval()
    torch.manual_seed(7)
    rgb, sph = torch.randn(1, 3, 256, 256), torch.rand(1, 1, 160, 160)
    with torch.no_grad():
        o1 = net.depth_and_inpaint.net1(types.SimpleNamespace(rgb=rgb))
        o2 = net.depth_and_inpaint.net2(sph)
    case["inputs_seed"] = 7
    case["net1"] = {k: signature(v) for k, v in o1.items()}
    case["net2"] = {k: signature(v) for k, v in o2.items()}
    p = subprocess.run([sys.executable, os.path.abspath(__file__), ref, "--original-forward-on-cpu"], stdout=subprocess.PIPE,
                       check=True, text=True)
    case["forward_cpu"] = json.loads(p.stdout.strip().splitlines()[-1])
    out["cases"]["GenReNet"] = case
    torch.manual_seed(1)
    out["cases"]["ShapeHDNet"] = {"seed": 1, **layout(shd.Net())}
    torch.manual_seed(2)
    out["cases"]["WganCritic"] = {"seed": 2, **layout(wg.D())}
    json.dump(out, open(os.path.join(HERE, "models_digest.json"), "w"), indent=1)


if __name__ == "__main__":
    if sys.argv[2:] == ["--original-forward-on-cpu"]:
        original_forward_on_cpu(sys.argv[1])
    else:
        main(sys.argv[1])
