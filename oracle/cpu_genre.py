"""The reference's CPU path of the GenRe forward (BASELINE configs[2]) — BASELINE INFRASTRUCTURE, see cpu_toolbox/README.md.

build_cpu_genre_net() returns genre_shapehd_b200.genre_models.GenReNet (the published models/genre_full_model.Net) on CPU with
    toolbox.*            -> oracle/cpu_toolbox (the CUDA-only ops restated on the CPU oracle, maps in parallel)
    networks.*           -> the 2D U-ResNets and networks/networks.py on torch CPU
Must run in a process that never called genre_shapehd_b200.install() (bench.py --impl reference is such a process).

    python oracle/cpu_genre.py        # one JSON line: forward_signatures() of that net
"""
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)


def build_cpu_genre_net():
    import torch
    for name in ("toolbox", "networks", "nndistance"):
        if name in sys.modules:
            raise RuntimeError("%s is already imported (from %s): the CPU reference path needs its own process"
                               % (name, getattr(sys.modules[name], "__file__", "?")))
    if REPO not in sys.path:
        sys.path.insert(0, REPO)
    sys.path.insert(0, os.path.join(REPO, "genre_shapehd_b200"))     # networks
    sys.path.insert(0, os.path.join(HERE, "cpu_toolbox"))           # toolbox -> CPU oracle stand-ins
    from genre_shapehd_b200.genre_models import GenReNet
    from genre_shapehd_b200.synth_genre import init_genre_net_for_bench
    import toolbox
    assert os.path.abspath(toolbox.__file__).startswith(os.path.join(HERE, "cpu_toolbox"))
    torch.manual_seed(0)
    net = GenReNet()
    init_genre_net_for_bench(net)
    return net.eval()


FORWARD_BATCH, FORWARD_SEED, FORWARD_THREADS = 1, 0, 4


def forward_signatures(net, n=64):
    """eval forward of a GenRe net on genre_inputs(FORWARD_BATCH, seed=FORWARD_SEED), FORWARD_THREADS torch threads:
    for every output, its shape, float64 sum and |sum| and n values at evenly spaced flat indices"""
    import torch
    from genre_shapehd_b200.synth_genre import genre_inputs
    torch.set_num_threads(FORWARD_THREADS)
    with torch.no_grad():
        out = net(genre_inputs(FORWARD_BATCH, seed=FORWARD_SEED))
    sig = {}
    for k, t in out.items():
        flat = t.detach().reshape(-1).double()
        idx = torch.linspace(0, flat.numel() - 1, n).long()
        sig[k] = {"shape": list(t.shape), "sum": float(flat.sum()), "abs_sum": float(flat.abs().sum()),
                  "samples": [float(v) for v in flat[idx]]}
    return sig


if __name__ == "__main__":
    import json
    sys.path[:] = [p for p in sys.path if os.path.abspath(p or ".") != HERE]     # `oracle` is the package, not oracle.py
    print(json.dumps(forward_signatures(build_cpu_genre_net())))
