"""Times ONE optimizer step over the parameters of the NTU model (274 tensors, 13.9 MB), fused against torch.optim (run on the GPU
box):  python tools/bench_optim.py [--steps K] [--warmup W] [--rounds R] [--out FILE]

Configurations: FusedAdam(amsgrad=True) vs torch.optim.Adam(amsgrad=True), FusedASGD vs torch.optim.ASGD (both with torch's
defaults otherwise, as the reference's YAML would build them), and the plain FusedAdam vs torch.optim.Adam as the control.  Every
optimizer steps its own copy of the parameters, with gradients drawn once from a fixed seed.  Each round times K steps of each
configuration with CUDA events after W warm-up steps; the rounds alternate fused and torch, and the median / min / max over the
rounds is printed.  Parameters, gradients and optimizer state (at most 5 x 13.9 MB) stay resident in the 126 MB L2 between steps.
The GPU name, its power limit and its maximum SM clock are read in the same run and printed with the numbers.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from fusion_gcn_b200 import capi, graph as G, modules as M, optim  # noqa: E402

CONFIGS = [   # name: (fused class, torch class, keyword arguments for both)
    ("adam_amsgrad", optim.FusedAdam, torch.optim.Adam, dict(lr=1e-3, amsgrad=True)),
    ("asgd", optim.FusedASGD, torch.optim.ASGD, dict(lr=1e-2)),
    ("adam_control", optim.FusedAdam, torch.optim.Adam, dict(lr=1e-3)),
]


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info.update(power_limit_w=float(out[0]), sm_max_mhz=float(out[1]))
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        info.update(power_limit_w=None, sm_max_mhz=None)
    return info


def ntu_parameters():
    torch.manual_seed(1)
    model = M.Model((2, 300, 25, 3), 60, G.SkeletonGraph(G.NTU_EDGES, center_joint=G.NTU_CENTER))
    return [p.detach().cuda() for p in model.parameters()]


def make_step(cls, base, grads, kw):
    params = [torch.nn.Parameter(p.clone()) for p in base]
    for p, g in zip(params, grads):
        p.grad = g.clone()
    return cls(params, **kw).step


def time_steps(step, k):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(k):
        step()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / k


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_optim.py needs a CUDA device")
    base = ntu_parameters()
    gen = torch.Generator(device="cuda").manual_seed(0)
    grads = [torch.randn(p.shape, generator=gen, device="cuda") * 1e-2 for p in base]
    nbytes = sum(p.numel() for p in base) * 4
    lines = [json.dumps(dict(gpu_info(), tensors=len(base), param_mb=round(nbytes / 1e6, 2), steps=args.steps, warmup=args.warmup,
                             rounds=args.rounds))]
    print(lines[-1], flush=True)
    for name, fused_cls, torch_cls, kw in CONFIGS:
        steps = {"fused": make_step(fused_cls, base, grads, kw), "torch": make_step(torch_cls, base, grads, kw)}
        for s in steps.values():
            for _ in range(args.warmup):
                s()
        before = capi.lib().agcn_launch_count()
        steps["fused"]()
        launches = capi.lib().agcn_launch_count() - before
        ms = {k: [] for k in steps}
        for _ in range(args.rounds):
            for k, s in steps.items():
                ms[k].append(time_steps(s, args.steps))
        rec = {"config": name, "kwargs": kw, "fused_launches_per_step": launches}
        for k, v in ms.items():
            rec[f"{k}_ms"] = {"median": round(statistics.median(v), 4), "min": round(min(v), 4), "max": round(max(v), 4)}
        rec["torch_over_fused"] = round(statistics.median(ms["torch"]) / statistics.median(ms["fused"]), 2)
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
