"""Times the training step eagerly against the same step replayed as one CUDA graph (graphed.GraphedStep), for the two step kinds the
launcher's --graph-step now captures besides the single-tensor step (run on the GPU box):

    python tools/bench_graph_step.py [--steps K] [--warmup W] [--rounds R] [--out FILE]

Cases:
  fusion_dict  the skeleton + inertial fusion model of tests/fusion_wrapper.py (skeleton branch at the UTD-MHAD shape M=1, T=100,
               V=20, C=3 with the default width 64; inertial branch on the 40-node IMU graph; nn.Linear head, torch cross-entropy)
               on dict batches of 8 sequences: the multimodal step of the early / late fusion configs.
  ntu_accum2   the NTU model (M=2, T=300, V=25, C=3, 60 classes) at 8 sequences per micro-batch with loss_quotient = 2: loss / 2,
               gradients summed over two micro-batches (GraphedStep(accumulate=True, loss_divisor=2)), fused classifier + loss head.

A timed step is one micro-batch: forward + loss + backward, with the gradients zeroed (eager: set to None; graph: zero_grads()) at the
first micro-batch of every optimizer step; the optimizer step itself is excluded, as in bench.py.  The batch is device resident and
the graphed step copies it into its static input every step, as the launcher does.  K (default 8) and W (default 3) are bench.py's
window and warm-up; every round times K steps of each variant with CUDA events, the rounds alternate eager and graph, and the median /
min / max over the rounds is reported.  Eager and graphed steps run on two copies of the same model; after the timing both run one
more optimizer step's micro-batches on the same batches and the report gives the largest relative difference of loss and gradients
(0 = bit-identical).  The GPU name, its power limit and its maximum SM clock are read in the same run.
"""
import argparse
import copy
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from fusion_gcn_b200 import graph as G, modules as M  # noqa: E402
from fusion_gcn_b200.graphed import GraphedStep, loss_and_logits  # noqa: E402
import fusion_wrapper as FW  # noqa: E402

BATCH = 8


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info.update(power_limit_w=float(out[0]), sm_max_mhz=float(out[1]))
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        info.update(power_limit_w=None, sm_max_mhz=None)
    return info


def fusion_dict_case():
    shape = (1, 100, 20, 3)
    torch.manual_seed(1)
    model = FW.SkeletonInertialNet(skeleton_shape=shape, start_feature_size=64).cuda().train()
    batches = [FW.batch(BATCH, skeleton_shape=shape, seed=s) for s in range(2)]
    return model, batches, 1


def ntu_accum_case():
    torch.manual_seed(1)
    model = M.Model((2, 300, 25, 3), 60, G.SkeletonGraph(G.NTU_EDGES, center_joint=G.NTU_CENTER)).cuda().train()
    g = torch.Generator().manual_seed(2)
    batches = [(torch.randn(BATCH, 2, 300, 25, 3, generator=g).cuda(), torch.randint(60, (BATCH,), generator=g).cuda())
               for _ in range(2)]
    return model, batches, 2


CASES = {"fusion_dict": fusion_dict_case, "ntu_accum2": ntu_accum_case}


def eager_step(model, loss_fn, lq):
    def run(i, x, y):
        if i % lq == 0:
            model.zero_grad(set_to_none=True)
        loss, _ = loss_and_logits(model, loss_fn, x, y)
        if lq != 1:
            loss = loss / lq
        loss.backward()
        return loss.detach()
    return run


def graph_step(gs, lq):
    def run(i, x, y):
        if lq != 1 and i % lq == 0:
            gs.zero_grads()
        return gs(x, y)
    return run


def time_steps(run, batches, k):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(k):
        run(i, *batches[i % len(batches)])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / k


def rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).abs().max()) / max(float(b.abs().max()), 1e-30)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--cases", nargs="*", default=list(CASES), choices=list(CASES))
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_graph_step.py needs a CUDA device")
    lines = [json.dumps(dict(gpu_info(), batch=BATCH, steps=args.steps, warmup=args.warmup, rounds=args.rounds,
                             unit="ms per micro-batch step (forward + loss + backward)"))]
    print(lines[-1], flush=True)
    loss_fn = torch.nn.CrossEntropyLoss()
    for name in args.cases:
        model, batches, lq = CASES[name]()
        if args.steps % lq:
            raise SystemExit(f"--steps must be a multiple of the loss quotient {lq}")
        twin = copy.deepcopy(model)
        gs = GraphedStep(twin, loss_fn, *batches[0], warmup=2, accumulate=lq > 1, loss_divisor=lq)
        runs = {"eager": eager_step(model, loss_fn, lq), "graph": graph_step(gs, lq)}
        for run in runs.values():
            for i in range(args.warmup * lq):
                run(i, *batches[i % len(batches)])
        ms = {k: [] for k in runs}
        for _ in range(args.rounds):
            for k, run in runs.items():
                ms[k].append(time_steps(run, batches, args.steps))
        for k, run in runs.items():                     # one more optimizer step's micro-batches on the same batches
            for i in range(lq):
                loss = run(i, *batches[i % len(batches)])
            ms[k + "_loss"] = loss.detach().clone()
        torch.cuda.synchronize()
        grads = [(p.grad, q.grad) for p, q in zip(twin.parameters(), model.parameters()) if q.grad is not None]
        rec = {"case": name, "loss_quotient": lq, "launches_per_replay": gs.launches_per_replay}
        for k in runs:
            v = ms[k]
            rec[f"{k}_ms"] = {"median": round(statistics.median(v), 3), "min": round(min(v), 3), "max": round(max(v), 3)}
        rec["eager_over_graph"] = round(statistics.median(ms["eager"]) / statistics.median(ms["graph"]), 2)
        rec["graph_sequences_per_s"] = round(BATCH * 1e3 / statistics.median(ms["graph"]), 1)
        rec["loss_rel_diff"] = rel(ms["graph_loss"], ms["eager_loss"])
        rec["grad_max_rel_diff"] = max(rel(a, b) for a, b in grads)
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)
        del model, twin, gs, runs
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
