"""Times the eval-mode forward eagerly (under no_grad) against the same forward replayed as one CUDA graph (graphed.GraphedForward)
(run on the GPU box):

    python tools/bench_graph_eval.py [--steps K] [--warmup W] [--rounds R] [--out FILE]

Cases:
  ntu_b8, ntu_b10  the NTU model (M=2, T=300, V=25, C=3, 60 classes) on 8 and 10 sequences: the reference's own batch sizes.
  fusion_dict      the skeleton + inertial fusion model of tests/fusion_wrapper.py (skeleton branch at the UTD-MHAD shape M=1, T=100,
                   V=20, C=3 with the default width 64; inertial branch on the 40-node IMU graph) on dict batches of 8 sequences.
  ntu_val          one validation pass of the NTU model over 101 sequences at batch 8: 12 full batches and one of 5, which the graph
                   zero-pads.  Timed end to end as the launcher runs it: every batch's forward, the clone of the replayed logits
                   into y_pred (graph only; the eager logits are already the session's own tensor) and the cross-entropy loss.

A timed step is one forward (ntu_val: one pass).  The batches are device resident; the graph copies each into its static input, as
the launcher does.  K (default 8) and W (default 3) are bench.py's window and warm-up; every round times K steps of each variant with
CUDA events, the rounds alternate eager and graph, and the median / min / max over the rounds is reported.  Both variants run on the
same model; the report gives the largest relative difference between their logits over every batch of the case (0 = bit-identical;
the shorter batch of ntu_val is compared with the eager forward of its 5 sequences alone, which sums in another order).  The GPU
name, its power limit and its maximum SM clock are read in the same run.
"""
import argparse
import itertools
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from fusion_gcn_b200 import graph as G, modules as M  # noqa: E402
from fusion_gcn_b200.graphed import GraphedForward  # noqa: E402
import fusion_wrapper as FW  # noqa: E402
from bench_graph_step import gpu_info, rel  # noqa: E402

VAL_SEQUENCES, VAL_BATCH = 101, 8


def ntu_model():
    torch.manual_seed(1)
    return M.Model((2, 300, 25, 3), 60, G.SkeletonGraph(G.NTU_EDGES, center_joint=G.NTU_CENTER)).cuda().eval()


def ntu_batches(sizes, seed=2):
    g = torch.Generator().manual_seed(seed)
    return [(torch.randn(n, 2, 300, 25, 3, generator=g).cuda(), torch.randint(60, (n,), generator=g).cuda()) for n in sizes]


def ntu_case(n):
    return lambda: (ntu_model(), ntu_batches([n, n]), False)


def fusion_dict_case():
    shape = (1, 100, 20, 3)
    torch.manual_seed(1)
    model = FW.SkeletonInertialNet(skeleton_shape=shape, start_feature_size=64).cuda().eval()
    return model, [FW.batch(8, skeleton_shape=shape, seed=s) for s in range(2)], False


def ntu_val_case():
    full, last = divmod(VAL_SEQUENCES, VAL_BATCH)
    return ntu_model(), ntu_batches([VAL_BATCH] * full + [last]), True


CASES = {"ntu_b8": ntu_case(8), "ntu_b10": ntu_case(10), "fusion_dict": fusion_dict_case, "ntu_val": ntu_val_case}


def eager_forward(model):
    def run(x):
        with torch.no_grad():
            return model(x)
    return run


def validation_pass(forward, loss_fn, batches, clone):
    """One pass of the session's validation loop: (y_pred, loss) of every batch."""
    def run():
        out = []
        for x, y in batches:
            y_pred = forward(x)
            if clone:
                y_pred = y_pred.clone()
            out.append((y_pred, loss_fn(y_pred, y)))
        return out
    return run


def time_steps(run, k):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(k):
        run()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / k


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--cases", nargs="*", default=list(CASES), choices=list(CASES))
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_graph_eval.py needs a CUDA device")
    lines = [json.dumps(dict(gpu_info(), steps=args.steps, warmup=args.warmup, rounds=args.rounds,
                             unit="ms per eval-mode forward (ntu_val: per validation pass)"))]
    print(lines[-1], flush=True)
    loss_fn = torch.nn.CrossEntropyLoss()
    for name in args.cases:
        model, batches, whole_pass = CASES[name]()
        gf = GraphedForward(model, batches[0][0])
        eager = eager_forward(model)
        if whole_pass:
            runs = {"eager": validation_pass(eager, loss_fn, batches, clone=False),
                    "graph": validation_pass(gf, loss_fn, batches, clone=True)}
        else:
            def step_runs(fwd):
                it = itertools.count()
                return lambda: fwd(batches[next(it) % len(batches)][0])
            runs = {"eager": step_runs(eager), "graph": step_runs(gf)}
        for run in runs.values():
            for _ in range(args.warmup):
                run()
        ms = {k: [] for k in runs}
        for _ in range(args.rounds):
            for k, run in runs.items():
                ms[k].append(time_steps(run, args.steps))
        diff = 0.0
        for x, _ in batches:
            a = gf(x).clone()
            diff = max(diff, rel(a, eager(x)))
        torch.cuda.synchronize()
        rec = {"case": name, "sequences": sum(int(y.shape[0]) for _, y in batches) if whole_pass else int(batches[0][1].shape[0]),
               "captured_batch": gf.batch_size, "launches_per_replay": gf.launches_per_replay}
        for k in runs:
            v = ms[k]
            rec[f"{k}_ms"] = {"median": round(statistics.median(v), 3), "min": round(min(v), 3), "max": round(max(v), 3)}
        rec["eager_over_graph"] = round(statistics.median(ms["eager"]) / statistics.median(ms["graph"]), 2)
        rec["graph_sequences_per_s"] = round(rec["sequences"] * 1e3 / statistics.median(ms["graph"]), 1)
        rec["logits_max_rel_diff"] = diff
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)
        del model, gf, runs
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
