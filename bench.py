#!/usr/bin/env python
"""AGCN fwd+bwd sequences/s on B200 (BASELINE.json metric), one process per GPU.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload ntu|utd|mmact_imu|utd_rgb] [--dump-outputs DIR]
  torchrun ... bench.py --gpus N ...        (N > 1: batch-sharded replicas + NCCL gradient all-reduce)

A step = zero_grad + forward + cross-entropy + backward (+ gradient all-reduce when N > 1) of the full 10-unit AGCN
model on one synthetic batch; the optimizer step is excluded (SURVEY 8d).  Default workload: BASELINE configs[1], the
2s-AGCN joint stream at NTU shape (64 sequences per GPU, M=2, T=300, V=25, C=3, 60 classes), train mode, fp32 parity mode.
Rank 0 prints ONE JSON line (see the task contract): value = device-resident throughput, e2e = through the public
module API from pinned HOST buffers with the H2D/D2H copies inside the timed region, roofline = the dominant kernel
timed live with CUDA events, cpu_baseline = the oracle port of the reference on the host cores (bounded sample).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {   # name: (M, T, V, C, classes, graph)
    "ntu": (2, 300, 25, 3, 60, "ntu"),
    "utd": (1, 100, 20, 3, 27, "utd"),
    "mmact_imu": (2, 300, 22, 3, 35, "mmact_imu"),
    "utd_rgb": (1, 100, 25, 515, 27, "ntu"),
}
# algorithmic work per sequence, fwd+bwd (SURVEY 8d / Appendix B): GFLOP and MB (model M1, fp32 activations)
WORK = {"ntu": (116.44, 1441.0), "utd": (15.39, 192.0), "mmact_imu": (101.92, 1268.0), "utd_rgb": (22.69, 271.0)}


def make_graph(kind):
    from fusion_gcn_b200 import graph as G
    if kind == "ntu":
        return G.SkeletonGraph(G.NTU_EDGES, center_joint=G.NTU_CENTER)
    if kind == "utd":
        return G.SkeletonGraph(G.UTD_EDGES, center_joint=G.UTD_CENTER)
    return G.imu_fusion_graph(G.SkeletonGraph(G.MMACT_EDGES, center_joint=G.MMACT_CENTER), 4, "append_center")


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    fallback = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}
    tf32 = {}
    tpath = os.path.join(ROOT, "profiles", "tf32_peak.json")            # tools/measure_peaks.py on a B200 of this pool (cuBLAS TF32 8192^3)
    if os.path.isfile(tpath):
        try:
            t = json.load(open(tpath))
            tf32 = {"tf32_tflops": float(t["tf32_tflops"]), "tf32_tflops_sustained": float(t["tf32_tflops_sustained"])}
        except (KeyError, TypeError, ValueError):
            tf32 = {}
    fallback.update(tf32)
    if os.path.isfile(path):
        try:
            d = json.load(open(path))
            return dict({"hbm_gbs": float(d["hbm_gbs"]), "bf16_tflops": float(d["bf16_tflops"]),
                         "bf16_tflops_sustained": d.get("bf16_tflops_sustained"), "source": "measured"}, **tf32)
        except (KeyError, TypeError, ValueError):          # unexpected layout: say so and use the recipe's fallback numbers
            fallback["source"] = "fallback (MEASURED_PEAKS.json present but not in the expected layout)"
    return fallback


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        self.thread.join(timeout=2)
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [s.strip() for s in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


DUMP_BUDGET = 60 << 20     # bytes of array data written by --dump-outputs: with the .npy headers, well inside 64 MB


def dump_outputs(outdir, arrays):
    """Writes every array as outdir/<name>.npy.  Past DUMP_BUDGET each array keeps its share of the budget as a fixed, seeded
    sample of its flattened elements, so that two runs with the same arguments still write the same elements (none of the
    workloads above gets there: a training step's outputs are about 14 MB)."""
    import numpy as np
    os.makedirs(outdir, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    rng = np.random.default_rng(0)
    for name, a in arrays.items():
        if total > DUMP_BUDGET:
            a = a.reshape(-1)[np.sort(rng.choice(a.size, max(1, a.size * DUMP_BUDGET // total), replace=False))]
        np.save(os.path.join(outdir, name + ".npy"), a)


def build_model(workload, precision, device, recompute=False):
    from fusion_gcn_b200 import modules as M
    m, t, v, c, ncls, gk = WORKLOADS[workload]
    torch.manual_seed(1)
    model = M.Model((m, t, v, c), ncls, make_graph(gk))
    M.set_precision(model, precision)
    M.set_recompute(model, recompute)
    return model.to(device).train()


def run_ours(args):
    import torch.distributed as dist
    from fusion_gcn_b200 import capi, ops
    from fusion_gcn_b200.distributed import GradientAllReducer
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch N>1 with torch.distributed.run")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    m, t, v, c, ncls, _ = WORKLOADS[args.workload]
    if args.scaling == "strong":
        if args.batch % world:
            raise SystemExit(f"--scaling strong: global batch {args.batch} is not divisible by {world} GPUs")
        n_local = args.batch // world         # strong scaling: the GLOBAL batch is fixed (BASELINE configs[1]: N=64 sharded 32/16/8 per GPU)
    else:
        n_local = args.batch                  # weak scaling: fixed per-GPU batch
    if args.no_overlap:
        import fusion_gcn_b200.functional as FN_
        FN_.set_overlap_leaves(False)
    model = build_model(args.workload, args.precision, dev, recompute=args.recompute)
    if args.sync_bn and world > 1:
        from fusion_gcn_b200 import modules as M_
        M_.set_sync_batchnorm(model, True)     # statistics over all ranks: the sharded batch normalises like the unsharded one
    reducer = GradientAllReducer(model.parameters()) if world > 1 else None
    gen = torch.Generator().manual_seed(1234 + rank)
    x_host = torch.randn(n_local, m, t, v, c, generator=gen).pin_memory()
    y_host = torch.randint(ncls, (n_local,), generator=gen).pin_memory()
    x_dev, y_dev = x_host.to(dev), y_host.to(dev)
    loss_fn = torch.nn.CrossEntropyLoss()

    from fusion_gcn_b200.graphed import loss_and_logits

    def step(x, y):
        model.zero_grad(set_to_none=True)
        loss, logits = loss_and_logits(model, loss_fn, x, y)       # fc + cross-entropy as one kernel (Model.loss)
        loss.backward()
        if reducer is not None:
            reducer()
        return loss.detach(), logits.detach()       # detached: a kept result must not keep the step's autograd graph alive
                                                    # (its AccumulateGrad nodes would invalidate the CUDA-graph capture below)

    def step_outputs(loss, logits):
        """What a caller of the training step receives: the loss, the logits and every parameter gradient."""
        out = {"loss": loss, "logits": logits}
        out.update({"grad." + k: p.grad for k, p in model.named_parameters() if p.grad is not None})
        return {k: v.detach().float().cpu().numpy() for k, v in out.items()}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step(x_dev, y_dev)
    # ---- device-resident timed region, with per-launch CUDA events on the conv entry points (roofline evidence)
    ops.start_timing(("*",))
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    l0 = capi.lib().agcn_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss, logits = step(x_dev, y_dev)
    e1.record()
    barrier()
    launches = capi.lib().agcn_launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    timings = ops.stop_timing()
    ms = e0.elapsed_time(e1)
    eager_outputs = step_outputs(loss, logits) if args.dump_outputs else None
    graph_outputs = None
    # ---- end-to-end: host pinned buffers -> device every step, loss read back every step
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(args.steps):
        xb = x_host.to(dev, non_blocking=True)
        yb = y_host.to(dev, non_blocking=True)
        loss_val = step(xb, yb)[0].item()
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    # ---- the same step replayed as ONE CUDA graph (SURVEY 8 f1; fusion_gcn_b200/graphed.py): device-resident and end to end
    ms_graph = ms_graph_e2e = 0.0
    graph_info = None
    graph_ok = 0.0
    if not args.no_graph:
        try:
            from fusion_gcn_b200.graphed import GraphedStep
            gs = GraphedStep(model, loss_fn, x_dev, y_dev, warmup=1, after_backward=reducer)
            for _ in range(args.warmup):
                gs()
            barrier()
            h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            h0.record()
            for _ in range(args.steps):
                gs()
            h1.record()
            barrier()
            ms_graph = h0.elapsed_time(h1)
            graph_outputs = step_outputs(gs.loss, gs.logits) if args.dump_outputs else None
            e2e_path = None
            nbar = 0                                     # barriers passed inside the try: a rank that falls back must not add any
            try:
                # end to end through the package's own input pipeline (SURVEY 8 f3): every step's batch is gathered out of a host array
                # into a pinned staging buffer by pipeline.PrefetchLoader's worker thread, copied H2D on its copy stream (inside the
                # timed region, overlapped with the previous step) and handed to the graphed step; the loss is read with .item() every step
                from fusion_gcn_b200.pipeline import FeatureStore, PrefetchLoader
                nb_e2e = args.steps + 2
                store = FeatureStore.from_arrays(
                    {"skeleton": x_host.numpy()[None].repeat(nb_e2e, axis=0).reshape((nb_e2e * n_local,) + tuple(x_host.shape[1:]))},
                    y_host.numpy()[None].repeat(nb_e2e, axis=0).reshape(-1))
                batches = iter(PrefetchLoader(store, n_local, shuffle=False, drop_last=True, device=dev, depth=3))
                for _ in range(2):                       # pipeline warm-up: the staging ring fills
                    xb, yb, _idx = next(batches)
                    gs(xb, yb).item()
                barrier()
                nbar = 1
                h0.record()
                for _ in range(args.steps):
                    xb, yb, _idx = next(batches)
                    graph_loss = gs(xb, yb).item()
                h1.record()
                barrier()
                nbar = 2
                ms_graph_e2e = h0.elapsed_time(h1)
                for _ in batches:                        # (drains the loader: its worker thread ends)
                    pass
                del store, batches
                e2e_path = ("pipeline.PrefetchLoader (host array -> pinned staging -> asynchronous H2D on a copy stream, one batch per step "
                            "inside the timed region) -> graphed.GraphedStep -> loss.item() every step")
            except Exception as exc:                     # noqa: BLE001 -- the plain synchronous loop stands in
                if nbar < 2:
                    e2e_path = f"synchronous copies (prefetch loader failed: {type(exc).__name__}: {exc})"[:200]
                    if nbar == 0:
                        barrier()
                    torch.cuda.synchronize()
                    h0.record()
                    for _ in range(args.steps):
                        graph_loss = gs(x_host, y_host).item()
                    h1.record()
                    barrier()
                    ms_graph_e2e = h0.elapsed_time(h1)
            graph_info = {"launches_per_replay": gs.launches_per_replay, "last_loss": round(graph_loss, 5), "e2e_path": e2e_path}
            graph_ok = 1.0
            del gs
        except Exception as exc:                     # noqa: BLE001 -- reported in the JSON line, the eager numbers stand
            graph_info = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        model.zero_grad(set_to_none=True)
        torch.cuda.empty_cache()
    # ---- the separately reported TF32 mode (single-pass tensor cores, own tolerance), device-resident, same step
    ms_tf32 = ms_tf32_graph = 0.0
    if args.precision in ("fp32", "bf16x3") and not args.no_tf32:
        from fusion_gcn_b200 import modules as M
        M.set_precision(model, "tf32")
        for _ in range(args.warmup):
            step(x_dev, y_dev)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(args.steps):
            step(x_dev, y_dev)
        g1.record()
        barrier()
        ms_tf32 = g0.elapsed_time(g1)
        if graph_ok and not args.no_graph:               # same launch mode as the headline: one CUDA graph per step
            try:
                gs = GraphedStep(model, loss_fn, x_dev, y_dev, warmup=1, after_backward=reducer)
                for _ in range(args.warmup):
                    gs()
                barrier()
                g0.record()
                for _ in range(args.steps):
                    gs()
                g1.record()
                barrier()
                ms_tf32_graph = g0.elapsed_time(g1)
                del gs
            except Exception:                            # noqa: BLE001 -- the eager TF32 number stands
                ms_tf32_graph = 0.0
            model.zero_grad(set_to_none=True)
        M.set_precision(model, args.precision)
    # ---- N > 1: the same GLOBAL batch sharded over the GPUs (strong scaling, BASELINE configs[1]), one CUDA graph per step
    ms_strong = 0.0
    n_strong = args.batch // world if args.batch % world == 0 else 0
    if world > 1 and args.scaling == "weak" and not args.no_strong and not args.no_graph and graph_ok and n_strong > 0:
        try:
            xs, ys = x_dev[:n_strong].contiguous(), y_dev[:n_strong].contiguous()
            gs = GraphedStep(model, loss_fn, xs, ys, warmup=2, after_backward=reducer)
            for _ in range(args.warmup):
                gs()
            barrier()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            for _ in range(args.steps):
                gs()
            s1.record()
            barrier()
            ms_strong = s0.elapsed_time(s1)
            del gs
        except Exception:                                # noqa: BLE001 -- the weak-scaling numbers stand
            ms_strong = 0.0
        model.zero_grad(set_to_none=True)
    t_all = torch.tensor([ms, ms_e2e, ms_tf32, ms_graph, ms_graph_e2e, -graph_ok, ms_tf32_graph, -float(ms_tf32_graph > 0),
                          ms_strong, -float(ms_strong > 0)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_all, op=dist.ReduceOp.MAX)
    ms, ms_e2e, ms_tf32, ms_graph, ms_graph_e2e = (float(t_all[i]) for i in range(5))
    ms_tf32_graph = float(t_all[6]) if float(t_all[7]) <= -1.0 else 0.0
    ms_strong = float(t_all[8]) if float(t_all[9]) <= -1.0 else 0.0
    graph_ok = float(t_all[5]) <= -1.0 and ms_graph > 0          # every rank captured and replayed
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, graph_outputs if graph_ok else eager_outputs)
    pk = peaks()
    n_global = n_local * world
    # headline: the step replayed as one CUDA graph (the package's GraphedStep) when every rank captured it, else the eager launches
    ms_head, ms_head_e2e = (ms_graph, ms_graph_e2e) if graph_ok else (ms, ms_e2e)
    value = n_global * args.steps / (ms_head / 1e3)
    e2e_value = n_global * args.steps / (ms_head_e2e / 1e3)
    if graph_ok:
        launches = graph_info["launches_per_replay"] * args.steps
        loss_val = graph_info["last_loss"]
    # dominant kernel: the C-ABI launch signature with the largest summed device time (CUDA events around every call)
    roof, top, families = None, [], {}
    if timings:
        traffic_db = {}
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.isfile(tpath):
            traffic_db = json.load(open(tpath))
        tensor_peak = pk["bf16_tflops_sustained"] or pk["bf16_tflops"]

        def describe(key, val):
            (name, sig), (tot_ms, cnt, flops, nbytes) = key, val
            avg_s = tot_ms / cnt / 1e3
            tf, gbs = flops / avg_s / 1e12, nbytes / avg_s / 1e9
            ident = f"{name}{list(sig)}"
            return {"kernel": ident, "avg_launch_ms": round(avg_s * 1e3, 4), "launches_timed": cnt, "share_of_step": round(tot_ms / ms, 4),
                    "tflops": round(tf, 2), "gbs": round(gbs, 1), "frac_tensor": round(tf / tensor_peak, 4), "frac_hbm": round(gbs / pk["hbm_gbs"], 4),
                    "traffic": (traffic_db.get(ident) or {}).get("dram_bytes")}

        ranked = sorted(timings.items(), key=lambda kv: -kv[1][0])
        top = [describe(k, v) for k, v in ranked[:6]]
        for (name, _sig), (tot_ms, cnt, _f, _b) in ranked:        # share of the step per C-ABI entry point (all signatures)
            fam = families.setdefault(name, [0.0, 0])
            fam[0] += tot_ms
            fam[1] += cnt
        if args.dump_kernels:
            with open(args.dump_kernels, "w") as fh:
                json.dump([describe(k, v) for k, v in ranked], fh, indent=0)
        # dominant kernel FAMILY (C-ABI entry point x temporal taps): all its launches summed, algorithmic work / device time
        fam_work = {}
        for (name, sig), (tot_ms, cnt, flops, nbytes) in ranked:
            label = name
            if name in ("agcn_conv_fwd", "agcn_conv_wgrad"):
                label = f"{name}[taps={sig[6]}]"
            f = fam_work.setdefault(label, [0.0, 0, 0.0, 0.0])
            f[0] += tot_ms; f[1] += cnt; f[2] += flops * cnt; f[3] += nbytes * cnt
        fl, (f_ms, f_cnt, f_flops, f_bytes) = max(fam_work.items(), key=lambda kv: kv[1][0])
        fam_tf, fam_gbs = f_flops / (f_ms / 1e3) / 1e12, f_bytes / (f_ms / 1e3) / 1e9
        family_roof = {"family": fl, "share_of_step": round(f_ms / ms, 4), "launches_per_step": round(f_cnt / args.steps, 1),
                       "tflops": round(fam_tf, 2), "gbs": round(fam_gbs, 1), "frac_tensor_bf16": round(fam_tf / tensor_peak, 4),
                       "frac_hbm": round(fam_gbs / pk["hbm_gbs"], 4)}
        if pk.get("tf32_tflops_sustained"):
            # issued-FLOP view: tensor-pipe time per algorithmic MAC = (TF32 products) / TF32 peak + (BF16 products) / BF16 peak.
            # strict fp32: hi*hi on kind::tf32 + lo*hi + hi*lo on kind::f16 (weight gradients: 3 BF16 products); bf16x3: 3 BF16; tf32: 1 TF32
            wgrad_family = fl.startswith("agcn_conv_wgrad")
            n_tf32, n_bf16, what = {"fp32": (0, 3, "3 x BF16") if wgrad_family else (1, 2, "1 x TF32 + 2 x BF16"),
                                    "bf16x3": (0, 3, "3 x BF16"), "tf32": (1, 0, "1 x TF32")}[args.precision]
            if not fl.startswith("agcn_conv_"):         # gram / mix stages: TF32 hi*hi + BF16 cross terms in both parity modes
                n_tf32, n_bf16, what = (1, 0, "1 x TF32") if args.precision == "tf32" else (1, 2, "1 x TF32 + 2 x BF16")
            ceiling = 1.0 / (n_tf32 / pk["tf32_tflops_sustained"] + n_bf16 / tensor_peak)
            family_roof["frac_tensor_mode"] = round(fam_tf / ceiling, 4)
            family_roof["mode_peak"] = (f"{what} products per MAC: ceiling {ceiling:.1f} algorithmic TFLOP/s from the measured sustained peaks "
                                        f"(TF32 {pk['tf32_tflops_sustained']}, BF16 {tensor_peak} TFLOP/s)")
        d = top[0]
        hbm_bound = d["frac_hbm"] >= d["frac_tensor"]
        roof = {"bound": "hbm" if hbm_bound else "tensor", "achieved": d["gbs"] if hbm_bound else d["tflops"],
                "peak": pk["hbm_gbs"] if hbm_bound else tensor_peak, "unit": "GB/s" if hbm_bound else "TFLOP/s",
                "frac": d["frac_hbm"] if hbm_bound else d["frac_tensor"], "traffic": d["traffic"], "traffic_unit": "DRAM bytes per launch (ncu --set full, "
                "dram__bytes_read.sum + dram__bytes_write.sum, profiles/ncu_traffic.json); algorithmic bytes per launch = gbs * avg_launch_ms * 1e6",
                "kernel": d["kernel"],
                "avg_launch_ms": d["avg_launch_ms"], "launches_timed": d["launches_timed"], "share_of_step": d["share_of_step"],
                "frac_tensor": d["frac_tensor"], "frac_hbm": d["frac_hbm"],
                "peak_source": pk["source"] + (" copy bandwidth" if hbm_bound else " bf16 sustained (kernel timed inside a long step)"),
                "top_family": family_roof,
                "note": "achieved = algorithmic work of one launch (DESIGN.md section 4) / mean CUDA-event time of that launch signature inside the "
                        "timed region; bound = the roof the kernel sits closer to. The strict fp32 mode issues one TF32 and two BF16 MMAs per product "
                        "(weight gradients: three BF16), so its tensor ceiling for algorithmic FLOPs is top_family.mode_peak, not the bf16 peak used as denominator."}
    gflop, mbytes = WORK[args.workload]
    line = {
        "metric": "AGCN fwd+bwd sequences/sec", "value": round(value, 2), "unit": "sequences/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(ms_head / args.steps, 3), "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "tf32" if args.precision == "tf32" else "f32", "data": "synthetic",
        "config": {"workload": f"{args.workload}: AGCN 10 units, N={n_local}/GPU (global {n_global}), M={m}, T={t}, V={v}, C={c}, "
                               f"{ncls} classes, train mode, fwd+CE+bwd, random init", "precision_mode": args.precision,
                   "l2_policy": "activations per step (GBs) exceed the 126 MB L2; no explicit flush",
                   "parallelism": f"dp{world} (batch shards, NCCL gradient all-reduce)" if world > 1 else "single GPU",
                   "launch_mode": "one CUDA graph per step (fusion_gcn_b200.graphed.GraphedStep)" if graph_ok else "eager launches",
                   "batchnorm": "synchronised over the ranks (--sync-bn)" if (args.sync_bn and world > 1) else "per-replica statistics",
                   "streams": "weight gradients on the main stream (--no-overlap)" if args.no_overlap else "weight gradients on a side stream beside the main chain",
                   "activation_policy": "theta/phi and the aggregated tensor recomputed in the backward (--recompute)" if args.recompute
                                        else "all activations kept"},
        "peak_memory_gb": round(torch.cuda.max_memory_allocated() / 2 ** 30, 2),
        "e2e": {"value": round(e2e_value, 2), "unit": "sequences/s", "h2d_bytes_per_step": x_host.numel() * 4 + y_host.numel() * 8,
                "d2h_bytes_per_step": 4, "ms_per_step": round(ms_head_e2e / args.steps, 3), "last_loss": round(loss_val, 5)},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roof,
        "top_kernels": top,
        "entry_point_shares": {k: {"share_of_step": round(v[0] / ms, 4), "launches_per_step": round(v[1] / args.steps, 1)}
                               for k, v in sorted(families.items(), key=lambda kv: -kv[1][0])},
        "tf32_mode": None if ms_tf32 <= 0 else {
            "value": round(n_global * args.steps / ((ms_tf32_graph or ms_tf32) / 1e3), 2), "unit": "sequences/s",
            "ms_per_step": round((ms_tf32_graph or ms_tf32) / args.steps, 3),
            "launch_mode": "one CUDA graph per step" if ms_tf32_graph else "eager launches",
            "eager_value": round(n_global * args.steps / (ms_tf32 / 1e3), 2),
            "note": "AGCN_PREC_TF32 (single-pass tcgen05 kind::tf32, operands truncated to TF32), reported separately from the fp32 parity "
                    "mode; tolerance: logits within 3e-2 of the fp64 oracle (tests/test_gpu_unit.py::test_tf32_mode_model_logits)"},
        "eager_mode": {"value": round(n_global * args.steps / (ms / 1e3), 2), "e2e_value": round(n_global * args.steps / (ms_e2e / 1e3), 2),
                       "unit": "sequences/s", "ms_per_step": round(ms / args.steps, 3),
                       "note": "the same step launched kernel by kernel from Python, with a CUDA-event pair around every C-ABI call "
                               "(this is the region `roofline`, `top_kernels` and `entry_point_shares` are measured in)"},
        "graph_mode": None if graph_info is None else dict(graph_info, **({} if ms_graph <= 0 else {
            "value": round(n_global * args.steps / (ms_graph / 1e3), 2), "e2e_value": round(n_global * args.steps / (ms_graph_e2e / 1e3), 2),
            "unit": "sequences/s", "ms_per_step": round(ms_graph / args.steps, 3),
            "note": "same step (zero-grad + fwd + CE + bwd [+ gradient all-reduce]) captured once and replayed as one CUDA graph; e2e_value "
                    "copies the batch from pinned host memory into the graph's static input and reads the loss back every step"})),
        "strong_scaling": None if ms_strong <= 0 else {
            "value": round(n_strong * world * args.steps / (ms_strong / 1e3), 2), "unit": "sequences/s", "global_batch": n_strong * world,
            "per_gpu_batch": n_strong, "ms_per_step": round(ms_strong / args.steps, 3),
            "note": "BASELINE configs[1]: the N=64 batch sharded over the GPUs (32/16/8 sequences per GPU at 2/4/8), one CUDA graph per step "
                    "with the bucketed all-reduce overlapped with backward; compare with the 1-GPU headline for strong-scaling efficiency"},
        "model_roofline": {"hbm_seq_s": round(pk["hbm_gbs"] * 1e3 / mbytes, 1), "achieved_frac_of_hbm_ceiling": round(value / world / (pk["hbm_gbs"] * 1e3 / mbytes), 4),
                           "algorithmic_gflop_per_seq": gflop, "algorithmic_mb_per_seq": mbytes,
                           "achieved_tflops": round(value * gflop / 1e3, 2), "achieved_gbs": round(value / world * mbytes / 1e3, 1)},
    }
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_reference(args.workload, steps=5, warmup=1)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_infer(args):
    """BASELINE config 5: forward only, eval mode, torch.no_grad(), large batch, replicas without communication."""
    import torch.distributed as dist
    from fusion_gcn_b200 import capi, ops
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch N>1 with torch.distributed.run")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    m, t, v, c, ncls, _ = WORKLOADS[args.workload]
    n_local, micro = args.batch, min(args.batch, args.micro_batch)
    model = build_model(args.workload, args.precision, dev).eval()
    gen = torch.Generator().manual_seed(1234 + rank)
    x_host = torch.randn(n_local, m, t, v, c, generator=gen).pin_memory()
    x_dev = x_host.to(dev)

    def step(x):
        with torch.no_grad():
            return torch.cat([model(x[i:i + micro]) for i in range(0, n_local, micro)])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step(x_dev)
    ops.start_timing(("*",))
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    l0 = capi.lib().agcn_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        logits = step(x_dev)
    e1.record()
    barrier()
    launches = capi.lib().agcn_launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    timings = ops.stop_timing()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"logits": logits.float().cpu().numpy()})
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(args.steps):
        pred = step(x_host.to(dev, non_blocking=True)).argmax(1).cpu()
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    t_all = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t_all, op=dist.ReduceOp.MAX)
        dist.destroy_process_group()
    if rank != 0:
        return
    ms, ms_e2e = float(t_all[0]), float(t_all[1])
    pk = peaks()
    n_global = n_local * world
    value = n_global * args.steps / (ms / 1e3)
    gflop, mbytes = WORK[args.workload][0] / 3.0, WORK[args.workload][1] / 3.0      # forward = a third of fwd+bwd (SURVEY Appendix B)
    fam = {}
    for (name, _sig), (tot_ms, cnt, _f, _b) in timings.items():
        e = fam.setdefault(name, [0.0, 0]); e[0] += tot_ms; e[1] += cnt
    (kname, ksig), (ktot, kcnt, kflops, kbytes) = max(timings.items(), key=lambda kv: kv[1][0])
    avg_s = ktot / kcnt / 1e3
    tensor_peak = pk["bf16_tflops_sustained"] or pk["bf16_tflops"]
    f_h, f_t = kbytes / avg_s / 1e9 / pk["hbm_gbs"], kflops / avg_s / 1e12 / tensor_peak
    hbm_bound = f_h >= f_t
    line = {
        "metric": "AGCN forward sequences/sec (inference sweep, BASELINE config 5)", "value": round(value, 2), "unit": "sequences/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32" if args.precision == "fp32" else "tf32", "data": "synthetic",
        "config": {"workload": f"{args.workload}: AGCN 10 units, forward only, eval mode, no_grad, N={n_local}/GPU (micro-batches of {micro}), "
                               f"M={m}, T={t}, V={v}, C={c}, {ncls} classes, random init", "precision_mode": args.precision,
                   "l2_policy": "activations per step (GBs) exceed the 126 MB L2; no explicit flush",
                   "parallelism": "replicas only, no communication" if world > 1 else "single GPU"},
        "e2e": {"value": round(n_global * args.steps / (ms_e2e / 1e3), 2), "unit": "sequences/s", "h2d_bytes_per_step": x_host.numel() * 4,
                "d2h_bytes_per_step": n_local * 8, "ms_per_step": round(ms_e2e / args.steps, 3), "last_pred0": int(pred[0])},
        "gpu_launches": int(launches), "clocks": clocks,
        "roofline": {"bound": "hbm" if hbm_bound else "tensor", "achieved": round(kbytes / avg_s / 1e9 if hbm_bound else kflops / avg_s / 1e12, 2),
                     "peak": pk["hbm_gbs"] if hbm_bound else tensor_peak, "unit": "GB/s" if hbm_bound else "TFLOP/s",
                     "frac": round(f_h if hbm_bound else f_t, 4), "traffic": None, "kernel": f"{kname}{list(ksig)}",
                     "avg_launch_ms": round(avg_s * 1e3, 4), "share_of_step": round(ktot / ms, 4), "peak_source": pk["source"]},
        "entry_point_shares": {k: {"share_of_step": round(v_[0] / ms, 4), "launches_per_step": round(v_[1] / args.steps, 1)}
                               for k, v_ in sorted(fam.items(), key=lambda kv: -kv[1][0])},
        "model_roofline": {"hbm_seq_s": round(pk["hbm_gbs"] * 1e3 / mbytes, 1), "achieved_frac_of_hbm_ceiling": round(value / world / (pk["hbm_gbs"] * 1e3 / mbytes), 4),
                           "algorithmic_gflop_per_seq": round(gflop, 2), "algorithmic_mb_per_seq": round(mbytes, 1)},
    }
    print(json.dumps(line), flush=True)


def _reference_graph(ref, gk):
    """The reference's own util.graph.Graph for the workload (datasets/*/constants.py edge lists, fusion.py:65-89)."""
    const = {"ntu": ref["ntu"], "utd": ref["utd"], "mmact_imu": ref["mmact"]}[gk]
    g = ref["Graph"](const.skeleton_edges, center_joint=const.center_joint)
    if gk == "mmact_imu":
        g = ref["fusion"].get_skeleton_imu_fusion_graph(g, "append_center", 4)
    return g


def cpu_reference(workload, steps, warmup, n=None):
    """The reference's CPU path on the host cores, all host threads, bounded sample of the same workload (N=16 sequences per
    step).  kind "reference": the UNMODIFIED torch_src/models/mmargcn/agcn.py::Model, imported from the byte copy that
    baseline/install_ref.py places under baseline/_ref (or /root/reference in the build container), with the reference's own
    Graph / partition strategy, nn.CrossEntropyLoss and loss.backward() as in torch_src/session/procedures/step.py:39-46.
    kind "port": oracle/agcn_oracle.py (same ATen ops), only when no reference copy is present."""
    from oracle import agcn_oracle as O, ref_loader
    from fusion_gcn_b200 import graph as G
    m, t, v, c, ncls, gk = WORKLOADS[workload]
    n = n or 16
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    gen = torch.Generator().manual_seed(1234)
    x = torch.randn(n, m, t, v, c, generator=gen)
    y = torch.randint(ncls, (n,), generator=gen)
    kind = "port"
    if ref_loader.available():
        try:
            ref = ref_loader.load()
            torch.manual_seed(1)
            model = ref["agcn"].Model((m, t, v, c), ncls, _reference_graph(ref, gk)).train()
            loss_fn = torch.nn.CrossEntropyLoss()

            def one_step():
                model.zero_grad(set_to_none=True)
                loss = loss_fn(model(x), y)
                loss.backward()
                return loss
            kind = "reference"
        except Exception as exc:            # noqa: BLE001 -- fall back to the port and say so
            sys.stderr.write(f"bench.py: reference import failed ({type(exc).__name__}: {exc}); timing the oracle port instead\n")
    if kind == "port":
        adj = G.adjacency_from_graph(make_graph(gk))
        p = O.as_leaves(O.init_state(adj, (m, t, v, c), ncls, seed=1))
        leaves = [a for a in p.values() if a.requires_grad]

        def one_step():
            for a in leaves:
                a.grad = None
            loss = torch.nn.functional.cross_entropy(O.model_forward(x, p, c, True), y)
            loss.backward()
            return loss
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        one_step()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    total = sum(times)
    return {"value": round(n * len(times) / total, 3), "unit": "sequences/s", "cores": torch.get_num_threads(), "kind": kind,
            "sample": f"{len(times)} steps of N={n} sequences at the {workload} shape (same model, fwd+CE+bwd, fp32, train mode)",
            "ms_per_step": round(total / len(times) * 1e3, 1)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    m, t, v, c, ncls, _ = WORKLOADS[args.workload]
    steps = args.steps
    base = cpu_reference(args.workload, steps=steps, warmup=max(1, min(args.warmup, 2)))
    line = {"impl": "reference", "metric": "AGCN fwd+bwd sequences/sec", "value": base["value"], "unit": "sequences/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": max(1, min(args.warmup, 2)), "ms_per_step": base["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.workload}: AGCN 10 units, M={m}, T={t}, V={v}, C={c}, {ncls} classes, train mode, fwd+CE+bwd; "
                                   f"reference CPU path ({base['kind']}) on the host cores, bounded sample: {base['sample']}"},
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": "sequences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="ntu", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=None, help="sequences per GPU (default 64; 256 for --mode infer)")
    ap.add_argument("--mode", default="train", choices=["train", "infer"], help="train: fwd+CE+bwd (the BASELINE metric); infer: forward only, eval mode")
    ap.add_argument("--micro-batch", type=int, default=512, help="--mode infer: sequences per forward call")
    ap.add_argument("--precision", default="fp32", choices=["fp32", "bf16x3", "tf32"],
                    help="fp32 = strict parity mode (TF32 hi*hi + BF16 cross terms), bf16x3 = bf16 triple-product parity mode (both meet 1e-4), tf32 = single pass (own tolerance)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --batch sequences per GPU (default); strong: --batch sequences in total, sharded over the GPUs")
    ap.add_argument("--no-strong", action="store_true", help="N > 1, weak scaling: skip the extra strong-scaling timing (global batch = --batch)")
    ap.add_argument("--dump-kernels", default=None, help="write the per-signature timing table (all C-ABI launches) to this JSON file")
    ap.add_argument("--sync-bn", action="store_true", help="N > 1: synchronised BatchNorm (modules.set_sync_batchnorm), default per-replica statistics")
    ap.add_argument("--no-overlap", action="store_true", help="weight gradients on the main stream (functional.OVERLAP_LEAVES off), for A/B")
    ap.add_argument("--recompute", action="store_true", help="activation-recompute policy (modules.set_recompute): less memory, two more launches per unit")
    ap.add_argument("--no-graph", action="store_true", help="skip the CUDA-graph replay timing")
    ap.add_argument("--no-tf32", action="store_true", help="skip the extra TF32-mode timing that the fp32 run reports beside the headline")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the headline path computed in its last step as DIR/<name>.npy (float32): "
                         "loss, logits and every parameter gradient (grad.<parameter>); --mode infer: the logits")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of this package's timed path (--impl ours)")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.batch is None:
        args.batch = 256 if args.mode == "infer" else 64
    if args.impl == "reference":
        run_reference(args)
    elif args.mode == "infer":
        run_infer(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
