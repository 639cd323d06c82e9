"""Per-kernel timing at the NTU layer shapes (run on the GPU box):  python tools/bench_stage.py [name ...] [--tf32] [--once]

Times single C-ABI entry points with CUDA events (L2 flushed between repetitions by the sheer tensor sizes) and prints the
algorithmic GB/s and TFLOP/s of each.  ``--once`` runs each case a single time (for use under ncu).
Cases are (unit width, T) pairs of the 10-unit NTU model at N'=128 person-sequences.
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from fusion_gcn_b200 import ops as K  # noqa: E402

NB, V = 128, 25
SHAPES = {"c64": (64, 300), "c128": (128, 150), "c256": (256, 75)}


def timeit(fn, once):
    if once:
        fn()
        torch.cuda.synchronize()
        return float("nan")
    for _ in range(2):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    reps = 5
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def report(name, ms, nbytes, flops):
    print(f"{name:34s} {ms:8.3f} ms  {nbytes / ms / 1e6:8.1f} GB/s  {flops / ms / 1e9:8.1f} TFLOP/s", flush=True)


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    once = "--once" in sys.argv
    prec = K.PREC_TF32 if "--tf32" in sys.argv else K.PREC_BF16X3 if "--bf16x3" in sys.argv else K.PREC_FP32
    want = lambda n: not args or any(a in n for a in args)   # noqa: E731
    dev = "cuda"
    for tag, (c, t) in SHAPES.items():
        ci = c // 4
        rows = NB * t * V
        x = torch.randn(NB, t, V, c, device=dev)
        act = rows * c * 4
        if want(f"gram_score_{tag}"):
            e = torch.randn(NB, t, V, 6 * ci, device=dev)
            nchunk = K.pick_nchunk(NB, t, V, ci)
            ms = timeit(lambda: K.joint_gram(e, e, groups=3, offa=0, stridea=2 * ci, offb=ci, strideb=2 * ci, width=ci, nchunk=nchunk, precision=prec), once)
            report(f"gram_score_{tag}", ms, e.numel() * 4, 3 * 2.0 * rows * V * ci)
            del e
        if want(f"gram_dg_{tag}"):
            dz = torch.randn(NB, t, V, 3 * c, device=dev)
            nchunk = K.pick_nchunk(NB, t, V, c)
            ms = timeit(lambda: K.joint_gram(x, dz, groups=3, offa=0, stridea=0, offb=0, strideb=c, width=c, nchunk=nchunk, precision=prec), once)
            report(f"gram_dg_{tag}", ms, act * 4, 3 * 2.0 * rows * V * c)
            del dz
        if want(f"mix_fwd_{tag}") or want(f"mix_bwd_{tag}"):
            g = torch.randn(NB, 3, V, V, device=dev)
            if want(f"mix_fwd_{tag}"):
                ms = timeit(lambda: K.joint_mix(x, g, width=c, mode=K.MIX_AGG_FWD, precision=prec), once)
                report(f"mix_fwd_{tag}", ms, act * 4, 3 * 2.0 * rows * V * c)
            if want(f"mix_bwd_{tag}"):
                dz = torch.randn(NB, t, V, 3 * c, device=dev)
                dx = torch.randn(NB, t, V, c, device=dev)
                ms = timeit(lambda: K.joint_mix(dz, g, width=c, mode=K.MIX_AGG_BWD, out=dx, accumulate=True, precision=prec), once)
                report(f"mix_bwd_{tag}", ms, act * 5, 3 * 2.0 * rows * V * c)
                del dz, dx
        if want(f"mix_score_bwd_{tag}"):
            e = torch.randn(NB, t, V, 6 * ci, device=dev)
            ds = torch.randn(NB, 3, V, V, device=dev)
            ms = timeit(lambda: K.joint_mix(e, ds, width=ci, mode=K.MIX_SCORE_BWD, precision=prec), once)
            report(f"mix_score_bwd_{tag}", ms, e.numel() * 8, 6 * 2.0 * rows * V * ci)
            del e, ds
        for nm, cin, cout, taps in (("emb", c, 6 * ci, 1), ("proj", 3 * c, c, 1), ("dproj", c, 3 * c, 1), ("tconv", c, c, 9)):
            if want(f"conv_{nm}_{tag}"):
                xi = torch.randn(NB, t, V, cin, device=dev)
                w = torch.randn(cout, taps, cin, device=dev) * 0.05
                b = torch.randn(cout, device=dev)
                ms = timeit(lambda: K.conv_fwd(xi, w, b, pad=(taps - 1) // 2, precision=prec), once)
                report(f"conv_{nm}_{tag}", ms, rows * (cin + cout) * 4, 2.0 * rows * cin * cout * taps)
                del xi
            if want(f"convstats_{nm}_{tag}") and nm in ("proj", "tconv"):
                xi = torch.randn(NB, t, V, cin, device=dev)
                w = torch.randn(cout, taps, cin, device=dev) * 0.05
                b = torch.randn(cout, device=dev)
                ms = timeit(lambda: K.conv_fwd_stats(xi, w, b, pad=(taps - 1) // 2, precision=prec), once)
                report(f"convstats_{nm}_{tag}", ms, rows * (cin + cout) * 4, 2.0 * rows * cin * cout * taps)
                del xi
            if want(f"wgradpre_{nm}_{tag}") and cin % 64 == 0 and cout % 64 == 0:      # operands arrive as bf16 pieces
                xs = K.bf16_split(torch.randn(NB, t, V, cin, device=dev))
                dys = K.bf16_split(torch.randn(NB, t, V, cout, device=dev))
                ms = timeit(lambda: K.conv_wgrad_presplit(dys, xs, (NB, t, V), taps=taps, pad=(taps - 1) // 2), once)
                report(f"wgradpre_{nm}_{tag}", ms, rows * (cin + cout) * 4, 2.0 * rows * cin * cout * taps)
                del xs, dys
            if want(f"wgrad_{nm}_{tag}"):
                xi = torch.randn(NB, t, V, cin, device=dev)
                dy = torch.randn(NB, t, V, cout, device=dev)
                ms = timeit(lambda: K.conv_wgrad(dy, xi, taps=taps, pad=(taps - 1) // 2, want_bias=False, precision=prec), once)
                report(f"wgrad_{nm}_{tag}", ms, rows * (cin + cout) * 4, 2.0 * rows * cin * cout * taps)
                del xi, dy
        if want(f"bn_{tag}"):
            # every operand is its own buffer: aliased operands (res = x, dout = y = mask) are served from L2 / one DRAM
            # stream and overstate the achieved bandwidth (VERDICT r1 item 7)
            gamma, beta = torch.ones(c, device=dev), torch.zeros(c, device=dev)
            rm, rv = torch.zeros(c, device=dev), torch.ones(c, device=dev)
            res, dout, msk = (torch.randn_like(x) for _ in range(3))
            ms = timeit(lambda: K.bn_stats(x, gamma, beta, rm, rv, None, 0.1, 1e-5, True), once)
            report(f"bn_stats_{tag}", ms, act, 0)
            sc, sh, mean, invstd = K.bn_stats(x, gamma, beta, rm, rv, None, 0.1, 1e-5, True)
            ms = timeit(lambda: K.bn_apply(x, sc, sh, res_mode=K.RES_TENSOR, res=res, relu=True), once)
            report(f"bn_apply_res_{tag}", ms, act * 3, 0)
            ms = timeit(lambda: K.bn_bwd(dout, msk, x, mean, invstd, gamma), once)
            report(f"bn_bwd_{tag}", ms, act * 7, 0)              # two passes over (dout, mask, y) + dy
            _, bits, _ = K.bn_apply(x, sc, sh, res_mode=K.RES_TENSOR, res=res, relu=True, want_mask=True)
            ms = timeit(lambda: K.bn_apply(x, sc, sh, res_mode=K.RES_TENSOR, res=res, relu=True, want_mask=True), once)
            report(f"bn_apply_res_mask_{tag}", ms, act * 3, 0)
            ms = timeit(lambda: K.bn_bwd(dout, None, x, mean, invstd, gamma, mask_bits=bits), once)
            report(f"bn_bwd_bits_{tag}", ms, act * 5, 0)         # two passes over (dout, y) + dy (+ 1/32 for the bits)
            if bits is not None:                                 # two BatchNorms over one upstream gradient (agcn_bn_bwd_bits_dual)
                ms = timeit(lambda: K.bn_bwd_dual(dout, (x, mean, invstd, gamma), (res, mean, invstd, gamma), mask_bits=bits), once)
                report(f"bn_bwd_dual_{tag}", ms, act * 8, 0)     # two passes over (dout, y_a, y_b) + dy_a + dy_b
            del res, dout, msk
        del x
        torch.cuda.empty_cache()
    if want("first_unit"):
        t = 300
        rows = NB * t * V
        for cin, cout in ((3, 96), (9, 64), (3, 64)):
            xs = torch.randn(NB, t, V, cin, device=dev)
            dy = torch.randn(NB, t, V, cout, device=dev)
            w = torch.randn(cout, 1, cin, device=dev)
            ms = timeit(lambda: K.conv_wgrad(dy, xs, want_bias=True, precision=prec), once)
            report(f"first_unit_wgrad_{cin}_{cout}", ms, rows * (cin + cout) * 4, 2.0 * rows * cin * cout)
            ms = timeit(lambda: K.conv_fwd(xs, w, None, precision=prec), once)
            report(f"first_unit_conv_{cin}_{cout}", ms, rows * (cin + cout) * 4, 2.0 * rows * cin * cout)
    if want("res_dgrad"):
        for cin, cout, t_out in ((256, 128, 150), (128, 64, 300)):      # input gradient of the strided 1x1 residual conv
            t_in = t_out // 2
            dy = torch.randn(NB, t_in, V, cin, device=dev)
            w = torch.randn(cout, 1, cin, device=dev) * 0.05
            ms = timeit(lambda: K.conv_fwd(dy, w, None, t_out=t_out, stride=2, pad=0, transposed=True, precision=prec), once)
            report(f"res_dgrad_{cin}_{cout}", ms, NB * V * (t_in * cin + t_out * cout) * 4, 2.0 * NB * t_in * V * cin * cout)
    if want("skinny"):
        t = 300
        rows = NB * t * V
        for cin, cout in ((64, 3), (96, 3), (64, 9)):
            xi = torch.randn(NB, t, V, cin, device=dev)
            w = torch.randn(cout, 1, cin, device=dev)
            ms = timeit(lambda: K.conv_fwd(xi, w, None, precision=prec), once)
            report(f"skinny_out_{cin}_{cout}", ms, rows * (cin + cout) * 4, 2.0 * rows * cin * cout)
            dy = torch.randn(NB, t, V, cin, device=dev)
            xs = torch.randn(NB, t, V, cout, device=dev)
            ms = timeit(lambda: K.conv_wgrad(dy, xs, want_bias=True, precision=prec), once)
            report(f"skinny_wgrad_{cout}_{cin}", ms, rows * (cin + cout) * 4, 2.0 * rows * cin * cout)


if __name__ == "__main__":
    main()
