"""Tensor-level wrappers over the C ABI (one function per entry point of include/agcn_b200.h).

Every function takes/returns fp32 CUDA tensors in the channels-last activation layout
``[nb, t, v, c]`` and launches on ``torch.cuda.current_stream()``.  PyTorch only provides the
device memory and the stream.  ``oracle/stages.py`` restates each function in plain torch for
the tests; nothing here falls back to it.
"""
import threading
from typing import Optional, Tuple

import torch

from . import capi
from .capi import (MIX_AGG_BWD, MIX_AGG_FWD, MIX_SCORE_BWD, PREC_BF16X3, PREC_FP32, PREC_FP32_FFMA, PREC_TF32, RES_AFFINE,  # noqa: F401
                   RES_NONE, RES_TENSOR)

NUM_SMS = 148


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


_tl = threading.local()          # device of the tensors of the call being assembled (forward and backward run on different host threads)


def _same_device(t):
    dev = getattr(_tl, "dev", None)
    if dev is None:
        _tl.dev = t.device
    elif t.device != dev:
        _tl.dev = None
        raise RuntimeError(f"fusion_gcn_b200: tensors of one call live on different devices ({dev} and {t.device})")


def _check_bf16(*tensors):
    """Split operands (bf16 pieces [2, rows, C]): CUDA, contiguous, on the call's device."""
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda or t.dtype != torch.bfloat16 or not t.is_contiguous() or t.dim() != 3 or t.shape[0] != 2:
            _tl.dev = None
            raise RuntimeError("contiguous CUDA bf16 tensor of shape [2, rows, C] expected")
        _same_device(t)


def _check(*tensors):
    for t in tensors:
        if t is None:
            continue
        if t.is_cuda:
            _same_device(t)
        if not t.is_cuda:
            _tl.dev = None
            raise RuntimeError("fusion_gcn_b200 kernels need CUDA tensors (there is no CPU path)")
        if t.dtype != torch.float32:
            _tl.dev = None
            raise RuntimeError(f"fp32 tensor expected, got {t.dtype}")
        if not t.is_contiguous():
            _tl.dev = None
            raise RuntimeError("contiguous tensor expected")


def _check_strided(*tensors):
    """Device / dtype check for tensors addressed through a rowmap (need not be contiguous)."""
    for t in tensors:
        if t is None:
            continue
        if t.is_cuda:
            _same_device(t)
        if not t.is_cuda:
            _tl.dev = None
            raise RuntimeError("fusion_gcn_b200 kernels need CUDA tensors (there is no CPU path)")
        if t.dtype != torch.float32:
            _tl.dev = None
            raise RuntimeError(f"fp32 tensor expected, got {t.dtype}")


def _stream():
    """Current stream of the device the call's tensors live on (not of the current device: the two differ when a caller
    drives cuda:1 tensors while cuda:0 is current)."""
    return torch.cuda.current_stream(getattr(_tl, "dev", None)).cuda_stream


_timing = None            # (set of entry-point names, list of (key, start_event, end_event)) while bench.py is timing


def start_timing(names):
    """Record a CUDA-event pair on the launching stream around every call of the named conv entry points."""
    global _timing
    _timing = (set(names), [])


def stop_timing():
    """-> {(name, signature): (total_ms, launches, algorithmic_flops, algorithmic_bytes)}; synchronises the device.
    ``signature`` is the tuple of shape arguments of the call; flops / bytes are per launch (DESIGN.md section 4)."""
    global _timing
    if _timing is None:
        return {}
    _, records = _timing
    _timing = None
    torch.cuda.synchronize()
    out = {}
    for key, work, e0, e1 in records:
        tot, cnt = out.get(key, (0.0, 0, 0.0, 0.0))[:2]
        out[key] = (tot + e0.elapsed_time(e1), cnt + 1, work[0], work[1])
    return out


def _call(name, *args, sig=None, work=(0.0, 0.0), alias=None):
    """``sig``: shape signature of the call, ``work``: (algorithmic FLOPs, algorithmic bytes) of one launch -- used only while
    bench.py is timing (CUDA events on the launching stream around the C-ABI call)."""
    capi.launch_count += 1
    fn = getattr(capi.lib(), name)
    dev = getattr(_tl, "dev", None)
    if dev is not None and dev.index is not None and dev.index != torch.cuda.current_device():
        # the C ABI launches on the CURRENT device and never changes it: make the tensors' device current for the call
        _tl.dev = None
        capi.launch_count -= 1
        with torch.cuda.device(dev):
            return _call(name, *args, sig=sig, work=work, alias=alias)
    _tl.dev = None                 # the next call collects its own device
    if _timing is not None and (name in _timing[0] or "*" in _timing[0]):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = fn(*args)
        e1.record()
        _timing[1].append(((alias or name, sig), work, e0, e1))
    else:
        rc = fn(*args)
    capi.check(rc, name)


# ----------------------------------------------------------------------------- dense contractions
def conv_fwd(x, w, bias=None, *, t_out=None, stride=1, pad=0, transposed=False, out=None, accumulate=False,
             precision=PREC_FP32):
    """x [nb,t_in,v,cin], w [cout,taps,cin] -> y [nb,t_out,v,cout]; see agcn_conv_fwd."""
    nb, t_in, v, cin = x.shape
    cout, taps, cin_w = w.shape
    if cin_w != cin:
        raise RuntimeError(f"conv_fwd: weight expects {cin_w} input channels, tensor has {cin}")
    if t_out is None:
        t_out = t_in
    if out is None:
        if accumulate:
            raise RuntimeError("conv_fwd: accumulate needs an output tensor")
        out = torch.empty((nb, t_out, v, cout), device=x.device, dtype=torch.float32)
    elif tuple(out.shape) != (nb, t_out, v, cout):
        raise RuntimeError(f"conv_fwd: out has shape {tuple(out.shape)}, expected {(nb, t_out, v, cout)}")
    _check(x, w, bias, out)
    ws_bytes = capi.lib().agcn_conv_fwd_workspace_bytes(cin, cout, taps, precision)
    ws = torch.empty((ws_bytes + 3) // 4, device=x.device, dtype=torch.float32) if ws_bytes else None
    rows = nb * t_out * v
    _call("agcn_conv_fwd", _ptr(x), _ptr(w), _ptr(bias), _ptr(out), nb, t_in, t_out, v, cin, cout, taps, stride, pad,
          int(transposed), int(accumulate), precision, _ptr(ws), ws_bytes, _stream(),
          sig=(nb, t_in, t_out, v, cin, cout, taps, stride, int(transposed), int(accumulate)),
          work=(2.0 * rows * cin * cout * taps, 4.0 * (x.numel() + rows * cout * (2 if accumulate else 1))))
    return out


def conv_fwd_post(x, w, bias=None, *, scale=None, shift=None, res=None, relu=False, t_out=None, stride=1, pad=0, precision=PREC_FP32):
    """Eval-mode convolution with its tail fused: act(scale * (conv(x, w) + bias) + shift + res); see agcn_conv_fwd_post."""
    nb, t_in, v, cin = x.shape
    cout, taps, cin_w = w.shape
    if cin_w != cin:
        raise RuntimeError(f"conv_fwd_post: weight expects {cin_w} input channels, tensor has {cin}")
    if t_out is None:
        t_out = t_in
    out = torch.empty((nb, t_out, v, cout), device=x.device, dtype=torch.float32)
    if res is not None and tuple(res.shape) != tuple(out.shape):
        raise RuntimeError(f"conv_fwd_post: residual has shape {tuple(res.shape)}, expected {tuple(out.shape)}")
    _check(x, w, bias, scale, shift, res, out)
    ws_bytes = capi.lib().agcn_conv_fwd_workspace_bytes(cin, cout, taps, precision)
    ws = torch.empty((ws_bytes + 3) // 4, device=x.device, dtype=torch.float32) if ws_bytes else None
    rows = nb * t_out * v
    _call("agcn_conv_fwd_post", _ptr(x), _ptr(w), _ptr(bias), _ptr(scale), _ptr(shift), _ptr(res), int(relu), _ptr(out),
          nb, t_in, t_out, v, cin, cout, taps, stride, pad, precision, _ptr(ws), ws_bytes, _stream(),
          sig=(nb, t_in, t_out, v, cin, cout, taps, stride, 2, int(res is not None)),
          work=(2.0 * rows * cin * cout * taps, 4.0 * (x.numel() + rows * cout * (2 if res is not None else 1))), alias="agcn_conv_fwd")
    return out


def conv_fwd_stats(x, w, bias=None, *, t_out=None, stride=1, pad=0, precision=PREC_FP32):
    """conv_fwd whose epilogue also accumulates the column sums of y for the training-mode BatchNorm that follows
    (agcn_conv_fwd_stats).  -> (y, part) with part [nparts, 4, cout] (shifted sum | shifted sum of squares | pivot | row count per
    partial), or (y, None) when the fused epilogue does not cover the shape (run bn_stats on y then)."""
    import ctypes
    nb, t_in, v, cin = x.shape
    cout, taps, cin_w = w.shape
    if cin_w != cin:
        raise RuntimeError(f"conv_fwd_stats: weight expects {cin_w} input channels, tensor has {cin}")
    if t_out is None:
        t_out = t_in
    out = torch.empty((nb, t_out, v, cout), device=x.device, dtype=torch.float32)
    _check(x, w, bias, out)
    L = capi.lib()
    ws_bytes = L.agcn_conv_fwd_workspace_bytes(cin, cout, taps, precision)
    ws = torch.empty((ws_bytes + 3) // 4, device=x.device, dtype=torch.float32) if ws_bytes else None
    part_bytes = L.agcn_conv_fwd_stats_bytes(cout)
    part = torch.empty(part_bytes // 4, device=x.device, dtype=torch.float32)
    nparts = ctypes.c_int(0)
    rows = nb * t_out * v
    _call("agcn_conv_fwd_stats", _ptr(x), _ptr(w), _ptr(bias), _ptr(out), nb, t_in, t_out, v, cin, cout, taps, stride, pad,
          precision, _ptr(ws), ws_bytes, _ptr(part), part_bytes, ctypes.byref(nparts), _stream(),
          sig=(nb, t_in, t_out, v, cin, cout, taps, stride, 0, 0),
          work=(2.0 * rows * cin * cout * taps, 4.0 * (x.numel() + rows * cout)), alias="agcn_conv_fwd")
    if nparts.value == 0:
        return out, None
    return out, part[:nparts.value * 4 * cout].view(nparts.value, 4, cout)


def bn_finalize(part, rows, gamma, beta, running_mean, running_var, nbt, momentum, eps):
    """Training-mode BatchNorm parameters from the partials of conv_fwd_stats: -> scale, shift, save_mean, save_invstd."""
    nparts, _, c = part.shape
    scale = torch.empty((4, c), device=part.device, dtype=torch.float32)
    _check(part, gamma, beta, running_mean, running_var)
    if nbt is not None and nbt.dtype != torch.int64:
        raise RuntimeError("num_batches_tracked must be int64")
    _call("agcn_bn_finalize", _ptr(part), nparts, int(rows), c, _ptr(gamma), _ptr(beta), _ptr(running_mean), _ptr(running_var),
          _ptr(nbt), float(momentum), float(eps), scale[0].data_ptr(), scale[1].data_ptr(), scale[2].data_ptr(), scale[3].data_ptr(),
          0, None, _stream(), sig=(nparts, c), work=(0.0, 0.0))
    return scale[0], scale[1], scale[2], scale[3]


def bn_moments(part, rows):
    """Phase 1 of a synchronised BatchNorm's statistics: the partials of this rank (conv_fwd_stats / bn_stats_partials) reduced to
    fp64 moments [2c + 1] = sum x per channel | sum x^2 per channel | rows.  The moments of all ranks add up (all-reduce, sum);
    bn_finalize_moments turns the total into the BatchNorm parameters."""
    nparts, _, c = part.shape
    _check(part)
    moments = torch.empty((2 * c + 1,), device=part.device, dtype=torch.float64)
    _call("agcn_bn_finalize", _ptr(part), nparts, int(rows), c, None, None, None, None, None, 0.0, 0.0, None, None, None, None,
          1, moments.data_ptr(), _stream(), sig=(nparts, c, 1), work=(0.0, 0.0))
    return moments


def bn_finalize_moments(moments, gamma, beta, running_mean, running_var, nbt, momentum, eps):
    """Phase 2: scale, shift, save_mean, save_invstd from moments summed over the ranks (bn_moments); the running statistics take
    the unbiased variance over the count in moments[-1], and ``nbt`` is incremented."""
    c = (moments.shape[0] - 1) // 2
    if moments.dtype != torch.float64 or not moments.is_cuda or not moments.is_contiguous() or moments.shape != (2 * c + 1,):
        raise RuntimeError("bn_finalize_moments: moments must be the contiguous CUDA float64 tensor [2c + 1] of bn_moments")
    _same_device(moments)
    scale = torch.empty((4, c), device=moments.device, dtype=torch.float32)
    _check(gamma, beta, running_mean, running_var)
    if nbt is not None and nbt.dtype != torch.int64:
        raise RuntimeError("num_batches_tracked must be int64")
    _call("agcn_bn_finalize", None, 0, 0, c, _ptr(gamma), _ptr(beta), _ptr(running_mean), _ptr(running_var),
          _ptr(nbt), float(momentum), float(eps), scale[0].data_ptr(), scale[1].data_ptr(), scale[2].data_ptr(), scale[3].data_ptr(),
          2, moments.data_ptr(), _stream(), sig=(0, c, 2), work=(0.0, 0.0))
    return scale[0], scale[1], scale[2], scale[3]


def conv_wgrad(dy, x, *, taps=1, stride=1, pad=0, want_bias=True, precision=PREC_FP32):
    """dy [nb,t_out,v,cout], x [nb,t_in,v,cin] -> dw [cout,taps,cin], dbias [cout] | None."""
    nb, t_out, v, cout = dy.shape
    nb2, t_in, v2, cin = x.shape
    if nb2 != nb or v2 != v:
        raise RuntimeError("conv_wgrad: dy / x batch or joint mismatch")
    _check(dy, x)
    L = capi.lib()
    ws_bytes = L.agcn_conv_wgrad_workspace_bytes(nb, t_in, t_out, v, cin, cout, taps)
    ws = torch.empty((ws_bytes + 3) // 4, device=x.device, dtype=torch.float32)
    dw = torch.empty((cout, taps, cin), device=x.device, dtype=torch.float32)
    db = torch.empty((cout,), device=x.device, dtype=torch.float32) if want_bias else None
    _call("agcn_conv_wgrad", _ptr(dy), _ptr(x), _ptr(dw), _ptr(db), nb, t_in, t_out, v, cin, cout, taps, stride, pad,
          _ptr(ws), ws_bytes, precision, _stream(), sig=(nb, t_in, t_out, v, cin, cout, taps, stride),
          work=(2.0 * nb * t_out * v * cin * cout * taps, 4.0 * (x.numel() + dy.numel())))
    return dw, db


def bf16_split(x):
    """[..., C] fp32 -> [2, rows, C] bf16 pieces (h = bf16(x), m = bf16(x - h), round to nearest ties away like the kernels).
    Test / reference helper: in the model the pieces come out of the BatchNorm kernels (bn_apply / bn_bwd ``want_split``)."""
    flat = x.reshape(-1, x.shape[-1]).contiguous()
    hb = ((flat.view(torch.int32) + 0x8000) & -65536)
    h = hb.view(torch.float32)
    mb = ((flat - h).view(torch.int32) + 0x8000) & -65536
    return torch.stack([(hb >> 16).to(torch.int16), (mb >> 16).to(torch.int16)]).view(torch.bfloat16)


def conv_wgrad_presplit(dy_split, x_split, shape, *, taps=1, stride=1, pad=0):
    """Weight gradient from pre-split operands (bf16 [2, rows, C] each); shape = (nb, t_in, v) of the convolution's input.
    -> dw [cout, taps, cin], or None when the kernel does not cover the channel counts (call conv_wgrad on the fp32 tensors then)."""
    nb, t_in, v = shape
    t_out = (t_in + 2 * pad - taps) // stride + 1
    cout, cin = dy_split.shape[-1], x_split.shape[-1]
    if cin % 64 or cout % 64:
        return None
    if dy_split.shape[1] != nb * t_out * v or x_split.shape[1] != nb * t_in * v:
        raise RuntimeError("conv_wgrad_presplit: operand rows do not match the shape")
    _check_bf16(dy_split, x_split)
    L = capi.lib()
    ws_bytes = L.agcn_conv_wgrad_workspace_bytes(nb, t_in, t_out, v, cin, cout, taps)
    ws = torch.empty((ws_bytes + 3) // 4, device=x_split.device, dtype=torch.float32)
    dw = torch.empty((cout, taps, cin), device=x_split.device, dtype=torch.float32)
    _call("agcn_conv_wgrad_presplit", _ptr(dy_split), _ptr(x_split), _ptr(dw), nb, t_in, t_out, v, cin, cout, taps, stride, pad,
          _ptr(ws), ws_bytes, _stream(),
          sig=(nb, t_in, t_out, v, cin, cout, taps, stride), work=(2.0 * nb * t_out * v * cin * cout * taps, 4.0 * nb * v * (t_in * cin + t_out * cout)),
          alias="agcn_conv_wgrad")
    return dw


# ----------------------------------------------------------------------------- V x V attention
def pick_nchunk(nb: int, t: int, v: int = 0, width: int = 0) -> int:
    """Chunks of the t axis of the joint-gram reduction (one CTA per (sample, chunk)).  Shapes the tensor-core kernel takes
    (3*v <= 80, width 16 or a multiple of 32) want ONE resident wave of long-running CTAs (<= 148); the FFMA kernel wants
    about four waves of short ones."""
    if v > 32:
        return 1          # large graphs (1-D graph convolution): batched GEMM over the node axis, one chunk
    if v and 3 * v <= 80 and (width == 16 or (width > 0 and width % 32 == 0)):
        return max(1, min(NUM_SMS // max(nb, 1), max(1, t // 8)))
    n = max(1, min((4 * NUM_SMS + nb - 1) // nb, max(1, t // 4)))
    return min(n, t)


def joint_gram(a, b, *, groups, offa, stridea, offb, strideb, width, nchunk, precision=PREC_FP32):
    nb, t, v, lda = a.shape
    ldb = b.shape[3]
    _check(a, b)
    out = torch.empty((nb, nchunk, groups, v, v), device=a.device, dtype=torch.float32)
    same = a.data_ptr() == b.data_ptr()
    _call("agcn_joint_gram", _ptr(a), _ptr(b), _ptr(out), nb, t, v, lda, ldb, groups, offa, stridea, offb, strideb, width,
          nchunk, precision, _stream(), sig=(nb, t, v, lda, ldb, groups, width, nchunk),
          work=(2.0 * nb * t * groups * v * v * width, 4.0 * (a.numel() + (0 if same else b.numel()))))
    return out


def attention_fwd(s_part, adj_a, adj_b, scale: float) -> Tuple[torch.Tensor, torch.Tensor]:
    nb, nchunk, groups, v, _ = s_part.shape
    _check(s_part, adj_a, adj_b)
    p = torch.empty((nb, groups, v, v), device=s_part.device, dtype=torch.float32)
    g = torch.empty_like(p)
    _call("agcn_attention_fwd", _ptr(s_part), _ptr(adj_a), _ptr(adj_b), _ptr(p), _ptr(g), nb, nchunk, groups, v, float(scale),
          _stream(), sig=(nb, nchunk, groups, v), work=(0.0, 4.0 * (s_part.numel() + 2 * p.numel())))
    return p, g


def attention_bwd(dg_part, p, scale: float) -> Tuple[torch.Tensor, torch.Tensor]:
    nb, nchunk, groups, v, _ = dg_part.shape
    _check(dg_part, p)
    dg_sum = torch.empty_like(p)
    ds = torch.empty_like(p)
    dadj_b = torch.empty((groups, v, v), device=p.device, dtype=torch.float32)
    _call("agcn_attention_bwd", _ptr(dg_part), _ptr(p), _ptr(dg_sum), _ptr(ds), _ptr(dadj_b), nb, nchunk, groups, v,
          float(scale), _stream(), sig=(nb, nchunk, groups, v), work=(0.0, 4.0 * (dg_part.numel() + 3 * p.numel())))
    return ds, dadj_b


def joint_mix(inp, mats, *, width, mode, out=None, accumulate=False, precision=PREC_FP32):
    nb, t, v, ldin = inp.shape
    ldout = {MIX_AGG_FWD: 3 * width, MIX_AGG_BWD: width, MIX_SCORE_BWD: 6 * width}[mode]
    if out is None:
        if accumulate:
            raise RuntimeError("joint_mix: accumulate needs an output tensor")
        out = torch.empty((nb, t, v, ldout), device=inp.device, dtype=torch.float32)
    _check(inp, mats, out)
    terms = {MIX_AGG_FWD: 3, MIX_AGG_BWD: 3, MIX_SCORE_BWD: 6}[mode]
    ws_bytes = capi.lib().agcn_joint_mix_workspace_bytes(nb) if precision != PREC_FP32_FFMA else 0
    ws = torch.empty((ws_bytes + 3) // 4, device=inp.device, dtype=torch.float32) if ws_bytes else None
    _call("agcn_joint_mix", _ptr(inp), _ptr(mats), _ptr(out), nb, t, v, ldin, ldout, width, mode, int(accumulate), precision,
          _ptr(ws), ws_bytes, _stream(),
          sig=(nb, t, v, ldin, ldout, width, mode, int(accumulate)),
          work=(2.0 * nb * t * terms * v * v * width, 4.0 * (inp.numel() + out.numel() * (2 if accumulate else 1))))
    return out


def joint_mix_score_bwd(e, ds, *, width, precision=PREC_FP32):
    """de = joint_mix(e, ds, mode=MIX_SCORE_BWD) together with the column sums of de over all (nb, t, v) rows -- the bias gradient of
    the theta / phi convolutions -- out of the same epilogue (agcn_joint_mix_score_bwd_colsum).  -> (de, colsum [6 * width]), or
    (de, None) for shapes the fused epilogue does not cover (sum the columns separately then)."""
    nb, t, v, ld = e.shape
    fused = (precision != PREC_FP32_FFMA and v <= 32 and ld == 6 * width and 6 * width <= 384 and (width == 16 or width % 32 == 0))
    if not fused:
        return joint_mix(e, ds, width=width, mode=MIX_SCORE_BWD, precision=precision), None
    out = torch.empty_like(e)
    colsum = torch.empty((ld,), device=e.device, dtype=torch.float32)
    _check(e, ds, out)
    ws_bytes = capi.lib().agcn_joint_mix_score_bwd_colsum_workspace_bytes(nb, width)
    ws = torch.empty((ws_bytes + 3) // 4, device=e.device, dtype=torch.float32)
    _call("agcn_joint_mix_score_bwd_colsum", _ptr(e), _ptr(ds), _ptr(out), _ptr(colsum), nb, t, v, width, precision, _ptr(ws), ws_bytes, _stream(),
          sig=(nb, t, v, ld, ld, width, MIX_SCORE_BWD, 0), work=(2.0 * nb * t * 6 * v * v * width, 4.0 * (e.numel() + out.numel())),
          alias="agcn_joint_mix")
    return out, colsum


# ----------------------------------------------------------------------------- batch norm
def _rowmap(x, rowmap):
    """rowmap = (outer, inner, outer_stride, channels) or None for a plain [rows, channels] view."""
    if rowmap is not None:
        return rowmap
    c = x.shape[-1]
    return (1, x.numel() // c, 0, c)


def _bn_ws(channels, device):
    nbytes = capi.lib().agcn_bn_workspace_bytes(channels)
    return torch.empty((nbytes + 3) // 4, device=device, dtype=torch.float32), nbytes


def bn_stats(x, gamma, beta, running_mean, running_var, nbt, momentum, eps, training, rowmap=None):
    """-> scale, shift, save_mean, save_invstd (each [channels]); running statistics updated in place."""
    outer, inner, ostride, c = _rowmap(x, rowmap)
    scale = torch.empty((4, c), device=x.device, dtype=torch.float32)
    ws, nbytes = _bn_ws(c, x.device)
    _check(gamma, beta, running_mean, running_var)
    _check_strided(x)
    if nbt is not None and nbt.dtype != torch.int64:
        raise RuntimeError("num_batches_tracked must be int64")
    _call("agcn_bn_stats", x.data_ptr(), outer, inner, ostride, c, _ptr(gamma), _ptr(beta), _ptr(running_mean), _ptr(running_var),
          _ptr(nbt), float(momentum), float(eps), int(training), scale[0].data_ptr(), scale[1].data_ptr(),
          scale[2].data_ptr(), scale[3].data_ptr(), _ptr(ws), nbytes, _stream(),
          sig=(outer, inner, c, int(training)), work=(0.0, 4.0 * outer * inner * c if training else 0.0))
    return scale[0], scale[1], scale[2], scale[3]


def bn_stats_partials(x, rowmap=None):
    """Column statistics of x as mergeable partials [nparts, 4, c] (shifted sum | shifted sum of squares | pivot | row count per row
    partition, the layout of conv_fwd_stats): what bn_finalize, or bn_moments in a synchronised BatchNorm, reduces."""
    import ctypes
    outer, inner, ostride, c = _rowmap(x, rowmap)
    ws, nbytes = _bn_ws(c, x.device)
    _check_strided(x)
    part_bytes = capi.lib().agcn_bn_stats_partials_bytes(c)
    part = torch.empty(part_bytes // 4, device=x.device, dtype=torch.float32)
    nparts = ctypes.c_int(0)
    _call("agcn_bn_stats_partials", x.data_ptr(), outer, inner, ostride, c, part.data_ptr(), part_bytes, ctypes.byref(nparts),
          _ptr(ws), nbytes, _stream(), sig=(outer, inner, c), work=(0.0, 4.0 * outer * inner * c))
    return part[:nparts.value * 4 * c].view(nparts.value, 4, c)


def bn_apply(y, scale, shift, *, res_mode=RES_NONE, res=None, scale2=None, shift2=None, relu=False, rowmap=None, out=None,
             want_mask=False, want_split=False):
    """out = act(scale*y + shift + R) -> (out, bits | None, split | None).  ``want_mask``: also the ReLU mask (out > 0) as one bit
    per element (int32 words) for bn_bwd(mask_bits=...), None when the layout is not supported.  ``want_split`` (with want_mask):
    also ``out`` as bf16 pieces [2, rows, c] for conv_wgrad_presplit, None when there is no bit mask or c is not a multiple of 64."""
    outer, inner, ostride, c = _rowmap(y, rowmap)
    if out is None:
        out = torch.empty_like(y)
    _check_strided(y, res, out)
    _check(scale, shift, scale2, shift2)
    bits = split = None
    if want_mask and y.is_contiguous() and out.is_contiguous() and (res is None or res.is_contiguous()):
        words = capi.lib().agcn_bn_mask_words(outer, inner, c)
        if words:
            bits = torch.empty(words, device=y.device, dtype=torch.int32)
            if want_split and c % 64 == 0:
                split = torch.empty((2, inner, c), device=y.device, dtype=torch.bfloat16)
    _call("agcn_bn_apply", y.data_ptr(), _ptr(scale), _ptr(shift), res_mode, _ptr(res), _ptr(scale2), _ptr(shift2), int(relu),
          out.data_ptr(), _ptr(bits), _ptr(split), outer, inner, ostride, c, _stream(),
          sig=(outer, inner, c, res_mode, int(relu), int(bits is not None), int(split is not None)),
          work=(0.0, 4.0 * outer * inner * c * (2 if res_mode == RES_NONE else 3) + (4.0 * inner * c if split is not None else 0.0)))
    return out, bits, split


def bn_bwd(dout, mask_out, y, save_mean, save_invstd, gamma, *, want_dy=True, dy=None, dres=None, dres_accumulate=False,
           rowmap=None, mask_bits=None, pool_rows=0, frozen=False, want_split=False, sync=None):
    """-> (dy | None, dgamma, dbeta, dy_split | None); optionally writes / accumulates the masked gradient into ``dres``.
    ``dy`` may be a preallocated tensor addressed with the same rowmap as ``y``.  ``mask_bits`` (from bn_apply(want_mask=True))
    replaces the fp32 tensor ``mask_out`` as the ReLU mask.  ``pool_rows`` > 0 (with mask_bits): ``dout`` is the gradient of the
    fused mean pool, [groups, c], broadcast over the pool_rows rows of each group.  ``frozen``: the statistics are constants
    (eval-mode BatchNorm).  ``want_split``: dy also as bf16 pieces [2, rows, c] for conv_wgrad_presplit, None when there is no bit
    mask or c is not a multiple of 64.  ``sync`` (distributed.SyncBatchNorm, ignored when frozen): the statistics were taken over all
    ranks, so the two column sums are all-reduced between the sum pass (phase 1) and the apply pass (phase 2); dgamma / dbeta stay
    this rank's own sums.  The rows of all ranks: ``sync.global_rows`` when the sync object has one, a CUDA float64 scalar -- the
    count the forward's all-reduced moments carry (bn_moments), right for shards of any size; otherwise rows x sync.world (equal
    shards)."""
    outer, inner, ostride, c = _rowmap(y, rowmap)
    if want_dy and dy is None:
        dy = torch.empty_like(y)
    _check_strided(dout, mask_out, y, dy, dres)
    _check(save_mean, save_invstd, gamma)
    if pool_rows and frozen:
        raise RuntimeError("bn_bwd: the pooled tail is a training-mode path")
    global_rows = getattr(sync, "global_rows", None) if (sync is not None and not frozen) else None
    if global_rows is not None and (global_rows.dtype != torch.float64 or not global_rows.is_cuda or global_rows.numel() != 1):
        raise RuntimeError("bn_bwd: sync.global_rows must be a CUDA float64 tensor with one element")
    if mask_bits is not None:
        if mask_bits.dtype != torch.int32 or not mask_bits.is_cuda:
            raise RuntimeError("bn_bwd: mask_bits must be the int32 CUDA tensor returned by bn_apply(want_mask=True)")
        mask_out = None                 # the bits replace the tensor mask
    if mask_bits is not None or pool_rows:
        _check(dout, y, dy, dres)
    dy_split = torch.empty((2, inner, c), device=y.device, dtype=torch.bfloat16) if (want_split and dy is not None and mask_bits is not None
                                                                                     and c % 64 == 0) else None
    dgb = torch.empty((2, c), device=y.device, dtype=torch.float32)
    ws, nbytes = _bn_ws(c, y.device)
    mask_kind = 2 if mask_bits is not None else int(mask_out is not None)
    writes = int(dy is not None) + int(dres is not None) * (1 + int(dres_accumulate))
    pieces = int(dy_split is not None)

    def run(phase, planes, sums=None, rows_all=None):
        # planes: the algorithmic bytes of the call in fp32 planes of y
        _call("agcn_bn_bwd", dout.data_ptr(), _ptr(mask_out), _ptr(mask_bits), y.data_ptr(), _ptr(save_mean), _ptr(save_invstd), _ptr(gamma),
              _ptr(dy), _ptr(dy_split), dgb[0].data_ptr(), dgb[1].data_ptr(), _ptr(dres), int(dres_accumulate), int(frozen),
              outer, inner, ostride, c, int(pool_rows), phase, _ptr(sums), _ptr(rows_all), _ptr(ws), nbytes, _stream(),
              sig=(outer, inner, c, mask_kind, int(pool_rows), phase, int(dy is not None), int(dres is not None), int(dres_accumulate), pieces),
              work=(0.0, 4.0 * outer * inner * c * planes))

    if sync is not None and not frozen:
        reads = 2 + (2.0 / 32 if mask_bits is not None else int(mask_out is not None))
        run(1, reads)
        if dy is not None or dres is not None:
            sums = sync.all_reduce(torch.stack([dgb[1], dgb[0]]))             # (sum g | sum g xhat) over all ranks
            if global_rows is None:
                global_rows = torch.full((1,), float(outer) * inner * sync.world, device=y.device, dtype=torch.float64)
            run(2, reads + writes + pieces, sums, global_rows)
    elif pool_rows:
        run(0, 2 + 2.0 / 32 + writes)                 # y and the bits in both passes; the pooled gradient is negligible
    else:
        # two passes over (dout, y[, mask]); the second writes dy [and its pieces, and dres, read first when accumulating]
        run(0, 2 * (2 + (1.0 / 32 if mask_bits is not None else int(mask_out is not None))) + writes + pieces)
    return dy, dgb[0], dgb[1], dy_split


def bn_bwd_dual(dout, a, b, *, mask_out=None, mask_bits=None, frozen=False, want_split=False, pool_rows=0, sync=None):
    """Two BatchNorm backwards over the same upstream gradient and ReLU mask: ``a`` / ``b`` = (y, save_mean, save_invstd, gamma) of
    the two BatchNorms.  -> (dy_a, dgamma_a, dbeta_a, dy_a_split | None, dy_b, dgamma_b, dbeta_b); only BatchNorm A gets bf16 pieces.
    Where agcn_bn_bwd_bits_dual covers the call (bit mask, no pooled gradient, no synchronised statistics, contiguous tensors) the
    masked gradient is read once per pass for both; otherwise this is two bn_bwd calls."""
    ya, mean_a, invstd_a, gamma_a = a
    yb, mean_b, invstd_b, gamma_b = b
    c = ya.shape[-1]
    inner = ya.numel() // c
    if mask_bits is None or pool_rows or (sync is not None and not frozen) or not ya.is_contiguous() or not yb.is_contiguous() \
            or not dout.is_contiguous() or tuple(ya.shape) != tuple(yb.shape) or tuple(dout.shape) != tuple(ya.shape) \
            or capi.lib().agcn_bn_mask_words(1, inner, c) == 0:
        kw = dict(mask_bits=mask_bits, frozen=frozen, pool_rows=pool_rows, sync=sync)
        return bn_bwd(dout, mask_out, *a, want_split=want_split, **kw) + bn_bwd(dout, mask_out, *b, **kw)[:3]
    _check(dout, ya, yb, mean_a, invstd_a, gamma_a, mean_b, invstd_b, gamma_b)
    dya, dyb = torch.empty_like(ya), torch.empty_like(yb)
    split = torch.empty((2, inner, c), device=ya.device, dtype=torch.bfloat16) if (want_split and c % 64 == 0) else None
    dgb = torch.empty((4, c), device=ya.device, dtype=torch.float32)
    one = capi.lib().agcn_bn_workspace_bytes(c)
    ws = torch.empty((2 * one + 3) // 4, device=ya.device, dtype=torch.float32)
    _call("agcn_bn_bwd_bits_dual", dout.data_ptr(), mask_bits.data_ptr(), ya.data_ptr(), _ptr(mean_a), _ptr(invstd_a), _ptr(gamma_a),
          dya.data_ptr(), _ptr(split), dgb[0].data_ptr(), dgb[1].data_ptr(), yb.data_ptr(), _ptr(mean_b), _ptr(invstd_b), _ptr(gamma_b),
          dyb.data_ptr(), dgb[2].data_ptr(), dgb[3].data_ptr(), int(frozen), inner, c, ws.data_ptr(), 2 * one, _stream(),
          sig=(1, inner, c, 3, 2, int(split is not None)), work=(0.0, 4.0 * inner * c * (2 * (3 + 1.0 / 32) + 2 + int(split is not None))),
          alias="agcn_bn_bwd")
    return dya, dgb[0], dgb[1], split, dyb, dgb[2], dgb[3]


def bn_pool_supported(rows: int, channels: int) -> bool:
    """Whether the fused BN-apply + mean-pool tail (agcn_bn_apply_pool, and bn_bwd with pool_rows) covers this layout."""
    return channels % 32 == 0 and capi.lib().agcn_bn_mask_words(1, rows, channels) > 0


def bn_apply_pool(y, scale, shift, *, groups, res_mode=RES_NONE, res=None, scale2=None, shift2=None):
    """pooled[g] = mean over the rows of group g of relu(scale*y + shift + R); the full-size output is never written.
    -> (pooled [groups, c], ReLU mask bits for bn_bwd(pool_rows=...))."""
    c = y.shape[-1]
    rows = y.numel() // c
    if rows % groups:
        raise RuntimeError("bn_apply_pool: rows not divisible by groups")
    _check(y, scale, shift, res, scale2, shift2)
    L = capi.lib()
    bits = torch.empty(L.agcn_bn_mask_words(1, rows, c), device=y.device, dtype=torch.int32)
    pooled = torch.empty((groups, c), device=y.device, dtype=torch.float32)
    ws_bytes = L.agcn_bn_apply_pool_workspace_bytes(groups, c)
    ws = torch.empty(ws_bytes // 4, device=y.device, dtype=torch.float32)
    _call("agcn_bn_apply_pool", _ptr(y), _ptr(scale), _ptr(shift), res_mode, _ptr(res), _ptr(scale2), _ptr(shift2), bits.data_ptr(),
          _ptr(pooled), groups, rows // groups, c, _ptr(ws), ws_bytes, _stream(), sig=(groups, rows // groups, c, res_mode),
          work=(0.0, 4.0 * rows * c * (1 if res_mode == RES_NONE else 2)), alias="agcn_bn_apply")
    return pooled, bits


# ----------------------------------------------------------------------------- pooling
def pool_fwd(x, groups: int):
    c = x.shape[-1]
    rows = x.numel() // c // groups
    _check(x)
    out = torch.empty((groups, c), device=x.device, dtype=torch.float32)
    _call("agcn_pool_fwd", _ptr(x), _ptr(out), groups, rows, c, _stream(), sig=(groups, rows, c), work=(0.0, 4.0 * x.numel()))
    return out


def pool_bwd(dout, shape):
    groups, c = dout.shape
    dx = torch.empty(shape, device=dout.device, dtype=torch.float32)
    rows = dx.numel() // c // groups
    _check(dout)
    _call("agcn_pool_bwd", _ptr(dout), _ptr(dx), groups, rows, c, _stream(), sig=(groups, rows, c), work=(0.0, 4.0 * dx.numel()))
    return dx


# ----------------------------------------------------------------------------- classifier head + loss
def linear_ce_fwd(x, w, bias, labels):
    """-> (loss scalar, logits [n, ncls], dlogits [n, ncls]); see agcn_linear_ce_fwd."""
    n, cin = x.shape
    ncls = w.shape[0]
    _check(x, w, bias)
    if labels.dtype != torch.int64 or not labels.is_cuda or labels.shape != (n,):
        raise RuntimeError("linear_ce_fwd: labels must be an int64 CUDA tensor of shape [n]")
    buf = torch.empty((2 * n * ncls + n + 1,), device=x.device, dtype=torch.float32)
    logits, dlogits = buf[:n * ncls].view(n, ncls), buf[n * ncls:2 * n * ncls].view(n, ncls)
    per, loss = buf[2 * n * ncls:2 * n * ncls + n], buf[2 * n * ncls + n:].view(())
    _call("agcn_linear_ce_fwd", _ptr(x), _ptr(w), _ptr(bias), labels.data_ptr(), logits.data_ptr(), dlogits.data_ptr(), per.data_ptr(),
          loss.data_ptr(), n, cin, ncls, _stream(), sig=(n, cin, ncls), work=(2.0 * n * cin * ncls, 4.0 * (x.numel() + w.numel())))
    return loss, logits, dlogits


def linear_ce_bwd(x, w, dlogits, grad_loss, need_dx=True, need_db=True):
    n, cin = x.shape
    ncls = w.shape[0]
    _check(x, w, dlogits, grad_loss)
    dw = torch.empty_like(w)
    db = torch.empty((ncls,), device=x.device, dtype=torch.float32) if need_db else None
    dx = torch.empty_like(x) if need_dx else None
    _call("agcn_linear_ce_bwd", _ptr(x), _ptr(w), dlogits.data_ptr(), _ptr(grad_loss), _ptr(dw), _ptr(db), _ptr(dx), n, cin, ncls, _stream(),
          sig=(n, cin, ncls), work=(4.0 * n * cin * ncls, 4.0 * (x.numel() + w.numel())))
    return dw, db, dx


# ----------------------------------------------------------------------------- fixed-matrix node mixing (STGCN graph convolution)
def node_mix(inp, mat, *, transpose=False, out=None, accumulate=False):
    """inp [batch, v, c], mat [v, v] -> out[b, v, c] (+)= sum_u mat[v, u] inp[b, u, c]   (transpose: mat[u, v])."""
    b, v, c = inp.shape
    if out is None:
        if accumulate:
            raise RuntimeError("node_mix: accumulate needs an output tensor")
        out = torch.empty_like(inp)
    _check(inp, mat, out)
    _call("agcn_node_mix", _ptr(inp), _ptr(mat), _ptr(out), b, v, c, int(transpose), int(accumulate), _stream(),
          sig=(b, v, c, int(transpose), int(accumulate)), work=(2.0 * b * v * v * c, 4.0 * (inp.numel() + out.numel())))
    return out
