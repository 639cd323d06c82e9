"""TEST INFRASTRUCTURE ONLY -- plain-torch restatement of every entry point of
include/agcn_b200.h, with the signatures of ``fusion_gcn_b200/ops.py``.

Two uses, both from ``tests/``:
  * ``-m gpu``: each CUDA kernel is compared with its function here on the same inputs;
  * ``-m "not gpu"``: the tests swap this module in for ``fusion_gcn_b200.functional.K`` so the
    host-side composition (forward order, every backward formula, parameter packing, state-dict
    handling) is checked against ``oracle/agcn_oracle.py`` / the golden fixtures on CPU.
The package itself never imports this file.  Works in fp32 or fp64 (dtype follows the inputs).

Maths: SURVEY.md Appendix A; reference lines torch_src/models/mmargcn/agcn.py:37-51,96-115,134-136.
"""
import torch

PREC_FP32, PREC_TF32, PREC_FP32_FFMA, PREC_BF16X3 = 0, 1, 2, 3
MIX_AGG_FWD, MIX_AGG_BWD, MIX_SCORE_BWD = 0, 1, 2
RES_NONE, RES_TENSOR, RES_AFFINE = 0, 1, 2
NUM_SMS = 148


def _gather_index(t_in, t_out, taps, stride, pad, transposed, device):
    """[t_out, taps] input time index, -1 where the tap falls outside / is not divisible."""
    to = torch.arange(t_out, device=device).view(-1, 1)
    tap = torch.arange(taps, device=device).view(1, -1)
    if not transposed:
        ti = stride * to + tap - pad
        ok = (ti >= 0) & (ti < t_in)
    else:
        num = to + pad - tap
        ok = (num >= 0) & (num % stride == 0)
        ti = torch.div(num, stride, rounding_mode="floor")
        ok = ok & (ti < t_in)
    return torch.where(ok, ti, torch.full_like(ti, -1))


def _gathered(x, t_out, taps, stride, pad, transposed):
    """x [nb,t_in,v,c] -> [nb,t_out,taps,v,c] with zeros for invalid taps."""
    nb, t_in, v, c = x.shape
    idx = _gather_index(t_in, t_out, taps, stride, pad, transposed, x.device)
    xp = torch.cat([x, x.new_zeros(nb, 1, v, c)], dim=1)           # index -1 -> zero row
    return xp[:, idx.reshape(-1)].reshape(nb, t_out, taps, v, c)


def conv_fwd(x, w, bias=None, *, t_out=None, stride=1, pad=0, transposed=False, out=None, accumulate=False,
             precision=PREC_FP32):
    nb, t_in, v, cin = x.shape
    cout, taps, _ = w.shape
    t_out = t_in if t_out is None else t_out
    g = _gathered(x, t_out, taps, stride, pad, transposed)
    y = torch.einsum("ntkvc,okc->ntvo", g, w)
    if bias is not None:
        y = y + bias
    if out is None:
        return y.contiguous()
    if accumulate:
        out += y
    else:
        out.copy_(y)
    return out


def conv_fwd_post(x, w, bias=None, *, scale=None, shift=None, res=None, relu=False, t_out=None, stride=1, pad=0, precision=PREC_FP32):
    y = conv_fwd(x, w, bias, t_out=t_out, stride=stride, pad=pad)
    if scale is not None:
        y = y * scale + shift
    if res is not None:
        y = y + res
    return torch.relu(y) if relu else y


def conv_wgrad(dy, x, *, taps=1, stride=1, pad=0, want_bias=True, precision=PREC_FP32):
    t_out = dy.shape[1]
    g = _gathered(x, t_out, taps, stride, pad, False)
    dw = torch.einsum("ntvo,ntkvc->okc", dy, g).contiguous()
    db = dy.sum(dim=(0, 1, 2)) if want_bias else None
    return dw, db


def node_mix(inp, mat, *, transpose=False, out=None, accumulate=False):
    res = torch.einsum("uv,buc->bvc" if transpose else "vu,buc->bvc", mat, inp)
    if out is None:
        return res.contiguous()
    if accumulate:
        out += res
    else:
        out.copy_(res)
    return out


def pick_nchunk(nb, t, v=0, width=0):
    if v > 32:
        return 1
    n = max(1, min((4 * NUM_SMS + nb - 1) // nb, max(1, t // 4)))
    return min(n, t)


def joint_gram(a, b, *, groups, offa, stridea, offb, strideb, width, nchunk, precision=0):
    nb, t, v, _ = a.shape
    t_per = (t + nchunk - 1) // nchunk
    out = a.new_zeros(nb, nchunk, groups, v, v)
    for c in range(nchunk):
        t0, t1 = c * t_per, min(t, (c + 1) * t_per)
        if t0 >= t1:
            continue
        for g in range(groups):
            aa = a[:, t0:t1, :, offa + g * stridea: offa + g * stridea + width]
            bb = b[:, t0:t1, :, offb + g * strideb: offb + g * strideb + width]
            out[:, c, g] = torch.einsum("ntuc,ntvc->nuv", aa, bb)
    return out


def attention_fwd(s_part, adj_a, adj_b, scale):
    s = s_part.sum(dim=1) * scale
    p = torch.softmax(s, dim=-2)
    return p.contiguous(), (p + adj_a + adj_b).contiguous()


def attention_bwd(dg_part, p, scale):
    dg = dg_part.sum(dim=1)
    dot = (p * dg).sum(dim=-2, keepdim=True)
    ds = scale * p * (dg - dot)
    return ds.contiguous(), dg.sum(dim=0).contiguous()


def conv_fwd_stats(x, w, bias=None, *, t_out=None, stride=1, pad=0, precision=0):
    """conv_fwd plus what a following training-mode BatchNorm needs: part [1, 4, cout] = (sum, sum of squares) of y - p, the pivot p
    (the first row of y) and the row count -- the layout of agcn_conv_fwd_stats with a single partial."""
    y = conv_fwd(x, w, bias, t_out=t_out, stride=stride, pad=pad)
    flat = y.reshape(-1, y.shape[-1]).double()
    pivot = flat[0].clone()
    flat = flat - pivot
    return y, torch.stack([flat.sum(0), (flat * flat).sum(0), pivot, torch.full_like(pivot, flat.shape[0])]).unsqueeze(0)


def bn_finalize(part, rows, gamma, beta, running_mean, running_var, nbt, momentum, eps):
    p = part.double()
    s1, s2, piv, cnt = p[:, 0], p[:, 1], p[:, 2], p[:, 3].clamp_min(1)
    mean_p = piv + s1 / cnt
    mean = (mean_p * p[:, 3]).sum(0) / rows
    var = (((s2 - s1 * s1 / cnt) + p[:, 3] * (mean_p - mean) ** 2).sum(0) / rows).clamp_min(0)          # pairwise-variance merge
    if running_mean is not None:
        unbiased = var * rows / (rows - 1) if rows > 1 else var
        running_mean.mul_(1 - momentum).add_((momentum * mean).to(running_mean.dtype))
        running_var.mul_(1 - momentum).add_((momentum * unbiased).to(running_var.dtype))
    if nbt is not None:
        nbt += 1
    invstd = 1.0 / torch.sqrt(var + eps)
    g = gamma.double() if gamma is not None else torch.ones_like(mean)
    b = beta.double() if beta is not None else torch.zeros_like(mean)
    dt = gamma.dtype if gamma is not None else torch.float32
    return (g * invstd).to(dt), (b - mean * g * invstd).to(dt), mean.to(dt), invstd.to(dt)


def joint_mix(inp, mats, *, width, mode, out=None, accumulate=False, precision=0):
    nb, t, v, _ = inp.shape
    w = width
    if mode == MIX_AGG_FWD:
        res = torch.einsum("ntuc,nkuv->ntvkc", inp, mats).reshape(nb, t, v, 3 * w)
    elif mode == MIX_AGG_BWD:
        res = torch.einsum("ntvkc,nkuv->ntuc", inp.reshape(nb, t, v, 3, w), mats)
    elif mode == MIX_SCORE_BWD:
        e = inp.reshape(nb, t, v, 3, 2, w)
        theta, phi = e[..., 0, :], e[..., 1, :]                       # [nb,t,v,3,w]
        dtheta = torch.einsum("nkuv,ntvkc->ntukc", mats, phi)
        dphi = torch.einsum("nkuv,ntukc->ntvkc", mats, theta)
        res = torch.stack([dtheta, dphi], dim=4).reshape(nb, t, v, 6 * w)
    else:
        raise RuntimeError("unknown mode")
    if out is None:
        return res.contiguous()
    if accumulate:
        out += res
    else:
        out.copy_(res)
    return out


def joint_mix_score_bwd(e, ds, *, width, precision=0):
    """(de, column sums of de over all rows): the score-backward mix and the theta / phi bias gradient it also produces."""
    de = joint_mix(e, ds, width=width, mode=MIX_SCORE_BWD)
    return de, de.reshape(-1, de.shape[-1]).sum(0)


def _rows_view(x, rowmap):
    """[..., channels] view honouring rowmap = (outer, inner, outer_stride, channels)."""
    if rowmap is None:
        return x.view(-1, x.shape[-1])
    outer, inner, ostride, c = rowmap
    return torch.as_strided(x, (outer, inner, c), (ostride if outer > 1 else inner * c, c, 1), x.storage_offset())


def bn_stats(x, gamma, beta, running_mean, running_var, nbt, momentum, eps, training, rowmap=None):
    xv = _rows_view(x, rowmap)
    xv = xv.reshape(-1, xv.shape[-1])
    m = xv.shape[0]
    if training:
        mean = xv.mean(dim=0)
        var = xv.var(dim=0, unbiased=False)
        if running_mean is not None:
            unbiased = var * m / (m - 1) if m > 1 else var
            running_mean.mul_(1 - momentum).add_(momentum * mean.to(running_mean.dtype))
            running_var.mul_(1 - momentum).add_(momentum * unbiased.to(running_var.dtype))
        if nbt is not None:
            nbt += 1
    else:
        mean, var = running_mean.to(x.dtype), running_var.to(x.dtype)
    invstd = torch.rsqrt(var + eps)
    g = gamma if gamma is not None else torch.ones_like(mean)
    b = beta if beta is not None else torch.zeros_like(mean)
    scale = g * invstd
    return scale, b - mean * scale, mean, invstd


def bn_stats_partials(x, rowmap=None):
    """Mergeable column statistics of x (agcn_bn_stats_partials): part [1, 4, c] = (sum, sum of squares) of x - p, the pivot p (the first
    row) and the row count -- what bn_finalize merges, here with a single partial."""
    xv = _rows_view(x, rowmap)
    flat = xv.reshape(-1, xv.shape[-1]).double()
    pivot = flat[0].clone()
    flat = flat - pivot
    return torch.stack([flat.sum(0), (flat * flat).sum(0), pivot, torch.full_like(pivot, flat.shape[0])]).unsqueeze(0)


def bf16_split(x):
    """[..., C] -> [2, rows, C] bf16 pieces h = bf16(x), m = bf16(x - h) (round to nearest, ties away): the split-operand format of the
    weight-gradient kernel (agcn_conv_wgrad_presplit).  fp64 inputs (the tests' reference runs) are carried exactly instead: [2, rows, C]
    with the value in plane 0 and zeros in plane 1."""
    flat = x.reshape(-1, x.shape[-1]).contiguous()
    if flat.dtype != torch.float32:
        return torch.stack([flat, torch.zeros_like(flat)])
    hb = (flat.view(torch.int32) + 0x8000) & -65536
    h = hb.view(torch.float32)
    mb = ((flat - h).view(torch.int32) + 0x8000) & -65536
    return torch.stack([(hb >> 16).to(torch.int16), (mb >> 16).to(torch.int16)]).view(torch.bfloat16)


def conv_wgrad_presplit(dy_split, x_split, shape, *, taps=1, stride=1, pad=0):
    nb, t_in, v = shape
    t_out = (t_in + 2 * pad - taps) // stride + 1
    cout, cin = dy_split.shape[-1], x_split.shape[-1]
    if cin % 64 or cout % 64:
        return None
    wide = torch.float32 if dy_split.dtype == torch.bfloat16 else dy_split.dtype
    dy = (dy_split[0].to(wide) + dy_split[1].to(wide)).reshape(nb, t_out, v, cout)
    x = (x_split[0].to(wide) + x_split[1].to(wide)).reshape(nb, t_in, v, cin)
    return conv_wgrad(dy, x, taps=taps, stride=stride, pad=pad, want_bias=False)[0]


def bn_apply(y, scale, shift, *, res_mode=RES_NONE, res=None, scale2=None, shift2=None, relu=False, rowmap=None, out=None,
             want_mask=False, want_split=False):
    r = _bn_apply(y, scale, shift, res_mode=res_mode, res=res, scale2=scale2, shift2=shift2, relu=relu, rowmap=rowmap, out=out)
    bits = (r > 0) if want_mask else None              # the "bit mask" of the CUDA path is a bool tensor here
    split = bf16_split(r) if (want_mask and want_split and r.shape[-1] % 64 == 0 and rowmap is None) else None
    return r, bits, split


def _bn_apply(y, scale, shift, *, res_mode=RES_NONE, res=None, scale2=None, shift2=None, relu=False, rowmap=None, out=None):
    if out is None:
        out = torch.empty_like(y)
    yv = _rows_view(y, rowmap)
    o = yv * scale + shift
    if res_mode == RES_TENSOR:
        o = o + _rows_view(res, rowmap)
    elif res_mode == RES_AFFINE:
        o = o + _rows_view(res, rowmap) * scale2 + shift2
    if relu:
        o = torch.relu(o)
    _rows_view(out, rowmap).copy_(o)
    return out


def bn_bwd(dout, mask_out, y, save_mean, save_invstd, gamma, *, want_dy=True, dy=None, dres=None, dres_accumulate=False,
           rowmap=None, mask_bits=None, pool_rows=0, frozen=False, want_split=False, sync=None):
    if pool_rows:          # dout is the pooled gradient [groups, c]: broadcast over the rows of each group, divided by their number
        groups, c = dout.shape
        dout = (dout / pool_rows).reshape(groups, 1, c).expand(groups, pool_rows, c).reshape(y.shape).contiguous()
    g = _rows_view(dout, rowmap)
    if mask_bits is not None:
        g = g * mask_bits.reshape(g.shape).to(g.dtype)
    elif mask_out is not None:
        g = g * (_rows_view(mask_out, rowmap) > 0).to(g.dtype)
    yv = _rows_view(y, rowmap)
    c = yv.shape[-1]
    xhat = (yv - save_mean) * save_invstd
    red = tuple(range(g.dim() - 1))
    m = g.numel() // c
    dbeta = g.sum(dim=red)
    dgamma = (g * xhat).sum(dim=red)
    s1, s2 = dbeta, dgamma
    if sync is not None and not frozen:
        # synchronised BatchNorm (agcn_bn_bwd phases 1 and 2): the two sums and the row count over all ranks; dgamma / dbeta stay this rank's own
        both = sync.all_reduce(torch.stack([dbeta, dgamma]))
        s1, s2, m = both[0], both[1], m * sync.world
    if want_dy:
        gam = gamma if gamma is not None else torch.ones_like(save_mean)
        if dy is None:
            dy = torch.empty_like(y)
        # frozen: eval-mode BatchNorm, the statistics are constants
        _rows_view(dy, rowmap).copy_(gam * save_invstd * (g if frozen else g - s1 / m - xhat * s2 / m))
    if dres is not None:
        dv = _rows_view(dres, rowmap)
        if dres_accumulate:
            dv += g
        else:
            dv.copy_(g)
    ok = want_split and dy is not None and mask_bits is not None and rowmap is None and dy.shape[-1] % 64 == 0
    return dy, dgamma, dbeta, (bf16_split(dy) if ok else None)


def bn_bwd_dual(dout, a, b, *, mask_out=None, mask_bits=None, frozen=False, want_split=False, pool_rows=0, sync=None):
    """Two BatchNorm backwards over the same upstream gradient and ReLU mask (agcn_bn_bwd_bits_dual, or two bn_bwd calls); only
    BatchNorm A gets bf16 pieces."""
    kw = dict(mask_bits=mask_bits, frozen=frozen, pool_rows=pool_rows, sync=sync)
    return bn_bwd(dout, mask_out, *a, want_split=want_split, **kw) + bn_bwd(dout, mask_out, *b, **kw)[:3]


def bn_pool_supported(rows, channels):
    return channels % 32 == 0


def bn_apply_pool(y, scale, shift, *, groups, res_mode=RES_NONE, res=None, scale2=None, shift2=None):
    """Fused tail: (mean over each group's rows of relu(scale*y + shift + R), ReLU mask)."""
    out = _bn_apply(y, scale, shift, res_mode=res_mode, res=res, scale2=scale2, shift2=shift2, relu=True)
    c = out.shape[-1]
    return out.reshape(groups, -1, c).mean(dim=1), (out > 0)


def pool_fwd(x, groups):
    c = x.shape[-1]
    return x.reshape(groups, -1, c).mean(dim=1)


def pool_bwd(dout, shape):
    groups, c = dout.shape
    rows = 1
    for s in shape:
        rows *= s
    rows = rows // c // groups
    return (dout / rows).reshape(groups, 1, c).expand(groups, rows, c).reshape(shape).contiguous()


def linear_ce_fwd(x, w, bias, labels):
    logits = x @ w.t() + (bias if bias is not None else 0)
    p = torch.softmax(logits, dim=1)
    n = x.shape[0]
    onehot = torch.nn.functional.one_hot(labels, w.shape[0]).to(x.dtype)
    loss = (torch.logsumexp(logits, dim=1) - (logits * onehot).sum(1)).mean()
    return loss, logits, (p - onehot) / n


def linear_ce_bwd(x, w, dlogits, grad_loss, need_dx=True, need_db=True):
    d = dlogits * grad_loss
    return d.t() @ x, (d.sum(0) if need_db else None), (d @ w if need_dx else None)


# --------------------------------------------------------------------------- TF32-mode emulation (tests only)
def _trunc_tf32(t):
    return (t.contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)


class Tf32Emulation:
    """Stage backend that restates AGCN_PREC_TF32: on the shapes the tcgen05 path takes, tcgen05.mma kind::tf32 reads the
    upper 19 bits of each fp32 operand (measured on B200), i.e. operands are TRUNCATED to TF32 and products are
    accumulated in fp32.  Everything else is the plain fp32 stage.  fp32 tensors only."""

    def __getattr__(self, name):
        return globals()[name]

    @staticmethod
    def _fwd_on_tc(x, w, transposed, stride):
        cout, taps, cin = w.shape
        ok = cin % 4 == 0 and cout % 16 == 0 and (cout <= 128 or any(cout % c == 0 for c in range(64, 257, 16)))
        return ok          # (a strided 1x1 input gradient has empty parity classes; the tensor-core kernel skips them)

    def conv_fwd(self, x, w, bias=None, *, stride=1, transposed=False, precision=PREC_FP32, **kw):
        if precision == PREC_TF32 and self._fwd_on_tc(x, w, transposed, stride):
            x, w = _trunc_tf32(x), _trunc_tf32(w)
        return conv_fwd(x, w, bias, stride=stride, transposed=transposed, **kw)

    def conv_fwd_stats(self, x, w, bias=None, *, stride=1, precision=PREC_FP32, **kw):
        if precision == PREC_TF32 and self._fwd_on_tc(x, w, False, stride):
            x, w = _trunc_tf32(x), _trunc_tf32(w)
        return conv_fwd_stats(x, w, bias, stride=stride, **kw)

    def joint_gram(self, a, b, *, precision=PREC_FP32, **kw):
        v, width, same_row = a.shape[2], kw["width"], a is b and kw["stridea"] == 32 and kw["strideb"] == 32 and kw["offb"] == kw["offa"] + 16
        on_tc = kw["groups"] == 3 and 3 * v <= 80 and ((width == 16 and same_row) or width % 32 == 0)
        if precision == PREC_TF32 and on_tc:
            a, b = _trunc_tf32(a), _trunc_tf32(b)
        return joint_gram(a, b, **kw)

    def joint_mix(self, inp, mats, *, width, mode, precision=PREC_FP32, **kw):
        if precision == PREC_TF32 and width % (16 if mode == MIX_SCORE_BWD else 32) == 0:
            inp, mats = _trunc_tf32(inp), _trunc_tf32(mats)
        return joint_mix(inp, mats, width=width, mode=mode, **kw)

    def joint_mix_score_bwd(self, e, ds, *, width, precision=PREC_FP32):
        de = self.joint_mix(e, ds, width=width, mode=MIX_SCORE_BWD, precision=precision)
        return de, de.reshape(-1, de.shape[-1]).sum(0)

    def conv_wgrad(self, dy, x, *, precision=PREC_FP32, **kw):
        _, db = conv_wgrad(dy, x, **kw)
        if precision == PREC_TF32 and x.shape[-1] % 4 == 0 and dy.shape[-1] % 4 == 0:
            dy, x = _trunc_tf32(dy), _trunc_tf32(x)
        dw, _ = conv_wgrad(dy, x, **kw)
        return dw, db
