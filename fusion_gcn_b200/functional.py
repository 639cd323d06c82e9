"""Host-side composition of the AGCN unit from the C-ABI kernels, forward and backward.

Activations are channels-last ``[nb, t, v, c]`` (nb = N*M person-sequences).  The module
parameters keep the reference's shapes and names; they are packed here, inside the autograd
Functions, into the layouts the kernels want and the gradients are unpacked on the way back:

  wab  [6*Ci, 1, Cin]    rows = theta_0 | phi_0 | theta_1 | phi_1 | theta_2 | phi_2   (conv_a / conv_b, agcn.py:71-72)
  wd   [Cout, 1, 3*Cin]  columns = subset 0 | 1 | 2 (conv_d, agcn.py:73): sum_k Wd_k (X G_k) = [Wd_0 Wd_1 Wd_2] . [X G_0; X G_1; X G_2]
  wt   [Cout, 9, Cout]   temporal taps (tcn1.conv, agcn.py:41-42)

Maths: SURVEY.md Appendix A.  Reference: torch_src/models/mmargcn/agcn.py:49-51,96-115,134-136.
"""
from dataclasses import dataclass, field
from typing import List, Optional

import torch

from . import ops as K      # tests swap this for oracle.stages on CPU; the package has no fallback

BN_EPS = 1e-5
BN_MOMENTUM = 0.1


@dataclass
class BnBuffers:
    running_mean: torch.Tensor
    running_var: torch.Tensor
    num_batches_tracked: Optional[torch.Tensor]


@dataclass
class UnitSpec:
    """Static description of one SpatialTemporalConv (or of its gcn / tcn half)."""
    cin: int
    cout: int
    stride: int = 1
    residual: str = "none"          # 'none' | 'identity' | 'conv'
    has_down: bool = False
    kernel_size: int = 9
    relu_out: bool = True
    training: bool = True
    precision: int = 0
    bn_gcn: Optional[BnBuffers] = None
    bn_down: Optional[BnBuffers] = None
    bn_tcn: Optional[BnBuffers] = None
    bn_res: Optional[BnBuffers] = None
    attention_out: Optional[List[torch.Tensor]] = field(default=None)   # receives adj_c (3 x [nb,V,V], detached)
    pool_groups: int = 0            # > 0 (last unit of Model): return the mean-pooled [pool_groups, cout] instead of the feature map
    # grad mode of the CALLER when the spec is built (inside autograd.Function.forward it is always off, and ctx.needs_input_grad does
    # not look at it): under torch.no_grad() nothing can ask for a backward, so eval mode takes the fused, nothing-saved path
    grad_enabled: bool = field(default_factory=torch.is_grad_enabled)
    sync: Optional[object] = None   # distributed.SyncBatchNorm: training-mode BatchNorm statistics over all ranks of its group (SURVEY 8e)
    recompute: bool = False         # do not keep theta / phi (e) and the aggregated tensor (z) for the backward; run their kernels again there


def _bn_forward(y, gamma, beta, buf: BnBuffers, training: bool, sync=None, rowmap=None, nbt=True):
    """-> scale, shift, save_mean, save_invstd.  ``sync`` (training mode): the statistics are taken over the rows of ALL ranks -- every
    rank's mergeable partials are all-gathered and finalised with the global row count (synchronised BatchNorm)."""
    tracked = buf.num_batches_tracked if nbt else None
    if training and sync is not None:
        part = K.bn_stats_partials(y, rowmap=rowmap)
        rows = (rowmap[0] * rowmap[1]) if rowmap is not None else y.numel() // y.shape[-1]
        return K.bn_finalize(sync.gather_partials(part), rows * sync.world, gamma, beta, buf.running_mean, buf.running_var, tracked,
                             BN_MOMENTUM, BN_EPS)
    return K.bn_stats(y, gamma, beta, buf.running_mean, buf.running_var, tracked, BN_MOMENTUM, BN_EPS, training,
                      **({} if rowmap is None else dict(rowmap=rowmap)))


def _conv_bn(x, w, bias, gamma, beta, buf: BnBuffers, training: bool, prec: int, sync=None, **kw):
    """Conv2d -> BatchNorm2d pair (agcn.py:41-51,73-83): y = conv(x) and the BN scale / shift / saved statistics of y.
    In training mode the column sums come out of the convolution's epilogue (conv_fwd_stats) when the kernel covers the
    shape, which saves the separate statistics pass over y."""
    if training:
        y, part = K.conv_fwd_stats(x, w, bias, precision=prec, **kw)
        if part is not None:
            rows = y.numel() // y.shape[-1]
            if sync is not None:
                part, rows = sync.gather_partials(part), rows * sync.world
            return y, K.bn_finalize(part, rows, gamma, beta, buf.running_mean, buf.running_var, buf.num_batches_tracked,
                                    BN_MOMENTUM, BN_EPS)
    else:
        y = K.conv_fwd(x, w, bias, precision=prec, **kw)
    return y, _bn_forward(y, gamma, beta, buf, training, sync)


def _eval_affine(gamma, beta, buf: BnBuffers):
    """(scale, shift) of an eval-mode BatchNorm: gamma / sqrt(running_var + eps), beta - running_mean * scale."""
    c = gamma.shape[0]
    sc, sh, _, _ = K.bn_stats(gamma, gamma, beta, buf.running_mean, buf.running_var, None, BN_MOMENTUM, BN_EPS, False, rowmap=(1, 1, 0, c))
    return sc, sh


def _zero_bias(like, n):
    """Gradient of a conv bias that feeds a training-mode BatchNorm: BN subtracts the batch mean, so the loss does not
    depend on the bias and its gradient is identically zero (SURVEY D8; the reference's autograd produces ~1e-9 rounding
    noise here).  Returned analytically instead of summing dy over all rows."""
    return torch.zeros((n,), device=like.device, dtype=torch.float32)


def _t(w):
    """[cout, taps, cin] -> [cin, taps, cout] (weight of the input-gradient contraction)."""
    return w.permute(2, 1, 0).contiguous()


# Weight gradients are LEAVES of the backward pass: nothing downstream in the unit reads them.  With OVERLAP_LEAVES they are launched on a
# side stream, so that the tensor-bound weight-gradient kernel of the temporal convolution shares the SMs with the HBM-bound BatchNorm
# backward that follows on the main stream (its CTAs need 0-12 KB of shared memory and fit beside the persistent CTA), instead of the
# two running back to back.  Fork / join are stream waits (capturable in the step's CUDA graph); the join happens before the unit's
# backward returns, so autograd, gradient hooks and optimizers see ordinary main-stream tensors.
OVERLAP_LEAVES = True
_side_streams = {}


def set_overlap_leaves(flag: bool) -> None:
    global OVERLAP_LEAVES
    OVERLAP_LEAVES = bool(flag)


class _Leaves:
    def __init__(self, like):
        self.on = bool(OVERLAP_LEAVES and like is not None and like.is_cuda)
        self.device = like.device if self.on else None          # the tensors' device, which need not be the current one
        self.side = None
        self.keep = []

    def run(self, fn, *inputs):
        """fn() on the side stream, after everything enqueued on the current stream so far.  ``inputs`` (main-stream tensors the
        side kernels read) are kept alive until join(), so the caching allocator cannot hand their memory to a later main-stream
        allocation while the side kernel still reads it."""
        if not self.on:
            return fn()
        cur = torch.cuda.current_stream(self.device)
        if self.side is None:
            key = (cur.device.index, cur.cuda_stream)
            self.side = _side_streams.get(key)
            if self.side is None:
                self.side = _side_streams[key] = torch.cuda.Stream(device=cur.device)
        self.side.wait_stream(cur)
        self.keep.extend(t for t in inputs if t is not None)
        with torch.cuda.stream(self.side):
            return fn()

    def join(self):
        if self.side is not None:
            torch.cuda.current_stream(self.device).wait_stream(self.side)
            self.side = None
        self.keep.clear()


# =============================================================================== gcn half
def gcn_forward(x, adj_a, adj_b, wa, ba, wb, bb, wd, bd, bn_w, bn_b, down_w, down_b, dbn_w, dbn_b, spec: UnitSpec, ctx):
    nb, t, v, cin = x.shape
    cout = spec.cout
    ci = wa[0].shape[0]
    prec = spec.precision
    wab = torch.cat([w.reshape(ci, 1, cin) for pair in zip(wa, wb) for w in pair], dim=0)
    bab = torch.cat([b for pair in zip(ba, bb) for b in pair], dim=0)
    wdc = torch.cat([w.reshape(cout, 1, cin) for w in wd], dim=2).contiguous()
    bdc = bd[0] + bd[1] + bd[2]

    want_mask = ctx is not None                          # the backward reads the ReLU mask as one bit per element
    e = K.conv_fwd(x, wab, bab, precision=prec)                                        # theta / phi embeddings
    nchunk = K.pick_nchunk(nb, t, v, ci)
    s_part = K.joint_gram(e, e, groups=3, offa=0, stridea=2 * ci, offb=ci, strideb=2 * ci, width=ci, nchunk=nchunk, precision=prec)
    scale = 1.0 / float(ci * t)
    p, g = K.attention_fwd(s_part, adj_a.contiguous(), adj_b.contiguous(), scale)
    z = K.joint_mix(x, g, width=cin, mode=K.MIX_AGG_FWD, precision=prec)                               # [nb,t,v,3*cin]
    if not spec.training and ctx is None:
        # eval mode without gradients (session.py:188-194): BatchNorm is a per-channel affine of the running statistics, so BN, the down / identity
        # branch and the ReLU ride in the projection's epilogue -- no pre-BN tensor, no separate normalise pass, nothing saved
        sc, sh = _eval_affine(bn_w, bn_b, spec.bn_gcn)
        if spec.has_down:
            sc2, sh2 = _eval_affine(dbn_w, dbn_b, spec.bn_down)
            res = K.conv_fwd_post(x, down_w.reshape(cout, 1, cin), down_b, scale=sc2, shift=sh2, precision=prec)
        else:
            res = x
        o = K.conv_fwd_post(z, wdc, bdc, scale=sc, shift=sh, res=res, relu=True, precision=prec)
        if spec.attention_out is not None:
            spec.attention_out[:] = [p[:, k] for k in range(3)]
        return o
    y, (sc, sh, mean, invstd) = _conv_bn(z, wdc, bdc, bn_w, bn_b, spec.bn_gcn, spec.training, prec, sync=spec.sync)
    # the temporal convolution that follows takes its weight gradient from bf16 pieces of `o` written here, by the pass that
    # produces `o` anyway (agcn_conv_wgrad_presplit): no conversion pass in the weight-gradient kernel
    want_split = want_mask and spec.training and cout % 64 == 0 and prec != K.PREC_FP32_FFMA and prec != K.PREC_TF32
    if spec.has_down:
        yd, (sc2, sh2, mean2, invstd2) = _conv_bn(x, down_w.reshape(cout, 1, cin), down_b, dbn_w, dbn_b, spec.bn_down, spec.training, prec, sync=spec.sync)
        o, o_bits, o_split = K.bn_apply(y, sc, sh, want_mask=want_mask, want_split=want_split, res_mode=K.RES_AFFINE, res=yd, scale2=sc2,
                                        shift2=sh2, relu=True)
    else:
        yd = mean2 = invstd2 = None
        o, o_bits, o_split = K.bn_apply(y, sc, sh, want_mask=want_mask, want_split=want_split, res_mode=K.RES_TENSOR, res=x, relu=True)
    if spec.attention_out is not None:
        spec.attention_out[:] = [p[:, k] for k in range(3)]
    if ctx is not None:
        # recompute policy (SURVEY 7.1 step 7): e (1.5 cout wide) and z (3 cin wide) are more than half of what a unit saves, and each is
        # ONE deterministic kernel away from x (and g) -- the backward runs those two kernels again and gets the same bits
        keep = not spec.recompute
        ctx.update(x=x, e=e if keep else None, p=p, g=g, z=z if keep else None, y=y, yd=yd, o=o.detach(), o_bits=o_bits, o_split=o_split,
                   mean=mean, invstd=invstd, mean2=mean2, invstd2=invstd2, wab=wab, bab=bab, wdc=wdc, nchunk=nchunk, scale=scale, ci=ci)
    return o


def gcn_backward(d_o, ctx, bn_w, dbn_w, down_w, spec: UnitSpec, dx=None, need_dx=True, leaves=None):
    """Returns (dx, grads) where grads follows the parameter order of gcn_forward.  ``dx`` may carry
    an already-written gradient buffer to accumulate into.  ``leaves``: the caller's _Leaves (it joins); None = own, joined here."""
    own_leaves = leaves is None
    if own_leaves:
        leaves = _Leaves(d_o)
    x, e, p, g, z, y, o = ctx["x"], ctx["e"], ctx["p"], ctx["g"], ctx["z"], ctx["y"], ctx["o"]
    nb, t, v, cin = x.shape
    cout, ci, prec = spec.cout, ctx["ci"], spec.precision
    have = dx is not None
    # eval mode with gradients (frozen-BN fine-tuning, saliency): the BatchNorms are affine maps of constants, and the biases of the
    # convolutions in front of them get real gradients (the column sums of dy) instead of the training mode's analytic zeros
    frozen = not spec.training
    if z is None:
        z = K.joint_mix(x, g, width=cin, mode=K.MIX_AGG_FWD, precision=prec)
    if spec.has_down:
        # bn and down.1 both feed the ReLU of agcn.py:113-115: one pair of passes over the shared masked gradient for both backwards
        dy, dgam, dbet, _, dyd, dgam2, dbet2 = K.bn_bwd_dual(d_o, (y, ctx["mean"], ctx["invstd"], bn_w), (ctx["yd"], ctx["mean2"], ctx["invstd2"], dbn_w),
                                                             mask_out=o, mask_bits=ctx["o_bits"], frozen=frozen, sync=spec.sync)
        wdown = down_w.reshape(cout, 1, cin)
        d_down_w, d_down_b = leaves.run(lambda: K.conv_wgrad(dyd, x, want_bias=frozen, precision=prec), dyd, x)
        if not frozen:
            d_down_b = _zero_bias(x, cout)
        if need_dx:
            dx = K.conv_fwd(dyd, _t(wdown), out=dx, accumulate=have, precision=prec)
            have = True
    else:
        if need_dx and dx is None:
            dx = torch.empty_like(x)
        dy, dgam, dbet, _ = K.bn_bwd(d_o, o, y, ctx["mean"], ctx["invstd"], bn_w, dres=dx if need_dx else None, dres_accumulate=have,
                                     mask_bits=ctx["o_bits"], frozen=frozen, sync=spec.sync)
        have = have or need_dx
        dgam2 = dbet2 = d_down_w = d_down_b = None
    dz = K.conv_fwd(dy, _t(ctx["wdc"]), precision=prec)                                # [nb,t,v,3*cin]
    d_wdc, d_bdc = leaves.run(lambda: K.conv_wgrad(dy, z, want_bias=frozen, precision=prec), dy, z)
    del z
    if not frozen:
        d_bdc = _zero_bias(x, cout)
    dg_part = K.joint_gram(x, dz, groups=3, offa=0, stridea=0, offb=0, strideb=cin, width=cin, nchunk=K.pick_nchunk(nb, t, v, cin),
                           precision=prec)
    ds, d_adj_b = K.attention_bwd(dg_part, p, ctx["scale"])
    if need_dx:
        dx = K.joint_mix(dz, g, width=cin, mode=K.MIX_AGG_BWD, out=dx, accumulate=have, precision=prec)
        have = True
    # d theta / d phi, and their column sums (= the bias gradients) out of the same epilogue where the kernel covers the shape
    if e is None:
        e = K.conv_fwd(x, ctx["wab"], ctx["bab"], precision=prec)
    de, d_bab = K.joint_mix_score_bwd(e, ds, width=ci, precision=prec)
    want_bab = d_bab is None
    d_wab, d_bab2 = leaves.run(lambda: K.conv_wgrad(de, x, want_bias=want_bab, precision=prec), de, x)
    if d_bab is None:
        d_bab = d_bab2
    if need_dx:
        dx = K.conv_fwd(de, _t(ctx["wab"]), out=dx, accumulate=have, precision=prec)
    if own_leaves:
        leaves.join()
    # unpack
    d_wa = [d_wab[(2 * k) * ci:(2 * k + 1) * ci].reshape(ci, cin, 1, 1) for k in range(3)]
    d_wb = [d_wab[(2 * k + 1) * ci:(2 * k + 2) * ci].reshape(ci, cin, 1, 1) for k in range(3)]
    d_ba = [d_bab[(2 * k) * ci:(2 * k + 1) * ci] for k in range(3)]
    d_bb = [d_bab[(2 * k + 1) * ci:(2 * k + 2) * ci] for k in range(3)]
    d_wd = [d_wdc[:, 0, k * cin:(k + 1) * cin].reshape(cout, cin, 1, 1) for k in range(3)]
    d_bd = [d_bdc, d_bdc.clone(), d_bdc.clone()]       # three parameters, three tensors: .grad tensors must not alias (in-place unscale / clipping)
    grads = dict(adj_b=d_adj_b, wa=d_wa, ba=d_ba, wb=d_wb, bb=d_bb, wd=d_wd, bd=d_bd, bn_w=dgam, bn_b=dbet,
                 down_w=None if d_down_w is None else d_down_w.reshape(cout, cin, 1, 1), down_b=d_down_b,
                 dbn_w=dgam2, dbn_b=dbet2)
    return dx, grads


# =============================================================================== tcn half
def _pack_taps(w):
    """[cout, cin, k, 1] -> [cout, k, cin]."""
    return w.squeeze(-1).permute(0, 2, 1).contiguous()


def tcn_forward(o, x_res, wt, bt, bn_w, bn_b, wr, br, rbn_w, rbn_b, spec: UnitSpec, ctx):
    nb, t, v, c = o.shape
    s, ksz = spec.stride, spec.kernel_size
    pad = (ksz - 1) // 2
    t_out = (t + 2 * pad - ksz) // s + 1
    prec = spec.precision
    wtp = _pack_taps(wt)
    if not spec.training and ctx is None:
        # eval mode without gradients: temporal conv + BN + residual + ReLU in one pass (the residual branch's conv + BN in one more)
        sc, sh = _eval_affine(bn_w, bn_b, spec.bn_tcn)
        if spec.residual == "identity":
            res = x_res
        elif spec.residual == "conv":
            sc2, sh2 = _eval_affine(rbn_w, rbn_b, spec.bn_res)
            res = K.conv_fwd_post(x_res, _pack_taps(wr), br, scale=sc2, shift=sh2, t_out=t_out, stride=s, pad=0, precision=prec)
        else:
            res = None
        out = K.conv_fwd_post(o, wtp, bt, scale=sc, shift=sh, res=res, relu=spec.relu_out, t_out=t_out, stride=s, pad=pad, precision=prec)
        return out
    u, (sc, sh, mean, invstd) = _conv_bn(o, wtp, bt, bn_w, bn_b, spec.bn_tcn, spec.training, prec, sync=spec.sync, t_out=t_out, stride=s, pad=pad)
    ur = mean2 = invstd2 = wrp = None
    want_mask = ctx is not None and spec.relu_out
    # the model's tail (agcn.py:194-196): the last unit's output only feeds the global mean pool, so the pooled means and the ReLU
    # mask bits come out of the normalise / residual / ReLU pass and the feature map itself is never written
    pool = spec.pool_groups if (spec.pool_groups and spec.training and spec.relu_out and
                                K.bn_pool_supported(u.numel() // u.shape[-1], u.shape[-1])) else 0
    apply = (lambda *a, **kw: K.bn_apply_pool(*a, groups=pool, **{k: v for k, v in kw.items() if k != "relu"})) if pool else \
        (lambda *a, **kw: K.bn_apply(*a, want_mask=want_mask, **kw)[:2])
    if spec.residual == "identity":
        out, out_bits = apply(u, sc, sh, res_mode=K.RES_TENSOR, res=x_res, relu=spec.relu_out)
    elif spec.residual == "conv":
        wrp = _pack_taps(wr)
        ur, (sc2, sh2, mean2, invstd2) = _conv_bn(x_res, wrp, br, rbn_w, rbn_b, spec.bn_res, spec.training, prec, sync=spec.sync, t_out=t_out, stride=s, pad=0)
        out, out_bits = apply(u, sc, sh, res_mode=K.RES_AFFINE, res=ur, scale2=sc2, shift2=sh2, relu=spec.relu_out)
    else:
        out, out_bits = apply(u, sc, sh, relu=spec.relu_out)
    if ctx is not None:
        ctx.update(t_o=o.detach(), t_o_shape=tuple(o.shape), t_x=x_res, u=u, ur=ur, out=None if (pool or out_bits is not None or not spec.relu_out) else out.data, out_bits=out_bits, t_mean=mean, t_invstd=invstd,
                   t_mean2=mean2, t_invstd2=invstd2, wtp=wtp, wrp=wrp, pad=pad, pool_rows=(u.numel() // u.shape[-1] // pool) if pool else 0)
    return out


def tcn_backward(d_out, ctx, bn_w, rbn_w, spec: UnitSpec, need_dres=True, need_do=True, leaves=None):
    """Returns (d_o, d_xres, grads).  ``leaves``: the caller's _Leaves (it joins); None = own, joined here."""
    own_leaves = leaves is None
    if own_leaves:
        leaves = _Leaves(d_out)
    o, x_res, u, out = ctx["t_o"], ctx["t_x"], ctx["u"], ctx["out"]
    o_shape = ctx["t_o_shape"]              # (`o` itself is released when its bf16 pieces serve the weight gradient, see UnitFn.forward)
    s, pad, prec = spec.stride, ctx["pad"], spec.precision
    ksz = spec.kernel_size
    mask = out if spec.relu_out else None
    bits = ctx["out_bits"] if spec.relu_out else None
    d_xres = None
    d_wr = d_br = dgam2 = dbet2 = None
    frozen = not spec.training          # eval mode with gradients, see gcn_backward
    # weight gradient of the temporal convolution from split operands: `o` as bf16 pieces from the gcn half's normalise pass, `du` as
    # bf16 pieces from the BatchNorm backward below (bit-mask forms only)
    o_split = ctx.get("o_split") if (not frozen and bits is not None) else None
    # pool_rows > 0: d_out is the pooled gradient [groups, c]
    kw = dict(mask_bits=bits, pool_rows=ctx.get("pool_rows", 0), frozen=frozen, sync=spec.sync, want_split=o_split is not None)
    if spec.residual == "identity":
        d_xres = torch.empty_like(x_res) if need_dres else None
        du, dgam, dbet, du_split = K.bn_bwd(d_out, mask, u, ctx["t_mean"], ctx["t_invstd"], bn_w, dres=d_xres, dres_accumulate=False, **kw)
    elif spec.residual == "conv":
        # the temporal BatchNorm and the residual branch's both feed the ReLU of agcn.py:135-136: one pair of passes for both backwards
        du, dgam, dbet, du_split, dur, dgam2, dbet2 = K.bn_bwd_dual(d_out, (u, ctx["t_mean"], ctx["t_invstd"], bn_w),
                                                                    (ctx["ur"], ctx["t_mean2"], ctx["t_invstd2"], rbn_w), mask_out=mask, **kw)
        d_wrp, d_br = leaves.run(lambda: K.conv_wgrad(dur, x_res, taps=1, stride=s, pad=0, want_bias=frozen, precision=prec), dur, x_res)
        if not frozen:
            d_br = _zero_bias(d_out, d_wrp.shape[0])
        d_wr = d_wrp.permute(0, 2, 1).unsqueeze(-1)
        if need_dres:
            d_xres = K.conv_fwd(dur, _t(ctx["wrp"]), t_out=x_res.shape[1], stride=s, pad=0, transposed=True, precision=prec)
    else:
        du, dgam, dbet, du_split = K.bn_bwd(d_out, mask, u, ctx["t_mean"], ctx["t_invstd"], bn_w, **kw)
    # the input gradient first (the gcn half's BatchNorm backward waits for it), then the weight gradient as a leaf beside that pass
    d_o = None
    if need_do:
        d_o = K.conv_fwd(du, _t(ctx["wtp"]), t_out=o_shape[1], stride=s, pad=pad, transposed=True, precision=prec)
    d_wtp = None
    if du_split is not None and o_split is not None:
        d_wtp = leaves.run(lambda: K.conv_wgrad_presplit(du_split, o_split, o_shape[:3], taps=ksz, stride=s, pad=pad), du_split, o_split)
        d_bt = _zero_bias(d_out, du.shape[-1])
    if d_wtp is None:
        d_wtp, d_bt = leaves.run(lambda: K.conv_wgrad(du, o, taps=ksz, stride=s, pad=pad, want_bias=frozen, precision=prec), du, o)
        if not frozen:
            d_bt = _zero_bias(d_out, d_wtp.shape[0])
    if own_leaves:
        leaves.join()
    grads = dict(wt=d_wtp.permute(0, 2, 1).unsqueeze(-1), bt=d_bt, bn_w=dgam, bn_b=dbet, wr=d_wr, br=d_br, rbn_w=dgam2, rbn_b=dbet2)
    return d_o, d_xres, grads


# =============================================================================== autograd wrappers
GCN_NPARAMS = 1 + 1 + 18 + 2 + 4      # adj_a, adj_b, (wa,ba,wb,bb,wd,bd)x3, bn w/b, down w/b + its bn w/b
TCN_NPARAMS = 4 + 4                   # wt, bt, bn w/b, wr, br, rbn w/b


def _split_gcn(params):
    adj_a, adj_b = params[0], params[1]
    wa, ba, wb, bb, wd, bd = [], [], [], [], [], []
    for k in range(3):
        a = params[2 + 6 * k: 8 + 6 * k]
        wa.append(a[0]); ba.append(a[1]); wb.append(a[2]); bb.append(a[3]); wd.append(a[4]); bd.append(a[5])
    bn_w, bn_b, down_w, down_b, dbn_w, dbn_b = params[20:26]
    return adj_a, adj_b, wa, ba, wb, bb, wd, bd, bn_w, bn_b, down_w, down_b, dbn_w, dbn_b


def _gcn_grad_tuple(g):
    out = [None, g["adj_b"]]
    for k in range(3):
        out += [g["wa"][k], g["ba"][k], g["wb"][k], g["bb"][k], g["wd"][k], g["bd"][k]]
    out += [g["bn_w"], g["bn_b"], g["down_w"], g["down_b"], g["dbn_w"], g["dbn_b"]]
    return out


def _tcn_grad_tuple(g):
    return [g["wt"], g["bt"], g["bn_w"], g["bn_b"], g["wr"], g["br"], g["rbn_w"], g["rbn_b"]]


def _like(grads, params):
    """Gradients in the shapes of their parameters (Conv1d weights of the 1-D graph convolution are (out, in, 1), Conv2d ones
    (out, in, 1, 1)); a gradient for an absent (None) parameter is dropped."""
    return [None if (g is None or p is None) else g.reshape(p.shape) for g, p in zip(grads, params)]


def _store(ctx, spec):
    """Activation store of one forward: a dict when a backward can follow (training mode, or eval mode with an input or parameter
    that requires a gradient), None otherwise -- eval mode then takes the fused, nothing-saved path."""
    return {} if (spec.training or (spec.grad_enabled and any(ctx.needs_input_grad))) else None


def _stash(ctx, store):
    """Hands the activation store to autograd: the tensors go through ``save_for_backward`` (the engine releases them as soon as the
    node's backward has run, keeps them under ``retain_graph=True`` -- a second backward then works -- and checks their version
    counters), everything else stays on the ctx."""
    ctx.has_store = store is not None
    if store is None:
        return
    keys = [k for k, v in store.items() if isinstance(v, torch.Tensor)]
    ctx.save_for_backward(*[store[k] for k in keys])
    ctx.store_keys = keys
    ctx.store_meta = {k: v for k, v in store.items() if not isinstance(v, torch.Tensor)}


def _unstash(ctx):
    if not ctx.has_store:
        raise RuntimeError("fusion_gcn_b200: this forward ran under torch.no_grad() in eval mode (fused path, nothing saved): no backward")
    store = dict(ctx.store_meta)
    store.update(zip(ctx.store_keys, ctx.saved_tensors))      # raises torch's own error on a second backward without retain_graph
    return store


class GcnFn(torch.autograd.Function):
    """SpatialGraphConv.forward (agcn.py:96-115) on a channels-last tensor."""

    @staticmethod
    def forward(ctx, x, spec, *params):
        store = _store(ctx, spec)
        o = gcn_forward(x, *_split_gcn(params), spec, store)
        ctx.spec, ctx.params = spec, params
        _stash(ctx, store)
        return o

    @staticmethod
    def backward(ctx, d_o):
        spec, p = ctx.spec, ctx.params
        dx, g = gcn_backward(d_o.contiguous(), _unstash(ctx), p[20], p[24], p[22], spec, need_dx=ctx.needs_input_grad[0])
        return (dx, None, *_like(_gcn_grad_tuple(g), p))


class TcnFn(torch.autograd.Function):
    """TemporalConv.forward (agcn.py:49-51), optionally with the unit's residual add and ReLU (agcn.py:135-136)."""

    @staticmethod
    def forward(ctx, o, x_res, spec, *params):
        store = _store(ctx, spec)
        out = tcn_forward(o, x_res, *params, spec, store)
        ctx.spec, ctx.params = spec, params
        _stash(ctx, store)
        return out

    @staticmethod
    def backward(ctx, d_out):
        spec, p = ctx.spec, ctx.params
        d_o, d_xres, g = tcn_backward(d_out.contiguous(), _unstash(ctx), p[2], p[6], spec,
                                      need_dres=ctx.needs_input_grad[1], need_do=ctx.needs_input_grad[0])
        return (d_o, d_xres, None, *_tcn_grad_tuple(g))


class UnitFn(torch.autograd.Function):
    """SpatialTemporalConv.forward (agcn.py:134-136): relu(tcn1(gcn1(x)) + residual(x)), one autograd node so the
    three gradient contributions to x are accumulated in place by the kernels."""

    @staticmethod
    def forward(ctx, x, spec, *params):
        store = _store(ctx, spec)
        gp, tp = params[:GCN_NPARAMS], params[GCN_NPARAMS:]
        o = gcn_forward(x, *_split_gcn(gp), spec, store)
        out = tcn_forward(o, x if spec.residual != "none" else None, *tp, spec, store)
        if store is not None and store.get("o_split") is not None and store.get("o_bits") is not None and store.get("out_bits") is not None:
            # the backward reads `o` only as the ReLU mask (one bit per element) and as the weight-gradient operand (bf16 pieces):
            # the fp32 copy is not kept, so the split operand costs no activation memory
            store["o"] = None
            store["t_o"] = None
        ctx.spec, ctx.params = spec, params
        _stash(ctx, store)
        return out

    @staticmethod
    def backward(ctx, d_out):
        spec, params = ctx.spec, ctx.params
        store = _unstash(ctx)
        gp, tp = params[:GCN_NPARAMS], params[GCN_NPARAMS:]
        need_dx = ctx.needs_input_grad[0]
        d_out = d_out.contiguous()
        leaves = _Leaves(d_out)
        d_o, d_xres, tg = tcn_backward(d_out, store, tp[2], tp[6], spec, need_dres=need_dx, need_do=True, leaves=leaves)
        dx, gg = gcn_backward(d_o, store, gp[20], gp[24], gp[22], spec, dx=d_xres, need_dx=need_dx, leaves=leaves)
        leaves.join()
        return (dx, None, *_like(_gcn_grad_tuple(gg) + _tcn_grad_tuple(tg), params))


# =============================================================================== model-level pieces
class DataBnFn(torch.autograd.Function):
    """data_bn of Model.forward (agcn.py:186-188) without the two permute copies: the input (N,M,T,V,C) is already
    channels-last, BatchNorm1d channel (m, v, c) has its statistics over (n, t)."""

    @staticmethod
    def forward(ctx, x, gamma, beta, buf: BnBuffers, training: bool, sync=None):
        n, m, t, v, c = x.shape
        vc = v * c
        out = torch.empty_like(x)
        saved = []
        for mi in range(m):
            sl = slice(mi * vc, (mi + 1) * vc)
            rowmap = (n, t, m * t * vc, vc)
            xv = x[:, mi]
            sc, sh, mean, invstd = _bn_forward(xv, gamma[sl], beta[sl], BnBuffers(buf.running_mean[sl], buf.running_var[sl], buf.num_batches_tracked),
                                               training, sync, rowmap=rowmap, nbt=(mi == 0))
            K.bn_apply(xv, sc, sh, rowmap=rowmap, out=out[:, mi])
            saved.append((mean, invstd))
        ctx.x, ctx.gamma, ctx.saved, ctx.training, ctx.sync = x, gamma, saved, training, sync
        return out.view(n * m, t, v, c)

    @staticmethod
    def backward(ctx, d_out):
        x, gamma = ctx.x, ctx.gamma
        n, m, t, v, c = x.shape
        vc = v * c
        d_out = d_out.contiguous().view(n, m, t, v, c)
        need_dx = ctx.needs_input_grad[0]
        dx = torch.empty_like(x) if need_dx else None
        dgamma = torch.empty_like(gamma)
        dbeta = torch.empty_like(gamma)
        for mi in range(m):
            sl = slice(mi * vc, (mi + 1) * vc)
            rowmap = (n, t, m * t * vc, vc)
            mean, invstd = ctx.saved[mi]
            _, dg, db, _ = K.bn_bwd(d_out[:, mi], None, x[:, mi], mean, invstd, gamma[sl], want_dy=need_dx,
                                    dy=dx[:, mi] if need_dx else None, rowmap=rowmap, frozen=not ctx.training, sync=ctx.sync)
            dgamma[sl] = dg
            dbeta[sl] = db
        return dx, dgamma, dbeta, None, None, None


class PoolFn(torch.autograd.Function):
    """x.view(N, M, C, -1).mean(3).mean(1) (agcn.py:194-196) on a channels-last tensor [N*M, T, V, C] -> [N, C]."""

    @staticmethod
    def forward(ctx, x, groups: int):
        ctx.shape = tuple(x.shape)
        return K.pool_fwd(x, groups)

    @staticmethod
    def backward(ctx, d_out):
        return K.pool_bwd(d_out.contiguous(), ctx.shape), None


class LinearFn(torch.autograd.Function):
    """fc (agcn.py:198-199) through the same contraction kernel (rows = batch)."""

    @staticmethod
    def forward(ctx, x, w, b, precision: int):
        n, cin = x.shape
        ctx.save_for_backward(x, w)
        ctx.precision = precision
        ctx.has_bias = b is not None
        y = K.conv_fwd(x.view(1, 1, n, cin), w.view(w.shape[0], 1, cin), b, precision=precision)
        return y.view(n, w.shape[0])

    @staticmethod
    def backward(ctx, dy):
        x, w = ctx.saved_tensors
        n, cin = x.shape
        cout = w.shape[0]
        dy4 = dy.contiguous().view(1, 1, n, cout)
        dw, db = K.conv_wgrad(dy4, x.view(1, 1, n, cin), want_bias=ctx.has_bias, precision=ctx.precision)
        dx = None
        if ctx.needs_input_grad[0]:
            dx = K.conv_fwd(dy4, _t(w.view(cout, 1, cin)), precision=ctx.precision).view(n, cin)
        return dx, dw.view(cout, cin), db, None


class LinearCrossEntropyFn(torch.autograd.Function):
    """fc (agcn.py:198-199) + nn.CrossEntropyLoss with default options (session.py:53, step.py:41-42) as one node:
    (features [n, cin], fc.weight, fc.bias, labels int64 [n]) -> (loss, logits).  ``logits`` is returned for the metrics and is
    not differentiable through this node."""

    @staticmethod
    def forward(ctx, x, w, b, labels):
        loss, logits, dlogits = K.linear_ce_fwd(x.contiguous(), w, b, labels)
        ctx.save_for_backward(x, w, dlogits)
        ctx.has_bias = b is not None
        ctx.mark_non_differentiable(logits)
        return loss, logits

    @staticmethod
    def backward(ctx, d_loss, _d_logits):
        x, w, dlogits = ctx.saved_tensors
        dw, db, dx = K.linear_ce_bwd(x.contiguous(), w, dlogits, d_loss.contiguous().to(torch.float32), need_dx=ctx.needs_input_grad[0],
                                     need_db=ctx.has_bias)
        return dx, dw, db, None
