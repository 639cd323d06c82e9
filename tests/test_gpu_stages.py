"""-m gpu: every C-ABI entry point against its plain-torch restatement (oracle/stages.py) on the same seeded
inputs, including ragged / odd shapes (V = 5..25, odd T, channel counts that are not multiples of 4)."""
import pytest
import torch

from helpers import rel_err
from oracle import stages as S

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def K():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from fusion_gcn_b200 import ops
    return ops


def rnd(*shape, seed=0):
    g = torch.Generator().manual_seed(seed + sum(shape))
    return torch.randn(*shape, generator=g)


def both(fn_name, K, tensors, **kw):
    ref = getattr(S, fn_name)(*[None if t is None else t.double() for t in tensors], **kw)
    out = getattr(K, fn_name)(*[None if t is None else t.cuda() for t in tensors], **kw)
    return out, ref


CONV_CASES = [  # nb, t_in, v, cin, cout, taps, stride
    (2, 12, 25, 3, 96, 1, 1), (2, 12, 25, 64, 64, 9, 1), (3, 13, 20, 16, 32, 9, 2), (2, 13, 20, 16, 32, 1, 2),
    (1, 7, 5, 515, 64, 1, 1), (2, 9, 22, 9, 16, 1, 1), (1, 1, 37, 256, 60, 1, 1), (2, 30, 25, 128, 256, 9, 2),
    (1, 300, 25, 64, 64, 9, 1), (2, 11, 20, 48, 48, 9, 1), (2, 9, 25, 32, 64, 3, 1),
    # BASELINE layer widths of the theta/phi, conv_d and temporal convolutions (half K chunks, multi-segment, 256-wide tiles)
    (2, 12, 25, 96, 64, 1, 1), (2, 20, 25, 256, 256, 9, 1), (2, 20, 25, 128, 128, 9, 1), (2, 10, 25, 768, 256, 1, 1),
    (2, 10, 25, 256, 768, 1, 1), (2, 10, 22, 384, 128, 1, 1), (2, 21, 25, 256, 256, 9, 2),
    # enough rows per CTA for several accumulator segments of the weight gradient: 256- and 192-wide tiles (master sums in the
    # partial buffer), also with two taps stacked along M
    (4, 150, 25, 256, 128, 9, 1), (4, 150, 25, 256, 64, 9, 1), (4, 120, 25, 192, 128, 9, 1)]


@pytest.mark.parametrize("mode", ["ffma", "fp32", "bf16x3"])
@pytest.mark.parametrize("nb,t_in,v,cin,cout,taps,stride", CONV_CASES)
def test_conv_fwd_dgrad_wgrad(K, nb, t_in, v, cin, cout, taps, stride, mode):
    """mode 'ffma' = AGCN_PREC_FP32_FFMA (pure FFMA kernels); mode 'fp32' = AGCN_PREC_FP32, the parity mode, which runs
    3xTF32 error-compensated tcgen05 MMAs on the shapes the tensor-core path takes (and FFMA on the rest)."""
    prec, tol = {"ffma": (K.PREC_FP32_FFMA, 3e-6), "fp32": (K.PREC_FP32, 1e-5), "bf16x3": (K.PREC_BF16X3, 4e-5)}[mode]
    # bf16x3: x = h + m to 2^-17 (two bf16 pieces), products h.h + h.m + m.h: per-stage error ~1e-5, unit-level 1e-5..3e-5
    pad = (taps - 1) // 2
    t_out = (t_in + 2 * pad - taps) // stride + 1
    x, w, b = rnd(nb, t_in, v, cin), rnd(cout, taps, cin, seed=1) * 0.1, rnd(cout, seed=2)
    y, y_ref = both("conv_fwd", K, (x, w, b), t_out=t_out, stride=stride, pad=pad, precision=prec)
    assert rel_err(y, y_ref) <= tol
    # accumulate into an existing tensor
    base = rnd(nb, t_out, v, cout, seed=3)
    acc = K.conv_fwd(x.cuda(), w.cuda(), None, t_out=t_out, stride=stride, pad=pad, out=base.cuda().clone(), accumulate=True, precision=prec)
    assert rel_err(acc, S.conv_fwd(x.double(), w.double(), None, t_out=t_out, stride=stride, pad=pad) + base.double()) <= tol
    # input gradient = transposed gather with the transposed weight
    dy = rnd(nb, t_out, v, cout, seed=4)
    wt = w.permute(2, 1, 0).contiguous()
    dx, dx_ref = both("conv_fwd", K, (dy, wt, None), t_out=t_in, stride=stride, pad=pad, transposed=True, precision=prec)
    xg = x.double().requires_grad_(True)
    (S.conv_fwd(xg, w.double(), b.double(), t_out=t_out, stride=stride, pad=pad) * dy.double()).sum().backward()
    assert rel_err(dx_ref, xg.grad) <= 1e-12            # the stage oracle itself is consistent with autograd
    assert rel_err(dx, xg.grad) <= tol
    (dw, db), (dw_ref, db_ref) = both("conv_wgrad", K, (dy, x), taps=taps, stride=stride, pad=pad, precision=prec)
    # both parity modes compute weight gradients with bf16 triple products (a leaf of the backward pass: the error does not propagate)
    assert rel_err(dw, dw_ref) <= (5e-6 if mode == "ffma" else 4e-5) and rel_err(db, db_ref) <= 5e-6


@pytest.mark.parametrize("rows,c", [(1000, 64), (4099, 256), (777, 128), (333, 192), (50, 32)])
def test_bn_apply_and_bn_bwd_bf16_pieces_are_optional_outputs(K, rows, c):
    """agcn_bn_apply / agcn_bn_bwd with their bf16-pieces output (out_split / dy_split): the fp32 results are those of the same calls
    without it bit for bit, the extra output is their (h, m) bf16 split -- the operand format of agcn_conv_wgrad_presplit; channel
    counts that are not a multiple of 64 return None in its place."""
    y, res = rnd(rows, c).cuda(), rnd(rows, c, seed=1).cuda()
    sc, sh = (rnd(c, seed=2) * 0.3 + 1).cuda(), (rnd(c, seed=3) * 0.1).cuda()
    o0, b0, sp0 = K.bn_apply(y, sc, sh, res_mode=K.RES_TENSOR, res=res, relu=True, want_mask=True)
    o1, b1, sp = K.bn_apply(y, sc, sh, res_mode=K.RES_TENSOR, res=res, relu=True, want_mask=True, want_split=True)
    assert sp0 is None
    assert torch.equal(o0, o1)
    if b0 is None:                       # (192 channels: no bit-mask layout, hence no fused pieces either)
        assert b1 is None and sp is None
        return
    assert torch.equal(b0, b1)
    dout = rnd(rows, c, seed=4).cuda()
    mean, invstd, gamma = (rnd(c, seed=5) * 0.1).cuda(), (rnd(c, seed=6).abs() + 0.5).cuda(), (rnd(c, seed=7) * 0.3 + 1).cuda()
    d0 = K.bn_bwd(dout, None, y, mean, invstd, gamma, mask_bits=b0)
    d1 = K.bn_bwd(dout, None, y, mean, invstd, gamma, mask_bits=b0, want_split=True)
    assert d0[3] is None
    assert all(torch.equal(a, b) for a, b in zip(d0[:3], d1[:3]))
    if c % 64:
        assert sp is None and d1[3] is None
        return
    assert torch.equal(sp.view(torch.int16), K.bf16_split(o0).view(torch.int16))
    assert torch.equal(d1[3].view(torch.int16), K.bf16_split(d0[0]).view(torch.int16))


@pytest.mark.parametrize("rows,c,frozen", [(1000, 64, False), (4099, 256, False), (777, 128, True), (333, 192, False), (120000, 128, False)])
def test_bn_bwd_dual_matches_two_bn_bwd_calls(K, rows, c, frozen):
    """bn_bwd_dual on agcn_bn_bwd_bits_dual (bn + down.1 of the gcn half, the temporal + residual BatchNorms of the unit): same sums in
    the same order and the same apply formula as two agcn_bn_bwd calls; layouts without a bit mask make exactly those two calls."""
    ya, yb, res = rnd(rows, c).cuda(), rnd(rows, c, seed=9).cuda(), rnd(rows, c, seed=1).cuda()
    sc, sh = (rnd(c, seed=2) * 0.3 + 1).cuda(), (rnd(c, seed=3) * 0.1).cuda()
    out, bits, _ = K.bn_apply(ya, sc, sh, res_mode=K.RES_TENSOR, res=res, relu=True, want_mask=True)
    dout = rnd(rows, c, seed=4).cuda()
    stats = [((rnd(c, seed=5 + i) * 0.1).cuda(), (rnd(c, seed=7 + i).abs() + 0.5).cuda(), (rnd(c, seed=11 + i) * 0.3 + 1).cuda()) for i in range(2)]
    a, b = (ya, *stats[0]), (yb, *stats[1])
    got = K.bn_bwd_dual(dout, a, b, mask_out=out, mask_bits=bits, frozen=frozen, want_split=True)
    wa = K.bn_bwd(dout, out, ya, *stats[0], mask_bits=bits, frozen=frozen, want_split=True)
    wb = K.bn_bwd(dout, out, yb, *stats[1], mask_bits=bits, frozen=frozen)
    if bits is None:
        assert got[3] is None and wa[3] is None
        assert all(torch.equal(g, w) for g, w in zip(got[:3] + got[4:], wa[:3] + wb[:3]))
        return
    for g, w in zip(got[:3] + got[4:], wa[:3] + wb[:3]):
        assert rel_err(g, w) <= 1e-6
    if c % 64 == 0:
        assert torch.equal(got[3].view(torch.int16), K.bf16_split(got[0]).view(torch.int16))
    else:
        assert got[3] is None


@pytest.mark.parametrize("nb,t,v,cin,cout,taps,stride", [(2, 40, 25, 64, 64, 9, 1), (4, 150, 25, 256, 128, 9, 1), (2, 31, 25, 192, 64, 1, 1),
                                                        (3, 20, 22, 128, 256, 9, 1), (2, 12, 25, 64, 192, 1, 1), (4, 150, 25, 256, 64, 9, 1),
                                                        (1, 7, 20, 96, 64, 1, 1), (4, 150, 25, 128, 128, 9, 2), (2, 21, 25, 256, 256, 9, 2),
                                                        (2, 16, 25, 128, 256, 1, 2)])
def test_weight_gradient_from_presplit_operands(K, nb, t, v, cin, cout, taps, stride):
    """agcn_conv_wgrad_presplit: the operands arrive as the bf16 pieces (h, m) the parity modes multiply; the result is the one of
    agcn_conv_wgrad in those modes bit for bit (same pieces, same MMA order), and within their tolerance of the fp64 contraction."""
    pad = (taps - 1) // 2
    t_out = (t + 2 * pad - taps) // stride + 1
    x, dy = rnd(nb, t, v, cin).cuda(), rnd(nb, t_out, v, cout, seed=4).cuda()
    xs, dys = K.bf16_split(x), K.bf16_split(dy)
    assert xs.shape == (2, nb * t * v, cin) and xs.dtype == torch.bfloat16
    assert rel_err(xs[0].float() + xs[1].float(), x.reshape(-1, cin)) <= 2 ** -16
    dw = K.conv_wgrad_presplit(dys, xs, (nb, t, v), taps=taps, stride=stride, pad=pad)
    if cin % 64 or cout % 64:
        assert dw is None
        return
    want, _ = K.conv_wgrad(dy, x, taps=taps, stride=stride, pad=pad, want_bias=False, precision=K.PREC_FP32)
    assert torch.equal(dw, want)
    ref, _ = S.conv_wgrad(dy.double().cpu(), x.double().cpu(), taps=taps, stride=stride, pad=pad)
    assert rel_err(dw, ref) <= 4e-5


@pytest.mark.parametrize("mode", ["fp32", "tf32", "bf16x3"])
@pytest.mark.parametrize("nb,t_in,v,cin,cout,taps,stride", [
    (3, 40, 25, 64, 64, 9, 1), (2, 31, 25, 192, 64, 1, 1), (4, 30, 20, 64, 128, 9, 2), (2, 24, 22, 384, 128, 1, 1),
    (2, 16, 25, 128, 256, 1, 2), (1, 12, 25, 256, 256, 9, 1), (2, 12, 25, 3, 64, 1, 1), (3, 700, 25, 64, 64, 1, 1)])
def test_conv_fwd_fused_bn_statistics(K, nb, t_in, v, cin, cout, taps, stride, mode):
    """agcn_conv_fwd_stats + agcn_bn_finalize against conv_fwd followed by bn_stats on its output (same y bit for bit; scale /
    shift / mean / invstd and the running statistics to 1e-5), including more tiles than CTAs and a shape the fused epilogue
    does not cover (cin = 3: part is None and the caller falls back)."""
    prec = {"fp32": K.PREC_FP32, "tf32": K.PREC_TF32, "bf16x3": K.PREC_BF16X3}[mode]
    pad = (taps - 1) // 2
    t_out = (t_in + 2 * pad - taps) // stride + 1
    x, w, b = rnd(nb, t_in, v, cin).cuda(), (rnd(cout, taps, cin, seed=1) * 0.1).cuda(), rnd(cout, seed=2).cuda()
    gamma, beta = (rnd(cout, seed=3) * 0.3 + 1).cuda(), (rnd(cout, seed=4) * 0.1).cuda()
    y_ref = K.conv_fwd(x, w, b, t_out=t_out, stride=stride, pad=pad, precision=prec)
    y, part = K.conv_fwd_stats(x, w, b, t_out=t_out, stride=stride, pad=pad, precision=prec)
    assert torch.equal(y, y_ref)
    if cin % 4:
        assert part is None
        return
    assert part is not None and part.shape[1:] == (4, cout)          # shifted sum | shifted sum of squares | pivot | rows per partial
    assert float(part[:, 3].sum(0).min()) == float(part[:, 3].sum(0).max()) == nb * t_out * v
    rm, rv, nbt = torch.zeros(cout).cuda(), torch.ones(cout).cuda(), torch.zeros((), dtype=torch.long).cuda()
    rm2, rv2, nbt2 = rm.clone(), rv.clone(), nbt.clone()
    got = K.bn_finalize(part, nb * t_out * v, gamma, beta, rm, rv, nbt, 0.1, 1e-5)
    ref = S.bn_stats(y_ref.double().cpu(), gamma.double().cpu(), beta.double().cpu(), rm2.double().cpu(), rv2.double().cpu(), None, 0.1, 1e-5, True)
    for a, r in zip(got, ref):
        assert rel_err(a, r) <= 1e-5
    want = K.bn_stats(y_ref, gamma, beta, rm2, rv2, nbt2, 0.1, 1e-5, True)
    for a, r in zip(got, want):
        assert rel_err(a, r) <= 1e-5
    assert rel_err(rm, rm2) <= 1e-5 and rel_err(rv, rv2) <= 1e-5 and int(nbt) == 1 == int(nbt2)


@pytest.mark.parametrize("nb,t,v,ci,nchunk", [(2, 12, 25, 16, 3), (3, 7, 20, 4, 7), (1, 30, 22, 64, 4), (2, 5, 5, 2, 1), (2, 9, 18, 3, 2)])
def test_joint_gram_score_and_dg(K, nb, t, v, ci, nchunk):
    e = rnd(nb, t, v, 6 * ci)
    kw = dict(groups=3, offa=0, stridea=2 * ci, offb=ci, strideb=2 * ci, width=ci, nchunk=nchunk)
    s, s_ref = both("joint_gram", K, (e, e), **kw)
    assert s.shape == (nb, nchunk, 3, v, v) and rel_err(s, s_ref) <= 2e-6
    x, dz = rnd(nb, t, v, ci, seed=5), rnd(nb, t, v, 3 * ci, seed=6)
    kw = dict(groups=3, offa=0, stridea=0, offb=0, strideb=ci, width=ci, nchunk=nchunk)
    dg, dg_ref = both("joint_gram", K, (x, dz), **kw)
    assert rel_err(dg, dg_ref) <= 2e-6


@pytest.mark.parametrize("mode", ["fp32", "tf32", "ffma"])
@pytest.mark.parametrize("nb,t,v,ci,nchunk", [(2, 12, 25, 16, 3), (3, 9, 20, 32, 2), (2, 7, 22, 64, 7), (1, 30, 25, 16, 1), (2, 5, 18, 32, 5)])
def test_joint_gram_tensor_core_shapes(K, nb, t, v, ci, nchunk, mode):
    """Shapes the tcgen05 gram kernel takes (score with theta|phi sharing a 32-channel row, 32/64-wide groups, dG with
    C = 4*ci channels): fp32 mode = 3xTF32 (1e-5), TF32 mode against TF32-truncated operands (1e-5) and raw operands
    (3e-3), FFMA mode = the SIMT kernel (2e-6)."""
    prec = {"fp32": K.PREC_FP32, "tf32": K.PREC_TF32, "ffma": K.PREC_FP32_FFMA}[mode]
    tol = {"fp32": 1e-5, "tf32": 3e-3, "ffma": 2e-6}[mode]
    e = rnd(nb, t, v, 6 * ci)
    kw = dict(groups=3, offa=0, stridea=2 * ci, offb=ci, strideb=2 * ci, width=ci, nchunk=nchunk)
    ec = e.cuda()            # one tensor for both operands, as in the unit (the shared theta|phi row needs a == b)
    s = K.joint_gram(ec, ec, precision=prec, **kw)
    assert rel_err(s, S.joint_gram(e.double(), e.double(), **kw)) <= tol
    if mode == "tf32":
        et = _trunc_tf32(e)
        assert rel_err(s, S.joint_gram(et.double(), et.double(), **kw)) <= 1e-5
    c = 4 * ci
    x, dz = rnd(nb, t, v, c, seed=5), rnd(nb, t, v, 3 * c, seed=6)
    kw = dict(groups=3, offa=0, stridea=0, offb=0, strideb=c, width=c, nchunk=nchunk)
    dg = K.joint_gram(x.cuda(), dz.cuda(), precision=prec, **kw)
    assert rel_err(dg, S.joint_gram(x.double(), dz.double(), **kw)) <= tol
    if mode == "tf32":
        assert rel_err(dg, S.joint_gram(_trunc_tf32(x).double(), _trunc_tf32(dz).double(), **kw)) <= 1e-5


def test_joint_gram_wide_channels(K):
    x, dz = rnd(2, 6, 25, 256), rnd(2, 6, 25, 768, seed=1)
    kw = dict(groups=3, offa=0, stridea=0, offb=0, strideb=256, width=256, nchunk=2)
    dg, dg_ref = both("joint_gram", K, (x, dz), **kw)
    assert rel_err(dg, dg_ref) <= 2e-6


@pytest.mark.parametrize("nb,v,nchunk", [(3, 25, 4), (2, 20, 1), (5, 5, 2), (2, 32, 3)])
def test_attention_fwd_bwd(K, nb, v, nchunk):
    sp, a, b = rnd(nb, nchunk, 3, v, v) * 3, rnd(3, v, v, seed=1), rnd(3, v, v, seed=2) * 0.1
    (p, g), (p_ref, g_ref) = both("attention_fwd", K, (sp, a, b), scale=0.37)
    assert rel_err(p, p_ref) <= 2e-6 and rel_err(g, g_ref) <= 2e-6
    assert torch.allclose(p.sum(dim=-2).cpu(), torch.ones(nb, 3, v), atol=1e-5)
    dgp = rnd(nb, nchunk, 3, v, v, seed=3)
    (ds, db), (ds_ref, db_ref) = both("attention_bwd", K, (dgp, p_ref.float()), scale=0.37)
    assert rel_err(ds, ds_ref) <= 5e-6 and rel_err(db, db_ref) <= 5e-6
    # autograd cross-check of the softmax backward formula
    spd = sp.double().requires_grad_(True)
    pp, gg = S.attention_fwd(spd, a.double(), b.double(), 0.37)
    dG = dgp.double().sum(1)
    (gg * dG).sum().backward()
    assert rel_err(ds_ref.unsqueeze(1).expand_as(spd.grad), spd.grad) <= 1e-6      # p was rounded to fp32 for the kernel


@pytest.mark.parametrize("mode", ["ffma", "fp32"])
@pytest.mark.parametrize("nb,t,v,w", [(2, 9, 25, 64), (2, 5, 20, 3), (1, 4, 22, 256), (3, 7, 5, 8), (2, 3, 18, 9), (1, 11, 25, 16),
                                      (3, 13, 25, 32), (2, 301, 25, 64), (5, 6, 20, 128), (2, 7, 32, 96)])
def test_joint_mix_modes(K, nb, t, v, w, mode):
    """mode 'ffma' = the FFMA kernel; 'fp32' = AGCN_PREC_FP32, which runs AGG_FWD / AGG_BWD as 3xTF32 tcgen05 MMAs when the
    width is a multiple of 32 (1e-5) and on the FFMA kernel otherwise."""
    prec, tol = (K.PREC_FP32_FFMA, 2e-6) if mode == "ffma" else (K.PREC_FP32, 1e-5)
    mats = rnd(nb, 3, v, v, seed=1)
    x = rnd(nb, t, v, w)
    z, z_ref = both("joint_mix", K, (x, mats), width=w, mode=S.MIX_AGG_FWD, precision=prec)
    assert rel_err(z, z_ref) <= tol
    dz = rnd(nb, t, v, 3 * w, seed=2)
    dx, dx_ref = both("joint_mix", K, (dz, mats), width=w, mode=S.MIX_AGG_BWD, precision=prec)
    assert rel_err(dx, dx_ref) <= tol
    base = rnd(nb, t, v, w, seed=3)
    acc = K.joint_mix(dz.cuda(), mats.cuda(), width=w, mode=K.MIX_AGG_BWD, out=base.cuda().clone(), accumulate=True, precision=prec)
    assert rel_err(acc, dx_ref + base.double()) <= tol
    e = rnd(nb, t, v, 6 * w, seed=4)
    de, de_ref = both("joint_mix", K, (e, mats), width=w, mode=S.MIX_SCORE_BWD, precision=prec)
    assert rel_err(de, de_ref) <= (tol if w % 16 == 0 else 2e-6)       # widths that are multiples of 16 run on the tensor cores


@pytest.mark.parametrize("mode", ["fp32", "tf32"])
@pytest.mark.parametrize("nb,t,v,w", [(2, 9, 25, 16), (3, 301, 25, 32), (2, 75, 22, 64), (130, 40, 25, 16), (2, 7, 20, 24)])
def test_score_backward_mix_with_fused_bias_gradient(K, nb, t, v, w, mode):
    """agcn_joint_mix_score_bwd_colsum: the same de as agcn_joint_mix(SCORE_BWD), bit for bit, plus its column sums (the theta / phi
    bias gradient) from the epilogue; widths outside the fused path (24) return None and the caller sums separately."""
    prec = K.PREC_FP32 if mode == "fp32" else K.PREC_TF32
    e, ds = rnd(nb, t, v, 6 * w).cuda(), rnd(nb, 3, v, v, seed=1).cuda()
    ref = K.joint_mix(e, ds, width=w, mode=K.MIX_SCORE_BWD, precision=prec)
    de, cs = K.joint_mix_score_bwd(e, ds, width=w, precision=prec)
    assert torch.equal(de, ref)
    if w == 24:
        assert cs is None
        return
    want = ref.double().reshape(-1, 6 * w).sum(0)
    assert cs.shape == (6 * w,) and rel_err(cs, want) <= 2e-6


@pytest.mark.parametrize("nb,t,v,w", [(2, 9, 25, 64), (3, 13, 20, 32), (1, 40, 22, 128)])
def test_joint_mix_tf32_mode(K, nb, t, v, w):
    """AGCN_PREC_TF32: the tensor-core mix sees TF32-truncated operands (1e-5 against that, 3e-3 against the raw operands)."""
    mats = rnd(nb, 3, v, v, seed=1)
    x = rnd(nb, t, v, w)
    z = K.joint_mix(x.cuda(), mats.cuda(), width=w, mode=K.MIX_AGG_FWD, precision=K.PREC_TF32)
    assert rel_err(z, S.joint_mix(_trunc_tf32(x).double(), _trunc_tf32(mats).double(), width=w, mode=S.MIX_AGG_FWD)) <= 1e-5
    assert rel_err(z, S.joint_mix(x.double(), mats.double(), width=w, mode=S.MIX_AGG_FWD)) <= 3e-3
    dz = rnd(nb, t, v, 3 * w, seed=2)
    dx = K.joint_mix(dz.cuda(), mats.cuda(), width=w, mode=K.MIX_AGG_BWD, precision=K.PREC_TF32)
    assert rel_err(dx, S.joint_mix(_trunc_tf32(dz).double(), _trunc_tf32(mats).double(), width=w, mode=S.MIX_AGG_BWD)) <= 1e-5
    ci = max(16, w // 4)                # the score backward runs on the tensor cores for widths that are multiples of 16
    e = rnd(nb, t, v, 6 * ci, seed=3)
    de = K.joint_mix(e.cuda(), mats.cuda(), width=ci, mode=K.MIX_SCORE_BWD, precision=K.PREC_TF32)
    assert rel_err(de, S.joint_mix(_trunc_tf32(e).double(), _trunc_tf32(mats).double(), width=ci, mode=S.MIX_SCORE_BWD)) <= 1e-5


@pytest.mark.parametrize("rows,c", [(20000, 64), (3001, 12), (9000, 256)])
def test_bn_statistics_of_channels_with_mean_far_from_zero(K, rows, c):
    """|mean| >> sigma (raw coordinates, near-constant channels): E[x^2] - mean^2 in fp32 loses (mean/sigma)^2 x 1e-6 of the variance
    -- at mean 100, sigma 0.1 everything.  The sums are shifted by a pivot (first row / running mean), like Welford in torch."""
    x = (rnd(rows, c) * 0.1 + 100.0)
    gamma, beta = rnd(c, seed=1) * 0.3 + 1, rnd(c, seed=2) * 0.1
    ref = S.bn_stats(x.double(), gamma.double(), beta.double(), torch.zeros(c).double(), torch.ones(c).double(), None, 0.1, 1e-5, True)
    rm, rv = torch.zeros(c).cuda(), torch.ones(c).cuda()
    out = K.bn_stats(x.cuda(), gamma.cuda(), beta.cuda(), rm, rv, None, 0.1, 1e-5, True)
    assert rel_err(out[3], ref[3]) <= 2e-5 and rel_err(out[2], ref[2]) <= 1e-6 and rel_err(out[0], ref[0]) <= 2e-5      # invstd, mean, scale
    assert rel_err(rv, 0.9 + 0.1 * x.double().var(dim=0, unbiased=True)) <= 1e-5
    if c % 32 == 0:
        # the same through the convolution epilogues (1x1: TMA-store path, 9 taps: per-warp staging path): an identity-like conv with a
        # large bias; every partial shifts its sums by the first value it sees and agcn_bn_finalize merges them pairwise in fp64
        nb, t, v = 2, rows // 50, 25
        xi = rnd(nb, t, v, c).cuda() * 0.1
        for taps in (1, 9):
            w = torch.zeros(c, taps, c)
            w[:, taps // 2] = torch.eye(c)
            b = torch.full((c,), 100.0).cuda()
            y, part = K.conv_fwd_stats(xi, w.cuda(), b, pad=taps // 2, precision=K.PREC_FP32)
            assert part is not None
            rm2, rv2 = torch.zeros(c).cuda(), torch.ones(c).cuda()
            got = K.bn_finalize(part, nb * t * v, gamma.cuda(), beta.cuda(), rm2, rv2, None, 0.1, 1e-5)
            yd = y.double().cpu().reshape(-1, c)
            invstd_ref = 1.0 / torch.sqrt(yd.var(dim=0, unbiased=False) + 1e-5)
            assert rel_err(got[3], invstd_ref) <= 2e-5 and rel_err(got[2], yd.mean(0)) <= 1e-6, taps
            assert rel_err(rm2, 0.1 * yd.mean(0)) <= 1e-6 and rel_err(rv2, 0.9 + 0.1 * yd.var(dim=0, unbiased=True)) <= 1e-5


@pytest.mark.parametrize("rows,c", [(1000, 64), (777, 3), (4099, 256), (300, 515), (50, 12), (9000, 128), (64, 8)])
def test_bn_stats_apply_bwd_against_the_oracle(K, rows, c):
    x = rnd(rows, c) * 2 + 0.5
    gamma, beta = rnd(c, seed=1) * 0.3 + 1, rnd(c, seed=2) * 0.1
    rm, rv = rnd(c, seed=3) * 0.1, rnd(c, seed=4).abs() + 0.5
    nbt = torch.zeros((), dtype=torch.long)
    d = lambda t: t.double().clone()
    c_ = lambda t: t.cuda().clone()
    rm_c, rv_c, nbt_c = c_(rm), c_(rv), nbt.cuda()
    rm_d, rv_d, nbt_d = d(rm), d(rv), nbt.clone()
    out = K.bn_stats(c_(x), c_(gamma), c_(beta), rm_c, rv_c, nbt_c, 0.1, 1e-5, True)
    ref = S.bn_stats(d(x), d(gamma), d(beta), rm_d, rv_d, nbt_d, 0.1, 1e-5, True)
    for a, b in zip(out, ref):
        assert rel_err(a, b) <= 5e-6
    assert rel_err(rm_c, rm_d) <= 2e-6 and rel_err(rv_c, rv_d) <= 2e-6 and int(nbt_c) == 1
    ev = K.bn_stats(c_(x), c_(gamma), c_(beta), rm_c, rv_c, nbt_c, 0.1, 1e-5, False)
    ev_ref = S.bn_stats(d(x), d(gamma), d(beta), rm_d, rv_d, nbt_d, 0.1, 1e-5, False)
    assert rel_err(ev[0], ev_ref[0]) <= 5e-6 and rel_err(ev[1], ev_ref[1]) <= 5e-6 and int(nbt_c) == 1
    sc, sh, mean, invstd = ref
    res = rnd(rows, c, seed=5)
    sc2, sh2 = rnd(c, seed=6), rnd(c, seed=7)
    for mode, relu in ((S.RES_NONE, False), (S.RES_TENSOR, True), (S.RES_AFFINE, True)):
        kw = dict(res_mode=mode, res=res, scale2=sc2, shift2=sh2, relu=relu)
        o = K.bn_apply(c_(x), sc.float().cuda(), sh.float().cuda(), **{k: (v.cuda() if torch.is_tensor(v) else v) for k, v in kw.items()})[0]
        o_ref = S.bn_apply(d(x), sc, sh, **{k: (v.double() if torch.is_tensor(v) else v) for k, v in kw.items()})[0]
        assert rel_err(o, o_ref) <= 2e-6
    dout, mask = rnd(rows, c, seed=8), rnd(rows, c, seed=9)
    dres0 = rnd(rows, c, seed=10)
    for use_mask, acc in ((True, False), (False, True)):
        dres_c, dres_d = c_(dres0), d(dres0)
        mk = mask if use_mask else None
        dy, dg, db, _ = K.bn_bwd(c_(dout), None if mk is None else c_(mk), c_(x), mean.float().cuda(), invstd.float().cuda(), c_(gamma),
                                 dres=dres_c, dres_accumulate=acc)
        dy_r, dg_r, db_r, _ = S.bn_bwd(d(dout), None if mk is None else d(mk), d(x), mean, invstd, d(gamma), dres=dres_d, dres_accumulate=acc)
        assert rel_err(dy, dy_r) <= 1e-5 and rel_err(dg, dg_r) <= 1e-5 and rel_err(db, db_r) <= 1e-5
        assert rel_err(dres_c, dres_d) <= 1e-6


def test_bn_rowmap_data_bn_addressing(K):
    n, m, t, v, c = 3, 2, 7, 5, 3
    x = rnd(n, m, t, v, c)
    vc = v * c
    xc = x.cuda()
    for mi in range(m):
        rowmap = (n, t, m * t * vc, vc)
        out = K.bn_stats(xc[:, mi], None, None, None, None, None, 0.1, 1e-5, True, rowmap=rowmap)
        ref = S.bn_stats(x.double()[:, mi], None, None, None, None, None, 0.1, 1e-5, True, rowmap=rowmap)
        for a, b in zip(out, ref):
            assert rel_err(a, b) <= 5e-6
        flat = x[:, mi].reshape(n * t, vc).double()
        assert rel_err(out[2], flat.mean(0)) <= 5e-6


@pytest.mark.parametrize("rows,c", [(1000, 64), (4099, 256), (777, 128), (9001, 16), (50, 12), (333, 515), (37, 32)])
def test_relu_bit_mask_from_bn_apply_matches_tensor_mask(K, rows, c):
    """agcn_bn_apply / agcn_bn_bwd with mask_bits: the ReLU mask as one bit per element gives bit-identical results to the fp32
    tensor mask (rows * c not a multiple of 32 included); unsupported layouts return no bit mask."""
    y, res = (rnd(rows, c) * 2).cuda(), rnd(rows, c, seed=1).cuda()
    sc, sh = (rnd(c, seed=2) * 0.3 + 1).cuda(), (rnd(c, seed=3) * 0.1).cuda()
    out_ref, no_bits, _ = K.bn_apply(y, sc, sh, res_mode=K.RES_TENSOR, res=res, relu=True)
    out, bits, _ = K.bn_apply(y, sc, sh, res_mode=K.RES_TENSOR, res=res, relu=True, want_mask=True)
    assert no_bits is None
    assert torch.equal(out, out_ref)
    if c % 4 or 256 % (c // 4):
        assert bits is None
        return
    assert bits is not None and bits.numel() == (rows * c + 31) // 32
    flat = (out_ref > 0).flatten().cpu()
    pad = torch.zeros(bits.numel() * 32, dtype=torch.bool)
    pad[:flat.numel()] = flat
    want = (pad.view(-1, 32).long() << torch.arange(32)).sum(1)
    assert torch.equal(bits.cpu().long() & 0xFFFFFFFF, want)
    dout, mean, invstd, gamma = rnd(rows, c, seed=4).cuda(), (rnd(c, seed=5) * 0.1).cuda(), (rnd(c, seed=6).abs() + 0.5).cuda(), (rnd(c, seed=7) + 1).cuda()
    for acc in (False, True):
        dres_a, dres_b = rnd(rows, c, seed=8).cuda(), rnd(rows, c, seed=8).cuda()
        a = K.bn_bwd(dout, out_ref, y, mean, invstd, gamma, dres=dres_a, dres_accumulate=acc)
        b = K.bn_bwd(dout, None, y, mean, invstd, gamma, dres=dres_b, dres_accumulate=acc, mask_bits=bits)
        assert a[3] is None and b[3] is None
        for u, v in zip(a[:3], b[:3]):
            assert torch.equal(u, v)
        assert torch.equal(dres_a, dres_b)


@pytest.mark.parametrize("groups,rows,c", [(4, 100, 256), (3, 37, 60), (2, 1, 8)])
def test_pool(K, groups, rows, c):
    x = rnd(groups * rows, c).view(groups, rows, c)
    o, o_ref = both("pool_fwd", K, (x,), groups=groups)
    assert rel_err(o, o_ref) <= 2e-6
    dout = rnd(groups, c, seed=1)
    dx = K.pool_bwd(dout.cuda(), (groups, rows, c))
    assert rel_err(dx, S.pool_bwd(dout.double(), (groups, rows, c))) <= 2e-6


def test_error_paths_raise(K):
    with pytest.raises(RuntimeError, match="CUDA"):
        K.conv_fwd(torch.randn(1, 2, 3, 4), torch.randn(4, 1, 4).cuda())
    with pytest.raises(RuntimeError, match="status 2"):       # graphs with more than 32 nodes reduce their gram in ONE chunk
        e = torch.randn(1, 4, 40, 8).cuda()
        K.joint_gram(e, e, groups=1, offa=0, stridea=0, offb=0, strideb=0, width=8, nchunk=2)


def _trunc_tf32(t):
    return (t.view(torch.int32) & ~0x1FFF).view(torch.float32)


TC_CASES = [  # nb, t_in, v, cin, cout, taps, stride  (shapes the tcgen05 path takes; others fall back to FFMA)
    (2, 20, 25, 64, 64, 9, 1), (2, 21, 25, 64, 128, 9, 2), (2, 12, 25, 16, 96, 1, 1), (2, 14, 20, 64, 128, 9, 1),
    (1, 10, 25, 768, 256, 1, 1), (2, 14, 22, 32, 32, 9, 1), (2, 20, 18, 128, 256, 1, 2), (2, 11, 20, 48, 48, 9, 1),
    (2, 9, 25, 32, 64, 3, 1)]


@pytest.mark.parametrize("nb,t_in,v,cin,cout,taps,stride", TC_CASES)
def test_tf32_tensor_core_path(K, nb, t_in, v, cin, cout, taps, stride):
    """AGCN_PREC_TF32 (tcgen05.mma kind::tf32): the hardware truncates fp32 operands to TF32, so against an fp64
    contraction of TF32-truncated inputs the result must be fp32-accumulation exact (1e-5); against the raw inputs the
    stated TF32 tolerance is 3e-3."""
    pad = (taps - 1) // 2
    t_out = (t_in + 2 * pad - taps) // stride + 1
    x, w, b = rnd(nb, t_in, v, cin), rnd(cout, taps, cin, seed=1) * 0.1, rnd(cout, seed=2)
    kw = dict(t_out=t_out, stride=stride, pad=pad)
    y = K.conv_fwd(x.cuda(), w.cuda(), b.cuda(), precision=K.PREC_TF32, **kw)
    assert rel_err(y, S.conv_fwd(_trunc_tf32(x).double(), _trunc_tf32(w).double(), b.double(), **kw)) <= 1e-5
    assert rel_err(y, S.conv_fwd(x.double(), w.double(), b.double(), **kw)) <= 3e-3
    dy = rnd(nb, t_out, v, cout, seed=4)
    wt = w.permute(2, 1, 0).contiguous()
    kw_t = dict(t_out=t_in, stride=stride, pad=pad, transposed=True)
    base = rnd(nb, t_in, v, cin, seed=5)
    dx = K.conv_fwd(dy.cuda(), wt.cuda(), None, out=base.cuda().clone(), accumulate=True, precision=K.PREC_TF32, **kw_t)
    # (a 1x1 stride-2 input gradient has an empty parity class: the tensor-core kernel skips it, those rows keep `base`)
    assert rel_err(dx, S.conv_fwd(_trunc_tf32(dy).double(), _trunc_tf32(wt).double(), None, **kw_t) + base.double()) <= 1e-5
    assert rel_err(dx, S.conv_fwd(dy.double(), wt.double(), None, **kw_t) + base.double()) <= 3e-3
    dw, db = K.conv_wgrad(dy.cuda(), x.cuda(), taps=taps, stride=stride, pad=pad, precision=K.PREC_TF32)
    dw_ref, db_ref = S.conv_wgrad(_trunc_tf32(dy).double(), _trunc_tf32(x).double(), taps=taps, stride=stride, pad=pad)
    assert rel_err(dw, dw_ref) <= 2e-5
    assert rel_err(db, S.conv_wgrad(dy.double(), x.double(), taps=taps, stride=stride, pad=pad)[1]) <= 5e-6


@pytest.mark.parametrize("groups,rpg,c,res_mode", [(4, 75, 256, 1), (3, 50, 64, 2), (2, 33, 128, 0), (64, 3750, 256, 1)])
def test_bn_apply_pool_tail_and_pooled_bn_bwd(K, groups, rpg, c, res_mode):
    """agcn_bn_apply_pool / agcn_bn_bwd with pool_rows (the model's fused tail) against bn_apply + pool_fwd and pool_bwd + bn_bwd."""
    rows = groups * rpg
    assert K.bn_pool_supported(rows, c)
    y, res = rnd(rows, c).cuda(), rnd(rows, c, seed=1).cuda()
    sc, sh = (rnd(c, seed=2) * 0.3 + 1).cuda(), (rnd(c, seed=3) * 0.2).cuda()
    sc2, sh2 = (rnd(c, seed=4) * 0.3 + 1).cuda(), (rnd(c, seed=5) * 0.2).cuda()
    kw = dict(res_mode=res_mode, res=res if res_mode else None, scale2=sc2 if res_mode == 2 else None, shift2=sh2 if res_mode == 2 else None)
    pooled, bits = K.bn_apply_pool(y, sc, sh, groups=groups, **kw)
    out, bits_ref, _ = K.bn_apply(y, sc, sh, relu=True, want_mask=True, **kw)
    assert torch.equal(bits, bits_ref)
    assert rel_err(pooled, out.double().reshape(groups, rpg, c).mean(1)) <= 2e-6
    d_pooled = rnd(groups, c, seed=6).cuda()
    mean, invstd, gamma = (rnd(c, seed=7) * 0.1).cuda(), (rnd(c, seed=8).abs() + 0.5).cuda(), (rnd(c, seed=9) * 0.3 + 1).cuda()
    d_full = K.pool_bwd(d_pooled, (rows, c))
    dres_a, dres_b = torch.empty_like(y), torch.empty_like(y)
    got = K.bn_bwd(d_pooled, None, y, mean, invstd, gamma, dres=dres_a, mask_bits=bits, pool_rows=rpg)
    want = K.bn_bwd(d_full, None, y, mean, invstd, gamma, dres=dres_b, mask_bits=bits)
    assert got[3] is None and want[3] is None
    for a, b in zip(got[:3], want[:3]):
        assert rel_err(a, b) <= 2e-6
    assert rel_err(dres_a, dres_b) <= 1e-6


@pytest.mark.parametrize("n,cin,ncls", [(64, 256, 60), (3, 64, 27), (16, 1024, 35), (1, 32, 5)])
def test_linear_cross_entropy_head(K, n, cin, ncls):
    x, w, b = rnd(n, cin), rnd(ncls, cin, seed=1) * 0.2, rnd(ncls, seed=2)
    labels = torch.randint(0, ncls, (n,), generator=torch.Generator().manual_seed(3))
    loss, logits, dlogits = K.linear_ce_fwd(x.cuda(), w.cuda(), b.cuda(), labels.cuda())
    xr, wr, br = x.double().requires_grad_(True), w.double().requires_grad_(True), b.double().requires_grad_(True)
    lr = torch.nn.functional.linear(xr, wr, br)
    loss_ref = torch.nn.functional.cross_entropy(lr, labels)
    (loss_ref * 1.7).backward()
    assert rel_err(logits, lr) <= 2e-6 and abs(float(loss) - float(loss_ref)) <= 2e-6 * max(1.0, abs(float(loss_ref)))
    dw, db, dx = K.linear_ce_bwd(x.cuda(), w.cuda(), dlogits, torch.tensor(1.7).cuda())
    assert rel_err(dw, wr.grad) <= 5e-6 and rel_err(db, br.grad) <= 5e-6 and rel_err(dx, xr.grad) <= 5e-6


@pytest.mark.parametrize("mode", ["ffma", "fp32", "bf16x3", "tf32"])
@pytest.mark.parametrize("nb,t_in,v,cin,cout,taps,stride,with_res", [
    (2, 12, 25, 192, 64, 1, 1, True), (2, 20, 25, 64, 64, 9, 1, True), (2, 21, 25, 128, 256, 9, 2, True), (3, 9, 20, 3, 64, 1, 1, False),
    (2, 10, 25, 768, 256, 1, 1, True), (2, 16, 22, 64, 128, 1, 2, False)])
def test_conv_fwd_post_eval_tail(K, nb, t_in, v, cin, cout, taps, stride, with_res, mode):
    """agcn_conv_fwd_post: act(scale * (conv + bias) + shift + res) in the convolution's epilogue (both tensor-core epilogues and
    the FFMA kernel) against the separate stage oracle."""
    prec, tol = {"ffma": (K.PREC_FP32_FFMA, 3e-6), "fp32": (K.PREC_FP32, 1e-5), "bf16x3": (K.PREC_BF16X3, 4e-5), "tf32": (K.PREC_TF32, 2e-3)}[mode]
    pad = (taps - 1) // 2
    t_out = (t_in + 2 * pad - taps) // stride + 1
    x, w, b = rnd(nb, t_in, v, cin), rnd(cout, taps, cin, seed=1) * 0.1, rnd(cout, seed=2)
    sc, sh = rnd(cout, seed=3) * 0.3 + 1, rnd(cout, seed=4) * 0.2
    res = rnd(nb, t_out, v, cout, seed=5) if with_res else None
    for relu in (False, True):
        y = K.conv_fwd_post(x.cuda(), w.cuda(), b.cuda(), scale=sc.cuda(), shift=sh.cuda(), res=None if res is None else res.cuda(), relu=relu,
                            t_out=t_out, stride=stride, pad=pad, precision=prec)
        ref = S.conv_fwd_post(x.double(), w.double(), b.double(), scale=sc.double(), shift=sh.double(), res=None if res is None else res.double(),
                              relu=relu, t_out=t_out, stride=stride, pad=pad)
        assert rel_err(y, ref) <= tol
    y = K.conv_fwd_post(x.cuda(), w.cuda(), None, res=None if res is None else res.cuda(), t_out=t_out, stride=stride, pad=pad, precision=prec)
    ref = S.conv_fwd_post(x.double(), w.double(), None, res=None if res is None else res.double(), t_out=t_out, stride=stride, pad=pad)
    assert rel_err(y, ref) <= tol
