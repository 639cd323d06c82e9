"""Kernel contracts that the stage tests leave open, each against the fp64 stage oracle (oracle/stages.py) on the CPU:

* accumulate in every joint-mix mode, for the resident kernels (V <= 32) and the batched GEMMs of large graphs (V > 32), plus the
  large-graph gram, attention and node mix at the edges of the 64 x 64 GEMM tiles and with many timesteps;
* synchronised BatchNorm over shards with different means and row counts, simulated in one process: the mergeable partials of
  agcn_bn_stats_partials / agcn_conv_fwd_stats, their merge in agcn_bn_finalize, and the two phases of agcn_bn_bwd;
* the one-launch pack / unpack of the data-parallel gradient buckets (agcn_bucket_copy).

Everything except the CPU anchor of the partials merge needs a GPU (-m gpu)."""
import math

import pytest
import torch

from helpers import rel_err
from oracle import stages as S


@pytest.fixture(scope="module")
def K():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from fusion_gcn_b200 import ops
    return ops


def rnd(*shape, seed=0):
    g = torch.Generator().manual_seed(seed + sum(shape))
    return torch.randn(*shape, generator=g)


def _trunc_tf32(t):
    return (t.contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)


# ============================================================================================ joint mix with accumulate, all V
MIX_CASES = [  # nb, t, v, width: resident kernels (V <= 32), then the batched GEMMs (V > 32) around their 64-row / 64-column tiles
    (3, 5, 5, 3), (3, 6, 25, 32), (3, 1, 32, 16), (4, 7, 25, 65), (3, 5, 32, 1),
    (3, 5, 33, 16), (3, 1, 63, 65), (3, 6, 64, 32), (3, 5, 65, 3), (3, 1, 129, 1), (3, 5, 129, 65)]
MIX_MODES = {"agg_fwd": S.MIX_AGG_FWD, "agg_bwd": S.MIX_AGG_BWD, "score_bwd": S.MIX_SCORE_BWD}
MIX_LD = {S.MIX_AGG_FWD: (1, 3), S.MIX_AGG_BWD: (3, 1), S.MIX_SCORE_BWD: (6, 6)}          # (ldin, ldout) in widths


def _mix_on_tensor_cores(mode, precision, v, w, accumulate):
    """Whether agcn_joint_mix runs on the tcgen05 kernel (mix_tc.cu); every other call runs an FFMA kernel, exact fp32."""
    if precision == S.PREC_FP32_FFMA or v > 32:
        return False
    if accumulate and mode != S.MIX_AGG_BWD:
        return False                     # the tensor-core mix accumulates only in AGG_BWD; the others fall back to the FFMA kernel
    return w % (16 if mode == S.MIX_SCORE_BWD else 32) == 0


def _mix_reference(inp, mats, w, mode, precision, on_tc):
    """(fp64 reference, tolerance): TF32 on the tensor cores is held to fp32 accuracy against TF32-truncated operands."""
    if on_tc and precision == S.PREC_TF32:
        return S.joint_mix(_trunc_tf32(inp).double(), _trunc_tf32(mats).double(), width=w, mode=mode), 1e-5
    return S.joint_mix(inp.double(), mats.double(), width=w, mode=mode), (1e-5 if on_tc else 2e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MIX_MODES))
@pytest.mark.parametrize("prec", ["ffma", "fp32", "tf32"])
@pytest.mark.parametrize("nb,t,v,w", MIX_CASES)
def test_joint_mix_accumulates_in_every_mode(K, nb, t, v, w, mode, prec):
    """agcn_joint_mix(accumulate=1) adds into `out` in every mode and for every V; accumulate=0 overwrites an `out` full of NaN."""
    mode, precision = MIX_MODES[mode], {"ffma": K.PREC_FP32_FFMA, "fp32": K.PREC_FP32, "tf32": K.PREC_TF32}[prec]
    ld_in, ld_out = MIX_LD[mode]
    inp, mats, base = rnd(nb, t, v, ld_in * w), rnd(nb, 3, v, v, seed=1), rnd(nb, t, v, ld_out * w, seed=2)
    on_tc = _mix_on_tensor_cores(mode, precision, v, w, True)
    ref, tol = _mix_reference(inp, mats, w, mode, precision, on_tc)
    acc = K.joint_mix(inp.cuda(), mats.cuda(), width=w, mode=mode, out=base.cuda(), accumulate=True, precision=precision)
    assert rel_err(acc, ref + base.double()) <= tol
    on_tc = _mix_on_tensor_cores(mode, precision, v, w, False)
    ref, tol = _mix_reference(inp, mats, w, mode, precision, on_tc)
    out = torch.full((nb, t, v, ld_out * w), float("nan"), device="cuda")
    fresh = K.joint_mix(inp.cuda(), mats.cuda(), width=w, mode=mode, out=out, accumulate=False, precision=precision)
    assert rel_err(fresh, ref) <= tol


GRAPH_CASES = [  # nb, t, v, ci: V = 32 on the resident kernels against V = 33 on the GEMMs, tile edges at 63 / 64 / 65 / 129 nodes
    (3, 9, 32, 3), (3, 5, 33, 16), (3, 1, 63, 65), (3, 6, 64, 1), (4, 5, 65, 32), (3, 7, 129, 3)]


@pytest.mark.gpu
@pytest.mark.parametrize("nb,t,v,ci", GRAPH_CASES)
def test_large_graph_gram_and_attention(K, nb, t, v, ci):
    """agcn_joint_gram in score form (theta | phi sharing one row) and dG form (stridea = 0, one segment per timestep), and
    agcn_attention_fwd / _bwd with several samples summed into dadj_b."""
    nchunk = K.pick_nchunk(nb, t, v, ci)
    e = rnd(nb, t, v, 6 * ci)
    kw = dict(groups=3, offa=0, stridea=2 * ci, offb=ci, strideb=2 * ci, width=ci, nchunk=nchunk)
    ec = e.cuda()
    s = K.joint_gram(ec, ec, **kw)
    assert s.shape == (nb, nchunk, 3, v, v) and rel_err(s, S.joint_gram(e.double(), e.double(), **kw)) <= 2e-6
    c = 4 * ci
    x, dz = rnd(nb, t, v, c, seed=1), rnd(nb, t, v, 3 * c, seed=2)
    kw = dict(groups=3, offa=0, stridea=0, offb=0, strideb=c, width=c, nchunk=nchunk)
    dg = K.joint_gram(x.cuda(), dz.cuda(), **kw)
    assert rel_err(dg, S.joint_gram(x.double(), dz.double(), **kw)) <= 2e-6
    sp, a, b = rnd(nb, nchunk, 3, v, v, seed=3) * 3, rnd(3, v, v, seed=4), rnd(3, v, v, seed=5) * 0.1
    p, g = K.attention_fwd(sp.cuda(), a.cuda(), b.cuda(), 0.37)
    p_ref, g_ref = S.attention_fwd(sp.double(), a.double(), b.double(), 0.37)
    assert rel_err(p, p_ref) <= 2e-6 and rel_err(g, g_ref) <= 2e-6
    dgp = rnd(nb, nchunk, 3, v, v, seed=6)
    ds, dadj = K.attention_bwd(dgp.cuda(), p, 0.37)
    ds_ref, dadj_ref = S.attention_bwd(dgp.double(), p.double().cpu(), 0.37)
    assert rel_err(ds, ds_ref) <= 5e-6 and rel_err(dadj, dadj_ref) <= 2e-6


@pytest.mark.gpu
@pytest.mark.parametrize("accumulate", [False, True])
@pytest.mark.parametrize("transpose", [False, True])
@pytest.mark.parametrize("batch,v,c", [(3, 7, 5), (4, 64, 16), (3, 65, 65), (3, 300, 3)])
def test_node_mix(K, batch, v, c, transpose, accumulate):
    """agcn_node_mix: one fixed V x V matrix for the whole batch, either orientation, adding into or overwriting `out`."""
    inp, mat, base = rnd(batch, v, c), rnd(v, v, seed=1) * 0.1, rnd(batch, v, c, seed=2)
    ref = S.node_mix(inp.double(), mat.double(), transpose=transpose)
    out = base.cuda() if accumulate else torch.full((batch, v, c), float("nan"), device="cuda")
    got = K.node_mix(inp.cuda(), mat.cuda(), transpose=transpose, out=out, accumulate=accumulate)
    assert rel_err(got, ref + base.double() if accumulate else ref) <= 2e-6


# ============================================================================================ synchronised BatchNorm over shards
def _shard_offset(r):
    """Per-shard mean: about 100 with sigma 0.1 inside a shard, so the pivots of the shifted sums matter, and different between shards."""
    return 100.0 + 0.25 * (r + 1) * (-1) ** r


def _bn_params(c):
    gamma, beta = rnd(c, seed=1) * 0.3 + 1, rnd(c, seed=2) * 0.1
    rm, rv = rnd(c, seed=3) * 0.1, rnd(c, seed=4).abs() + 0.5
    return gamma, beta, rm, rv


def _check_merged_statistics(K, part, x_all, c):
    """bn_finalize over the concatenated partials against bn_stats over the whole batch, running statistics included."""
    gamma, beta, rm, rv = _bn_params(c)
    rm_c, rv_c, nbt_c = rm.cuda(), rv.cuda(), torch.zeros((), dtype=torch.long).cuda()
    rm_d, rv_d, nbt_d = rm.double(), rv.double(), torch.zeros((), dtype=torch.long)
    got = K.bn_finalize(part, x_all.shape[0], gamma.cuda(), beta.cuda(), rm_c, rv_c, nbt_c, 0.1, 1e-5)
    ref = S.bn_stats(x_all.double(), gamma.double(), beta.double(), rm_d, rv_d, nbt_d, 0.1, 1e-5, True)
    scale, shift, mean, invstd = got
    assert rel_err(scale, ref[0]) <= 2e-5 and rel_err(shift, ref[1]) <= 2e-5
    assert rel_err(mean, ref[2]) <= 1e-6 and rel_err(invstd, ref[3]) <= 2e-5
    assert rel_err(rm_c, rm_d) <= 1e-6 and rel_err(rv_c, rv_d) <= 1e-5 and int(nbt_c) == 1


@pytest.mark.gpu
@pytest.mark.parametrize("c,sizes", [(3, (4099, 3001)), (12, (20000, 64, 777)), (64, (40000, 1)), (256, (9000, 4099, 5000))])
def test_sync_bn_statistics_over_distinct_shards(K, c, sizes):
    """Each shard's agcn_bn_stats_partials, concatenated in rank order and merged by agcn_bn_finalize with the total row count, give the
    statistics of the unsharded batch: shards of unequal size (down to one row; 40000 rows leave trailing partials with no rows) whose
    means differ, so every shard's partials carry their own pivot."""
    shards = [rnd(n, c, seed=10 * r) * 0.1 + _shard_offset(r) for r, n in enumerate(sizes)]
    parts = [K.bn_stats_partials(x.cuda()) for x in shards]
    for x, part in zip(shards, parts):
        assert part.shape[1:] == (4, c) and float(part[:, 3].sum(0).min()) == float(part[:, 3].sum(0).max()) == x.shape[0]
    _check_merged_statistics(K, torch.cat(parts), torch.cat(shards), c)
    # one shard alone: the kernel's partials (layout-specific) and the oracle's single partial merge to the same statistics
    gamma, beta = (t.cuda() for t in _bn_params(c)[:2])
    got = K.bn_finalize(parts[0], sizes[0], gamma, beta, None, None, None, 0.1, 1e-5)
    ref = S.bn_finalize(S.bn_stats_partials(shards[0].double()), sizes[0], gamma.double().cpu(), beta.double().cpu(), None, None, None, 0.1, 1e-5)
    for a, r, tol in zip(got, ref, (2e-5, 2e-5, 1e-6, 2e-5)):
        assert rel_err(a, r) <= tol


@pytest.mark.gpu
@pytest.mark.parametrize("ranks", [2, 3])
def test_sync_bn_statistics_with_the_data_bn_row_map(K, ranks):
    """The same through the data-BatchNorm row map (n, t, m*t*v*c, v*c): body mi of a [n, m, t, v, c] batch, sharded along n."""
    n, m, t, v, c = 5, 2, 40, 25, 3
    vc = v * c
    x = rnd(n, m, t, v, c) * 0.1
    bounds = [0, 2, 5] if ranks == 2 else [0, 1, 3, 5]
    for r in range(ranks):
        x[bounds[r]:bounds[r + 1]] += _shard_offset(r)
    xc = x.cuda()
    for mi in range(m):
        parts = [K.bn_stats_partials(xc[n0:n1, mi], rowmap=(n1 - n0, t, m * t * vc, vc)) for n0, n1 in zip(bounds, bounds[1:])]
        _check_merged_statistics(K, torch.cat(parts), x[:, mi].reshape(n * t, vc), vc)


@pytest.mark.gpu
def test_sync_bn_statistics_from_mixed_sources(K):
    """A rank whose convolution writes the statistics in its epilogue (agcn_conv_fwd_stats, one pivot per partial) exchanges them with
    a rank that ran agcn_bn_stats_partials: both write the same layout and agcn_bn_finalize merges them, in either order."""
    nb, t, v, c = 2, 40, 25, 64
    w = torch.zeros(c, 1, c)
    w[:, 0] = torch.eye(c)
    y, conv_part = K.conv_fwd_stats((rnd(nb, t, v, c) * 0.1).cuda(), w.cuda(), torch.full((c,), _shard_offset(0)).cuda(), precision=K.PREC_FP32)
    assert conv_part is not None
    other = rnd(3001, c, seed=1) * 0.1 + _shard_offset(1)
    bn_part = K.bn_stats_partials(other.cuda())
    conv_rows = y.reshape(-1, c).cpu()
    _check_merged_statistics(K, torch.cat([conv_part, bn_part]), torch.cat([conv_rows, other]), c)
    _check_merged_statistics(K, torch.cat([bn_part, conv_part]), torch.cat([other, conv_rows]), c)


class _Totals:
    """Stands in for distributed.SyncBatchNorm in the backward of one rank: all_reduce returns the column sums of all ranks (summed by
    the test from each rank's phase 1; None: this rank's own) and keeps what this rank contributed."""

    def __init__(self, world, totals):
        self.world, self.totals, self.sent = world, totals, None

    def all_reduce(self, t):
        self.sent = t.clone()
        return t if self.totals is None else t.copy_(self.totals)


@pytest.mark.gpu
@pytest.mark.parametrize("dres_accumulate", [False, True])
@pytest.mark.parametrize("ranks,c,mask", [(2, 64, "bits"), (3, 64, "bits"), (2, 64, "tensor"), (3, 12, "tensor"), (2, 12, None)])
def test_sync_bn_backward_over_distinct_shards(K, ranks, c, mask, dres_accumulate):
    """agcn_bn_bwd phase 1 on every shard, the sums added up, then phase 2 per shard (ops.bn_bwd with a sync object): the shards' dy
    and dres are the whole-batch BatchNorm backward; dgamma / dbeta stay each shard's own sums; with bit masks at 64 channels the bf16
    pieces of dy are bf16_split(dy) bit for bit.  Equal shards, as ops.bn_bwd counts rows x world."""
    rows = 3000
    ys = [rnd(rows, c, seed=10 * r) + _shard_offset(r) for r in range(ranks)]
    y_all = torch.cat(ys)
    gamma = rnd(c, seed=1) * 0.3 + 1
    _, _, mean_d, invstd_d = S.bn_stats(y_all.double(), None, None, None, None, None, 0.1, 1e-5, True)
    mean, invstd = mean_d.float(), invstd_d.float()            # what the forward saved for the backward
    douts = [rnd(rows, c, seed=10 * r + 1) for r in range(ranks)]
    dres0 = [rnd(rows, c, seed=10 * r + 2) for r in range(ranks)]
    masks, bits = [None] * ranks, [None] * ranks
    if mask is not None:                 # the ReLU after the BatchNorm: about half of the elements pass
        sc = rnd(c, seed=3) * 0.3 + 1
        sh = rnd(c, seed=4) * 0.1 - mean * sc
        for r in range(ranks):
            masks[r], bits[r], _ = K.bn_apply(ys[r].cuda(), sc.cuda(), sh.cuda(), relu=True, want_mask=mask == "bits")
            assert (bits[r] is not None) == (mask == "bits")
        assert 0.2 < float((torch.cat(masks) > 0).float().mean()) < 0.8
    want_split = mask == "bits"
    stats = (mean.cuda(), invstd.cuda(), gamma.cuda())

    def call(r, **kw):
        return K.bn_bwd(douts[r].cuda(), masks[r] if mask == "tensor" else None, ys[r].cuda(), *stats,
                        mask_bits=bits[r], **kw)

    local = [call(r, want_dy=False, sync=_Totals(ranks, None)) for r in range(ranks)]          # phase 1 only
    totals = sum(torch.stack([db, dg]).double() for _, dg, db, _ in local).float()
    dys, dress = [], []
    for r in range(ranks):
        sync = _Totals(ranks, totals.cuda())
        dres = dres0[r].cuda()
        dy, dg, db, split = call(r, dres=dres, dres_accumulate=dres_accumulate, want_split=want_split, sync=sync)
        assert torch.equal(sync.sent, torch.stack([local[r][2], local[r][1]]))                 # phase 1 sent this shard's own sums
        assert torch.equal(dg, local[r][1]) and torch.equal(db, local[r][2])
        _, dg_ref, db_ref, _ = S.bn_bwd(douts[r].double(), None if mask is None else masks[r].double().cpu(), ys[r].double(),
                                        mean.double(), invstd.double(), gamma.double())
        assert rel_err(dg, dg_ref) <= 1e-5 and rel_err(db, db_ref) <= 1e-5
        if want_split:
            assert torch.equal(split.view(torch.int16), K.bf16_split(dy).view(torch.int16))
        else:
            assert split is None
        dys.append(dy.cpu())
        dress.append(dres.cpu())
    dres_ref = torch.cat(dres0).double()
    dy_ref, _, _, _ = S.bn_bwd(torch.cat(douts).double(), None if mask is None else torch.cat(masks).double().cpu(), y_all.double(),
                               mean.double(), invstd.double(), gamma.double(), dres=dres_ref, dres_accumulate=dres_accumulate)
    assert rel_err(torch.cat(dys), dy_ref) <= 1e-5
    assert rel_err(torch.cat(dress), dres_ref) <= 1e-6


def test_oracle_merges_partials_with_different_pivots():
    """CPU anchor of the tests above: the oracle's bn_finalize over single-partial bn_stats_partials of shards with different pivots
    (their first rows) is the fp64 mean / variance of the concatenation."""
    shards = [rnd(n, 7, seed=r) * 0.1 + _shard_offset(r) * (r + 1) for r, n in enumerate((50, 1, 333, 20))]
    x = torch.cat(shards).double()
    part = torch.cat([S.bn_stats_partials(s.double()) for s in shards])
    assert len({float(p) for p in part[:, 2, 0]}) == len(shards)
    one, zero = torch.ones(7, dtype=torch.float64), torch.zeros(7, dtype=torch.float64)
    rm, rv = zero.clone(), one.clone()
    _, _, mean, invstd = S.bn_finalize(part, x.shape[0], one, zero, rm, rv, None, 0.1, 0.0)
    assert rel_err(mean, x.mean(0)) <= 1e-12
    assert rel_err(invstd.pow(-2), x.var(0, unbiased=False)) <= 1e-12
    assert rel_err(rm, 0.1 * x.mean(0)) <= 1e-12 and rel_err(rv, 0.9 + 0.1 * x.var(0, unbiased=True)) <= 1e-12


# ============================================================================================ gradient buckets
@pytest.mark.gpu
def test_gradient_bucket_copies(K):
    """GradientAllReducer._copy on agcn_bucket_copy: one launch packs every gradient of a bucket into its flat buffer and one writes
    flat * scale back (both bit for bit: a copy and one fp32 multiply), across the 4096-element work chunks and an empty parameter;
    a reallocated gradient rebuilds the device table; a non-contiguous gradient takes the torch path with the same values."""
    from fusion_gcn_b200 import capi
    from fusion_gcn_b200.distributed import GradientAllReducer, _Bucket
    lib = capi.lib()
    chunk = lib.agcn_optim_chunk()
    shapes = [(1,), (3,), (chunk - 1,), (64, chunk // 64), (0, 5), (17, 241), (19, 647)]      # 4097 and 3 * 4096 + 5 elements
    assert [math.prod(s) for s in shapes] == [1, 3, chunk - 1, chunk, 0, chunk + 1, 3 * chunk + 5]
    params = [torch.nn.Parameter(torch.zeros(s, device="cuda")) for s in shapes]
    for i, p in enumerate(params):
        p.grad = rnd(*p.shape, seed=i).cuda()
    bucket = _Bucket(params)

    def copy(to_flat, scale, launches=1):
        before = lib.agcn_launch_count()
        GradientAllReducer._copy(bucket, to_flat, scale)
        torch.cuda.synchronize()
        assert lib.agcn_launch_count() - before == launches

    def check_pack(launches=1):
        bucket.flat.fill_(float("nan"))
        copy(True, 1.0, launches)
        assert torch.equal(bucket.flat, torch.cat([p.grad.reshape(-1) for p in params]))

    def check_unpack(scale, seed, launches=1):
        bucket.flat.copy_(rnd(bucket.numel, seed=seed).cuda())
        for p in params:
            p.grad.fill_(float("nan"))
        copy(False, scale, launches)
        for p, v in zip(params, bucket.views()):
            assert torch.equal(p.grad, (v * scale).view_as(p.grad))

    check_pack()
    for k, scale in enumerate((1.0, 0.25, 1 / 3)):
        check_unpack(scale, 100 + k)
    # a reallocated gradient: the new tensor is read and written, the old one is left alone
    old = params[3].grad
    kept = old.clone()
    params[3].grad = rnd(*shapes[3], seed=50).cuda()
    check_pack()
    check_unpack(0.25, 200)
    assert torch.equal(old, kept)
    # a non-contiguous gradient: no library launch, the same values
    params[5].grad = rnd(241, 17, seed=60).cuda().t()
    assert not params[5].grad.is_contiguous()
    check_pack(launches=0)
    check_unpack(1 / 3, 300, launches=0)
