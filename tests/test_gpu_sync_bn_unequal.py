"""-m gpu: synchronised BatchNorm over unequal shards on the CUDA library.  In one process, shards of different sizes (down to one row)
and means go through agcn_bn_finalize phase 1 (fp64 moments), are summed as the all-reduce would, and finalised by phase 2; the
backward's phase 2 reads the summed count on the device.  With two GPUs, a batch of 5 split 3/2 over NCCL against the unsharded
batch on one GPU, eagerly and as one captured CUDA graph."""
import copy
import os
import socket
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from helpers import rel_err
from oracle import stages as S

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def K():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from fusion_gcn_b200 import ops
    return ops


def rnd(*shape, seed=0):
    g = torch.Generator().manual_seed(seed + sum(shape))
    return torch.randn(*shape, generator=g)


def _offset(r):
    return 100.0 + 0.25 * (r + 1) * (-1) ** r


def _bn_params(c):
    gamma, beta = rnd(c, seed=1) * 0.3 + 1, rnd(c, seed=2) * 0.1
    rm, rv = rnd(c, seed=3) * 0.1, rnd(c, seed=4).abs() + 0.5
    return gamma, beta, rm, rv


def _moments_route(K, parts_rows, c):
    """Phase 1 per shard, the moments summed in rank order (the all-reduce), phase 2 -> (outputs, running mean, running var, nbt)."""
    total = None
    for part, rows in parts_rows:
        m = K.bn_moments(part, rows)
        assert m.dtype == torch.float64 and m.shape == (2 * c + 1,) and float(m[-1]) == rows
        total = m if total is None else total + m
    gamma, beta, rm, rv = _bn_params(c)
    rm_c, rv_c, nbt = rm.cuda(), rv.cuda(), torch.zeros((), dtype=torch.long, device="cuda")
    out = K.bn_finalize_moments(total, gamma.cuda(), beta.cuda(), rm_c, rv_c, nbt, 0.1, 1e-5)
    return out, rm_c, rv_c, nbt, total


def _check_against_whole_batch(K, parts_rows, x_all, c):
    (scale, shift, mean, invstd), rm_c, rv_c, nbt, total = _moments_route(K, parts_rows, c)
    assert float(total[-1]) == x_all.shape[0]
    gamma, beta, rm, rv = _bn_params(c)
    rm_d, rv_d, nbt_d = rm.double(), rv.double(), torch.zeros((), dtype=torch.long)
    ref = S.bn_stats(x_all.double(), gamma.double(), beta.double(), rm_d, rv_d, nbt_d, 0.1, 1e-5, True)
    assert rel_err(scale, ref[0]) <= 2e-5 and rel_err(shift, ref[1]) <= 2e-5
    assert rel_err(mean, ref[2]) <= 1e-6 and rel_err(invstd, ref[3]) <= 2e-5
    assert rel_err(rm_c, rm_d) <= 1e-6 and rel_err(rv_c, rv_d) <= 1e-5 and int(nbt) == 1


@pytest.mark.parametrize("c,sizes", [(3, (4099, 1, 3001)), (64, (40000, 1)), (256, (9000, 4099, 5000))])
def test_moments_over_unequal_shards(K, c, sizes):
    """agcn_bn_stats_partials per shard (different sizes and means), phase 1, summed moments, phase 2 == the whole batch's statistics."""
    shards = [rnd(n, c, seed=10 * r) * 0.1 + _offset(r) for r, n in enumerate(sizes)]
    parts = [(K.bn_stats_partials(x.cuda()), x.shape[0]) for x in shards]
    _check_against_whole_batch(K, parts, torch.cat(shards), c)


def test_moments_from_mixed_sources(K):
    """One shard's partials come from the convolution epilogue (agcn_conv_fwd_stats), the others from agcn_bn_stats_partials, one of
    them a single row."""
    nb, t, v, c = 2, 40, 25, 64
    w = torch.zeros(c, 1, c)
    w[:, 0] = torch.eye(c)
    y, conv_part = K.conv_fwd_stats((rnd(nb, t, v, c) * 0.1).cuda(), w.cuda(), torch.full((c,), _offset(0)).cuda(), precision=K.PREC_FP32)
    assert conv_part is not None
    others = [rnd(3001, c, seed=1) * 0.1 + _offset(1), rnd(1, c, seed=2) * 0.1 + _offset(2)]
    parts = [(conv_part, nb * t * v)] + [(K.bn_stats_partials(o.cuda()), o.shape[0]) for o in others]
    _check_against_whole_batch(K, parts, torch.cat([y.reshape(-1, c).cpu()] + others), c)


def test_moments_with_the_data_bn_row_map(K):
    """Body mi of a [n, m, t, v, c] batch through the data-BatchNorm row map, sharded 1/3/1 along n."""
    n, m, t, v, c = 5, 2, 40, 25, 3
    vc = v * c
    x = rnd(n, m, t, v, c) * 0.1
    bounds = [0, 1, 4, 5]
    for r in range(3):
        x[bounds[r]:bounds[r + 1]] += _offset(r)
    xc = x.cuda()
    for mi in range(m):
        parts = [(K.bn_stats_partials(xc[n0:n1, mi], rowmap=(n1 - n0, t, m * t * vc, vc)), (n1 - n0) * t)
                 for n0, n1 in zip(bounds, bounds[1:])]
        _check_against_whole_batch(K, parts, x[:, mi].reshape(n * t, vc), vc)


@pytest.mark.parametrize("c,sizes", [(64, (3000, 3000)), (256, (2048, 2048, 2048)), (12, (777, 777))])
def test_equal_shards_moments_route_matches_phase_0(K, c, sizes):
    """Equal shards: phase 1 + sum + phase 2 against phase 0 over the concatenated partials, within 2 fp32 ulp on mean and invstd."""
    shards = [rnd(n, c, seed=10 * r) * 0.1 + _offset(r) for r, n in enumerate(sizes)]
    parts = [K.bn_stats_partials(x.cuda()) for x in shards]
    (sc, sh, mean, invstd), rm_c, rv_c, _, _ = _moments_route(K, [(p, n) for p, n in zip(parts, sizes)], c)
    gamma, beta, rm, rv = (t.cuda() for t in _bn_params(c))
    _, _, mean0, invstd0 = K.bn_finalize(torch.cat(parts), sum(sizes), gamma, beta, rm, rv, None, 0.1, 1e-5)
    for a, b in ((mean, mean0), (invstd, invstd0)):
        ulp = torch.abs(torch.nextafter(b, torch.full_like(b, float("inf"))) - b)
        assert bool(((a - b).abs() <= 2 * ulp).all()), float(((a - b).abs() / ulp).max())
    assert rel_err(rm_c, rm) <= 1e-6 and rel_err(rv_c, rv) <= 1e-6


class _Totals:
    """Stands in for the sync object of one rank's backward: all_reduce returns the column sums of all ranks (None: this rank's own);
    ``global_rows``: the device count of all ranks' rows (None: ops.bn_bwd counts rows x world)."""

    def __init__(self, world, totals, global_rows=None):
        self.world, self.totals, self.global_rows = world, totals, global_rows

    def all_reduce(self, t):
        return t if self.totals is None else t.copy_(self.totals)


@pytest.mark.parametrize("dres_accumulate", [False, True])
@pytest.mark.parametrize("sizes,c,mask", [((3000, 1, 1999), 64, "bits"), ((2500, 700), 64, "tensor"), ((1, 4000, 33), 12, "tensor"),
                                          ((900, 2), 12, None)])
def test_backward_phase2_with_the_device_count(K, sizes, c, mask, dres_accumulate):
    """agcn_bn_bwd phase 1 per shard, the sums added, phase 2 per shard with the global count as a device scalar (the moments' count
    slot): the shards' dy and dres are the whole-batch bn_bwd; with bit masks the bf16 pieces of dy are bf16_split(dy) bit for bit."""
    ranks = len(sizes)
    ys = [rnd(n, c, seed=10 * r) + _offset(r) for r, n in enumerate(sizes)]
    y_all = torch.cat(ys)
    gamma = rnd(c, seed=1) * 0.3 + 1
    _, _, mean_d, invstd_d = S.bn_stats(y_all.double(), None, None, None, None, None, 0.1, 1e-5, True)
    mean, invstd = mean_d.float(), invstd_d.float()
    douts = [rnd(n, c, seed=10 * r + 1) for r, n in enumerate(sizes)]
    dres0 = [rnd(n, c, seed=10 * r + 2) for r, n in enumerate(sizes)]
    masks, bits = [None] * ranks, [None] * ranks
    if mask is not None:
        sc = rnd(c, seed=3) * 0.3 + 1
        sh = rnd(c, seed=4) * 0.1 - mean * sc
        for r in range(ranks):
            masks[r], bits[r], _ = K.bn_apply(ys[r].cuda(), sc.cuda(), sh.cuda(), relu=True, want_mask=mask == "bits")
            assert (bits[r] is not None) == (mask == "bits")
    want_split = mask == "bits"
    stats = (mean.cuda(), invstd.cuda(), gamma.cuda())
    count = torch.tensor([float(sum(sizes))], dtype=torch.float64, device="cuda")

    def call(r, **kw):
        return K.bn_bwd(douts[r].cuda(), masks[r] if mask == "tensor" else None, ys[r].cuda(), *stats, mask_bits=bits[r], **kw)

    local = [call(r, want_dy=False, sync=_Totals(ranks, None)) for r in range(ranks)]
    totals = sum(torch.stack([db, dg]).double() for _, dg, db, _ in local).float()
    dys, dress = [], []
    for r in range(ranks):
        dres = dres0[r].cuda()
        dy, dg, db, split = call(r, dres=dres, dres_accumulate=dres_accumulate, want_split=want_split,
                                 sync=_Totals(ranks, totals.cuda(), count))
        assert torch.equal(dg, local[r][1]) and torch.equal(db, local[r][2])
        if want_split:
            assert torch.equal(split.view(torch.int16), K.bf16_split(dy).view(torch.int16))
        dys.append(dy.cpu())
        dress.append(dres.cpu())
    m_all = None if mask is None else torch.cat([t.cpu() for t in masks]).cuda()
    dres_whole = torch.cat(dres0).cuda()
    dy_whole, _, _, _ = K.bn_bwd(torch.cat(douts).cuda(), m_all, y_all.cuda(), *stats, dres=dres_whole, dres_accumulate=dres_accumulate)
    dy_ref, _, _, _ = S.bn_bwd(torch.cat(douts).double(), None if m_all is None else m_all.double().cpu(), y_all.double(),
                               mean.double(), invstd.double(), gamma.double())
    assert rel_err(torch.cat(dys), dy_whole) <= 1e-5 and rel_err(torch.cat(dys), dy_ref) <= 1e-5
    assert torch.equal(torch.cat(dress), dres_whole.cpu())
    # the equal-shard default (rows x world) would be wrong here: the count really comes from the device scalar
    dy_eq, _, _, _ = call(0, sync=_Totals(ranks, totals.cuda()))
    assert rel_err(dy_eq.cpu(), dys[0]) > 1e-4


# ============================================================================================ two GPUs over NCCL
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


class _Weighted(torch.nn.Module):
    """A model whose fused loss is multiplied by loss_weight, so that GraphedStep captures (loss * w).backward() through Model.loss."""

    def __init__(self, model, weight):
        super().__init__()
        self.inner, self.fc, self.loss_weight = model, model.fc, weight

    def loss(self, x, labels):
        loss, logits = self.inner.loss(x, labels)
        return loss * self.loss_weight, logits


def _worker(rank, world, port, out):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from fusion_gcn_b200 import graph as G, modules as M
        from fusion_gcn_b200.distributed import GradientAllReducer, SyncBatchNorm, split_batch
        from fusion_gcn_b200.graphed import GraphedStep, loss_and_logits
        from helpers import ZERO_GRAD, stat_err
        from oracle import agcn_oracle as O
        shape, ncls, n_global, layers = (2, 40, 25, 3), 12, 5, 5
        torch.manual_seed(5)
        graph = G.SkeletonGraph(G.NTU_EDGES, center_joint=G.NTU_CENTER)
        state = O.init_state(G.adjacency_from_graph(graph), shape, ncls, start=64, num_layers=layers, seed=3, loud=True)
        model = M.Model(shape, ncls, graph, start_feature_size=64, num_layers=layers)
        model.load_state_dict(state, strict=True)
        model = model.to(dev).train()
        x = torch.randn(n_global, *shape, device=dev)
        labels = torch.randint(0, ncls, (n_global,), device=dev)
        lo, hi, weight = split_batch(n_global, rank, world)
        full = copy.deepcopy(model)
        loss_full, _ = full.loss(x, labels)
        loss_full.backward()
        sharded = M.set_sync_batchnorm(copy.deepcopy(model), SyncBatchNorm())
        reducer = GradientAllReducer(sharded.parameters())
        loss, _ = sharded.loss(x[lo:hi], labels[lo:hi])
        (loss * weight).backward()
        reducer()
        torch.cuda.synchronize()
        scale = max(float(q.grad.abs().max()) for q in full.parameters())
        worst_l2 = 0.0
        for (k, p), q in zip(sharded.named_parameters(), full.parameters()):
            if ZERO_GRAD.search(k):
                assert float((p.grad - q.grad).abs().max()) <= 1e-5 * scale, k
                continue
            worst_l2 = max(worst_l2, float((p.grad.double() - q.grad.double()).norm() / q.grad.double().norm().clamp_min(1e-30)))
        stats = max(stat_err(a, b) for (k, a), b in zip(sharded.state_dict().items(), full.state_dict().values()) if "running" in k)
        # the mean losses of the shards, weighted, average to the unsharded mean loss
        lw = (loss.detach() * weight).reshape(1)
        dist.all_reduce(lw)
        loss_err = abs(float(lw) / world - float(loss_full)) / abs(float(loss_full))

        # how far two correct fp32 evaluations of the unsharded batch are apart (the FFMA kernels: another summation order), for the
        # bound on the gradients: a ReLU input within rounding of zero may take the other bracket (see test_gpu_multi.py)
        calib = M.set_precision(copy.deepcopy(model), "fp32_ffma")
        calib.loss(x, labels)[0].backward()
        noise_l2 = max(float((c.grad.double() - q.grad.double()).norm() / q.grad.double().norm().clamp_min(1e-30))
                       for (k, c), q in zip(calib.named_parameters(), full.parameters()) if not ZERO_GRAD.search(k))

        # the same step captured with the gradient all-reduce: a replay equals the eager step bit for bit
        eager = M.set_sync_batchnorm(copy.deepcopy(model), SyncBatchNorm())
        graphed = M.set_sync_batchnorm(copy.deepcopy(model), SyncBatchNorm())
        lf = torch.nn.CrossEntropyLoss()
        w_eager, w_graphed = _Weighted(eager, weight), _Weighted(graphed, weight)
        r_eager, r_graphed = GradientAllReducer(eager.parameters()), GradientAllReducer(graphed.parameters())
        xs, ys = x[lo:hi].contiguous(), labels[lo:hi].contiguous()
        step = GraphedStep(w_graphed, lf, xs, ys, warmup=1, after_backward=r_graphed, preserve_buffers=True)
        eager.zero_grad(set_to_none=True)
        l_eager, _ = loss_and_logits(w_eager, lf, xs, ys)
        l_eager.backward()
        r_eager()
        l_graph = step()
        torch.cuda.synchronize()
        bitwise = torch.equal(l_graph, l_eager.detach()) and all(torch.equal(p.grad, q.grad) for p, q in zip(graphed.parameters(), eager.parameters()))
        bitwise = bitwise and all(torch.equal(a, b) for a, b in zip(graphed.state_dict().values(), eager.state_dict().values()))
        if rank == 0:
            out.put((worst_l2, noise_l2, float(stats), loss_err, bitwise))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(600)
def test_two_gpu_unequal_shards_weighted_loss_and_graph_replay():
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=560)
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    worst_l2, noise_l2, stats, loss_err, bitwise = out.get(timeout=5)
    print(f"[unequal shards 3/2 over NCCL] gradients worst L2 {worst_l2:.2e} (two fp32 evaluations of the unsharded batch: {noise_l2:.2e}), "
          f"running statistics {stats:.2e}, loss {loss_err:.2e}")
    assert loss_err <= 1e-5 and stats <= 1e-5, (loss_err, stats)
    assert worst_l2 <= max(1e-4, 4 * noise_l2), (worst_l2, noise_l2)
    assert bitwise, "the captured step does not reproduce the eager step bit for bit"
