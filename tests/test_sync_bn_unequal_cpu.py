"""Data parallelism over unequal batch shards, without a GPU: ``distributed.split_batch``, the fp64 moments that a synchronised
BatchNorm all-reduces (the host composition's form of agcn_bn_finalize phases 1 and 2), the C ABI's rejections of the new operands, and
gloo runs with 3 ranks (N = 7, shards 3/2/2) and 2 ranks (N = 5, shards 3/2) of the host composition on the stage oracle against the
unsharded fp64 model."""
import os
import socket
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LAYERS = 5


# ============================================================================================ split_batch
@pytest.mark.parametrize("n,world", [(7, 3), (5, 2), (10, 4), (64, 3), (64, 5), (64, 6), (64, 7), (3, 3), (64, 8), (1, 1)])
def test_split_batch_partitions_like_tensor_split(n, world):
    from fusion_gcn_b200.distributed import split_batch
    shards = [split_batch(n, r, world) for r in range(world)]
    assert shards[0][0] == 0 and shards[-1][1] == n
    assert all(a[1] == b[0] for a, b in zip(shards, shards[1:]))                    # contiguous, in rank order
    assert [hi - lo for lo, hi, _ in shards] == [len(t) for t in torch.tensor_split(torch.arange(n), world)]
    assert all(w == (hi - lo) * world / n for lo, hi, w in shards)
    assert sum(w for _, _, w in shards) == pytest.approx(world, rel=1e-15)


def test_split_batch_equal_shards_reproduce_shard_batch():
    from fusion_gcn_b200.distributed import shard_batch, split_batch
    for n, world in [(64, 4), (64, 8), (12, 3), (5, 1)]:
        for r in range(world):
            lo, hi, w = split_batch(n, r, world)
            assert (lo, hi) == shard_batch(n, r, world) and w == 1.0


def test_split_batch_rejects_empty_shards_and_bad_ranks():
    from fusion_gcn_b200.distributed import split_batch
    with pytest.raises(ValueError):
        split_batch(3, 0, 4)
    with pytest.raises(ValueError):
        split_batch(8, 4, 4)


# ============================================================================================ fp64 moments
def test_moments_of_shards_add_up_to_the_whole_batch(monkeypatch):
    """Shards with means about 100 (sigma 0.1) that differ between shards, sizes down to one row: their fp64 moments (the formulas of
    agcn_bn_finalize phase 1), summed as the all-reduce does, hold the whole batch's sum x / sum x^2 / row count, and the synchronised
    finalize of the host composition gives the whole batch's statistics and the backward's row factor."""
    import fusion_gcn_b200.functional as FN
    from oracle import stages as S
    monkeypatch.setattr(FN, "K", S)
    g = torch.Generator().manual_seed(3)
    shards = [torch.randn(n, 7, generator=g).double() * 0.1 + 100.0 + 0.25 * (r + 1) * (-1) ** r for r, n in enumerate((50, 1, 333, 20))]
    x = torch.cat(shards)
    total = sum(FN.host_moments(S.bn_stats_partials(s), s.shape[0]) for s in shards)
    assert float(total[-1]) == x.shape[0]
    assert (total[:7] - x.sum(0)).abs().max() <= 1e-12 * x.sum(0).abs().max()
    assert (total[7:14] - (x * x).sum(0)).abs().max() <= 1e-12 * (x * x).sum(0).abs().max()

    class _Sum:                     # the all-reduce of rank 1 (the one-row shard): every rank's moments added up
        world = len(shards)

        def all_reduce(self, t):
            return t.copy_(total)

    one, zero = torch.ones(7, dtype=torch.float64), torch.zeros(7, dtype=torch.float64)
    buf = FN.BnBuffers(zero.clone(), one.clone(), torch.zeros((), dtype=torch.long))
    _, _, mean, invstd, shard = FN._sync_finalize(S.bn_stats_partials(shards[1]), 1, one, zero, buf, buf.num_batches_tracked, _Sum())
    assert ((mean - x.mean(0)).abs() <= 1e-12 * x.mean(0).abs()).all()
    # E[x^2] - mean^2 in fp64 (as in the kernel): its rounding is (mean / sigma)^2 ~ 1e6 times 1e-16 of the variance
    assert ((invstd.pow(-2) - (x.var(0, unbiased=False) + FN.BN_EPS)).abs() <= 1e-12 * x.pow(2).mean(0)).all()
    assert ((buf.running_mean - 0.1 * x.mean(0)).abs() <= 1e-12 * x.mean(0).abs()).all()
    assert ((buf.running_var - (0.9 + 0.1 * x.var(0, unbiased=True))).abs() <= 1e-12 * x.pow(2).mean(0)).all()
    assert int(buf.num_batches_tracked) == 1
    assert shard.global_rows is None and shard.world == x.shape[0]           # 404 rows in all over this rank's one row


# ============================================================================================ C ABI rejections
def _lib():
    from fusion_gcn_b200 import build, capi
    build.build()
    return capi.lib()


@pytest.mark.parametrize("phase,part,nparts,rows,moments,status,message", [
    (3, 8, 1, 64, 8, 2, b"phase 3"),
    (-1, 8, 1, 64, 8, 2, b"phase -1"),
    (1, 8, 1, 64, None, 6, b"phase 1 needs moments"),
    (2, None, 0, 0, None, 6, b"phase 2 needs moments"),
    (1, 8, 1, 64, 12, 3, b"8-byte aligned"),
    (2, None, 0, 0, 4, 3, b"8-byte aligned"),
    (1, 8, 1, 0, 8, 1, b"bad shape"),
    (1, 8, 1, -5, 8, 1, b"bad shape"),
    (0, 8, 1, 0, None, 1, b"bad shape"),
    (1, None, 1, 64, 8, 6, b"null pointer"),
])
def test_bn_finalize_rejects_bad_phase_operands_without_gpu(phase, part, nparts, rows, moments, status, message):
    """agcn_bn_finalize checks the phase, the moments pointer and the row count before it launches anything."""
    lib = _lib()
    rc = lib.agcn_bn_finalize(part, nparts, rows, 16, None, None, None, None, None, 0.1, 1e-5, 16, 16, None, None, phase, moments, None)
    assert rc == status and message in lib.agcn_last_error_string()


@pytest.mark.parametrize("count,status,message", [(None, 6, b"global row count"), (12, 3, b"global_rows must be 8-byte aligned")])
def test_bn_bwd_phase2_rejects_a_missing_or_misaligned_count_without_gpu(count, status, message):
    lib = _lib()
    ws = lib.agcn_bn_workspace_bytes(64)
    rc = lib.agcn_bn_bwd(16, None, None, 16, 16, 16, 16, 16, None, None, None, None, 0, 0, 1, 64, 0, 64, 0, 2, 16, count, 16, ws, None)
    assert rc == status and message in lib.agcn_last_error_string()


# ============================================================================================ gloo, unequal shards
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, n_global, out):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.set_num_threads(2)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import fusion_gcn_b200.functional as FN
        from fusion_gcn_b200 import graph as G, modules as M
        from fusion_gcn_b200.distributed import GradientAllReducer, SyncBatchNorm, split_batch
        from helpers import ZERO_GRAD, check_grads, rel_err
        from oracle import agcn_oracle as O, stages
        FN.K = stages                                   # TEST ONLY: torch stage oracle instead of the CUDA library
        shape, ncls, start = (2, 12, 20, 3), 7, 8
        graph = G.SkeletonGraph(G.UTD_EDGES, center_joint=G.UTD_CENTER)
        state = O.init_state(G.adjacency_from_graph(graph), shape, ncls, start=start, num_layers=LAYERS, seed=3, loud=True)
        gen = torch.Generator().manual_seed(11)
        x = torch.randn(n_global, *shape, generator=gen)
        w = torch.randn(n_global, ncls, generator=gen)
        labels = torch.randint(0, ncls, (n_global,), generator=gen)
        lo, hi, weight = split_batch(n_global, rank, world)
        model = M.Model(shape, ncls, graph, start_feature_size=start, num_layers=LAYERS)
        model.load_state_dict(state, strict=True)
        M.set_sync_batchnorm(model, SyncBatchNorm())
        model.train()
        reducer = GradientAllReducer(model.parameters(), bucket_bytes=4096)
        names = [k for k, _ in model.named_parameters()]

        def sharded_step(loss_of):
            model.zero_grad(set_to_none=True)
            loss_of().backward()
            reducer()
            return {k: p.grad.clone() for k, p in model.named_parameters()}

        def full_batch(dtype, loss_of):
            p = O.as_leaves(state, dtype)
            logits = O.model_forward(x.to(dtype), p, shape[3], True, start=start, num_layers=LAYERS)
            loss_of(logits).backward()
            return logits.detach(), {k: p[k].grad for k in names}

        y = model(x[lo:hi])
        # sum loss: the all-reduced mean of the ranks' gradients is the full-batch gradient / world
        g_sum = sharded_step(lambda: (model(x[lo:hi]) * w[lo:hi]).sum())
        y64, e_sum = full_batch(torch.float64, lambda lg: (lg * w.to(lg.dtype)).sum() / world)
        _, e_sum32 = full_batch(torch.float32, lambda lg: (lg * w.to(lg.dtype)).sum() / world)
        err_y = rel_err(y, y64[lo:hi])
        assert err_y <= 2e-5, err_y
        check_grads(g_sum, e_sum, 1e-4, f"sum loss rank {rank}", ref32=e_sum32)
        # mean cross-entropy of the shard (fused head) x loss_weight: the gradient of the unsharded batch's mean loss
        g_ce = sharded_step(lambda: model.loss(x[lo:hi], labels[lo:hi])[0] * weight)
        _, e_ce = full_batch(torch.float64, lambda lg: torch.nn.functional.cross_entropy(lg, labels))
        _, e_ce32 = full_batch(torch.float32, lambda lg: torch.nn.functional.cross_entropy(lg, labels))
        check_grads(g_ce, e_ce, 1e-4, f"weighted mean loss rank {rank}", ref32=e_ce32)
        # negative control: the same step without loss_weight misses the bound
        g_plain = sharded_step(lambda: model.loss(x[lo:hi], labels[lo:hi])[0])
        unweighted = max(rel_err(g_plain[k], e_ce[k]) for k in names if not ZERO_GRAD.search(k))
        # running statistics: identical on every rank
        stats = torch.cat([b.reshape(-1).double() for k, b in model.named_buffers() if "running" in k or "num_batches" in k])
        gathered = [torch.empty_like(stats) for _ in range(world)]
        dist.all_gather(gathered, stats)
        same = all(torch.equal(gathered[0], t) for t in gathered)
        if rank == 0:
            out.put((float(err_y), unweighted, same))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(600)
@pytest.mark.parametrize("world,n_global", [(3, 7), (2, 5)])
def test_unequal_shards_with_sync_batchnorm_match_the_unsharded_batch(world, n_global):
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, n_global, out)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=560)
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    err_y, unweighted, same = out.get(timeout=5)
    assert same, "ranks disagree on the running statistics"
    assert err_y <= 2e-5, err_y
    assert unweighted > 1e-2, f"without loss_weight the gradients should miss the bound, error {unweighted:.2e}"
