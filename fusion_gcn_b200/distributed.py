"""Batch-sharded data parallelism for the AGCN model: one process per GPU, full replica per rank, bucketed gradient
all-reduce overlapped with the backward pass (NCCL over NVLink 5 / NVSwitch on the GPU box; gloo in the CPU tests).

The reference has no distributed code at all (SURVEY 2.1); the only natural shard of the path is the batch
(SURVEY 8e).  BatchNorm statistics stay per replica, which is what DistributedDataParallel does by default.

Buckets are filled in reverse parameter order (the order backward produces gradients).  Each bucket owns a persistent flat
buffer; when the last gradient of a bucket has been accumulated (post-accumulate-grad hooks) ONE kernel packs the bucket
(``agcn_bucket_copy``), the all-reduce starts asynchronously on NCCL's stream while backward continues with the earlier layers,
and ``finish()`` waits and writes the averaged values back with one kernel per bucket -- no ``torch.cat``, no per-parameter
copy kernels.  Everything is stream-ordered, so the whole thing is capturable in the step's CUDA graph.
"""
from typing import Iterable, List

import torch
import torch.distributed as dist

from . import capi


def shard_batch(n_global: int, rank: int, world: int):
    """Rank r takes samples [r*N/R, (r+1)*N/R) (SURVEY 8e).  Equal shards only; see split_batch for any N >= R."""
    if n_global % world:
        raise ValueError(f"global batch {n_global} is not divisible by world size {world}")
    per = n_global // world
    return rank * per, (rank + 1) * per


def split_batch(n_global: int, rank: int, world: int):
    """Rank r's shard of a global batch of N sequences over R ranks, for any N >= R: -> (lo, hi, loss_weight).

    The shards follow ``torch.tensor_split``: the first N mod R ranks take one sequence more.  ``loss_weight`` = n_r * R / N (exactly
    1.0 for equal shards) is the factor a MEAN-reduced loss of the shard must be multiplied by before ``backward()``: the gradient
    all-reduce then averages to the gradient of the unsharded batch's mean loss.  Scaling at the all-reduce instead is not enough with
    synchronised BatchNorm, whose backward adds the ranks' upstream gradients, so every rank's must be on the same scale.
    ``(loss * loss_weight).backward()`` reaches the fused classifier (``Model.loss``) through its device-side loss gradient."""
    if not 0 <= rank < world:
        raise ValueError(f"rank {rank} outside a world of {world}")
    if n_global < world:
        raise ValueError(f"global batch {n_global} is smaller than world size {world}: a rank would get no sequence")
    per, extra = divmod(n_global, world)
    lo = rank * per + min(rank, extra)
    hi = lo + per + (1 if rank < extra else 0)
    return lo, hi, (hi - lo) * world / n_global


class SyncBatchNorm:
    """The collectives of a synchronised BatchNorm (``modules.set_sync_batchnorm``): training-mode statistics and their backward sums
    over all ranks of ``group``, so that a batch sharded over R GPUs normalises exactly like the unsharded batch (SURVEY 8e), whether
    or not the shards are of equal size.  In the forward each rank reduces its partials to fp64 moments (sum x | sum x^2 | rows,
    2C + 1 doubles: at most 4 KB at C = 256) and all-reduces them; the count travels with the moments to the backward, which
    all-reduces its two fp32 column sums between its sum pass and its apply pass.  Both payloads have a fixed size whatever the
    shard or world size.  Stream-ordered on NCCL: capturable in the step's CUDA graph."""

    def __init__(self, group=None):
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1

    def all_reduce(self, t: torch.Tensor) -> torch.Tensor:
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
        return t


class _Bucket:
    def __init__(self, params: List[torch.nn.Parameter]):
        self.params = params
        self.numel = sum(p.numel() for p in params)
        self.flat = torch.empty(self.numel, device=params[0].device, dtype=params[0].dtype)
        self.ready = 0
        self.work = None
        self._key = None
        self._table = self._items = None
        self._nitems = 0

    def views(self):
        out, off = [], 0
        for p in self.params:
            out.append(self.flat[off:off + p.numel()])
            off += p.numel()
        return out

    def table(self):
        """Device table (flat slice, gradient tensor, numel) of the bucket, rebuilt only when a gradient was reallocated."""
        key = tuple(p.grad.data_ptr() for p in self.params)
        if key != self._key:
            chunk = capi.lib().agcn_optim_chunk()
            rows, items, off = [], [], 0
            for i, p in enumerate(self.params):
                n = p.numel()
                rows.append([self.flat.data_ptr() + 4 * off, p.grad.data_ptr(), 0, 0, n])
                items += [(i, c) for c in range((n + chunk - 1) // chunk)]
                off += n
            # pinned staging (kept alive): the upload is then legal inside a CUDA-graph capture, where the gradients get their
            # final, static addresses
            self._host = (torch.tensor(rows, dtype=torch.int64).pin_memory(), torch.tensor(items, dtype=torch.int32).pin_memory())
            self._table = self._host[0].to(self.flat.device, non_blocking=True)
            self._items = self._host[1].to(self.flat.device, non_blocking=True)
            self._nitems, self._key = len(items), key
        return self._table, self._items, self._nitems


class GradientAllReducer:
    """``reducer = GradientAllReducer(model.parameters())``; after ``loss.backward()`` call ``reducer()`` (or ``finish()``):
    ``p.grad`` then holds the average over the ranks.  With ``overlap=True`` (default) the buckets' all-reduces start from
    gradient hooks DURING backward; ``reducer()`` only waits for them and writes the averages back."""

    def __init__(self, params: Iterable[torch.nn.Parameter], bucket_bytes: int = 4 << 20, group=None, overlap: bool = True):
        self.params: List[torch.nn.Parameter] = [p for p in params if p.requires_grad]
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.buckets: List[_Bucket] = []
        cur, size = [], 0
        for p in reversed(self.params):
            cur.append(p)
            size += p.numel() * p.element_size()
            if size >= bucket_bytes:
                self.buckets.append(_Bucket(cur))
                cur, size = [], 0
        if cur:
            self.buckets.append(_Bucket(cur))
        self._hooks = []
        if overlap and self.world > 1:
            for b in self.buckets:
                for p in b.params:
                    self._hooks.append(p.register_post_accumulate_grad_hook(lambda _p, b=b: self._grad_ready(b)))

    # ---- bucket <-> gradient tensors
    @staticmethod
    def _copy(bucket: _Bucket, to_flat: bool, scale: float):
        grads = [p.grad for p in bucket.params]
        if bucket.flat.is_cuda and all(g.dtype == torch.float32 and g.is_contiguous() for g in grads):
            table, items, n = bucket.table()
            rc = capi.lib().agcn_bucket_copy(table.data_ptr(), items.data_ptr(), n, int(to_flat), float(scale),
                                             torch.cuda.current_stream(bucket.flat.device).cuda_stream)
            capi.check(rc, "agcn_bucket_copy")
        elif to_flat:                                   # CPU tensors (gloo groups in the tests) / non-contiguous gradients
            torch._foreach_copy_(bucket.views(), [g.reshape(-1) for g in grads])
        else:
            for g, v in zip(grads, bucket.views()):
                g.copy_((v * scale).view_as(g))

    def _launch(self, bucket: _Bucket):
        for p in bucket.params:
            if p.grad is None:
                p.grad = torch.zeros_like(p)
        self._copy(bucket, True, 1.0)
        bucket.work = dist.all_reduce(bucket.flat, op=dist.ReduceOp.SUM, group=self.group, async_op=True)

    def _grad_ready(self, bucket: _Bucket):
        bucket.ready += 1
        if bucket.ready == len(bucket.params) and bucket.work is None:
            self._launch(bucket)

    def start(self):
        """Starts the all-reduce of every bucket that the hooks have not started already."""
        if self.world == 1:
            return
        for b in self.buckets:
            if b.work is None:
                self._launch(b)

    def finish(self):
        for b in self.buckets:
            if b.work is not None:
                b.work.wait()
                self._copy(b, False, 1.0 / self.world)
                b.work = None
            b.ready = 0

    wait = finish

    def __call__(self):
        self.start()
        self.finish()

    def remove_hooks(self):
        for h in self._hooks:
            h.remove()
        self._hooks = []
