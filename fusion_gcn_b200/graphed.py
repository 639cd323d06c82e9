"""Whole training step (forward + loss + backward of any model whose step is capturable) replayed as ONE CUDA graph (SURVEY 8 f1).

The reference launches every ATen kernel of a step from Python (torch_src/session/procedures/step.py:39-43).  The C ABI
of this package never allocates, never synchronises and takes the stream from the caller, so a step is capturable: the
~630 launches of the NTU model become one ``cudaGraphLaunch`` and the host leaves the critical path (the eager step is
launch-bound below ~8 sequences per GPU, profiles/r1q).  Inputs, logits, loss and the parameter gradients live at fixed
addresses; ``__call__`` copies a new batch into the static input and replays.  The input is one tensor or, for the fusion
models whose dataset yields one tensor per modality (torch_src/dataset.py:42-49), a dict of tensors.

``GraphedForward`` does the same for the eval-mode forward alone (validation, evaluation sessions, inference), and serves batches
shorter than the captured one by zero padding.
"""
from typing import Callable, Dict, Optional, Union

import torch

from . import capi

Features = Union[torch.Tensor, Dict[str, torch.Tensor]]


def loss_and_logits(model: torch.nn.Module, loss_fn: Callable, x: Features, y: torch.Tensor):
    """loss_fn(model(x), y) -- through the fused classifier + cross-entropy head (``Model.loss``) when ``loss_fn`` is a plain
    ``nn.CrossEntropyLoss()`` (mean reduction, no class weights, no label smoothing: what the reference builds at
    torch_src/session/session.py:53) and the model has one; any other loss runs as given."""
    fused = (isinstance(loss_fn, torch.nn.CrossEntropyLoss) and loss_fn.weight is None and loss_fn.reduction == "mean"
             and loss_fn.label_smoothing == 0.0 and getattr(model, "fc", None) is not None and hasattr(model, "loss")
             and y.dtype == torch.int64 and y.dim() == 1)
    if fused:
        return model.loss(x, y)
    logits = model(x)
    return loss_fn(logits, y), logits


def _describe(t) -> str:
    if not isinstance(t, torch.Tensor):
        return type(t).__name__
    return f"{tuple(t.shape)} {t.dtype} on {t.device}"


def _items(x: Features):
    return list(x.items()) if isinstance(x, dict) else [(None, x)]


def _require_cuda(x: Features, who: str) -> None:
    for key, t in _items(x):
        if not (isinstance(t, torch.Tensor) and t.is_cuda):
            where = "" if key is None else f" (input {key!r}: {_describe(t)})"
            raise RuntimeError(f"{who} needs CUDA tensors (there is no CPU path){where}")


def _static_copy(x: Features) -> Features:
    if isinstance(x, dict):
        return {k: v.detach().clone() for k, v in x.items()}
    return x.detach().clone()


def _pair_inputs(static: Features, x, who: str, check: Optional[Callable] = None):
    """[(key, static tensor, new entry)] for a batch ``x`` with the captured structure: one tensor (key None), or a dict with
    exactly the captured keys.  ValueError otherwise, and whatever ``check(key, static tensor, new entry)`` raises."""
    check = check or (lambda key, s, t: None)
    if not isinstance(static, dict):
        if isinstance(x, dict):
            raise ValueError(f"{who} was captured with one input tensor, got a dict with keys {sorted(x)}")
        check(None, static, x)
        return [(None, static, x)]
    if not isinstance(x, dict):
        raise ValueError(f"{who} was captured with the inputs {sorted(static)}, got {_describe(x)}")
    for key in static:
        if key not in x:
            raise ValueError(f"input {key!r} is missing (captured inputs: {sorted(static)})")
    for key, t in x.items():
        if key not in static:
            raise ValueError(f"input {key!r} was not captured (captured inputs: {sorted(static)})")
        check(key, static[key], t)
    return [(key, static[key], t) for key, t in x.items()]


def _check_entry(key, s: torch.Tensor, t, rows: bool = False) -> None:
    """ValueError naming the input unless ``t`` has the dtype, device and shape of the static tensor ``s``.  ``rows``: the leading
    (batch) dim may be anything from 1 to ``s``'s."""
    fits = isinstance(t, torch.Tensor) and t.dtype == s.dtype and t.device == s.device
    if fits and rows:
        fits = t.dim() == s.dim() and t.shape[1:] == s.shape[1:] and 1 <= t.shape[0] <= s.shape[0]
    elif fits:
        fits = t.shape == s.shape
    if not fits:
        name = "input" if key is None else f"input {key!r}"
        limit = f" (any batch size from 1 to {s.shape[0]})" if rows else ""
        raise ValueError(f"{name}: {_describe(t)} differs from the captured {_describe(s)}{limit}")


class GraphedStep:
    """``step = GraphedStep(model, loss_fn, x_example, y_example)``; ``loss = step(x, y)`` runs forward + loss + backward and
    leaves the gradients in ``p.grad`` (static tensors).  ``after_backward`` (for instance a gradient all-reduce) is captured
    into the same graph when given.

    ``x_example`` is a CUDA tensor or a dict of CUDA tensors (one per modality); every later ``x`` must have the same keys, and
    the same shape, dtype and device per key.

    ``loss_divisor``: the captured loss is ``loss_fn(model(x), y) / loss_divisor``, as the reference divides by ``loss_quotient``
    for gradient accumulation (procedures/step.py:41-42).  ``loss_fn`` keeps its own type, so the fused head stays in use.

    ``accumulate``: False (default) -- every replay overwrites the gradients with this batch's.  True -- every replay adds this
    batch's gradient to them, as ``loss.backward()`` does on defined ``.grad`` tensors; ``zero_grads()`` starts a new sum."""

    def __init__(self, model: torch.nn.Module, loss_fn: Callable, x_example: Features, y_example: torch.Tensor,
                 warmup: int = 3, after_backward: Optional[Callable[[], None]] = None, preserve_buffers: bool = False,
                 accumulate: bool = False, loss_divisor: float = 1):
        """``preserve_buffers``: the warm-up steps run real forward passes (BatchNorm running statistics move); with this flag the
        module buffers are put back afterwards, so that the first replay is the first step the model sees (training sessions that
        build the graph lazily on their first batch)."""
        _require_cuda(x_example, "GraphedStep")
        self.model, self.loss_fn = model, loss_fn
        self.accumulate, self.loss_divisor, self.after_backward = bool(accumulate), loss_divisor, after_backward
        self.x = _static_copy(x_example)
        self.y = y_example.detach().clone()
        saved_buffers = [b.detach().clone() for b in model.buffers()] if preserve_buffers else None
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):          # warm-up off the default stream: lazy initialisation (function attributes,
            for _ in range(max(1, warmup)):    # driver entry points, allocator) must not happen during capture
                model.zero_grad(set_to_none=True)
                self._step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        reached = [p for p in model.parameters() if p.grad is not None]
        model.zero_grad(set_to_none=True)
        if self.accumulate:
            # allocated here, outside the capture and after the warm-up: the captured backward adds into them in place
            # (AccumulateGrad on a defined .grad); without accumulate they are allocated inside the capture, from the graph's pool
            for p in reached:
                p.grad = torch.zeros_like(p)
        self.graph = torch.cuda.CUDAGraph()
        before = capi.lib().agcn_launch_count()
        with torch.cuda.graph(self.graph):
            self.loss, self.logits = self._step()
        self.launches_per_replay = int(capi.lib().agcn_launch_count() - before)   # kernels of libagcn_b200.so in the graph
        # the static gradient tensors: a caller whose loop sets p.grad to None (optimizer.zero_grad()) re-attaches them after a replay
        self.grads = [(p, p.grad) for p in model.parameters() if p.grad is not None]
        if saved_buffers is not None:
            with torch.no_grad():
                for b, old in zip(model.buffers(), saved_buffers):
                    b.copy_(old)

    def _step(self):
        loss, logits = loss_and_logits(self.model, self.loss_fn, self.x, self.y)
        if self.loss_divisor != 1:
            loss = loss / self.loss_divisor
        loss.backward()
        if self.after_backward is not None:
            self.after_backward()
        return loss, logits

    def attach_grads(self) -> None:
        """p.grad <- the graph's static gradient tensor, for every parameter the captured backward reaches."""
        for p, g in self.grads:
            p.grad = g

    def zero_grads(self) -> None:
        """Zeroes the static gradient tensors in place: with ``accumulate``, the next replay then starts a new sum."""
        torch._foreach_zero_([g for _, g in self.grads])

    def _copy_features(self, x: Features) -> None:
        # (a single tensor goes straight to copy_)
        for _, s, t in _pair_inputs(self.x, x, "GraphedStep", _check_entry if isinstance(self.x, dict) else None):
            s.copy_(t, non_blocking=True)

    def __call__(self, x: Optional[Features] = None, y: Optional[torch.Tensor] = None) -> torch.Tensor:
        if x is not None:
            self._copy_features(x)
        if y is not None:
            self.y.copy_(y, non_blocking=True)
        self.graph.replay()
        return self.loss


class GraphedForward:
    """``gf = GraphedForward(model, x_example)``; ``logits = gf(x)`` replays the eval-mode forward ``model(x)`` as one CUDA graph.

    Evaluation (``Session.validate_epoch``, ``EvaluationSession``, inference) at the reference's batch sizes is as launch bound as
    training: the eval forward is a chain of library kernels with BatchNorm, residual and ReLU in the convolution epilogues, no host
    synchronisation and nothing saved, so it is captured as it stands.  Warm-up and capture run under ``torch.no_grad()``, whatever
    the caller's grad mode; no loss is captured, the caller applies any loss to the returned logits.

    ``model`` must be in eval mode (``ValueError`` otherwise: a training-mode forward moves the BatchNorm running statistics and its
    batch statistics couple the samples).  ``x_example`` is a CUDA tensor or a dict of CUDA tensors, all batch-first with one batch
    size B; its output must be a tensor with leading dim B.

    Shorter batches: ``gf(x)`` takes any n from 1 to B sequences (every dict entry with the same n).  They are copied into the first n
    rows of the static input, the other rows are zeroed, and ``logits[:n]`` is returned.  This relies on the eval-mode forward
    treating every sample independently (BatchNorm is a per-channel affine of the running statistics; the attention softmax, the
    pool and the classifier are per sample), which holds for every model of the reference and of this package.  The first n rows
    are bit-identical to the eager forward of the zero-padded batch; against the eager forward of the n sequences alone they differ
    by rounding, because the eager kernels pick their T-chunking from the batch size.  Trailing shapes, dtypes, keys and device
    must match the capture (``ValueError`` naming the input).

    The returned logits are a view of the graph's static output: the next call overwrites them, so clone what has to outlive it.

    ``adj_c`` (the attention maps of ``SpatialGraphConv`` / ``AGCNGraphConvolution``): after every call each ``adj_c[k]`` is the
    graph's own tensor, sliced to the rows of the n valid samples -- also when an eager forward rebound it in between.

    Weights and buffers: the graph reads the tensors the model held at capture time, so in-place changes (optimizer steps, BatchNorm
    running statistics moved by training steps, ``load_state_dict``, which copies in place) are picked up by the next replay.  A
    replaced tensor is not: new ``Parameter`` objects, ``model.to(...)`` that moves or casts, ``load_state_dict(assign=True)`` need a
    new ``GraphedForward``."""

    def __init__(self, model: torch.nn.Module, x_example: Features, warmup: int = 2):
        if model.training:
            raise ValueError("GraphedForward captures the eval-mode forward: call model.eval() first (in training mode the forward "
                             "moves the BatchNorm running statistics and the batch statistics couple the samples)")
        _require_cuda(x_example, "GraphedForward")
        sizes = {t.shape[0] if t.dim() else 0 for _, t in _items(x_example)}
        if len(sizes) != 1 or 0 in sizes:
            raise ValueError("GraphedForward needs batch-first inputs with one batch size, got "
                             + ", ".join(f"{k!r}: {_describe(t)}" for k, t in _items(x_example)))
        self.model, self.batch_size = model, sizes.pop()
        self.x = _static_copy(x_example)
        holders = [m for m in model.modules() if isinstance(getattr(m, "adj_c", None), list)]
        with torch.no_grad():
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):       # warm-up off the default stream, as GraphedStep's
                for _ in range(max(1, warmup)):
                    model(self.x)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            before_capture = [list(m.adj_c) for m in holders]
            self.graph = torch.cuda.CUDAGraph()
            before = capi.lib().agcn_launch_count()
            with torch.cuda.graph(self.graph):
                self.logits = model(self.x)
            self.launches_per_replay = int(capi.lib().agcn_launch_count() - before)
        if not (isinstance(self.logits, torch.Tensor) and self.logits.dim() >= 1 and self.logits.shape[0] == self.batch_size):
            raise ValueError(f"GraphedForward needs a model output with leading dim {self.batch_size}, got {_describe(self.logits)}")
        # the attention maps the capture wrote (modules the forward did not reach keep what they held)
        self.attention = [(m, list(m.adj_c)) for m, old in zip(holders, before_capture)
                          if any(a is not b for a, b in zip(m.adj_c, old))]

    def __call__(self, x: Features) -> torch.Tensor:
        pairs = _pair_inputs(self.x, x, "GraphedForward", lambda key, s, t: _check_entry(key, s, t, rows=True))
        first, _, t0 = pairs[0]
        n = t0.shape[0]
        for key, _, t in pairs:
            if t.shape[0] != n:
                raise ValueError(f"input {key!r} has {t.shape[0]} sequences, input {first!r} has {n}: every input needs the same batch size")
        for _, s, t in pairs:
            s[:n].copy_(t, non_blocking=True)
            s[n:].zero_()
        self.graph.replay()
        for m, maps in self.attention:
            m.adj_c[:] = [a[:a.shape[0] * n // self.batch_size] for a in maps]
        return self.logits[:n]
