"""Whole training step (forward + loss + backward of any model whose step is capturable) replayed as ONE CUDA graph (SURVEY 8 f1).

The reference launches every ATen kernel of a step from Python (torch_src/session/procedures/step.py:39-43).  The C ABI
of this package never allocates, never synchronises and takes the stream from the caller, so a step is capturable: the
~630 launches of the NTU model become one ``cudaGraphLaunch`` and the host leaves the critical path (the eager step is
launch-bound below ~8 sequences per GPU, profiles/r1q).  Inputs, logits, loss and the parameter gradients live at fixed
addresses; ``__call__`` copies a new batch into the static input and replays.  The input is one tensor or, for the fusion
models whose dataset yields one tensor per modality (torch_src/dataset.py:42-49), a dict of tensors.
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
        examples = x_example.items() if isinstance(x_example, dict) else [(None, x_example)]
        for key, t in examples:
            if not (isinstance(t, torch.Tensor) and t.is_cuda):
                where = "" if key is None else f" (input {key!r}: {_describe(t)})"
                raise RuntimeError(f"GraphedStep needs CUDA tensors (there is no CPU path){where}")
        self.model, self.loss_fn = model, loss_fn
        self.accumulate, self.loss_divisor, self.after_backward = bool(accumulate), loss_divisor, after_backward
        if isinstance(x_example, dict):
            self.x = {k: v.detach().clone() for k, v in x_example.items()}
        else:
            self.x = x_example.detach().clone()
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
        if not isinstance(self.x, dict):
            if isinstance(x, dict):
                raise ValueError(f"GraphedStep was captured with one input tensor, got a dict with keys {sorted(x)}")
            self.x.copy_(x, non_blocking=True)
            return
        if not isinstance(x, dict):
            raise ValueError(f"GraphedStep was captured with the inputs {sorted(self.x)}, got {_describe(x)}")
        for key in self.x:
            if key not in x:
                raise ValueError(f"input {key!r} is missing (captured inputs: {sorted(self.x)})")
        for key, t in x.items():
            if key not in self.x:
                raise ValueError(f"input {key!r} was not captured (captured inputs: {sorted(self.x)})")
            s = self.x[key]
            if not (isinstance(t, torch.Tensor) and t.shape == s.shape and t.dtype == s.dtype and t.device == s.device):
                raise ValueError(f"input {key!r}: {_describe(t)} differs from the captured {_describe(s)}")
        for key, t in x.items():
            self.x[key].copy_(t, non_blocking=True)

    def __call__(self, x: Optional[Features] = None, y: Optional[torch.Tensor] = None) -> torch.Tensor:
        if x is not None:
            self._copy_features(x)
        if y is not None:
            self.y.copy_(y, non_blocking=True)
        self.graph.replay()
        return self.loss
