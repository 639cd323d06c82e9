"""Fused multi-tensor optimizers for the AGCN model (SURVEY 8 f4).

Drop-in subclasses of ``torch.optim.Optimizer`` with the constructor arguments, ``param_groups`` and ``state_dict`` layout of
``torch.optim.SGD`` / ``Adam`` / ``AdamW`` / ``ASGD`` -- the classes the reference instantiates from its YAML ``optimizer`` /
``optimizer_args`` keys (torch_src/session_helper.py:48-82) -- so learning-rate schedulers (session_helper.py:56-89) and the
reference's ``CheckpointManager`` (torch_src/progress.py:203-276) keep working.  ``step()`` is ONE kernel launch per parameter
group (``agcn_optim_sgd`` / ``agcn_optim_adam`` / ``agcn_optim_asgd``) instead of hundreds of per-tensor kernels: the 274
parameter tensors of the model stay where PyTorch put them and are reached through a device table of pointers.

Options torch's classes take: ``maximize`` (all four), ``amsgrad`` (Adam / AdamW; the state gains ``max_exp_avg_sq``).  They
are kept in each parameter group under torch's names and read from the group at every step, so a checkpoint written by
torch.optim with other settings steps the way torch would after loading it.  ``foreach`` / ``fused`` / ``capturable`` /
``differentiable`` are accepted and ignored (the step is always one capturable launch); sparse gradients are refused.

Mixed precision (torch_src/session/procedures/step.py:55-78): the classes declare ``_step_supports_amp_scaling``, so
``GradScaler.step`` hands them its device scalars ``grad_scale`` / ``found_inf`` and the kernel unscales the gradients and skips
the step on overflow -- no ``.item()`` synchronisation, capturable in a CUDA graph.  There is no CPU path.
"""
from typing import Dict, List

import torch

from . import capi


def _stream(dev):
    return torch.cuda.current_stream(dev).cuda_stream


class _FusedOptimizer(torch.optim.Optimizer):
    _step_supports_amp_scaling = True          # GradScaler passes grad_scale / found_inf instead of unscaling + syncing itself

    def _tensors(self, group) -> List[torch.nn.Parameter]:
        out = []
        for p in group["params"]:
            if p.grad is None:
                continue
            if not p.is_cuda or p.dtype != torch.float32 or not p.is_contiguous():
                raise RuntimeError("fusion_gcn_b200.optim: contiguous fp32 CUDA parameters expected (there is no CPU path)")
            if p.grad.is_sparse or p.grad.dtype != torch.float32:
                raise RuntimeError("fusion_gcn_b200.optim: dense fp32 gradients expected")
            if not p.grad.is_contiguous():
                p.grad = p.grad.contiguous()
            out.append(p)
        return out

    def __setstate__(self, state):
        super().__setstate__(state)
        for group in self.param_groups:            # a checkpoint written before the option existed
            group.setdefault("maximize", False)

    def _work(self, group, params, states):
        """Device table + work list for ``params`` (rebuilt only when a pointer changed, e.g. after zero_grad(set_to_none=True)).
        ``states``: per parameter the state tensors of its row, between gradient and numel (None: an unused column)."""
        key = tuple((p.data_ptr(), p.grad.data_ptr(), *(0 if t is None else t.data_ptr() for t in st), p.numel()) for p, st in zip(params, states))
        cache = self._cache.get(id(group))
        if cache is not None and cache[0] == key:
            return cache[1], cache[2], cache[3]
        dev = params[0].device
        chunk = capi.lib().agcn_optim_chunk()
        rows, items = [], []
        for i, k in enumerate(key):
            rows.append(list(k))
            items += [(i, c) for c in range((k[-1] + chunk - 1) // chunk)]
        host = (torch.tensor(rows, dtype=torch.int64).pin_memory(), torch.tensor(items, dtype=torch.int32).pin_memory())
        table, work = host[0].to(dev, non_blocking=True), host[1].to(dev, non_blocking=True)      # pinned: legal under graph capture
        self._cache[id(group)] = (key, table, work, len(items), host)
        return table, work, len(items)

    def _amp(self):
        gs, fi = getattr(self, "grad_scale", None), getattr(self, "found_inf", None)
        return gs, fi

    @staticmethod
    def _ptr(t):
        return None if t is None else t.data_ptr()

    @staticmethod
    def _group_scalar(value, device, init):
        """A device scalar shared by the whole group: ``value`` as loaded from a checkpoint (any device, dtype or Python number), or a
        new one holding ``init``."""
        if value is None:
            return torch.full((), init, dtype=torch.float32, device=device)
        if isinstance(value, torch.Tensor) and value.is_cuda and value.dtype == torch.float32 and value.dim() == 0:
            return value
        return torch.as_tensor(value).detach().to(device=device, dtype=torch.float32).reshape(()).clone()

    def _lr_args(self, group):
        """(host lr, device lr pointer): a tensor ``lr`` (capturable schedulers) is read on the device."""
        lr = group["lr"]
        if isinstance(lr, torch.Tensor):
            if lr.is_cuda:
                return 0.0, lr.data_ptr()
            return float(lr), None
        return float(lr), None


class FusedSGD(_FusedOptimizer):
    """torch.optim.SGD(params, lr, momentum=0, dampening=0, weight_decay=0, nesterov=False, maximize=False) with one launch per
    group."""

    def __init__(self, params, lr=1e-3, momentum=0.0, dampening=0.0, weight_decay=0.0, nesterov=False, maximize=False, **unused):
        if nesterov and (momentum <= 0 or dampening != 0):
            raise ValueError("Nesterov momentum requires a momentum and zero dampening")
        super().__init__(params, dict(lr=lr, momentum=momentum, dampening=dampening, weight_decay=weight_decay, nesterov=nesterov,
                                      maximize=maximize))
        self._cache: Dict[int, tuple] = {}

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        gs, fi = self._amp()
        for group in self.param_groups:
            params = self._tensors(group)
            if not params:
                continue
            first = False
            states = []
            for p in params:
                st = self.state[p]
                if group["momentum"] != 0 and "momentum_buffer" not in st:
                    st["momentum_buffer"] = torch.zeros_like(p, memory_format=torch.contiguous_format)
                    first = True                    # torch: buf = clone(grad) on the first step
                states.append((st.get("momentum_buffer", p), None))
            table, work, nitems = self._work(group, params, states)
            lr, lr_dev = self._lr_args(group)
            rc = capi.lib().agcn_optim_sgd(table.data_ptr(), work.data_ptr(), nitems, lr, lr_dev, float(group["momentum"]),
                                           float(group["dampening"]), float(group["weight_decay"]), int(group["nesterov"]), int(first),
                                           int(group["maximize"]), self._ptr(gs), self._ptr(fi), _stream(params[0].device))
            capi.check(rc, "agcn_optim_sgd")
        return loss


class FusedAdam(_FusedOptimizer):
    """torch.optim.Adam(params, lr, betas, eps, weight_decay, amsgrad=False, maximize=False) -- L2 weight decay added to the
    gradient."""
    _decoupled = False

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, amsgrad=False, maximize=False, **unused):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, amsgrad=amsgrad, maximize=maximize))
        self._cache: Dict[int, tuple] = {}

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        gs, fi = self._amp()
        for group in self.param_groups:
            params = self._tensors(group)
            if not params:
                continue
            amsgrad = bool(group["amsgrad"])
            states = []
            master = None          # ONE device step counter shared by the group (state[p]["step"] of every parameter is this tensor)
            for p in params:
                st = self.state[p]
                if "exp_avg" not in st:
                    st["exp_avg"] = torch.zeros_like(p, memory_format=torch.contiguous_format)
                    st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.contiguous_format)
                if amsgrad and "max_exp_avg_sq" not in st:
                    st["max_exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.contiguous_format)
                if master is None:
                    master = self._group_scalar(st.get("step"), p.device, 0.0)
                st["step"] = master
                states.append((st["exp_avg"], st["exp_avg_sq"]) + ((st["max_exp_avg_sq"],) if amsgrad else ()))
            table, work, nitems = self._work(group, params, states)
            lr, lr_dev = self._lr_args(group)
            b1, b2 = group["betas"]
            rc = capi.lib().agcn_optim_adam(table.data_ptr(), work.data_ptr(), nitems, lr, lr_dev, float(b1), float(b2), float(group["eps"]),
                                            float(group["weight_decay"]), int(self._decoupled), int(amsgrad), int(group["maximize"]),
                                            master.data_ptr(), self._ptr(gs), self._ptr(fi), _stream(params[0].device))
            capi.check(rc, "agcn_optim_adam")
            if fi is None:
                master.add_(1.0)
            else:                                   # GradScaler skipped the step on overflow: the counter does not advance
                master.add_((fi == 0).to(torch.float32).reshape(()))
        return loss


class FusedAdamW(FusedAdam):
    """torch.optim.AdamW: decoupled weight decay (p *= 1 - lr * wd)."""
    _decoupled = True

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, amsgrad=False, maximize=False, **unused):
        super().__init__(params, lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, amsgrad=amsgrad, maximize=maximize)


class FusedASGD(_FusedOptimizer):
    """torch.optim.ASGD(params, lr, lambd, alpha, t0, weight_decay, maximize): averaged SGD with the state keys step / eta / mu / ax.

    torch keeps step, eta and mu per parameter, all equal; here they are ONE set of device scalars for the group, advanced inside
    the launch (state[p]["step"] of every parameter is the same tensor, likewise eta and mu).  ``state_dict()`` hands out a copy per
    parameter, so that torch.optim.ASGD loads it and advances each parameter's counters once per step."""
    _SCALARS = ("step", "eta", "mu")

    def __init__(self, params, lr=1e-2, lambd=1e-4, alpha=0.75, t0=1e6, weight_decay=0.0, maximize=False, **unused):
        super().__init__(params, dict(lr=lr, lambd=lambd, alpha=alpha, t0=t0, weight_decay=weight_decay, maximize=maximize))
        self._cache: Dict[int, tuple] = {}
        self._done: Dict[int, torch.Tensor] = {}         # per group: the kernel's block counter, zero between launches

    def state_dict(self):
        sd = super().state_dict()
        sd["state"] = {k: {n: v.clone() if n in self._SCALARS else v for n, v in st.items()} for k, st in sd["state"].items()}
        return sd

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        gs, fi = self._amp()
        for group in self.param_groups:
            params = self._tensors(group)
            if not params:
                continue
            dev = params[0].device
            shared, states = None, []
            for p in params:
                st = self.state[p]
                if "ax" not in st:
                    st["ax"] = torch.zeros_like(p, memory_format=torch.contiguous_format)
                if shared is None:                  # torch's initial state: step 0, eta = lr, mu = 1
                    shared = {"step": self._group_scalar(st.get("step"), dev, 0.0),
                              "eta": self._group_scalar(st.get("eta"), dev, float(group["lr"])),
                              "mu": self._group_scalar(st.get("mu"), dev, 1.0)}
                st.update(shared)
                states.append((st["ax"], None))
            table, work, nitems = self._work(group, params, states)
            lr, lr_dev = self._lr_args(group)
            done = self._done.get(id(group))
            if done is None:
                done = self._done[id(group)] = torch.zeros((), dtype=torch.int32, device=dev)
            rc = capi.lib().agcn_optim_asgd(table.data_ptr(), work.data_ptr(), nitems, lr, lr_dev, float(group["lambd"]),
                                            float(group["alpha"]), float(group["t0"]), float(group["weight_decay"]),
                                            int(group["maximize"]), shared["eta"].data_ptr(), shared["mu"].data_ptr(),
                                            shared["step"].data_ptr(), done.data_ptr(), self._ptr(gs), self._ptr(fi), _stream(dev))
            capi.check(rc, "agcn_optim_asgd")
        return loss


# the names the reference's YAML files use (torch_src/session_helper.py:48-53)
FUSED_OPTIMIZERS = {"SGD": FusedSGD, "ADAM": FusedAdam, "ADAMW": FusedAdamW, "ASGD": FusedASGD}
