"""Drop-in installer / launcher: runs the UNMODIFIED reference (main.py, YAML configs, fusion wrappers) on top of the
B200 unit.

The reference discovers its model with ``import_model(cfg.model)`` -> ``models.<name>.<name>.Model``
(torch_src/session/session.py:50, util/dynamic_import.py:29-38) and every multimodal wrapper builds the backbone as
``agcn.Model(...)`` through the module attribute (torch_src/models/mmargcn/early_fusion_models.py:18,36,71,108,144,187,
228,265; late_fusion_models.py:19,55; rgb_feature_models.py:22,43,89).  The reference tree is read-only, so the drop-in
is a rebinding of those module attributes:

    models.mmargcn.agcn.{TemporalConv, SpatialGraphConv, SpatialTemporalConv, Model}  -> fusion_gcn_b200.modules.*
    models.agcn.agcn.{unit_tcn, unit_gcn, TCN_GCN_unit, Model}                        -> fusion_gcn_b200.modules_original.*
    models.mmargcn.{graph_convolution, gcn}.{AGCNGraphConvolution, STGCNGraphConvolution} -> fusion_gcn_b200.graphconv.*

Usage (on a box that has both the reference checkout and a B200):

    python -m fusion_gcn_b200.dropin --reference /path/to/fusion-gcn [--precision fp32|tf32] -- -f config/<...>.yaml

which installs the import shims the reference needs on a current software stack (SURVEY D5 / Appendix D), rebinds the
classes and then ``runpy``s ``torch_src/main.py`` with cwd = the reference root (its config code scans cwd for models and
datasets, torch_src/config.py:21-41).  YAML files, main.py and the session code stay byte-identical.
"""
import importlib
import os
import runpy
import sys
from unittest.mock import MagicMock

_ORIGINALS = {}          # (module name, attribute) -> reference object, for uninstall()

_MMARGCN_NAMES = ("TemporalConv", "SpatialGraphConv", "SpatialTemporalConv", "Model")
_ORIGINAL_NAMES = ("unit_tcn", "unit_gcn", "TCN_GCN_unit", "Model")


def install_shims(reference_root: str, host_stubs: bool = True) -> None:
    """Makes the reference importable on numpy >= 1.24 / a box without matplotlib, seaborn or ray (SURVEY Appendix D)."""
    import numpy as np
    for p in (os.path.join(reference_root, "torch_src"), reference_root):
        if p not in sys.path:
            sys.path.insert(0, p)
    names = ["matplotlib", "matplotlib.pyplot"]
    if host_stubs:
        names += ["seaborn", "ray", "ray.tune", "ray.tune.schedulers"]
    for name in names:
        try:
            importlib.import_module(name)
        except Exception:                                   # absent (or broken) optional dependency: stub it
            sys.modules.setdefault(name, MagicMock(name=name))
    if not hasattr(np, "int"):
        np.int = int                                        # util/graph.py:75,88
    if not hasattr(np, "float"):
        np.float = float                                    # util/graph.py:117,127
    # np.bool is deliberately left alone (numpy >= 2 defines it; overriding it breaks numpy.ma / scipy)


def install(reference_root: str, precision="fp32", host_stubs: bool = True, fused_optimizers: bool = False, prefetch: bool = False,
            recompute: bool = False) -> dict:
    """Rebinds the reference's unit / backbone classes to the B200 implementations.  Returns the patched modules.
    ``fused_optimizers``: the YAML optimizer names SGD / ADAM / ADAMW / ASGD (torch_src/session_helper.py:48-53) build the multi-tensor
    classes of fusion_gcn_b200.optim.  ``prefetch``: the sessions' ``DataLoader`` (session/training.py:18-25, evaluation.py:20-24,
    debugging.py:15-21) becomes fusion_gcn_b200.pipeline.PrefetchLoader (same batches, pinned staging + asynchronous H2D)."""
    from . import modules, modules_original
    if not os.path.isfile(os.path.join(reference_root, "torch_src", "models", "mmargcn", "agcn.py")):
        raise FileNotFoundError(f"{reference_root} does not look like a fusion-gcn checkout (torch_src/models/mmargcn/agcn.py missing)")
    install_shims(reference_root, host_stubs)
    modules.set_default_precision(precision)
    modules.set_default_recompute(recompute)             # activation-recompute policy of the units the session builds
    ref_m = importlib.import_module("models.mmargcn.agcn")
    ref_o = importlib.import_module("models.agcn.agcn")
    for mod, names, impl in ((ref_m, _MMARGCN_NAMES, modules), (ref_o, _ORIGINAL_NAMES, modules_original)):
        for name in names:
            _ORIGINALS.setdefault((mod.__name__, name), getattr(mod, name))
            setattr(mod, name, getattr(impl, name))
    patched = {"models.mmargcn.agcn": ref_m, "models.agcn.agcn": ref_o}
    # 1-D graph convolutions of the IMU / late-fusion models (graph_convolution.py:12-113); gcn.py binds the names at import time
    from . import graphconv
    ref_g = importlib.import_module("models.mmargcn.graph_convolution")
    ref_gcn = importlib.import_module("models.mmargcn.gcn")
    for mod in (ref_g, ref_gcn):
        for name in ("AGCNGraphConvolution", "STGCNGraphConvolution"):
            _ORIGINALS.setdefault((mod.__name__, name), getattr(mod, name))
            setattr(mod, name, getattr(graphconv, name))
        patched[mod.__name__] = mod
    if fused_optimizers:
        from .optim import FUSED_OPTIMIZERS
        helper = importlib.import_module("session_helper")
        _ORIGINALS.setdefault((helper.__name__, "available_optimizers"), helper.available_optimizers)
        helper.available_optimizers = dict(helper.available_optimizers, **FUSED_OPTIMIZERS)
        patched["session_helper"] = helper
    if prefetch:
        import torch
        from .pipeline import PrefetchLoader
        device = "cuda" if torch.cuda.is_available() else "cpu"

        def loader(dataset, batch_size=1, shuffle=False, drop_last=False, **kw):
            return PrefetchLoader(dataset, batch_size, shuffle=shuffle, drop_last=drop_last, device=device)
        importlib.import_module("session_helper")      # first, as main.py does: session <-> session_helper import each other
        for name in ("session.training", "session.evaluation", "session.debugging"):
            mod = importlib.import_module(name)
            _ORIGINALS.setdefault((mod.__name__, "DataLoader"), mod.DataLoader)
            mod.DataLoader = loader
            patched[name] = mod
    return patched


def uninstall() -> None:
    """Restores the reference classes (used by the tests)."""
    for (mod_name, name), obj in _ORIGINALS.items():
        setattr(sys.modules[mod_name], name, obj)
    _ORIGINALS.clear()


def graph_step_key(model, features, label, loss_quotient=1):
    """The key under which ``--graph-step`` caches the captured training step of ``DefaultStep.forward(model, loss_function,
    features, label, loss_quotient)``, or None when that step has to run eagerly.

    A step is graphable when the features are a CUDA tensor or a dict of CUDA tensors (the fusion models' multimodal batches),
    the label is a CUDA tensor, ``loss_quotient >= 1``, the model is in training mode, grad mode is on and autocast is off
    (``MixedPrecisionStep``'s ``GradScaler`` is not captured).  The key holds the model's identity, every feature entry's name,
    shape and dtype, the label's shape and dtype and ``loss_quotient``: a replay of a graph captured under another key would
    read the wrong model, shapes or loss scale."""
    import torch
    entries = _cuda_entries(features)
    if entries is None or not (isinstance(label, torch.Tensor) and label.is_cuda):
        return None
    if not (loss_quotient >= 1 and model.training and torch.is_grad_enabled()) or torch.is_autocast_enabled():
        return None
    return (id(model), tuple((name, tuple(t.shape), t.dtype) for name, t in entries), tuple(label.shape), label.dtype, loss_quotient)


def graph_eval_key(model, features):
    """The key under which ``--graph-step`` caches the captured eval-mode forward (``graphed.GraphedForward``) of
    ``DefaultStep.forward(model, ...)``, or None when that forward has to run eagerly.

    A forward is graphable when the features are a batch-first CUDA tensor or a non-empty dict of them, the model is in eval mode,
    grad mode is off (the sessions' ``torch.no_grad()`` validation) and autocast is off.  The key holds the model's identity and
    every feature entry's name, trailing shape and dtype.  The batch size is not part of it: the graph serves any batch up to the
    captured one by zero padding."""
    import torch
    entries = _cuda_entries(features)
    if entries is None or any(t.dim() == 0 for _, t in entries):
        return None
    if model.training or torch.is_grad_enabled() or torch.is_autocast_enabled():
        return None
    return (id(model), tuple((name, tuple(t.shape[1:]), t.dtype) for name, t in entries))


def _cuda_entries(features):
    """[(name, tensor)] sorted by name (name None for a single tensor) when the features are a CUDA tensor or a non-empty dict of
    CUDA tensors, else None."""
    import torch
    if isinstance(features, torch.Tensor):
        entries = [(None, features)]
    elif isinstance(features, dict) and features and all(isinstance(v, torch.Tensor) for v in features.values()):
        entries = sorted(features.items(), key=lambda kv: str(kv[0]))
    else:
        return None
    return entries if all(t.is_cuda for _, t in entries) else None


def _graph_steps() -> None:
    """The sessions' training step (procedures/step.py:39-46: forward, loss, backward launched op by op from Python) replayed as ONE
    CUDA graph per step.  At the reference's own batch sizes (8 - 10, SURVEY appendix E) the eager single-tensor step is launch
    bound: 20.8 ms against 11.2 ms replayed at 8 sequences (profiles/r17_bench_b8.json).  ``DefaultStep.forward`` builds a
    ``graphed.GraphedStep`` lazily on the first graphable training batch (``graph_step_key``; BatchNorm buffers preserved across the
    warm-up), replays it for every batch of that key and hands back (logits, loss / loss_quotient); ``DefaultStep.backward`` then only
    re-attaches the graph's static gradients (the session's ``optimizer.zero_grad()`` sets them to None).  Dict features of the
    fusion models are captured like a tensor.  With ``loss_quotient > 1`` (gradient accumulation, batch_train.py:63) the graph adds
    each micro-batch's gradient into its static gradients: a step whose gradients are all None starts a new sum (``zero_grads()``),
    a step whose gradients are all the graph's own adds to it, and any other state (gradients of an eager step) runs eagerly.
    Autocast and a second training key (another model, batch shape -- a shorter last batch -- or quotient) take the reference's own
    code path; only one training graph is cached.

    Evaluation (``validate_epoch`` and the evaluation sessions: eval mode under ``torch.no_grad()``, ``graph_eval_key``) gets a graph
    of its own beside the training graph: a ``graphed.GraphedForward`` of the model's forward, built lazily on the first such batch
    and replayed for every batch of that key with at most as many sequences, so a shorter last batch is zero-padded to the captured
    size and sliced afterwards.  The step hands back a clone of the replayed logits as ``y_pred`` (the session keeps it for its
    metrics; the next replay overwrites the graph's output) and computes ``loss_function(y_pred, label) / loss_quotient`` eagerly, as
    the reference does.  A larger batch, another key, eval under autocast or with gradients runs eagerly; a failed eval capture is
    reported on stderr and leaves evaluation eager for the rest of the session, the training graph untouched."""
    import torch
    from .graphed import GraphedForward, GraphedStep
    importlib.import_module("session_helper")          # first, as main.py does: session <-> session_helper import each other
    step = importlib.import_module("session.procedures.step")
    inner_forward, inner_backward = step.DefaultStep.forward, step.DefaultStep.backward
    state = {"graph": None, "key": None, "pending": None, "disabled": False,
             "eval": None, "eval_key": None, "eval_disabled": False}

    def forward(self, model, loss_function, features, label, loss_quotient=1):
        state["pending"] = None
        key = None if state["disabled"] else graph_step_key(model, features, label, loss_quotient)
        if key is not None:
            trainable = [p for p in model.parameters() if p.requires_grad]
            fresh = all(p.grad is None for p in trainable)
            if state["graph"] is None and fresh:        # (capture resets .grad: never over gradients the session still holds)
                try:
                    state["graph"] = GraphedStep(model, loss_function, features, label, warmup=2, preserve_buffers=True,
                                                 accumulate=loss_quotient > 1, loss_divisor=loss_quotient)
                    state["key"] = key
                except Exception as exc:                 # noqa: BLE001 -- the eager step stands in for the rest of the session
                    state["disabled"] = True
                    model.zero_grad(set_to_none=True)
                    print(f"fusion_gcn_b200.dropin: CUDA-graph step disabled ({type(exc).__name__}: {exc})", file=sys.stderr)
            gs = state["graph"]
            if gs is not None and key == state["key"]:
                static = {id(p): g for p, g in gs.grads}
                if fresh and gs.accumulate:
                    gs.zero_grads()
                if fresh or (gs.accumulate and all(p.grad is static.get(id(p)) for p in trainable)):
                    loss = gs(features, label)
                    state["pending"] = gs
                    return gs.logits, loss
        eval_key = None if state["eval_disabled"] else graph_eval_key(model, features)
        if eval_key is not None:
            if state["eval"] is None:
                try:
                    state["eval"], state["eval_key"] = GraphedForward(model, features, warmup=2), eval_key
                except Exception as exc:                 # noqa: BLE001 -- evaluation stays eager, the training graph is kept
                    state["eval_disabled"] = True
                    print(f"fusion_gcn_b200.dropin: CUDA-graph evaluation disabled ({type(exc).__name__}: {exc})", file=sys.stderr)
            gf = state["eval"]
            rows = {t.shape[0] for t in (features.values() if isinstance(features, dict) else [features])}
            if gf is not None and eval_key == state["eval_key"] and len(rows) == 1 and 1 <= min(rows) <= gf.batch_size:
                y_pred = gf(features).clone()
                return y_pred, loss_function(y_pred, label) / loss_quotient
        return inner_forward(self, model, loss_function, features, label, loss_quotient)

    def backward(self, loss):
        gs, state["pending"] = state["pending"], None
        if gs is not None and loss is gs.loss:
            gs.attach_grads()                            # the replay already ran the backward
        else:
            inner_backward(self, loss)
    step.DefaultStep.forward, step.DefaultStep.backward = forward, backward


def _trace_losses(path: str) -> None:
    """Appends every training-step loss (procedures/step.py:39-43) to ``path`` as text, one value per line."""
    importlib.import_module("session_helper")          # first, as main.py does: session <-> session_helper import each other
    step = importlib.import_module("session.procedures.step")
    inner = step.DefaultStep.forward

    def forward(self, model, loss_function, features, label, loss_quotient=1):
        y_pred, loss = inner(self, model, loss_function, features, label, loss_quotient)
        if model.training:
            with open(path, "a") as fh:
                fh.write(repr(float(loss.detach())) + "\n")
        return y_pred, loss
    step.DefaultStep.forward = forward


def main(argv=None) -> None:
    argv = list(sys.argv[1:] if argv is None else argv)
    rest = []
    if "--" in argv:
        i = argv.index("--")
        argv, rest = argv[:i], argv[i + 1:]
    import argparse
    ap = argparse.ArgumentParser(prog="python -m fusion_gcn_b200.dropin", description=__doc__.split("\n")[0])
    ap.add_argument("--reference", default=os.environ.get("FUSION_GCN_REFERENCE", "/root/reference"))
    ap.add_argument("--precision", default="fp32", choices=["fp32", "bf16x3", "tf32", "fp32_ffma"])
    ap.add_argument("--recompute", action="store_true", help="units recompute theta / phi and the aggregated tensor in the backward (~40 %% less activation memory)")
    ap.add_argument("--graph-step", action="store_true", help="replay the training step (forward + loss + backward) as one CUDA graph per "
                    "batch, and the evaluation forward (eval mode, no_grad; a shorter last batch zero-padded) as another")
    ap.add_argument("--no-dropin", action="store_true", help="run the UNMODIFIED reference under the same import shims (A/B baseline)")
    ap.add_argument("--reference-fp32", action="store_true", help="with --no-dropin: disable cuDNN / cuBLAS TF32 so the reference is an fp32 oracle (SURVEY D9)")
    ap.add_argument("--no-fused-optimizers", action="store_true", help="keep torch.optim instead of fusion_gcn_b200.optim")
    ap.add_argument("--no-prefetch", action="store_true", help="keep torch's DataLoader instead of fusion_gcn_b200.pipeline.PrefetchLoader")
    ap.add_argument("--trace-loss", default=None, metavar="FILE", help="append every training-step loss to FILE")
    args = ap.parse_args(argv)
    root = os.path.abspath(args.reference)
    if args.no_dropin:
        if not os.path.isfile(os.path.join(root, "torch_src", "main.py")):
            raise FileNotFoundError(f"{root} does not look like a fusion-gcn checkout")
        install_shims(root)
        if args.reference_fp32:
            import torch
            torch.backends.cudnn.allow_tf32 = False
            torch.backends.cuda.matmul.allow_tf32 = False
    else:
        install(root, args.precision, fused_optimizers=not args.no_fused_optimizers, prefetch=not args.no_prefetch, recompute=args.recompute)
        from . import capi
        capi.lib()                                           # fail before training starts if the extension is not built
        if args.graph_step:
            _graph_steps()
    if args.trace_loss:
        _trace_losses(args.trace_loss)
    os.chdir(root)
    sys.argv = [os.path.join(root, "torch_src", "main.py")] + rest
    runpy.run_path(sys.argv[0], run_name="__main__")


if __name__ == "__main__":
    main()
