"""-m gpu: the CUDA-graph training step (graphed.GraphedStep) with dict (multimodal) inputs and with gradient accumulation, and the
launcher's decision of which steps it graphs (dropin.graph_step_key and the --graph-step wrapper of DefaultStep).

The captured step launches the same kernels in the same order as the eager step, so wherever both take the same loss head the
results are compared with torch.equal: loss, logits, every gradient and every buffer (running statistics, num_batches_tracked).
Every op of the fusion wrapper (tests/fusion_wrapper.py: the package's kernels, torch.cat / mean, nn.Linear, cross-entropy) is
bitwise reproducible under capture.  The NTU model's graphed step takes the fused classifier + cross-entropy head (Model.loss), its
eager twin torch's: those are held to the tolerances of test_gpu_unit.py::test_graphed_step_matches_eager."""
import copy
import sys
import types

import pytest
import torch

import fusion_wrapper as FW
from helpers import ZERO_GRAD, rel_err, stat_err

pytestmark = pytest.mark.gpu
LQ = 3                                  # micro-batches per optimizer step


@pytest.fixture(scope="module")
def pkg():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import fusion_gcn_b200
    from fusion_gcn_b200 import capi
    capi.lib()
    return fusion_gcn_b200


def _assert_same(model, twin, what):
    for (k, p), q in zip(model.named_parameters(), twin.parameters()):
        assert (p.grad is None) == (q.grad is None), (what, k)
        assert p.grad is None or torch.equal(p.grad, q.grad), (what, "grad", k)
        assert torch.equal(p, q), (what, "parameter", k)
    for (k, a), b in zip(model.named_buffers(), twin.buffers()):
        assert torch.equal(a, b), (what, "buffer", k)


def _eager(model, loss_fn, x, y, divisor=1):
    logits = model(x)
    loss = loss_fn(logits, y)
    if divisor != 1:
        loss = loss / divisor
    loss.backward()
    return loss.detach(), logits.detach()


def test_dict_input_replay_matches_eager_bitwise(pkg):
    from fusion_gcn_b200.graphed import GraphedStep
    torch.manual_seed(11)
    model = FW.SkeletonInertialNet().cuda().train()
    twin = copy.deepcopy(model)
    loss_fn = torch.nn.CrossEntropyLoss()
    batches = [FW.batch(5, seed=s) for s in range(4)]
    warm = 2
    step = GraphedStep(model, loss_fn, *batches[0], warmup=warm)
    assert step.launches_per_replay > 100
    for _ in range(warm):                       # the twin sees the same number of warm-up steps (running statistics)
        twin.zero_grad(set_to_none=True)
        _eager(twin, loss_fn, *batches[0])
    for i, (x, y) in enumerate(batches[1:]):    # every replay overwrites the gradients: the twin zeroes before each step
        loss = step(x, y)
        twin.zero_grad(set_to_none=True)
        ref, logits = _eager(twin, loss_fn, x, y)
        torch.cuda.synchronize()
        assert torch.equal(loss, ref) and torch.equal(step.logits, logits), i
        _assert_same(model, twin, f"step {i}")
    # the static inputs are the captured keys, shapes, dtypes and device: anything else is refused before the copy
    x, y = batches[1]
    for bad, name in (({"skeleton": x["skeleton"]}, "'inertial'"),
                      (dict(x, extra=x["inertial"]), "'extra'"),
                      (dict(x, inertial=x["inertial"][:4]), "'inertial'"),
                      (dict(x, skeleton=x["skeleton"].double()), "'skeleton'"),
                      (dict(x, skeleton=x["skeleton"].cpu()), "'skeleton'")):
        with pytest.raises(ValueError, match=name):
            step(bad, y)
    with pytest.raises(ValueError):
        step(x["skeleton"], y)


def test_replay_without_accumulate_overwrites_the_gradients(pkg):
    from fusion_gcn_b200.graphed import GraphedStep
    torch.manual_seed(12)
    model = FW.SkeletonInertialNet().cuda().train()
    loss_fn = torch.nn.CrossEntropyLoss()
    (xa, ya), (xb, yb) = FW.batch(4, seed=1), FW.batch(4, seed=2)
    twin = copy.deepcopy(model)
    step = GraphedStep(model, loss_fn, xa, ya, warmup=1, preserve_buffers=True)
    step(xa, ya)
    _eager(twin, loss_fn, xa, ya)
    step(xb, yb)
    twin.zero_grad(set_to_none=True)
    _eager(twin, loss_fn, xb, yb)
    torch.cuda.synchronize()
    _assert_same(model, twin, "second replay")


def _ntu_model():
    from fusion_gcn_b200 import graph as G, modules as M
    graph = G.SkeletonGraph(G.NTU_EDGES, center_joint=G.NTU_CENTER)
    return M.Model((2, 300, 25, 3), 60, graph).cuda().train()


def _assert_close(named, ref, what):
    """The tolerances of test_gpu_unit.py::test_graphed_step_matches_eager (fused head against torch's): 2e-5 relative per tensor,
    and on the absolute scale 1e-6 x the largest magnitude for the mathematically-zero families and for tensors already below that
    level (the phi-bias gradients of the first units are ~1e-11 here, ten orders under the largest gradient: rounding of the two
    heads alone moves them by a few 1e-5 of their own size)."""
    scale = max(float(q.abs().max()) for q in ref)
    for (k, p), q in zip(named, ref):
        if ZERO_GRAD.search(k) or float(q.abs().max()) <= 1e-6 * scale:
            assert float((p - q).abs().max()) <= 1e-6 * scale, (what, k)
        else:
            assert rel_err(p, q) <= 2e-5, (what, k)


def test_accumulated_replays_match_eager_accumulation_fused_head(pkg):
    """NTU model, 4 sequences per micro-batch, loss / 3 over 3 micro-batches per FusedSGD step, two steps.  The graphed step takes
    the fused classifier + cross-entropy head, which receives the 1/3 as its device-side loss gradient.  Against an eager twin on the
    same head every loss, gradient, parameter and buffer is bit-identical; against a twin on torch's head (classifier, then
    nn.CrossEntropyLoss) they agree to the fused head's rounding.  That twin starts every optimizer step from the graphed model's
    parameters and buffers: carried through an optimizer step, the two heads' rounding flips ReLU inputs that lie within rounding of
    zero and moves whole gradient tensors by ~1e-2 (measured: data_bn.weight 1.2e-2 at the second step), which says nothing about
    the capture."""
    from fusion_gcn_b200.graphed import GraphedStep, loss_and_logits
    from fusion_gcn_b200.optim import FusedSGD
    torch.manual_seed(13)
    model = _ntu_model()
    same_head, torch_head = copy.deepcopy(model), copy.deepcopy(model)
    loss_fn = torch.nn.CrossEntropyLoss()

    def fused(m, x, y):
        loss, _ = loss_and_logits(m, loss_fn, x, y)
        loss = loss / LQ
        loss.backward()
        return loss.detach()

    def plain(m, x, y):
        return _eager(m, loss_fn, x, y, LQ)[0]

    g = torch.Generator().manual_seed(5)
    xs = [torch.randn(4, 2, 300, 25, 3, generator=g).cuda() for _ in range(2 * LQ)]
    ys = [torch.randint(60, (4,), generator=g).cuda() for _ in range(2 * LQ)]
    twins = [(same_head, fused), (torch_head, plain)]
    opts = [FusedSGD(m.parameters(), lr=0.01, momentum=0.9) for m in (model, same_head, torch_head)]
    warm = 2
    step = GraphedStep(model, loss_fn, xs[0], ys[0], warmup=warm, accumulate=True, loss_divisor=LQ)
    for twin, run in twins:
        for _ in range(warm):
            twin.zero_grad(set_to_none=True)
            run(twin, xs[0], ys[0])
        twin.zero_grad(set_to_none=True)
    assert all(float(g.abs().max()) == 0.0 for _, g in step.grads), "the warm-up left something in the static gradients"
    for s in range(2):
        step.zero_grads()
        torch_head.load_state_dict(model.state_dict())
        for o in opts[1:]:
            o.zero_grad()
        for i in range(LQ):
            x, y = xs[s * LQ + i], ys[s * LQ + i]
            loss = step(x, y)
            ref_same, ref_torch = fused(same_head, x, y), plain(torch_head, x, y)
            torch.cuda.synchronize()
            assert torch.equal(loss, ref_same), (s, i)
            _assert_same(model, same_head, f"step {s} micro-batch {i}")
            assert rel_err(loss, ref_torch) <= 1e-6, (s, i)
            _assert_close([(k, p.grad) for k, p in model.named_parameters()], [q.grad for q in torch_head.parameters()], (s, i))
        for o in opts:
            o.step()
        torch.cuda.synchronize()
        _assert_same(model, same_head, f"after optimizer step {s}")
        _assert_close([(k, p.detach()) for k, p in model.named_parameters()], [q.detach() for q in torch_head.parameters()], s)
    for (k, a), b in zip(model.named_buffers(), torch_head.buffers()):
        assert stat_err(a, b) <= 1e-6, k


def test_accumulated_replays_match_eager_accumulation_dict_input(pkg):
    from fusion_gcn_b200.graphed import GraphedStep
    from fusion_gcn_b200.optim import FusedSGD
    torch.manual_seed(14)
    model = FW.SkeletonInertialNet().cuda().train()
    twin = copy.deepcopy(model)
    loss_fn = torch.nn.CrossEntropyLoss()
    batches = [FW.batch(4, seed=20 + s) for s in range(2 * LQ)]
    opt, opt_twin = FusedSGD(model.parameters(), lr=0.05, momentum=0.9), FusedSGD(twin.parameters(), lr=0.05, momentum=0.9)
    step = GraphedStep(model, loss_fn, *batches[0], warmup=2, accumulate=True, loss_divisor=LQ, preserve_buffers=True)
    for s in range(2):
        step.zero_grads()
        opt_twin.zero_grad()
        for i in range(LQ):
            x, y = batches[s * LQ + i]
            loss = step(x, y)
            ref, logits = _eager(twin, loss_fn, x, y, LQ)
            torch.cuda.synchronize()
            assert torch.equal(loss, ref) and torch.equal(step.logits, logits), (s, i)
            _assert_same(model, twin, f"step {s} micro-batch {i}")
        opt.step()
        opt_twin.step()
        torch.cuda.synchronize()
        _assert_same(model, twin, f"after optimizer step {s}")


# ---------------------------------------------------------------------------------------------------- the launcher's decision
def test_graph_step_key(pkg):
    from fusion_gcn_b200.dropin import graph_step_key
    model = FW.SkeletonInertialNet().cuda().train()
    x, y = FW.batch(4)
    key = graph_step_key(model, x, y, 1)
    assert key is not None
    assert graph_step_key(model, x["skeleton"], y, 1) is not None
    assert graph_step_key(model, {k: v.cpu() for k, v in x.items()}, y, 1) is None
    assert graph_step_key(model, dict(x, inertial=x["inertial"].cpu()), y, 1) is None
    assert graph_step_key(model, x, y.cpu(), 1) is None
    assert graph_step_key(model, x, y, 0) is None
    with torch.no_grad():
        assert graph_step_key(model, x, y, 1) is None
    with torch.autocast("cuda", dtype=torch.float16):
        assert graph_step_key(model, x, y, 1) is None
    model.eval()
    assert graph_step_key(model, x, y, 1) is None
    model.train()
    assert graph_step_key(model, dict(reversed(list(x.items()))), y, 1) == key          # the dict's order does not matter
    assert graph_step_key(model, dict(x, inertial=x["inertial"][:, :, :39].contiguous()), y, 1) != key
    assert graph_step_key(model, dict(x, skeleton=x["skeleton"][:, :, :20].contiguous()), y, 1) != key
    assert graph_step_key(model, dict(x, skeleton=x["skeleton"].double()), y, 1) != key
    assert graph_step_key(model, {"skel": x["skeleton"], "inertial": x["inertial"]}, y, 1) != key
    assert graph_step_key(model, x, y[:, None], 1) != key
    assert graph_step_key(model, x, y, 2) != key
    assert graph_step_key(copy.deepcopy(model), x, y, 1) != key


class _DefaultStep:
    """procedures/step.py:38-49 of the reference restated: the class the launcher's --graph-step wraps."""

    def forward(self, model, loss_function, features, label, loss_quotient=1):
        y_pred = model(features)
        loss = loss_function(y_pred, label) / loss_quotient
        return y_pred, loss

    def backward(self, loss):
        loss.backward()


def test_launcher_graph_step_accumulates_like_the_eager_session(pkg, monkeypatch):
    """The --graph-step wrapper of DefaultStep over a gradient-accumulating session (loss_quotient = 3, optimizer.zero_grad()
    after every optimizer step), with steps that must stay eager mixed in: a shorter batch (another key) in the middle of a sum and
    at the start of one.  Every loss, gradient, parameter and buffer equals the same session run eagerly, bit for bit, and the
    graph is replayed exactly for the steps it may take."""
    from fusion_gcn_b200 import dropin, graphed
    from fusion_gcn_b200.optim import FusedSGD
    replays = []

    class Counting(graphed.GraphedStep):
        def __call__(self, x=None, y=None):
            replays.append(True)
            return super().__call__(x, y)

    monkeypatch.setattr(graphed, "GraphedStep", Counting)
    step_mod = types.ModuleType("session.procedures.step")
    step_mod.DefaultStep = type("DefaultStep", (_DefaultStep,), {})
    for name, mod in (("session_helper", types.ModuleType("session_helper")), ("session", types.ModuleType("session")),
                      ("session.procedures", types.ModuleType("session.procedures")), ("session.procedures.step", step_mod)):
        monkeypatch.setitem(sys.modules, name, mod)
    dropin._graph_steps()
    assert step_mod.DefaultStep.forward is not _DefaultStep.forward
    graph_session, eager_session = step_mod.DefaultStep(), _DefaultStep()

    torch.manual_seed(15)
    model = FW.SkeletonInertialNet().cuda().train()
    twin = copy.deepcopy(model)
    loss_fn = torch.nn.CrossEntropyLoss()
    opt, opt_twin = FusedSGD(model.parameters(), lr=0.05, momentum=0.9), FusedSGD(twin.parameters(), lr=0.05, momentum=0.9)
    # (batch size, expected to replay): three optimizer steps of LQ micro-batches each
    plan = [(4, True), (3, False), (4, True),           # a shorter batch adds eagerly into the graph's own gradients
            (3, False), (4, False), (4, False),         # a sum started eagerly stays eager
            (4, True), (4, True), (4, True)]
    for i, (n, graphed_expected) in enumerate(plan):
        x, y = FW.batch(n, seed=40 + i)
        before = len(replays)
        _, loss = graph_session.forward(model, loss_fn, x, y, LQ)
        graph_session.backward(loss)
        _, ref = eager_session.forward(twin, loss_fn, x, y, LQ)
        eager_session.backward(ref)
        torch.cuda.synchronize()
        assert (len(replays) > before) == graphed_expected, i
        assert torch.equal(loss.detach(), ref.detach()), i
        _assert_same(model, twin, f"micro-batch {i}")
        if i % LQ == LQ - 1:
            opt.step()
            opt_twin.step()
            opt.zero_grad()
            opt_twin.zero_grad()
            torch.cuda.synchronize()
            _assert_same(model, twin, f"after optimizer step {i // LQ}")
