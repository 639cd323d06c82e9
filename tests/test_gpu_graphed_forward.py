"""-m gpu: the eval-mode forward replayed as one CUDA graph (graphed.GraphedForward), and the launcher's evaluation graph under
--graph-step (dropin.graph_eval_key and the DefaultStep wrapper).

The captured forward launches the same kernels as the eager forward at the captured batch size, so a replay is compared with
torch.equal against eager ``model(x)`` under ``no_grad`` at that size.  A shorter batch of n sequences is zero-padded to the captured
size: its logits are bit-identical to the first n rows of the eager forward of the padded batch, and within rounding of the eager
forward of the n sequences alone (the eager kernels pick their T-chunking from the batch size, so their sums run in another order)."""
import copy
import sys
import types

import pytest
import torch

import fusion_wrapper as FW
from helpers import rel_err

pytestmark = pytest.mark.gpu
B = 8


@pytest.fixture(scope="module")
def pkg():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import fusion_gcn_b200
    from fusion_gcn_b200 import capi
    capi.lib()
    return fusion_gcn_b200


def _ntu_model():
    from fusion_gcn_b200 import graph as G, modules as M
    graph = G.SkeletonGraph(G.NTU_EDGES, center_joint=G.NTU_CENTER)
    return M.Model((2, 300, 25, 3), 60, graph).cuda()


def _ntu_batch(n, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, 2, 300, 25, 3, generator=g).cuda()


def _pad(x, rows):
    if isinstance(x, dict):
        return {k: _pad(v, rows) for k, v in x.items()}
    return torch.cat([x, x.new_zeros(rows - x.shape[0], *x.shape[1:])])


def _head(x, n):
    return {k: v[:n] for k, v in x.items()} if isinstance(x, dict) else x[:n]


def _eager(model, x):
    with torch.no_grad():
        return model(x)


def _check_replays(model, batches, shorter=(1, 5)):
    """Every full batch replays bit-identical to the eager forward; every shorter one to the padded eager forward's first rows and
    within 1e-5 of the eager forward of its n sequences."""
    from fusion_gcn_b200.graphed import GraphedForward
    gf = GraphedForward(model, batches[0])
    assert gf.launches_per_replay > 50
    for i, x in enumerate(batches):
        logits = gf(x)
        ref = _eager(model, x)
        torch.cuda.synchronize()
        assert logits.shape == ref.shape and torch.equal(logits, ref), i
    x = batches[-1]
    for n in shorter:
        logits = gf(_head(x, n)).clone()
        padded = _eager(model, _pad(_head(x, n), B))[:n]
        alone = _eager(model, _head(x, n))
        torch.cuda.synchronize()
        assert logits.shape == alone.shape, n
        assert torch.equal(logits, padded), n
        assert rel_err(logits, alone) <= 1e-5, n
    return gf


def test_replay_matches_eager_bitwise_and_serves_shorter_batches(pkg):
    torch.manual_seed(21)
    model = _ntu_model().eval()
    _check_replays(model, [_ntu_batch(B, seed=s) for s in range(4)])


def test_dict_input_replay_matches_eager(pkg):
    """The skeleton + inertial fusion model: dict batches, and the 40-node large-graph kernels inside the capture."""
    torch.manual_seed(22)
    model = FW.SkeletonInertialNet().cuda().eval()
    _check_replays(model, [FW.batch(B, seed=s)[0] for s in range(4)])


def test_grad_mode_of_the_caller_does_not_matter(pkg):
    """Warm-up and capture run under no_grad whatever the caller's grad mode: nothing is saved for a backward."""
    from fusion_gcn_b200.graphed import GraphedForward
    torch.manual_seed(23)
    model = FW.SkeletonInertialNet().cuda().eval()
    x = FW.batch(B, seed=1)[0]
    with torch.enable_grad():
        gf = GraphedForward(model, x)
        logits = gf(x)
    assert not logits.requires_grad
    assert torch.equal(logits, _eager(model, x))
    assert all(p.grad is None for p in model.parameters())


def test_attention_maps_view_the_graph(pkg):
    from fusion_gcn_b200.graphed import GraphedForward
    torch.manual_seed(24)
    model = _ntu_model().eval()
    x = _ntu_batch(B, seed=3)
    gf = GraphedForward(model, x)
    units = [m for m in model.modules() if isinstance(getattr(m, "adj_c", None), list)]
    assert len(units) == 10 and len(gf.attention) == 10
    n = 5
    gf(x[:n])
    torch.cuda.synchronize()
    got = [[a.clone() for a in m.adj_c] for m in units]
    graph_ptrs = [[a.data_ptr() for a in m.adj_c] for m in units]
    _eager(model, x[:n])                                 # rebinds every adj_c to the eager tensors
    torch.cuda.synchronize()
    assert any(m.adj_c[0].data_ptr() != p[0] for m, p in zip(units, graph_ptrs))
    for u, (m, maps) in enumerate(zip(units, got)):
        for k in range(3):
            assert maps[k].shape == (n * 2, 25, 25), (u, k)
            assert rel_err(maps[k], m.adj_c[k]) <= 1e-5, (u, k)
    gf(x[:n])
    for m, maps, ptrs in zip(units, got, graph_ptrs):
        assert [a.data_ptr() for a in m.adj_c] == ptrs
        assert all(a.shape == b.shape for a, b in zip(m.adj_c, maps))
    gf(x)
    assert all(a.shape[0] == B * 2 for m in units for a in m.adj_c)


def test_updates_between_replays_are_picked_up(pkg):
    """Training replays (GraphedStep) + FusedSGD steps move the parameters and the BatchNorm running statistics in place; every
    eval replay in between equals the eager eval of the same model state."""
    from fusion_gcn_b200.graphed import GraphedForward, GraphedStep
    from fusion_gcn_b200.optim import FusedSGD
    torch.manual_seed(25)
    model = FW.SkeletonInertialNet().cuda().train()
    loss_fn = torch.nn.CrossEntropyLoss()
    train = [FW.batch(B, seed=30 + s) for s in range(3)]
    evals = [FW.batch(B, seed=40 + s)[0] for s in range(3)]
    opt = FusedSGD(model.parameters(), lr=0.05, momentum=0.9)
    gs = GraphedStep(model, loss_fn, *train[0], warmup=2)
    model.eval()
    gf = GraphedForward(model, evals[0])
    stats = [b.clone() for b in model.buffers()]
    for s in range(3):
        gs(*train[s])
        opt.step()
        for n in (B, 3):
            x = _head(evals[s], n)
            logits = gf(x)
            ref = _eager(model, _pad(x, B))[:n]
            torch.cuda.synchronize()
            assert torch.equal(logits, ref), (s, n)
    assert any(not torch.equal(a, b) for a, b in zip(model.buffers(), stats)), "the running statistics did not move"
    # load_state_dict copies in place: the replay reads the loaded weights
    other = FW.SkeletonInertialNet().cuda().eval()
    model.load_state_dict(other.state_dict())
    assert torch.equal(gf(evals[0]), _eager(other, evals[0]))


def test_refusals(pkg):
    from fusion_gcn_b200.graphed import GraphedForward
    torch.manual_seed(26)
    model = FW.SkeletonInertialNet().cuda()
    x = FW.batch(4, seed=5)[0]
    with pytest.raises(ValueError, match="eval"):
        GraphedForward(model.train(), x)
    model.eval()
    with pytest.raises(ValueError, match="batch size"):
        GraphedForward(model, dict(x, inertial=x["inertial"][:3]))
    gf = GraphedForward(model, x)
    big = FW.batch(5, seed=6)[0]
    for bad, name in ((big, "'skeleton'"),                                              # n > B
                      (dict(x, skeleton=x["skeleton"][:0]), "'skeleton'"),              # n = 0
                      (dict(x, inertial=x["inertial"][:, :, :39]), "'inertial'"),       # trailing shape
                      (dict(x, skeleton=x["skeleton"].double()), "'skeleton'"),         # dtype
                      (dict(x, skeleton=x["skeleton"].cpu()), "'skeleton'"),            # device
                      ({"skeleton": x["skeleton"]}, "'inertial'"),                      # missing key
                      (dict(x, extra=x["inertial"]), "'extra'"),                        # extra key
                      (dict(x, inertial=x["inertial"][:2]), "'inertial'")):             # entries with different n
        with pytest.raises(ValueError, match=name):
            gf(bad)
    with pytest.raises(ValueError):
        gf(x["skeleton"])
    single = _ntu_model().eval()
    xs = _ntu_batch(2, seed=7)
    gs = GraphedForward(single, xs)
    for bad in (_ntu_batch(3, seed=8), xs[:, :, :299], xs.double(), {"skeleton": xs}):
        with pytest.raises(ValueError, match="input"):
            gs(bad)


# ---------------------------------------------------------------------------------------------------- the launcher's decision
def test_graph_eval_key(pkg):
    from fusion_gcn_b200.dropin import graph_eval_key
    model = FW.SkeletonInertialNet().cuda().eval()
    x, _ = FW.batch(4)
    with torch.no_grad():
        key = graph_eval_key(model, x)
        assert key is not None
        assert graph_eval_key(model, x["skeleton"]) is not None
        assert graph_eval_key(model, {k: v.cpu() for k, v in x.items()}) is None
        assert graph_eval_key(model, dict(x, inertial=x["inertial"].cpu())) is None
        assert graph_eval_key(model, {}) is None
        with torch.autocast("cuda", dtype=torch.float16):
            assert graph_eval_key(model, x) is None
        model.train()
        assert graph_eval_key(model, x) is None
        model.eval()
        assert graph_eval_key(model, dict(reversed(list(x.items())))) == key          # the dict's order does not matter
        assert graph_eval_key(model, _head(x, 3)) == key                               # nor the batch size
        assert graph_eval_key(model, FW.batch(9)[0]) == key
        assert graph_eval_key(model, dict(x, inertial=x["inertial"][:, :, :39].contiguous())) != key
        assert graph_eval_key(model, dict(x, skeleton=x["skeleton"][:, :, :20].contiguous())) != key
        assert graph_eval_key(model, dict(x, skeleton=x["skeleton"].double())) != key
        assert graph_eval_key(model, {"skel": x["skeleton"], "inertial": x["inertial"]}) != key
        assert graph_eval_key(copy.deepcopy(model), x) != key
    assert graph_eval_key(model, x) is None                                            # grad mode on


class _DefaultStep:
    """procedures/step.py:38-49 of the reference restated: the class the launcher's --graph-step wraps."""

    def forward(self, model, loss_function, features, label, loss_quotient=1):
        y_pred = model(features)
        loss = loss_function(y_pred, label) / loss_quotient
        return y_pred, loss

    def backward(self, loss):
        loss.backward()


def _assert_same(model, twin, what):
    for (k, p), q in zip(model.named_parameters(), twin.parameters()):
        assert (p.grad is None) == (q.grad is None), (what, k)
        assert p.grad is None or torch.equal(p.grad, q.grad), (what, "grad", k)
        assert torch.equal(p, q), (what, "parameter", k)
    for (k, a), b in zip(model.named_buffers(), twin.buffers()):
        assert torch.equal(a, b), (what, "buffer", k)


def test_launcher_graphs_validation_passes(pkg, monkeypatch):
    """The --graph-step wrapper of DefaultStep over a session of graphed training steps + FusedSGD, with a validation pass
    (model.eval() + no_grad, last batch shorter) after every epoch.  Every validation batch replays the eval graph; y_pred and the
    loss equal an eager twin session (bitwise for full batches, within 1e-5 for the shorter one, which the twin runs unpadded); a
    y_pred kept from an earlier batch survives later replays; training is bit-identical to the twin; eval under autocast or with
    gradients stays eager."""
    from fusion_gcn_b200 import dropin, graphed
    from fusion_gcn_b200.optim import FusedSGD
    replays = {"train": 0, "eval": 0}

    class CountingStep(graphed.GraphedStep):
        def __call__(self, x=None, y=None):
            replays["train"] += 1
            return super().__call__(x, y)

    class CountingForward(graphed.GraphedForward):
        def __call__(self, x):
            replays["eval"] += 1
            return super().__call__(x)

    monkeypatch.setattr(graphed, "GraphedStep", CountingStep)
    monkeypatch.setattr(graphed, "GraphedForward", CountingForward)
    step_mod = types.ModuleType("session.procedures.step")
    step_mod.DefaultStep = type("DefaultStep", (_DefaultStep,), {})
    for name, mod in (("session_helper", types.ModuleType("session_helper")), ("session", types.ModuleType("session")),
                      ("session.procedures", types.ModuleType("session.procedures")), ("session.procedures.step", step_mod)):
        monkeypatch.setitem(sys.modules, name, mod)
    dropin._graph_steps()
    graph_session, eager_session = step_mod.DefaultStep(), _DefaultStep()

    torch.manual_seed(27)
    model = FW.SkeletonInertialNet().cuda().train()
    twin = copy.deepcopy(model)
    loss_fn = torch.nn.CrossEntropyLoss()
    opt, opt_twin = FusedSGD(model.parameters(), lr=0.05, momentum=0.9), FusedSGD(twin.parameters(), lr=0.05, momentum=0.9)
    val = [FW.batch(n, seed=70 + i) for i, n in enumerate((4, 4, 3))]
    kept = []
    for epoch in range(3):
        model.train()
        twin.train()
        for i in range(2):
            x, y = FW.batch(4, seed=50 + 2 * epoch + i)
            before = replays["train"]
            _, loss = graph_session.forward(model, loss_fn, x, y, 1)
            graph_session.backward(loss)
            _, ref = eager_session.forward(twin, loss_fn, x, y, 1)
            eager_session.backward(ref)
            opt.step()
            opt_twin.step()
            opt.zero_grad()
            opt_twin.zero_grad()
            torch.cuda.synchronize()
            assert replays["train"] == before + 1, (epoch, i)
            assert torch.equal(loss.detach(), ref.detach()), (epoch, i)
            _assert_same(model, twin, f"epoch {epoch} step {i}")
        model.eval()
        twin.eval()
        with torch.no_grad():
            for i, (x, y) in enumerate(val):
                before = replays["eval"]
                y_pred, loss = graph_session.forward(model, loss_fn, x, y, 1)
                ref_pred, ref = eager_session.forward(twin, loss_fn, x, y, 1)
                torch.cuda.synchronize()
                assert replays["eval"] == before + 1, (epoch, i)
                if x["skeleton"].shape[0] == 4:
                    assert torch.equal(y_pred, ref_pred) and torch.equal(loss, ref), (epoch, i)
                else:
                    assert rel_err(y_pred, ref_pred) <= 1e-5 and rel_err(loss, ref) <= 1e-5, (epoch, i)
                kept.append((y_pred, y_pred.clone()))
        for y_pred, copy_ in kept:
            assert torch.equal(y_pred, copy_)
        _assert_same(model, twin, f"after validation {epoch}")
    before = dict(replays)
    x, y = val[0]
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
        graph_session.forward(model, loss_fn, x, y, 1)
    graph_session.forward(model, loss_fn, x, y, 1)                     # eval mode, grad mode on
    big = FW.batch(5, seed=90)
    with torch.no_grad():
        graph_session.forward(model, loss_fn, *big, 1)                 # more sequences than the graph holds
    torch.cuda.synchronize()
    assert replays == before
