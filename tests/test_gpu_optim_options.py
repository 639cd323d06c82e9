"""-m gpu: the options of the fused optimizers -- AMSGrad (Adam / AdamW), maximize (SGD / Adam / AdamW) -- and the fused ASGD,
against torch.optim with the same arguments: under a learning-rate scheduler with ONE launch per step, across state_dict round
trips with torch, through GradScaler with a skipped overflow step, and inside a captured training-step graph."""
import copy

import pytest
import torch

from helpers import rel_err

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def O():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from fusion_gcn_b200 import capi, optim
    capi.lib()
    return optim


def make_params(seed=0):
    g = torch.Generator().manual_seed(seed)
    shapes = [(64, 3, 1, 1), (64,), (3, 25, 25), (256, 256, 9, 1), (60, 256), (1,), (128, 64, 1, 1), (5000,)]
    return [torch.nn.Parameter(torch.randn(*s, generator=g).cuda()) for s in shapes]


def grads_for(params, step, seed=100):
    g = torch.Generator().manual_seed(seed + step)
    return [torch.randn(*p.shape, generator=g).cuda() * 0.1 for p in params]


TORCH = {"SGD": torch.optim.SGD, "ADAM": torch.optim.Adam, "ADAMW": torch.optim.AdamW, "ASGD": torch.optim.ASGD}
# beta2 = 0.5 lets exp_avg_sq fall below its running maximum within six steps, so AMSGrad's maximum decides the step
AMSGRAD_ADAM = ("ADAM", dict(lr=1e-3, betas=(0.9, 0.5), weight_decay=0.01, amsgrad=True))
# t0 = 2: mu < 1 from step 4 on (averaging acts); lambd and weight decay large enough to move the parameters visibly
ASGD_AVERAGING = ("ASGD", dict(lr=0.05, lambd=1e-2, t0=2, weight_decay=1e-2))
CASES = [
    AMSGRAD_ADAM,
    ("ADAM", dict(lr=1e-3, amsgrad=True)),
    ("ADAMW", dict(lr=1e-3, betas=(0.9, 0.5), weight_decay=0.05, amsgrad=True)),
    ("SGD", dict(lr=0.05, maximize=True)),
    ("SGD", dict(lr=0.1, momentum=0.9, nesterov=True, weight_decay=1e-4, maximize=True)),
    ("ADAM", dict(lr=1e-3, weight_decay=0.01, maximize=True)),
    ("ADAMW", dict(lr=1e-3, weight_decay=0.05, maximize=True)),
    ("ADAM", dict(lr=3e-3, betas=(0.8, 0.5), eps=1e-6, amsgrad=True, maximize=True)),
    ("ADAMW", dict(lr=1e-3, betas=(0.9, 0.5), weight_decay=0.05, amsgrad=True, maximize=True)),
    ("ASGD", dict()),
    ASGD_AVERAGING,
    ("ASGD", dict(lr=0.05, lambd=1e-2, t0=3, weight_decay=1e-2, maximize=True)),
]


def assert_states_match(ours, ref, tol=2e-6):
    """Every state entry torch keeps (max_exp_avg_sq, ax, eta, mu, step, ...) exists in the fused state and agrees."""
    sd_ref, sd_ours = ref.state_dict(), ours.state_dict()
    for k, st in sd_ref["state"].items():
        assert st.keys() == sd_ours["state"][k].keys(), k
        for key, val in st.items():
            assert rel_err(sd_ours["state"][k][key], val) <= tol, (k, key)


def run_steps(ref, ours, p_ref, p_ours, steps, schedulers=()):
    for step in steps:
        for a, b, g in zip(p_ref, p_ours, grads_for(p_ref, step)):
            a.grad, b.grad = g.clone(), g.clone()
        ref.step(); ours.step()
        for s in schedulers:
            s.step()


@pytest.mark.parametrize("name,kw", CASES)
def test_options_match_torch_optim_with_scheduler(O, name, kw):
    from fusion_gcn_b200 import capi
    p_ref, p_ours = make_params(), make_params()
    ref, ours = TORCH[name](p_ref, **kw), O.FUSED_OPTIMIZERS[name](p_ours, **kw)
    scheds = [torch.optim.lr_scheduler.MultiStepLR(o, milestones=[2, 4], gamma=0.5) for o in (ref, ours)]
    before = capi.lib().agcn_launch_count()
    run_steps(ref, ours, p_ref, p_ours, range(6), scheds)
    assert capi.lib().agcn_launch_count() - before == 6          # ONE launch per step for all eight tensors
    for a, b in zip(p_ref, p_ours):
        assert rel_err(b, a) <= 2e-6
    assert ref.param_groups[0]["lr"] == ours.param_groups[0]["lr"]
    assert_states_match(ours, ref)
    st = ref.state[p_ref[3]]
    if kw.get("amsgrad") and kw.get("betas", (0, 0.999))[1] == 0.5:     # the maximum took part
        assert not torch.equal(st["max_exp_avg_sq"], st["exp_avg_sq"])
    if name == "ASGD" and kw.get("t0", 1e6) < 6:                        # the average lags the parameters
        assert float(st["mu"]) < 1 and not torch.allclose(st["ax"], p_ref[3])


@pytest.mark.parametrize("name,kw", [AMSGRAD_ADAM, ASGD_AVERAGING])
def test_state_dict_round_trip_through_the_fused_class(O, name, kw):
    """torch -> fused -> torch: a torch checkpoint loads into the fused class, which then steps as torch does; the fused state
    loads back into torch.optim.  ASGD's fused state_dict() carries one copy of step / eta / mu per parameter, so torch.optim.ASGD
    trains on from it identically.  (The Adam state goes back with ONE step tensor shared by the group -- the CUDA step counter of
    the fused Adam classes, a separate matter -- so that leg checks the loaded state only.)"""
    p_ref, p_ours = make_params(1), make_params(1)
    ref = TORCH[name](p_ref, **kw)
    for step in range(2):
        for a, g in zip(p_ref, grads_for(p_ref, step)):
            a.grad = g
        ref.step()
    for a, b in zip(p_ref, p_ours):
        b.data.copy_(a.data)
    ours = O.FUSED_OPTIMIZERS[name](p_ours, **kw)
    ours.load_state_dict(copy.deepcopy(ref.state_dict()))
    run_steps(ref, ours, p_ref, p_ours, range(2, 5))
    for a, b in zip(p_ref, p_ours):
        assert rel_err(b, a) <= 2e-6
    assert_states_match(ours, ref)
    p_back = make_params(1)
    for a, b in zip(p_ref, p_back):
        b.data.copy_(a.data)
    back = TORCH[name](p_back, **kw)
    back.load_state_dict(copy.deepcopy(ours.state_dict()))
    assert_states_match(back, ours, tol=0.0)
    if name == "ASGD":
        for step in range(5, 8):
            for a, b, g in zip(p_ref, p_back, grads_for(p_ref, step)):
                a.grad, b.grad = g.clone(), g.clone()
            ref.step(); back.step()
        for a, b in zip(p_ref, p_back):
            assert rel_err(b, a) <= 2e-6
        assert_states_match(back, ref)


def test_torch_amsgrad_checkpoint_into_a_fused_adam_built_without_it(O):
    """The options live in the parameter groups: a torch AMSGrad checkpoint switches AMSGrad on in a FusedAdam constructed
    without it, which then keeps max_exp_avg_sq and steps as torch does."""
    name, kw = AMSGRAD_ADAM
    p_ref, p_ours = make_params(3), make_params(3)
    ref = torch.optim.Adam(p_ref, **kw)
    for step in range(2):
        for a, g in zip(p_ref, grads_for(p_ref, step)):
            a.grad = g
        ref.step()
    for a, b in zip(p_ref, p_ours):
        b.data.copy_(a.data)
    ours = O.FusedAdam(p_ours, lr=kw["lr"], betas=kw["betas"], weight_decay=kw["weight_decay"])
    assert ours.param_groups[0]["amsgrad"] is False
    ours.load_state_dict(copy.deepcopy(ref.state_dict()))
    assert ours.param_groups[0]["amsgrad"] is True
    run_steps(ref, ours, p_ref, p_ours, range(2, 6))
    for a, b in zip(p_ref, p_ours):
        assert rel_err(b, a) <= 2e-6
    assert_states_match(ours, ref)


def _snapshot(opt, params):
    return [p.detach().clone() for p in params], {id(p): {k: v.clone() for k, v in opt.state[p].items()} for p in params}


@pytest.mark.parametrize("name,kw", [AMSGRAD_ADAM, ASGD_AVERAGING])
def test_gradscaler_overflow_step_leaves_everything_untouched(O, name, kw):
    """GradScaler with an inf in step 2: the fused step is skipped on the device -- parameters and every state entry (including
    max_exp_avg_sq, ax and ASGD's eta / mu / step) stay bit for bit -- and the run ends where torch's ends."""
    p_ref, p_ours = make_params(2), make_params(2)
    ref, ours = TORCH[name](p_ref, **kw), O.FUSED_OPTIMIZERS[name](p_ours, **kw)
    sc_ref = torch.amp.GradScaler("cuda", init_scale=256.0, growth_interval=1000)
    sc_ours = torch.amp.GradScaler("cuda", init_scale=256.0, growth_interval=1000)
    for sc in (sc_ref, sc_ours):
        sc.scale(torch.zeros(1, device="cuda"))
    for step in range(6):
        gs = grads_for(p_ref, step)
        if step == 2:
            gs[3][0, 0, 0, 0] = float("inf")
            params0, state0 = _snapshot(ours, p_ours)
        for a, b, g in zip(p_ref, p_ours, gs):
            a.grad, b.grad = g * sc_ref.get_scale(), g * sc_ours.get_scale()
        sc_ref.step(ref); sc_ref.update()
        sc_ours.step(ours); sc_ours.update()
        assert sc_ref.get_scale() == sc_ours.get_scale()
        if step == 2:
            params1, state1 = _snapshot(ours, p_ours)
            assert all(torch.equal(a, b) for a, b in zip(params0, params1))
            assert state0.keys() == state1.keys()
            for k, st in state0.items():
                assert st.keys() == state1[k].keys() and all(torch.equal(v, state1[k][n]) for n, v in st.items()), k
    assert sc_ours.get_scale() == 128.0
    for a, b in zip(p_ref, p_ours):
        assert torch.isfinite(b).all() and rel_err(b, a) <= 2e-6
    assert_states_match(ours, ref)


ADAM_STATE = ("exp_avg", "exp_avg_sq", "max_exp_avg_sq")


@pytest.mark.parametrize("name,kw", [("ADAM", dict(lr=1e-3, weight_decay=1e-4, amsgrad=True)),
                                     ("ASGD", dict(lr=0.02, lambd=1e-2, t0=0, weight_decay=1e-4))])
def test_optimizer_step_inside_the_captured_step_graph(O, name, kw):
    """FusedAdam(amsgrad=True) / FusedASGD as GraphedStep(after_backward=opt.step): with the state created before capture, the
    first replay (zero-grad + forward + backward + the optimizer step, ASGD's scalar update included) matches one eager torch step
    on a twin model."""
    from fusion_gcn_b200 import graph as G, modules as M
    from fusion_gcn_b200.graphed import GraphedStep, loss_and_logits
    torch.manual_seed(1)
    graph = G.SkeletonGraph(G.UTD_EDGES, center_joint=G.UTD_CENTER)
    m1 = M.Model((1, 16, 20, 3), 27, graph, start_feature_size=16).cuda().train()
    m2 = copy.deepcopy(m1)
    x = torch.randn(4, 1, 16, 20, 3, device="cuda")
    y = torch.randint(0, 27, (4,), device="cuda")
    lf = torch.nn.CrossEntropyLoss()
    o1 = O.FUSED_OPTIMIZERS[name](m1.parameters(), **kw)

    def reset_state(create):             # torch's initial state; reset in place once the graph holds the tensors' addresses
        for p in m1.parameters():
            st = o1.state[p]
            if create:
                st.update({k: torch.zeros_like(p) for k in (ADAM_STATE if name == "ADAM" else ("ax",))})
                st["step"] = torch.zeros((), device="cuda")
                if name == "ASGD":
                    st["eta"], st["mu"] = torch.full((), kw["lr"], device="cuda"), torch.ones((), device="cuda")
            else:
                for k, v in st.items():
                    v.fill_(kw["lr"] if k == "eta" else 1.0 if k == "mu" else 0.0)
    reset_state(True)
    state0 = copy.deepcopy(m1.state_dict())
    step = GraphedStep(m1, lf, x, y, warmup=1, after_backward=o1.step)
    m1.load_state_dict(state0)
    reset_state(False)
    o2 = TORCH[name](m2.parameters(), **kw)
    step()
    o2.zero_grad(set_to_none=True)
    loss_and_logits(m2, lf, x, y)[0].backward()
    o2.step()
    torch.cuda.synchronize()
    for (k, a), (_, b) in zip(m2.named_parameters(), m1.named_parameters()):
        assert rel_err(b, a) <= 2e-6, k
        for key, val in o2.state[a].items():
            assert rel_err(o1.state[b][key], val) <= 2e-6, (k, key)
