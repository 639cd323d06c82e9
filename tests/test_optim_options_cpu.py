"""The fused optimizers' options and ASGD without a GPU: constructor arguments and parameter-group keys against torch.optim, the
optimizer names against the reference's table, and the argument checks of agcn_optim_asgd through the C ABI."""
import ast
import os

import pytest
import torch

from oracle import ref_loader

TORCH = {"SGD": torch.optim.SGD, "ADAM": torch.optim.Adam, "ADAMW": torch.optim.AdamW, "ASGD": torch.optim.ASGD}
OPTIONS = [
    ("SGD", dict(lr=0.1, momentum=0.9, nesterov=True, maximize=True)),
    ("ADAM", dict(lr=1e-3, amsgrad=True)),
    ("ADAM", dict(lr=1e-3, amsgrad=True, maximize=True)),
    ("ADAMW", dict(lr=1e-3, weight_decay=0.05, amsgrad=True, maximize=True)),
    ("ASGD", dict()),
    ("ASGD", dict(lr=0.05, lambd=1e-3, alpha=0.5, t0=2, weight_decay=1e-3, maximize=True)),
]


@pytest.mark.parametrize("name,kw", OPTIONS)
def test_fused_groups_carry_torchs_keys_and_values(name, kw):
    """Every hyper-parameter the fused class keeps in its group is one torch's class keeps, under the same name and with the same
    value, defaults included (the class is built on CPU parameters: construction needs no device)."""
    from fusion_gcn_b200 import optim
    ours = optim.FUSED_OPTIMIZERS[name]([torch.nn.Parameter(torch.zeros(3))], **kw).param_groups[0]
    ref = TORCH[name]([torch.nn.Parameter(torch.zeros(3))], **kw).param_groups[0]
    assert "maximize" in ours and (name not in ("ADAM", "ADAMW") or "amsgrad" in ours)
    for key, value in ours.items():
        if key != "params":
            assert key in ref and ref[key] == value, key


def test_fused_asgd_has_torchs_constructor_defaults():
    from fusion_gcn_b200 import optim
    group = optim.FusedASGD([torch.nn.Parameter(torch.zeros(3))]).param_groups[0]
    assert {k: group[k] for k in ("lr", "lambd", "alpha", "t0", "weight_decay", "maximize")} == \
        dict(lr=1e-2, lambd=1e-4, alpha=0.75, t0=1e6, weight_decay=0, maximize=False)
    optim.FusedASGD([torch.nn.Parameter(torch.zeros(3))], foreach=True, capturable=True)        # absorbed, as by the other classes


def test_a_checkpoint_without_maximize_loads_with_the_default():
    """A fused checkpoint written before ``maximize`` existed has no such key in its groups; loading it leaves the option off."""
    from fusion_gcn_b200 import optim
    opt = optim.FusedSGD([torch.nn.Parameter(torch.zeros(3))], lr=0.1, maximize=True)
    sd = opt.state_dict()
    del sd["param_groups"][0]["maximize"]
    opt.load_state_dict(sd)
    assert opt.param_groups[0]["maximize"] is False


def test_fused_optimizer_names_match_the_reference_table():
    """FUSED_OPTIMIZERS replaces entries of session_helper.available_optimizers (dropin.install): the names must be the table's."""
    if not ref_loader.available():
        pytest.skip("reference copy not present")
    from fusion_gcn_b200 import optim
    tree = ast.parse(open(os.path.join(ref_loader.REFERENCE_ROOT, "torch_src", "session_helper.py")).read())
    tables = [node.value for node in ast.walk(tree) if isinstance(node, ast.Assign) and isinstance(node.value, ast.Dict)
              and any(isinstance(t, ast.Name) and t.id == "available_optimizers" for t in node.targets)]
    assert len(tables) == 1
    assert sorted(k.value for k in tables[0].keys) == sorted(optim.FUSED_OPTIMIZERS)


def _asgd(lib, table=8, items=8, nitems=1, eta=16, mu=16, step=16, done=16):
    return lib.agcn_optim_asgd(table, items, nitems, 0.01, None, 1e-4, 0.75, 1e6, 0.0, 0, eta, mu, step, done, None, None, None)


@pytest.mark.parametrize("operands,status,message", [
    (dict(table=None), 6, b"null table"),
    (dict(items=None), 6, b"null table"),
    (dict(nitems=0), 1, b"empty work list"),
    (dict(table=12), 3, b"not 8-byte aligned"),
    (dict(eta=None), 6, b"null eta / mu / step / done"),
    (dict(mu=None), 6, b"null eta / mu / step / done"),
    (dict(step=None), 6, b"null eta / mu / step / done"),
    (dict(done=None), 6, b"null eta / mu / step / done"),
])
def test_asgd_entry_point_rejects_bad_operands_without_gpu(operands, status, message):
    """agcn_optim_asgd checks its table, work list and scalars before it launches anything, so a CPU box sees the rejections."""
    from fusion_gcn_b200 import build, capi
    build.build()
    lib = capi.lib()
    assert lib.agcn_version() == 102
    assert _asgd(lib, **operands) == status and message in lib.agcn_last_error_string()
