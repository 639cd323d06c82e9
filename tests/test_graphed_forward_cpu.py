"""not gpu: what the CUDA-graph eval forward (graphed.GraphedForward) and the launcher's evaluation decision (dropin.graph_eval_key)
refuse on the host.  There is no CPU path: host tensors, in a dict as alone, are rejected before anything is captured."""
import pytest
import torch

from fusion_gcn_b200.dropin import graph_eval_key
from fusion_gcn_b200.graphed import GraphedForward


@pytest.fixture(scope="module")
def pkg():
    import fusion_gcn_b200
    return fusion_gcn_b200


def test_graphed_forward_refuses_host_tensors(pkg):
    model = torch.nn.Linear(4, 3).eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        GraphedForward(model, torch.zeros(2, 4))
    with pytest.raises(RuntimeError, match="'inertial'"):
        GraphedForward(model, {"inertial": torch.zeros(2, 4)})


def test_graphed_forward_refuses_a_training_mode_model(pkg):
    with pytest.raises(ValueError, match="eval"):
        GraphedForward(torch.nn.Linear(4, 3).train(), torch.zeros(2, 4))


def test_graph_eval_key_rejects_host_features(pkg):
    model = torch.nn.Linear(4, 3).eval()
    with torch.no_grad():
        assert graph_eval_key(model, torch.zeros(2, 4)) is None
        assert graph_eval_key(model, {"skeleton": torch.zeros(2, 4), "inertial": torch.zeros(2, 4)}) is None
        assert graph_eval_key(model, {}) is None
        assert graph_eval_key(model, [torch.zeros(2, 4)]) is None
