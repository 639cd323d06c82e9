"""not gpu: what the CUDA-graph step (graphed.GraphedStep) and the launcher's --graph-step decision (dropin.graph_step_key) refuse on
the host.  There is no CPU path: host tensors, in a dict as alone, are rejected before anything is captured."""
import pytest
import torch

from fusion_gcn_b200.dropin import graph_step_key
from fusion_gcn_b200.graphed import GraphedStep


def test_graphed_step_refuses_host_tensors():
    model = torch.nn.Linear(4, 3)
    y = torch.zeros(2, dtype=torch.int64)
    with pytest.raises(RuntimeError, match="CUDA"):
        GraphedStep(model, torch.nn.CrossEntropyLoss(), torch.zeros(2, 4), y)
    with pytest.raises(RuntimeError, match="'inertial'"):
        GraphedStep(model, torch.nn.CrossEntropyLoss(), {"inertial": torch.zeros(2, 4)}, y)


def test_graph_step_key_rejects_host_features():
    model = torch.nn.Linear(4, 3).train()
    y = torch.zeros(2, dtype=torch.int64)
    assert graph_step_key(model, torch.zeros(2, 4), y, 1) is None
    assert graph_step_key(model, {"skeleton": torch.zeros(2, 4), "inertial": torch.zeros(2, 4)}, y, 2) is None
    assert graph_step_key(model, {}, y, 1) is None
    assert graph_step_key(model, [torch.zeros(2, 4)], y, 1) is None
