"""bench.py --dump-outputs: what the timed step computed in its last step, written as .npy files for output-for-output comparison of
two builds."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import check_grads, rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N = 4                 # sequences per benchmark step in the GPU tests


def test_dump_outputs_writes_every_array_and_samples_past_the_budget(tmp_path, monkeypatch):
    import bench
    arrays = {"loss": np.float32(1.5).reshape(()), "logits": np.arange(600, dtype=np.float32).reshape(20, 30),
              "grad.w": np.linspace(-1, 1, 400).astype(np.float32)}
    bench.dump_outputs(str(tmp_path / "full"), arrays)
    for k, a in arrays.items():
        got = np.load(tmp_path / "full" / (k + ".npy"))
        assert got.dtype == np.float32 and np.array_equal(got, a), k
    monkeypatch.setattr(bench, "DUMP_BUDGET", 1000)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays)
    a = {k: np.load(tmp_path / "a" / (k + ".npy")) for k in arrays}
    b = {k: np.load(tmp_path / "b" / (k + ".npy")) for k in arrays}
    assert sum(v.nbytes for v in a.values()) <= 1000
    for k in arrays:
        assert np.array_equal(a[k], b[k]) and a[k].size >= 1, k                 # a fixed sample: the same elements every run
        assert np.isin(a[k], arrays[k]).all() and (np.diff(a[k]) > 0).all(), k   # elements of the array, in their original order


def _bench(out_dir, *extra):
    """bench.py at the UTD shape, N=4, two timed steps, dumping into out_dir: (JSON line, {name: array})."""
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "utd", "--batch", str(N), "--steps", "2", "--warmup", "1",
           "--no-cpu-baseline", "--no-tf32", "--dump-outputs", str(out_dir), *extra]
    out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2
    return line, {p.name[:-4]: np.load(p) for p in out_dir.glob("*.npy")}


def _seeded_batch():
    """The benchmark's batch: the same generator, seed and draws as bench.py (rank 0)."""
    import bench
    m, t, v, c, ncls, _ = bench.WORKLOADS["utd"]
    gen = torch.Generator().manual_seed(1234)
    x = torch.randn(N, m, t, v, c, generator=gen)
    return x.cuda(), torch.randint(ncls, (N,), generator=gen).cuda()


def _check_step(got, want, what):
    assert set(got) == set(want), what
    assert all(a.dtype == np.float32 for a in got.values()), what
    assert got["logits"].shape == tuple(want["logits"].shape) and got["loss"].shape == (), what
    assert rel_err(got["loss"], want["loss"]) <= 1e-5 and rel_err(got["logits"], want["logits"]) <= 1e-5, what
    check_grads({k[5:]: v for k, v in got.items() if k.startswith("grad.")}, {k[5:]: v for k, v in want.items() if k.startswith("grad.")},
                1e-5, what)


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_training_step(tmp_path):
    """The dump is the training step's loss, logits and parameter gradients (recomputed here from the benchmark's seeded model and
    batch), the same arrays on a second run with the same arguments, and the same step on the eager path (--no-graph)."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import bench
    from fusion_gcn_b200.graphed import loss_and_logits
    model = bench.build_model("utd", "fp32", "cuda")
    x, y = _seeded_batch()
    loss, logits = loss_and_logits(model, torch.nn.CrossEntropyLoss(), x, y)
    loss.backward()
    want = {"loss": loss, "logits": logits}
    want.update({"grad." + k: p.grad for k, p in model.named_parameters()})
    want = {k: v.detach().double().cpu() for k, v in want.items()}

    line, got = _bench(tmp_path / "graph")
    assert "last_loss" in line["graph_mode"], line["graph_mode"]          # the headline path is the captured step graph
    _check_step(got, want, "graph")
    assert abs(float(got["loss"]) - line["graph_mode"]["last_loss"]) <= 1e-4
    _, again = _bench(tmp_path / "again")
    for k in got:                                                           # same arguments, same inputs: the same outputs
        assert np.array_equal(again[k], got[k]), k
    line, eager = _bench(tmp_path / "eager", "--no-graph")
    assert line["config"]["launch_mode"] == "eager launches"
    _check_step(eager, want, "eager")


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_inference_step(tmp_path):
    """--mode infer dumps the logits of the last timed forward: eval mode, the benchmark's seeded model and batch."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import bench
    model = bench.build_model("utd", "fp32", "cuda").eval()
    x, _ = _seeded_batch()
    with torch.no_grad():
        want = model(x)
    _, got = _bench(tmp_path, "--mode", "infer")
    assert set(got) == {"logits"} and got["logits"].dtype == np.float32 and got["logits"].shape == tuple(want.shape)
    assert rel_err(got["logits"], want) <= 1e-5
