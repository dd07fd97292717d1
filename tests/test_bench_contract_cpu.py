"""CPU: the JSON contract of ``bench.py --impl reference`` (the arm the driver runs next to the GPU arm): one line on rank 0 with
the GPU arm's metric / unit / direction, ``impl``, a ``cpu_baseline`` describing the run and an ``e2e`` object with zero copy
bytes; the other ranks of a torchrun launch print nothing and exit 0.  Runs the small configs[0] workload (4 layers, batch 8)."""
import json
import os
import subprocess
import sys
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra):
    env = dict(os.environ, **env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c1", "--steps", "1", "--warmup", "1"],
                          capture_output=True, text=True, env=env, timeout=600)


def test_reference_arm_prints_the_contract_line_on_rank_0_only():
    r = _run({"RANK": "0"})
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"].startswith("audio-sec/sec train") and d["unit"] == "audio-s/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["steps"] == 1 and d["n_gpus"] == 1 and "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and "utterances" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0
    other = _run({"RANK": "1"})
    assert other.returncode == 0 and other.stdout.strip() == ""


def test_dump_outputs_writes_a_fixed_sample_of_the_step_results(tmp_path, monkeypatch):
    """--dump-outputs: arrays named after what the step returns (float32; the optimizer's counters float64); the parameter /
    gradient sample is the same seeded set of positions in every run, in state_dict order, and holds the model's own values."""
    import numpy as np
    import torch
    import bench
    torch.manual_seed(0)
    model = torch.nn.Sequential(torch.nn.Linear(6, 5), torch.nn.BatchNorm1d(5), torch.nn.Linear(5, 3))
    with torch.no_grad():
        for p in model.parameters():  # distinct values: a sampled value identifies its position
            p.uniform_(-1.0, 1.0)
    model(torch.randn(4, 6)).sum().backward()
    model.last_losses = torch.tensor([3.0, 2.0, 4.0])
    opt = SimpleNamespace(state=torch.tensor([7.0, 1.5, 2e-4, 0.0, 1.0, 0.0, 0.0, 0.0]))  # [updates, grad norm, lr, ...]
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 17)
    bench.dump_outputs(str(tmp_path / "a"), model, opt, torch.tensor(3.0))
    bench.dump_outputs(str(tmp_path / "b"), model, opt, torch.tensor(3.0))
    names = {"loss", "loss_terms", "params_sample", "grads_sample", "bn_running_stats", "optimizer_state"}
    assert {p.name for p in (tmp_path / "a").iterdir()} == {n + ".npy" for n in names}
    got = {n: np.load(tmp_path / "a" / f"{n}.npy") for n in names}
    for n in names:
        assert got[n].dtype == (np.float64 if n == "optimizer_state" else np.float32), n
        assert np.array_equal(got[n], np.load(tmp_path / "b" / f"{n}.npy")), n
    assert got["loss"] == 3.0 and got["loss_terms"].tolist() == [3.0, 2.0, 4.0]
    assert got["optimizer_state"].tolist() == opt.state[:3].double().tolist()
    flat_p = torch.cat([p.detach().reshape(-1) for p in model.parameters()]).numpy()
    flat_g = torch.cat([p.grad.reshape(-1) for p in model.parameters()]).numpy()
    assert got["params_sample"].shape == got["grads_sample"].shape == (17,)
    pos = [int(np.flatnonzero(flat_p == v)[0]) for v in got["params_sample"]]
    assert pos == sorted(set(pos)) and np.array_equal(flat_g[pos], got["grads_sample"])
    bn = model[1]
    assert np.array_equal(got["bn_running_stats"], torch.cat([bn.running_mean, bn.running_var]).numpy())
