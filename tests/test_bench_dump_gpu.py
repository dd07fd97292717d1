"""GPU: ``bench.py --dump-outputs`` on the timed path (the small configs[0] workload, headline numbers only).

Two runs with the same arguments write the same arrays: the inputs are seeded, so the only differences left are the order of
floating-point atomics in the gradient reductions.  A different batch or initialisation would differ by orders of magnitude
more.  The optimizer's update count in the dump is that of the last timed step: bench.py runs 5 eager steps, ``max(3, W)``
warm-up replays, ``K`` timed replays, 2 end-to-end warm-up steps and ``K`` timed end-to-end steps before it dumps, so one
more ``--steps`` is exactly two more updates."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("loss", "loss_terms", "params_sample", "grads_sample", "bn_running_stats", "optimizer_state")


def _bench(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--workload", "c1", "--quick", "--steps", str(steps),
                        "--warmup", "1", "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0]), {n: np.load(os.path.join(out_dir, n + ".npy")) for n in NAMES}


def _rel(x, y):
    return np.linalg.norm(x.astype(np.float64) - y) / np.linalg.norm(x)


def test_dump_outputs_same_arguments_same_arrays(tmp_path):
    line, a = _bench(tmp_path / "a", 3)
    assert sorted(os.listdir(tmp_path / "a")) == sorted(n + ".npy" for n in NAMES)
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for n, v in a.items():
        assert v.dtype == (np.float64 if n == "optimizer_state" else np.float32) and np.isfinite(v).all(), n
    assert a["loss"] == a["loss_terms"][0] and a["loss"] > 0
    assert np.abs(a["grads_sample"]).max() > 0 and a["bn_running_stats"].size > 0
    assert a["optimizer_state"][0] == 5 + line["warmup"] + 2 + 2 * 3
    _, b = _bench(tmp_path / "b", 3)
    # rel-L2 between two runs of the bench workload on a B200: loss 1e-6, parameters 1e-7, BatchNorm statistics 1e-5, gradients 2e-4
    for n, tol in (("loss_terms", 1e-4), ("params_sample", 1e-5), ("bn_running_stats", 1e-3), ("grads_sample", 2e-3)):
        assert _rel(a[n], b[n]) <= tol, (n, _rel(a[n], b[n]))
    assert b["optimizer_state"][0] == a["optimizer_state"][0]
    # one more timed step: two more updates, and parameters further from the first run than run-to-run noise
    _, c = _bench(tmp_path / "c", 4)
    assert c["optimizer_state"][0] == a["optimizer_state"][0] + 2
    assert _rel(a["params_sample"], c["params_sample"]) > 10 * _rel(a["params_sample"], b["params_sample"])
