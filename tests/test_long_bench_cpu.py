"""CPU: tools/long_bench.py parses its arguments without a GPU and, having no CPU fallback, exits non-zero without one; its
byte count is the one DESIGN §4.12 states."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCRIPT = os.path.join(ROOT, "tools", "long_bench.py")


def test_help():
    r = subprocess.run([sys.executable, SCRIPT, "--help"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "--blank-bias" in r.stdout and "--skip-model" in r.stdout


def test_no_gpu_exits_nonzero():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, SCRIPT, "--skip-model", "--iters", "1"], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode != 0
    assert r.stdout.strip() == ""


def test_softmax_bytes():
    sys.path.insert(0, ROOT)
    from tools.long_bench import softmax_bytes
    # bf16/bf16: forward reads ac + bd and writes probs (6 B per element); backward reads probs + dprobs, writes dscores + dbd (8 B)
    assert softmax_bytes(10, 1032, 2, 2) == (10 * 1032 * 6, 10 * 1032 * 8)
    assert softmax_bytes(3, 2048, 4, 4) == (3 * 2048 * 12, 3 * 2048 * 16)
