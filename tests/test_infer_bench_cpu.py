"""CPU: tools/infer_bench.py parses its arguments without a GPU and, having no CPU fallback, exits non-zero without one."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCRIPT = os.path.join(ROOT, "tools", "infer_bench.py")


def test_help():
    r = subprocess.run([sys.executable, SCRIPT, "--help"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "--blank-bias" in r.stdout and "--precision" in r.stdout


def test_no_gpu_exits_nonzero():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, SCRIPT, "--n", "4"], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode != 0
    assert r.stdout.strip() == ""
