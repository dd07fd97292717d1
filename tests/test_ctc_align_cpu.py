"""CPU: the forced-alignment ABI (include/lasr_align.h), the numpy reference the GPU test trusts, the frame -> seconds
conversion and tools/align_bench.py's command line."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from ctc_align_ref import brute_force_best, collapse, emissions, min_frames, viterbi
from test_abi_bindings_cpu import _C_KIND, _Recorder  # the recorder and C-type table of the lasr.h binding check

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCRIPT = os.path.join(ROOT, "tools", "align_bench.py")


def _align_prototypes():
    import re
    from liteasr_b200 import _lib
    src = re.sub(r"/\*.*?\*/", "", open(_lib.ALIGN_HEADER_PATH).read(), flags=re.S)
    src = re.sub(r"#.*", "", src)
    protos = {}
    for m in re.finditer(r"\b(lasr_[a-z0-9_]+)\s*\(([^()]*)\)\s*;", src):
        kinds = []
        for p in " ".join(m.group(2).split()).split(","):
            p = p.strip()
            kinds.append("ptr" if "*" in p else _C_KIND[" ".join(p.replace("const ", "").split()[:-1])])
        protos[m.group(1)] = kinds
    return protos


def test_align_binding_matches_the_header(monkeypatch):
    from liteasr_b200 import _lib, ops
    rec = _Recorder()
    monkeypatch.setattr(_lib, "_lib", rec)
    monkeypatch.setattr(ops, "_require_cuda", lambda *ts: None)
    monkeypatch.setattr(ops, "_stream", lambda: C.c_void_p(0))
    protos = _align_prototypes()
    assert set(protos) == {"lasr_ctc_forced_align_workspace", "lasr_ctc_forced_align"}
    i64 = lambda *s: torch.zeros(*s, dtype=torch.int64)  # noqa: E731
    ops.ctc_forced_align(torch.zeros(8, 16), torch.zeros(8), i64(2, 3), i64(2), i64(2), 4, 0, vocab=13)
    ops.ctc_forced_align(torch.zeros(8, 16, dtype=torch.bfloat16), torch.zeros(8), i64(2, 0), i64(2), i64(2), 4, 0)
    seen = set()
    for name, kinds in rec.calls:
        assert name in protos, f"{name} is called but not declared in include/lasr_align.h"
        assert kinds == protos[name], f"{name}: passed {kinds}, declared {protos[name]}"
        seen.add(name)
    assert seen == set(protos)


def test_align_symbols_are_exported():
    from liteasr_b200 import _lib, build
    build.build()
    lib = C.CDLL(_lib.LIB_PATH)
    names = _lib.declared_symbols(_lib.ALIGN_HEADER_PATH)
    assert names == ["lasr_ctc_forced_align", "lasr_ctc_forced_align_workspace"]
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/lasr_align.h but not exported"
    # size query: B * Tmax * NT * 8 bytes, 0 outside the limits
    q = lib.lasr_ctc_forced_align_workspace
    q.restype = C.c_size_t
    assert q(2, 10, 40) == 2 * 10 * 32 * 8
    assert q(1, 16384, 16383) == 16384 * 1024 * 8
    assert q(1, 16385, 10) == 0 and q(1, 10, 16384) == 0 and q(0, 10, 10) == 0


def _all_cases(rng, n):
    """Tiny (T, C, y) cases over C <= 4 classes (blank 0): random, repeated labels, exactly the minimum length and one below."""
    for _ in range(n):
        C_ = int(rng.integers(2, 5))
        L = int(rng.integers(0, 4))
        y = [int(v) for v in rng.integers(1, C_, size=L)]
        if rng.random() < 0.3 and L >= 2:
            y = [y[0]] * L
        lo = min_frames(y)
        T = int(rng.choice([max(lo - 1, 0), lo, lo + 1, lo + 2]))
        T = min(max(T, 1), 6)
        yield T, C_, y


def test_numpy_viterbi_equals_brute_force():
    rng = np.random.default_rng(5)
    n_inf = n_fin = 0
    for T, C_, y in _all_cases(rng, 150):
        lp = rng.normal(size=(T, C_)) * 2.0
        lp -= np.log(np.exp(lp).sum(1, keepdims=True))
        e = emissions(lp, np.zeros(T), y, 0, dtype=np.float64)
        state, logp, score, spans = viterbi(e, y, dtype=np.float64)
        ref = brute_force_best(lp, y, 0)
        if ref == -np.inf:
            assert score == -np.inf and (state == -1).all() and (spans == -1).all() and (logp == -np.inf).all()
            assert T < min_frames(y)
            n_inf += 1
            continue
        n_fin += 1
        assert T >= min_frames(y)
        assert abs(score - ref) <= 1e-12 * max(1.0, abs(ref)), (T, y, score, ref)
        # the path is a valid CTC path for y and its frame log-probs sum to the score
        z = np.full(2 * len(y) + 1, 0)
        z[1::2] = y
        cls = z[state]
        assert collapse(cls, 0) == list(y)
        assert abs(logp.sum() - score) <= 1e-12 * max(1.0, abs(ref))
        for k in range(len(y)):
            run = np.nonzero(state == 2 * k + 1)[0]
            assert (spans[k] == (run[0], run[-1])).all() and len(run) == run[-1] - run[0] + 1
    assert n_inf >= 10 and n_fin >= 100


def test_numpy_viterbi_tie_rules():
    # all-equal emissions: the trailing blank wins the end, and stay beats s-1 beats s-2, so walking back from the end the
    # path stays on each state while that state was reachable: the labels come as early as possible, then blanks
    y = [1, 2]
    e = np.zeros((6, 5), np.float32)
    state, _, score, spans = viterbi(e, y)
    assert score == 0.0
    assert list(state) == [1, 3, 4, 4, 4, 4]
    assert spans.tolist() == [[0, 0], [1, 1]]
    # a repeated label cannot skip the blank between its copies
    state, _, _, _ = viterbi(np.zeros((4, 5), np.float32), [1, 1])
    assert list(state) == [1, 2, 3, 4]
    # L = 0: the all-blank path
    state, _, score, spans = viterbi(np.full((3, 1), -0.5, np.float32), [])
    assert list(state) == [0, 0, 0] and score == np.float32(-1.5) and spans.shape == (0, 2)


def test_span_seconds():
    from liteasr_b200.decoding import span_seconds
    assert span_seconds(0, 0) == (0.0, 0.04)
    assert span_seconds(10, 12) == pytest.approx((0.4, 0.52))
    assert span_seconds(3, 3, frame_shift=0.02) == pytest.approx((0.24, 0.32))


def test_align_bench_help():
    r = subprocess.run([sys.executable, SCRIPT, "--help"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "--n" in r.stdout and "--tmax" in r.stdout


def test_align_bench_no_gpu_exits_nonzero():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, SCRIPT, "--n", "4"], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode != 0
    assert r.stdout.strip() == ""
