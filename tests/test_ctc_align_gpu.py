"""GPU: the CTC Viterbi forced aligner (``lasr_ctc_forced_align``, include/lasr_align.h) against the numpy float32 restatement
in tests/ctc_align_ref.py bit for bit, against a float64 optimum and torchaudio, and ``decoding.align`` /
``decode_batch(timestamps=True)`` on synthetic models.

Every output buffer starts as NaN (fp32) or -7 (int32), so an element the kernel never writes fails the comparison.

Optimality bound (test_path_is_optimal_in_float64): the kernel's path re-scored in float64 may fall short of the float64 optimum
only through fp32 rounding.  A path's fp32 score is T rounded subtractions (emissions) and T - 1 rounded adds whose partial sums
stay below T * max|e| in magnitude, so it is within u * T * (T + 1) * max|e| of its exact score (u = 2^-24); the gap between
the two paths is at most twice that: 2^-23 * T * (T + 1) * max|e|.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from ctc_align_ref import emissions, min_frames, viterbi

pytestmark = pytest.mark.gpu


def _run(logits, lse, ys_list, tps, Tmax, blank=0, V=None):
    """Call the kernel with sentinel-filled outputs.  logits (B*Tmax, ld) device, lse (B*Tmax,) device fp32."""
    from liteasr_b200 import _lib, ops
    dev = logits.device
    B = len(tps)
    V = logits.shape[1] if V is None else V
    lmax = max([0] + [len(y) for y in ys_list])
    ys = np.full((B, lmax), -1, np.int64)
    for b, y in enumerate(ys_list):
        ys[b, : len(y)] = y
    ys_d = torch.from_numpy(ys).to(dev)
    yl = torch.tensor([len(y) for y in ys_list], dtype=torch.int64, device=dev)
    fr = torch.tensor(tps, dtype=torch.int64, device=dev)
    state = torch.full((B, Tmax), -7, dtype=torch.int32, device=dev)
    logp = torch.full((B, Tmax), float("nan"), dtype=torch.float32, device=dev)
    score = torch.full((B,), float("nan"), dtype=torch.float32, device=dev)
    spans = torch.full((B, lmax, 2), -7, dtype=torch.int32, device=dev)
    L = _lib.lib()
    ws = torch.empty(max(8, int(L.lasr_ctc_forced_align_workspace(B, Tmax, lmax))), dtype=torch.uint8, device=dev)
    _lib.check(L.lasr_ctc_forced_align(ops._ptr(logits), ops._i(ops.dtype_code(logits)), ops._l(logits.stride(0)), ops._ptr(lse),
                                       ops._ptr(ys_d), ops._ptr(yl), ops._ptr(fr), ops._i(B), ops._i(Tmax), ops._i(lmax), ops._i(V),
                                       ops._i(blank), ops._ptr(state), ops._ptr(logp), ops._ptr(score), ops._ptr(spans), ops._ptr(ws),
                                       C.c_size_t(ws.numel()), ops._stream()), "ctc_forced_align")
    return state.cpu().numpy(), logp.cpu().numpy(), score.cpu().numpy(), spans.cpu().numpy()


def _compare(logits, lse, ys_list, tps, Tmax, blank=0, V=None):
    """Kernel vs numpy, bit for bit; -> number of feasible utterances."""
    st, lp, sc, sp = _run(logits, lse, ys_list, tps, Tmax, blank, V)
    V = logits.shape[1] if V is None else V
    lg = logits.float().cpu().numpy()[:, :V]
    ls = lse.cpu().numpy()
    lmax = sp.shape[1]
    feasible = 0
    for b, (y, T) in enumerate(zip(ys_list, tps)):
        e = emissions(lg[b * Tmax: b * Tmax + T], ls[b * Tmax: b * Tmax + T], y, blank)
        rs, rl, rsc, rsp = viterbi(e, y)
        L = len(y)
        ctx = (b, L, T)
        assert np.array_equal(st[b, :T], rs), ctx
        assert np.array_equal(lp[b, :T].view(np.int32), rl.astype(np.float32).view(np.int32)), ctx
        assert np.float32(sc[b]).view(np.int32) == np.float32(rsc).view(np.int32), (ctx, sc[b], rsc)
        assert np.array_equal(sp[b, :L], rsp), ctx
        assert (st[b, T:] == -1).all() and np.isneginf(lp[b, T:]).all() and (sp[b, L:lmax] == -1).all(), ctx
        feasible += int(np.isfinite(rsc))
        assert bool(np.isfinite(rsc)) == (T >= min_frames(y)), ctx
    return feasible


def _logits(rows, ld, dtype, seed, scale=3.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (scale * torch.randn(rows, ld, generator=g, device="cuda")).to(dtype)


def _lse(logits, V):
    from liteasr_b200 import ops
    return ops.logsoftmax_topk(logits, 0, vocab=V, want_lse=True)[2]


def _labels(rng, L, V, repeats=True):
    y = rng.integers(1, V, size=L)
    if not repeats:
        for i in range(1, L):
            while y[i] == y[i - 1]:
                y[i] = rng.integers(1, V)
    return [int(v) for v in y]


# ---------------------------------------------------------------------------------------------------- kernel vs numpy
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_kernel_equals_numpy_short(dtype):
    """L in {0, 1, 2, 15, 16, 31, 32, 33}, each at its minimum length, one frame below it and with slack; a transcript of one
    repeated token; a small vocabulary (V = 12, many adjacent repeats) and a padded row (ld = 16 > V)."""
    rng = np.random.default_rng(1)
    V, ld = 12, 16
    ys_list, tps = [], []
    for L in (0, 1, 2, 15, 16, 31, 32, 33):
        y = _labels(rng, L, V)
        lo = min_frames(y)
        for T in (lo - 1, lo, lo + 17):
            if T >= 1:
                ys_list.append(y)
                tps.append(T)
    for L in (5, 32):
        y = [7] * L
        for T in (2 * L - 2, 2 * L - 1, 3 * L):
            ys_list.append(y)
            tps.append(T)
    Tmax = max(tps)
    lg = _logits(len(tps) * Tmax, ld, dtype, 3)
    n = _compare(lg, _lse(lg, V), ys_list, tps, Tmax, V=V)
    assert 0 < n < len(tps)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_kernel_equals_numpy_long(dtype):
    """L in {1023, 1024, 4000} (three thread-block shapes in one batch selected from lmax = 4000), mixed with short transcripts,
    at the minimum length, one below it and with slack; V = 300 in a 304-wide buffer."""
    rng = np.random.default_rng(2)
    V, ld = 300, 304
    ys_list, tps = [], []
    for L in (1023, 1024, 4000, 3, 40):
        y = _labels(rng, L, V)
        lo = min_frames(y)
        for T in (lo - 1, lo, lo + 300):
            ys_list.append(y)
            tps.append(T)
    Tmax = max(tps)
    lg = _logits(len(tps) * Tmax, ld, dtype, 4)
    n = _compare(lg, _lse(lg, V), ys_list, tps, Tmax, V=V)
    assert n == 10


def test_kernel_equals_numpy_largest():
    """The limits: Tmax = 16 384 frames and L = 16 383 labels with no adjacent repeats (one spare frame), next to an L = 16 383
    utterance one frame short and an L = 0 one; fp32, V = 4233 as at C2."""
    rng = np.random.default_rng(3)
    V = 4233
    y = _labels(rng, 16383, V, repeats=False)
    ys_list, tps = [y, y[:-1] + [y[-2]], []], [16384, 16384, 16384]   # the second ends on a repeat: needs 16 384 frames, fits
    ys_list.append(y)
    tps.append(16382)                                                    # one short of the 16 383 it needs
    Tmax = 16384
    lg = _logits(len(tps) * Tmax, V, torch.float32, 5)
    assert _compare(lg, _lse(lg, V), ys_list, tps, Tmax, V=V) == 3


# ---------------------------------------------------------------------------------------------------- ties
def test_ties_follow_the_documented_rule():
    """Emissions that are multiples of 0.25 (exact in fp32, lse = 0) and all-equal rows: every tie the lattice meets is
    resolved as the header says (stay over s-1 over s-2; end state S-1 over S-2), which the numpy restatement encodes."""
    rng = np.random.default_rng(4)
    V = 6
    ys_list, tps, rows = [], [], []
    for i in range(40):
        y = _labels(rng, int(rng.integers(0, 9)), V)
        T = max(1, min_frames(y) + int(rng.integers(0, 6)))
        q = rng.integers(-4, 1, size=(T, 8)).astype(np.float32) * 0.25
        if i % 4 == 0:
            q[:] = -0.5
        ys_list.append(y)
        tps.append(T)
        rows.append(q)
    Tmax = max(tps)
    lg = np.zeros((len(tps) * Tmax, 8), np.float32)
    for b, q in enumerate(rows):
        lg[b * Tmax: b * Tmax + tps[b]] = q
    lg_d = torch.from_numpy(lg).cuda()
    lse = torch.zeros(len(tps) * Tmax, dtype=torch.float32, device="cuda")
    assert _compare(lg_d, lse, ys_list, tps, Tmax, V=V) == 40
    # the worked example of tests/test_ctc_align_cpu.py on the device
    st, _, sc, sp = _run(torch.zeros(6, 8, device="cuda"), torch.zeros(6, device="cuda"), [[1, 2]], [6], 6, V=V)
    assert st[0].tolist() == [1, 3, 4, 4, 4, 4] and sc[0] == 0.0 and sp[0].tolist() == [[0, 0], [1, 1]]


# ---------------------------------------------------------------------------------------------------- float64 optimum
def test_path_is_optimal_in_float64():
    rng = np.random.default_rng(6)
    V = 40
    ys_list, tps = [], []
    for L in (1, 7, 30, 200, 1000):
        y = _labels(rng, L, V)
        ys_list.append(y)
        tps.append(min_frames(y) + int(rng.integers(0, 2 * L + 5)))
    Tmax = max(tps)
    lg = _logits(len(tps) * Tmax, V, torch.float32, 7)
    lse = _lse(lg, V)
    st, _, sc, _ = _run(lg, lse, ys_list, tps, Tmax, V=V)
    lgh = lg.cpu().numpy().astype(np.float64)
    lsh = lse.cpu().numpy().astype(np.float64)
    for b, (y, T) in enumerate(zip(ys_list, tps)):
        e = emissions(lgh[b * Tmax: b * Tmax + T], lsh[b * Tmax: b * Tmax + T], y, 0, dtype=np.float64)
        _, _, opt, _ = viterbi(e, y, dtype=np.float64)
        path64 = float(e[np.arange(T), st[b, :T]].sum())
        bound = 2.0 ** -23 * T * (T + 1) * float(np.abs(e[np.isfinite(e)]).max())
        assert path64 <= opt + 1e-9 * abs(opt)
        assert opt - path64 <= bound, (b, opt, path64, bound)
        assert abs(float(sc[b]) - path64) <= bound


# ---------------------------------------------------------------------------------------------------- torchaudio
def test_path_equals_torchaudio():
    TAF = pytest.importorskip("torchaudio.functional")
    rng = np.random.default_rng(8)
    V = 30
    ys_list, tps = [], []
    for _ in range(24):
        y = _labels(rng, int(rng.integers(1, 40)), V)
        ys_list.append(y)
        tps.append(min_frames(y) + int(rng.integers(0, 80)))
    Tmax = max(tps)
    lg = _logits(len(tps) * Tmax, V, torch.float32, 9)
    lse = _lse(lg, V)
    st, _, _, _ = _run(lg, lse, ys_list, tps, Tmax, V=V)
    lp = (lg - lse[:, None]).view(len(tps), Tmax, V).cpu()
    for b, (y, T) in enumerate(zip(ys_list, tps)):
        ali, _ = TAF.forced_align(lp[b:b + 1, :T], torch.tensor(y, dtype=torch.int32)[None], blank=0)
        z = np.zeros(2 * len(y) + 1, np.int64)
        z[1::2] = y
        assert np.array_equal(z[st[b, :T]], ali[0].numpy()), b


# ---------------------------------------------------------------------------------------------------- errors (kernel)
def test_kernel_limits():
    from liteasr_b200 import ops
    lg = torch.zeros(4, 8, device="cuda")
    lse = torch.zeros(4, device="cuda")
    one = torch.ones(1, dtype=torch.int64, device="cuda")
    with pytest.raises(RuntimeError, match="16383"):
        ops.ctc_forced_align(lg, lse, torch.ones(1, 16384, dtype=torch.int64, device="cuda"), one, one, 4, 0)
    big = torch.zeros(16385, 8, device="cuda")
    with pytest.raises(RuntimeError, match="16384"):
        ops.ctc_forced_align(big, torch.zeros(16385, device="cuda"), torch.ones(1, 1, dtype=torch.int64, device="cuda"), one, one, 16385, 0)


# ---------------------------------------------------------------------------------------------------- model level
def _model(precision, dims=None, seed=7):
    import json
    import os
    from liteasr_b200.models.u2 import U2, U2Config
    from liteasr_b200.schema import U2Dims
    from liteasr_b200.utils.synthetic import synth_state_dict
    if dims is None:
        g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "u2_tiny.json")))
        dims, seed = g["dims"], g["seed"]
    model = U2(U2Config(**{**dims, "precision": precision}))
    model.load_state_dict(synth_state_dict(U2Dims(**dims), seed=seed))
    return model.cuda().eval()


def _padded(utts, feat=80, seed=0):
    T = max(u.shape[0] for u in utts)
    g = torch.Generator().manual_seed(seed)
    xs = torch.randn(len(utts), T, feat, generator=g)   # padding frames hold noise, not zeros
    for i, u in enumerate(utts):
        xs[i, : u.shape[0]] = u
    return xs.cuda()


def _targets(lists):
    ys = torch.full((len(lists), max([1] + [len(y) for y in lists])), -1, dtype=torch.int64)
    for b, y in enumerate(lists):
        ys[b, : len(y)] = torch.tensor(y, dtype=torch.int64)
    return ys, torch.tensor([len(y) for y in lists])


# frame counts 4 T' + 3: T' in {1, 9, 40, 75, 300}; the last batch adds T' = 1100 (> 1024: the wide attention softmax)
FRAMES = [7, 39, 163, 303, 1203]


@pytest.mark.parametrize("precision,frames", [("fp32", FRAMES), ("bf16", FRAMES), ("fp32", FRAMES[:2] + [4 * 1100 + 3])])
def test_align_batch_equals_batch1(precision, frames):
    from liteasr_b200 import decoding
    model = _model(precision)
    gen = torch.Generator().manual_seed(len(frames))
    rng = np.random.default_rng(11)
    utts = [torch.randn(n, 80, generator=gen) for n in frames]
    tps = [int(model.get_pred_len(n)) for n in frames]
    lists = [_labels(rng, max(0, min(tp // 3, 60) - (b % 2)), model.vocab_size) for b, tp in enumerate(tps)]
    lists = [[t if t != model.blank else 1 for t in y] for y in lists]
    lists.append(_labels(rng, tps[1] + 3, model.vocab_size, repeats=False))   # does not fit: -inf, empty path
    utts.append(utts[1])
    xs = _padded(utts)
    ys, yl = _targets(lists)
    out = decoding.align(model, xs, torch.tensor([u.shape[0] for u in utts]), ys, yl)
    assert out[-1] == dict(score=-np.inf, path=[], tokens=[])
    for b, (u, y) in enumerate(zip(utts, lists)):
        ys1, yl1 = _targets([y])
        one = decoding.align(model, u.unsqueeze(0).cuda(), torch.tensor([u.shape[0]]), ys1, yl1)[0]
        assert out[b] == one, b
        if b < len(utts) - 1:
            T = int(model.get_pred_len(u.shape[0]))
            assert np.isfinite(one["score"]) and len(one["path"]) == T and [t for t, *_ in one["tokens"]] == y
            for tok, f0, f1, s0, s1 in one["tokens"]:
                assert one["path"][f0:f1 + 1] == [tok] * (f1 - f0 + 1)
                assert (s0, s1) == decoding.span_seconds(f0, f1)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_aligning_greedy_tokens_gives_the_greedy_path(precision):
    from liteasr_b200 import decoding, ops
    model = _model(precision)
    gen = torch.Generator().manual_seed(5)
    frames = [303, 163, 4 * 1100 + 3, 39]
    utts = [torch.randn(n, 80, generator=gen) for n in frames]
    xs = _padded(utts, seed=1)
    xlens = torch.tensor(frames)
    dec = decoding.decode_batch(model, xs, xlens)
    ys, yl = _targets([d["greedy"] for d in dec])
    al = decoding.align(model, xs, xlens, ys, yl)
    _, logits, tps, _, Tp = decoding._ragged_encode(model, xs, xlens)
    tv, ti, lse, _ = ops.logsoftmax_topk(logits, 2, vocab=model.vocab_size, want_lse=True)
    tv, ti = tv.view(len(frames), Tp, 2).cpu().numpy(), ti.view(len(frames), Tp, 2).cpu().numpy()
    lse = lse.view(len(frames), Tp).cpu().numpy()
    n_exact = 0
    for b, T in enumerate(tps):
        # the top-K values round (x - max) - log(sum), the aligner x - lse: both within 2^-24 (|x| + |lse|) of the exact value
        top1 = tv[b, :T, 0].astype(np.float64)
        tol = 2.0 ** -23 * T * (T + 1) * float(np.abs(top1).max()) + 2.0 ** -22 * T * (float(np.abs(lse[b, :T]).max()) + 1.0)
        assert abs(al[b]["score"] - top1.sum()) <= tol, (b, al[b]["score"], top1.sum(), tol)
        if (tv[b, :T, 0] - tv[b, :T, 1] > 1e-4).all():
            assert al[b]["path"] == [int(v) for v in ti[b, :T, 0]]
            n_exact += 1
    assert n_exact >= 1


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_decode_batch_timestamps(precision):
    from liteasr_b200 import decoding
    model = _model(precision)
    gen = torch.Generator().manual_seed(9)
    frames = [163, 7, 303, 67]
    utts = [torch.randn(n, 80, generator=gen) for n in frames]
    xs = _padded(utts, seed=2)
    xlens = torch.tensor(frames)
    plain = decoding.decode_batch(model, xs, xlens)
    with_ts = decoding.decode_batch(model, xs, xlens, timestamps=True)
    assert all(set(p) == {"best", "hyps", "scores", "greedy"} for p in plain)
    ys, yl = _targets([p["best"] for p in plain])
    al = decoding.align(model, xs, xlens, ys, yl)
    for p, w, a in zip(plain, with_ts, al):
        assert {k: v for k, v in w.items() if k != "timestamps"} == p
        assert w["timestamps"] == a["tokens"]
        assert [t for t, *_ in w["timestamps"]] == p["best"]


def test_align_errors():
    from liteasr_b200 import decoding
    model = _model("fp32")
    xs = torch.randn(2, 40, 80, device="cuda")
    xl = torch.tensor([40, 30])
    ys, yl = _targets([[1, 2], [3]])
    with pytest.raises(ValueError):
        decoding.align(model, xs, torch.tensor([40, 6]), ys, yl)                    # shorter than 7 frames
    for bad in (model.blank, -1, model.vocab_size):
        y2 = ys.clone()
        y2[0, 1] = bad
        with pytest.raises(ValueError):
            decoding.align(model, xs, xl, y2, yl)                                    # blank / negative / >= V token
    with pytest.raises(ValueError):
        decoding.align(model, xs, xl, ys, torch.tensor([3, 1]))                      # ylens > Lmax
    long = torch.ones(2, 16384, dtype=torch.int64)
    with pytest.raises(ValueError):
        decoding.align(model, xs, xl, long, torch.tensor([16384, 1]))                # L > 16383
    model.train()
    with pytest.raises(RuntimeError):
        decoding.align(model, xs, xl, ys, yl)
