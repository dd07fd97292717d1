"""numpy restatement of the CTC Viterbi forced alignment of include/lasr_align.h, shared by tests/test_ctc_align_cpu.py (which
checks it against brute-force enumeration) and tests/test_ctc_align_gpu.py (which checks the kernel against it bit for bit).

With dtype float32 every step is the kernel's: one fp32 subtraction per emission, an exact max, one fp32 add per state.
"""
import itertools

import numpy as np


def emissions(logits, lse, y, blank, dtype=np.float32):
    """e (T, S): logits (T, >=V) and lse (T,) of one utterance, y (L,) labels -> e[t, s] = logits[t, z[s]] - lse[t]."""
    z = np.full(2 * len(y) + 1, blank, dtype=np.int64)
    z[1::2] = y
    lg = np.asarray(logits, dtype=dtype)
    return lg[:, z] - np.asarray(lse, dtype=dtype)[:, None]


def viterbi(e, y, dtype=np.float32):
    """e (T, S) emissions, y (L,) labels -> (state (T,) int32, frame_logp (T,), score, spans (L, 2) int32) with the header's
    rules: predecessors s, s-1 and s-2 (odd s >= 3 with y[k] != y[k-1]), ties to the higher predecessor index, end state S-1 over
    S-2 on a tie.  An optimum of -inf gives state / spans -1, frame_logp -inf and score -inf."""
    e = np.asarray(e, dtype=dtype)
    T, S = e.shape
    L = len(y)
    assert S == 2 * L + 1
    ninf = dtype(-np.inf)
    state = np.full(T, -1, np.int32)
    logp = np.full(T, ninf, dtype)
    spans = np.full((L, 2), -1, np.int32)
    if T == 0:
        return state, logp, ninf, spans
    skip = np.zeros(S, bool)
    if L >= 2:
        skip[3::2] = np.asarray(y[1:]) != np.asarray(y[:-1])
    delta = np.full(S, ninf, dtype)
    delta[: min(2, S)] = e[0, : min(2, S)]
    bp = np.zeros((T, S), np.int8)
    for t in range(1, T):
        c1 = np.concatenate(([ninf], delta[:-1]))
        c2 = np.concatenate(([ninf, ninf], delta[:-2]))[:S]
        c2 = np.where(skip, c2, ninf)
        best = delta.copy()
        p = np.zeros(S, np.int8)
        m = c1 > best
        best[m], p[m] = c1[m], 1
        m = c2 > best
        best[m], p[m] = c2[m], 2
        delta = (best + e[t]).astype(dtype)
        bp[t] = p
    end = S - 1
    score = delta[S - 1]
    if S >= 2 and delta[S - 2] > score:
        end, score = S - 2, delta[S - 2]
    if not score > ninf:
        return state, logp, ninf, spans
    s = end
    for t in range(T - 1, -1, -1):
        state[t] = s
        s -= int(bp[t, s])
    logp = e[np.arange(T), state.astype(np.int64)]
    for k in range(L):
        fr = np.nonzero(state == 2 * k + 1)[0]
        spans[k] = fr[0], fr[-1]
    return state, logp, dtype(score), spans


def collapse(path, blank):
    """CTC collapse of a per-frame class path: merge repeats, drop blanks."""
    out = []
    prev = None
    for c in path:
        if c != prev and c != blank:
            out.append(int(c))
        prev = c
    return out


def brute_force_best(logp, y, blank):
    """max over every class path of length T that collapses to y of sum_t logp[t, path[t]] (float64), or -inf."""
    T, C = logp.shape
    best = -np.inf
    for path in itertools.product(range(C), repeat=T):
        if collapse(path, blank) == list(y):
            best = max(best, float(sum(logp[t, c] for t, c in enumerate(path))))
    return best


def min_frames(y):
    """The fewest frames that can hold y: L plus one blank between each pair of adjacent equal labels."""
    y = list(y)
    return len(y) + sum(1 for a, b in zip(y, y[1:]) if a == b)
