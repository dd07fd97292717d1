"""CTC forced-alignment benchmark: the device Viterbi aligner (``lasr_ctc_forced_align``) and ``decode_batch(timestamps=True)``.

    python tools/align_bench.py [--n 256] [--tmax 1200] [--iters 20] [--seed 7] [--no-torchaudio]

Arms, in one process, each warmed up before it is timed (CUDA events around the launches):
  kernel_c2     the aligner on seeded emissions shaped like a C2 batch: N utterances of T' <= T'(tmax) encoder frames (tmax input
                frames, 4x sub-sampling), V = 4233, transcripts of 30-60 tokens; fp32 and bf16 logits
  kernel_long   one utterance of T' = 16 384 frames (10.9 min of audio) with L = 4000 and L = 16 383 tokens (no adjacent
                repeats: 16 383 tokens need 16 383 frames plus one per repeat), fp32 logits
  decode        ``decode_batch`` on N C2-shape utterances (bf16, synthetic weights) without and with ``timestamps=True``, and the
                timestamps stage alone (the aligner on the best hypotheses over the same CTC logits, with the host-side assembly)
  torchaudio    ``torchaudio.functional.forced_align`` on the CPU over the same emissions (log-probs formed from the same logits
                and lse), one utterance at a time, for scale; skipped (and said so) when torchaudio is not importable
Prints one JSON line.  Needs a GPU: without one it exits non-zero.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

C2_DIMS = (80, 4233, 256, 2048, 4, 12, 256, 2048, 4, 6)


def _gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        name, power = out[0].split(",")
        return name.strip(), power.strip()
    except Exception as e:  # the query is informative only
        return f"unknown ({e})", "unknown"


def _no_repeats(rng, n, V):
    """n tokens in [1, V) with no two adjacent equal."""
    y = rng.integers(1, V, size=n)
    for i in range(1, n):
        while y[i] == y[i - 1]:
            y[i] = rng.integers(1, V)
    return y


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--n", type=int, default=256, help="utterances of the C2-shape arms")
    ap.add_argument("--tmax", type=int, default=1200, help="longest C2 utterance in input frames")
    ap.add_argument("--iters", type=int, default=20, help="timed launches per kernel arm (median reported)")
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--no-torchaudio", action="store_true", help="skip the CPU torchaudio arm")
    args = ap.parse_args(argv)

    import numpy as np
    import torch
    if not torch.cuda.is_available():
        print("align_bench: no CUDA device (liteasr_b200 has no CPU fallback)", file=sys.stderr)
        return 2
    from liteasr_b200 import build, decoding, ops
    from liteasr_b200.models.u2 import U2, U2Config
    from liteasr_b200.schema import U2Dims
    from liteasr_b200.utils.synthetic import synth_batch, synth_state_dict
    build.build()
    dev = torch.device("cuda")
    V = C2_DIMS[1]
    rng = np.random.default_rng(args.seed)
    gen = torch.Generator(device="cuda").manual_seed(args.seed)

    def timed(fn, iters):
        fn()
        torch.cuda.synchronize()
        ms = []
        for _ in range(iters):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn()
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        return float(np.median(ms)), out

    def problem(tps, ys_list, dtype):
        B, Tp = len(tps), max(tps)
        logits = (3.0 * torch.randn(B * Tp, V, generator=gen, device=dev)).to(dtype)
        _, _, lse, _ = ops.logsoftmax_topk(logits, 0, vocab=V, want_lse=True)
        lmax = max(len(y) for y in ys_list)
        ys = np.full((B, lmax), -1, np.int64)
        for b, y in enumerate(ys_list):
            ys[b, : len(y)] = y
        return (logits, lse, torch.from_numpy(ys).to(dev), torch.tensor([len(y) for y in ys_list], dtype=torch.int64).to(dev),
                torch.tensor(tps, dtype=torch.int64).to(dev), Tp)

    def run_torchaudio(p, tps, ys_list, kernel_state):
        """CPU forced_align per utterance on the same log-probs; -> (ms, utterances whose per-frame token path equals the kernel's)."""
        import torchaudio.functional as TAF
        logits, lse, _, _, _, Tp = p
        lp = (logits.float() - lse[:, None]).view(len(tps), Tp, V).cpu()
        st = kernel_state.cpu().numpy()
        t0 = time.perf_counter()
        paths = []
        for b, (T, y) in enumerate(zip(tps, ys_list)):
            ali, _ = TAF.forced_align(lp[b:b + 1, :T], torch.tensor(np.asarray(y), dtype=torch.int32)[None], blank=0)
            paths.append(ali[0].numpy())
        ms = (time.perf_counter() - t0) * 1e3
        same = frames_same = 0
        for b, (T, y) in enumerate(zip(tps, ys_list)):
            s = st[b, :T].astype(np.int64)
            path = np.where(s & 1, np.asarray(y, np.int64)[np.minimum(s >> 1, len(y) - 1)], 0)
            same += int((path == paths[b]).all())
            frames_same += int((path == paths[b]).sum())
        return ms, same, frames_same / sum(tps)

    try:
        import torchaudio  # noqa: F401
        ta_note = None if not args.no_torchaudio else "skipped (--no-torchaudio)"
    except Exception as e:
        ta_note = f"skipped: torchaudio not importable ({type(e).__name__})"

    res = {}
    # ---- kernel, C2 batch
    tp_max = ((args.tmax - 1) // 2 - 1) // 2
    tps = [int(v) for v in rng.integers(tp_max // 2, tp_max + 1, size=args.n)]
    tps[0] = tp_max
    ys_c2 = [_no_repeats(rng, int(rng.integers(30, 61)), V) for _ in tps]
    for dt, name in ((torch.float32, "fp32"), (torch.bfloat16, "bf16")):
        p = problem(tps, ys_c2, dt)
        ms, out = timed(lambda: ops.ctc_forced_align(p[0], p[1], p[2], p[3], p[4], p[5], 0, vocab=V), args.iters)
        assert bool(torch.isfinite(out[2]).all()), "a C2 transcript came out infeasible"
        arm = dict(utterances=args.n, tp_max=tp_max, frames=sum(tps), labels=sum(len(y) for y in ys_c2), kernel_ms=round(ms, 4),
                   frames_per_s=round(sum(tps) / ms * 1e3, 1))
        if name == "fp32" and ta_note is None:
            ta_ms, same, fr = run_torchaudio(p, tps, ys_c2, out[0])
            arm["torchaudio_cpu"] = dict(ms=round(ta_ms, 2), same_path=f"{same}/{args.n}", same_frames=round(fr, 6),
                                         over_kernel=round(ta_ms / ms, 1))
        res[f"kernel_c2_{name}"] = arm
        del p

    # ---- kernel, long form
    for L in (4000, 16383):
        y = _no_repeats(rng, L, V)
        p = problem([16384], [y], torch.float32)
        ms, out = timed(lambda: ops.ctc_forced_align(p[0], p[1], p[2], p[3], p[4], p[5], 0, vocab=V), max(3, args.iters // 4))
        assert bool(torch.isfinite(out[2]).all())
        arm = dict(frames=16384, labels=L, states=2 * L + 1, kernel_ms=round(ms, 3),
                   ns_per_frame=round(ms * 1e6 / 16384, 1), workspace_mb=round(ops._lib.lib().lasr_ctc_forced_align_workspace(1, 16384, L) / 2**20, 1))
        if ta_note is None:
            ta_ms, same, fr = run_torchaudio(p, [16384], [y], out[0])
            arm["torchaudio_cpu"] = dict(ms=round(ta_ms, 1), same_path=f"{same}/1", same_frames=round(fr, 6), over_kernel=round(ta_ms / ms, 1))
        res[f"kernel_long_L{L}"] = arm
        del p, out
        torch.cuda.empty_cache()

    # ---- decode_batch without / with timestamps
    dims = U2Dims(*C2_DIMS)
    model = U2(U2Config(**dims.__dict__, precision="bf16"))
    model.load_state_dict(synth_state_dict(dims, seed=args.seed))
    model = model.cuda().eval()
    xs, xlens, _, _ = synth_batch(args.n, args.tmax, 40, V, seed=args.seed)
    xs = xs.cuda()
    iters = 3
    ms_plain, plain = timed(lambda: decoding.decode_batch(model, xs, xlens), iters)
    ms_ts, with_ts = timed(lambda: decoding.decode_batch(model, xs, xlens, timestamps=True), iters)
    same = all({k: v for k, v in w.items() if k != "timestamps"} == p_ for w, p_ in zip(with_ts, plain))
    # the timestamps stage alone: the aligner on the best hypotheses over the same CTC logits, with the host-side assembly
    best = [o["best"] for o in plain]
    ys = np.full((args.n, max(len(b) for b in best)), -1, np.int64)
    for b, hy in enumerate(best):
        ys[b, : len(hy)] = hy
    with torch.no_grad():
        _, logits, tp_list, sub, Tp = decoding._ragged_encode(model, xs, xlens)
        _, _, lse, _ = ops.logsoftmax_topk(logits, 0, vocab=V, want_lse=True)
        ms_stage, al = timed(lambda: decoding._align_rows(model, logits, lse, ys, [len(b) for b in best], sub, tp_list, Tp, 0.01), iters)
        ms_kernel, _ = timed(lambda: ops.ctc_forced_align(logits, lse, torch.from_numpy(ys).to(dev),
                                                          torch.tensor([len(b) for b in best], dtype=torch.int64).to(dev), sub, Tp, 0,
                                                          vocab=V), args.iters)
    same = same and all(a["tokens"] == w["timestamps"] for a, w in zip(al, with_ts))
    res["decode_batch_bf16"] = dict(utterances=args.n, tmax=args.tmax, ms=round(ms_plain, 2), timestamps_ms=round(ms_ts, 2),
                                    timestamps_overhead_ms=round(ms_ts - ms_plain, 2), align_stage_ms=round(ms_stage, 3),
                                    align_kernel_ms=round(ms_kernel, 4), lmax=int(ys.shape[1]), consistent=bool(same),
                                    mean_best_tokens=round(float(np.mean([len(o["best"]) for o in plain])), 1))

    name, power = _gpu_info()
    print(json.dumps(dict(metric="CTC Viterbi forced alignment (device kernel; decode_batch timestamps)", gpu=name, power_limit=power,
                          torchaudio=ta_note or "CPU forced_align on the same log-probs, one utterance at a time", **res)))
    return 0


if __name__ == "__main__":
    sys.exit(main())
