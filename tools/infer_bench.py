"""Batched inference benchmark (BASELINE config 5): CTC prefix beam search + attention rescoring of N utterances on one GPU.

    python tools/infer_bench.py [--n 256] [--tmax 1200] [--beam 10] [--precision bf16|fp32] [--blank-bias X] [--iters 3]

Model: the C2 shape (12L d256 H4 f2048 Conformer + 6L decoder, V = 4233) with ``synth_state_dict`` weights; N utterances from
``synth_batch`` (Tmax frames).  Random weights give near-uniform posteriors in which the best prefix grows every frame (the
search's worst case); ``--blank-bias X`` adds X to the blank logit's bias (ctc.ctc_lo.bias[0]), which approximates a trained
model's blank-dominated posteriors.  The fraction of frames whose argmax is blank is reported.

Arms, in one process, each warmed up before it is timed:
  batch1   ``attention_rescore`` per utterance on the first 32 utterances (the batch-1 path)
  batched  ``decode_batch`` on all N, CUDA events per stage: encoder + CTC head, top-K, device search, D2H of the n-best, rescoring
  host     the host search (``lasr_ctc_prefix_beam_search``) on the same top-K arrays as the device search
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
N_BATCH1 = 32


def _gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        name, power = out[0].split(",")
        return name.strip(), power.strip()
    except Exception as e:  # the query is informative only
        return f"unknown ({e})", "unknown"


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--n", type=int, default=256, help="utterances decoded by the batched arm")
    ap.add_argument("--tmax", type=int, default=1200, help="longest utterance in frames")
    ap.add_argument("--beam", type=int, default=10)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--blank-bias", type=float, default=0.0, help="added to ctc.ctc_lo.bias[0]")
    ap.add_argument("--iters", type=int, default=3, help="timed repetitions of the batched arm (median reported)")
    ap.add_argument("--seed", type=int, default=7)
    args = ap.parse_args(argv)

    import numpy as np
    import torch
    if not torch.cuda.is_available():
        print("infer_bench: no CUDA device (liteasr_b200 has no CPU fallback)", file=sys.stderr)
        return 2
    from liteasr_b200 import build, decoding, ops
    from liteasr_b200.models.u2 import U2, U2Config
    from liteasr_b200.schema import U2Dims
    from liteasr_b200.utils.synthetic import synth_batch, synth_state_dict
    build.build()

    dims = U2Dims(*C2_DIMS)
    model = U2(U2Config(**dims.__dict__, precision=args.precision))
    sd = synth_state_dict(dims, seed=args.seed)
    sd["ctc.ctc_lo.bias"][0] += args.blank_bias
    model.load_state_dict(sd)
    model = model.cuda().eval()
    xs, xlens, _, _ = synth_batch(args.n, args.tmax, 40, dims.vocab_size, seed=args.seed)
    xs, xlens = xs.cuda(), xlens.cuda()
    lens = [int(v) for v in xlens.cpu()]
    dev = xs.device

    def ev():
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    # stage-timed restatement of decode_batch
    def run_batched():
        st = {}
        with torch.no_grad():
            e0 = ev()
            tps = [int(model.get_pred_len(n)) for n in lens]
            sub = torch.tensor(tps, dtype=torch.int64).to(dev)
            from liteasr_b200 import functions as F
            s_, eng, _ = F.bind(model, dev)
            F.bind(model.encoder, dev)
            F.bind(model.ctc, dev)
            s_.refresh_operands(force=True)
            enc = eng.encoder_fwd(model.encoder, xs, None, False, sub_lens=sub)
            head = eng.ctc_head_fwd(model.ctc, enc.out)
            e1 = ev()
            k = min(args.beam, dims.vocab_size)
            tv, ti, _, _ = ops.logsoftmax_topk(head.out, k, vocab=dims.vocab_size)
            e2 = ev()
            Tp = enc.Tp
            toks, tl, sc, cnt = ops.ctc_prefix_beam_search_batch(tv, ti, sub, Tp, beam=args.beam, blank=model.blank)
            e3 = ev()
            toks, tl, sc, cnt, top1 = (t.cpu().numpy() for t in (toks, tl, sc, cnt, ti[:, 0].view(-1, Tp)))
            e4 = ev()
            nbest = [[(tuple(int(x) for x in toks[b, i, : tl[b, i]]), float(sc[b, i])) for i in range(cnt[b])] for b in range(len(tps))]
            res = decoding._rescore_padded(model, nbest, enc.out, tps)
            e5 = ev()
        torch.cuda.synchronize()
        st = dict(encoder_head_ms=e0.elapsed_time(e1), topk_ms=e1.elapsed_time(e2), search_ms=e2.elapsed_time(e3),
                  d2h_ms=e3.elapsed_time(e4), rescore_ms=e4.elapsed_time(e5), total_ms=e0.elapsed_time(e5))
        out = [dict(best=list(hy[bi][0]), hyps=hy) for hy, (bi, _) in zip(nbest, res)]
        return st, out, tv, ti, tps, top1

    # ---- batched arm
    run_batched()  # warm-up (module loads, graph of allocations)
    runs = [run_batched() for _ in range(args.iters)]
    stages = {k: float(np.median([r[0][k] for r in runs])) for k in runs[0][0]}
    _, out, tv, ti, tps, top1 = runs[-1]
    blank_frac = float(np.mean(np.concatenate([top1[b, : tps[b]] == model.blank for b in range(len(tps))])))
    # the public entry point gives the same result
    pub = decoding.decode_batch(model, xs, xlens, beam=args.beam)
    assert all(p["best"] == o["best"] and p["hyps"] == o["hyps"] for p, o in zip(pub, out)), "decode_batch differs from its stages"

    # ---- host search on the same top-K arrays
    Tp = tv.shape[0] // args.n
    tvh, tih = tv.view(args.n, Tp, -1).cpu().numpy(), ti.view(args.n, Tp, -1).cpu().numpy()
    ops.ctc_prefix_beam_search_host(tvh[0, : tps[0]], tih[0, : tps[0]], beam=args.beam, blank=model.blank)
    t0 = time.perf_counter()
    host = [ops.ctc_prefix_beam_search_host(tvh[b, : tps[b]], tih[b, : tps[b]], beam=args.beam, blank=model.blank) for b in range(args.n)]
    host_ms = (time.perf_counter() - t0) * 1e3
    same_prefixes = sum([p for p, _ in h] == [p for p, _ in o["hyps"]] for h, o in zip(host, out))
    max_rel = max((abs(a[1] - b[1]) / max(1e-300, abs(a[1])) for h, o in zip(host, out) for a, b in zip(h, o["hyps"])
                   if a[0] == b[0] and np.isfinite(a[1])), default=0.0)

    # ---- batch-1 arm on the first 32 utterances
    n1 = min(N_BATCH1, args.n)
    utts = [xs[b:b + 1, : lens[b]] for b in range(n1)]
    decoding.attention_rescore(model, utts[0], beam=args.beam)  # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    single = [decoding.attention_rescore(model, u, beam=args.beam, return_details=True) for u in utts]
    torch.cuda.synchronize()
    b1_ms = (time.perf_counter() - t0) * 1e3
    identical = sum(s["best"] == o["best"] and [p for p, _ in s["hyps"]] == [p for p, _ in o["hyps"]] for s, o in zip(single, out))

    name, power = _gpu_info()
    audio_s = sum(lens) * 0.01
    res = dict(
        metric="batched CTC prefix beam search + attention rescoring (C2 shape, synthetic weights)",
        gpu=name, power_limit=power, precision=args.precision, n=args.n, tmax=args.tmax, beam=args.beam, blank_bias=args.blank_bias,
        blank_frac=round(blank_frac, 4),
        batched=dict(utt_per_s=round(args.n / stages["total_ms"] * 1e3, 1), audio_s_per_s=round(audio_s / stages["total_ms"] * 1e3, 1),
                     **{k: round(v, 3) for k, v in stages.items()}),
        batch1=dict(n=n1, ms=round(b1_ms, 2), utt_per_s=round(n1 / b1_ms * 1e3, 2),
                    audio_s_per_s=round(sum(lens[:n1]) * 0.01 / b1_ms * 1e3, 2)),
        batched_over_batch1_utt_per_s=round((args.n / stages["total_ms"]) / (n1 / b1_ms), 2),
        host_search=dict(ms=round(host_ms, 2), same_prefix_lists=same_prefixes, max_rel_score_diff=max_rel),
        host_over_device_search=round(host_ms / stages["search_ms"], 1),
        batch1_identical=f"{identical}/{n1}",
    )
    print(json.dumps(res))
    return 0


if __name__ == "__main__":
    sys.exit(main())
