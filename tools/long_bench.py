"""Long-utterance benchmark: the attention softmax on rows wider than 1024 columns, and the whole model on 60-300 s of audio.

    python tools/long_bench.py [--iters 20] [--precision bf16|fp32] [--blank-bias X] [--skip-model]

Kernel arm: ``lasr_attn_softmax_fwd`` / ``_bwd`` (encoder self-attention: rel-pos term, key mask mode 3, every key valid) timed
with CUDA events at T' in {1024 (warp kernel), 1032, 2048, 4096, 8192, 16384} (CTA-per-row kernels), bf16/bf16 and fp32/fp32.
B*H is chosen so that each (B,H,T',ld) tensor holds at least 512 MB, four times the 126 MB L2 and more, so every timed pass
reads from HBM (no buffer rotation).  Algorithmic bytes: forward ac + bd read, probs written; backward probs + dprobs read,
dscores + dbd written.  Reported: time per call, GB/s and the fraction of 7.7 TB/s (the HBM3e bandwidth of one B200).

Model arm: the C2 shape (12L d256 H4 f2048 Conformer + 6L decoder, V = 4233) with ``synth_state_dict`` weights.
  decode   ``decoding.decode_batch`` on 60 / 120 / 300 s utterances (random features; random weights give near-uniform
           posteriors, so hypotheses grow about one token per frame and rescoring runs the decoder on targets as long as T';
           ``--blank-bias`` shifts the blank logit towards a trained model's blank-dominated posteriors)
  train    one eager training step (``TrainStep.step_eager``: forward, backward, clip + Noam + Adam) on 60 s utterances
           with 200 labels each: audio-s/s and peak memory
Prints one JSON line with the GPU name and power limit read in the same run.  Needs a GPU: without one it exits non-zero.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

C2_DIMS = (80, 4233, 256, 2048, 4, 12, 256, 2048, 4, 6)
HBM_BPS = 7.7e12
KERNEL_T = (1024, 1032, 2048, 4096, 8192, 16384)
DECODE = ((60, 8), (120, 4), (300, 2))   # (seconds per utterance, utterances)
TRAIN = (60, 8)


def _gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        name, power = out[0].split(",")
        return name.strip(), power.strip()
    except Exception as e:  # the query is informative only
        return f"unknown ({e})", "unknown"


def softmax_bytes(rows: int, ld: int, e_s: int, e_p: int):
    """Algorithmic bytes of one forward and one backward call (rel-pos attention)."""
    return rows * ld * (2 * e_s + e_p), rows * ld * (e_p + e_s + 2 * e_p)


def kernel_arm(torch, ops, iters: int):
    out = []
    for sdt, pdt, tag in ((torch.bfloat16, torch.bfloat16, "bf16/bf16"), (torch.float32, torch.float32, "fp32/fp32")):
        e_s, e_p = torch.finfo(sdt).bits // 8, torch.finfo(pdt).bits // 8
        for T in KERNEL_T:
            ld = (T + 7) // 8 * 8
            BH = max(1, -(-(512 << 20) // (T * ld * min(e_s, e_p))))
            B, H = BH, 1
            g = torch.Generator(device="cuda").manual_seed(T)
            ac = (torch.randn(B, H, T, ld, generator=g, device="cuda") * 3).to(sdt)
            bd = (torch.randn(B, H, T, ld, generator=g, device="cuda") * 3).to(sdt)
            dp = torch.randn(B, H, T, ld, generator=g, device="cuda").to(sdt)
            probs, dsc, dbd = (torch.empty(B, H, T, ld, device="cuda", dtype=pdt) for _ in range(3))
            lens = torch.full((B,), 4 * T, dtype=torch.int64, device="cuda")

            def fwd():
                ops.attn_softmax_fwd(ac, bd, probs, lens, 3, 0, 0.125, T)

            def bwd():
                ops.attn_softmax_bwd(probs, dp, dsc, dbd, 0.125, T)
            res = dict(dtypes=tag, T=T, ld=ld, B=B, H=H, kernel="warp" if ld <= 1024 else "cta")
            for name, fn, nbytes in zip(("fwd", "bwd"), (fwd, bwd), softmax_bytes(B * H * T, ld, e_s, e_p)):
                for _ in range(3):
                    fn()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(iters):
                    fn()
                e1.record()
                torch.cuda.synchronize()
                s = e0.elapsed_time(e1) / 1e3 / iters
                res[name] = dict(us=round(s * 1e6, 1), bytes=nbytes, gbps=round(nbytes / s / 1e9, 1), frac_hbm=round(nbytes / s / HBM_BPS, 3))
            out.append(res)
            del ac, bd, dp, probs, dsc, dbd
            torch.cuda.empty_cache()
    return out


def model_arm(torch, args):
    import numpy as np
    from liteasr_b200 import decoding
    from liteasr_b200.criterions.hybrid_ctc_attn import HybridCTCLoss, HybridCTCLossConfig
    from liteasr_b200.models.u2 import U2, U2Config
    from liteasr_b200.schema import U2Dims
    from liteasr_b200.trainer import TrainStep
    from liteasr_b200.utils.synthetic import synth_state_dict
    dims = U2Dims(*C2_DIMS)
    sd = synth_state_dict(dims, seed=args.seed)
    g = torch.Generator().manual_seed(args.seed)

    def timed(fn, reps):
        fn()  # warm-up: module loads, allocator growth
        ts = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) / 1e3)
        return float(np.median(ts)), r

    model = U2(U2Config(**dims.__dict__, precision=args.precision))
    sdd = {k: v.clone() for k, v in sd.items()}
    sdd["ctc.ctc_lo.bias"][0] += args.blank_bias
    model.load_state_dict(sdd)
    model = model.cuda().eval()
    decode = []
    for sec, n in DECODE:
        T = int(sec * 100)
        xs = torch.randn(n, T, dims.input_dim, generator=g).cuda()
        xlens = torch.full((n,), T)
        torch.cuda.reset_peak_memory_stats()
        s, res = timed(lambda: decoding.decode_batch(model, xs, xlens), args.model_reps)
        decode.append(dict(seconds=sec, n=n, T_sub=int(model.get_pred_len(T)), s=round(s, 4), utt_per_s=round(n / s, 2),
                           audio_s_per_s=round(n * sec / s, 1), longest_hyp=max(len(p) for r in res for p, _ in r["hyps"]),
                           peak_gb=round(torch.cuda.max_memory_allocated() / 1e9, 2)))
        del xs
    del model
    torch.cuda.empty_cache()

    sec, n = TRAIN
    T = int(sec * 100)
    model = U2(U2Config(**dims.__dict__, precision=args.precision))
    model.load_state_dict(sd)
    model = model.cuda().train()
    crit = HybridCTCLoss(HybridCTCLossConfig(vocab_size=dims.vocab_size, smoothing=0.1, ctc_weight=0.3))
    step = TrainStep(model, crit, use_graph=False, device=torch.device("cuda:0"))
    xs = torch.randn(n, T, dims.input_dim, generator=g).cuda()
    xlens = torch.full((n,), T).cuda()
    ys = torch.randint(1, dims.vocab_size - 1, (n, 200), generator=g).cuda()
    ylens = torch.full((n,), 200).cuda()
    torch.cuda.reset_peak_memory_stats()
    s, loss = timed(lambda: step.step_eager(xs, xlens, ys, ylens), args.model_reps)
    train = dict(seconds=sec, n=n, T_sub=int(model.get_pred_len(T)), labels=200, s=round(s, 4), audio_s_per_s=round(n * sec / s, 1),
                 peak_gb=round(torch.cuda.max_memory_allocated() / 1e9, 2), loss_finite=bool(torch.isfinite(torch.as_tensor(float(loss)))))
    return dict(decode=decode, train=train)


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--iters", type=int, default=20, help="timed calls per kernel point")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"], help="model arm precision")
    ap.add_argument("--blank-bias", type=float, default=0.0, help="added to ctc.ctc_lo.bias[0] in the decode arm")
    ap.add_argument("--model-reps", type=int, default=3, help="timed repetitions per model point (median reported)")
    ap.add_argument("--skip-model", action="store_true", help="run the kernel arm only")
    ap.add_argument("--seed", type=int, default=7)
    args = ap.parse_args(argv)

    import torch
    if not torch.cuda.is_available():
        print("long_bench: no CUDA device (liteasr_b200 has no CPU fallback)", file=sys.stderr)
        return 2
    from liteasr_b200 import build, ops
    build.build()
    name, power = _gpu_info()
    res = dict(metric="attention softmax past 1024 columns + long-utterance decode / train (C2 shape, synthetic weights)",
               gpu=name, power_limit=power, precision=args.precision, blank_bias=args.blank_bias, l2_note="tensors >= 512 MB each, no rotation",
               kernels=kernel_arm(torch, ops, args.iters))
    if not args.skip_model:
        res["model"] = model_arm(torch, args)
    print(json.dumps(res))
    return 0


if __name__ == "__main__":
    sys.exit(main())
