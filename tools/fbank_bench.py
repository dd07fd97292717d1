"""Filterbank benchmark: the device log-mel front end (``lasr_fbank``) against torchaudio, and what it adds to decoding.

    python tools/fbank_bench.py [--n 256] [--seconds 12] [--long-frames 65542] [--iters 20] [--seed 7] [--no-torchaudio]

Workloads (16 kHz int16, 80 bins, 25 / 10 ms; seeded noise with a sine, a chirp and a clipped square wave mixed in):
  batch   N utterances of --seconds each (the C2 shape: 256 x 12 s)
  long    one utterance of --long-frames frames (65 542 frames = 10.9 min, the encoder's limit)
Arms, each warmed up before it is timed:
  kernel       ``ops.fbank`` (one launch), median of CUDA-event timings; audio-s/s, and bytes/s (int16 samples in, fp32
               features out) against the 7.7 TB/s HBM bound.  The long workload's 42 MB fit the 126 MB L2, so its repeated
               launches read from L2.
  transcribe   ``decoding.transcribe`` against ``decode_batch`` on the precomputed features (C2 model, bf16, synthetic
               weights): the difference is what the front end adds per call
  torchaudio   ``torchaudio.compliance.kaldi.fbank`` one utterance at a time on CUDA fp32 tensors (median of 3 passes) and on
               the host CPU (one pass); skipped (and said so) when torchaudio is not importable or with --no-torchaudio
Every kernel output is checked against torchaudio in float64 on the same samples (FLT_EPSILON floor): the largest |dE| over
the frame's total energy, the largest |d log| on strong bins (E >= 1e-3 x the frame's largest) and on all bins.
Prints one JSON line.  Needs a GPU: without one it exits non-zero.
"""
from __future__ import annotations

import argparse
import dataclasses
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

C2_DIMS = (80, 4233, 256, 2048, 4, 12, 256, 2048, 4, 6)
HBM_BYTES_PER_S = 7.7e12   # one B200, NVIDIA data sheet


def _gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()
        name, power = out[0].split(",")
        return name.strip(), power.strip()
    except Exception as e:  # the query is informative only
        return f"unknown ({e})", "unknown"


def _signal(rng, n, sr):
    """n int16 samples: noise, then a 1 kHz sine, a 100 Hz - 7.1 kHz chirp and a clipped square wave, a quarter each."""
    import numpy as np
    q = n // 4
    t = np.arange(n) / sr
    x = rng.normal(0.0, 6000.0, size=n)
    x[q: 2 * q] = 12000.0 * np.sin(2 * np.pi * 1000.0 * t[q: 2 * q])
    tc = t[2 * q: 3 * q] - t[2 * q]
    dur = max(tc[-1], 1e-9) if tc.size else 1.0
    x[2 * q: 3 * q] = 12000.0 * np.sin(2 * np.pi * (100.0 * tc + 0.5 * (7000.0 / dur) * tc * tc))
    x[3 * q:] = np.clip(40000.0 * np.sign(np.sin(2 * np.pi * 220.0 * t[3 * q:])), -32768, 32767)
    return np.clip(np.round(x), -32768, 32767).astype(np.int16)


def _errors(out, x_list, cfg):
    """Kernel output (B, Fmax, nb) against float64 torchaudio per utterance -> error summary dict."""
    import numpy as np
    import torch
    import torchaudio.compliance.kaldi as K
    eps = float(np.finfo(np.float32).eps)
    o = out.cpu().numpy().astype(np.float64)
    rel = dlog_strong = dlog_all = 0.0
    pad_ok = True
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        for b, x in enumerate(x_list):
            E = K.fbank(torch.from_numpy(x.astype(np.float64))[None], use_log_fbank=False, **dataclasses.asdict(cfg)).numpy()
            F = E.shape[0]
            pad_ok &= bool((o[b, F:] == 0).all())
            ob = o[b, :F]
            ref = np.log(np.maximum(E, eps))
            rel = max(rel, float((np.abs(np.exp(ob) - np.maximum(E, eps)) / E.sum(1, keepdims=True)).max()))
            strong = E >= 1e-3 * E.max(1, keepdims=True)
            dlog_strong = max(dlog_strong, float(np.abs(ob - ref)[strong].max()))
            dlog_all = max(dlog_all, float(np.abs(ob - ref).max()))
    finally:
        torch.set_default_dtype(old)
    return dict(max_dE_over_frame_total=rel, max_dlog_strong=dlog_strong, max_dlog_all=dlog_all, padding_rows_zero=pad_ok)


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--n", type=int, default=256, help="utterances of the batch workload")
    ap.add_argument("--seconds", type=float, default=12.0, help="length of each batch utterance")
    ap.add_argument("--long-frames", type=int, default=65542, help="frames of the long utterance")
    ap.add_argument("--iters", type=int, default=20, help="timed launches per kernel arm (median reported)")
    ap.add_argument("--seed", type=int, default=7)
    ap.add_argument("--no-torchaudio", action="store_true", help="skip the torchaudio arms")
    args = ap.parse_args(argv)

    import numpy as np
    import torch
    if not torch.cuda.is_available():
        print("fbank_bench: no CUDA device (liteasr_b200 has no CPU fallback)", file=sys.stderr)
        return 2
    from liteasr_b200 import build, decoding, features, ops
    from liteasr_b200.models.u2 import U2, U2Config
    from liteasr_b200.schema import U2Dims
    from liteasr_b200.utils.synthetic import synth_state_dict
    build.build()
    dev = torch.device("cuda")
    cfg = features.FbankConfig()
    sr, W, S, nb = int(cfg.sample_frequency), cfg.window_size, cfg.window_shift, cfg.num_mel_bins
    rng = np.random.default_rng(args.seed)
    try:
        import torchaudio.compliance.kaldi as K
        ta_note = None if not args.no_torchaudio else "skipped (--no-torchaudio)"
    except Exception as e:
        ta_note = f"skipped: torchaudio not importable ({type(e).__name__})"

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

    dims = U2Dims(*C2_DIMS)
    model = U2(U2Config(**dims.__dict__, precision="bf16"))
    model.load_state_dict(synth_state_dict(dims, seed=args.seed))
    model = model.cuda().eval()

    res = {}
    n_long = W + (args.long_frames - 1) * S
    for name, lens in (("batch", [int(args.seconds * sr)] * args.n), ("long", [n_long])):
        x_list = [_signal(rng, n, sr) for n in lens]
        waves = torch.zeros((len(lens), max(lens)), dtype=torch.int16)
        for b, x in enumerate(x_list):
            waves[b, : len(x)] = torch.from_numpy(x)
        waves = waves.to(dev)
        nsamp = torch.tensor(lens, dtype=torch.int64).to(dev)
        win, lo, off, w = features._tables(cfg, dev)
        ms, out = timed(lambda: ops.fbank(waves, nsamp, W, S, win, lo, off, w), args.iters)
        audio_s = sum(lens) / sr
        frames = sum(features.num_frames(n, cfg) for n in lens)
        nbytes = 2 * sum(lens) + 4 * out.numel()
        arm = dict(utterances=len(lens), audio_s=round(audio_s, 2), frames=frames, kernel_ms=round(ms, 4),
                   audio_s_per_s=round(audio_s / ms * 1e3, 0), frames_per_s=round(frames / ms * 1e3, 0), bytes=nbytes,
                   bytes_per_s=round(nbytes / ms * 1e3, 0), hbm_bound_share=round(nbytes / ms * 1e3 / HBM_BYTES_PER_S, 4),
                   fits_l2=nbytes < 126e6, vs_float64_torchaudio=_errors(out, x_list, cfg))

        # transcribe against decode_batch on the precomputed features
        iters = 3 if name == "batch" else 1
        feats, flens = features.fbank(waves, nsamp, cfg)
        ms_dec, dec = timed(lambda: decoding.decode_batch(model, feats, flens.cpu()), iters)
        ms_tr, tr = timed(lambda: decoding.transcribe(model, waves, nsamp, cfg), iters)
        arm["decode"] = dict(decode_batch_on_features_ms=round(ms_dec, 2), transcribe_ms=round(ms_tr, 2),
                             front_end_adds_ms=round(ms_tr - ms_dec, 3), same_result=tr == dec)
        del feats, flens, dec, tr

        if ta_note is None:
            xs_dev = [torch.from_numpy(x.astype(np.float32)).to(dev)[None] for x in x_list]
            kw = dataclasses.asdict(cfg)

            def ta_cuda():
                return [K.fbank(x, **kw) for x in xs_dev]

            ta_ms = []
            ta_cuda()
            for _ in range(3):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                ta_cuda()
                torch.cuda.synchronize()
                ta_ms.append((time.perf_counter() - t0) * 1e3)
            xs_cpu = [torch.from_numpy(x.astype(np.float32))[None] for x in x_list]
            t0 = time.perf_counter()
            for x in xs_cpu:
                K.fbank(x, **kw)
            cpu_ms = (time.perf_counter() - t0) * 1e3
            tcu = float(np.median(ta_ms))
            arm["torchaudio_cuda_per_utterance"] = dict(ms=round(tcu, 2), over_kernel=round(tcu / ms, 1))
            arm["torchaudio_cpu_per_utterance"] = dict(ms=round(cpu_ms, 1), over_kernel=round(cpu_ms / ms, 1),
                                                       threads=torch.get_num_threads())
            del xs_dev
        res[name] = arm
        del waves, out
        torch.cuda.empty_cache()

    gpu, power = _gpu_info()
    print(json.dumps(dict(metric="Kaldi-compatible log-mel filterbank (device kernel; transcribe vs decode_batch)", gpu=gpu,
                          power_limit=power, config=dataclasses.asdict(cfg),
                          torchaudio=ta_note or "torchaudio.compliance.kaldi.fbank fp32, one utterance at a time", **res)))
    return 0


if __name__ == "__main__":
    sys.exit(main())
