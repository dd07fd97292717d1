#!/usr/bin/env python
"""Benchmark of the hot path: one U2 Conformer training step (fwd + bwd + hybrid CTC/attention loss + gradient all-reduce +
fused clip/Adam) on synthetic 80-dim fbank batches.  Metric: audio-seconds per second (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c2|c1|c3] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

One JSON line on rank 0.  `value` = whole-job audio-s/s with the batch resident in HBM (CUDA-graph replay, CUDA-event timed,
max over ranks); `e2e` = the same step through the public API with the batch in pinned HOST memory (H2D inside the timed
region, loss read back every step).  The headline trains with the reference's shipped rates (config/model/my_U2.yaml: dropout
0.1, attention-probability rates 0.0; BASELINE.md section 3: "0.1 for the throughput run"); `extra.dropout_0` is the same step
with every rate 0 (round-1's configuration).  `roofline` = the dominant kernel family (every tcgen05 contraction of the step: lasr_gemm,
the implicit-GEMM convolutions, the fused feed-forward kernels and the paired attention-backward kernel) timed live with CUDA events
(the family's launches of one step replayed from a CUDA graph), `roofline_split` = its tensor-bound (K >= 1024, convolutions) and
HBM-bound (K < 1024) halves against their own peaks, `roofline_ctc` = the standalone fused CTC over the whole BASELINE config-4
grid; `gpu_incumbent` = the reference's own modules (unmodified copy under baseline/_ref, else the oracle port) on torch-CUDA on
the same GPU, eager fp32 and autocast(bf16), same batch; `cpu_baseline` = the same reference path on the box's host cores, one
step over (at most) 126 utterances of the batch.  `--impl reference` runs only the CPU arm on a bounded sample and prints the same line shape.
"""
from __future__ import annotations

import argparse
import contextlib
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FRAME_SHIFT_S = 0.01  # Kaldi fbank default frame shift (the reference never states it; SURVEY 8d)

WORKLOADS = {
    # BASELINE.json configs[1]: AISHELL-1 shape
    "c2": dict(dims=(80, 4233, 256, 2048, 4, 12, 256, 2048, 4, 6), batch=252, tmax=1200, lmax=40, ctc_weight=0.3, smoothing=0.1,
               desc="C2: U2 Conformer 12L d256 H4 f2048 + 6L Transformer decoder, V=4233 (AISHELL-1 shape), Tmax=1200 (T'=299), "
                    "per-GPU batch 252 (builder's choice, SURVEY 8: 252 x 299 rows = 589 row tiles = four waves of the 148 SMs, 3.98 of "
                    "them full; rounds 1 and most of 2 ran two waves = `--batch 126`, 4 % slower per utterance; the reference default 32 "
                    "is `--batch 32`), Lmax=40, hybrid ctc_weight 0.3, smoothing 0.1, dropout 0 (U2Config default)"),
    # configs[0]: the reference's CPU-runnable case
    "c1": dict(dims=(80, 500, 256, 2048, 4, 4, 256, 2048, 4, 6), batch=8, tmax=500, lmax=30, ctc_weight=0.3, smoothing=0.1,
               desc="C1: U2 Conformer 4L d256 H4 + 6L decoder, V=500, batch 8, Tmax=500"),
    # configs[2]: LibriSpeech-960 shape
    "c3": dict(dims=(80, 5000, 512, 2048, 8, 12, 512, 2048, 8, 6), batch=92, tmax=1600, lmax=100, ctc_weight=0.3, smoothing=0.1,
               desc="C3: Conformer-large 12L d512 H8 + 6L decoder d512, V=5000, Tmax=1600 (T'=399), per-GPU batch 92 (92 x 399 rows = 287 "
                    "row tiles = two waves of the 148 SMs, chosen like C2's batch; round 1 and the first half of round 2 ran 16 = a third "
                    "of ONE wave: 13.2 k audio-s/s), Lmax=100"),
}


REF_COPY = os.path.join(ROOT, "baseline", "_ref")  # git-ignored copy of the unmodified reference package (travels with gpurun)


def reference_root():
    """Where the unmodified reference package can be imported from on THIS machine (None: only the oracle port is available)."""
    for cand in (REF_COPY, "/root/reference"):
        if os.path.isdir(os.path.join(cand, "liteasr", "nets")):
            return cand
    return None


def my_u2_rates(p: float) -> dict:
    """config/model/my_U2.yaml: one rate everywhere, the three attention-probability rates 0.0."""
    if p <= 0:
        return {}
    return dict(dropout_rate=p, enc_attn_dropout_rate=0.0, dec_self_attn_dropout_rate=0.0, dec_src_attn_dropout_rate=0.0)


def build_reference_step(wl, device, dropout: float, batch):
    """One training step of the reference path in stock torch ops: HybridCTCLoss(U2) forward + backward + clip_grad_norm_ + Adam
    (trainer.py:140-171).  With a copy of the reference available the UNMODIFIED modules run (kind "reference", loaded through
    oracle/ref_shims.py); otherwise the oracle's functional restatement of the same arithmetic (kind "port").
    -> (step(autocast: bool) -> loss, kind)"""
    import torch
    from liteasr_b200.schema import U2Dims
    dims = U2Dims(*wl["dims"])
    xs, xlens, ys, ylens = batch
    root = reference_root()
    if root is not None:
        os.environ["LITEASR_REFERENCE_ROOT"] = root
        from oracle import ref_shims
        ref_shims.REFERENCE_ROOT = root
        ref_shims.install()
        from liteasr.criterions.hybrid_ctc_attn import HybridCTCLoss, HybridCTCLossConfig
        from liteasr.models.u2 import U2, U2Config
        cfg = U2Config(**dims.__dict__)
        for f in ref_shims._DROPOUT_FIELDS:
            setattr(cfg, f, float(dropout))
        for k, v in my_u2_rates(dropout).items():
            setattr(cfg, k, v)
        torch.manual_seed(42)
        model = U2(cfg).to(device).train()
        crit = HybridCTCLoss(HybridCTCLossConfig(vocab_size=dims.vocab_size, smoothing=wl["smoothing"], ctc_weight=wl["ctc_weight"]))
        params = list(model.parameters())
        opt = torch.optim.Adam(params, lr=1e-4, betas=(0.9, 0.98), eps=1e-9)

        def step(autocast=False):
            opt.zero_grad(set_to_none=True)
            with torch.autocast(device_type=device.type, dtype=torch.bfloat16, enabled=autocast):
                loss = crit(model, xs, xlens, ys, ylens)
            loss.backward()
            torch.nn.utils.clip_grad_norm_(params, 5.0)
            opt.step()
            return loss
        return step, "reference"
    # oracle port (CPU: C lattice through the oracle; CUDA: torch.ctc_loss, the call of criterions/hybrid_ctc_attn.py:67-75)
    from liteasr_b200.utils.synthetic import synth_state_dict
    from oracle import u2_oracle as O
    sd = synth_state_dict(dims, seed=42)
    sd = {k: (v.to(device).requires_grad_(True) if v.is_floating_point() and "running" not in k and ".pe.pe" not in k else v.to(device))
          for k, v in sd.items()}
    cfg = O.U2Shape(**dims.__dict__)
    params = [v for v in sd.values() if getattr(v, "requires_grad", False)]
    opt = torch.optim.Adam(params, lr=1e-4, betas=(0.9, 0.98), eps=1e-9)
    rates = O.DropRates.uniform(dropout, 0.0)

    class TorchDropper:  # the reference's own dropout: torch's generator stream (nn.Dropout / F.dropout)
        r, training = rates, True

        def __call__(self, x, net, layer, kind, p, always=False):
            return torch.nn.functional.dropout(x, p, True) if p > 0 else x
    dp = TorchDropper() if dropout > 0 else None

    # on the GPU the oracle's factory calls (masks, position tables) must follow its inputs there
    on_device = contextlib.nullcontext() if device.type == "cpu" else torch.device(device)

    def step(autocast=False):
        opt.zero_grad(set_to_none=True)
        with torch.autocast(device_type=device.type, dtype=torch.bfloat16, enabled=autocast), on_device:
            if device.type == "cpu":
                loss = O.hybrid_loss(sd, cfg, xs, xlens, ys, ylens, wl["ctc_weight"], wl["smoothing"], True, {}, dp)["loss"]
            else:
                h_attn, h_ctc, _ = O.u2_forward(sd, cfg, xs, xlens, ys, ylens, True, {}, dp)
                b = ys.size(0)
                la = O.label_smoothing_kl(h_attn.float(), O.attention_targets(ys, ylens, cfg.vocab_size), wl["smoothing"]) / b
                lp = torch.log_softmax(h_ctc.float().transpose(0, 1), dim=-1)
                lc = torch.nn.functional.ctc_loss(lp, ys.clamp(min=0), O.subsampled_len(xlens), ylens, blank=0, reduction="sum") / b
                loss = wl["ctc_weight"] * lc + (1 - wl["ctc_weight"]) * la
        loss.backward()
        torch.nn.utils.clip_grad_norm_(params, 5.0)
        opt.step()
        return loss
    return step, "port"


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm=p["hbm_gbs"], tc_burst=p["bf16_tflops"], tc_sustained=p["bf16_tflops_sustained"], src="measured")
    except Exception:  # noqa: BLE001
        return dict(hbm=6650.0, tc_burst=1590.0, tc_sustained=1400.0, src="fallback")


class ClockSampler(threading.Thread):
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.max_sm = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            self.nv = None

    def run(self):
        while not self.stop_flag and self.nv is not None:
            try:
                self.sm.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.05)

    def result(self):
        s = sorted(self.sm)
        return dict(sm_mhz=(s[len(s) // 2] if s else None), sm_max_mhz=self.max_sm, reasons=sorted(self.reasons), samples=len(s))


# --------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's path, on the host cores, on a bounded sample
# --------------------------------------------------------------------------------------------------
def cpu_oracle_run(wl, steps: int, warmup: int, sample_batch: int = 2, dropout: float = 0.0):
    """The reference's path on the host cores (all threads): `sample_batch` utterances of the workload's batch (the batch's own
    seeded draw when sample_batch == wl['batch']), fwd + bwd + clip + Adam."""
    import torch
    from liteasr_b200.schema import U2Dims
    from liteasr_b200.utils.synthetic import synth_batch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    dims = U2Dims(*wl["dims"])
    batch = synth_batch(sample_batch, wl["tmax"], wl["lmax"], dims.vocab_size, seed=42)
    if reference_root() is None:
        from oracle import u2_oracle as O
        O._clib()  # compile (if needed) and load the C lattice before the timed steps
    one, kind = build_reference_step(wl, torch.device("cpu"), dropout, batch)
    for _ in range(max(0, warmup)):
        one()
    t0 = time.perf_counter()
    for _ in range(steps):
        float(one())
    dt = (time.perf_counter() - t0) / steps
    audio = float(batch[1].sum()) * FRAME_SHIFT_S
    what = "the unmodified reference modules (baseline/_ref copy through oracle/ref_shims.py)" if kind == "reference" else "the oracle port of the reference path"
    return dict(value=audio / dt, ms_per_step=dt * 1e3, cores=cores, threads=torch.get_num_threads(), kind=kind,
                sample=f"{what}: {sample_batch} of {wl['batch']} utterances of the same workload (Tmax={wl['tmax']}), dropout {dropout}, "
                       f"fwd+bwd+clip+Adam, {steps} timed step(s) after {warmup} warm-up, torch {torch.__version__} CPU fp32, {cores} threads")


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_oracle_run(wl, args.steps, max(1, min(args.warmup, 2)), sample_batch=8, dropout=args.dropout)
    line = {
        "impl": "reference", "metric": "audio-sec/sec train (Conformer fwd+bwd+CTC)", "value": r["value"], "unit": "audio-s/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": max(1, min(args.warmup, 2)), "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": wl["desc"], "parallelism": "cpu", "frame_shift_ms": 10, "dropout": args.dropout},
        "cpu_baseline": {"value": r["value"], "unit": "audio-s/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
def _record_gemms(step_fn, batch):
    """One eager step with every `ops.gemm` / implicit-GEMM convolution call recorded (operands stay alive).
    -> list of (fn, args, kwargs, flops, algorithmic bytes, K)."""
    import torch
    from liteasr_b200 import ops
    rec = []
    orig = ops.gemm
    conv_names = ("conv2_fwd", "conv2_dgrad", "conv2_wgrad")  # the implicit-GEMM convolutions run on the same kernel
    conv_orig = {n: getattr(ops, n) for n in conv_names}

    def es(t):
        return t.element_size() if t is not None else 0

    def recording(a, b, c, m, n, k, **kw):
        bt = kw.get("batch", (1, 1))
        nb = bt[0] * bt[1]

        def distinct(strides):  # how many different (b1, b2) slices of an operand exist (stride 0 = broadcast over that level)
            s1, s2 = strides
            return (bt[0] if s1 != 0 else 1) * (bt[1] if s2 != 0 else 1)

        # algorithmic bytes: every distinct operand element once -- A, B, C and the epilogue's extra tensors
        byt = m * k * es(a) * distinct(kw.get("sa", (0, 0))) + n * k * es(b) * distinct(kw.get("sb", (0, 0)))
        byt += m * max(n, kw.get("n_store", 0)) * es(c) * distinct(kw.get("sc", (0, 0)))
        for extra in ("res", "aux", "dact"):
            if kw.get(extra) is not None:
                byt += m * n * es(kw[extra])
        rec.append((orig, (a, b, c, m, n, k), kw, 2.0 * m * n * k * nb, float(byt), k))
        orig(a, b, c, m, n, k, **kw)

    def conv_recorder(name):
        fn = conv_orig[name]

        def wrapped(*args):
            B, T, F = args[-3:]
            h1p = {"conv2_fwd": args[0], "conv2_dgrad": args[2], "conv2_wgrad": args[1]}[name]
            d = h1p.shape[-1]
            _, _, _, _, T2, F2 = ops.plane_dims(T, F)
            byt = sum(t.numel() * t.element_size() for t in args if isinstance(t, torch.Tensor))
            rec.append((fn, args, {}, 2.0 * B * T2 * F2 * d * 9 * d, float(byt), 9 * d))
            fn(*args)
        return wrapped

    ffn_orig = ops.ffn_bwd

    def ffn_recorder(dy, g, w2, w1, dh, dln, **kw):  # the fused feed-forward backward: two contractions (2 x 2 m d f flops) in one kernel
        m, d = dy.shape
        f = g.shape[1]
        byt = sum(t.numel() * t.element_size() for t in (dy, g, w2, w1, dh, dln))
        rec.append((ffn_orig, (dy, g, w2, w1, dh, dln), kw, 4.0 * m * d * f, float(byt), d))
        ffn_orig(dy, g, w2, w1, dh, dln, **kw)

    pair_orig = ops.attn_bwd_pair

    def pair_recorder(x, r, l, dl, dr, B, H, Tq, Tk, dk, **kw):  # the paired attention-backward contractions: 2 x (2 B H Tq Tk dk) flops
        byt = B * H * Tq * Tk * x.element_size() + sum(t.numel() * t.element_size() for t in (l, dl))
        byt += (B if kw.get("r_batched", True) else 1) * Tk * H * dk * r.element_size() + dr.numel() * dr.element_size()
        rec.append((pair_orig, (x, r, l, dl, dr, B, H, Tq, Tk, dk), kw, 4.0 * B * H * Tq * Tk * dk, float(byt), dk))
        pair_orig(x, r, l, dl, dr, B, H, Tq, Tk, dk, **kw)

    ffwd_orig = ops.ffn_fwd

    def ffwd_recorder(ln, w1, b1, w2, b2, res, a, g, out, **kw):  # the fused feed-forward forward: two contractions (2 x 2 m d f flops)
        m, d = ln.shape
        f = w1.shape[0]
        byt = sum(t.numel() * t.element_size() for t in (ln, w1, w2, res, a, g, out))
        rec.append((ffwd_orig, (ln, w1, b1, w2, b2, res, a, g, out), kw, 4.0 * m * d * f, float(byt), d))
        ffwd_orig(ln, w1, b1, w2, b2, res, a, g, out, **kw)

    wg2_orig = ops.wgrad2

    def wg2_recorder(dy, x, gw, **kw):  # weight gradients on CTA pairs
        rows, mo = dy.shape
        no = x.shape[1]
        byt = sum(t.numel() * t.element_size() for t in (dy, x, gw))
        rec.append((wg2_orig, (dy, x, gw), kw, 2.0 * rows * mo * no, float(byt), rows))
        wg2_orig(dy, x, gw, **kw)

    ops.wgrad2 = wg2_recorder
    ops.gemm = recording
    ops.ffn_bwd = ffn_recorder
    ops.ffn_fwd = ffwd_recorder
    ops.attn_bwd_pair = pair_recorder
    for n in conv_names:
        setattr(ops, n, conv_recorder(n))
    try:
        step_fn.step_eager(*batch)
        torch.cuda.synchronize()
    finally:
        ops.gemm = orig
        ops.wgrad2 = wg2_orig
        ops.ffn_bwd = ffn_orig
        ops.ffn_fwd = ffwd_orig
        ops.attn_bwd_pair = pair_orig
        for n in conv_names:
            setattr(ops, n, conv_orig[n])
    return rec


def _replay_ms(rec, reps: int = 5) -> float:
    """CUDA-event time of one back-to-back replay of the recorded launches from a CUDA graph (no host gaps, nothing else)."""
    import torch
    if not rec:
        return 0.0

    def replay():
        for fn, args, kw, *_ in rec:
            fn(*args, **kw)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        replay()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        replay()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    del g
    return ms


def gemm_family_replay(step_fn, batch, reps: int = 5, split: bool = False):
    """The dominant kernel family (every tcgen05 GEMM of one training step) timed live and alone: one eager step records each
    `ops.gemm` call, a CUDA graph replays exactly those launches back to back on the real operands, CUDA events time `reps`
    replays: flops / time is the family's own tensor-pipe throughput.  -> (flops, ms, launches[, split dict]): with `split`
    the two halves of the family are also replayed on their own -- K >= 1024 and the convolutions (tensor-bound: judged
    against the tensor peak) and K < 1024 (at most 120 FLOP per algorithmic byte: judged against the HBM peak)."""
    rec = _record_gemms(step_fn, batch)
    flops = sum(r[3] for r in rec)
    ms = _replay_ms(rec, reps)
    if not split:
        return flops, ms, len(rec)
    hi = [r for r in rec if r[5] >= 1024]
    lo = [r for r in rec if r[5] < 1024]
    out = {}
    for name, part in (("tensor", hi), ("hbm", lo)):
        out[name] = dict(launches=len(part), flops=sum(r[3] for r in part), bytes=sum(r[4] for r in part), ms=_replay_ms(part, reps))
    return flops, ms, len(rec), out


C4_GRID = [(T, L, V) for (T, L) in ((200, 20), (400, 50), (800, 100), (1600, 200)) for V in (500, 1000, 2000, 5000)]


def ctc_standalone(pk, torch_too: bool = True):
    """BASELINE config 4, the whole grid: standalone fused CTC fwd+bwd (B = 64, fp32), algorithmic GB/s = T*B*V*(4+4) bytes / time
    (SURVEY 8d), next to the reference's torch path on the same GPU (log_softmax + ctc_loss(sum) forward + backward,
    criterions/hybrid_ctc_attn.py:67-75).  The headline fields are the largest point (2.05 GB of logits)."""
    import torch
    from liteasr_b200 import ops
    B = 64
    grid = []
    for T, L, V in C4_GRID:
        g = torch.Generator(device="cuda").manual_seed(1000 * T + V)
        x = torch.randn(T, B, V, generator=g, device="cuda")
        il = torch.randint(int(0.6 * T), T + 1, (B,), generator=g, device="cuda"); il[0] = T
        tl = torch.randint(L // 2, L + 1, (B,), generator=g, device="cuda"); tl[0] = L
        tg = torch.randint(1, V, (B, L), generator=g, device="cuda")
        tg[1, 1] = tg[1, 0]
        grad = torch.empty_like(x)
        ws = torch.empty(ops.ctc_workspace_bytes(T, B, L), dtype=torch.uint8, device="cuda")

        def timed(fn, n):
            for _ in range(3):
                fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / n

        # small points fit the 126 MB L2 (x + grad = 2 * T*B*V*4 bytes): rotate over enough copies to exceed it
        ncopy = max(1, min(8, int(2.6e8 // (2 * x.numel() * 4)) + 1))
        xs_ = [x] + [x.clone() for _ in range(ncopy - 1)]
        gs_ = [grad] + [torch.empty_like(x) for _ in range(ncopy - 1)]
        it = {"i": 0}

        def fused():
            i = it["i"] % ncopy
            it["i"] += 1
            ops.ctc_fwdbwd(xs_[i], tg, il, tl, time_major=True, grad=gs_[i], workspace=ws)

        ms = timed(fused, 10 if T * V >= 4e6 else 30)
        gbs = T * B * V * 8 / (ms * 1e-3) / 1e9
        row = {"T": T, "L": L, "V": V, "ms": ms, "achieved": gbs, "frac": gbs / pk["hbm"], "l2_rotation": ncopy}
        if torch_too:
            xr = x.clone().requires_grad_(True)

            def ref():
                xr.grad = None
                torch.nn.functional.ctc_loss(xr.log_softmax(-1), tg, il, tl, blank=0, reduction="sum", zero_infinity=False).backward()

            row["torch_cuda_ms"] = timed(ref, 3)
            row["vs_torch_cuda"] = row["torch_cuda_ms"] / ms
            del xr
        grid.append(row)
        del x, grad, ws, xs_, gs_
        torch.cuda.empty_cache()
    big = grid[-1]
    return {"workload": f"standalone CTC fwd+bwd B={B} T={big['T']} V={big['V']} L={big['L']} fp32 (2.05 GB logits > L2); `grid` = all 16 BASELINE config-4 points",
            "ms": big["ms"], "bound": "hbm", "achieved": big["achieved"], "peak": pk["hbm"], "unit": "GB/s", "frac": big["frac"],
            "traffic": None, "grid": grid}


def _traffic():
    """DRAM bytes per step / per launch of the dominant kernel family from the committed ncu capture (profiles/r2_traffic.json,
    written by tools/traffic_summary.py --json from `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum`)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            return json.load(f)
    except Exception:  # noqa: BLE001
        return None


def measure_step(args, wl, dev, dropout: float, rank: int, world: int, want_e2e: bool, want_clocks: bool, steps: int):
    """Build the model + TrainStep for one (workload, dropout) and time it.  -> dict with the step object and the numbers."""
    import torch
    import torch.distributed as dist
    from liteasr_b200 import _lib
    from liteasr_b200.criterions.hybrid_ctc_attn import HybridCTCLoss, HybridCTCLossConfig
    from liteasr_b200.models.u2 import U2, U2Config
    from liteasr_b200.optims import FusedNoam, NoamConfig
    from liteasr_b200.schema import U2Dims
    from liteasr_b200.trainer import Prefetcher, TrainStep
    from liteasr_b200.utils.synthetic import synth_batch
    dims = U2Dims(*wl["dims"])
    torch.manual_seed(42)
    model = U2(U2Config(**dims.__dict__, precision=args.precision, **my_u2_rates(dropout))).to(dev).train()
    crit = HybridCTCLoss(HybridCTCLossConfig(vocab_size=dims.vocab_size, smoothing=wl["smoothing"], ctc_weight=wl["ctc_weight"]))
    step = TrainStep(model, crit, None, clip_grad_norm=5.0, use_graph=not args.no_graph, device=dev)
    step.optimizer = FusedNoam(step.store, NoamConfig(model_dim=dims.enc_dim))
    host = synth_batch(wl["batch"], wl["tmax"], wl["lmax"], dims.vocab_size, seed=42 + rank)
    host = tuple(t.pin_memory() for t in host)
    batch = tuple(t.to(dev) for t in host)
    audio_local = float(host[1].sum()) * FRAME_SHIFT_S

    def barrier():
        if world > 1:
            dist.barrier()

    def timed(fn, k):
        barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        torch.cuda.synchronize()
        barrier()
        ms = e0.elapsed_time(e1) / k
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms

    # launches per step (eager, before capture) -- counts kernels launched by liblasr only; the eager step is also timed: it is
    # what a run with a new input shape every step would see (no graph to replay)
    step.step_eager(*batch)
    torch.cuda.synchronize()
    c0 = _lib.launch_count()
    step.step_eager(*batch)
    torch.cuda.synchronize()
    launches_per_step = _lib.launch_count() - c0
    ms_eager = timed(lambda: step.step_eager(*batch), 3)

    t0 = time.perf_counter()
    static = step.static_inputs(*batch) if step.use_graph else batch
    torch.cuda.synchronize()
    capture_s = time.perf_counter() - t0
    loss = None
    for _ in range(max(3, args.warmup)):
        loss = step(*static)
    torch.cuda.synchronize()

    sampler = ClockSampler(dev.index or 0) if want_clocks else None
    if sampler:
        sampler.start()
    ms = timed(lambda: step(*static), steps)
    res = dict(step=step, batch=batch, host=host, ms=ms, ms_eager=ms_eager, capture_s=capture_s, audio_local=audio_local,
               launches_per_step=int(launches_per_step), loss=float(loss), dims=dims)
    if want_e2e:
        # end-to-end: pinned host batch -> H2D -> step through the public TrainStep call -> loss read back on the host
        loss_host = torch.zeros((), dtype=torch.float32).pin_memory()
        pf = Prefetcher(dev)
        pf.put(host)

        def e2e_step():
            # the public training API: Prefetcher (pinned host -> device on a copy stream, one step ahead) + TrainStep.__call__
            # (device-to-device into the graph's static inputs, graph replay); every step starts one H2D copy of a full batch
            # and reads the loss back on the host
            dev_batch = pf.get()
            pf.put(host)
            l = step(*dev_batch)
            loss_host.copy_(l, non_blocking=False)  # D2H + host sync: the loss is read every step

        for _ in range(2):
            e2e_step()
        res["ms_e2e"] = timed(e2e_step, steps)
        res["h2d"] = sum(t.numel() * t.element_size() for t in host)
        res["loss_last"] = loss_host
    if sampler:
        sampler.stop_flag = True
        sampler.join(timeout=1.0)
        res["clocks"] = sampler.result()
    audio = audio_local
    if world > 1:
        t = torch.tensor([audio_local], device=dev, dtype=torch.float64)
        dist.all_reduce(t)
        audio = float(t)
    res["audio"] = audio
    return res


def variable_shape_run(args, wl, dev, dropout: float):
    """VERDICT r1 item 9: training over the shapes the reference's length-bucketed batching produces (utils/batchify.py:76-112,
    `SeqBatch` over a length-sorted corpus): every batch has its own (Tmax, Lmax).  One epoch runs eagerly (no shape has been
    seen before), the second captures each shape at its second occurrence (bounded LRU cache), the third replays."""
    import types

    import torch
    from liteasr_b200.criterions.hybrid_ctc_attn import HybridCTCLoss, HybridCTCLossConfig
    from liteasr_b200.models.u2 import U2, U2Config
    from liteasr_b200.optims import FusedNoam, NoamConfig
    from liteasr_b200.schema import U2Dims
    from liteasr_b200.trainer import TrainStep
    from liteasr_b200.utils.batchify import SeqBatch, length_sorted_indices
    from liteasr_b200.utils.synthetic import pred_len
    dims = U2Dims(*wl["dims"])
    g = torch.Generator().manual_seed(7)
    # at most 126 utterances per batch and eight shapes: their private graph pools (up to 12 GB each at 126) all stay resident
    # under the cache's memory cap, so the third epoch replays every step; with more shapes than pools the cache keeps what
    # fits and runs the rest eagerly (tests/test_u2_gpu.py::test_graph_cache_is_bounded_by_pool_memory)
    nb, B = 8, min(wl["batch"], 126)
    n = nb * B
    xl = torch.randint(int(0.3 * wl["tmax"]), wl["tmax"] + 1, (n,), generator=g)
    yl = torch.minimum(torch.randint(wl["lmax"] // 2, wl["lmax"] + 1, (n,), generator=g), torch.clamp(pred_len(xl) // 2, min=1))
    order = length_sorted_indices(xl.tolist())
    pol = SeqBatch(types.SimpleNamespace(batch_size=B, min_batch_size=1, max_len_in=10 ** 9, max_len_out=10 ** 9))
    pol.batchify(order, [types.SimpleNamespace(xlen=int(xl[i]), ylen=int(yl[i])) for i in order])
    batches = []
    for idx in pol.data:
        xlens, ylens = xl[idx], yl[idx]
        tmax, lmax = int(xlens.max()), int(ylens.max())
        xs = torch.randn(len(idx), tmax, 80, generator=g) * (torch.arange(tmax).view(1, -1, 1) < xlens.view(-1, 1, 1))
        ys = torch.randint(1, dims.vocab_size - 1, (len(idx), lmax), generator=g)
        ys = ys.masked_fill(torch.arange(lmax).view(1, -1) >= ylens.view(-1, 1), -1)
        batches.append(tuple(t.to(dev) for t in (xs, xlens, ys, ylens)))
    audio = float(xl.sum()) * FRAME_SHIFT_S
    torch.manual_seed(42)
    model = U2(U2Config(**dims.__dict__, precision=args.precision, **my_u2_rates(dropout))).to(dev).train()
    crit = HybridCTCLoss(HybridCTCLossConfig(vocab_size=dims.vocab_size, smoothing=wl["smoothing"], ctc_weight=wl["ctc_weight"]))
    step = TrainStep(model, crit, None, clip_grad_norm=5.0, use_graph=True, device=dev, graph_min_hits=2, max_graphs=len(batches),
                     graph_mem_fraction=0.7)
    step.optimizer = FusedNoam(step.store, NoamConfig(model_dim=dims.enc_dim))
    step.step_eager(*batches[0])  # library warm-up (lazy module load), not timed

    def epoch():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for b in batches:
            step(*b)
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    t_eager, t_capture, t_replay = epoch(), epoch(), epoch()
    return {"what": f"{len(batches)} length-bucketed batches of {B} utterances (SeqBatch over {n} utterances, Tmax {int(xl.min())}..{int(xl.max())}), "
                    f"{len(set((tuple(b[0].shape), tuple(b[2].shape)) for b in batches))} distinct (Tmax, Lmax) shapes; host-timed epochs",
            "audio_s_per_epoch": audio,
            "epoch1_eager": {"value": audio / t_eager, "unit": "audio-s/s", "s": t_eager},
            "epoch2_capturing": {"value": audio / t_capture, "unit": "audio-s/s", "s": t_capture},
            "epoch3_replaying": {"value": audio / t_replay, "unit": "audio-s/s", "s": t_replay},
            "cache": dict(step.stats, entries=len(step.graphs), pool_gb=sum(e[3] for e in step.graphs.values()) / 1e9)}


def gpu_incumbent(wl, dev, dropout: float, host_batch):
    """SURVEY 8d / BASELINE.md 3.7: the reference's own modules on torch-CUDA on this GPU -- eager fp32 and autocast(bf16) --
    same batch, same step (fwd + bwd + clip + Adam).  torch's library kernels are the only GPU incumbent the reference has."""
    import torch
    batch = tuple(t.to(dev) for t in host_batch)
    audio = float(host_batch[1].sum()) * FRAME_SHIFT_S
    out = {}
    kind = None
    for name, autocast in (("fp32", False), ("autocast_bf16", True)):
        step, kind = build_reference_step(wl, dev, dropout, batch)
        for _ in range(2):
            step(autocast)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n = 3
        e0.record()
        for _ in range(n):
            loss = step(autocast)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        out[name] = {"value": audio / (ms * 1e-3), "unit": "audio-s/s", "ms_per_step": ms, "loss": float(loss),
                     "peak_mem_gb": torch.cuda.max_memory_allocated(dev) / 1e9}
        del step
        torch.cuda.empty_cache()
    out["kind"] = kind
    out["what"] = ("the UNMODIFIED reference U2 + HybridCTCLoss modules (copy under baseline/_ref, loaded through oracle/ref_shims.py)"
                   if kind == "reference" else "oracle port of the reference modules (no reference copy on this machine)") + \
                  f" on torch {torch.__version__} CUDA, eager, same {wl['batch']}-utterance batch, dropout {dropout}, fwd+bwd+clip_grad_norm_+Adam, 3 timed steps after 2 warm-up"
    return out


DUMP_SAMPLE = 4 << 20  # parameter / gradient elements written by --dump-outputs: 2 x 16 MB in float32


def dump_outputs(out_dir: str, model, optimizer, loss) -> None:
    """What a caller of the timed step holds after its last step, as DIR/<name>.npy: the loss the call returned, its
    [loss, CTC term, attention term], the updated parameters and their gradients (the same seeded sample of DUMP_SAMPLE
    elements of all parameters concatenated in state_dict order: the whole model is larger than the dump's 64 MB), the
    BatchNorm running statistics and the optimizer's [updates so far, gradient norm, learning rate] of that step (float64).
    Same arguments, same inputs: two builds can be compared array by array.  The names are listed in .gitignore."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    params = [p for _, p in model.named_parameters()]
    n = sum(p.numel() for p in params)
    idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values.to(params[0].device)
    arrays = {
        "loss": loss.float(),
        "loss_terms": model.last_losses.float(),
        "params_sample": torch.cat([p.detach().reshape(-1) for p in params])[idx],
        "grads_sample": torch.cat([p.grad.reshape(-1) for p in params])[idx],
        "bn_running_stats": torch.cat([b.reshape(-1).float() for k, b in model.state_dict().items() if "running" in k]),
        "optimizer_state": optimizer.state[:3].double(),
    }
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().cpu().numpy())


def run_gpu(args, wl):
    import torch
    import torch.distributed as dist
    from liteasr_b200.distributed.utils import distributed_init

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (liteasr_b200 has no CPU fallback); use --impl reference for the CPU arm")
    local = distributed_init("nccl")
    world = dist.get_world_size() if dist.is_initialized() else 1
    rank = dist.get_rank() if dist.is_initialized() else 0
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    pk = peaks()
    extras = rank == 0 and world == 1 and not args.quick

    ddp_check = None
    if world > 1 and not args.no_ddp_check:
        from liteasr_b200.distributed.check import ddp_numeric_check
        ddp_check = ddp_numeric_check(dev)
        if args.check_ddp_shapes:  # opt-in: ranks with different batch shapes capturing graphs at different steps
            from liteasr_b200.distributed.check import ddp_varshape_check
            ddp_check["varshape"] = ddp_varshape_check(dev)

    r = measure_step(args, wl, dev, args.dropout, rank, world, want_e2e=True, want_clocks=True, steps=args.steps)
    ms, audio, dims, step = r["ms"], r["audio"], r["dims"], r["step"]
    if args.dump_outputs and rank == 0:  # before anything below runs another step on the same model
        dump_outputs(args.dump_outputs, step.model, step.optimizer, r["loss_last"])

    # roofline of the dominant kernel family (tcgen05 GEMM), measured live with CUDA events
    flops, gemm_ms, n_gemm, split = gemm_family_replay(step, r["batch"], split=True)
    tflops = flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    traffic = _traffic()
    fam_traffic = (traffic or {}).get("gemm_family_bytes_per_step")
    roof = {"kernel": "gemm_tc_kernel + ffn_fwd_kernel + ffn_bwd_kernel + attn_pair_kernel (tcgen05.mma bf16: every GEMM, implicit-GEMM convolution, fused FFN forward / backward and paired attention-backward contraction of one step)" if args.precision == "bf16" else "gemm_simt_kernel",
            "bound": "tensor", "achieved": tflops, "peak": pk["tc_sustained"], "unit": "TFLOP/s", "frac": tflops / pk["tc_sustained"],
            "traffic": fam_traffic,
            "traffic_note": ((traffic or {}).get("note") if traffic else "no ncu capture found under profiles/"),
            "algorithmic_bytes_per_step": sum(v["bytes"] for v in split.values()),
            "peak_source": pk["src"] + " (sustained bf16: the family's launches of one step replayed back to back from a CUDA graph)",
            "launches": n_gemm, "kernel_ms_per_step": gemm_ms, "share_of_step": gemm_ms / ms, "algorithmic_tflop_per_step": flops / 1e12}
    t, h = split["tensor"], split["hbm"]
    roof_split = {
        "tensor": {"what": "GEMMs with K >= 1024 and the implicit-GEMM convolutions", "bound": "tensor", "launches": t["launches"],
                   "kernel_ms_per_step": t["ms"], "achieved": t["flops"] / (t["ms"] * 1e-3) / 1e12 if t["ms"] else 0.0, "peak": pk["tc_sustained"],
                   "unit": "TFLOP/s", "frac": (t["flops"] / (t["ms"] * 1e-3) / 1e12 / pk["tc_sustained"]) if t["ms"] else 0.0},
        "hbm": {"what": "GEMMs with K < 1024 (K = 256 / 512 / 64: <= 120 FLOP per algorithmic byte, below the 210 FLOP/B machine balance)",
                "bound": "hbm", "launches": h["launches"], "kernel_ms_per_step": h["ms"],
                "achieved": h["bytes"] / (h["ms"] * 1e-3) / 1e9 if h["ms"] else 0.0, "peak": pk["hbm"], "unit": "GB/s",
                "frac": (h["bytes"] / (h["ms"] * 1e-3) / 1e9 / pk["hbm"]) if h["ms"] else 0.0,
                "tflops": h["flops"] / (h["ms"] * 1e-3) / 1e12 if h["ms"] else 0.0},
    }

    tp = (((wl["tmax"] - 3) // 2 + 1) - 3) // 2 + 1
    ctc_logit_mb = wl["batch"] * tp * ((dims.vocab_size + 7) // 8 * 8) * 2 // 1000000
    line = {
        "metric": "audio-sec/sec train (Conformer fwd+bwd+CTC)", "value": audio / (ms * 1e-3), "unit": "audio-s/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
        "config": {"workload": wl["desc"], "global_batch": wl["batch"] * world, "audio_s_per_step": audio, "parallelism": f"dp{world}",
                   "frame_shift_ms": 10, "cuda_graph": bool(step.use_graph), "dropout": args.dropout,
                   "l2": f"per-step working set (several GB of activations, {ctc_logit_mb} MB of CTC logits) exceeds the 126 MB L2; no explicit flush"},
        "clocks": r.get("clocks"),
        "e2e": {"value": audio / (r["ms_e2e"] * 1e-3), "unit": "audio-s/s", "ms_per_step": r["ms_e2e"], "h2d_bytes_per_step": r["h2d"],
                "d2h_bytes_per_step": 4},
        "gpu_launches": int(r["launches_per_step"] * args.steps),
        "gpu_launches_per_step": r["launches_per_step"],
        "eager_no_graph": {"ms_per_step": r["ms_eager"], "value": r["audio_local"] / (r["ms_eager"] * 1e-3), "unit": "audio-s/s (one GPU)",
                           "graph_capture_s": r["capture_s"],
                           "note": "the same step launched kernel by kernel (what every NEW input shape costs before its graph exists)"},
        "roofline": roof,
        "roofline_split": roof_split,
        "loss": r["loss"],
    }
    if ddp_check is not None:
        line["ddp_check"] = ddp_check
    if extras:
        host = r["host"]
        del step, r
        torch.cuda.empty_cache()
        extra = {}
        try:  # the same step with every dropout rate 0 (round-1's configuration)
            if args.dropout > 0:
                r0 = measure_step(args, wl, dev, 0.0, rank, world, want_e2e=False, want_clocks=False, steps=max(5, args.steps // 2))
                extra["dropout_0"] = {"value": r0["audio"] / (r0["ms"] * 1e-3), "unit": "audio-s/s", "ms_per_step": r0["ms"],
                                      "gpu_launches_per_step": r0["launches_per_step"], "eager_ms_per_step": r0["ms_eager"]}
                del r0
                torch.cuda.empty_cache()
        except Exception as e:  # noqa: BLE001
            extra["dropout_0"] = {"error": str(e)}
        try:  # BASELINE configs[2] (C3: d = 512, T' = 399) on one GPU
            if args.workload == "c2":
                w3 = dict(WORKLOADS["c3"])
                r3 = measure_step(args, w3, dev, args.dropout, rank, world, want_e2e=False, want_clocks=False, steps=max(5, args.steps // 2))
                f3, g3, n3 = gemm_family_replay(r3["step"], r3["batch"])
                extra["c3"] = {"workload": w3["desc"], "value": r3["audio"] / (r3["ms"] * 1e-3), "unit": "audio-s/s", "ms_per_step": r3["ms"],
                               "gpu_launches_per_step": r3["launches_per_step"], "dropout": args.dropout,
                               "roofline": {"bound": "tensor", "achieved": f3 / (g3 * 1e-3) / 1e12, "peak": pk["tc_sustained"], "unit": "TFLOP/s",
                                            "frac": f3 / (g3 * 1e-3) / 1e12 / pk["tc_sustained"], "kernel_ms_per_step": g3, "launches": n3}}
                del r3
                torch.cuda.empty_cache()
        except Exception as e:  # noqa: BLE001
            extra["c3"] = {"error": str(e)}
        try:
            extra["variable_shapes"] = variable_shape_run(args, wl, dev, args.dropout)
        except Exception as e:  # noqa: BLE001
            extra["variable_shapes"] = {"error": str(e)}
        torch.cuda.empty_cache()
        line["extra"] = extra
        try:
            line["roofline_ctc"] = ctc_standalone(pk)
        except Exception as e:  # noqa: BLE001
            line["roofline_ctc"] = {"error": str(e)}
        torch.cuda.empty_cache()
        try:
            gi = gpu_incumbent(wl, dev, args.dropout, host)
            line["gpu_incumbent"] = gi
            line["vs_gpu_incumbent"] = {k: line["value"] / gi[k]["value"] for k in ("fp32", "autocast_bf16")}
        except Exception as e:  # noqa: BLE001
            line["gpu_incumbent"] = {"error": str(e)}
        torch.cuda.empty_cache()
        if not args.no_cpu_baseline:
            try:
                # a bounded sample (about 30 s of CPU work): at most 126 utterances of the batch -- the reference's CPU step is
                # linear in the batch (33 s at 126, 68 s at 252 on 16 cores: 36.3 vs 35.5 audio-s/s), so audio-s/s is comparable
                rc = cpu_oracle_run(wl, 1, 0, sample_batch=min(wl["batch"], 126), dropout=args.dropout)
                line["cpu_baseline"] = {"value": rc["value"], "unit": "audio-s/s", "cores": rc["cores"], "kind": rc["kind"], "sample": rc["sample"],
                                        "ms_per_step": rc["ms_per_step"]}
            except Exception as e:  # noqa: BLE001
                line["cpu_baseline"] = {"error": str(e)}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        # the captured graph holds NCCL kernels: tearing the communicator down under it can block, so leave without destructors
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch override (0 = the workload's default)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--dropout", type=float, default=0.1,
                    help="model.dropout_rate: default 0.1 = the reference's shipped training config (config/model/my_U2.yaml; the three "
                         "attention-probability rates stay 0.0); 0 = U2Config's dataclass default (round-1's bench)")
    ap.add_argument("--quick", action="store_true", help="headline numbers only (no extras: dropout-0 / C3 / CTC grid / GPU incumbent / CPU baseline)")
    ap.add_argument("--no-ddp-check", action="store_true", help="skip the NCCL gradient / buffer numeric check that runs first at N > 1")
    ap.add_argument("--check-ddp-shapes", action="store_true", help="N > 1: also run TrainStep with rank-dependent batch shapes (graph capture at different steps)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step computed (loss, sampled parameters and gradients, "
                         "BatchNorm statistics, optimizer step count / gradient norm / learning rate) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's outputs (--impl b200)")
    wl = dict(WORKLOADS[args.workload])
    for k in WORKLOADS:
        WORKLOADS[k]["desc"] = WORKLOADS[k]["desc"].replace("dropout 0 (U2Config default)", f"dropout {args.dropout}")
    wl["desc"] = wl["desc"].replace("dropout 0 (U2Config default)",
                                    f"dropout {args.dropout} (config/model/my_U2.yaml: attention-probability rates 0.0; own Philox stream)" if args.dropout > 0
                                    else "dropout 0 (U2Config dataclass default)")
    if args.batch > 0:
        wl["desc"] = wl["desc"].replace(f"per-GPU batch {wl['batch']}", f"per-GPU batch {args.batch}").replace(f"batch {wl['batch']},", f"batch {args.batch},")
        wl["batch"] = args.batch
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_gpu(args, wl)


if __name__ == "__main__":
    main()
