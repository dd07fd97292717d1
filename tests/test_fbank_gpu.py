"""GPU: the log-mel filterbank kernel (``lasr_fbank``, include/lasr_fbank.h) against torchaudio.compliance.kaldi.fbank in
float64 on the same samples, and ``decoding.transcribe`` against ``decode_batch`` on the same features.

Every output buffer starts as NaN, so a row the kernel never writes fails.  Criteria, per frame, with E64 the float64 mel
energies and the FLT_EPSILON floor applied to both sides:
  - linear: |exp(out) - E64| <= 1e-6 * sum_m E64[m] + E64 * ulp(out).  The second term is the output format's own resolution:
    out is log E rounded to fp32, and one ulp of a log value near 30 is a relative 1.9e-6 in E, more than the 1e-6 budget of
    the frame total when one bin holds most of the frame's energy (a sine).
  - strong bins (E64 >= 1e-3 x the frame's largest): |out - log E64| <= 1e-4.
  - silence and integer constants: every bin is the floor log(FLT_EPSILON) = -15.942385 to within 1 ulp, one constant.
  - rows t >= F_b are exactly 0.
"""
import dataclasses

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

FLT_EPS = float(np.finfo(np.float32).eps)
FLOOR = np.float32(np.log(np.float32(FLT_EPS)))


def _cfg(**kw):
    from liteasr_b200.features import FbankConfig
    return FbankConfig(**kw)


def _run(waves, nsamp, cfg):
    """The kernel on a NaN-filled output.  waves (B, Nmax) CUDA int16 | fp32, nsamp a list."""
    from liteasr_b200 import _lib, features, ops
    win, lo, off, w = features._tables(cfg, waves.device)
    B, nmax = waves.shape
    out = torch.full((B, features.num_frames(nmax, cfg), cfg.num_mel_bins), float("nan"), device=waves.device)
    n = torch.tensor(nsamp, dtype=torch.int64, device=waves.device)
    code = _lib.I16 if waves.dtype == torch.int16 else _lib.F32
    _lib.check(_lib.lib().lasr_fbank(ops._ptr(waves), ops._i(code), ops._l(waves.stride(0)), ops._ptr(n), ops._i(B), ops._l(nmax),
                                     ops._i(cfg.window_size), ops._i(cfg.window_shift), ops._ptr(win), ops._i(cfg.num_mel_bins),
                                     ops._ptr(lo), ops._ptr(off), ops._ptr(w), ops._ptr(out), ops._stream()), "fbank")
    return out.cpu().numpy()


def _oracle(x, cfg):
    """torchaudio's fbank in float64 (mel bank included) -> linear mel energies (F, nb)."""
    import torchaudio.compliance.kaldi as K
    if len(x) < cfg.window_size:
        return np.zeros((0, cfg.num_mel_bins))
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        return K.fbank(torch.from_numpy(np.asarray(x, np.float64))[None], use_log_fbank=False, **dataclasses.asdict(cfg)).numpy()
    finally:
        torch.set_default_dtype(old)


def _check(o, x, cfg, floor_only=False):
    """o (Fmax, nb) kernel rows of one utterance with samples x (float64, exactly the values the kernel read)."""
    E = _oracle(x, cfg)
    F = E.shape[0]
    assert not np.isnan(o).any()
    assert (o[F:] == 0).all()
    o = o[:F]
    if floor_only:
        if F:
            assert (o == o[0, 0]).all() and abs(float(o[0, 0]) - float(FLOOR)) <= float(np.spacing(np.abs(FLOOR)))
        return
    Ef = np.maximum(E, FLT_EPS)
    lin = np.abs(np.exp(o.astype(np.float64)) - Ef)
    tol = 1e-6 * E.sum(1, keepdims=True) + Ef * np.spacing(np.abs(o)).astype(np.float64)
    assert (lin <= tol).all(), float((lin / tol).max())
    strong = E >= 1e-3 * E.max(1, keepdims=True)
    d = np.abs(o.astype(np.float64) - np.log(Ef))
    assert (d[strong] <= 1e-4).all(), float(d[strong].max())


def _signals(n, sr, dtype, rng):
    """name -> float64 samples in int16 scale, integral for int16 (fractional noise / sines / chirp for fp32)."""
    t = np.arange(n) / sr

    def q(x):  # the values the kernel reads
        return np.clip(np.round(x), -32768, 32767) if dtype == torch.int16 else x.astype(np.float32).astype(np.float64)

    f1 = min(7100.0, 0.45 * sr)
    dur = max(n / sr, 1e-3)
    return {
        "noise": q(rng.uniform(-32768, 32767, size=n)),
        "quiet_noise": rng.integers(-3, 4, size=n).astype(np.float64),
        "sines": q(9000.0 * np.sin(2 * np.pi * 440.0 * t) + 6000.0 * np.sin(2 * np.pi * 3000.0 * t + 0.3)),
        "chirp": q(12000.0 * np.sin(2 * np.pi * (100.0 * t + 0.5 * (f1 - 100.0) / dur * t * t))),
        "square": np.clip(40000.0 * np.sign(np.sin(2 * np.pi * 220.0 * t)), -32768, 32767),
        "silence": np.zeros(n),
        "dc": np.full(n, 32767.0),
        "dc_negative": np.full(n, -1234.0),
    }


def _batch(xs, dtype, garbage=None, rng=None):
    """Pad float64 sample arrays into a CUDA (B, Nmax) tensor; the padding holds `garbage` values."""
    nmax = max(len(x) for x in xs)
    w = np.zeros((len(xs), nmax))
    if garbage is not None:
        w[:] = rng.choice(garbage, size=w.shape)
    for b, x in enumerate(xs):
        w[b, : len(x)] = x
    return torch.from_numpy(w).to(dtype).cuda()


@pytest.mark.parametrize("nb", [23, 40, 80, 128])
@pytest.mark.parametrize("sr", [16000, 8000])
@pytest.mark.parametrize("dtype", [torch.int16, torch.float32])
def test_signals_match_float64_torchaudio(dtype, sr, nb):
    cfg = _cfg(num_mel_bins=nb, sample_frequency=float(sr))
    rng = np.random.default_rng(nb + sr)
    sig = _signals(int(1.5 * sr), sr, dtype, rng)
    names = list(sig)
    xs = [sig[k][: len(sig[k]) - 37 * i] for i, k in enumerate(names)]     # ragged lengths
    out = _run(_batch(xs, dtype), [len(x) for x in xs], cfg)
    for b, (k, x) in enumerate(zip(names, xs)):
        _check(out[b], x, cfg, floor_only=k in ("silence", "dc", "dc_negative"))


@pytest.mark.parametrize("sr", [16000, 8000])
@pytest.mark.parametrize("dtype", [torch.int16, torch.float32])
def test_edge_lengths_and_padding_garbage(dtype, sr):
    """N in {0, W-1, W, W+1, W+S-1, W+S, 1 s, 30 s + 123} in one padded batch whose samples past nsamp hold large garbage
    (NaN and 1e30 for fp32): each row matches the oracle and equals the same utterance run alone, bit for bit."""
    cfg = _cfg(sample_frequency=float(sr))
    W, S = cfg.window_size, cfg.window_shift
    rng = np.random.default_rng(sr)
    lens = [0, W - 1, W, W + 1, W + S - 1, W + S, sr, 30 * sr + 123]
    xs = [rng.integers(-32768, 32768, size=n).astype(np.float64) for n in lens]
    garbage = [32767.0, -32768.0] if dtype == torch.int16 else [np.nan, 1e30, -1e30]
    out = _run(_batch(xs, dtype, garbage, rng), lens, cfg)
    for b, x in enumerate(xs):
        _check(out[b], x, cfg)
        if len(x) >= W:
            one = _run(_batch([x], dtype), [len(x)], cfg)[0]
            F = one.shape[0]
            assert np.array_equal(out[b, :F], one), b
    # nsamp clamps to [0, Nmax]: a negative length gives no frame, a length past Nmax reads Nmax samples
    big = _run(_batch([xs[-1], xs[-2]], dtype), [-5, 10 ** 9], cfg)
    assert (big[0] == 0).all()
    _check(big[1], np.concatenate([xs[-2], np.zeros(len(xs[-1]) - len(xs[-2]))]), cfg)


def test_c2_batch_of_256():
    """256 utterances of 6-12 s (the C2 shape), int16, 80 bins at 16 kHz."""
    cfg = _cfg()
    rng = np.random.default_rng(256)
    lens = [int(v) for v in rng.integers(6 * 16000, 12 * 16000 + 1, size=256)]
    lens[0] = 12 * 16000
    xs = []
    for i, n in enumerate(lens):
        sig = _signals(n, 16000, torch.int16, rng)
        xs.append(sig[("noise", "sines", "chirp", "square", "quiet_noise")[i % 5]])
    out = _run(_batch(xs, torch.int16), lens, cfg)
    for b, x in enumerate(xs):
        _check(out[b], x, cfg)


def test_longest_utterance():
    """One 10.9-minute utterance: 65 542 frames, the encoder's limit (T' = 16 384)."""
    cfg = _cfg()
    n = cfg.window_size + 65541 * cfg.window_shift
    rng = np.random.default_rng(65542)
    sig = _signals(n, 16000, torch.int16, rng)
    x = np.concatenate([sig["chirp"][: n // 3], sig["noise"][n // 3: 2 * n // 3], sig["square"][2 * n // 3:]])
    out = _run(_batch([x], torch.int16), [n], cfg)
    assert out.shape == (1, 65542, 80)
    _check(out[0], x, cfg)


def test_features_fbank_entry_point():
    """features.fbank: a padded tensor, a list and nsamp=None agree with the kernel; flens = num_frames; rows past flens are 0."""
    from liteasr_b200 import features
    cfg = _cfg()
    rng = np.random.default_rng(3)
    lens = [16000, 399, 7000, 400]
    xs = [rng.integers(-32768, 32768, size=n).astype(np.float64) for n in lens]
    waves = _batch(xs, torch.int16)
    feats, flens = features.fbank(waves, torch.tensor(lens), cfg)
    assert feats.shape == (4, features.num_frames(16000, cfg), 80) and feats.dtype == torch.float32
    assert flens.device == waves.device and flens.tolist() == [features.num_frames(n, cfg) for n in lens]
    assert np.array_equal(feats.cpu().numpy(), _run(waves, lens, cfg))
    f2, l2 = features.fbank([waves[b, :n] for b, n in enumerate(lens)], None, cfg)
    assert torch.equal(f2, feats) and torch.equal(l2, flens)
    f3, l3 = features.fbank(waves[:1], None, cfg)
    assert torch.equal(f3[0], feats[0]) and l3.tolist() == [flens[0].item()]
    fp, _ = features.fbank(waves.float(), lens, cfg)
    assert torch.equal(fp, feats)                       # int16 and fp32 samples of the same values give the same bits


def test_fbank_captures_in_a_cuda_graph():
    from liteasr_b200 import features
    cfg = _cfg()
    rng = np.random.default_rng(4)
    waves = torch.from_numpy(rng.integers(-32768, 32768, size=(4, 20000)).astype(np.int16)).cuda()
    nsamp = torch.tensor([20000, 12000, 400, 5000], device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        features.fbank(waves, nsamp, cfg)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        feats, flens = features.fbank(waves, nsamp, cfg)
    waves.copy_(torch.from_numpy(rng.integers(-32768, 32768, size=(4, 20000)).astype(np.int16)))
    nsamp.copy_(torch.tensor([1000, 20000, 19999, 0]))
    g.replay()
    ref, rl = features.fbank(waves, nsamp, cfg)
    torch.cuda.synchronize()
    assert torch.equal(feats, ref) and torch.equal(flens, rl)


def test_fbank_errors():
    from liteasr_b200 import features, ops
    cfg = _cfg()
    win, lo, off, w = features._tables(cfg, torch.device("cuda"))
    waves = torch.zeros(2, 4000, dtype=torch.int16, device="cuda")
    n = torch.tensor([4000, 4000], device="cuda")
    with pytest.raises(RuntimeError, match="2048-point"):
        ops.fbank(waves, n, 1025, 160, torch.ones(1025, device="cuda"), lo, off, w)           # NFFT 2048
    lo129 = torch.zeros(129, dtype=torch.int32, device="cuda")
    off129 = torch.zeros(130, dtype=torch.int32, device="cuda")
    with pytest.raises(RuntimeError, match=r"\[4, 128\]"):
        ops.fbank(waves, n, 400, 160, win, lo129, off129, w)                                 # nb = 129
    with pytest.raises(RuntimeError):
        features.fbank(waves.cpu(), n.cpu(), cfg)                                           # host tensor
    with pytest.raises(ValueError):
        features.fbank(waves.double(), n, cfg)                                              # float64 samples
    with pytest.raises(ValueError):
        features.fbank(waves, n[:1], cfg)                                                   # nsamp size


# ---------------------------------------------------------------------------------------------------- transcribe
def _model(precision="fp32"):
    import json
    import os
    from liteasr_b200.models.u2 import U2, U2Config
    from liteasr_b200.schema import U2Dims
    from liteasr_b200.utils.synthetic import synth_state_dict
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "u2_tiny.json")))
    model = U2(U2Config(**{**g["dims"], "precision": precision}))
    model.load_state_dict(synth_state_dict(U2Dims(**g["dims"]), seed=g["seed"]))
    return model.cuda().eval()


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_transcribe_equals_decode_batch_on_features(precision):
    from liteasr_b200 import decoding, features
    model = _model(precision)
    rng = np.random.default_rng(12)
    lens = [16000, 1360, 24000, 8000]                      # 1360 samples: exactly 7 frames
    xs = [rng.integers(-8000, 8000, size=n).astype(np.float64) for n in lens]
    waves = _batch(xs, torch.int16)
    nsamp = torch.tensor(lens)
    ref = decoding.decode_batch(model, *features.fbank(waves, nsamp))
    out = decoding.transcribe(model, waves, nsamp)
    assert out == ref
    assert decoding.transcribe(model, [waves[b, :n] for b, n in enumerate(lens)]) == ref
    # timestamps in seconds at the configured frame shift (the 1360-sample utterance has 5 frames at 12.5 ms: left out)
    cfg = features.FbankConfig(frame_shift=12.5)
    keep = [0, 2, 3]
    ref_ts = decoding.decode_batch(model, *features.fbank(waves[keep], nsamp[keep], cfg), timestamps=True, frame_shift=0.0125)
    out_ts = decoding.transcribe(model, waves[keep], nsamp[keep], cfg, timestamps=True)
    assert out_ts == ref_ts
    for o in out_ts:
        for tok, f0, f1, s0, s1 in o["timestamps"]:
            assert (s0, s1) == decoding.span_seconds(f0, f1, 0.0125)


def test_transcribe_errors():
    from liteasr_b200 import decoding, features
    model = _model()
    waves = torch.zeros(2, 16000, dtype=torch.int16, device="cuda")
    with pytest.raises(ValueError, match="7"):
        decoding.transcribe(model, waves, torch.tensor([16000, 1359]))                # 6 frames
    with pytest.raises(ValueError):
        decoding.transcribe(model, waves, None, features.FbankConfig(num_mel_bins=40))  # encoder takes 80
