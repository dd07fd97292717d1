"""CPU: the filterbank's tables and frame counts against torchaudio, the ABI of include/lasr_fbank.h, the configuration checks
and tools/fbank_bench.py's command line."""
import ctypes as C
import dataclasses
import os
import re
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

from test_abi_bindings_cpu import _C_KIND, _Recorder  # the recorder and C-type table of the lasr.h binding check

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCRIPT = os.path.join(ROOT, "tools", "fbank_bench.py")


def _configs():
    """Every NFFT (256 / 512 / 1024) at the common sample rates, bin counts from the smallest to the largest supported, and
    explicit frequency limits (low > 0, high below and at Nyquist)."""
    from liteasr_b200.features import FbankConfig
    out = []
    for sr, fl in ((8000, 25.0), (16000, 25.0), (8000, 60.0), (16000, 32.0), (16000, 50.0), (16000, 64.0), (22050, 25.0), (44100, 10.0)):
        for nb in (4, 23, 40, 80, 128):
            for lo, hi in ((20.0, 0.0), (0.0, -400.0), (64.0, 3800.0)):
                out.append(FbankConfig(num_mel_bins=nb, sample_frequency=float(sr), frame_length=fl, low_freq=lo, high_freq=hi))
    assert {c.padded_window_size for c in out} == {256, 512, 1024}
    return out


@pytest.fixture
def float64_default():
    """torchaudio builds its mel bank in the default dtype: float64 for a float64 reference."""
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    yield
    torch.set_default_dtype(old)


def test_tables_equal_torchaudio(float64_default):
    import torchaudio.compliance.kaldi as K
    from liteasr_b200 import features
    for cfg in _configs():
        W, nfft = cfg.window_size, cfg.padded_window_size
        win = K._feature_window_function("povey", W, 0.42, torch.device("cpu"), torch.float64).numpy()
        assert np.abs(features.povey_window(W) - win).max() <= 1e-12, cfg
        ref, _ = K.get_mel_banks(cfg.num_mel_bins, nfft, cfg.sample_frequency, cfg.low_freq, cfg.high_freq, 100.0, -500.0, 1.0)
        M = features.mel_banks(cfg.num_mel_bins, nfft, cfg.sample_frequency, cfg.low_freq, cfg.high_freq)
        assert M.shape == tuple(ref.shape) == (cfg.num_mel_bins, nfft // 2)
        assert np.abs(M - ref.numpy()).max() <= 1e-12, cfg
        # the sparse form the kernel reads is the fp32 rounding of the same bank, ranges in bounds
        lo, off, w = features.sparse_mel_banks(cfg)
        assert off[0] == 0 and (np.diff(off) >= 0).all() and w.size == off[-1] and w.dtype == np.float32
        dense = np.zeros_like(M, dtype=np.float32)
        for m in range(cfg.num_mel_bins):
            n = off[m + 1] - off[m]
            assert 0 <= lo[m] and lo[m] + n <= nfft // 2
            dense[m, lo[m]: lo[m] + n] = w[off[m]: off[m + 1]]
        assert (dense == M.astype(np.float32)).all(), cfg


def test_num_frames_equals_torchaudio():
    import torchaudio.compliance.kaldi as K
    from liteasr_b200.features import FbankConfig, num_frames
    for cfg in (FbankConfig(), FbankConfig(sample_frequency=8000.0), FbankConfig(frame_length=64.0, frame_shift=12.5)):
        W, S = cfg.window_size, cfg.window_shift
        ns = [0, 1, W - 1, W, W + 1, W + S - 1, W + S, W + S + 1, 16000, 480123]
        for n in ns:
            ref = K._get_strided(torch.zeros(n), W, S, True).shape[0]
            assert num_frames(n, cfg) == ref, (cfg, n)
        t = num_frames(torch.tensor(ns), cfg)
        assert t.dtype == torch.int64 and t.tolist() == [num_frames(n, cfg) for n in ns]
    assert FbankConfig().window_size == 400 and FbankConfig().window_shift == 160 and FbankConfig().padded_window_size == 512


def test_config_rejects_unsupported_options():
    from liteasr_b200.features import FbankConfig
    for kw in (dict(dither=1.0), dict(window_type="hamming"), dict(snip_edges=False), dict(use_energy=True), dict(vtln_warp=0.9),
               dict(frame_length=64.1),                    # 1025 samples: a 2048-point FFT
               dict(frame_length=8.0),                     # 128 samples: a 128-point FFT
               dict(num_mel_bins=3), dict(num_mel_bins=129),
               dict(frame_shift=0.01),                     # less than one sample
               dict(sample_frequency=0.0),
               dict(low_freq=8000.0), dict(low_freq=-1.0), dict(high_freq=8001.0), dict(high_freq=-8000.0),
               dict(low_freq=4000.0, high_freq=3000.0)):
        with pytest.raises(ValueError):
            FbankConfig(**kw)
    FbankConfig(frame_length=64.0)                         # 1024 samples: the largest supported FFT
    FbankConfig(num_mel_bins=4)
    FbankConfig(num_mel_bins=128)
    # the field names are torchaudio's: a config is a valid keyword set for torchaudio.compliance.kaldi.fbank
    import inspect

    import torchaudio.compliance.kaldi as K
    assert set(dataclasses.asdict(FbankConfig())) <= set(inspect.signature(K.fbank).parameters)


def test_fbank_rejects_host_tensors_and_bad_inputs():
    from liteasr_b200 import decoding, features
    with pytest.raises(RuntimeError):
        features.fbank(torch.zeros(2, 1000, dtype=torch.int16), torch.tensor([1000, 500]))
    with pytest.raises(RuntimeError):
        features.fbank([torch.zeros(1000), torch.zeros(500)])
    with pytest.raises(ValueError):
        features.fbank([torch.zeros(1000)], [1000])               # a list carries its own lengths
    with pytest.raises(ValueError):
        features.fbank(torch.zeros(1000))                          # 1-D: not a padded batch
    model = types.SimpleNamespace(encoder=types.SimpleNamespace(i_dim=80))
    with pytest.raises(ValueError):
        decoding.transcribe(model, torch.zeros(1, 16000), None, features.FbankConfig(num_mel_bins=40))


def _fbank_prototypes():
    from liteasr_b200 import _lib
    src = re.sub(r"/\*.*?\*/", "", open(_lib.FBANK_HEADER_PATH).read(), flags=re.S)
    src = re.sub(r"#.*", "", src)
    protos = {}
    for m in re.finditer(r"\b(lasr_[a-z0-9_]+)\s*\(([^()]*)\)\s*;", src):
        kinds = []
        for p in " ".join(m.group(2).split()).split(","):
            p = p.strip()
            kinds.append("ptr" if "*" in p else _C_KIND[" ".join(p.replace("const ", "").split()[:-1])])
        protos[m.group(1)] = kinds
    return protos


def test_fbank_binding_matches_the_header(monkeypatch):
    from liteasr_b200 import _lib, features, ops
    rec = _Recorder()
    monkeypatch.setattr(_lib, "_lib", rec)
    monkeypatch.setattr(ops, "_require_cuda", lambda *ts: None)
    monkeypatch.setattr(ops, "_stream", lambda: C.c_void_p(0))
    protos = _fbank_prototypes()
    assert set(protos) == {"lasr_fbank"}
    cfg = features.FbankConfig()
    lo, off, w = (torch.from_numpy(a) for a in features.sparse_mel_banks(cfg))
    win = torch.from_numpy(features.povey_window(cfg.window_size).astype(np.float32))
    for dt in (torch.int16, torch.float32):
        out = ops.fbank(torch.zeros(3, 1000, dtype=dt), torch.zeros(3, dtype=torch.int64), 400, 160, win, lo, off, w)
        assert out.shape == (3, 1 + (1000 - 400) // 160, 80)
    assert ops.fbank(torch.zeros(1, 399), torch.zeros(1, dtype=torch.int64), 400, 160, win, lo, off, w).shape == (1, 0, 80)
    assert len(rec.calls) == 3
    for name, kinds in rec.calls:
        assert name in protos, f"{name} is called but not declared in include/lasr_fbank.h"
        assert kinds == protos[name], f"{name}: passed {kinds}, declared {protos[name]}"


def test_fbank_symbols_are_exported():
    from liteasr_b200 import _lib, build
    build.build()
    lib = C.CDLL(_lib.LIB_PATH)
    names = _lib.declared_symbols(_lib.FBANK_HEADER_PATH)
    assert names == ["lasr_fbank"]
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/lasr_fbank.h but not exported"


def test_fbank_argument_checks_need_no_device():
    """The argument checks run before any CUDA call: the returned codes and messages are host-side."""
    from liteasr_b200 import _lib, build
    build.build()
    lib = C.CDLL(_lib.LIB_PATH)
    lib.lasr_last_error.restype = C.c_char_p
    p = C.c_void_p(8)

    def call(frame_len=400, nb=80, shift=160, dtype=2, B=1):
        return lib.lasr_fbank(p, C.c_int(dtype), C.c_int64(1000), p, C.c_int(B), C.c_int64(1000), C.c_int(frame_len), C.c_int(shift),
                              p, C.c_int(nb), p, p, p, p, None)

    for kw, needle in ((dict(frame_len=1025), b"2048-point"), (dict(frame_len=128), b"128-point"), (dict(nb=129), b"[4, 128]"),
                       (dict(nb=3), b"[4, 128]"), (dict(shift=0), b">= 1"), (dict(dtype=1), b"dtype"), (dict(B=70000), b"65535")):
        assert call(**kw) == -1, kw
        assert needle in lib.lasr_last_error(), (kw, lib.lasr_last_error())


def test_fbank_bench_help():
    r = subprocess.run([sys.executable, SCRIPT, "--help"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "--n" in r.stdout and "--seconds" in r.stdout


def test_fbank_bench_no_gpu_exits_nonzero():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, SCRIPT, "--n", "4"], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode != 0
    assert r.stdout.strip() == ""
