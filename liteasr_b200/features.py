"""Kaldi-compatible log-mel filterbank features on the device: raw audio in, the ``(xs, xlens)`` input of training and decoding out.

``fbank(waves, nsamp, cfg)`` equals ``torchaudio.compliance.kaldi.fbank(w, dither=0.0, **cfg)`` per utterance (Kaldi's
``compute-fbank-feats`` with dither 0), except that the log floor is FLT_EPSILON whatever the input dtype, as in Kaldi; the
definition is written out in include/lasr_fbank.h.  The whole padded batch runs in one kernel launch (``lasr_fbank``).

Samples are in int16 scale, Kaldi's convention: pass int16 PCM as is, and multiply a float waveform normalised to [-1, 1] by
32768 first.  No CMVN is applied (the reference's loader applies none).  The window and the mel bank are computed here in numpy
float64 (torchaudio is not a dependency of this module), rounded to fp32 and cached per (config, device).
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, Optional, Sequence, Tuple, Union

import numpy as np
import torch
from torch import Tensor

from . import ops

MS = 0.001                      # torchaudio's MILLISECONDS_TO_SECONDS: frame sizes are int(sr * ms * 0.001), as it computes them
SUPPORTED_NFFT = (256, 512, 1024)
MIN_MEL_BINS, MAX_MEL_BINS = 4, 128


@dataclass(frozen=True)
class FbankConfig:
    """The options of torchaudio.compliance.kaldi.fbank this implementation takes (same names and units: Hz, milliseconds;
    ``high_freq <= 0`` is an offset from the Nyquist frequency).  The last five fields exist so that a Kaldi or torchaudio
    option set converts field by field; values other than their defaults are rejected.  ``dataclasses.asdict(cfg)`` is a valid
    keyword set for torchaudio's fbank."""
    num_mel_bins: int = 80
    sample_frequency: float = 16000.0
    frame_length: float = 25.0
    frame_shift: float = 10.0
    low_freq: float = 20.0
    high_freq: float = 0.0
    dither: float = 0.0
    window_type: str = "povey"
    snip_edges: bool = True
    use_energy: bool = False
    vtln_warp: float = 1.0

    def __post_init__(self):
        if self.dither != 0.0:
            raise ValueError("dither != 0 is not supported: features are deterministic (use dither=0.0)")
        if self.window_type != "povey":
            raise ValueError(f"window_type {self.window_type!r} is not supported: only 'povey'")
        if not self.snip_edges:
            raise ValueError("snip_edges=False is not supported: frames that do not fit the utterance are dropped")
        if self.use_energy:
            raise ValueError("use_energy=True is not supported: the output holds the mel bins only")
        if self.vtln_warp != 1.0:
            raise ValueError("VTLN (vtln_warp != 1.0) is not supported")
        if not self.sample_frequency > 0:
            raise ValueError(f"sample_frequency {self.sample_frequency} must be > 0")
        W, S = self.window_size, self.window_shift
        if S < 1:
            raise ValueError(f"frame_shift {self.frame_shift} ms is less than one sample at {self.sample_frequency} Hz")
        nfft = self.padded_window_size
        if W < 2 or nfft not in SUPPORTED_NFFT:
            raise ValueError(f"frame_length {self.frame_length} ms = {W} samples needs a {nfft}-point FFT; supported are "
                             f"{SUPPORTED_NFFT} (129 to 1024 samples per frame)")
        if not MIN_MEL_BINS <= self.num_mel_bins <= MAX_MEL_BINS:
            raise ValueError(f"num_mel_bins {self.num_mel_bins} outside the supported [{MIN_MEL_BINS}, {MAX_MEL_BINS}]")
        nyq = 0.5 * self.sample_frequency
        hi = self.high_freq + nyq if self.high_freq <= 0.0 else self.high_freq
        if not (0.0 <= self.low_freq < nyq and 0.0 < hi <= nyq and self.low_freq < hi):
            raise ValueError(f"bad low_freq {self.low_freq} / high_freq {self.high_freq} (-> {hi}) for Nyquist {nyq}: need "
                             "0 <= low < Nyquist, 0 < high <= Nyquist and low < high")

    @property
    def window_size(self) -> int:
        """W, samples per frame."""
        return int(self.sample_frequency * self.frame_length * MS)

    @property
    def window_shift(self) -> int:
        """S, samples between frame starts."""
        return int(self.sample_frequency * self.frame_shift * MS)

    @property
    def padded_window_size(self) -> int:
        """NFFT, the next power of two >= W."""
        return 1 << max(self.window_size - 1, 0).bit_length()


def num_frames(nsamp: Union[int, Tensor], cfg: FbankConfig = FbankConfig()) -> Union[int, Tensor]:
    """Frames of an utterance of ``nsamp`` samples (snip_edges): 0 below one window, else 1 + (nsamp - W) // S.
    An int gives an int; an integer tensor gives an int64 tensor on its device."""
    W, S = cfg.window_size, cfg.window_shift
    if isinstance(nsamp, Tensor):
        return torch.div(nsamp.to(torch.int64) - W + S, S, rounding_mode="floor").clamp_min(0)
    n = int(nsamp)
    return 0 if n < W else 1 + (n - W) // S


def povey_window(W: int) -> np.ndarray:
    """(0.5 - 0.5 cos(2 pi j / (W - 1)))^0.85, j < W, float64 (torchaudio's _feature_window_function('povey'))."""
    return np.power(0.5 - 0.5 * np.cos(2.0 * math.pi * np.arange(W) / (W - 1)), 0.85)


def mel_banks(num_bins: int, nfft: int, sample_freq: float, low_freq: float, high_freq: float) -> np.ndarray:
    """Kaldi's triangular mel bank (num_bins, nfft // 2) in float64, without the Nyquist column (torchaudio's get_mel_banks
    without VTLN): bin m rises from mel_low + m * d to its peak at mel_low + (m + 1) * d and falls to zero at mel_low + (m + 2) * d,
    d = (mel_high - mel_low) / (num_bins + 1), with mel(f) = 1127 ln(1 + f / 700)."""
    def mel(f):
        return 1127.0 * np.log(1.0 + np.asarray(f, dtype=np.float64) / 700.0)

    nyq = 0.5 * sample_freq
    if high_freq <= 0.0:
        high_freq += nyq
    mlo, mhi = float(mel(low_freq)), float(mel(high_freq))
    d = (mhi - mlo) / (num_bins + 1)
    b = np.arange(num_bins, dtype=np.float64)[:, None]
    left, center, right = mlo + b * d, mlo + (b + 1.0) * d, mlo + (b + 2.0) * d
    m = mel(sample_freq / nfft * np.arange(nfft // 2, dtype=np.float64))[None, :]
    return np.maximum(0.0, np.minimum((m - left) / (center - left), (right - m) / (right - center)))


def sparse_mel_banks(cfg: FbankConfig) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """The mel bank as lasr_fbank takes it: (mel_lo (nb,) int32, mel_off (nb+1,) int32, mel_w fp32): bin m weights FFT bins
    mel_lo[m] + j, j < mel_off[m+1] - mel_off[m], by mel_w[mel_off[m] + j].  The nonzero weights of a triangle are contiguous."""
    M = mel_banks(cfg.num_mel_bins, cfg.padded_window_size, cfg.sample_frequency, cfg.low_freq, cfg.high_freq)
    lo = np.zeros(M.shape[0], np.int32)
    off = np.zeros(M.shape[0] + 1, np.int32)
    ws = []
    for i, row in enumerate(M):
        nz = np.flatnonzero(row > 0.0)
        if nz.size:
            lo[i] = nz[0]
            ws.append(row[nz[0]: nz[-1] + 1])
            assert (ws[-1] > 0.0).all()
        off[i + 1] = off[i] + nz.size
    w = np.concatenate(ws).astype(np.float32) if ws else np.zeros(0, np.float32)
    return lo, off, w


_TABLES: Dict[Tuple[FbankConfig, torch.device], Tuple[Tensor, Tensor, Tensor, Tensor]] = {}


def _tables(cfg: FbankConfig, device: torch.device):
    key = (cfg, device)
    if key not in _TABLES:
        lo, off, w = sparse_mel_banks(cfg)
        win = povey_window(cfg.window_size).astype(np.float32)
        _TABLES[key] = tuple(torch.from_numpy(a).to(device) for a in (win, lo, off, w))
    return _TABLES[key]


def fbank(waves: Union[Tensor, Sequence[Tensor]], nsamp: Optional[Union[Tensor, Sequence[int]]] = None,
          cfg: FbankConfig = FbankConfig()) -> Tuple[Tensor, Tensor]:
    """Log-mel filterbank features of a batch of waveforms in one kernel launch.
    waves: a padded (B, Nmax) CUDA tensor of int16 or fp32 samples in int16 scale, with nsamp (B,) valid lengths (None: every row
    is Nmax samples long; lengths are clamped to [0, Nmax]); or a list of 1-D CUDA tensors of one dtype (nsamp must be None).
    -> (feats (B, Fmax, num_mel_bins) fp32, flens (B,) int64), both on the device: Fmax = num_frames(Nmax), rows t >= flens[b]
    are 0.  Utterance b equals torchaudio.compliance.kaldi.fbank(waves[b, :nsamp[b]][None], dither=0.0, **asdict(cfg)) with
    the log floor at FLT_EPSILON.
    Raises RuntimeError for tensors not on a CUDA device, ValueError for any other unsupported input."""
    if isinstance(waves, (list, tuple)):
        if not waves or nsamp is not None:
            raise ValueError("a list of waveforms must be non-empty and carries its own lengths (nsamp must be None)")
        for w in waves:
            if not isinstance(w, Tensor) or w.dim() != 1:
                raise ValueError("a list of waveforms must hold 1-D tensors")
            if not w.is_cuda:
                raise RuntimeError("features.fbank needs CUDA tensors (there is no CPU fallback)")
            if w.dtype != waves[0].dtype or w.device != waves[0].device:
                raise ValueError("the waveforms of a list must share one dtype and one device")
        x = torch.nn.utils.rnn.pad_sequence(list(waves), batch_first=True)
        n = torch.tensor([w.shape[0] for w in waves], dtype=torch.int64).to(x.device)
    else:
        if not isinstance(waves, Tensor) or waves.dim() != 2:
            raise ValueError("waves must be a padded (B, Nmax) tensor or a list of 1-D tensors")
        if not waves.is_cuda:
            raise RuntimeError("features.fbank needs CUDA tensors (there is no CPU fallback)")
        x = waves if waves.stride(1) == 1 else waves.contiguous()
        if nsamp is None:
            n = torch.full((x.shape[0],), x.shape[1], dtype=torch.int64, device=x.device)
        else:
            n = torch.as_tensor(nsamp).reshape(-1).to(device=x.device, dtype=torch.int64)
            if n.numel() != x.shape[0]:
                raise ValueError(f"nsamp has {n.numel()} entries for a batch of {x.shape[0]}")
    if x.dtype not in (torch.int16, torch.float32):
        raise ValueError(f"samples must be int16 or fp32 (in int16 scale), not {x.dtype}")
    if x.shape[0] == 0:
        raise ValueError("an empty batch")
    win, lo, off, w = _tables(cfg, x.device)
    feats = ops.fbank(x, n, cfg.window_size, cfg.window_shift, win, lo, off, w)
    return feats, num_frames(n.clamp(0, x.shape[1]), cfg)
