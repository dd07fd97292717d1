"""TEST INFRASTRUCTURE ONLY -- CPU restatement of LiteASR's U2 + hybrid CTC/attention path.

This file is the *oracle*: a functional (state_dict in, tensors out) restatement, in plain
torch CPU ops plus a C/numpy CTC lattice, of exactly the arithmetic the reference performs
on its training hot path.  It is pinned against the unmodified reference (imported through
``oracle/ref_shims.py``) by ``oracle/make_golden.py`` -> ``tests/golden/*.json``; see
``tests/test_oracle_golden.py``.  Only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may import it.  The product
(``liteasr_b200``) never does.

Every function cites the reference lines it restates (paths relative to
``/root/reference/liteasr``).  Tensors are ``(B, T, feat)`` unless stated otherwise; all
functions are dtype-agnostic (float32 reproduces the reference bit-for-bit on the same
torch build for most ops, float64 is used for tight pins).
"""
from __future__ import annotations

import ctypes
import hashlib
import math
import os
import subprocess
import tempfile
from dataclasses import dataclass
from typing import Dict, Optional, Tuple

import numpy as np
import torch

Tensor = torch.Tensor
SD = Dict[str, Tensor]

LN_EPS = 1e-12  # nets/layer_norm.py:10
BN_EPS = 1e-5  # torch BatchNorm1d default, nets/conformer_convolution.py:41
BN_MOMENTUM = 0.1
MASK_FILL = -1e38  # nets/attention.py:54
DW_KERNEL = 15  # nets/transformer_encoder.py:98


@dataclass
class U2Shape:
    """The subset of ``U2Config`` (models/u2.py:35-67) that changes arithmetic."""

    input_dim: int = 80
    vocab_size: int = 500
    enc_dim: int = 256
    enc_ff_dim: int = 2048
    enc_attn_heads: int = 4
    enc_layers: int = 12
    dec_dim: int = 256
    dec_ff_dim: int = 2048
    dec_attn_heads: int = 4
    dec_layers: int = 6

    def as_ref_cfg(self) -> dict:
        return dict(self.__dict__)


# --------------------------------------------------------------------------------------
# dropout (nn.Dropout / F.dropout sites of the reference; masks = the product's own Philox stream, replayed)
# --------------------------------------------------------------------------------------
NET_ENC, NET_DEC, NET_CTC = 1, 2, 3
(ENC_POS_X, ENC_POS_EMB, ENC_FFM_INNER, ENC_FFM_OUT, ENC_ATT_PROB, ENC_ATT_OUT, ENC_CONV_OUT, ENC_FF_INNER,
 ENC_FF_OUT) = range(1, 10)
DEC_POS, DEC_SELF_PROB, DEC_SELF_OUT, DEC_SRC_PROB, DEC_SRC_OUT, DEC_FF_INNER, DEC_FF_OUT = range(1, 8)
CTC_IN = 1
GLOBAL_LAYER = 0xFFFF


@dataclass
class DropRates:
    """The ten dropout fields of ``U2Config`` (models/u2.py:39,49-52,62-66) after interpolation."""

    dropout_rate: float = 0.0            # CTC head input (nets/ctc.py:29; applied in train AND eval, quirk Q3)
    enc_dropout_rate: float = 0.0        # Conformer sub-layer outputs (nets/conformer_layer.py:42,54,63,125)
    enc_pos_dropout_rate: float = 0.0    # x * sqrt(d) and pos_emb (nets/positional_encoding.py:75)
    enc_attn_dropout_rate: float = 0.0   # attention probabilities (nets/attention.py:55)
    enc_ff_dropout_rate: float = 0.0     # FFN inner (nets/feed_forward.py:19)
    dec_dropout_rate: float = 0.0
    dec_pos_dropout_rate: float = 0.0
    dec_self_attn_dropout_rate: float = 0.0
    dec_src_attn_dropout_rate: float = 0.0
    dec_ff_dropout_rate: float = 0.0

    @classmethod
    def uniform(cls, p: float, attn: float = 0.0) -> "DropRates":
        """config/model/my_U2.yaml: one rate everywhere, the three attention rates overridden."""
        return cls(p, p, p, attn, p, p, p, attn, attn, p)


class Dropper:
    """x -> x * keep / (1 - p) with keep from oracle/philox_oracle.py (the published Philox4x32-10 + the product's site /
    row / column indexing, restated).  The reference draws its masks from torch's global generator, which fused kernels cannot
    replay (SURVEY 8a): parity with dropout is therefore stated as 'the reference arithmetic under the SAME masks'."""

    def __init__(self, rates: DropRates, seed: int, step: int, training: bool = True):
        self.r, self.seed, self.step, self.training = rates, int(seed), int(step), training

    def __call__(self, x: Tensor, net: int, layer: int, kind: int, p: float, always: bool = False) -> Tensor:
        if p <= 0.0 or not (self.training or always):
            return x
        from oracle import philox_oracle
        site = ((net & 0xFF) << 24) | ((layer & 0xFFFF) << 8) | (kind & 0xFF)
        return philox_oracle.apply(x, site, self.seed, self.step, p)


def _nodrop(x, *a, **k):
    return x


# --------------------------------------------------------------------------------------
# masks / lengths / targets
# --------------------------------------------------------------------------------------
def pad_mask(lens: Tensor, width: Optional[int] = None) -> Tensor:
    """utils/mask.py:8-27 -- True marks padding. Width defaults to max(lens)."""
    w = int(lens.max()) if width is None else width
    return torch.arange(w).unsqueeze(0) >= lens.unsqueeze(1)


def causal_mask(n: int) -> Tensor:
    """utils/mask.py:30-90 with col=0, stage=1, diagonal=1 -- True above the diagonal."""
    r = torch.arange(n)
    return r.unsqueeze(0) > r.unsqueeze(1)


def subsampled_len(xlens: Tensor) -> Tensor:
    """models/u2.py:319-321 ``get_pred_len``."""
    return ((xlens - 1) // 2 - 1) // 2


def subsample_mask(mask: Tensor) -> Tensor:
    """nets/transformer_encoder.py:118 ("convolution simulation")."""
    return mask[:, :-2:2][:, :-2:2]


def decoder_inputs(ys: Tensor, ylens: Tensor, vocab: int) -> Tuple[Tensor, Tensor]:
    """models/u2.py:339-358 -- ys_in = [sos | ys with -1 -> eos]; ys_mask over ylens+1."""
    eos = vocab - 1
    ys_ = torch.where(ys == -1, torch.full_like(ys, eos), ys)
    sos = torch.full((ys.size(0), 1), eos, dtype=ys.dtype)
    return torch.cat([sos, ys_], dim=1), pad_mask(ylens + 1)


def attention_targets(ys: Tensor, ylens: Tensor, vocab: int) -> Tensor:
    """models/u2.py:323-328 -- [ys | -1] with eos written at column ylens[b]."""
    tgt = torch.cat([ys, torch.full((ys.size(0), 1), -1, dtype=ys.dtype)], dim=1)
    tgt[torch.arange(ys.size(0)), ylens] = vocab - 1
    return tgt


# --------------------------------------------------------------------------------------
# primitive blocks
# --------------------------------------------------------------------------------------
def layer_norm(sd: SD, p: str, x: Tensor) -> Tensor:
    """nets/layer_norm.py:8-29 (eps = 1e-12, affine)."""
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    return (x - mu) / torch.sqrt(var + LN_EPS) * sd[p + ".weight"] + sd[p + ".bias"]


def dense(sd: SD, p: str, x: Tensor, bias: bool = True) -> Tensor:
    y = x @ sd[p + ".weight"].t()
    return y + sd[p + ".bias"] if bias else y


def swish(x: Tensor) -> Tensor:
    """nets/swish.py:14-16."""
    return x * torch.sigmoid(x)


def sinusoid_table(n: int, d: int, dtype) -> Tensor:
    """nets/positional_encoding.py:29-38 (computed in float32 like the buffer, then cast)."""
    pos = torch.arange(0, n).unsqueeze(1).float()
    div = torch.exp(torch.arange(0, d, 2).float() * -(math.log(10000.0) / d))
    pe = torch.zeros(n, d)
    pe[:, 0::2] = torch.sin(pos * div)
    pe[:, 1::2] = torch.cos(pos * div)
    return pe.to(dtype)


def conv2d_subsampling(sd: SD, p: str, x: Tensor) -> Tensor:
    """nets/subsampling.py:42-48 -- two 3x3 stride-2 convs + ReLU, (c,f)-major flatten, Linear."""
    F = torch.nn.functional
    h = F.relu(F.conv2d(x.unsqueeze(1), sd[p + ".conv.0.weight"], sd[p + ".conv.0.bias"], stride=2))
    h = F.relu(F.conv2d(h, sd[p + ".conv.2.weight"], sd[p + ".conv.2.bias"], stride=2))
    b, c, t, f = h.shape
    h = h.permute(0, 2, 1, 3).reshape(b, t, c * f)
    return dense(sd, p + ".out", h)


def rel_shift_index(t: int) -> Tuple[Tensor, Tensor, Tensor]:
    """Closed form of the legacy ``rel_shift`` (nets/attention.py:99-118, zero_triu=False).

    out[i, j] = BD[i, t-1-(i-j)]   if j <= i
              = 0                   if j == i + 1
              = BD[i+1, j-i-2]      if j >  i + 1
    Derived from the pad/view trick: flat = (i+1)*t + j in the (t, t+1) zero-padded buffer,
    row r = flat // (t+1), col c = flat % (t+1); c == 0 is the pad, else BD[r, c-1].
    Returns (row, col, is_zero) index tensors of shape (t, t).
    """
    i = torch.arange(t).unsqueeze(1).expand(t, t)
    j = torch.arange(t).unsqueeze(0).expand(t, t)
    flat = (i + 1) * t + j
    r = flat // (t + 1)
    c = flat % (t + 1)
    zero = c == 0
    return r.clamp(max=t - 1), (c - 1).clamp(min=0), zero


def rel_shift(bd: Tensor) -> Tensor:
    t = bd.size(-1)
    r, c, zero = rel_shift_index(t)
    out = bd[..., r, c]
    return out.masked_fill(zero, 0.0)


def split_heads(x: Tensor, h: int) -> Tensor:
    b, t, d = x.shape
    return x.view(b, t, h, d // h).transpose(1, 2)  # (B,H,T,dk)


def softmax_attend(scores: Tensor, v: Tensor, mask: Optional[Tensor], drop=_nodrop) -> Tensor:
    """nets/attention.py:46-59 minus linear_o: masked_fill(-1e38) -> softmax -> dropout -> @V -> merge heads.
    No post-softmax re-zeroing (quirk Q4)."""
    if mask is not None:
        scores = scores.masked_fill(mask, MASK_FILL)
    a = drop(torch.softmax(scores, dim=-1))
    o = a @ v
    b, h, t, dk = o.shape
    return o.transpose(1, 2).reshape(b, t, h * dk)


def rel_self_attention(sd: SD, p: str, x: Tensor, pos: Tensor, mask: Optional[Tensor], h: int, drop=_nodrop) -> Tensor:
    """nets/attention.py:120-154.  x (B,T,d) already layer-normed; pos (1,T,d); mask (B,1,1,T)."""
    d = x.size(-1)
    dk = d // h
    q = split_heads(dense(sd, p + ".linear_q", x), h)
    k = split_heads(dense(sd, p + ".linear_k", x), h)
    v = split_heads(dense(sd, p + ".linear_v", x), h)
    pp = split_heads(dense(sd, p + ".linear_pos", pos, bias=False), h)  # (1,H,T,dk)
    qu = q + sd[p + ".pos_bias_u"].unsqueeze(0).unsqueeze(2)
    qv = q + sd[p + ".pos_bias_v"].unsqueeze(0).unsqueeze(2)
    ac = qu @ k.transpose(-2, -1)
    bd = rel_shift(qv @ pp.transpose(-2, -1))
    scores = (ac + bd) * (dk ** -0.5)
    return dense(sd, p + ".linear_o", softmax_attend(scores, v, mask, drop))


def attention(sd: SD, p: str, xq: Tensor, xkv: Tensor, mask: Optional[Tensor], h: int, drop=_nodrop) -> Tensor:
    """nets/attention.py:61-71 (plain scaled dot-product MHA; decoder self/src attention)."""
    dk = xq.size(-1) // h
    q = split_heads(dense(sd, p + ".linear_q", xq), h)
    k = split_heads(dense(sd, p + ".linear_k", xkv), h)
    v = split_heads(dense(sd, p + ".linear_v", xkv), h)
    scores = (dk ** -0.5) * (q @ k.transpose(-2, -1))
    return dense(sd, p + ".linear_o", softmax_attend(scores, v, mask, drop))


def feed_forward(sd: SD, p: str, x: Tensor, act, drop=_nodrop) -> Tensor:
    """nets/feed_forward.py:18-19: fc2(dropout(act(fc1 x)))."""
    return dense(sd, p + ".fc2", drop(act(dense(sd, p + ".fc1", x))))


def conv_module(sd: SD, p: str, x: Tensor, training: bool, bn_out: Optional[dict]) -> Tensor:
    """nets/conformer_convolution.py:44-57.  x (B,T,d) already layer-normed.

    pointwise(d->2d) -> GLU(first half * sigmoid(second half)) -> depthwise k=15 pad 7 ->
    BatchNorm1d (train: biased batch stats over ALL B*T frames incl. padding, quirk Q2;
    eval: running stats) -> Swish -> pointwise(d->d).  ``bn_out`` receives the running-stat
    update torch would have applied (momentum 0.1, unbiased variance)."""
    F = torch.nn.functional
    d = x.size(-1)
    y = x @ sd[p + ".pointwise_conv1.weight"].squeeze(-1).t() + sd[p + ".pointwise_conv1.bias"]
    y = y[..., :d] * torch.sigmoid(y[..., d:])
    y = F.conv1d(
        y.transpose(1, 2), sd[p + ".depthwise_conv.weight"], sd[p + ".depthwise_conv.bias"],
        padding=(DW_KERNEL - 1) // 2, groups=d,
    ).transpose(1, 2)  # (B,T,d)
    if training:
        n = y.size(0) * y.size(1)
        mean = y.mean(dim=(0, 1))
        var = ((y - mean) ** 2).mean(dim=(0, 1))
        if bn_out is not None:
            rm, rv = sd[p + ".norm.running_mean"], sd[p + ".norm.running_var"]
            bn_out[p + ".norm.running_mean"] = ((1 - BN_MOMENTUM) * rm + BN_MOMENTUM * mean).detach()
            bn_out[p + ".norm.running_var"] = (
                (1 - BN_MOMENTUM) * rv + BN_MOMENTUM * var * (n / max(n - 1, 1))
            ).detach()
            bn_out[p + ".norm.num_batches_tracked"] = sd[p + ".norm.num_batches_tracked"] + 1
    else:
        mean, var = sd[p + ".norm.running_mean"], sd[p + ".norm.running_var"]
    y = (y - mean) / torch.sqrt(var + BN_EPS) * sd[p + ".norm.weight"] + sd[p + ".norm.bias"]
    y = swish(y)
    return y @ sd[p + ".pointwise_conv2.weight"].squeeze(-1).t() + sd[p + ".pointwise_conv2.bias"]


def conformer_layer(sd: SD, p: str, x: Tensor, pos: Tensor, mask, h: int, training: bool, bn_out, dp=None, li: int = 0) -> Tensor:
    """nets/conformer_layer.py:130-147 (pre-norm, macaron FFN scale 0.5, extra final_norm); ``dp`` = Dropper or None."""
    def d(kind, rate):
        return (lambda t: dp(t, NET_ENC, li, kind, rate)) if dp is not None else _nodrop
    r = dp.r if dp is not None else DropRates()
    out = r.enc_dropout_rate
    x = x + 0.5 * d(ENC_FFM_OUT, out)(feed_forward(sd, p + ".feed_forward_macaron", layer_norm(sd, p + ".feed_forward_macaron_norm", x),
                                                     swish, d(ENC_FFM_INNER, r.enc_ff_dropout_rate)))
    x = x + d(ENC_ATT_OUT, out)(rel_self_attention(sd, p + ".self_attn", layer_norm(sd, p + ".self_attn_norm", x), pos, mask, h,
                                                    d(ENC_ATT_PROB, r.enc_attn_dropout_rate)))
    x = x + d(ENC_CONV_OUT, out)(conv_module(sd, p + ".conv", layer_norm(sd, p + ".conv_norm", x), training, bn_out))
    x = x + 0.5 * d(ENC_FF_OUT, out)(feed_forward(sd, p + ".feed_forward", layer_norm(sd, p + ".feed_forward_norm", x), swish,
                                                    d(ENC_FF_INNER, r.enc_ff_dropout_rate)))
    return layer_norm(sd, p + ".final_norm", x)


def encoder(sd: SD, cfg: U2Shape, xs: Tensor, xs_mask: Optional[Tensor], training: bool = True,
            bn_out: Optional[dict] = None, dp=None) -> Tensor:
    """nets/transformer_encoder.py:107-127 with use_rel=True, arch=conformer, activation=swish."""
    d = cfg.enc_dim
    x = conv2d_subsampling(sd, "encoder.embed", xs)
    x = x * math.sqrt(d)  # positional_encoding.py:73
    pos = sinusoid_table(x.size(1), d, x.dtype).unsqueeze(0)  # :74 -- absolute positions 0..T'-1
    if dp is not None:  # :75 -- dropout on both, ONE dropped pos_emb for all layers
        x = dp(x, NET_ENC, GLOBAL_LAYER, ENC_POS_X, dp.r.enc_pos_dropout_rate)
        pos = dp(pos, NET_ENC, GLOBAL_LAYER, ENC_POS_EMB, dp.r.enc_pos_dropout_rate)
    mask = None
    if xs_mask is not None:
        assert tuple(xs_mask.shape) == tuple(xs.shape[:2])
        m = subsample_mask(xs_mask)
        mask = m.view(m.size(0), 1, 1, m.size(1))
    for i in range(cfg.enc_layers):
        x = conformer_layer(sd, f"encoder.enc_layers.{i}", x, pos, mask, cfg.enc_attn_heads, training, bn_out, dp, i)
    return layer_norm(sd, "encoder.after_norm", x)


def decoder(sd: SD, cfg: U2Shape, ys_in: Tensor, self_mask: Tensor, memory: Tensor,
            memory_mask: Optional[Tensor], dp=None) -> Tensor:
    """nets/transformer_decoder.py:70-93 + nets/transformer_layer.py:179-221 (ReLU FFN, pre-norm)."""
    d = cfg.dec_dim
    h = cfg.dec_attn_heads
    r = dp.r if dp is not None else DropRates()

    def dr(li, kind, rate):
        return (lambda t: dp(t, NET_DEC, li, kind, rate)) if dp is not None else _nodrop
    y = sd["decoder.embed.weight"][ys_in]
    y = y * math.sqrt(d) + sinusoid_table(y.size(1), d, y.dtype).unsqueeze(0)
    y = dr(GLOBAL_LAYER, DEC_POS, r.dec_pos_dropout_rate)(y)  # positional_encoding.py:54-55
    smask = self_mask.unsqueeze(1)
    mmask = None
    if memory_mask is not None:
        m = subsample_mask(memory_mask)
        assert tuple(m.shape) == tuple(memory.shape[:2])
        mmask = m.view(m.size(0), 1, 1, m.size(1))
    for i in range(cfg.dec_layers):
        p = f"decoder.dec_layers.{i}"
        out = r.dec_dropout_rate
        z = layer_norm(sd, p + ".self_attn_norm", y)
        y = y + dr(i, DEC_SELF_OUT, out)(attention(sd, p + ".self_attn", z, z, smask, h, dr(i, DEC_SELF_PROB, r.dec_self_attn_dropout_rate)))
        z = layer_norm(sd, p + ".src_attn_norm", y)
        y = y + dr(i, DEC_SRC_OUT, out)(attention(sd, p + ".src_attn", z, memory, mmask, h, dr(i, DEC_SRC_PROB, r.dec_src_attn_dropout_rate)))
        y = y + dr(i, DEC_FF_OUT, out)(feed_forward(sd, p + ".feed_forward", layer_norm(sd, p + ".feed_forward_norm", y), torch.relu,
                                                     dr(i, DEC_FF_INNER, r.dec_ff_dropout_rate)))
    return dense(sd, "decoder.linear_out", layer_norm(sd, "decoder.after_norm", y))


def u2_forward(sd: SD, cfg: U2Shape, xs, xlens, ys, ylens, training: bool = True, bn_out=None, dp=None):
    """models/u2.py:116-159 -> (h_attn (B,L+1,V), h_ctc (B,T',V), h_enc).  ``dp`` = Dropper (its ``training`` flag gates every
    site except the CTC head's, which the reference applies unconditionally: nets/ctc.py:29, quirk Q3)."""
    xs_mask = pad_mask(xlens, xs.size(1))
    ys_in, ys_mask = decoder_inputs(ys, ylens, cfg.vocab_size)
    h_enc = encoder(sd, cfg, xs, xs_mask, training, bn_out, dp)
    dec_mask = ys_mask.unsqueeze(1) | causal_mask(ys_mask.size(1)).unsqueeze(0)
    h_attn = decoder(sd, cfg, ys_in, dec_mask, h_enc, xs_mask, dp)
    h_in = h_enc if dp is None else dp(h_enc, NET_CTC, GLOBAL_LAYER, CTC_IN, dp.r.dropout_rate, always=True)
    h_ctc = dense(sd, "ctc.ctc_lo", h_in)
    return h_attn, h_ctc, h_enc


# --------------------------------------------------------------------------------------
# CTC alpha-beta (restates torch.nn.CTCLoss == ATen LossCTC.cpp semantics; torch 2.11.0 pin)
# --------------------------------------------------------------------------------------
_HERE = os.path.dirname(os.path.abspath(__file__))
_CLIB = None


def build_c_oracle(force: bool = False) -> str:
    """gcc -O2 oracle/ctc_oracle.c -> oracle/_build/libctc_oracle.so (plain C, no deps).  In a read-only tree whose library
    is missing or older than its source, the library goes to a private per-user cache directory under the system's temporary
    directory instead, named after a hash of the source: built once, reused by later processes."""
    out_dir = os.path.join(_HERE, "_build")
    so = os.path.join(out_dir, "libctc_oracle.so")
    src = os.path.join(_HERE, "ctc_oracle.c")
    if not force and os.path.exists(so) and os.path.getmtime(so) >= os.path.getmtime(src):
        return so
    if not os.access(out_dir if os.path.isdir(out_dir) else _HERE, os.W_OK):
        out_dir = os.path.join(tempfile.gettempdir(), f"ctc_oracle-{os.getuid()}")
        os.makedirs(out_dir, mode=0o700, exist_ok=True)
        st = os.stat(out_dir)
        if st.st_uid != os.getuid() or st.st_mode & 0o077:  # a library loaded from here must be this user's own
            raise RuntimeError(f"{out_dir} is not a private directory of this user")
        with open(src, "rb") as f:
            so = os.path.join(out_dir, f"libctc_oracle-{hashlib.sha256(f.read()).hexdigest()[:16]}.so")
        if not force and os.path.exists(so):
            return so
    os.makedirs(out_dir, exist_ok=True)
    tmp = f"{so}.{os.getpid()}.tmp"  # concurrent builders each write their own file; the rename is atomic
    subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-fopenmp", "-o", tmp, src, "-lm"])
    os.replace(tmp, so)
    return so


def _clib():
    global _CLIB
    if _CLIB is None:
        lib = ctypes.CDLL(build_c_oracle())
        lib.ctc_alpha_beta_f64.restype = ctypes.c_int
        lib.ctc_alpha_beta_f64.argtypes = [ctypes.c_void_p] * 7 + [ctypes.c_long] * 4 + [ctypes.c_int]
        _CLIB = lib
    return _CLIB


def ctc_alpha_beta_numpy(lp: np.ndarray, targets: np.ndarray, in_len: np.ndarray, tgt_len: np.ndarray,
                         blank: int = 0):
    """Pure-numpy float64 alpha-beta (small cases only).  lp (T,B,V) log-probs.

    Returns (nll (B,), dnll_dlp (T,B,V)) where dnll_dlp = -occupancy (the true partial
    derivative wrt the log-probs; rows t >= in_len[b] are 0).  Infeasible -> nll = +inf."""
    T, B, V = lp.shape
    nll = np.zeros(B)
    g = np.zeros_like(lp, dtype=np.float64)
    NEG = -np.inf

    def lse(*a):
        m = max(a)
        if m == NEG:
            return NEG
        return m + math.log(sum(math.exp(x - m) for x in a))

    for b in range(B):
        Tb, L = int(in_len[b]), int(tgt_len[b])
        ext = [blank] * (2 * L + 1)
        for k in range(L):
            ext[2 * k + 1] = int(targets[b, k])
        S = 2 * L + 1
        al = np.full((Tb, S), NEG)
        be = np.full((Tb, S), NEG)
        if Tb == 0:
            nll[b] = 0.0 if L == 0 else np.inf
            continue
        al[0, 0] = lp[0, b, blank]
        if S > 1:
            al[0, 1] = lp[0, b, ext[1]]
        for t in range(1, Tb):
            for s in range(S):
                a = [al[t - 1, s]]
                if s >= 1:
                    a.append(al[t - 1, s - 1])
                if s >= 2 and ext[s] != blank and ext[s] != ext[s - 2]:
                    a.append(al[t - 1, s - 2])
                al[t, s] = lp[t, b, ext[s]] + lse(*a)
        tot = lse(al[Tb - 1, S - 1], al[Tb - 1, S - 2]) if S > 1 else al[Tb - 1, 0]
        nll[b] = -tot
        if not np.isfinite(tot):
            g[:Tb, b, :] = np.nan
            continue
        be[Tb - 1, S - 1] = lp[Tb - 1, b, ext[S - 1]]
        if S > 1:
            be[Tb - 1, S - 2] = lp[Tb - 1, b, ext[S - 2]]
        for t in range(Tb - 2, -1, -1):
            for s in range(S):
                a = [be[t + 1, s]]
                if s + 1 < S:
                    a.append(be[t + 1, s + 1])
                if s + 2 < S and ext[s] != blank and ext[s] != ext[s + 2]:
                    a.append(be[t + 1, s + 2])
                be[t, s] = lp[t, b, ext[s]] + lse(*a)
        for t in range(Tb):
            for s in range(S):
                ab = al[t, s] + be[t, s]
                if ab > NEG:
                    g[t, b, ext[s]] -= math.exp(ab - lp[t, b, ext[s]] - tot)
    return nll, g


def ctc_alpha_beta_c(lp: np.ndarray, targets: np.ndarray, in_len: np.ndarray, tgt_len: np.ndarray):
    """Same contract as ``ctc_alpha_beta_numpy`` through oracle/ctc_oracle.c (fast)."""
    lp = np.ascontiguousarray(lp, dtype=np.float64)
    T, B, V = lp.shape
    targets = np.ascontiguousarray(targets, dtype=np.int64)
    if targets.ndim == 1:
        targets = targets.reshape(B, -1)
    in_len = np.ascontiguousarray(in_len, dtype=np.int64)
    tgt_len = np.ascontiguousarray(tgt_len, dtype=np.int64)
    nll = np.zeros(B, dtype=np.float64)
    g = np.zeros_like(lp)
    lmax = targets.shape[1]
    ws = np.zeros(1, dtype=np.float64)
    rc = _clib().ctc_alpha_beta_f64(
        lp.ctypes.data, targets.ctypes.data, in_len.ctypes.data, tgt_len.ctypes.data,
        nll.ctypes.data, g.ctypes.data, ws.ctypes.data, T, B, V, lmax, 0,
    )
    if rc != 0:
        raise RuntimeError(f"ctc_alpha_beta_f64 failed rc={rc}")
    return nll, g


class _CTCNll(torch.autograd.Function):
    @staticmethod
    def forward(ctx, lp, targets, in_len, tgt_len):
        nll, g = ctc_alpha_beta_c(lp.detach().double().numpy(), targets.numpy(), in_len.numpy(), tgt_len.numpy())
        ctx.save_for_backward(torch.from_numpy(g).to(lp.dtype))
        return torch.from_numpy(nll).to(lp.dtype)

    @staticmethod
    def backward(ctx, gout):
        (g,) = ctx.saved_tensors
        return g * gout.view(1, -1, 1), None, None, None


def ctc_nll(lp: Tensor, targets: Tensor, in_len: Tensor, tgt_len: Tensor) -> Tensor:
    """Per-utterance -log p(l|x) with autograd; lp (T,B,V) log-probs."""
    return _CTCNll.apply(lp, targets, in_len, tgt_len)


# --------------------------------------------------------------------------------------
# criterion
# --------------------------------------------------------------------------------------
def label_smoothing_kl(h_attn: Tensor, tgt: Tensor, smoothing: float) -> Tensor:
    """criterions/hybrid_ctc_attn.py:49-64 -- sum over non-ignored rows of KL(q || softmax),
    q = eps/(V-1) off-target, 1-eps on target.  Returns the SUM (caller divides by B)."""
    v = h_attn.size(-1)
    flat = h_attn.reshape(-1, v)
    t = tgt.reshape(-1)
    ign = t == -1
    t0 = t.masked_fill(ign, 0)
    q = torch.full_like(flat, smoothing / (v - 1))
    q.scatter_(1, t0.unsqueeze(1), 1.0 - smoothing)
    logp = torch.log_softmax(flat, dim=1)
    # KLDivLoss(reduction="none") = xlogy(q, q) - q * logp  (0 where q == 0)
    kl = torch.xlogy(q, q) - q * logp
    return kl.masked_fill(ign.unsqueeze(1), 0).sum()


def hybrid_loss(sd: SD, cfg: U2Shape, xs, xlens, ys, ylens, ctc_weight: float, smoothing: float,
                training: bool = True, bn_out=None, dp=None):
    """criterions/hybrid_ctc_attn.py:39-79 -> dict(loss, loss_ctc, loss_attn, h_attn, h_ctc, h_enc)."""
    h_attn, h_ctc, h_enc = u2_forward(sd, cfg, xs, xlens, ys, ylens, training, bn_out, dp)
    b = ys.size(0)
    loss_attn = label_smoothing_kl(h_attn, attention_targets(ys, ylens, cfg.vocab_size), smoothing) / b
    lp = torch.log_softmax(h_ctc.transpose(0, 1), dim=-1)
    loss_ctc = ctc_nll(lp, ys, subsampled_len(xlens), ylens).sum() / b
    loss = ctc_weight * loss_ctc + (1 - ctc_weight) * loss_attn
    return dict(loss=loss, loss_ctc=loss_ctc, loss_attn=loss_attn, h_attn=h_attn, h_ctc=h_ctc, h_enc=h_enc)


def greedy_ctc(sd: SD, cfg: U2Shape, xs: Tensor, xlens: Optional[Tensor] = None):
    """Greedy CTC decode (not in the reference; defined from nets/ctc.py:25-26 as
    argmax_v log_softmax(ctc_lo(encoder(x))) -> collapse repeats -> drop blank 0).
    xlens=None mirrors the reference's maskless inference encoder call (models/u2.py:222)."""
    mask = None if xlens is None else pad_mask(xlens, xs.size(1))
    h = encoder(sd, cfg, xs, mask, training=False)
    ids = torch.log_softmax(dense(sd, "ctc.ctc_lo", h), dim=-1).argmax(-1)
    out = []
    for b in range(ids.size(0)):
        n = ids.size(1) if xlens is None else int(subsampled_len(xlens[b]))
        seq, prev = [], -1
        for t in range(n):
            c = int(ids[b, t])
            if c != prev and c != 0:
                seq.append(c)
            prev = c
        out.append(seq)
    return out, ids


# --------------------------------------------------------------------------------------
# inference (models/u2.py:221-317): CTC prefix beam search + attention rescoring, batch 1
# --------------------------------------------------------------------------------------
def log_add(args) -> float:
    """models/u2.py:367-375 (stable log-add over a list of Python floats)."""
    if all(a == -float("inf") for a in args):
        return -float("inf")
    a_max = max(args)
    lsp = math.log(sum(math.exp(a - a_max) for a in args))
    return a_max + lsp


def prefix_beam_search_logp(ctc_probs: Tensor, beam_size: int = 10):
    """models/u2.py:226-261 on a (frames, vocab) log-probability matrix.  Returns [(prefix tuple, score)] best first.
    Kept structurally identical to the reference: per frame torch.topk prune, dict in insertion order, Python floats,
    stable sort on log_add(pb, pnb) descending."""
    from collections import defaultdict
    cur_hyps = [(tuple(), (0.0, -float("inf")))]
    for logp in ctc_probs:
        next_hyps = defaultdict(lambda: (-float("inf"), -float("inf")))
        _, index_topk = torch.topk(logp, beam_size)
        for s in index_topk:
            s = s.item()
            ps = logp[s].item()
            for prefix, (pb, pnb) in cur_hyps:
                last = prefix[-1] if len(prefix) > 0 else None
                if s == 0:  # blank
                    n_pb, n_pnb = next_hyps[prefix]
                    n_pb = log_add([n_pb, pb + ps, pnb + ps])
                    next_hyps[prefix] = (n_pb, n_pnb)
                elif s == last:
                    n_pb, n_pnb = next_hyps[prefix]
                    n_pnb = log_add([n_pnb, pnb + ps])
                    next_hyps[prefix] = (n_pb, n_pnb)
                    n_prefix = prefix + (s,)
                    n_pb, n_pnb = next_hyps[n_prefix]
                    n_pnb = log_add([n_pnb, pb + ps])
                    next_hyps[n_prefix] = (n_pb, n_pnb)
                else:
                    n_prefix = prefix + (s,)
                    n_pb, n_pnb = next_hyps[n_prefix]
                    n_pnb = log_add([n_pnb, pb + ps, pnb + ps])
                    next_hyps[n_prefix] = (n_pb, n_pnb)
        next_hyps = sorted(next_hyps.items(), key=lambda x: log_add(list(x[1])), reverse=True)
        cur_hyps = next_hyps[:beam_size]
    return [(y[0], log_add([y[1][0], y[1][1]])) for y in cur_hyps]


def rescore_scores(attn_score: Tensor, hyps, eos: int, ctc_weight: float = 0.5):
    """models/u2.py:303-315: per hypothesis sum_j logp[j, y_j] + logp[len, eos] + 0.5 * ctc score, accumulated left to right
    in the tensor dtype exactly like the reference's `score += attn_score[i][j][w]` (a 0-dim tensor after the first add).
    Returns (best index, [scores])."""
    best_score, best_index, scores = -float("inf"), 0, []
    for i, hyp in enumerate(hyps):
        score = 0.0
        for j, w in enumerate(hyp[0]):
            score += attn_score[i][j][w]
        score += attn_score[i][len(hyp[0])][eos]
        score += hyp[1] * ctc_weight
        scores.append(float(score))
        if score > best_score:
            best_score = score
            best_index = i
    return best_index, scores


def attention_rescore(sd: SD, cfg: U2Shape, x: Tensor, beam_size: int = 10):
    """models/u2.py:269-317 for one utterance x (1, T, F): maskless encoder (eval-mode BatchNorm), CTC prefix beam search,
    decoder pass over the padded n-best ([sos | hyp, pad -> eos], mask = padding | causal, memory unmasked), rescoring.
    Deviation (SURVEY 8c-i): the reference passes Python lists to `_preprocess` and crashes at HEAD (quirk Q13); the lengths are
    tensors here.  Returns dict(best, hyps, scores, ctc_logp)."""
    h = encoder(sd, cfg, x, None, training=False)
    ctc_logp = torch.log_softmax(dense(sd, "ctc.ctc_lo", h), dim=-1).squeeze(0)
    hyps = prefix_beam_search_logp(ctc_logp, beam_size)
    ylens = torch.tensor([len(hy[0]) for hy in hyps], dtype=torch.long)
    lmax = int(ylens.max())
    ys = torch.full((len(hyps), max(lmax, 0)), -1, dtype=torch.long)
    for i, hy in enumerate(hyps):
        if len(hy[0]):
            ys[i, : len(hy[0])] = torch.tensor(hy[0], dtype=torch.long)
    ys_in, ys_mask = decoder_inputs(ys, ylens, cfg.vocab_size)
    dec_mask = ys_mask.unsqueeze(1) | causal_mask(ys_mask.size(1)).unsqueeze(0)
    h_attn = decoder(sd, cfg, ys_in, dec_mask, h.repeat(len(hyps), 1, 1), None)
    attn_score = torch.log_softmax(h_attn, dim=-1)
    best, scores = rescore_scores(attn_score, hyps, cfg.vocab_size - 1)
    return dict(best=list(hyps[best][0]), hyps=[(list(p), s) for p, s in hyps], scores=scores, ctc_logp=ctc_logp)
