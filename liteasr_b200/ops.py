"""Thin tensor-level wrappers over the C ABI (one Python function per ``lasr_*`` entry point).

All wrappers take CUDA tensors, pass raw device pointers + the current torch stream, and raise on any
non-zero return code.  Nothing here computes on the host and nothing falls back to torch ops.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import ACT_MUL, ACT_NONE, ACT_RELU, ACT_SWISH, BF16, F32  # noqa: F401

_P = C.c_void_p


def _ptr(t: Optional[torch.Tensor]):
    return _P(t.data_ptr()) if t is not None else _P(0)


def _stream():
    return _P(torch.cuda.current_stream().cuda_stream)


def dtype_code(t: torch.Tensor) -> int:
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.bfloat16:
        return BF16
    raise TypeError(f"unsupported dtype {t.dtype}")


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("liteasr_b200 ops need CUDA tensors (there is no CPU fallback)")


def gemm(a: torch.Tensor, b: torch.Tensor, c: torch.Tensor, m: int, n: int, k: int, *, lda: int, ldb: int, ldc: int,
         ta: bool = False, tb: bool = False, bias: Optional[torch.Tensor] = None, res: Optional[torch.Tensor] = None,
         ldres: int = 0, aux: Optional[torch.Tensor] = None, alpha: float = 1.0, act: int = ACT_NONE,
         accumulate: bool = False, split_k: int = 1, batch: Tuple[int, int] = (1, 1), sa: Tuple[int, int] = (0, 0),
         sb: Tuple[int, int] = (0, 0), sc: Tuple[int, int] = (0, 0), dact: Optional[torch.Tensor] = None,
         colsum: Optional[torch.Tensor] = None, cs: Tuple[int, int] = (0, 0), n_store: int = 0,
         drop=None, drop_mark_aux: bool = False, aux_deriv: bool = False) -> None:
    """C[b1,b2] = alpha * act(A.B^T + bias) (+ res); see include/lasr.h ``lasr_gemm``.  ``drop`` = ``Drop`` (dropout on the
    output before the residual add) or None."""
    _require_cuda(a, b, c, bias, res, aux, dact, colsum)
    if a.dtype != b.dtype:
        raise TypeError("gemm operands must share a dtype")
    g = _lib.GemmArgs()
    g.a, g.b, g.c = a.data_ptr(), b.data_ptr(), c.data_ptr()
    g.bias = bias.data_ptr() if bias is not None else None
    g.res = res.data_ptr() if res is not None else None
    g.aux = aux.data_ptr() if aux is not None else None
    g.m, g.n, g.k = m, n, k
    g.ab_dtype, g.c_dtype = dtype_code(a), dtype_code(c)
    g.trans_a, g.trans_b = int(ta), int(tb)
    g.lda, g.ldb, g.ldc, g.ldres = lda, ldb, ldc, (ldres if res is not None else 0)
    g.batch1, g.batch2 = batch
    g.sa1, g.sa2 = sa
    g.sb1, g.sb2 = sb
    g.sc1, g.sc2 = sc
    g.alpha, g.act, g.accumulate, g.split_k = alpha, act, int(accumulate), split_k
    g.dact = dact.data_ptr() if dact is not None else None
    g.lddact = dact.stride(0) if dact is not None else 0
    g.colsum = colsum.data_ptr() if colsum is not None else None
    g.cs1, g.cs2 = cs
    g.n_store = n_store
    if drop is not None and drop.thr:
        g.drop_state, g.drop_site, g.drop_thr, g.drop_scale = drop.state.data_ptr(), drop.site, drop.thr, drop.scale
        g.drop_mark_aux = int(drop_mark_aux)
    g.aux_deriv = int(aux_deriv)
    if dact is not None and (dact.dtype != a.dtype or dact.dim() != 2 or dact.stride(1) != 1):
        raise TypeError("dact must be a 2-D row-major tensor of the operand dtype")
    if colsum is not None and colsum.dtype != torch.float32:
        raise TypeError("colsum must be fp32")
    if bias is not None and bias.dtype != torch.float32:
        raise TypeError("bias must be fp32")
    if res is not None and res.dtype != torch.float32:
        raise TypeError("res must be fp32")
    if aux is not None and aux.dtype != c.dtype:
        raise TypeError("aux must have C's dtype")
    _lib.check(_lib.lib().lasr_gemm(C.byref(g), _stream()), "gemm")


def linear(x: torch.Tensor, w: torch.Tensor, out: torch.Tensor, *, bias=None, res=None, aux=None, alpha=1.0,
           act=ACT_NONE) -> torch.Tensor:
    """out (M,N) = alpha * act(x (M,K) @ w (N,K)^T + bias) (+ res); rows may be strided (stride(0))."""
    m, k = x.shape
    n = w.shape[0]
    gemm(x, w, out, m, n, k, lda=x.stride(0), ldb=w.stride(0), ldc=out.stride(0), bias=bias, res=res,
         ldres=(res.stride(0) if res is not None else 0), aux=aux, alpha=alpha, act=act)
    return out


def wgrad2_supported(m: int, n: int) -> bool:
    return bool(_lib.lib().lasr_wgrad2_supported(C.c_int(m), C.c_int(n)))


def wgrad2(dy, x, gw, alpha: float = 1.0, split_k: int = 1) -> None:
    """gw (N_out, K_in) fp32 += alpha * dy^T x on CTA pairs (include/lasr.h ``lasr_wgrad2``); dy (rows, N_out), x (rows, K_in) bf16."""
    _require_cuda(dy, x, gw)
    if dy.dtype != torch.bfloat16 or x.dtype != torch.bfloat16 or gw.dtype != torch.float32:
        raise TypeError("wgrad2 takes bf16 operands and an fp32 gradient")
    rows, m = dy.shape
    n = x.shape[1]
    assert x.shape[0] == rows and gw.shape == (m, n) and dy.stride(1) == 1 and x.stride(1) == 1 and gw.stride(1) == 1
    _lib.check(_lib.lib().lasr_wgrad2(_ptr(dy), C.c_int64(dy.stride(0)), _ptr(x), C.c_int64(x.stride(0)), _ptr(gw), C.c_int64(gw.stride(0)),
                                      C.c_float(alpha), C.c_int(m), C.c_int(n), C.c_int(rows), C.c_int(split_k), _stream()), "wgrad2")


def ffn_bwd_supported(d: int, f: int) -> bool:
    return bool(_lib.lib().lasr_ffn_bwd_supported(C.c_int(d), C.c_int(f)))


def ffn_bwd(dy, g, w2, w1, dh, dln, colsum=None, alpha: float = 1.0) -> None:
    """dh = alpha * (dy @ w2) * g ; colsum += sum_rows dh ; dln = dh @ w1  (one fused tcgen05 kernel, include/lasr.h)."""
    _require_cuda(dy, g, w2, w1, dh, dln, colsum)
    for t in (dy, g, w2, w1, dh, dln):
        if t.dtype != torch.bfloat16 or t.dim() != 2 or t.stride(1) != 1:
            raise TypeError("ffn_bwd takes 2-D row-major bf16 tensors")
    m, d = dy.shape
    f = g.shape[1]
    assert g.shape == (m, f) and w2.shape == (d, f) and w1.shape == (f, d) and dh.shape == (m, f) and dln.shape == (m, d)
    if colsum is not None:
        assert colsum.dtype == torch.float32 and colsum.numel() == f
    _lib.check(_lib.lib().lasr_ffn_bwd(_ptr(dy), C.c_int64(dy.stride(0)), _ptr(g), C.c_int64(g.stride(0)), _ptr(w2), C.c_int64(w2.stride(0)),
                                       _ptr(w1), C.c_int64(w1.stride(0)), _ptr(dh), C.c_int64(dh.stride(0)), _ptr(dln),
                                       C.c_int64(dln.stride(0)), _ptr(colsum), C.c_float(alpha), C.c_int(m), C.c_int(d), C.c_int(f),
                                       _stream()), "ffn_bwd")


def ffn_fwd_supported(d: int, f: int) -> bool:
    return bool(_lib.lib().lasr_ffn_fwd_supported(C.c_int(d), C.c_int(f)))


def ffn_fwd(ln, w1, b1, w2, b2, res, a, g, out, alpha: float = 1.0, drop_in=None, drop_out=None) -> None:
    """a = drop_in(swish(ln @ w1^T + b1)), g = swish'(.) (0 where dropped), out = res + drop_out(alpha * (a @ w2^T + b2)):
    one fused tcgen05 kernel (include/lasr.h ``lasr_ffn_fwd``).  ``drop_in`` / ``drop_out``: ``Drop`` of the two sites (same pass)."""
    _require_cuda(ln, w1, b1, w2, b2, res, a, g, out)
    for t in (ln, w1, w2, a, g):
        if t.dtype != torch.bfloat16 or t.dim() != 2 or t.stride(1) != 1:
            raise TypeError("ffn_fwd takes 2-D row-major bf16 operands")
    for t in (b1, b2, res, out):
        if t.dtype != torch.float32:
            raise TypeError("ffn_fwd: biases, residual and output are fp32")
    m, d = ln.shape
    f = w1.shape[0]
    assert w1.shape == (f, d) and w2.shape == (d, f) and a.shape == (m, f) and g.shape == (m, f) and res.shape == (m, d) and out.shape == (m, d)
    assert b1.numel() == f and b2.numel() == d and res.stride(1) == 1 and out.stride(1) == 1
    di = drop_in if (drop_in is not None and drop_in.thr) else None
    do = drop_out if (drop_out is not None and drop_out.thr) else None
    state = (di or do).state if (di or do) is not None else None
    if di is not None and do is not None:
        assert di.state.data_ptr() == do.state.data_ptr(), "the two dropout sites of a block share the pass's RNG snapshot"
    _lib.check(_lib.lib().lasr_ffn_fwd(_ptr(ln), C.c_int64(ln.stride(0)), _ptr(w1), C.c_int64(w1.stride(0)), _ptr(b1), _ptr(w2),
                                       C.c_int64(w2.stride(0)), _ptr(b2), _ptr(res), C.c_int64(res.stride(0)), _ptr(a), C.c_int64(a.stride(0)),
                                       _ptr(g), C.c_int64(g.stride(0)), _ptr(out), C.c_int64(out.stride(0)), C.c_float(alpha), C.c_int(m),
                                       C.c_int(d), C.c_int(f), _ptr(state), C.c_uint32(di.site if di else 0), C.c_uint32(di.thr if di else 0),
                                       C.c_float(di.scale if di else 1.0), C.c_uint32(do.site if do else 0), C.c_uint32(do.thr if do else 0),
                                       C.c_float(do.scale if do else 1.0), _stream()), "ffn_fwd")


def ctc_workspace_bytes(T: int, B: int, lmax: int) -> int:
    return int(_lib.lib().lasr_ctc_workspace_bytes(C.c_int(T), C.c_int(B), C.c_int(lmax)))


def ctc_fwdbwd(logits: torch.Tensor, targets: torch.Tensor, in_len: torch.Tensor, tgt_len: torch.Tensor, *,
               time_major: bool, grad: Optional[torch.Tensor] = None, grad_scale: float = 1.0,
               upstream: Optional[torch.Tensor] = None, blank: int = 0, vocab: Optional[int] = None,
               workspace: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Fused CTC fwd+bwd.  logits (T,B,V) if time_major else (B,T,V) (last dim contiguous; may be a
    narrowed view of a padded buffer).  Returns (nll (B,) fp32, grad wrt logits with logits' layout)."""
    _require_cuda(logits, targets, in_len, tgt_len, grad, upstream, workspace)
    assert logits.dim() == 3 and logits.stride(2) == 1
    if time_major:
        T, B, V = logits.shape
        st, sb = logits.stride(0), logits.stride(1)
    else:
        B, T, V = logits.shape
        sb, st = logits.stride(0), logits.stride(1)
    if vocab is not None:
        V = vocab
    if grad is None:
        grad = torch.empty_like(logits)
    gst, gsb = (grad.stride(0), grad.stride(1)) if time_major else (grad.stride(1), grad.stride(0))
    assert grad.stride(2) == 1 and grad.dtype == logits.dtype
    assert targets.dtype == torch.int64 and in_len.dtype == torch.int64 and tgt_len.dtype == torch.int64
    targets = targets.contiguous()
    lmax = max(1, targets.shape[1])
    if targets.shape[1] == 0:
        targets = torch.zeros(B, 1, dtype=torch.int64, device=logits.device)
    nbytes = ctc_workspace_bytes(T, B, lmax)
    if workspace is None or workspace.numel() * workspace.element_size() < nbytes:
        workspace = torch.empty(nbytes, dtype=torch.uint8, device=logits.device)
    nll = torch.empty(B, dtype=torch.float32, device=logits.device)
    rc = _lib.lib().lasr_ctc_fwdbwd(
        _ptr(logits), C.c_int(dtype_code(logits)), C.c_int64(st), C.c_int64(sb), _ptr(targets), _ptr(in_len),
        _ptr(tgt_len), C.c_int(T), C.c_int(B), C.c_int(V), C.c_int(lmax), C.c_int(blank), C.c_float(grad_scale),
        _ptr(upstream), _ptr(nll), _ptr(grad), C.c_int64(gst), C.c_int64(gsb), _ptr(workspace),
        C.c_size_t(workspace.numel() * workspace.element_size()), _stream())
    _lib.check(rc, "ctc_fwdbwd")
    return nll, grad


# ----------------------------------------------------------------------------------------------
# remaining entry points (see include/lasr.h for the contracts)
# ----------------------------------------------------------------------------------------------
def _i(v):
    return C.c_int(int(v))


def _l(v):
    return C.c_int64(int(v))


def _f(v):
    return C.c_float(float(v))


def zero_(t: torch.Tensor) -> torch.Tensor:
    _require_cuda(t)
    assert t.is_contiguous()
    _lib.check(_lib.lib().lasr_zero(_ptr(t), C.c_size_t(t.numel() * t.element_size()), _stream()), "zero")
    return t


def cast_bf16(src: torch.Tensor, dst: torch.Tensor) -> torch.Tensor:
    _require_cuda(src, dst)
    assert src.dtype == torch.float32 and dst.dtype == torch.bfloat16 and src.is_contiguous() and dst.is_contiguous()
    _lib.check(_lib.lib().lasr_cast_f32_bf16(_ptr(src), _ptr(dst), _l(src.numel()), _stream()), "cast_f32_bf16")
    return dst


def permute4d(src, dst, n, src_strides, dst_strides, accumulate=False):
    _require_cuda(src, dst)
    A = C.c_int64 * 4
    _lib.check(_lib.lib().lasr_permute4d(_ptr(src), _i(dtype_code(src)), _ptr(dst), _i(dtype_code(dst)), A(*n), A(*src_strides),
                                         A(*dst_strides), _i(accumulate), _stream()), "permute4d")


def layernorm_fwd(x, gamma, beta, y, mean=None, rstd=None, eps=1e-12):
    _require_cuda(x, gamma, beta, y)
    rows, d = x.shape
    _lib.check(_lib.lib().lasr_layernorm_fwd(_ptr(x), _l(x.stride(0)), _ptr(gamma), _ptr(beta), _ptr(y), _i(dtype_code(y)),
                                             _l(y.stride(0)), _ptr(mean), _ptr(rstd), _i(rows), _i(d), _f(eps), _stream()),
               "layernorm_fwd")
    return y


def layernorm_bwd(dy, x, mean, rstd, gamma, dx, dgamma, dbeta, accumulate: bool, dx_lo=None, colsum=None, colsum_scale=1.0,
                  drop=None):
    """dx (+)= LN'(dy); optional fused outputs: dx_lo (bf16 or fp32 copy of the final dx), colsum += colsum_scale * sum_rows dx.
    ``drop``: the dropout site of the block that consumes dx_lo / colsum (mask applied to those two outputs only)."""
    _require_cuda(dy, x, dx, dx_lo, colsum)
    rows, d = x.shape
    if drop is not None and not drop.thr:
        drop = None
    _lib.check(_lib.lib().lasr_layernorm_bwd_drop(
        _ptr(dy), _i(dtype_code(dy)), _l(dy.stride(0)), _ptr(x), _l(x.stride(0)), _ptr(mean), _ptr(rstd), _ptr(gamma), _ptr(dx),
        _l(dx.stride(0)), _i(accumulate), _ptr(dgamma), _ptr(dbeta), _i(rows), _i(d), _ptr(dx_lo),
        _i(dtype_code(dx_lo) if dx_lo is not None else BF16), _l(dx_lo.stride(0) if dx_lo is not None else 0), _ptr(colsum),
        _f(colsum_scale), _ptr(drop.state if drop is not None else None), C.c_uint32(drop.site if drop is not None else 0),
        C.c_uint32(drop.thr if drop is not None else 0), _f(drop.scale if drop is not None else 1.0), _stream()), "layernorm_bwd")


DROP_P_MAX = 0.96875  # thr = round(p * 32768) <= 0x7c00


class Drop:
    """One dropout site of one step: device RNG state {seed, step}, site id, 15-bit threshold and the 1/(1-p) scale
    (include/lasr.h, "Dropout"; liteasr_b200/dropout.py builds these)."""
    __slots__ = ("state", "site", "thr", "scale")

    def __init__(self, state: torch.Tensor, site: int, p: float):
        self.state, self.site = state, int(site)
        if not 0.0 <= float(p) <= DROP_P_MAX:
            raise ValueError(f"dropout rate {p!r} outside [0, {DROP_P_MAX}] (15-bit lanes compared as fp16 patterns: csrc/philox.cuh)")
        self.thr = int(max(0, round(float(p) * 32768.0)))
        self.scale = 32768.0 / (32768.0 - self.thr)


def rng_advance(state: torch.Tensor) -> None:
    """state[1] += 1 on the device (inside the captured step: every replay draws fresh masks)."""
    _require_cuda(state)
    assert state.dtype == torch.int64 and state.numel() >= 2
    _lib.check(_lib.lib().lasr_rng_advance(_ptr(state), _stream()), "rng_advance")


def philox_raw(ctr_key: torch.Tensor, rounds: int) -> torch.Tensor:
    """Known-answer hook: philox4x32 with ``rounds`` (10 or 7) rounds of counter ctr_key[0:4], key ctr_key[4:6] (int32 bit patterns)."""
    _require_cuda(ctr_key)
    assert ctr_key.dtype == torch.int32 and ctr_key.numel() == 6 and ctr_key.is_contiguous()
    out = torch.empty(4, dtype=torch.int32, device=ctr_key.device)
    _lib.check(_lib.lib().lasr_philox_raw(_ptr(ctr_key), _ptr(out), _i(rounds), _stream()), "philox_raw")
    return out


def dropout(x: torch.Tensor, y: torch.Tensor, drop: Drop) -> torch.Tensor:
    """y = keep * scale * x over the logical (rows, cols) = (numel / last, last) tensor; x, y 2-D views (or contiguous N-D)."""
    _require_cuda(x, y)
    if x.dim() != 2:
        assert x.is_contiguous() and y.is_contiguous()
        x, y2 = x.view(-1, x.shape[-1]), y.view(-1, y.shape[-1])
    else:
        y2 = y
    assert x.shape == y2.shape and x.stride(1) == 1 and y2.stride(1) == 1
    rows, cols = x.shape
    _lib.check(_lib.lib().lasr_dropout(_ptr(x), _i(dtype_code(x)), _l(x.stride(0)), _ptr(y2), _i(dtype_code(y2)), _l(y2.stride(0)),
                                       _l(rows), _i(cols), _ptr(drop.state), C.c_uint32(drop.site), C.c_uint32(drop.thr),
                                       _f(drop.scale), _stream()), "dropout")
    return y


def act_bwd(da, saved, dh, dbias, act, scale=1.0):
    """dh = scale * da * act'(saved); dbias += colsum(dh).  2-D (rows, cols) views; dh/saved/dbias optional."""
    _require_cuda(da, saved, dh, dbias)
    rows, cols = da.shape
    _lib.check(_lib.lib().lasr_act_bwd(_ptr(da), _l(da.stride(0)), _ptr(saved), _l(saved.stride(0) if saved is not None else 0),
                                       _ptr(dh), _l(dh.stride(0) if dh is not None else 0), _ptr(dbias), _i(rows), _i(cols),
                                       _i(act), _f(scale), _i(dtype_code(da)), _stream()), "act_bwd")


def pos_bias_fwd(q, u, v, qu, qv):
    rows, d = q.shape
    _lib.check(_lib.lib().lasr_pos_bias_fwd(_ptr(q), _l(q.stride(0)), _ptr(u), _ptr(v), _ptr(qu), _ptr(qv), _l(qu.stride(0)),
                                            _i(rows), _i(d), _i(dtype_code(q)), _stream()), "pos_bias_fwd")


def pos_bias_bwd(dqu, dqv, dq, du, dv, dqbias=None):
    rows, d = dqu.shape
    _lib.check(_lib.lib().lasr_pos_bias_bwd(_ptr(dqu), _ptr(dqv), _l(dqu.stride(0)), _ptr(dq), _l(dq.stride(0)), _ptr(du), _ptr(dv),
                                            _ptr(dqbias), _i(rows), _i(d), _i(dtype_code(dqu)), _stream()), "pos_bias_bwd")


def embed_fwd(tokens, emb, pe, out, scale):
    B, L = tokens.shape
    _lib.check(_lib.lib().lasr_embed_fwd(_ptr(tokens), _i(L), _ptr(emb), _ptr(pe), _ptr(out), _i(B), _i(emb.shape[1]), _f(scale),
                                         _stream()), "embed_fwd")


def embed_bwd(tokens, dout, demb, scale):
    _lib.check(_lib.lib().lasr_embed_bwd(_ptr(tokens), _ptr(dout), _ptr(demb), _l(tokens.numel()), _i(demb.shape[1]), _f(scale),
                                         _stream()), "embed_bwd")


def scale_by_scalar(x, scalar):
    assert x.is_contiguous() and scalar.dtype == torch.float32
    _lib.check(_lib.lib().lasr_scale_by_scalar(_ptr(x), _i(dtype_code(x)), _l(x.numel()), _ptr(scalar), _stream()), "scale_by_scalar")


def glu_dwconv_fwd(y2, w, bias, z, partial, B, T, d):
    _lib.check(_lib.lib().lasr_glu_dwconv_fwd(_ptr(y2), _i(dtype_code(y2)), _l(y2.stride(0)), _ptr(w), _ptr(bias), _ptr(z),
                                              _ptr(partial), _i(B), _i(T), _i(d), _stream()), "glu_dwconv_fwd")


def glu_dwconv_fwd_lens(y2, w, bias, z, partial, B, T, d, lens):
    """glu_dwconv_fwd with GLU rows t >= lens[b] (int64 (B,), sub-sampled frames) read as zero: per-utterance inference."""
    _require_cuda(y2, lens)
    assert lens.dtype == torch.int64 and lens.numel() == B and lens.is_contiguous()
    _lib.check(_lib.lib().lasr_glu_dwconv_fwd_lens(_ptr(y2), _i(dtype_code(y2)), _l(y2.stride(0)), _ptr(w), _ptr(bias), _ptr(z),
                                                   _ptr(partial), _i(B), _i(T), _i(d), _ptr(lens), _stream()), "glu_dwconv_fwd_lens")


def bn_finalize(partial, nblk, d, count, mean, rstd, running_mean, running_var, nbt, training, eps=1e-5, momentum=0.1):
    _lib.check(_lib.lib().lasr_bn_finalize(_ptr(partial), _i(nblk), _i(d), _l(count), _f(eps), _f(momentum), _ptr(mean), _ptr(rstd),
                                           _ptr(running_mean), _ptr(running_var), _ptr(nbt), _i(training), _stream()), "bn_finalize")


def bn_swish_fwd(z, mean, rstd, gamma, beta, a):
    rows, d = z.shape
    _lib.check(_lib.lib().lasr_bn_swish_fwd(_ptr(z), _ptr(mean), _ptr(rstd), _ptr(gamma), _ptr(beta), _ptr(a), _i(dtype_code(a)),
                                            _l(rows), _i(d), _stream()), "bn_swish_fwd")


def bn_swish_bwd_stats(da, z, mean, rstd, gamma, beta, partial, sums, dgamma, dbeta):
    rows, d = z.shape
    _lib.check(_lib.lib().lasr_bn_swish_bwd_stats(_ptr(da), _i(dtype_code(da)), _ptr(z), _ptr(mean), _ptr(rstd), _ptr(gamma), _ptr(beta),
                                                  _ptr(partial), _ptr(sums), _ptr(dgamma), _ptr(dbeta), _l(rows), _i(d), _stream()),
               "bn_swish_bwd_stats")


def dwconv_glu_bwd(da, z, y2, mean, rstd, gamma, beta, sums, w, dy2, dw, dbias, B, T, d, colsum=None, wpartial=None):
    _lib.check(_lib.lib().lasr_dwconv_glu_bwd(_ptr(da), _ptr(z), _ptr(y2), _i(dtype_code(y2)), _l(y2.stride(0)), _ptr(mean), _ptr(rstd),
                                              _ptr(gamma), _ptr(beta), _ptr(sums), _ptr(w), _ptr(dy2), _l(dy2.stride(0)), _ptr(dw),
                                              _ptr(dbias), _ptr(colsum), _ptr(wpartial), _i(B), _i(T), _i(d), _stream()), "dwconv_glu_bwd")


def conv1_fwd(x, w, bias, h1):
    B, T, F = x.shape
    _lib.check(_lib.lib().lasr_conv1_fwd(_ptr(x), _ptr(w), _ptr(bias), _ptr(h1), _i(dtype_code(h1)), _i(B), _i(T), _i(F),
                                         _i(h1.shape[-1]), _stream()), "conv1_fwd")


def conv1_bwd(x, dh1, dw, dbias):
    B, T, F = x.shape
    _lib.check(_lib.lib().lasr_conv1_bwd(_ptr(x), _ptr(dh1), _i(dtype_code(dh1)), _ptr(dw), _ptr(dbias), _i(B), _i(T), _i(F),
                                         _i(dh1.shape[-1]), _stream()), "conv1_bwd")


def im2col_s2(h1, col):
    B, T1, F1, d = h1.shape
    _lib.check(_lib.lib().lasr_im2col_s2(_ptr(h1), _ptr(col), _i(dtype_code(h1)), _i(B), _i(T1), _i(F1), _i(d), _stream()), "im2col")


def col2im_s2_relu(dcol, h1, dh1):
    B, T1, F1, d = h1.shape
    _lib.check(_lib.lib().lasr_col2im_s2_relu(_ptr(dcol), _ptr(h1), _ptr(dh1), _i(dtype_code(h1)), _i(B), _i(T1), _i(F1), _i(d),
                                              _stream()), "col2im")


def plane_dims(T: int, F: int):
    """(T1, F1, U, V, T2, F2) of the parity-plane sub-sampling front end (include/lasr.h)."""
    T1, F1 = (T - 3) // 2 + 1, (F - 3) // 2 + 1
    return T1, F1, (T1 + 1) // 2, (F1 + 1) // 2, (T1 - 3) // 2 + 1, (F1 - 3) // 2 + 1


def planes_supported(d: int, T: int, F: int) -> bool:
    return d % 64 == 0 and 64 <= d <= 1024 and 256 % (d // 4) == 0 and T >= 7 and F >= 7


def conv1_fwd_planes(x, w, bias, h1p):
    B, T, F = x.shape
    _require_cuda(x, w, bias, h1p)
    _lib.check(_lib.lib().lasr_conv1_fwd_planes(_ptr(x), _ptr(w), _ptr(bias), _ptr(h1p), _i(B), _i(T), _i(F), _i(h1p.shape[-1]), _stream()),
               "conv1_fwd_planes")


def conv1_bwd_planes(x, dh1p, dw, dbias):
    B, T, F = x.shape
    _require_cuda(x, dh1p, dw, dbias)
    _lib.check(_lib.lib().lasr_conv1_bwd_planes(_ptr(x), _ptr(dh1p), _ptr(dw), _ptr(dbias), _i(B), _i(T), _i(F), _i(dh1p.shape[-1]),
                                                _stream()), "conv1_bwd_planes")


def conv2_fwd(h1p, w2k, bias, h2p, B, T, F):
    _require_cuda(h1p, w2k, bias, h2p)
    assert h1p.dtype == torch.bfloat16 and w2k.dtype == torch.bfloat16 and h2p.dtype == torch.bfloat16 and bias.dtype == torch.float32
    _lib.check(_lib.lib().lasr_conv2_fwd(_ptr(h1p), _ptr(w2k), _ptr(bias), _ptr(h2p), _i(B), _i(T), _i(F), _i(h1p.shape[-1]), _stream()),
               "conv2_fwd")


def conv2_dgrad(dy2p, w2k, h1p, dh1p, B, T, F):
    _require_cuda(dy2p, w2k, h1p, dh1p)
    assert dy2p.dtype == torch.bfloat16 and dh1p.dtype == torch.bfloat16
    _lib.check(_lib.lib().lasr_conv2_dgrad(_ptr(dy2p), _ptr(w2k), _ptr(h1p), _ptr(dh1p), _i(B), _i(T), _i(F), _i(h1p.shape[-1]), _stream()),
               "conv2_dgrad")


def conv2_wgrad(dy2p, h1p, dw2k, B, T, F):
    _require_cuda(dy2p, h1p, dw2k)
    assert dy2p.dtype == torch.bfloat16 and dw2k.dtype == torch.float32
    _lib.check(_lib.lib().lasr_conv2_wgrad(_ptr(dy2p), _ptr(h1p), _ptr(dw2k), _i(B), _i(T), _i(F), _i(h1p.shape[-1]), _stream()),
               "conv2_wgrad")


def attn_softmax_fwd(ac, bd, probs, lens, mask_mode, causal, scale, Tk):
    B, H, Tq, ld = ac.shape
    assert bd is None or bd.dtype == ac.dtype
    _lib.check(_lib.lib().lasr_attn_softmax_fwd(_ptr(ac), _ptr(bd), _i(dtype_code(ac)), _ptr(probs), _i(dtype_code(probs)), _ptr(lens), _i(mask_mode),
                                                _i(causal), _f(scale), _i(B), _i(H), _i(Tq), _i(Tk), _i(ld), _stream()),
               "attn_softmax_fwd")


def rel_attn_fwd_supported(T: int, dk: int) -> bool:
    return bool(_lib.lib().lasr_rel_attn_fwd_supported(_i(T), _i(dk)))


def rel_attn_fwd(qu, qv, k, v, pos, probs, o, lens, mask_mode, scale, B, H, T, dk):
    """Fused rel-pos attention forward (bf16): probs (B,H,T,ld) and o (B*T, H*dk) from qu/qv/k/v (B*T, H*dk views) and pos (T, H*dk)."""
    _require_cuda(qu, qv, k, v, pos, probs, o, lens)
    for t in (qu, qv, k, v, pos, probs, o):
        if t.dtype != torch.bfloat16:
            raise TypeError("rel_attn_fwd takes bf16 tensors")
    assert qu.stride(0) == qv.stride(0) and k.stride(0) == v.stride(0) and probs.is_contiguous()
    _lib.check(_lib.lib().lasr_rel_attn_fwd(_ptr(qu), _ptr(qv), _l(qu.stride(0)), _ptr(k), _ptr(v), _l(k.stride(0)), _ptr(pos), _l(pos.stride(0)),
                                            _ptr(probs), _i(probs.shape[-1]), _ptr(o), _l(o.stride(0)), _ptr(lens), _i(mask_mode), _f(scale),
                                            _i(B), _i(H), _i(T), _i(dk), _stream()), "rel_attn_fwd")


def attn_bwd_pair_supported(Tk: int, dk: int) -> bool:
    return bool(_lib.lib().lasr_attn_bwd_pair_supported(_i(Tk), _i(dk)))


def attn_bwd_pair(x, r, l, dl, dr, B, H, Tq, Tk, dk, r_batched=True, reduce_b=False, colsum=None):
    """dl = X . r and dr = X^T . l per (utterance, head) with X (B,H,Tq,ld) read once (include/lasr.h ``lasr_attn_bwd_pair``)."""
    _require_cuda(x, r, l, dl, dr, colsum)
    for t in (x, r, l, dl):
        if t.dtype != torch.bfloat16:
            raise TypeError("attn_bwd_pair takes bf16 operands")
    if dr.dtype != (torch.float32 if reduce_b else torch.bfloat16):
        raise TypeError("attn_bwd_pair: dr is fp32 with reduce_b, bf16 otherwise")
    assert x.is_contiguous() and x.shape[:3] == (B, H, Tq) and r.stride(1) == 1 and l.stride(1) == 1 and dl.stride(1) == 1 and dr.stride(1) == 1
    _lib.check(_lib.lib().lasr_attn_bwd_pair(_ptr(x), _l(x.shape[-1]), _ptr(r), _l(r.stride(0)), _i(1 if r_batched else 0), _ptr(l), _l(l.stride(0)),
                                             _ptr(dl), _l(dl.stride(0)), _ptr(dr), _l(dr.stride(0)), _i(1 if reduce_b else 0), _ptr(colsum),
                                             _i(B), _i(H), _i(Tq), _i(Tk), _i(dk), _stream()), "attn_bwd_pair")


def attn_softmax_bwd(probs, dprobs, dsc, dbd, scale, Tk):
    B, H, Tq, ld = probs.shape
    _lib.check(_lib.lib().lasr_attn_softmax_bwd(_ptr(probs), _ptr(dprobs), _i(dtype_code(dprobs)), _ptr(dsc), _ptr(dbd), _i(dtype_code(probs)), _f(scale),
                                                _i(B), _i(H), _i(Tq), _i(Tk), _i(ld), _stream()), "attn_softmax_bwd")


def lsmooth_kl_fwdbwd(logits, ys, ylens, V, smoothing, grad_scale, upstream, row_loss, grad):
    """logits/grad: (B*(lmax+1), >=V) 2-D views (row stride = padded vocab)."""
    B, lmax = ys.shape
    _lib.check(_lib.lib().lasr_lsmooth_kl_fwdbwd(_ptr(logits), _i(dtype_code(logits)), _l(logits.stride(0)), _ptr(ys), _ptr(ylens), _i(B),
                                                 _i(lmax), _i(V), _f(smoothing), _f(grad_scale), _ptr(upstream), _ptr(row_loss),
                                                 _ptr(grad), _l(grad.stride(0)), _stream()), "lsmooth_kl")


def hybrid_combine(nll, row_kl, ctc_weight, out):
    _lib.check(_lib.lib().lasr_hybrid_combine(_ptr(nll), _i(nll.numel()), _ptr(row_kl), _i(row_kl.numel()), _f(ctc_weight), _ptr(out),
                                              _stream()), "hybrid_combine")


def clip_adam_step(params, grads, exp_avg, exp_avg_sq, state, workspace, *, grad_mult=1.0, max_norm=5.0, beta1=0.9, beta2=0.999,
                   eps=1e-8, weight_decay=0.0, noam_factor=0.0, model_dim=256.0, warmup=25000.0, lr=1e-3):
    _lib.check(_lib.lib().lasr_clip_adam_step(_ptr(params), _ptr(grads), _ptr(exp_avg), _ptr(exp_avg_sq), _l(params.numel()),
                                              _f(grad_mult), _f(max_norm), _f(beta1), _f(beta2), _f(eps), _f(weight_decay),
                                              _f(noam_factor), _f(model_dim), _f(warmup), _f(lr), _ptr(state), _ptr(workspace),
                                              _stream()), "clip_adam_step")


# ----------------------------------------------------------------------------------------------
# inference
# ----------------------------------------------------------------------------------------------
def logsoftmax_topk(logits: torch.Tensor, k: int, *, vocab: Optional[int] = None, want_lse: bool = False, want_full: bool = False):
    """logits (rows, >=V) 2-D view (row stride = padded vocab).  Returns (top_val (rows,k) fp32 log-probs, top_idx (rows,k) int32,
    lse (rows,) or None, logp (rows,V) fp32 or None)."""
    _require_cuda(logits)
    assert logits.dim() == 2 and logits.stride(1) == 1
    rows = logits.shape[0]
    V = logits.shape[1] if vocab is None else vocab
    dev = logits.device
    tv = torch.empty((rows, k), dtype=torch.float32, device=dev) if k else None
    ti = torch.empty((rows, k), dtype=torch.int32, device=dev) if k else None
    lse = torch.empty(rows, dtype=torch.float32, device=dev) if want_lse else None
    full = torch.empty((rows, V), dtype=torch.float32, device=dev) if want_full else None
    _lib.check(_lib.lib().lasr_logsoftmax_topk(_ptr(logits), _i(dtype_code(logits)), _l(logits.stride(0)), _l(rows), _i(V), _i(k), _ptr(lse),
                                               _ptr(full), _l(V), _ptr(tv), _ptr(ti), _stream()), "logsoftmax_topk")
    return tv, ti, lse, full


def gather_logp(logits: torch.Tensor, lse: torch.Tensor, tokens: torch.Tensor, vocab: int) -> torch.Tensor:
    """out[r] = logits[r, tokens[r]] - lse[r] (0 where tokens[r] < 0)."""
    _require_cuda(logits, lse, tokens)
    rows = logits.shape[0]
    assert tokens.dtype == torch.int64 and tokens.numel() == rows and lse.numel() == rows
    out = torch.empty(rows, dtype=torch.float32, device=logits.device)
    _lib.check(_lib.lib().lasr_gather_logp(_ptr(logits), _i(dtype_code(logits)), _l(logits.stride(0)), _ptr(lse), _ptr(tokens.contiguous()),
                                           _ptr(out), _l(rows), _i(vocab), _stream()), "gather_logp")
    return out


def ctc_prefix_beam_search_host(top_val, top_idx, beam: int = 10, blank: int = 0):
    """HOST: top_val (frames,K) float32 / top_idx (frames,K) int32 numpy arrays -> [(prefix tuple, score float64)] best first."""
    import numpy as np
    tv = np.ascontiguousarray(top_val, dtype=np.float32)
    ti = np.ascontiguousarray(top_idx, dtype=np.int32)
    frames, K = tv.shape if tv.ndim == 2 else (0, max(1, beam))
    max_len = max(1, frames)
    toks = np.empty((beam, max_len), dtype=np.int32)
    lens = np.empty(beam, dtype=np.int32)
    scores = np.empty(beam, dtype=np.float64)
    n = C.c_int32(0)
    _lib.check(_lib.lib().lasr_ctc_prefix_beam_search(tv.ctypes.data_as(_P), ti.ctypes.data_as(_P), _i(frames), _i(K), _i(beam), _i(blank),
                                                      toks.ctypes.data_as(_P), lens.ctypes.data_as(_P), scores.ctypes.data_as(_P),
                                                      _i(max_len), C.byref(n)), "ctc_prefix_beam_search")
    return [(tuple(int(x) for x in toks[i, : lens[i]]), float(scores[i])) for i in range(n.value)]


def ctc_prefix_beam_search_batch(top_val: torch.Tensor, top_idx: torch.Tensor, frames: torch.Tensor, Tmax: int, beam: int = 10,
                                 blank: int = 0):
    """DEVICE prefix search over a ragged batch (one launch, no host synchronisation).  top_val / top_idx (B*Tmax, K) as
    ``logsoftmax_topk`` returns them, frames (B,) int64 on the device.  -> (tokens (B,beam,Tmax) int32 padded -1, lengths (B,beam)
    int32, scores (B,beam) float64, counts (B,) int32), all on the device."""
    _require_cuda(top_val, top_idx, frames)
    assert top_val.dtype == torch.float32 and top_idx.dtype == torch.int32 and frames.dtype == torch.int64
    assert top_val.is_contiguous() and top_idx.is_contiguous() and frames.is_contiguous() and top_val.shape == top_idx.shape
    B = frames.numel()
    K = top_val.shape[1]
    assert top_val.shape[0] == B * Tmax
    dev = top_val.device
    toks = torch.empty((B, beam, Tmax), dtype=torch.int32, device=dev)
    lens = torch.empty((B, beam), dtype=torch.int32, device=dev)
    scores = torch.empty((B, beam), dtype=torch.float64, device=dev)
    count = torch.empty(B, dtype=torch.int32, device=dev)
    L = _lib.lib()
    ws_bytes = int(L.lasr_ctc_prefix_beam_search_batch_workspace(_i(B), _i(Tmax), _i(beam)))
    ws = torch.empty(max(ws_bytes, 8), dtype=torch.uint8, device=dev)
    _lib.check(L.lasr_ctc_prefix_beam_search_batch(_ptr(top_val), _ptr(top_idx), _ptr(frames), _i(B), _i(Tmax), _i(K), _i(beam), _i(blank),
                                                   _ptr(toks), _ptr(lens), _ptr(scores), _ptr(count), _i(Tmax), _ptr(ws),
                                                   C.c_size_t(ws.numel()), _stream()), "ctc_prefix_beam_search_batch")
    return toks, lens, scores, count


def ctc_forced_align(logits: torch.Tensor, lse: torch.Tensor, targets: torch.Tensor, tgt_len: torch.Tensor, frames: torch.Tensor, Tmax: int,
                     blank: int = 0, *, vocab: Optional[int] = None):
    """DEVICE CTC Viterbi forced alignment of a ragged batch (include/lasr_align.h, one launch, no host synchronisation).
    logits (B*Tmax, >=V) fp32 | bf16 2-D view (utterance b at rows [b*Tmax, b*Tmax + frames[b])), lse (B*Tmax,) fp32 as
    ``logsoftmax_topk(..., want_lse=True)`` returns it, targets (B, lmax) int64 padded -1, tgt_len / frames (B,) int64.
    -> (state (B,Tmax) int32, frame_logp (B,Tmax) fp32, score (B,) fp32, spans (B,lmax,2) int32), all on the device."""
    _require_cuda(logits, lse, targets, tgt_len, frames)
    assert logits.dim() == 2 and logits.stride(1) == 1 and lse.dtype == torch.float32 and lse.is_contiguous()
    assert targets.dtype == torch.int64 and tgt_len.dtype == torch.int64 and frames.dtype == torch.int64 and targets.dim() == 2
    B, lmax = targets.shape
    assert tgt_len.numel() == B and frames.numel() == B and logits.shape[0] == B * Tmax and lse.numel() == B * Tmax
    V = logits.shape[1] if vocab is None else vocab
    dev = logits.device
    targets, tgt_len, frames = targets.contiguous(), tgt_len.contiguous(), frames.contiguous()
    state = torch.empty((B, Tmax), dtype=torch.int32, device=dev)
    logp = torch.empty((B, Tmax), dtype=torch.float32, device=dev)
    score = torch.empty(B, dtype=torch.float32, device=dev)
    spans = torch.empty((B, lmax, 2), dtype=torch.int32, device=dev)
    L = _lib.lib()
    ws_bytes = int(L.lasr_ctc_forced_align_workspace(_i(B), _i(Tmax), _i(lmax)))
    ws = torch.empty(max(ws_bytes, 8), dtype=torch.uint8, device=dev)
    _lib.check(L.lasr_ctc_forced_align(_ptr(logits), _i(dtype_code(logits)), _l(logits.stride(0)), _ptr(lse), _ptr(targets), _ptr(tgt_len),
                                       _ptr(frames), _i(B), _i(Tmax), _i(lmax), _i(V), _i(blank), _ptr(state), _ptr(logp), _ptr(score),
                                       _ptr(spans), _ptr(ws), C.c_size_t(ws.numel()), _stream()), "ctc_forced_align")
    return state, logp, score, spans


def fbank(wave: torch.Tensor, nsamp: torch.Tensor, frame_len: int, frame_shift: int, window: torch.Tensor, mel_lo: torch.Tensor,
          mel_off: torch.Tensor, mel_w: torch.Tensor) -> torch.Tensor:
    """DEVICE Kaldi log-mel filterbank of a padded batch (include/lasr_fbank.h, one launch, no host synchronisation).
    wave (B, Nmax) int16 | fp32 in int16 scale, row stride >= Nmax; nsamp (B,) int64; frame_len / frame_shift in samples;
    window (frame_len,) fp32; the sparse mel bank mel_lo (nb,) int32, mel_off (nb+1,) int32, mel_w (mel_off[nb],) fp32.
    -> (B, Fmax, nb) fp32, Fmax = the frame count of Nmax, rows past each utterance's frames 0."""
    _require_cuda(wave, nsamp, window, mel_lo, mel_off, mel_w)
    assert wave.dim() == 2 and wave.stride(1) == 1 and nsamp.dtype == torch.int64 and nsamp.numel() == wave.shape[0]
    assert window.dtype == torch.float32 and mel_w.dtype == torch.float32 and mel_lo.dtype == torch.int32 and mel_off.dtype == torch.int32
    assert mel_off.numel() == mel_lo.numel() + 1
    if wave.dtype == torch.int16:
        code = _lib.I16
    elif wave.dtype == torch.float32:
        code = F32
    else:
        raise TypeError(f"fbank takes int16 or fp32 samples, not {wave.dtype}")
    B, nmax = wave.shape
    nb = mel_lo.numel()
    fmax = 0 if nmax < frame_len else 1 + (nmax - frame_len) // frame_shift
    out = torch.empty((B, fmax, nb), dtype=torch.float32, device=wave.device)
    _lib.check(_lib.lib().lasr_fbank(_ptr(wave), _i(code), _l(wave.stride(0) if B > 1 else nmax), _ptr(nsamp.contiguous()), _i(B), _l(nmax),
                                     _i(frame_len), _i(frame_shift), _ptr(window.contiguous()), _i(nb), _ptr(mel_lo.contiguous()),
                                     _ptr(mel_off.contiguous()), _ptr(mel_w.contiguous()), _ptr(out), _stream()), "fbank")
    return out
