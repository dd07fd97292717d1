"""Forward / backward pipelines of the U2 hot path, written against the C ABI (``ops``) and the flat ``ParamStore``.

This is the host-side schedule: which kernel runs on which buffer in which order.  Every arithmetic step is a
``lasr_*`` kernel; torch is used for allocation (caching allocator -> CUDA-graph friendly), views and streams only.

Numerics / layout decisions (see DESIGN.md):
  * residual stream and all statistics in fp32; GEMM operands in ``adt`` (bf16 on tcgen05, or fp32 on the SIMT path);
  * activations are (rows, features) row-major with rows = (batch, time): the reference's transposes for Conv1d /
    Conv2d / heads disappear (heads are addressed in place through the GEMM's two-level batch strides);
  * every backward accumulates parameter gradients straight into ``store.gflat`` (split-K ``red.add`` wgrads, column-sum
    bias gradients), so gradient accumulation and the flat all-reduce need no extra pass.

Reference lines restated by each block are cited inline (paths relative to /root/reference/liteasr).
"""
from __future__ import annotations

import math
import os
from types import SimpleNamespace as NS
from typing import Optional

import torch

from . import dropout as DR
from . import ops
from .ops import ACT_MUL, ACT_NONE, ACT_RELU, ACT_SWISH
from .store import ParamStore

LN_EPS = 1e-12
KW = 15


def _ceil(a: int, b: int) -> int:
    return (a + b - 1) // b * b


def _empty(shape, dtype, dev):
    return torch.empty(shape, dtype=dtype, device=dev)


class Engine:
    def __init__(self, store: ParamStore):
        self.st = store
        self.adt = store.adt
        # attention score tensors that still round-trip through HBM (dprobs of every attention backward; ac / bd of the unfused
        # forward: decoder attentions, T' > 320): the operand dtype in bf16 mode -- what torch autocast's matmul hands to the softmax
        # in the reference's bf16 run -- which halves their traffic (183 -> 91 MB per tensor at C2/B=126; 0.9 % of the step).
        self.sdt = store.adt
        self.dev = store.device
        # LASR_FUSED_ATTN=0: developer switch back to GEMM -> softmax kernel -> GEMM for the rel-pos attention forward
        self.fused_attn = os.environ.get("LASR_FUSED_ATTN", "1") != "0"
        self.fused_attn_bwd = os.environ.get("LASR_FUSED_ATTN_BWD", "1") != "0"
        # off by default: correct but measured slower than the GEMM pair (csrc/ffn_fused.cu, "STATUS")
        self.fused_ffn_fwd = store.adt == torch.bfloat16 and os.environ.get("LASR_FUSED_FFN_FWD", "0") == "1"

    # ------------------------------------------------------------------------------------------
    # small helpers
    # ------------------------------------------------------------------------------------------
    def to_adt(self, x32: torch.Tensor) -> torch.Tensor:
        """fp32 -> operand dtype copy (identity in fp32 mode)."""
        if self.adt == torch.float32:
            return x32
        out = _empty(x32.shape, torch.bfloat16, self.dev)
        ops.cast_bf16(x32.reshape(-1), out.reshape(-1))
        return out

    def layernorm(self, x: torch.Tensor, pfx: str, out_dtype) -> NS:
        rows, d = x.shape
        y = _empty((rows, d), out_dtype, self.dev)
        mean = _empty((rows,), torch.float32, self.dev)
        rstd = _empty((rows,), torch.float32, self.dev)
        ops.layernorm_fwd(x, self.st.p(pfx + ".weight"), self.st.p(pfx + ".bias"), y, mean, rstd, LN_EPS)
        return NS(x=x, y=y, mean=mean, rstd=rstd, pfx=pfx)

    def layernorm_bwd(self, ln: NS, dy: torch.Tensor, dx: torch.Tensor, accumulate: bool, nxt=None, want_lo: bool = False):
        """dx (+)= LN'(dy) and the LayerNorm parameter gradients.  ``nxt = (bias_grad, scale, drop)``: the updated residual-stream
        gradient dx is also the output gradient of the block that runs next in backward order, so its output Linear's bias
        gradient (scale * colsum(dx)) and the operand-dtype copy of dx that block's GEMMs read are produced here, in the same
        pass -- both masked with that block's output-dropout site ``drop`` (None = no dropout there).  Returns that copy (dx
        itself in fp32 mode without dropout), or None when not requested."""
        want_lo = want_lo or nxt is not None
        drop = nxt[2] if nxt is not None and len(nxt) > 2 else None
        lo = None
        if want_lo and (self.adt != torch.float32 or drop is not None):
            lo = _empty(dx.shape, self.adt, self.dev)
        ops.layernorm_bwd(dy, ln.x, ln.mean, ln.rstd, self.st.p(ln.pfx + ".weight"), dx, self.st.g(ln.pfx + ".weight"),
                          self.st.g(ln.pfx + ".bias"), accumulate, dx_lo=lo, colsum=(nxt[0] if nxt is not None else None),
                          colsum_scale=(nxt[1] if nxt is not None else 1.0), drop=drop)
        if not want_lo:
            return None
        return lo if lo is not None else dx

    @staticmethod
    def _pick_bn(n: int, gran: int) -> int:
        if n <= 256:
            return (n + gran - 1) // gran * gran
        best, best_pad = 256, (n + 255) // 256 * 256
        for bn in range(256 - gran, 127, -gran):
            pad = (n + bn - 1) // bn * bn
            if pad < best_pad:
                best, best_pad = bn, pad
        return best

    def _split_k(self, n_out: int, k_out: int, rows: int) -> int:
        if self.adt == torch.float32:
            # parity mode: the SIMT kernel accumulates in fp64; a moderate split only adds parallelism
            return max(1, min(64, rows // 512))
        bn = self._pick_bn(k_out, 64)  # the wgrad GEMM is (n_out x k_out), B operand MN-major
        tiles = ((n_out + 127) // 128) * ((k_out + bn - 1) // bn)
        s = max(1, min(74, 148 // max(1, tiles)))  # one work unit per SM (a 256 x 256 weight gradient is 2 tiles -> 74 splits)
        s = min(s, max(1, rows // 256))
        return s

    def linear(self, x, wname, out_dtype, *, bias=True, act=ACT_NONE, res=None, alpha=1.0, aux=False, w=None, n=None,
               bias_t=None, drop=None, drop_mark_aux=False, aux_deriv=False):
        """y = drop(alpha * act(x @ W^T + b)) (+ res).  W (N,K) from the store (or ``w``)."""
        w = self.st.w(wname + ".weight") if w is None else w
        n = w.shape[0] if n is None else n
        m = x.shape[0]
        ld = _ceil(n, 8)
        buf = _empty((m, ld), out_dtype, self.dev)
        out = buf[:, :n] if ld != n else buf
        auxbuf = None
        if aux:
            ab = _empty((m, ld), out_dtype, self.dev)
            auxbuf = ab[:, :n] if ld != n else ab
        b = bias_t if bias_t is not None else (self.st.p(wname + ".bias") if bias else None)
        ops.gemm(x, w, out, m, n, x.shape[1], lda=x.stride(0), ldb=w.stride(0), ldc=ld, bias=b, res=res,
                 ldres=(res.stride(0) if res is not None else 0), aux=auxbuf, alpha=alpha, act=act, drop=drop,
                 drop_mark_aux=drop_mark_aux, aux_deriv=aux_deriv)
        return (out, auxbuf) if aux else out

    def wgrad(self, dy, x, gw, alpha=1.0) -> None:
        """gw (N_out, K_in) += alpha * dy^T x   (split-K tcgen05 / SIMT GEMM with red.add)."""
        m, n = dy.shape
        k = x.shape[1]
        if (dy.dtype == torch.bfloat16 and x.dtype == torch.bfloat16 and ops.wgrad2_supported(n, k) and m >= 1024
                and dy.stride(0) % 8 == 0 and x.stride(0) % 8 == 0 and gw.stride(0) % 4 == 0):
            # CTA pairs (tcgen05.mma.cta_group::2): each SM stages half of both operands of a 256 x 256 tile (csrc/gemm2_wgrad.cu);
            # one work unit per pair, split-K so that the units cover the 74 pairs of the machine
            tiles = (n // 256) * (k // 256)
            ops.wgrad2(dy, x, gw, alpha=alpha, split_k=max(1, min(74 // tiles if tiles <= 74 else 1, m // 512)))
            return
        ops.gemm(dy, x, gw, n, k, m, lda=dy.stride(0), ldb=x.stride(0), ldc=gw.stride(0), ta=True, tb=True, accumulate=True,
                 split_k=self._split_k(n, k, m), alpha=alpha)

    def dgrad(self, dy, w, *, out_dtype=None, alpha=1.0, dx_res=None, dact=None, act=ACT_NONE, colsum=None, drop=None):
        """dx = alpha * dy @ W (W stored (N_out, K_in)); optional fused activation backward (``dact``/``act``), bias-gradient
        column sum of the result (``colsum``) and fp32 accumulation into ``dx_res``."""
        m, n = dy.shape
        k = w.shape[1]
        dx = _empty((m, k), self.adt if out_dtype is None else out_dtype, self.dev) if dx_res is None else dx_res
        ops.gemm(dy, w, dx, m, k, n, lda=dy.stride(0), ldb=w.stride(0), ldc=dx.stride(0), tb=True, alpha=alpha,
                 res=dx_res, ldres=(dx_res.stride(0) if dx_res is not None else 0), dact=dact, act=act, colsum=colsum, drop=drop)
        return dx

    def linear_bwd(self, dy, x, wname, *, need_dx=True, dx_dtype=None, bias=True, dbias_done=False, alpha=1.0, w=None,
                   gw=None, gb=None, dx_res=None, dx_drop=None):
        """dW += alpha * dy^T x ; db += colsum(dy) (unless fused earlier) ; returns dx = alpha * dy @ W."""
        w = self.st.w(wname + ".weight") if w is None else w
        gw = self.st.gw(wname + ".weight") if gw is None else gw
        if bias and not dbias_done:
            ops.act_bwd(dy, None, None, self.st.g(wname + ".bias") if gb is None else gb, ACT_NONE, alpha)
        self.wgrad(dy, x, gw, alpha)
        if not need_dx:
            return None
        return self.dgrad(dy, w, out_dtype=dx_dtype, alpha=alpha, dx_res=dx_res, drop=dx_drop)

    # ------------------------------------------------------------------------------------------
    # feed-forward block   x <- x + scale * fc2(act(fc1(LN x)))      nets/feed_forward.py:18-19,
    #                                                               nets/conformer_layer.py:37-47,58-66
    # ------------------------------------------------------------------------------------------
    def ffn_fwd(self, x, pfx_norm, pfx_ff, act, scale, d_in=None, d_out=None) -> NS:
        """d_in: dropout on the activation (feed_forward.py:19); d_out: dropout on the block output before the residual add
        (conformer_layer.py:42,63, transformer_layer.py:58).  Swish: what fc1 saves for the backward pass is ``g = swish'(h)``
        (``aux_deriv``), not the pre-activation ``h``: the backward epilogue then multiplies by ``g`` instead of re-evaluating
        swish' (it is instruction-bound), and the inner dropout mask needs no regeneration either -- ``g`` is 0 at dropped
        elements (ReLU: the saved output is 0 there)."""
        ln = self.layernorm(x, pfx_norm, self.adt)
        w1, w2 = self.st.w(pfx_ff + ".fc1.weight"), self.st.w(pfx_ff + ".fc2.weight")
        if (act == ACT_SWISH and self.fused_ffn_fwd and ops.ffn_fwd_supported(w1.shape[1], w1.shape[0])
                and ln.y.stride(0) % 8 == 0 and x.stride(0) % 4 == 0):
            # ONE kernel: a and g = swish'(h) are written once, the second contraction reads a from shared memory (csrc/ffn_fused.cu)
            m, f = ln.y.shape[0], w1.shape[0]
            a, h = _empty((m, f), self.adt, self.dev), _empty((m, f), self.adt, self.dev)
            out = _empty((m, x.shape[1]), torch.float32, self.dev)
            ops.ffn_fwd(ln.y, w1, self.st.p(pfx_ff + ".fc1.bias"), w2, self.st.p(pfx_ff + ".fc2.bias"), x, a, h, out, alpha=scale,
                        drop_in=d_in, drop_out=d_out)
            return NS(out=out, ln=ln, a=a, h=h, act=act, scale=scale, pfx=pfx_ff, d_in=d_in, d_out=d_out)
        if act == ACT_SWISH:
            a, h = self.linear(ln.y, pfx_ff + ".fc1", self.adt, act=act, aux=True, drop=d_in, drop_mark_aux=True, aux_deriv=True)
        else:  # ReLU: act'(.) from the output
            a, h = self.linear(ln.y, pfx_ff + ".fc1", self.adt, act=act, drop=d_in), None
        out = self.linear(a, pfx_ff + ".fc2", torch.float32, res=x, alpha=scale, drop=d_out)
        return NS(out=out, ln=ln, a=a, h=h, act=act, scale=scale, pfx=pfx_ff, d_in=d_in, d_out=d_out)

    def ffn_bwd(self, c: NS, dres: torch.Tensor, dy: torch.Tensor, nxt=None, want_lo=False):
        """dres (fp32, in/out): gradient wrt the block output on entry, wrt the block input on exit.  dy = operand-dtype copy of
        dres on entry (fc2's bias gradient was taken by the producer of dy).  Returns the operand copy of the updated dres."""
        st = self.st
        self.wgrad(dy, c.a, st.gw(c.pfx + ".fc2.weight"), c.scale)
        # dh = scale * (dy @ W2) * act'(.)  and  db1 += colsum(dh), both in the dgrad epilogue; with inner dropout the 1/(1-p)
        # factor rides on alpha and the mask is implied by the saved tensor (marker / zero)
        s_in = c.scale * (c.d_in.scale if c.d_in is not None else 1.0)
        if (c.act == ACT_SWISH and self.adt == torch.bfloat16 and ops.ffn_bwd_supported(dy.shape[1], c.h.shape[1]) and c.h.stride(0) % 8 == 0
              and dy.stride(0) % 8 == 0):
            # ONE kernel: dh = s (dy @ W2) * g, db1 += colsum(dh), dln = dh @ W1 -- dh is written once (the fc1 weight gradient
            # needs it) and never read back by the second contraction
            dh = _empty(c.h.shape, self.adt, self.dev)
            dln = _empty(dy.shape, self.adt, self.dev)
            ops.ffn_bwd(dy, c.h, st.w(c.pfx + ".fc2.weight"), st.w(c.pfx + ".fc1.weight"), dh, dln, colsum=st.g(c.pfx + ".fc1.bias"),
                        alpha=s_in)
            self.wgrad(dh, c.ln.y, st.gw(c.pfx + ".fc1.weight"))
            return self.layernorm_bwd(c.ln, dln, dres, True, nxt, want_lo)
        else:
            dh = self.dgrad(dy, st.w(c.pfx + ".fc2.weight"), alpha=s_in, dact=(c.h if c.act == ACT_SWISH else c.a),
                            act=(ACT_MUL if c.act == ACT_SWISH else c.act), colsum=st.g(c.pfx + ".fc1.bias"))
        self.wgrad(dh, c.ln.y, st.gw(c.pfx + ".fc1.weight"))
        dln = self.dgrad(dh, st.w(c.pfx + ".fc1.weight"))
        return self.layernorm_bwd(c.ln, dln, dres, True, nxt, want_lo)

    # ------------------------------------------------------------------------------------------
    # attention core on projected q/k/v  (nets/attention.py:46-59,61-71,120-154)
    # q: (B*Tq, *) view with row stride ldq, k/v: (B*Tk, *) views; heads addressed via batch strides.
    # ------------------------------------------------------------------------------------------
    def attn_core_fwd(self, q, k, v, B, H, Tq, Tk, dk, lens, mask_mode, causal, qv=None, p=None, drop=None) -> NS:
        """``drop``: dropout on the attention probabilities (attention.py:55).  0.0 in the reference's shipped config; a
        non-zero rate keeps the unfused sequence and costs one extra pass in each direction (probabilities are saved undropped
        for the softmax backward, the dropped copy feeds probs.V and dV)."""
        d = H * dk
        ld = _ceil(Tk, 8)
        scale = dk ** -0.5
        fused = (qv is not None and drop is None and Tq == Tk and self.adt == torch.bfloat16 and self.fused_attn
                 and ops.rel_attn_fwd_supported(Tk, dk) and q.stride(0) == qv.stride(0) and k.stride(0) == v.stride(0))
        if fused:
            ld = _ceil(Tk, 64)  # 128-byte aligned probability rows: every 128-byte piece the kernel stores is a whole line
            # one tcgen05 kernel: both score contractions, rel_shift, scale, mask, softmax and probs.V (csrc/attn_fused.cu)
            probs = _empty((B, H, Tq, ld), self.adt, self.dev)
            o = _empty((B * Tq, d), self.adt, self.dev)
            ops.rel_attn_fwd(q, qv, k, v, p, probs, o, lens, mask_mode, scale, B, H, Tq, dk)
            return NS(q=q, k=k, v=v, qv=qv, p=p, probs=probs, probs_d=probs, drop=None, o=o, B=B, H=H, Tq=Tq, Tk=Tk, dk=dk, ld=ld,
                      scale=scale)
        ac = _empty((B, H, Tq, ld), self.sdt, self.dev)
        # n_store = ld: the padding columns [Tk, ld) are written too (zeros), which keeps the whole epilogue on the vector path
        ops.gemm(q, k, ac, Tq, Tk, dk, lda=q.stride(0), ldb=k.stride(0), ldc=ld, batch=(B, H), sa=(Tq * q.stride(0), dk),
                 sb=(Tk * k.stride(0), dk), sc=(H * Tq * ld, Tq * ld), n_store=ld)
        bd = None
        if qv is not None:  # rel-pos term (q + v_bias) . P^T, P broadcast over the batch
            bd = _empty((B, H, Tq, ld), self.sdt, self.dev)
            ops.gemm(qv, p, bd, Tq, Tk, dk, lda=qv.stride(0), ldb=p.stride(0), ldc=ld, batch=(B, H),
                     sa=(Tq * qv.stride(0), dk), sb=(0, dk), sc=(H * Tq * ld, Tq * ld), n_store=ld)
        probs = _empty((B, H, Tq, ld), self.adt, self.dev)
        ops.attn_softmax_fwd(ac, bd, probs, lens, mask_mode, causal, scale, Tk)
        probs_d = probs
        if drop is not None:  # logical tensor (B*H*Tq, Tk); the padding columns [Tk, ld) stay zero
            probs_d = _empty(probs.shape, self.adt, self.dev)
            if ld != Tk:
                ops.zero_(probs_d)
            ops.dropout(probs.view(-1, ld)[:, :Tk], probs_d.view(-1, ld)[:, :Tk], drop)
        o = _empty((B * Tq, d), self.adt, self.dev)
        ops.gemm(probs_d, v, o, Tq, dk, Tk, lda=ld, ldb=v.stride(0), ldc=d, tb=True, batch=(B, H), sa=(H * Tq * ld, Tq * ld),
                 sb=(Tk * v.stride(0), dk), sc=(Tq * d, dk))
        return NS(q=q, k=k, v=v, qv=qv, p=p, probs=probs, probs_d=probs_d, drop=drop, o=o, B=B, H=H, Tq=Tq, Tk=Tk, dk=dk, ld=ld,
                  scale=scale)

    def attn_core_bwd(self, c: NS, do, dq, dk_, dv, dqv=None, dp32=None, bq=None, bk=None, bv=None) -> None:
        """do (B*Tq,d) adt.  Writes dq/dk_/dv (views with the same strides as q/k/v); rel-pos: dqv and dp32 (+=).
        bq/bk/bv: bias-gradient vectors (d,) of the q/k/v projections, accumulated in the GEMM epilogues (head h -> [h*dk, (h+1)*dk))."""
        B, H, Tq, Tk, dk, ld = c.B, c.H, c.Tq, c.Tk, c.dk, c.ld
        bs = (H * Tq * ld, Tq * ld)
        dprobs = _empty((B, H, Tq, ld), self.sdt, self.dev)
        ops.gemm(do, c.v, dprobs, Tq, Tk, dk, lda=do.stride(0), ldb=c.v.stride(0), ldc=ld, batch=(B, H), sa=(Tq * do.stride(0), dk),
                 sb=(Tk * c.v.stride(0), dk), sc=bs, n_store=ld)
        if c.drop is not None:  # d(probs) = keep * scale * d(dropped probs): the forward mask, regenerated in place
            ops.dropout(dprobs.view(-1, ld)[:, :Tk], dprobs.view(-1, ld)[:, :Tk], c.drop)
        # dV[j] = sum_i probs[i,j] dO[i]   (the probabilities that multiplied V: the dropped copy)
        ops.gemm(c.probs_d, do, dv, Tk, dk, Tq, lda=ld, ldb=do.stride(0), ldc=dv.stride(0), ta=True, tb=True, batch=(B, H), sa=bs,
                 sb=(Tq * do.stride(0), dk), sc=(Tk * dv.stride(0), dk), colsum=bv, cs=(0, dk))
        dsc = _empty((B, H, Tq, ld), self.adt, self.dev)
        dbd = _empty((B, H, Tq, ld), self.adt, self.dev) if c.qv is not None else None
        ops.attn_softmax_bwd(c.probs, dprobs, dsc, dbd, c.scale, Tk)
        pair = (self.fused_attn_bwd and self.adt == torch.bfloat16 and ops.attn_bwd_pair_supported(Tk, dk) and bq is None
                and c.k.stride(0) % 8 == 0 and c.q.stride(0) % 8 == 0 and dq.stride(0) % 8 == 0 and dk_.stride(0) % 8 == 0
                and (c.qv is None or (c.p.stride(0) % 8 == 0 and c.qv.stride(0) % 8 == 0 and dqv.stride(0) % 8 == 0)))
        if pair:
            # each (B,H,Tq,Tk) gradient tensor feeds its two contractions from ONE pass through HBM (csrc/attn_pair.cu)
            ops.attn_bwd_pair(dsc, c.k, c.q, dq, dk_, B, H, Tq, Tk, dk, colsum=bk)
            if c.qv is not None:
                ops.attn_bwd_pair(dbd, c.p, c.qv, dqv, dp32, B, H, Tq, Tk, dk, r_batched=False, reduce_b=True)
            return
        # dQ[i] = sum_j ds[i,j] K[j] ; dK[j] = sum_i ds[i,j] Q[i]
        ops.gemm(dsc, c.k, dq, Tq, dk, Tk, lda=ld, ldb=c.k.stride(0), ldc=dq.stride(0), tb=True, batch=(B, H), sa=bs,
                 sb=(Tk * c.k.stride(0), dk), sc=(Tq * dq.stride(0), dk), colsum=bq, cs=(0, dk))
        ops.gemm(dsc, c.q, dk_, Tk, dk, Tq, lda=ld, ldb=c.q.stride(0), ldc=dk_.stride(0), ta=True, tb=True, batch=(B, H), sa=bs,
                 sb=(Tq * c.q.stride(0), dk), sc=(Tk * dk_.stride(0), dk), colsum=bk, cs=(0, dk))
        if c.qv is not None:
            ops.gemm(dbd, c.p, dqv, Tq, dk, Tk, lda=ld, ldb=c.p.stride(0), ldc=dqv.stride(0), tb=True, batch=(B, H), sa=bs,
                     sb=(0, dk), sc=(Tq * dqv.stride(0), dk))
            ops.gemm(dbd, c.qv, dp32, Tk, dk, Tq, lda=ld, ldb=c.qv.stride(0), ldc=dp32.stride(0), ta=True, tb=True, batch=(B, H),
                     sa=bs, sb=(Tq * c.qv.stride(0), dk), sc=(0, dk), accumulate=True)

    # ------------------------------------------------------------------------------------------
    # relative-position self-attention block (nets/conformer_layer.py:107-128, nets/attention.py:120-154)
    # ------------------------------------------------------------------------------------------
    def rel_mha_fwd(self, x, pfx_norm, pfx, pos, B, T, H, xlens, d_att=None, d_out=None, sub_lens=None) -> NS:
        """sub_lens: sub-sampled lengths -> mask mode 4 (per-utterance shift, inference only) instead of xlens' mode 3."""
        d = x.shape[1]
        dk = d // H
        ln = self.layernorm(x, pfx_norm, self.adt)
        wqkv = self.st.w(pfx + ".linear_q.weight", 3 * d, d)
        bqkv = self.st.p_span(pfx + ".linear_q.bias", 3 * d)
        qkv = self.linear(ln.y, None, self.adt, w=wqkv, bias_t=bqkv)
        q, k, v = qkv[:, :d], qkv[:, d:2 * d], qkv[:, 2 * d:]
        qu = _empty((B * T, d), self.adt, self.dev)
        qv = _empty((B * T, d), self.adt, self.dev)
        ops.pos_bias_fwd(q, self.st.p(pfx + ".pos_bias_u").view(-1), self.st.p(pfx + ".pos_bias_v").view(-1), qu, qv)
        p = self.linear(pos, pfx + ".linear_pos", self.adt, bias=False)
        if sub_lens is not None:
            core = self.attn_core_fwd(qu, k, v, B, H, T, T, dk, sub_lens, 4, 0, qv=qv, p=p, drop=d_att)
        else:
            core = self.attn_core_fwd(qu, k, v, B, H, T, T, dk, xlens, 3 if xlens is not None else 0, 0, qv=qv, p=p, drop=d_att)
        out = self.linear(core.o, pfx + ".linear_o", torch.float32, res=x, drop=d_out)
        return NS(out=out, ln=ln, qkv=qkv, core=core, pos=pos, pfx=pfx, d=d, d_out=d_out)

    def rel_mha_bwd(self, c: NS, dres, dy, nxt=None, want_lo=False):
        st, d, core = self.st, c.d, c.core
        B, T = core.B, core.Tq
        self.wgrad(dy, core.o, st.gw(c.pfx + ".linear_o.weight"))
        do = self.dgrad(dy, st.w(c.pfx + ".linear_o.weight"))
        dqkv = _empty((B * T, 3 * d), self.adt, self.dev)
        dqu = _empty((B * T, d), self.adt, self.dev)
        dqv = _empty((B * T, d), self.adt, self.dev)
        dp32 = torch.empty((T, d), dtype=torch.float32, device=self.dev)
        ops.zero_(dp32)
        gb = st.g_span(c.pfx + ".linear_q.bias", 3 * d)
        self.attn_core_bwd(core, do, dqu, dqkv[:, d:2 * d], dqkv[:, 2 * d:], dqv=dqv, dp32=dp32, bk=gb[d:2 * d], bv=gb[2 * d:])
        ops.pos_bias_bwd(dqu, dqv, dqkv[:, :d], st.g(c.pfx + ".pos_bias_u").view(-1), st.g(c.pfx + ".pos_bias_v").view(-1), gb[:d])
        # linear_pos (no bias): dW_pos += dP^T pos
        self.wgrad(self.to_adt(dp32), c.pos, st.gw(c.pfx + ".linear_pos.weight"))
        # fused q/k/v projection
        self.wgrad(dqkv, c.ln.y, st.gw(c.pfx + ".linear_q.weight", 3 * d, d))
        dln = self.dgrad(dqkv, st.w(c.pfx + ".linear_q.weight", 3 * d, d))
        return self.layernorm_bwd(c.ln, dln, dres, True, nxt, want_lo)

    # ------------------------------------------------------------------------------------------
    # plain MHA blocks of the decoder (nets/transformer_layer.py:29-51,161-177, nets/attention.py:61-71)
    # ------------------------------------------------------------------------------------------
    def self_mha_fwd(self, y, pfx_norm, pfx, B, L, H, ylens, d_att=None, d_out=None) -> NS:
        d = y.shape[1]
        ln = self.layernorm(y, pfx_norm, self.adt)
        qkv = self.linear(ln.y, None, self.adt, w=self.st.w(pfx + ".linear_q.weight", 3 * d, d),
                          bias_t=self.st.p_span(pfx + ".linear_q.bias", 3 * d))
        core = self.attn_core_fwd(qkv[:, :d], qkv[:, d:2 * d], qkv[:, 2 * d:], B, H, L, L, d // H, ylens, 2, 1, drop=d_att)
        out = self.linear(core.o, pfx + ".linear_o", torch.float32, res=y, drop=d_out)
        return NS(out=out, ln=ln, core=core, pfx=pfx, d=d, d_out=d_out)

    def self_mha_bwd(self, c: NS, dres, dy, nxt=None, want_lo=False):
        st, d, core = self.st, c.d, c.core
        self.wgrad(dy, core.o, st.gw(c.pfx + ".linear_o.weight"))
        do = self.dgrad(dy, st.w(c.pfx + ".linear_o.weight"))
        dqkv = _empty((core.B * core.Tq, 3 * d), self.adt, self.dev)
        gb = st.g_span(c.pfx + ".linear_q.bias", 3 * d)
        self.attn_core_bwd(core, do, dqkv[:, :d], dqkv[:, d:2 * d], dqkv[:, 2 * d:], bq=gb[:d], bk=gb[d:2 * d], bv=gb[2 * d:])
        self.wgrad(dqkv, c.ln.y, st.gw(c.pfx + ".linear_q.weight", 3 * d, d))
        dln = self.dgrad(dqkv, st.w(c.pfx + ".linear_q.weight", 3 * d, d))
        return self.layernorm_bwd(c.ln, dln, dres, True, nxt, want_lo)

    def src_mha_fwd(self, y, mem, pfx_norm, pfx, B, L, T, H, xlens, mask_mode=3, d_att=None, d_out=None) -> NS:
        d = y.shape[1]
        ln = self.layernorm(y, pfx_norm, self.adt)
        q = self.linear(ln.y, pfx + ".linear_q", self.adt)
        kv = self.linear(mem, None, self.adt, w=self.st.w(pfx + ".linear_k.weight", 2 * d, d),
                         bias_t=self.st.p_span(pfx + ".linear_k.bias", 2 * d))
        core = self.attn_core_fwd(q, kv[:, :d], kv[:, d:], B, H, L, T, d // H, xlens, mask_mode if xlens is not None else 0, 0,
                                  drop=d_att)
        out = self.linear(core.o, pfx + ".linear_o", torch.float32, res=y, drop=d_out)
        return NS(out=out, ln=ln, core=core, mem=mem, pfx=pfx, d=d, d_out=d_out)

    def src_mha_bwd(self, c: NS, dres, dy, dmem32, nxt=None, want_lo=False):
        st, d, core = self.st, c.d, c.core
        self.wgrad(dy, core.o, st.gw(c.pfx + ".linear_o.weight"))
        do = self.dgrad(dy, st.w(c.pfx + ".linear_o.weight"))
        dq = _empty((core.B * core.Tq, d), self.adt, self.dev)
        dkv = _empty((core.B * core.Tk, 2 * d), self.adt, self.dev)
        gkv = st.g_span(c.pfx + ".linear_k.bias", 2 * d)
        self.attn_core_bwd(core, do, dq, dkv[:, :d], dkv[:, d:], bq=st.g(c.pfx + ".linear_q.bias"), bk=gkv[:d], bv=gkv[d:])
        self.wgrad(dq, c.ln.y, st.gw(c.pfx + ".linear_q.weight"))
        dln = self.dgrad(dq, st.w(c.pfx + ".linear_q.weight"))
        lo = self.layernorm_bwd(c.ln, dln, dres, True, nxt, want_lo)
        # dmem += dkv @ W_kv   (fp32, accumulated across the decoder layers through the residual input)
        self.wgrad(dkv, c.mem, st.gw(c.pfx + ".linear_k.weight", 2 * d, d))
        self.dgrad(dkv, st.w(c.pfx + ".linear_k.weight", 2 * d, d), dx_res=dmem32)
        return lo

    # ------------------------------------------------------------------------------------------
    # convolution block (nets/conformer_layer.py:49-56, nets/conformer_convolution.py:44-57)
    # ------------------------------------------------------------------------------------------
    def conv_fwd(self, x, pfx_norm, pfx, B, T, bn_mod, training, d_out=None, sub_lens=None) -> NS:
        """sub_lens: sub-sampled lengths -> rows t >= sub_lens[b] enter the depthwise conv as zeros (inference only)."""
        st, d = self.st, x.shape[1]
        ln = self.layernorm(x, pfx_norm, self.adt)
        y2 = self.linear(ln.y, None, self.adt, w=st.w(pfx + ".pointwise_conv1.weight"), bias_t=st.p(pfx + ".pointwise_conv1.bias"))
        z = _empty((B * T, d), torch.float32, self.dev)
        nblk = B * ((T + 31) // 32)
        partial = _empty((nblk, 2, d), torch.float32, self.dev)
        if sub_lens is not None:
            ops.glu_dwconv_fwd_lens(y2, st.p(pfx + ".depthwise_conv.weight").view(d, KW), st.p(pfx + ".depthwise_conv.bias"), z, partial, B,
                                    T, d, sub_lens)
        else:
            ops.glu_dwconv_fwd(y2, st.p(pfx + ".depthwise_conv.weight").view(d, KW), st.p(pfx + ".depthwise_conv.bias"), z, partial, B, T, d)
        mean = _empty((d,), torch.float32, self.dev)
        rstd = _empty((d,), torch.float32, self.dev)
        if bn_mod.momentum is None:  # cumulative moving average: never configured by the reference (conformer_convolution.py:41)
            raise NotImplementedError("BatchNorm1d(momentum=None) is not implemented (the reference uses the default 0.1)")
        ops.bn_finalize(partial, nblk, d, B * T, mean, rstd, bn_mod.running_mean, bn_mod.running_var, bn_mod.num_batches_tracked,
                        training, eps=bn_mod.eps, momentum=bn_mod.momentum)
        a = _empty((B * T, d), self.adt, self.dev)
        ops.bn_swish_fwd(z, mean, rstd, st.p(pfx + ".norm.weight"), st.p(pfx + ".norm.bias"), a)
        out = self.linear(a, None, torch.float32, w=st.w(pfx + ".pointwise_conv2.weight"), bias_t=st.p(pfx + ".pointwise_conv2.bias"), res=x,
                          drop=d_out)
        return NS(out=out, ln=ln, y2=y2, z=z, mean=mean, rstd=rstd, a=a, pfx=pfx, B=B, T=T, d=d, training=training, d_out=d_out)

    def conv_bwd(self, c: NS, dres, dy, nxt=None, want_lo=False):
        st, d, pfx = self.st, c.d, c.pfx
        if not c.training:
            raise RuntimeError("conv-module backward needs batch statistics (module must be in training mode)")
        self.wgrad(dy, c.a, st.gw(pfx + ".pointwise_conv2.weight"))
        da = self.dgrad(dy, st.w(pfx + ".pointwise_conv2.weight"))
        rows = c.B * c.T
        partial = _empty(((rows + 31) // 32, 2, d), torch.float32, self.dev)
        sums = _empty((2, d), torch.float32, self.dev)
        gam, bet = st.p(pfx + ".norm.weight"), st.p(pfx + ".norm.bias")
        ops.bn_swish_bwd_stats(da, c.z, c.mean, c.rstd, gam, bet, partial, sums, st.g(pfx + ".norm.weight"), st.g(pfx + ".norm.bias"))
        dy2 = _empty((rows, 2 * d), self.adt, self.dev)
        wpart = _empty((c.B * ((c.T + 31) // 32), KW + 3, d), torch.float32, self.dev) if d % 4 == 0 else None
        ops.dwconv_glu_bwd(da, c.z, c.y2, c.mean, c.rstd, gam, bet, sums, st.p(pfx + ".depthwise_conv.weight").view(d, KW), dy2,
                           st.g(pfx + ".depthwise_conv.weight").view(d, KW), st.g(pfx + ".depthwise_conv.bias"), c.B, c.T, d,
                           colsum=st.g(pfx + ".pointwise_conv1.bias"), wpartial=wpart)
        self.wgrad(dy2, c.ln.y, st.gw(pfx + ".pointwise_conv1.weight"))
        dln = self.dgrad(dy2, st.w(pfx + ".pointwise_conv1.weight"))
        return self.layernorm_bwd(c.ln, dln, dres, True, nxt, want_lo)

    # ------------------------------------------------------------------------------------------
    # Conv2d subsampling front end (nets/subsampling.py:42-48) + x*sqrt(d) (nets/positional_encoding.py:73)
    # ------------------------------------------------------------------------------------------
    def _conv2_weight(self, pfx, d):
        key = pfx + ".conv.2.weight/khkwc"
        if key not in self.st.derived:  # (o,i,kh,kw) -> (o,kh,kw,i): K index matches the channel-last im2col
            w = _empty((d, 9 * d), self.adt, self.dev)
            ops.permute4d(self.st.p(pfx + ".conv.2.weight"), w, (d, 3, 3, d), (9 * d, 3, 1, 9), (9 * d, 3 * d, d, 1))
            self.st.derived[key] = w
        return self.st.derived[key]

    def _out_weight(self, pfx, d, f2):
        key = pfx + ".out.weight/fc"
        if key not in self.st.derived:  # columns (c*F2 + f) -> (f*d + c)
            w = _empty((d, f2 * d), self.adt, self.dev)
            ops.permute4d(self.st.p(pfx + ".out.weight"), w, (d, f2, d, 1), (f2 * d, 1, f2, 0), (f2 * d, d, 1, 0))
            self.st.derived[key] = w
        return self.st.derived[key]

    def embed_fwd(self, xs, pfx, d, d_out=None) -> NS:
        """d_out: dropout on ``x * sqrt(d)`` (positional_encoding.py:73-75), applied in the output Linear's epilogue."""
        B, T, F = xs.shape
        if self.adt == torch.bfloat16 and ops.planes_supported(d, T, F):
            return self._embed_fwd_planes(xs, pfx, d, d_out)
        T1, F1 = (T - 3) // 2 + 1, (F - 3) // 2 + 1
        T2, F2 = (T1 - 3) // 2 + 1, (F1 - 3) // 2 + 1
        st = self.st
        h1 = _empty((B, T1, F1, d), self.adt, self.dev)
        ops.conv1_fwd(xs, st.p(pfx + ".conv.0.weight").view(d, 9), st.p(pfx + ".conv.0.bias"), h1)
        col = _empty((B * T2 * F2, 9 * d), self.adt, self.dev)
        ops.im2col_s2(h1, col)
        h2 = self.linear(col, None, self.adt, w=self._conv2_weight(pfx, d), bias_t=st.p(pfx + ".conv.2.bias"), act=ACT_RELU)
        h2v = h2.view(B * T2, F2 * d)
        x0 = self.linear(h2v, None, torch.float32, w=self._out_weight(pfx, d, F2), bias_t=st.p(pfx + ".out.bias"), alpha=math.sqrt(d),
                         drop=d_out)
        return NS(out=x0, xs=xs, h1=h1, col=col, h2=h2, B=B, T1=T1, F1=F1, T2=T2, F2=F2, d=d, pfx=pfx, planes=False, d_out=d_out)

    def _embed_fwd_planes(self, xs, pfx, d, d_out=None) -> NS:
        """bf16 mode: conv1 writes parity planes, conv2 runs as an implicit GEMM on them (no im2col matrix); conv2's output keeps
        V = F2 + 1 slots per frame, the output Linear reads the first F2 of them through its row stride."""
        B, T, F = xs.shape
        T1, F1, U, V, T2, F2 = ops.plane_dims(T, F)
        st = self.st
        h1p = _empty((B, 4, U * V, d), self.adt, self.dev)
        ops.conv1_fwd_planes(xs, st.p(pfx + ".conv.0.weight").view(d, 9), st.p(pfx + ".conv.0.bias"), h1p)
        h2p = _empty((B * T2, V * d), self.adt, self.dev)
        ops.conv2_fwd(h1p, self._conv2_weight(pfx, d), st.p(pfx + ".conv.2.bias"), h2p, B, T, F)
        h2v = h2p[:, : F2 * d]
        x0 = self.linear(h2v, None, torch.float32, w=self._out_weight(pfx, d, F2), bias_t=st.p(pfx + ".out.bias"), alpha=math.sqrt(d),
                         drop=d_out)
        return NS(out=x0, xs=xs, h1p=h1p, h2p=h2p, h2v=h2v, B=B, T=T, F=F, T1=T1, F1=F1, U=U, V=V, T2=T2, F2=F2, d=d, pfx=pfx, planes=True,
                  d_out=d_out)

    def embed_bwd(self, c: NS, dy) -> None:
        """dy: operand-dtype gradient wrt the front end's output (out.bias gradient already taken by the producer of dy)."""
        if c.planes:
            return self._embed_bwd_planes(c, dy)
        st, d, pfx = self.st, c.d, c.pfx
        B, T2, F2 = c.B, c.T2, c.F2
        s = math.sqrt(d)
        gwo = torch.empty((d, F2 * d), dtype=torch.float32, device=self.dev)
        ops.zero_(gwo)
        h2v = c.h2.view(B * T2, F2 * d)
        self.wgrad(dy, h2v, gwo, s)
        ops.permute4d(gwo, st.g(pfx + ".out.weight"), (d, F2, d, 1), (F2 * d, d, 1, 0), (F2 * d, 1, F2, 0), accumulate=True)
        # dh2 = s * (dy @ W_out) * relu'(h2): conv2's ReLU backward fused into the dgrad epilogue
        dh2 = self.dgrad(dy, self._out_weight(pfx, d, F2), alpha=s, dact=h2v, act=ACT_RELU).view(B * T2 * F2, d)
        ops.act_bwd(dh2, None, None, st.g(pfx + ".conv.2.bias"), ACT_NONE)
        gw2 = torch.empty((d, 9 * d), dtype=torch.float32, device=self.dev)
        ops.zero_(gw2)
        self.wgrad(dh2, c.col, gw2)
        dcol = self.dgrad(dh2, self._conv2_weight(pfx, d))
        ops.permute4d(gw2, st.g(pfx + ".conv.2.weight"), (d, 3, 3, d), (9 * d, 3 * d, d, 1), (9 * d, 3, 1, 9), accumulate=True)
        dh1 = _empty(c.h1.shape, self.adt, self.dev)
        ops.col2im_s2_relu(dcol, c.h1, dh1)
        ops.conv1_bwd(c.xs, dh1, st.g(pfx + ".conv.0.weight").view(d, 9), st.g(pfx + ".conv.0.bias"))

    def _embed_bwd_planes(self, c: NS, dy) -> None:
        st, d, pfx = self.st, c.d, c.pfx
        B, T2, F2, V = c.B, c.T2, c.F2, c.V
        s = math.sqrt(d)
        gwo = torch.empty((d, F2 * d), dtype=torch.float32, device=self.dev)
        ops.zero_(gwo)
        self.wgrad(dy, c.h2v, gwo, s)
        ops.permute4d(gwo, st.g(pfx + ".out.weight"), (d, F2, d, 1), (F2 * d, d, 1, 0), (F2 * d, 1, F2, 0), accumulate=True)
        # dh2 = s * (dy @ W_out) * relu'(h2) into the padded (B*T2, V*d) layout, conv.2.bias gradient as the epilogue's column sums
        dh2p = _empty((B * T2, V * d), self.adt, self.dev)
        ops.zero_(dh2p)  # the padding slot of every frame must be zero for the implicit GEMMs (one memset; the GEMM fills the rest)
        wo = self._out_weight(pfx, d, F2)
        csum = torch.empty((F2 * d,), dtype=torch.float32, device=self.dev)
        ops.zero_(csum)
        ops.gemm(dy, wo, dh2p, B * T2, F2 * d, d, lda=dy.stride(0), ldb=wo.stride(0), ldc=V * d, tb=True, alpha=s, dact=c.h2v,
                 act=ACT_RELU, colsum=csum)
        # conv.2.bias gradient = the F2 per-slot column sums folded over the slots (column sums of the (F2, d) view)
        ops.act_bwd(csum.view(F2, d), None, None, st.g(pfx + ".conv.2.bias"), ACT_NONE)
        gw2 = torch.empty((d, 9 * d), dtype=torch.float32, device=self.dev)
        ops.zero_(gw2)
        ops.conv2_wgrad(dh2p, c.h1p, gw2, B, c.T, c.F)
        ops.permute4d(gw2, st.g(pfx + ".conv.2.weight"), (d, 3, 3, d), (9 * d, 3 * d, d, 1), (9 * d, 3, 1, 9), accumulate=True)
        dh1p = _empty(c.h1p.shape, self.adt, self.dev)
        ops.conv2_dgrad(dh2p, self._conv2_weight(pfx, d), c.h1p, dh1p, B, c.T, c.F)
        ops.conv1_bwd_planes(c.xs, dh1p, st.g(pfx + ".conv.0.weight").view(d, 9), st.g(pfx + ".conv.0.bias"))

    # ------------------------------------------------------------------------------------------
    # encoder (nets/transformer_encoder.py:107-127; use_rel=True, arch=conformer, activation=swish)
    # ------------------------------------------------------------------------------------------
    def encoder_fwd(self, enc, xs, xlens, training: bool, rng=None, sub_lens=None) -> NS:
        """xs (B,T,F) fp32, xlens (B,) int64 or None (maskless inference call).  Returns ctx with ctx.out (B,T',d) fp32.
        rng: RNG snapshot of this pass (dropout.RngState.begin_pass) -- dropout is applied iff training and rng is given.
        sub_lens (B,) int64 device tensor of sub-sampled lengths T'_b (xlens must be None): per-utterance inference on a padded
        batch -- rows t < T'_b of utterance b equal the maskless batch-1 call on xs[b, :T_b] (attention mask mode 4, the
        length-aware depthwise conv), rows t >= T'_b hold finite values.  Eval only: training keeps the padded-batch semantics."""
        if sub_lens is not None and (training or xlens is not None):
            raise RuntimeError("encoder_fwd: per-utterance lengths are an inference-only, maskless mode (training=False, xlens=None)")
        d, H = enc.h_dim, enc.n_head
        B = xs.shape[0]
        pfx = enc._lasr_prefix
        if not training:
            rng = None
        E, G = DR.NET_ENC, DR.GLOBAL_LAYER
        emb = self.embed_fwd(xs, pfx + "embed", d, DR.drop(rng, E, G, DR.ENC_POS_X, enc.pe.dropout_rate))
        Tp = emb.T2
        enc.pe.ensure(Tp, self.dev)  # extend_pe (positional_encoding.py:40-53): T' may exceed max_len = 5000
        d_pos = DR.drop(rng, E, G, DR.ENC_POS_EMB, enc.pe.dropout_rate)
        if d_pos is None:
            pos = self.to_adt(enc.pe.pe[0, :Tp])  # absolute positions 0..T'-1 (positional_encoding.py:74); contiguous slice
        else:  # ONE dropped pos_emb shared by every layer, as in the reference (transformer_encoder.py:116-124)
            pos = ops.dropout(enc.pe.pe[0, :Tp], _empty((Tp, d), self.adt, self.dev), d_pos)
        x = emb.out
        layers = []
        for i, layer in enumerate(enc.enc_layers):
            lp = f"{pfx}enc_layers.{i}"
            p_out, p_ffm, p_ff = layer.dropout_rate, layer.feed_forward_macaron.dropout_rate, layer.feed_forward.dropout_rate
            c1 = self.ffn_fwd(x, lp + ".feed_forward_macaron_norm", lp + ".feed_forward_macaron", ACT_SWISH, 0.5,
                              DR.drop(rng, E, i, DR.ENC_FFM_INNER, p_ffm), DR.drop(rng, E, i, DR.ENC_FFM_OUT, p_out))
            c2 = self.rel_mha_fwd(c1.out, lp + ".self_attn_norm", lp + ".self_attn", pos, B, Tp, H, xlens,
                                  DR.drop(rng, E, i, DR.ENC_ATT_PROB, layer.self_attn.dropout_rate), DR.drop(rng, E, i, DR.ENC_ATT_OUT, p_out),
                                  sub_lens=sub_lens)
            c3 = self.conv_fwd(c2.out, lp + ".conv_norm", lp + ".conv", B, Tp, layer.conv.norm, training,
                               DR.drop(rng, E, i, DR.ENC_CONV_OUT, p_out), sub_lens=sub_lens)
            c4 = self.ffn_fwd(c3.out, lp + ".feed_forward_norm", lp + ".feed_forward", ACT_SWISH, 0.5,
                              DR.drop(rng, E, i, DR.ENC_FF_INNER, p_ff), DR.drop(rng, E, i, DR.ENC_FF_OUT, p_out))
            c5 = self.layernorm(c4.out, lp + ".final_norm", torch.float32)
            layers.append((c1, c2, c3, c4, c5))
            x = c5.y
        fin = self.layernorm(x, pfx + "after_norm", torch.float32)
        return NS(out=fin.y.view(B, Tp, d), emb=emb, layers=layers, fin=fin, B=B, Tp=Tp, d=d, pfx=pfx)

    def encoder_bwd(self, c: NS, dh: torch.Tensor) -> None:
        dh = dh.contiguous().view(c.B * c.Tp, c.d)
        if dh.dtype != torch.float32:
            raise TypeError("encoder gradient must be fp32")
        st, g = self.st, self.st.g
        dres = _empty(dh.shape, torch.float32, self.dev)
        self.layernorm_bwd(c.fin, dh, dres, accumulate=False)
        hook = st.grad_ready_hook
        if hook is not None:
            hook(*st.range_of(c.pfx + "after_norm."))
        for i in range(len(c.layers) - 1, -1, -1):
            c1, c2, c3, c4, c5 = c.layers[i]
            lp = f"{c.pfx}enc_layers.{i}"
            nxt = _empty(dres.shape, torch.float32, self.dev)
            # every LayerNorm backward also emits the bias gradient of the Linear that closes the block that runs NEXT in
            # backward order (its output gradient is exactly the residual-stream gradient being written) + the bf16 copy
            dy = self.layernorm_bwd(c5, dres, nxt, False, (g(lp + ".feed_forward.fc2.bias"), 0.5, c4.d_out))
            dres = nxt
            dy = self.ffn_bwd(c4, dres, dy, (g(lp + ".conv.pointwise_conv2.bias"), 1.0, c3.d_out))
            dy = self.conv_bwd(c3, dres, dy, (g(lp + ".self_attn.linear_o.bias"), 1.0, c2.d_out))
            dy = self.rel_mha_bwd(c2, dres, dy, (g(lp + ".feed_forward_macaron.fc2.bias"), 0.5, c1.d_out))
            dy = self.ffn_bwd(c1, dres, dy, (g(c.pfx + "embed.out.bias"), math.sqrt(c.d), c.emb.d_out) if i == 0 else None)
            if hook is not None:
                hook(*st.range_of(lp + "."))
        if len(c.layers) == 0:
            if c.emb.d_out is not None:
                dy = ops.dropout(dres, _empty(dres.shape, self.adt, self.dev), c.emb.d_out)
            else:
                dy = self.to_adt(dres)
            ops.act_bwd(dy, None, None, g(c.pfx + "embed.out.bias"), ACT_NONE, math.sqrt(c.d))
        self.embed_bwd(c.emb, dy)
        if hook is not None:
            hook(*st.range_of(c.pfx + "embed."))

    # ------------------------------------------------------------------------------------------
    # CTC head (nets/ctc.py:28-30): logits = ctc_lo(dropout(h)); dropout p must be 0 here
    # ------------------------------------------------------------------------------------------
    def ctc_head_fwd(self, ctc, h_enc, rng=None) -> NS:
        """rng given: ``ctc_lo(F.dropout(h, p))`` -- the reference applies this dropout in train AND eval mode (nets/ctc.py:29,
        quirk Q3), so callers pass an rng whenever they go through ``CTC.forward``; the inference path
        (``CTC.log_softmax``, nets/ctc.py:25-26) has no dropout and passes None."""
        B, Tp, d = h_enc.shape
        drop = DR.drop(rng, DR.NET_CTC, DR.GLOBAL_LAYER, DR.CTC_IN, ctc.dropout_rate)
        h2 = h_enc.reshape(B * Tp, d)
        if drop is None:
            hb = self.to_adt(h2)
        else:  # dropout fused with the fp32 -> operand-dtype cast
            hb = ops.dropout(h2, _empty((B * Tp, d), self.adt, self.dev), drop)
        pfx = ctc._lasr_prefix + "ctc_lo"
        logits = self.linear(hb, pfx, self.adt)
        V = logits.shape[1]
        return NS(out=logits, hb=hb, pfx=pfx, B=B, Tp=Tp, V=V, d=d, drop=drop)

    def ctc_head_bwd(self, c: NS, dlogits, dh32=None) -> torch.Tensor:
        """dlogits (B*T', V) adt view -> dh (B*T', d) fp32 (accumulated into dh32 when given)."""
        if dh32 is None:
            return self.linear_bwd(dlogits, c.hb, c.pfx, dx_dtype=torch.float32, dx_drop=c.drop)
        return self.linear_bwd(dlogits, c.hb, c.pfx, dx_res=dh32, dx_drop=c.drop)

    # ------------------------------------------------------------------------------------------
    # decoder (nets/transformer_decoder.py:70-93, nets/transformer_layer.py:179-221)
    # ------------------------------------------------------------------------------------------
    def decoder_fwd(self, dec, ys, ylens, h_enc, xlens, mem_mask_mode: int = 3, training: bool = False, rng=None) -> NS:
        """ys (B,L) int64 decoder input tokens ([sos | ys], models/u2.py:339-358); ylens (B,) so that key j of the
        self-attention is valid iff j < ylens[b]+1 (and j <= i); h_enc (B,T',d) fp32; xlens raw input lengths or None.
        mem_mask_mode 3: memory key j valid iff 4j < xlens[b] (training: the reference's re-subsampled padding mask);
        1: xlens holds sub-sampled memory lengths directly (batched rescoring of utterances encoded one by one)."""
        B, L = ys.shape
        d, H = dec.h_dim, dec.n_head
        Tp = h_enc.shape[1]
        pfx = dec._lasr_prefix
        V = dec.vocab
        st = self.st
        y = _empty((B * L, d), torch.float32, self.dev)
        dec.pe.ensure(L, self.dev)
        ops.embed_fwd(ys, st.p(pfx + "embed.weight"), dec.pe.pe[0], y, math.sqrt(d))
        if not training:
            rng = None
        D = DR.NET_DEC
        d_pos = DR.drop(rng, D, DR.GLOBAL_LAYER, DR.DEC_POS, dec.pe.dropout_rate)
        if d_pos is not None:  # dropout(embed * sqrt(d) + pe), positional_encoding.py:54-55 (a (B*L, d) tensor: in place)
            ops.dropout(y, y, d_pos)
        mem = self.to_adt(h_enc.reshape(B * Tp, d))
        layers = []
        for i, layer in enumerate(dec.dec_layers):
            lp = f"{pfx}dec_layers.{i}"
            p_out = layer.dropout_rate
            c1 = self.self_mha_fwd(y, lp + ".self_attn_norm", lp + ".self_attn", B, L, H, ylens,
                                   DR.drop(rng, D, i, DR.DEC_SELF_PROB, layer.self_attn.dropout_rate), DR.drop(rng, D, i, DR.DEC_SELF_OUT, p_out))
            c2 = self.src_mha_fwd(c1.out, mem, lp + ".src_attn_norm", lp + ".src_attn", B, L, Tp, H, xlens, mem_mask_mode,
                                  DR.drop(rng, D, i, DR.DEC_SRC_PROB, layer.src_attn.dropout_rate), DR.drop(rng, D, i, DR.DEC_SRC_OUT, p_out))
            c3 = self.ffn_fwd(c2.out, lp + ".feed_forward_norm", lp + ".feed_forward", ACT_RELU, 1.0,
                              DR.drop(rng, D, i, DR.DEC_FF_INNER, layer.feed_forward.dropout_rate), DR.drop(rng, D, i, DR.DEC_FF_OUT, p_out))
            layers.append((c1, c2, c3))
            y = c3.out
        fin = self.layernorm(y, pfx + "after_norm", self.adt)
        logits = self.linear(fin.y, pfx + "linear_out", self.adt)
        return NS(out=logits, ys=ys, layers=layers, fin=fin, mem=mem, B=B, L=L, Tp=Tp, d=d, V=V, pfx=pfx, d_pos=d_pos)

    def decoder_bwd(self, c: NS, dlogits, dmem32: torch.Tensor) -> None:
        """dlogits (B*L, V) adt view; dmem32 (B*T', d) fp32 is accumulated into (memory gradient)."""
        st, g = self.st, self.st.g
        dfin = self.linear_bwd(dlogits, c.fin.y, c.pfx + "linear_out")
        dres = _empty((c.B * c.L, c.d), torch.float32, self.dev)
        n = len(c.layers)
        dy = self.layernorm_bwd(c.fin, dfin, dres, False,
                                (g(f"{c.pfx}dec_layers.{n - 1}.feed_forward.fc2.bias"), 1.0, c.layers[n - 1][2].d_out) if n else None)
        for i in range(n - 1, -1, -1):
            c1, c2, c3 = c.layers[i]
            lp = f"{c.pfx}dec_layers.{i}"
            dy = self.ffn_bwd(c3, dres, dy, (g(lp + ".src_attn.linear_o.bias"), 1.0, c2.d_out))
            dy = self.src_mha_bwd(c2, dres, dy, dmem32, (g(lp + ".self_attn.linear_o.bias"), 1.0, c1.d_out))
            dy = self.self_mha_bwd(c1, dres, dy, (g(f"{c.pfx}dec_layers.{i - 1}.feed_forward.fc2.bias"), 1.0, c.layers[i - 1][2].d_out)
                                   if i > 0 else None)
        if c.d_pos is not None:  # gradient through dropout(embed * sqrt(d) + pe)
            dres = ops.dropout(dres, _empty(dres.shape, torch.float32, self.dev), c.d_pos)
        ops.embed_bwd(c.ys, dres, st.g(c.pfx + "embed.weight"), math.sqrt(c.d))
        if st.grad_ready_hook is not None:
            st.grad_ready_hook(*st.range_of(c.pfx))
