"""Inference side of the path (models/u2.py:221-317 of the reference, driven per utterance by infer.py:97-120).

* ``greedy_ctc``              argmax_v log_softmax(ctc_lo(encoder(x))) -> collapse repeats -> drop blank (batched; defined from
                              nets/ctc.py:25-26, the reference itself ships no greedy decoder).
* ``ctc_prefix_beam_search``  models/u2.py:221-261: maskless eval-mode encoder on ONE utterance, per-frame top-``beam`` prune on
                              the GPU (``lasr_logsoftmax_topk``), the dictionary search itself on the host in float64 with the
                              reference's operation order (``lasr_ctc_prefix_beam_search``).
* ``attention_rescore``       models/u2.py:269-317: one decoder pass over the padded n-best, the (beam, L, V) log-softmax is never
                              materialised (row log-sum-exp + ``lasr_gather_logp``), scores summed left to right in fp32.
* ``decode_batch``            a padded batch in ONE encoder pass with per-utterance semantics (attention mask mode 4 and the
                              length-aware depthwise conv: every valid row equals the maskless batch-1 call on the utterance cut
                              to its length), one top-K over all rows, the prefix search for every utterance in one device launch
                              (``lasr_ctc_prefix_beam_search_batch``), one copy of the n-best to the host, ONE decoder pass
                              rescoring every n-best of every utterance (memory masked by its sub-sampled length).
* ``inference_batch``         a list of utterances through the same encoder pass and top-K, with the host search per utterance:
                              token- and score-identical to calling ``attention_rescore`` one by one.
* ``align``                   CTC Viterbi forced alignment of known transcripts on the same encoder pass: the most likely CTC
                              path per utterance in one device launch (``lasr_ctc_forced_align``), token spans in frames and
                              seconds (defined from nets/ctc.py:25-26; the reference ships no aligner).
* ``transcribe``              raw audio in: Kaldi-compatible log-mel features on the device (``features.fbank``, one launch),
                              then ``decode_batch``.

``greedy_ctc(xs, xlens)`` keeps the reference's padded-batch semantics (mask mode 3, the padded rows inside the depthwise conv
window), so its tokens can differ from those of a batch-1 call; ``decode_batch(...)["greedy"]`` has per-utterance semantics and
equals ``greedy_ctc(x_b, None)`` on each utterance.

Everything runs under ``torch.no_grad()`` on the hand-written CUDA kernels; there is no CPU fallback.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch
from torch import Tensor

from . import functions as F
from . import ops
from .features import FbankConfig
from .features import fbank as _fbank

BEAM = 10          # models/u2.py:223 (hard-coded in the reference)
CTC_WEIGHT = 0.5   # models/u2.py:312


def log_softmax(logits: Tensor) -> Tensor:
    """(…, V) logits (fp32 or bf16, last-dim stride 1) -> fp32 log-probabilities (nets/ctc.py:25-26)."""
    V = logits.shape[-1]
    x2 = logits.reshape(-1, V) if logits.is_contiguous() else logits.flatten(0, -2)
    _, _, _, full = ops.logsoftmax_topk(x2, 0, vocab=V, want_full=True)
    return full.view(*logits.shape[:-1], V)


def _encode(model, xs: Tensor, xlens: Optional[Tensor]):
    """Eval-mode encoder + CTC head -> (h_enc (B,T',d) fp32, logits 2-D view (B*T', >=V), T')."""
    st, eng, _ = F.bind(model, xs.device)
    F.bind(model.encoder, xs.device)
    F.bind(model.ctc, xs.device)
    st.refresh_operands(force=True)
    enc = eng.encoder_fwd(model.encoder, xs.contiguous().float(), xlens, False)
    head = eng.ctc_head_fwd(model.ctc, enc.out)
    return enc.out, head.out, enc.Tp


def _greedy_rows(ids, n: int, blank: int) -> List[int]:
    """Frame ids -> greedy CTC tokens: the first n frames, repeats collapsed, blanks dropped."""
    row = ids[:n]
    keep = np.ones(len(row), dtype=bool)
    keep[1:] = row[1:] != row[:-1]
    keep &= row != blank
    return [int(v) for v in row[keep]]


@torch.no_grad()
def greedy_ctc(model, xs: Tensor, xlens: Optional[Tensor] = None) -> Tuple[List[List[int]], Tensor]:
    """xs (B,T,F); xlens (B,) or None (maskless, every frame decoded).  -> (token lists, frame ids (B,T') int32)."""
    if model.training:
        raise RuntimeError("greedy_ctc runs on the BatchNorm running statistics: call model.eval() first")
    h, logits, Tp = _encode(model, xs, xlens)
    B = xs.shape[0]
    _, idx, _, _ = ops.logsoftmax_topk(logits, 1, vocab=model.vocab_size)
    ids = idx.view(B, Tp)
    host = ids.cpu().numpy()
    n = [Tp] * B if xlens is None else [int(v) for v in model.get_pred_len(xlens.cpu())]
    return [_greedy_rows(host[b], n[b], model.blank) for b in range(B)], ids


@torch.no_grad()
def _prefix_search(model, x: Tensor, beam: int = BEAM):
    """-> (hyps [(prefix tuple, score)], h_enc (1,T',d))."""
    if model.training:
        raise RuntimeError("inference runs on the BatchNorm running statistics: call model.eval() first")
    assert x.dim() == 3 and x.size(0) == 1, "the reference decodes one utterance at a time (infer.py:97-120)"
    h, logits, Tp = _encode(model, x, None)
    k = min(beam, model.vocab_size)
    tv, ti, _, _ = ops.logsoftmax_topk(logits, k, vocab=model.vocab_size)
    hyps = ops.ctc_prefix_beam_search_host(tv.cpu().numpy(), ti.cpu().numpy(), beam=beam, blank=model.blank)
    return hyps, h


def ctc_prefix_beam_search(model, x: Tensor, beam: int = BEAM):
    """models/u2.py:221-261 -> (hyps, h) like the reference's ``_ctc_prefix_beam_search``."""
    return _prefix_search(model, x, beam)


@torch.no_grad()
def _rescore(model, nbest: Sequence[Sequence[Tuple[tuple, float]]], mem: Tensor, mlens: Optional[Tensor]):
    """One decoder pass over every hypothesis of every utterance.  nbest[u] = [(prefix, ctc score)]; mem (n,T',d) fp32 holds the
    encoder output each of the n hypotheses attends to, mlens (n,) its key lengths (None: every key, memory_mask=None as in
    models/u2.py:297).  -> per utterance (best index, [scores])."""
    dev = mem.device
    st, eng, _ = F.bind(model, dev)
    F.bind(model.decoder, dev)
    flat = [(u, hy) for u, hyps in enumerate(nbest) for hy in hyps]
    n = len(flat)
    lmax = max(len(hy[0]) for _, hy in flat)
    toks = np.full((n, lmax + 1), model.eos, dtype=np.int64)      # [sos | hyp | eos padding]  (models/u2.py:346-353)
    toks[:, 0] = model.sos
    look = np.full((n, lmax + 1), -1, dtype=np.int64)             # class looked up at each position (-1 = none)
    ylens = np.zeros(n, dtype=np.int64)
    for i, (_, hy) in enumerate(flat):
        L = len(hy[0])
        ylens[i] = L
        if L:
            toks[i, 1:L + 1] = hy[0]
            look[i, :L] = hy[0]
        look[i, L] = model.eos
    model.decoder.pe.ensure(lmax + 1, dev)
    c = eng.decoder_fwd(model.decoder, torch.from_numpy(toks).to(dev), torch.from_numpy(ylens).to(dev), mem, mlens, mem_mask_mode=1)
    V = model.vocab_size
    _, _, lse, _ = ops.logsoftmax_topk(c.out, 0, vocab=V, want_lse=True)
    lp = ops.gather_logp(c.out, lse, torch.from_numpy(look.reshape(-1)).to(dev), V).view(n, lmax + 1).cpu().numpy()
    out, i = [], 0
    for hyps in nbest:
        best_score, best_index, scores = -float("inf"), 0, []
        for j, hy in enumerate(hyps):
            s = np.float32(0.0)
            for t in range(len(hy[0]) + 1):                       # left-to-right fp32 sum like `score += attn_score[i][j][w]`
                s = np.float32(s + lp[i, t])
            s = np.float32(s + np.float32(hy[1] * CTC_WEIGHT))
            scores.append(float(s))
            if s > best_score:
                best_score, best_index = s, j
            i += 1
        out.append((best_index, scores))
    return out


def attention_rescore(model, x: Tensor, beam: int = BEAM, return_details: bool = False):
    """models/u2.py:269-317 for one utterance x (1,T,F) -> best hypothesis (list of token ids)."""
    hyps, h = _prefix_search(model, x, beam)
    (best, scores), = _rescore(model, [hyps], h.expand(len(hyps), -1, -1).contiguous(), None)  # h.repeat(len(hyps), 1, 1) (u2.py:273)
    if return_details:
        return dict(best=list(hyps[best][0]), hyps=hyps, scores=scores)
    return list(hyps[best][0])


@torch.no_grad()
def _ragged_encode(model, xs: Tensor, xlens):
    """Per-utterance encoder pass over a padded batch + the CTC head.
    -> (h (B,T'max,d) fp32, CTC logits (B*T'max, >=V) 2-D view, T'_b list, T'_b device tensor, T'max)."""
    if model.training:
        raise RuntimeError("inference runs on the BatchNorm running statistics: call model.eval() first")
    if xs.dim() != 3:
        raise ValueError("xs must be a padded batch (B, T, F)")
    B, T = xs.shape[0], xs.shape[1]
    lens = [int(v) for v in torch.as_tensor(xlens).reshape(-1).cpu()]
    if len(lens) != B:
        raise ValueError(f"xlens has {len(lens)} entries for a batch of {B}")
    for n in lens:
        if n > T:
            raise ValueError(f"xlens holds {n} frames, more than the {T} of the padded batch")
        if n < 7:
            raise ValueError(f"an utterance of {n} frames has no frame after sub-sampling (needs >= 7)")
    tps = [int(model.get_pred_len(n)) for n in lens]
    dev = xs.device
    sub = torch.tensor(tps, dtype=torch.int64).to(dev)
    st, eng, _ = F.bind(model, dev)
    F.bind(model.encoder, dev)
    F.bind(model.ctc, dev)
    st.refresh_operands(force=True)
    enc = eng.encoder_fwd(model.encoder, xs.contiguous().float(), None, False, sub_lens=sub)
    head = eng.ctc_head_fwd(model.ctc, enc.out)
    return enc.out, head.out, tps, sub, enc.Tp


@torch.no_grad()
def _ragged_topk(model, xs: Tensor, xlens, beam: int, want_lse: bool = False):
    """``_ragged_encode`` + one top-K over every row (and, with want_lse, the row log-sum-exp from the same launch).
    -> (h (B,T'max,d) fp32, top_val / top_idx (B*T'max, K), T'_b list, T'_b device tensor, T'max, CTC logits, lse or None)."""
    h, logits, tps, sub, Tp = _ragged_encode(model, xs, xlens)
    k = min(beam, model.vocab_size)
    tv, ti, lse, _ = ops.logsoftmax_topk(logits, k, vocab=model.vocab_size, want_lse=want_lse)
    return h, tv, ti, tps, sub, Tp, logits, lse


@torch.no_grad()
def _rescore_padded(model, nbest, h: Tensor, tps: Sequence[int]):
    """``_rescore`` with the padded encoder output as memory: hypothesis i of utterance u reads h[u], keys j < T'_u."""
    dev = h.device
    utt = [u for u, hyps in enumerate(nbest) for _ in hyps]
    idx = torch.tensor(utt, dtype=torch.int64).to(dev)
    return _rescore(model, nbest, h.index_select(0, idx), torch.tensor([tps[u] for u in utt], dtype=torch.int64).to(dev))


def decode_batch(model, xs: Tensor, xlens, beam: int = BEAM, timestamps: bool = False, frame_shift: float = 0.01):
    """Decode a padded batch xs (B,T,F) fp32 with lengths xlens (B,): the batch-1 inference of every utterance (models/u2.py:
    221-317 on xs[b, :xlens[b]]) in one encoder pass, one top-K, one device prefix search and one decoder pass.
    -> one dict per utterance: ``best`` (token list), ``hyps`` [(prefix tuple, CTC score)], ``scores`` (rescoring scores) and
    ``greedy`` (greedy CTC tokens of the same rows, = ``greedy_ctc(x_b, None)``).  CTC scores are float64 with CUDA's exp / log:
    they may differ from the host search's in the last bits (see ``lasr_ctc_prefix_beam_search_batch``).
    ``timestamps=True`` adds ``timestamps``: ``align``'s ``tokens`` for ``best`` (token, first frame, last frame, start s, end s
    at ``frame_shift`` seconds per input frame), from the same encoder pass and CTC logits (one more device launch); the other
    keys do not change.
    Raises RuntimeError in training mode, ValueError for an utterance shorter than 7 frames or longer than T."""
    h, tv, ti, tps, sub, Tp, logits, lse = _ragged_topk(model, xs, xlens, beam, want_lse=timestamps)
    toks, lens, scores, count = ops.ctc_prefix_beam_search_batch(tv, ti, sub, Tp, beam=beam, blank=model.blank)
    toks, lens, scores, count, top1 = (t.cpu().numpy() for t in (toks, lens, scores, count, ti[:, 0].view(-1, Tp)))
    nbest = [[(tuple(int(x) for x in toks[b, i, : lens[b, i]]), float(scores[b, i])) for i in range(count[b])] for b in range(len(tps))]
    res = _rescore_padded(model, nbest, h, tps)
    out = [dict(best=list(hy[bi][0]), hyps=hy, scores=sc, greedy=_greedy_rows(top1[b], tps[b], model.blank))
           for b, (hy, (bi, sc)) in enumerate(zip(nbest, res))]
    if timestamps:
        best = [o["best"] for o in out]
        ys = np.full((len(best), max(len(b) for b in best)), -1, dtype=np.int64)
        for b, hy in enumerate(best):
            ys[b, : len(hy)] = hy
        al = _align_rows(model, logits, lse, ys, [len(b) for b in best], sub, tps, Tp, frame_shift)
        for o, a in zip(out, al):
            o["timestamps"] = a["tokens"]
    return out


def transcribe(model, waves, nsamp=None, cfg: FbankConfig = FbankConfig(), beam: int = BEAM, timestamps: bool = False):
    """Decode raw audio: ``features.fbank(waves, nsamp, cfg)`` (Kaldi-compatible log-mel features in one device launch; waves a
    padded (B, Nmax) CUDA int16 / fp32 tensor in int16 scale with lengths nsamp, or a list of 1-D CUDA tensors), then
    ``decode_batch`` on the features.  -> what ``decode_batch`` returns; with ``timestamps=True`` the seconds use
    ``cfg.frame_shift``.
    Raises ValueError when cfg.num_mel_bins differs from the encoder's input size or an utterance gives fewer than 7 feature
    frames, and what ``features.fbank`` and ``decode_batch`` raise."""
    if cfg.num_mel_bins != model.encoder.i_dim:
        raise ValueError(f"cfg.num_mel_bins = {cfg.num_mel_bins}, but the encoder takes {model.encoder.i_dim} features per frame")
    feats, flens = _fbank(waves, nsamp, cfg)
    fl = flens.cpu()
    for b, f in enumerate(fl.tolist()):
        if f < 7:
            raise ValueError(f"utterance {b} gives {f} feature frames; the encoder needs >= 7 "
                             f"({cfg.frame_length + 6 * cfg.frame_shift:g} ms of audio)")
    return decode_batch(model, feats, fl, beam=beam, timestamps=timestamps, frame_shift=cfg.frame_shift / 1000)


# ----------------------------------------------------------------------------------------------
# forced alignment
# ----------------------------------------------------------------------------------------------
SUBSAMPLE = 4          # input frames per encoder frame (nets/subsampling.py: two stride-2 convolutions)
MAX_ALIGN_LABELS = 16383


def span_seconds(first: int, last: int, frame_shift: float = 0.01) -> Tuple[float, float]:
    """Encoder frames [first, last] -> (start, end) in seconds: encoder frame t stands for input frames [4t, 4t + 4), so
    start = 4 * first * frame_shift and end = 4 * (last + 1) * frame_shift."""
    return SUBSAMPLE * first * frame_shift, SUBSAMPLE * (last + 1) * frame_shift


def _align_rows(model, logits: Tensor, lse: Tensor, ys: np.ndarray, ylens: Sequence[int], sub: Tensor, tps: Sequence[int], Tp: int,
                frame_shift: float):
    """Forced alignment of the ragged CTC logits against host targets ys (B, Lmax) int64 padded -1 -> one dict per utterance."""
    dev = logits.device
    state, _, score, spans = ops.ctc_forced_align(logits, lse, torch.from_numpy(ys).to(dev), torch.tensor(list(ylens), dtype=torch.int64).to(dev),
                                                  sub, Tp, model.blank, vocab=model.vocab_size)
    state, score, spans = state.cpu().numpy(), score.cpu().numpy(), spans.cpu().numpy()
    out = []
    for b, (L, T) in enumerate(zip(ylens, tps)):
        sc = float(score[b])
        if sc == -np.inf:
            out.append(dict(score=sc, path=[], tokens=[]))
            continue
        st = state[b, :T].astype(np.int64)
        y = ys[b, :L]
        path = np.full(T, model.blank, dtype=np.int64)
        odd = (st & 1) == 1
        path[odd] = y[st[odd] >> 1]
        toks = [(tok, f0, f1, *span_seconds(f0, f1, frame_shift)) for tok, (f0, f1) in zip(y.tolist(), spans[b, :L].tolist())]
        out.append(dict(score=sc, path=path.tolist(), tokens=toks))
    return out


def align(model, xs: Tensor, xlens, ys, ylens, frame_shift: float = 0.01):
    """CTC Viterbi forced alignment of known transcripts (include/lasr_align.h): the single most likely CTC path of each
    transcript over log_softmax(ctc_lo(encoder(x))) (nets/ctc.py:25-26; the reference ships no aligner, this definition is
    ours).  xs (B,T,F) fp32 padded with lengths xlens (B,); ys (B,Lmax) int64 padded -1 with lengths ylens (B,): the training
    batch contract.  The encoder pass is ``decode_batch``'s (per-utterance semantics), so each result equals ``align`` on the
    utterance alone.
    -> one dict per utterance: ``score`` (float, the path's summed fp32 log-probability; -inf when the T'_b encoder frames
    cannot hold the transcript: T'_b < L + the number of adjacent repeated tokens), ``path`` (T'_b token ids, the blank id on
    blank frames; [] when infeasible) and ``tokens`` [(token, first frame, last frame, start s, end s)] ([] when infeasible).
    Frames are encoder frames: frame t covers input frames [4t, 4t + 4) at ``frame_shift`` seconds each, so start_s =
    4 * first * frame_shift and end_s = 4 * (last + 1) * frame_shift.
    Raises RuntimeError in training mode; ValueError for an utterance shorter than 7 frames or longer than T, a token that is
    blank, negative or >= V, a transcript longer than 16383 tokens, or ylens larger than Lmax."""
    if model.training:
        raise RuntimeError("inference runs on the BatchNorm running statistics: call model.eval() first")
    y = torch.as_tensor(ys).cpu()
    if y.dim() != 2 or y.dtype != torch.int64:
        raise ValueError("ys must be a padded (B, Lmax) int64 batch")
    y = y.numpy()
    lens = [int(v) for v in torch.as_tensor(ylens).reshape(-1).cpu()]
    if len(lens) != y.shape[0] or y.shape[0] != xs.shape[0]:
        raise ValueError(f"ys / ylens hold {y.shape[0]} / {len(lens)} transcripts for a batch of {xs.shape[0]}")
    V = model.vocab_size
    for b, L in enumerate(lens):
        if L < 0 or L > y.shape[1]:
            raise ValueError(f"ylens[{b}] = {L} outside [0, Lmax = {y.shape[1]}]")
        if L > MAX_ALIGN_LABELS:
            raise ValueError(f"a transcript of {L} tokens exceeds the aligner's limit of {MAX_ALIGN_LABELS}")
        row = y[b, :L]
        bad = (row < 0) | (row >= V) | (row == model.blank)
        if bad.any():
            raise ValueError(f"ys[{b}] holds token {int(row[bad][0])}: tokens must lie in [0, {V}) and differ from blank {model.blank}")
    _, logits, tps, sub, Tp = _ragged_encode(model, xs, xlens)
    _, _, lse, _ = ops.logsoftmax_topk(logits, 0, vocab=V, want_lse=True)
    return _align_rows(model, logits, lse, np.ascontiguousarray(y[:, : max(lens, default=0)]), lens, sub, tps, Tp, frame_shift)


def inference_batch(model, xs_list: Sequence[Tensor], beam: int = BEAM, return_details: bool = False):
    """Decode a list of utterances (each (T_u,F) or (1,T_u,F)); token-identical to calling ``attention_rescore`` one by one.
    The utterances share one per-utterance encoder pass and one top-K; the prefix search runs on the host per utterance, so
    that the CTC scores are bit-identical to the batch-1 path's (``decode_batch`` runs it on the device instead)."""
    utts = [x[0] if x.dim() == 3 else x for x in xs_list]
    lens = [u.shape[0] for u in utts]
    xs = torch.zeros((len(utts), max(lens), utts[0].shape[1]), dtype=torch.float32, device=utts[0].device)
    for i, u in enumerate(utts):
        xs[i, : lens[i]] = u
    h, tv, ti, tps, _, Tp, _, _ = _ragged_topk(model, xs, torch.tensor(lens), beam)
    tv, ti = tv.view(len(utts), Tp, -1).cpu().numpy(), ti.view(len(utts), Tp, -1).cpu().numpy()
    nbest = [ops.ctc_prefix_beam_search_host(tv[b, : tps[b]], ti[b, : tps[b]], beam=beam, blank=model.blank) for b in range(len(utts))]
    res = _rescore_padded(model, nbest, h, tps)
    if return_details:
        return [dict(best=list(h[b][0]), hyps=h, scores=s) for h, (b, s) in zip(nbest, res)]
    return [list(h[b][0]) for h, (b, _) in zip(nbest, res)]
