"""GPU: the attention loss (lasr_lsmooth_kl_fwdbwd) and the hybrid loss mix (lasr_hybrid_combine) against float64 references
(oracle.u2_oracle.label_smoothing_kl / attention_targets, criterions/hybrid_ctc_attn.py:49-64,78), element by element.

Bounds (u = 2^-24; V up to 8200 is summed by 256 threads, so a row sum takes at most V/256 + 16 sequential adds):
  row loss : the log-sum-exp is off by e = u (V/256 + 16 + 2 |lse|); the loss by
             4 [e (qt + (V-1) qo) + u (qt |lp_t| + qo (V/256 + 16)(sum |x| + V |lse|)) + 2^-22 (qt |log qt| + eps |log qo| + |ref|)]
  gradient : s (p - q) with p off by p u (2 |x - max| + V/256 + 20) and two more roundings; bf16 adds 2^-8 |ref|.
Ignored rows must be exactly 0, and columns [V, ldg) of the gradient keep their NaN sentinel.
"""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu

U32 = 2.0 ** -24


def _lsmooth_case(B, lmax, V, smoothing, dtype, seed):
    from liteasr_b200 import ops
    from oracle.u2_oracle import attention_targets, label_smoothing_kl
    g = torch.Generator().manual_seed(seed)
    rows = B * (lmax + 1)
    ld = (V + 7) // 8 * 8 + 8
    ylens = torch.randint(1, lmax, (B,), generator=g)
    ylens[0], ylens[1] = 0, lmax                                    # an utterance with no tokens (eos only) and a full one
    ys = torch.randint(0, V - 1, (B, lmax), generator=g)
    ys[torch.arange(lmax)[None, :] >= ylens[:, None]] = -1          # the reference's padding
    logits = torch.full((rows, ld), float("nan"), dtype=dtype)     # padding columns are never read
    logits[:, :V] = (torch.randn(rows, V, generator=g) * 3).to(dtype)
    grad_scale, up = 0.37, 1.9
    dl = logits.cuda()
    grad = torch.full((rows, ld), float("nan"), device="cuda", dtype=dtype)
    row_loss = torch.full((rows,), float("nan"), device="cuda")
    upstream = torch.tensor([up], device="cuda")
    ops.lsmooth_kl_fwdbwd(dl, ys.cuda(), ylens.cuda(), V, smoothing, grad_scale, upstream, row_loss, grad)
    loss, gr = row_loss.double().cpu(), grad.double().cpu()

    tgt = attention_targets(ys, ylens, V).reshape(-1)              # eos (V-1) at l == ylens[b], -1 beyond
    x = logits[:, :V].double().requires_grad_(True)
    per_row = torch.stack([label_smoothing_kl(x[r:r + 1], tgt[r:r + 1], smoothing) for r in range(rows)])
    s = float(torch.tensor(grad_scale, dtype=torch.float32) * torch.tensor(up, dtype=torch.float32))   # the kernel's fp32 factor
    (gref,) = torch.autograd.grad(per_row.sum() * s, x)
    ign = tgt == -1
    assert ign.any() and (~ign).any()

    # loss
    xd = x.detach()
    lse = torch.logsumexp(xd, 1)
    qo = smoothing / (V - 1)
    qt = 1.0 - smoothing
    lpt = (xd.gather(1, tgt.clamp(min=0)[:, None])[:, 0] - lse).abs()
    nred = V / 256 + 16
    e = U32 * (nred + 2 * lse.abs())
    xlogx = lambda q: abs(q * math.log(q)) if q > 0 else 0.0  # noqa: E731
    bound = 4 * (e * (qt + (V - 1) * qo) + U32 * (qt * lpt + qo * nred * (xd.abs().sum(1) + V * lse.abs()))
                 + 2.0 ** -22 * (xlogx(qt) + (V - 1) * xlogx(qo) + per_row.detach().abs()))
    assert not torch.isnan(loss).any()
    assert (loss[ign] == 0).all(), "ignored rows must have loss exactly 0"
    err = (loss - per_row.detach()).abs()
    assert (err[~ign] <= bound[~ign]).all(), f"row loss: worst excess {float((err - bound)[~ign].max()):.3g}"

    # gradient
    p = torch.softmax(xd, 1)
    gb = abs(s) * (p * U32 * (2 * (xd - xd.max(1, keepdim=True).values).abs() + nred + 20) + 3 * U32 * (gref.abs() / abs(s)))
    if dtype == torch.bfloat16:
        gb = gb + 2.0 ** -8 * (gref.abs() + gb)
    assert not torch.isnan(gr[:, :V]).any(), "gradient element left unwritten"
    assert (gr[ign, :V] == 0).all(), "ignored rows must have a zero gradient"
    gerr = (gr[:, :V] - gref).abs()
    assert (gerr <= gb).all(), f"gradient: worst excess {float((gerr - gb).max()):.3g}"
    assert torch.isnan(gr[:, V:]).all(), "gradient columns [V, ldg) must keep their contents"
    # the eos row of the utterance without tokens targets V-1: the only negative gradient entry at smoothing 0
    if smoothing == 0.0:
        assert int(gr[0, :V].argmin()) == V - 1


@pytest.mark.parametrize("V", [37, 256, 257, 4233, 5000, 8200])
@pytest.mark.parametrize("smoothing", [0.0, 0.1])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_lsmooth_kl_fwdbwd(V, smoothing, dtype):
    """Per-row loss and gradient of the label-smoothed KL, targets built on the fly from ys / ylens (eos at l == ylens[b],
    ignored beyond), padded row buffer ld = ceil(V, 8) + 8, grad_scale != 1 and a device upstream scalar."""
    _lsmooth_case(4, 6, V, smoothing, dtype, seed=V + int(smoothing * 10))


@pytest.mark.parametrize("ctc_weight", [0.0, 0.3, 1.0])
def test_hybrid_combine(ctc_weight):
    """out = {w lc + (1-w) la, lc, la}, lc = sum(nll)/B, la = sum(row_kl)/B with B and M > 256 (several trips per thread)."""
    from liteasr_b200 import ops
    g = torch.Generator().manual_seed(7)
    B, M = 300, 300 * 7 + 11
    nll = torch.rand(B, generator=g) * 200
    kl = torch.rand(M, generator=g) * 30
    kl[::5] = 0.0                                                   # ignored rows
    out = torch.full((3,), float("nan"), device="cuda")
    ops.hybrid_combine(nll.cuda(), kl.cuda(), ctc_weight, out)
    o = out.double().cpu()
    w = float(torch.tensor(ctc_weight, dtype=torch.float32))
    lc, la = nll.double().sum() / B, kl.double().sum() / B
    # fp32 sums: at most ceil(n/256) + 10 sequential adds, then the division and the mix
    bc = U32 * (math.ceil(B / 256) + 12) * lc
    ba = U32 * (math.ceil(M / 256) + 12) * la
    assert abs(o[1] - lc) <= bc and abs(o[2] - la) <= ba
    ref = w * lc + (1 - w) * la
    assert abs(o[0] - ref) <= w * bc + (1 - w) * ba + 4 * U32 * (w * lc + (1 - w) * la)
    if ctc_weight == 0.3:   # zero_infinity = False: an infeasible utterance makes the CTC term and the loss +inf
        nll[17] = float("inf")
        ops.hybrid_combine(nll.cuda(), kl.cuda(), ctc_weight, out)
        o = out.double().cpu()
        assert o[0] == math.inf and o[1] == math.inf and abs(o[2] - la) <= ba
