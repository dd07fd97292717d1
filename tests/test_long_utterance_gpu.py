"""GPU: whole-model runs on utterances longer than 41 s (T' > 1024 sub-sampled frames), where every attention -- encoder
self-attention, decoder source attention and, for long hypotheses, decoder self-attention -- takes the CTA-per-row softmax
kernels of csrc/attention.cu.  A 2-layer d256 model (the D256_2L dims of tests/test_batch_decode_gpu.py), synthetic weights.

Tolerances (the float64 oracle, oracle/u2_oracle.py, evaluated on the GPU as in tests/test_full_shape_gpu.py):
  training step, fp32 mode : loss rel 1e-5; whole-gradient rel-L2 1e-4 with ctc_weight 0 (the attention loss alone: both
                             encoder and decoder attentions past 1024 keys, forward and backward).  With ctc_weight 0.3 the
                             CTC gradient carries the T-dependent fp32 error of the log-domain lattice (DESIGN §2.1: abs error
                             per logit up to 2e-6 T', 4.2e-3 at T' = 2100; whole-gradient rel-L2 measured 7.3e-4), bound 3e-3
  training step, bf16 mode : loss rel 3e-3, whole-gradient rel-L2 3e-2 (ctc_weight 0.3)
  decoder forward (fp32, eval, L + 1 = 1100): max-abs error of the logits <= 1e-4 * max|ref|
  decode_batch: fp32 encoder rows of utterances with T'_b > 1024 are bit-identical to the batch-1 call (both take the wide kernels,
  whose results do not depend on the row width); rows with T'_b <= 1024 < T'max run the warp kernels in the batch-1 call and the
  wide ones in the batch: max-abs difference <= 2e-2 of max|h| (as for the fused / unfused pair, DESIGN §4.11)."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

D256_2L = dict(input_dim=80, vocab_size=300, enc_dim=256, enc_ff_dim=1024, enc_attn_heads=4, enc_layers=2, dec_dim=256, dec_ff_dim=1024,
               dec_attn_heads=4, dec_layers=1)
SEED, SM = 11, 0.1


def _frames_for(tp):
    """Input frames whose sub-sampled length is tp: ((T-1)//2-1)//2 == tp for T = 4 tp + 3."""
    return 4 * tp + 3


def _sd():
    from liteasr_b200.schema import U2Dims
    from liteasr_b200.utils.synthetic import synth_state_dict
    return synth_state_dict(U2Dims(**D256_2L), seed=SEED)


def _model(precision, train=False):
    from liteasr_b200.models.u2 import U2, U2Config
    model = U2(U2Config(**{**D256_2L, "precision": precision}))
    model.load_state_dict(_sd())
    model = model.cuda()
    return model.train() if train else model.eval()


def _sd_on_gpu(sd, dtype, grad):
    return {k: (v.to(dtype).cuda().requires_grad_(grad) if v.is_floating_point() and "running" not in k and ".pe.pe" not in k
                else (v.to(dtype).cuda() if v.is_floating_point() else v.cuda())) for k, v in sd.items()}


def _train_batch():
    """Two utterances, T' = 1100 and 2100 (44 s and 84 s), 60 / 120 labels."""
    g = torch.Generator().manual_seed(7)
    tps = [2100, 1100]
    xlens = torch.tensor([_frames_for(t) for t in tps])
    T = int(xlens.max())
    xs = torch.randn(2, T, 80, generator=g) * (torch.arange(T).view(1, -1, 1) < xlens.view(-1, 1, 1))
    ylens = torch.tensor([120, 60])
    ys = torch.full((2, 120), -1, dtype=torch.int64)
    for b, L in enumerate(ylens.tolist()):
        ys[b, :L] = torch.randint(1, D256_2L["vocab_size"] - 1, (L,), generator=g)
    return xs, xlens, ys, ylens


@pytest.fixture(scope="module")
def oracle_step():
    """The oracle's attention loss and CTC loss of the batch and the gradient of each, in float64 on the GPU."""
    from oracle import u2_oracle as O
    xs, xlens, ys, ylens = (t.cuda() for t in _train_batch())
    sd64 = _sd_on_gpu(_sd(), torch.float64, True)
    cfg = O.U2Shape(**D256_2L)
    with torch.device("cuda"):
        h_attn, h_ctc, _ = O.u2_forward(sd64, cfg, xs.double(), xlens, ys, ylens, True, {}, None)
        la = O.label_smoothing_kl(h_attn, O.attention_targets(ys, ylens, cfg.vocab_size), SM) / 2
        lp = torch.log_softmax(h_ctc.transpose(0, 1), dim=-1)
        lc = torch.nn.functional.ctc_loss(lp, ys.clamp(min=0), O.subsampled_len(xlens), ylens, blank=0, reduction="sum") / 2
        names = [k for k, v in sd64.items() if v.requires_grad]
        params = [sd64[k] for k in names]
        ga = torch.autograd.grad(la, params, retain_graph=True, allow_unused=True)
        gc = torch.autograd.grad(lc, params, allow_unused=True)
    zero = lambda p, g: torch.zeros_like(p) if g is None else g
    return (float(la.detach()), float(lc.detach()), {n: zero(p, g) for n, p, g in zip(names, params, ga)},
            {n: zero(p, g) for n, p, g in zip(names, params, gc)})


@pytest.mark.parametrize("precision,W", [("fp32", 0.0), ("fp32", 0.3), ("bf16", 0.3)])
def test_long_training_step_matches_float64_oracle(oracle_step, precision, W):
    """A batch of two utterances, T' = 2100 and 1100, through HybridCTCLoss.direct_step (the fused forward + hand-written
    backward) against the float64 oracle."""
    from liteasr_b200.criterions.hybrid_ctc_attn import HybridCTCLoss, HybridCTCLossConfig
    from liteasr_b200.trainer import TrainStep
    la, lc, ga, gc = oracle_step
    ref_loss = W * lc + (1 - W) * la
    model = _model(precision, train=True)
    crit = HybridCTCLoss(HybridCTCLossConfig(vocab_size=D256_2L["vocab_size"], smoothing=SM, ctc_weight=W))
    step = TrainStep(model, crit, use_graph=False, device=torch.device("cuda:0"))
    step.store.zero_grads()
    loss = crit.direct_step(model, *(t.cuda() for t in _train_batch()))
    assert loss is not None, "the fused step did not take the direct path"
    torch.cuda.synchronize()
    num = den = 0.0
    for n, p in model.named_parameters():
        got = p.grad.double()
        assert torch.isfinite(got).all(), n
        want = W * gc[n] + (1 - W) * ga[n]
        num += float((got - want).pow(2).sum())
        den += float(want.pow(2).sum())
    rel = math.sqrt(num / den)
    print(f"\n{precision}, ctc_weight {W}, T' = 2100 / 1100: loss {float(loss):.7f} vs {ref_loss:.7f}, gradient rel-L2 {rel:.3e}")
    if precision == "fp32":
        assert math.isclose(float(loss), ref_loss, rel_tol=1e-5)
        assert rel <= (1e-4 if W == 0 else 3e-3)
    else:
        assert math.isclose(float(loss), ref_loss, rel_tol=3e-3)
        assert rel <= 3e-2


def test_long_decoder_matches_float64_oracle():
    """Decoder forward in eval mode on L + 1 = 1100 target tokens (decoder self-attention past 1024 keys; only rescoring reaches
    it) over a memory of T' = 1200 frames with a key mask, against the oracle's decoder in float64."""
    from liteasr_b200 import functions as F
    from oracle import u2_oracle as O
    model = _model("fp32")
    V = D256_2L["vocab_size"]
    g = torch.Generator().manual_seed(3)
    L, Tp = 1099, 1200
    ylens = torch.tensor([L, 700])
    ys = torch.full((2, L), -1, dtype=torch.int64)
    for b, n in enumerate(ylens.tolist()):
        ys[b, :n] = torch.randint(1, V - 1, (n,), generator=g)
    ys_in, ys_mask = O.decoder_inputs(ys, ylens, V)
    mem = torch.randn(2, Tp, D256_2L["dec_dim"], generator=g)
    xlens = torch.tensor([_frames_for(Tp), _frames_for(1031)])   # raw frame counts: memory keys 4j < xlens
    dev = torch.device("cuda")
    st, eng, _ = F.bind(model, dev)
    F.bind(model.decoder, dev)
    st.refresh_operands(force=True)
    with torch.no_grad():
        c = eng.decoder_fwd(model.decoder, ys_in.to(dev), ylens.to(dev), mem.to(dev), xlens.to(dev), mem_mask_mode=3)
        got = c.out[:, :V].float().reshape(2, L + 1, V).double()
    sd64 = _sd_on_gpu(_sd(), torch.float64, False)
    cfg = O.U2Shape(**D256_2L)
    with torch.no_grad(), torch.device("cuda"):
        self_mask = ys_mask.cuda().unsqueeze(1) | O.causal_mask(L + 1).unsqueeze(0)
        ref = O.decoder(sd64, cfg, ys_in.cuda(), self_mask, mem.double().cuda(), O.pad_mask(xlens.cuda(), _frames_for(Tp)))
    # padded target rows (i > ylens[b]) are not compared: the reference's loss ignores them
    worst = max(float((got[b, : n + 1] - ref[b, : n + 1]).abs().max()) for b, n in enumerate(ylens.tolist()))
    scale = float(ref.abs().max())
    print(f"\ndecoder L + 1 = 1100, T' = 1200: max-abs error {worst:.3g} of max|ref| {scale:.3g}")
    assert worst <= 1e-4 * scale


def _ragged(model, xs, tps):
    from liteasr_b200 import functions as F
    dev = xs.device
    st, eng, _ = F.bind(model, dev)
    F.bind(model.encoder, dev)
    F.bind(model.ctc, dev)
    st.refresh_operands(force=True)
    with torch.no_grad():
        enc = eng.encoder_fwd(model.encoder, xs.contiguous().float(), None, False, sub_lens=torch.tensor(tps, dtype=torch.int64, device=dev))
    return enc.out.clone()


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_long_decode_batch_equals_batch1(precision):
    """decode_batch on a padded batch with T'_b = 1500 / 1030 / 300 / 40 against attention_rescore per utterance."""
    from liteasr_b200 import decoding
    model = _model(precision)
    tps = [1500, 1030, 300, 40]
    gen = torch.Generator().manual_seed(sum(tps))
    utts = [torch.randn(_frames_for(t), 80, generator=gen) for t in tps]
    T = max(u.shape[0] for u in utts)
    xs = torch.randn(len(utts), T, 80, generator=gen)  # padding frames hold noise, not zeros
    for i, u in enumerate(utts):
        xs[i, : u.shape[0]] = u
    xs = xs.cuda()
    xlens = torch.tensor([u.shape[0] for u in utts])

    # encoder rows of the padded batch against the batch-1 rows
    h = _ragged(model, xs, tps)
    for b, (u, tp) in enumerate(zip(utts, tps)):
        with torch.no_grad():
            hr, _, tpr = decoding._encode(model, u.unsqueeze(0).cuda(), None)
        assert tpr == tp
        hr = hr[0]
        if precision == "fp32" and tp > 1024:
            assert torch.equal(h[b, :tp], hr), f"utterance {b} (T' = {tp}): rows differ from the batch-1 call"
        else:
            rel = float((h[b, :tp] - hr).abs().max() / hr.abs().max())
            print(f"\n{precision} T'_b = {tp}: max-abs / max|h| {rel:.3g}")
            assert rel <= 2e-2

    out = decoding.decode_batch(model, xs, xlens)
    for b, (u, o) in enumerate(zip(utts, out)):
        one = decoding.attention_rescore(model, u.unsqueeze(0).cuda(), return_details=True)
        lmax = max(len(p) for p, _ in one["hyps"])
        print(f"utterance {b} (T' = {tps[b]}): {len(one['hyps'])} hypotheses, the longest {lmax} tokens")
        if precision == "fp32":
            assert o["best"] == one["best"]
            assert [p for p, _ in o["hyps"]] == [p for p, _ in one["hyps"]]
            assert np.allclose([s for _, s in o["hyps"]], [s for _, s in one["hyps"]], rtol=0, atol=1e-4)
            assert np.allclose(o["scores"], one["scores"], rtol=0, atol=1e-4)
        else:
            assert o["best"] == one["best"] or abs(o["hyps"][0][1] - one["hyps"][0][1]) <= 2e-2 * abs(one["hyps"][0][1])


def test_long_greedy_ctc_matches_float64_oracle():
    """greedy_ctc on one 45 s utterance (T' = 1124) in fp32 mode against the oracle's greedy decode in float64."""
    from liteasr_b200 import decoding
    from oracle import u2_oracle as O
    model = _model("fp32")
    x = torch.randn(1, _frames_for(1124), 80, generator=torch.Generator().manual_seed(45))
    got, ids = decoding.greedy_ctc(model, x.cuda(), None)
    assert ids.shape == (1, 1124)
    sd64 = _sd_on_gpu(_sd(), torch.float64, False)
    with torch.no_grad(), torch.device("cuda"):
        want, _ = O.greedy_ctc(sd64, O.U2Shape(**D256_2L), x.double().cuda(), None)
    assert got == [list(w) for w in want]
