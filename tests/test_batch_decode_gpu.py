"""GPU: per-utterance decoding of a padded batch -- the ragged encoder pass (attention mask mode 4, the length-aware depthwise
conv), the device CTC prefix beam search and ``decoding.decode_batch`` -- against the batch-1 path, the host search and torch."""
import json
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as TF

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _frames_for(tp):
    """Input frames whose sub-sampled length is tp: ((T-1)//2-1)//2 == tp for T = 4 tp + 3."""
    return 4 * tp + 3


def _model_from(dims_kw, precision, seed):
    from liteasr_b200.models.u2 import U2, U2Config
    from liteasr_b200.schema import U2Dims
    from liteasr_b200.utils.synthetic import synth_state_dict
    model = U2(U2Config(**{**dims_kw, "precision": precision}))
    model.load_state_dict(synth_state_dict(U2Dims(**dims_kw), seed=seed))
    return model.cuda().eval()


def _golden(case):
    return json.load(open(os.path.join(GOLDEN, f"u2_{case}.json")))


def _ragged(model, xs, tps):
    from liteasr_b200 import functions as F
    dev = xs.device
    st, eng, _ = F.bind(model, dev)
    F.bind(model.encoder, dev)
    F.bind(model.ctc, dev)
    st.refresh_operands(force=True)
    with torch.no_grad():
        enc = eng.encoder_fwd(model.encoder, xs.contiguous().float(), None, False, sub_lens=torch.tensor(tps, dtype=torch.int64, device=dev))
        head = eng.ctc_head_fwd(model.ctc, enc.out)
    V = model.vocab_size
    return enc.out.clone(), head.out[:, :V].float().reshape(xs.shape[0], enc.Tp, V).clone()


def _padded(utts, feat=80, seed=0):
    T = max(u.shape[0] for u in utts)
    g = torch.Generator().manual_seed(seed)
    xs = torch.randn(len(utts), T, feat, generator=g)  # padding frames hold noise, not zeros
    for i, u in enumerate(utts):
        xs[i, : u.shape[0]] = u
    return xs.cuda()


D256_2L = dict(input_dim=80, vocab_size=300, enc_dim=256, enc_ff_dim=1024, enc_attn_heads=4, enc_layers=2, dec_dim=256, dec_ff_dim=1024,
               dec_attn_heads=4, dec_layers=1)


@pytest.mark.parametrize("case,precision,tps", [
    ("tiny", "fp32", [3, 1, 14, 8, 15]),
    ("tiny_odd", "fp32", [6, 15, 1, 9]),
    ("c1", "fp32", [124, 1, 7, 30, 61, 99]),
    ("c1", "bf16", [124, 1, 7, 30, 61, 99]),
    ("d256", "bf16", [254, 1, 300, 127, 33, 128, 255, 40]),    # T'max <= 320: fused attention
    ("d256", "bf16", [340, 128, 1, 255, 127, 254, 77]),        # T'max > 320: unfused mode 4
    ("d256", "fp32", [340, 128, 1, 255, 127, 254, 77]),
])
def test_ragged_encoder_equals_batch1_rows(case, precision, tps):
    from liteasr_b200 import decoding
    if case == "d256":
        dims, seed = D256_2L, 11
    else:
        g = _golden(case)
        dims, seed = g["dims"], g["seed"]
    model = _model_from(dims, precision, seed)
    gen = torch.Generator().manual_seed(sum(tps))
    utts = [torch.randn(_frames_for(t), dims["input_dim"], generator=gen) for t in tps]
    xs = _padded(utts, dims["input_dim"])
    h, logits = _ragged(model, xs, tps)
    # large finite garbage in the padded input frames must not change a valid row
    xs2 = xs.clone()
    for i, u in enumerate(utts):
        xs2[i, u.shape[0]:] = 1e4 * torch.randn(xs.shape[1] - u.shape[0], xs.shape[2], generator=gen).cuda()
    h2, logits2 = _ragged(model, xs2, tps)
    assert torch.isfinite(h).all() and torch.isfinite(logits).all() and torch.isfinite(h2).all()
    worst_h = worst_l = worst_g = 0.0
    for b, (u, tp) in enumerate(zip(utts, tps)):
        with torch.no_grad():
            hr, lr, tpr = decoding._encode(model, u.unsqueeze(0).cuda(), None)
        assert tpr == tp
        hr = hr[0].clone()
        lr = lr[:, : model.vocab_size].float().clone()
        worst_h = max(worst_h, ((h[b, :tp] - hr).abs().max() / hr.abs().max()).item())
        worst_l = max(worst_l, ((logits[b, :tp] - lr).abs().max() / lr.abs().max()).item())
        worst_g = max(worst_g, max((h2[b, :tp] - h[b, :tp]).abs().max().item(), (logits2[b, :tp] - logits[b, :tp]).abs().max().item()))
    bound = 1e-6 if precision == "fp32" else 2e-2
    print(f"{case} {precision}: max-abs / max|.| encoder {worst_h:.3g}, logits {worst_l:.3g}; garbage-padding change {worst_g:.3g}")
    assert worst_h <= bound and worst_l <= bound
    assert worst_g == 0.0


# ---------------------------------------------------------------------------------------------------- kernel level
def _shift_ref(bd, klen):
    """torch restatement of the mode-4 shift for one (T, T) bd matrix: bd[i, klen-1-(i-j)] (j <= i), 0 (j == i+1),
    bd[i+1, j-i-2] (i+1 < j < klen); rows and columns >= klen are left zero."""
    T = bd.shape[0]
    out = torch.zeros_like(bd)
    i = torch.arange(klen, device=bd.device)[:, None]
    j = torch.arange(klen, device=bd.device)[None, :]
    low = bd[i, (klen - 1 - i + j).clamp(0, T - 1)]
    up = bd[(i + 1).clamp(max=T - 1), (j - i - 2).clamp(min=0)]
    out[:klen, :klen] = torch.where(j <= i, low, torch.where(j > i + 1, up, torch.zeros_like(low)))
    return out


def _attn_ref(ac, bd, klen, scale):
    s = (ac + _shift_ref(bd, klen)) * scale
    s[:, klen:] = -1e38
    return torch.softmax(s, dim=-1)


@pytest.mark.parametrize("T,lens", [(37, [37, 1, 20, 2]), (130, [129, 64, 130]), (350, [350, 121, 5])])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_attn_softmax_mode4(T, lens, dtype):
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(T)
    B, H = len(lens), 2
    ld = (T + 7) // 8 * 8
    ac = torch.randn(B, H, T, ld, generator=g, device="cuda").to(dtype)
    bd = torch.randn(B, H, T, ld, generator=g, device="cuda").to(dtype)
    probs = torch.empty(B, H, T, ld, device="cuda", dtype=dtype)
    lt = torch.tensor(lens, dtype=torch.int64, device="cuda")
    scale = 0.125
    ops.attn_softmax_fwd(ac, bd, probs, lt, 4, 0, scale, T)
    assert torch.isfinite(probs.float()).all()
    tol = 2e-6 if dtype == torch.float32 else 8e-3
    for b, k in enumerate(lens):
        for h in range(H):
            ref = _attn_ref(ac[b, h, :, :T].float(), bd[b, h, :, :T].float(), k, scale)
            assert (probs[b, h, :k, :T].float() - ref[:k]).abs().max().item() <= tol


@pytest.mark.parametrize("T,lens", [(300, [300, 1, 127, 128, 254, 255, 33]), (37, [37, 2, 19])])
def test_rel_attn_fused_mode4(T, lens):
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(T + 1)
    B, H, dk = len(lens), 4, 64
    d = H * dk
    qu, qv, k, v = (torch.randn(B * T, d, generator=g, device="cuda").to(torch.bfloat16) for _ in range(4))
    pos = torch.randn(T, d, generator=g, device="cuda").to(torch.bfloat16)
    ld = (T + 63) // 64 * 64
    probs = torch.empty(B, H, T, ld, device="cuda", dtype=torch.bfloat16)
    o = torch.empty(B * T, d, device="cuda", dtype=torch.bfloat16)
    lt = torch.tensor(lens, dtype=torch.int64, device="cuda")
    scale = dk ** -0.5
    ops.rel_attn_fwd(qu, qv, k, v, pos, probs, o, lt, 4, scale, B, H, T, dk)
    assert torch.isfinite(o.float()).all() and torch.isfinite(probs.float()).all()
    worst_p = worst_o = 0.0
    for b, kl in enumerate(lens):
        for h in range(H):
            sl = slice(h * dk, (h + 1) * dk)
            q1, q2 = qu[b * T:(b + 1) * T, sl].float(), qv[b * T:(b + 1) * T, sl].float()
            kk, vv = k[b * T:(b + 1) * T, sl].float(), v[b * T:(b + 1) * T, sl].float()
            p = _attn_ref(q1 @ kk.T, q2 @ pos[:, sl].float().T, kl, scale)
            worst_p = max(worst_p, (probs[b, h, :kl, :T].float() - p[:kl]).abs().max().item())
            worst_o = max(worst_o, (o[b * T:b * T + kl, sl].float() - p[:kl] @ vv).abs().max().item())
    print(f"fused mode 4, T={T}: max |dp| {worst_p:.3g}, max |dO| {worst_o:.3g}")
    assert worst_p <= 1e-2 and worst_o <= 5e-2


@pytest.mark.parametrize("d,dtype,variant", [(6, torch.float32, "generic"), (6, torch.bfloat16, "generic"), (132, torch.float32, "tiled"),
                                             (132, torch.bfloat16, "tiled"), (128, torch.bfloat16, "stream")])
def test_glu_dwconv_fwd_lens(d, dtype, variant):
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(d)
    lens = [70, 1, 33, 64, 8, 7]
    B, T = len(lens), max(lens)
    y2 = (2 * torch.randn(B * T, 2 * d, generator=g, device="cuda")).to(dtype)
    w = torch.randn(d, 15, generator=g, device="cuda") * 0.3
    bias = torch.randn(d, generator=g, device="cuda") * 0.1
    z = torch.empty(B * T, d, device="cuda")
    partial = torch.empty(B * ((T + 31) // 32), 2, d, device="cuda")
    ops.glu_dwconv_fwd_lens(y2, w, bias, z, partial, B, T, d, torch.tensor(lens, dtype=torch.int64, device="cuda"))
    assert torch.isfinite(z).all()
    tol = 2e-5 if variant != "stream" else 2e-2
    for b, L in enumerate(lens):
        y = y2[b * T:b * T + L].float()
        glu = y[:, :d] * torch.sigmoid(y[:, d:])
        ref = TF.conv1d(glu.T.unsqueeze(0), w.view(d, 1, 15), bias, padding=7, groups=d)[0].T
        assert (z[b * T:b * T + L] - ref).abs().max().item() <= tol * max(1.0, ref.abs().max().item())


# ---------------------------------------------------------------------------------------------------- device search
def _corpus(K, beam, n, rng):
    """n (frames, K) matrices: blank-dominated rows, exact value ties, a small vocabulary (repeated tokens), idx = -1 columns."""
    mats = []
    for u in range(n):
        frames = int(rng.integers(0, 401)) if u else 0
        V = max(K + 1, int(rng.integers(K + 1, K + 6)))
        tv = np.empty((frames, K), np.float32)
        ti = np.empty((frames, K), np.int32)
        kind = u % 4
        for t in range(frames):
            cls = rng.permutation(V)[:K]
            logit = rng.normal(size=K) * (3.0 if kind != 2 else 1.0)
            if kind == 0 and rng.random() < 0.8:  # blank-dominated frame
                if 0 not in cls:
                    cls[0] = 0
                logit[list(cls).index(0)] = 8.0
            if kind == 1:  # exact ties
                logit = np.round(logit * 2) / 2
            lp = logit - np.log(np.exp(logit).sum() + 1.0)
            order = np.lexsort((cls, -lp))
            tv[t], ti[t] = lp[order].astype(np.float32), cls[order]
            if kind == 3 and rng.random() < 0.3:  # classes that do not exist (fewer than K in the vocabulary)
                m = int(rng.integers(1, K + 1))
                tv[t, K - m:], ti[t, K - m:] = -np.inf, -1
        mats.append((tv, ti))
    return mats


def test_device_search_equals_host_search():
    from liteasr_b200 import ops
    rng = np.random.default_rng(1234)
    total, worst = 0, 0.0
    for K in (1, 3, 10, 16):
        for beam in (1, 4, 10, 16):
            mats = _corpus(K, beam, 32, rng)
            Tmax = max(1, max(m[0].shape[0] for m in mats))
            tv = np.full((len(mats), Tmax, K), -np.inf, np.float32)
            ti = np.full((len(mats), Tmax, K), -1, np.int32)
            for b, (v, i) in enumerate(mats):
                tv[b, : v.shape[0]], ti[b, : v.shape[0]] = v, i
            frames = torch.tensor([m[0].shape[0] for m in mats], dtype=torch.int64, device="cuda")
            toks, lens, scores, count = ops.ctc_prefix_beam_search_batch(torch.from_numpy(tv.reshape(-1, K)).cuda(),
                                                                         torch.from_numpy(ti.reshape(-1, K)).cuda(), frames, Tmax, beam=beam)
            toks, lens, scores, count = (t.cpu().numpy() for t in (toks, lens, scores, count))
            for b, (v, i) in enumerate(mats):
                host = ops.ctc_prefix_beam_search_host(v, i, beam=beam, blank=0)
                dev = [(tuple(int(x) for x in toks[b, h, : lens[b, h]]), float(scores[b, h])) for h in range(count[b])]
                assert [p for p, _ in dev] == [p for p, _ in host], (K, beam, b)
                for (_, sd), (_, sh) in zip(dev, host):
                    if math.isinf(sh):
                        assert sd == sh
                    else:
                        rel = abs(sd - sh) / max(abs(sh), 1e-300)
                        worst = max(worst, rel)
                        assert rel <= 1e-9, (K, beam, b, sd, sh)
                total += 1
    print(f"device vs host search: {total} matrices, prefix lists identical, largest relative score difference {worst:.3g}")
    assert total >= 500


# ---------------------------------------------------------------------------------------------------- decode_batch
@pytest.mark.parametrize("case", ["tiny", "tiny_odd", "c1"])
def test_decode_batch_fp32_equals_batch1_and_golden(case):
    from liteasr_b200 import decoding
    from liteasr_b200.utils.synthetic import synth_batch
    g = _golden(case)
    model = _model_from(g["dims"], "fp32", g["seed"])
    batch = synth_batch(g["batch"], g["tmax"], g["lmax"], g["dims"]["vocab_size"], seed=g["seed"])
    recs = list(zip(g["f32"]["inference"], g["f64"]["inference"]))
    utts = [batch[0][r32["utt"], : r32["frames"]] for r32, _ in recs][::-1]  # shortest first: unsorted lengths
    recs = recs[::-1]
    xs = _padded(utts, g["dims"]["input_dim"])
    xlens = torch.tensor([u.shape[0] for u in utts])
    out = decoding.decode_batch(model, xs, xlens)
    for u, (r32, r64), o in zip(utts, recs, out):
        x = u.unsqueeze(0).cuda()
        one = decoding.attention_rescore(model, x, return_details=True)
        assert o["best"] == one["best"] == r64["best"]
        assert [p for p, _ in o["hyps"]] == [p for p, _ in one["hyps"]] == [tuple(p) for p, _ in r64["hyps"]]
        assert np.allclose([s for _, s in o["hyps"]], [s for _, s in one["hyps"]], rtol=0, atol=1e-4)
        assert np.allclose([s for _, s in o["hyps"]], [s for _, s in r64["hyps"]], rtol=0, atol=1e-4)
        assert np.allclose(o["scores"], one["scores"], rtol=0, atol=1e-4)
        greedy, _ = decoding.greedy_ctc(model, x, None)
        assert o["greedy"] == greedy[0] == r64["greedy"]


def test_decode_batch_bf16_c1():
    from liteasr_b200 import decoding
    from liteasr_b200.utils.synthetic import synth_batch
    g = _golden("c1")
    m16 = _model_from(g["dims"], "bf16", g["seed"])
    batch = synth_batch(g["batch"], g["tmax"], g["lmax"], g["dims"]["vocab_size"], seed=g["seed"])
    xs, xlens = batch[0].cuda(), batch[1]
    out = decoding.decode_batch(m16, xs, xlens)
    for b, o in enumerate(out):
        one = decoding.attention_rescore(m16, xs[b:b + 1, : int(xlens[b])], return_details=True)
        assert o["best"] == one["best"] or abs(o["hyps"][0][1] - one["hyps"][0][1]) <= 2e-2 * abs(one["hyps"][0][1])


def test_decode_batch_errors():
    from liteasr_b200 import decoding
    g = _golden("tiny")
    model = _model_from(g["dims"], "fp32", g["seed"])
    xs = torch.randn(2, 40, g["dims"]["input_dim"], device="cuda")
    with pytest.raises(ValueError):
        decoding.decode_batch(model, xs, torch.tensor([40, 6]))
    with pytest.raises(ValueError):
        decoding.decode_batch(model, xs, torch.tensor([41, 20]))
    model.train()
    with pytest.raises(RuntimeError):
        decoding.decode_batch(model, xs, torch.tensor([40, 20]))
    from liteasr_b200 import functions as F
    _, eng, _ = F.bind(model, xs.device)
    with pytest.raises(RuntimeError):
        eng.encoder_fwd(model.encoder, xs, None, True, sub_lens=torch.tensor([9, 4], device="cuda"))
