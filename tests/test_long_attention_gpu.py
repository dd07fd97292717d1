"""GPU: the attention softmax forward and backward (csrc/attention.cu) on rows wider than 1024 columns -- the CTA-per-row kernels
that serve encoder self-attention and decoder source attention past T' = 1024 (~41 s of audio) and decoder self-attention past
L + 1 = 1024 -- against a float64 reference evaluated on the GPU from the same rounded inputs the kernel reads.

Element-wise bounds (u = 2^-24, S = the largest |scaled logit| of the call, NPW = column pairs per thread of the bucket that ld
selects: 2 / 4 / 8 / 16 for ld <= 2048 / 4096 / 8192 / 16384):
  forward, fp32 probs : |p - ref| <= ref * u * (6 S + 2 NPW + 24).  The row sum is 2 NPW sequential adds per thread, 5 of the warp
                        butterfly and 5 of a second butterfly over the 16 warp partials (block_sum; lanes 16-31 hold 0):
                        at most 2 NPW + 10 roundings; two expf at <= 2 ulp, 1/sum and the product add 6; the logit add /
                        subtract is the 6 S term, as for the warp kernels.
  forward, bf16 probs : one more rounding, + 2^-8 * ref
  backward            : ds = p (dp - D) scale with D = sum_j p_j dp_j; the fp32 dot product is off by at most
                        (2 NPW + 12) u sum_j |p_j dp_j| (one rounding per product, at most 2 NPW + 10 per sum), the three roundings of the
                        element by 2^-22 |p scale| (|dp| + |D|); bf16 outputs add 2^-8 |ref|.  dbd holds the same values moved
                        through the inverse shift.
Columns [Tk, ld) of probs / dscores / dbd must be exactly 0; every output buffer starts as NaN."""
import pytest
import torch

pytestmark = pytest.mark.gpu

U32 = 2.0 ** -24
MAX_LD = 16384
DTYPES = [(torch.float32, torch.float32), (torch.float32, torch.bfloat16), (torch.bfloat16, torch.bfloat16)]  # (scores, probs)


def _npw(ld):
    return 2 if ld <= 2048 else 4 if ld <= 4096 else 8 if ld <= 8192 else 16


def _c8(n):
    return (n + 7) // 8 * 8


def _rel_shift(x):
    """The legacy rel_shift (nets/attention.py:99-118) as the reference writes it: pad a zero column, re-view, drop a row."""
    *lead, t1, t2 = x.shape
    xp = torch.cat([x.new_zeros(*lead, t1, 1), x], -1).view(*lead, t2 + 1, t1)
    return xp[..., 1:, :].reshape(x.shape)


def _key_len(lens, mode, B, Tk):
    if mode == 0:
        return [Tk] * B
    out = []
    for l in lens.tolist():
        k = l + 1 if mode == 2 else (l + 3) // 4 if mode == 3 else l
        out.append(max(0, min(Tk, k)))
    return out


def _fill(shape, Tk, dtype, g, mult):
    """(…, ld) buffer of NaN with N(0, mult^2) values in columns [0, Tk), generated one leading slice at a time."""
    t = torch.full(shape, float("nan"), device="cuda", dtype=dtype)
    flat = t.view(-1, *shape[-2:])
    for s in range(flat.shape[0]):
        flat[s, :, :Tk] = (torch.randn(shape[-2], Tk, generator=g, device="cuda") * mult).to(dtype)
    return t


def _check(name, got, ref, bound, Tk):
    assert not torch.isnan(got).any(), f"{name}: element left unwritten or NaN"
    err = (got[..., :Tk].double() - ref).abs()
    assert (err <= bound).all(), f"{name}: worst excess {float((err - bound).max()):.3g}"
    assert (got[..., Tk:] == 0).all(), f"{name}: padding columns not zeroed"


def _softmax_case(B, H, Tq, Tk, ld, sdt, pdt, mode, causal, rel, lens, seed, scale=0.125, bwd=True):
    """Run lasr_attn_softmax_fwd (and _bwd) once and check every output element; the float64 reference runs per utterance."""
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(seed)
    ac = _fill((B, H, Tq, ld), Tk, sdt, g, 3)   # padding columns are never read as scores
    bd = _fill((B, H, Tq, ld), Tk, sdt, g, 3) if rel else None
    probs = torch.full((B, H, Tq, ld), float("nan"), device="cuda", dtype=pdt)
    ops.attn_softmax_fwd(ac, bd, probs, lens, mode, causal, scale, Tk)
    if bwd:
        dp = _fill((B, H, Tq, ld), Tk, sdt, g, 1)
        dsc = torch.full((B, H, Tq, ld), float("nan"), device="cuda", dtype=pdt)
        dbd = torch.full((B, H, Tq, ld), float("nan"), device="cuda", dtype=pdt) if rel else None
        ops.attn_softmax_bwd(probs, dp, dsc, dbd, scale, Tk)
    npw = _npw(ld)
    klens = _key_len(lens, mode, B, Tk)
    j = torch.arange(Tk, device="cuda")
    for b in range(B):
        # float64 reference (masked_fill(-1e38) + softmax: a row without keys is uniform 1/Tk, quirk Q4)
        s = ac[b, ..., :Tk].double()
        if rel:
            s = s + _rel_shift(bd[b, ..., :Tk].double())
        s = s * scale
        S = float(s.abs().max())
        mask = (j >= klens[b])[None, :]
        if causal:
            mask = mask | (j[None, :] > torch.arange(Tq, device="cuda")[:, None])
        ref = torch.softmax(s.masked_fill(mask, -1e38), -1)
        del s
        bound = ref * U32 * (6 * S + 2 * npw + 24)
        if pdt == torch.bfloat16:
            bound = bound + 2.0 ** -8 * ref
        _check("probs", probs[b], ref, bound, Tk)
        del ref, bound
        if not bwd:
            continue
        p64, g64 = probs[b, ..., :Tk].double(), dp[b, ..., :Tk].double()
        D = (p64 * g64).sum(-1, keepdim=True)
        ds_ref = p64 * (g64 - D) * scale
        ds_bound = p64.abs() * abs(scale) * ((2 * npw + 12) * U32 * (p64 * g64).abs().sum(-1, keepdim=True)
                                             + 2.0 ** -22 * (g64.abs() + D.abs()))
        del p64, g64
        if pdt == torch.bfloat16:
            ds_bound = ds_bound + 2.0 ** -8 * (ds_ref.abs() + ds_bound)
        _check("dscores", dsc[b], ds_ref, ds_bound, Tk)
        if rel:
            x = torch.zeros(H, Tq, Tk, dtype=torch.float64, device="cuda", requires_grad=True)
            y = _rel_shift(x)
            dbd_ref = torch.autograd.grad(y, x, ds_ref, retain_graph=True)[0]
            dbd_bound = torch.autograd.grad(y, x, ds_bound)[0]
            del x, y, ds_ref, ds_bound
            _check("dbd", dbd[b], dbd_ref, dbd_bound, Tk)
    return probs


def test_rel_shift_restatement_matches_oracle():
    from oracle.u2_oracle import rel_shift
    x = torch.randn(2, 3, 37, 37, dtype=torch.float64)
    assert torch.equal(_rel_shift(x), rel_shift(x))


# T on both sides of 1024 and of every wide-bucket edge (2048, 4096, 8192) up to the bound 16 384
@pytest.mark.parametrize("T", [1025, 1031, 1088, 2048, 2049, 4097, 8192, 16384])
@pytest.mark.parametrize("sdt,pdt", DTYPES)
@pytest.mark.parametrize("mode", [0, 1, 3])
def test_wide_softmax_relshift_fwd_bwd(T, sdt, pdt, mode):
    """Encoder self-attention (rel_shift of bd, Tq = Tk) at ld = ceil(T, 8) as the engine allocates it.  With a key mask the
    second utterance has no keys at all: every score of its rows is -1e38 and the softmax is uniform 1/Tk, like the reference."""
    g = torch.Generator().manual_seed(T * 7 + mode)
    lens = None
    B = 1 if mode == 0 else 3
    if mode == 1:
        lens = torch.tensor([T + 5, 0, int(torch.randint(1, T, (1,), generator=g))])
    elif mode == 3:                                           # raw frame counts: klen = ceil(l / 4)
        lens = torch.tensor([4 * T, 0, int(torch.randint(1, 4 * T - 3, (1,), generator=g))])
    lens = lens.cuda() if lens is not None else None
    probs = _softmax_case(B, 1, T, T, _c8(T), sdt, pdt, mode, 0, True, lens, seed=T + 100 * mode)
    if mode:
        assert torch.allclose(probs[1, ..., :T].double(), torch.full((1, T, T), 1.0 / T, dtype=torch.float64, device="cuda"),
                              rtol=2.0 ** -8, atol=0)


@pytest.mark.parametrize("sdt,pdt", DTYPES)
@pytest.mark.parametrize("Tq,Tk", [(1, 1025), (41, 1025), (1, 3000), (41, 3000)])
def test_wide_softmax_cross_attention(Tq, Tk, sdt, pdt):
    """Decoder source attention: Tq = L + 1 queries against T' encoder frames, encoder key mask (mode 3), no rel-pos term."""
    lens = torch.tensor([4 * Tk, 0, 4 * Tk - 13, 5], device="cuda")
    _softmax_case(4, 2, Tq, Tk, _c8(Tk), sdt, pdt, 3, 0, False, lens, seed=Tq * Tk)


@pytest.mark.parametrize("sdt,pdt", DTYPES)
def test_wide_softmax_decoder_self_attention(sdt, pdt):
    """Decoder self-attention at L + 1 = 1100 (rescoring a long hypothesis): causal, keys j < ylen + 1 (mode 2)."""
    lens = torch.tensor([1099, 0, 1030, 17], device="cuda")
    _softmax_case(4, 2, 1100, 1100, 1104, sdt, pdt, 2, 1, False, lens, seed=1100)


@pytest.mark.parametrize("sdt,pdt", DTYPES)
@pytest.mark.parametrize("Tk,ld", [(600, 1026), (1025, 2050), (2049, 8192), (1030, 16384)])
def test_wide_softmax_padding_columns(Tk, ld, sdt, pdt):
    """Row buffers wider than the bucket Tk alone would pick; ld decides the kernel, so (600, 1026) takes the wide path too."""
    lens = torch.tensor([4 * Tk, 4 * Tk - 9], device="cuda")
    _softmax_case(2, 1, Tk, Tk, ld, sdt, pdt, 3, 0, True, lens, seed=Tk + ld)


def _mode4_ref(ac, bd, klen, scale):
    """Mode 4 for one (T, T) matrix pair: the shift over klen, keys >= klen masked; rows >= klen are not compared."""
    T = ac.shape[0]
    i = torch.arange(klen, device=ac.device)[:, None]
    j = torch.arange(klen, device=ac.device)[None, :]
    low = bd[i, (klen - 1 - i + j).clamp(0, T - 1)]
    up = bd[(i + 1).clamp(max=T - 1), (j - i - 2).clamp(min=0)]
    sh = torch.where(j <= i, low, torch.where(j > i + 1, up, torch.zeros_like(low)))
    s = ac[:klen].clone()
    s[:, :klen] += sh
    s = s * scale
    s[:, klen:] = -1e38
    return torch.softmax(s, -1), float(s[:, :klen].abs().max())


@pytest.mark.parametrize("sdt,pdt", DTYPES)
def test_wide_softmax_mode4(sdt, pdt):
    """Per-utterance rows of a padded batch (mask mode 4, forward only): valid rows equal the batch-1 call on the cut utterance."""
    from liteasr_b200 import ops
    T, lens = 2049, [2049, 1500, 1025, 300, 1]
    B, H, ld = len(lens), 1, _c8(T)
    g = torch.Generator(device="cuda").manual_seed(T)
    ac = _fill((B, H, T, ld), T, sdt, g, 3)
    bd = _fill((B, H, T, ld), T, sdt, g, 3)
    probs = torch.full((B, H, T, ld), float("nan"), device="cuda", dtype=pdt)
    scale = 0.125
    ops.attn_softmax_fwd(ac, bd, probs, torch.tensor(lens, device="cuda"), 4, 0, scale, T)
    assert torch.isfinite(probs.float()).all()
    assert (probs[..., T:] == 0).all()
    for b, k in enumerate(lens):
        ref, S = _mode4_ref(ac[b, 0, :, :T].double(), bd[b, 0, :, :T].double(), k, scale)
        bound = ref * U32 * (6 * S + 2 * _npw(ld) + 24)
        if pdt == torch.bfloat16:
            bound = bound + 2.0 ** -8 * ref
        err = (probs[b, 0, :k, :T].double() - ref).abs()
        assert (err <= bound).all(), f"utterance {b}: worst excess {float((err - bound).max()):.3g}"


@pytest.mark.parametrize("sdt,pdt", DTYPES)
def test_wide_softmax_is_independent_of_ld(sdt, pdt):
    """The column -> thread mapping and the reduction tree do not depend on ld: the same rows at ld = ceil(Tk, 8) and in wider
    buffers (other NPW buckets) are bit-identical, forward and backward; so is a mode-4 row of a padded batch and the batch-1 call."""
    from liteasr_b200 import ops
    Tk, scale = 1030, 0.125
    g = torch.Generator(device="cuda").manual_seed(5)
    ac0 = (torch.randn(2, 2, Tk, Tk, generator=g, device="cuda") * 3).to(sdt)
    bd0 = (torch.randn(2, 2, Tk, Tk, generator=g, device="cuda") * 3).to(sdt)
    dp0 = torch.randn(2, 2, Tk, Tk, generator=g, device="cuda").to(sdt)
    lens = torch.tensor([4 * Tk, 4 * Tk - 999], device="cuda")
    outs = []
    for ld in (_c8(Tk), 2050, 4100, 9000, MAX_LD):
        ac, bd, dp = (torch.zeros(2, 2, Tk, ld, device="cuda", dtype=sdt) for _ in range(3))
        ac[..., :Tk], bd[..., :Tk], dp[..., :Tk] = ac0, bd0, dp0
        probs, dsc, dbd = (torch.full((2, 2, Tk, ld), float("nan"), device="cuda", dtype=pdt) for _ in range(3))
        ops.attn_softmax_fwd(ac, bd, probs, lens, 3, 0, scale, Tk)
        ops.attn_softmax_bwd(probs, dp, dsc, dbd, scale, Tk)
        outs.append((ld, probs[..., :Tk].clone(), dsc[..., :Tk].clone(), dbd[..., :Tk].clone()))
    for ld, p, d, db in outs[1:]:
        assert torch.equal(p, outs[0][1]), f"probs differ at ld {ld}"
        assert torch.equal(d, outs[0][2]), f"dscores differ at ld {ld}"
        assert torch.equal(db, outs[0][3]), f"dbd differ at ld {ld}"
    # mode 4: utterance 1 (klen = Tk) of a batch padded to 2100 frames against the maskless batch-1 call
    Tp = 2100
    ac, bd = (torch.randn(2, 2, Tp, _c8(Tp), generator=g, device="cuda") * 3).to(sdt), (torch.randn(2, 2, Tp, _c8(Tp), generator=g, device="cuda") * 3).to(sdt)
    ac[1, :, :Tk, :Tk], bd[1, :, :Tk, :Tk] = ac0[0], bd0[0]
    probs = torch.full((2, 2, Tp, _c8(Tp)), float("nan"), device="cuda", dtype=pdt)
    ops.attn_softmax_fwd(ac, bd, probs, torch.tensor([Tp, Tk], device="cuda"), 4, 0, scale, Tp)
    one = torch.full((1, 2, Tk, _c8(Tk)), float("nan"), device="cuda", dtype=pdt)
    a1, b1 = (torch.zeros(1, 2, Tk, _c8(Tk), device="cuda", dtype=sdt) for _ in range(2))
    a1[0, ..., :Tk], b1[0, ..., :Tk] = ac0[0], bd0[0]
    ops.attn_softmax_fwd(a1, b1, one, None, 0, 0, scale, Tk)
    assert torch.equal(probs[1, :, :Tk, :Tk], one[0, ..., :Tk])


def test_wide_softmax_bound():
    """ld above 16 384 is rejected with an error that names the bound; ld = 16 384 itself runs."""
    from liteasr_b200 import ops
    for Tk in (MAX_LD + 1, MAX_LD + 7):
        ld = _c8(Tk)
        ac = torch.zeros(1, 1, 1, ld, device="cuda")
        probs = torch.zeros(1, 1, 1, ld, device="cuda")
        with pytest.raises(RuntimeError, match="16384"):
            ops.attn_softmax_fwd(ac, None, probs, None, 0, 0, 1.0, Tk)
        with pytest.raises(RuntimeError, match="16384"):
            ops.attn_softmax_bwd(probs, ac, torch.zeros_like(probs), None, 1.0, Tk)
    ac = torch.zeros(1, 1, 1, MAX_LD, device="cuda")
    probs = torch.full((1, 1, 1, MAX_LD), float("nan"), device="cuda")
    ops.attn_softmax_fwd(ac, None, probs, None, 0, 0, 1.0, MAX_LD - 3)
    torch.cuda.synchronize()
    assert torch.allclose(probs[..., :MAX_LD - 3].double(), torch.full((MAX_LD - 3,), 1.0 / (MAX_LD - 3), dtype=torch.float64, device="cuda"))
    assert (probs[..., MAX_LD - 3:] == 0).all()


def test_wide_softmax_more_than_2_31_elements():
    """B = 3, H = 4, T' = 16 384 in bf16: 3.2e9 elements per (B,H,T',ld) tensor, past the int32 range.  Forward and backward with
    the rel-pos term, checked on a seeded sample of rows that includes the last rows of the last (utterance, head)."""
    from liteasr_b200 import ops
    B, H, T = 3, 4, 16384
    ld, scale = T, 0.125
    assert B * H * T * ld > 2 ** 31
    free, _ = torch.cuda.mem_get_info()
    if free < 60e9:
        pytest.skip(f"needs 60 GB of free HBM ({free / 1e9:.0f} GB free)")
    dt = torch.bfloat16
    g = torch.Generator(device="cuda").manual_seed(31)
    ac = _fill((B, H, T, ld), T, dt, g, 3)
    bd = _fill((B, H, T, ld), T, dt, g, 3)
    lens = torch.tensor([4 * T, 4 * T - 4001, 4 * 9000], device="cuda")
    probs = torch.full((B, H, T, ld), float("nan"), device="cuda", dtype=dt)
    ops.attn_softmax_fwd(ac, bd, probs, lens, 3, 0, scale, T)
    dp = _fill((B, H, T, ld), T, dt, g, 1)
    dbd = torch.full((B, H, T, ld), float("nan"), device="cuda", dtype=dt)
    dsc = torch.full((B, H, T, ld), float("nan"), device="cuda", dtype=dt)
    ops.attn_softmax_bwd(probs, dp, dsc, dbd, scale, T)
    torch.cuda.synchronize()
    klens = _key_len(lens, 3, B, T)
    rng = torch.Generator().manual_seed(2024)
    npw = _npw(ld)
    j = torch.arange(T, device="cuda")
    for b in range(B):
        for h in range(H):
            rows = torch.randint(1, T - 1, (6,), generator=rng).tolist() + [0, T - 2, T - 1]
            if (b, h) == (B - 1, H - 1):
                rows += list(range(T - 8, T))
            for i in sorted(set(rows)):
                a = ac[b, h, i].double()
                sh = torch.where(j <= i, bd[b, h, i, (T - 1 - i + j).clamp(0, T - 1)].double(),
                                 torch.where(j > i + 1, bd[b, h, min(i + 1, T - 1), (j - i - 2).clamp(min=0)].double(), torch.zeros_like(a)))
                s = ((a + sh) * scale).masked_fill(j >= klens[b], -1e38)
                ref = torch.softmax(s, -1)
                S = float(((a + sh) * scale).abs().max())
                bound = ref * U32 * (6 * S + 2 * npw + 24) + 2.0 ** -8 * ref
                _check(f"probs[{b},{h},{i}]", probs[b, h, i], ref, bound, T)

            def ds_row(i):
                p64, g64 = probs[b, h, i].double(), dp[b, h, i].double()
                D = (p64 * g64).sum()
                r = p64 * (g64 - D) * scale
                bnd = p64.abs() * scale * ((2 * npw + 12) * U32 * (p64 * g64).abs().sum() + 2.0 ** -22 * (g64.abs() + D.abs()))
                return r, bnd + 2.0 ** -8 * (r.abs() + bnd)
            for r in sorted(set(rows)):
                ds, dsb = ds_row(r)
                _check(f"dscores[{b},{h},{r}]", dsc[b, h, r], ds, dsb, T)
                # dbd row r = [ds row r-1, columns r+1 .. T-1 | ds row r, columns 0 .. r]; row 0 starts with zeros
                prev, prevb = ds_row(r - 1) if r > 0 else (torch.zeros(T, dtype=torch.float64, device="cuda"),) * 2
                want = torch.cat([prev[r + 1:], ds[: r + 1]])
                wb = torch.cat([prevb[r + 1:], dsb[: r + 1]])
                _check(f"dbd[{b},{h},{r}]", dbd[b, h, r], want, wb, T)
