"""GPU: the bandwidth kernels (LayerNorm, conv-module middle, attention softmax) through the C ABI vs plain torch fp32
references of the same op (the torch ops the reference calls: nets/layer_norm.py:15, nets/conformer_convolution.py:49-53,
nets/attention.py:46-59,99-118)."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _close(a, b, tol):
    a, b = a.float(), b.float()
    return (a - b).abs().max().item() <= tol * max(1.0, b.abs().max().item())


@pytest.mark.parametrize("rows,d", [(37, 64), (1000, 128), (9568, 256), (700, 512), (129, 1024)])
@pytest.mark.parametrize("dy_dtype", [torch.float32, torch.bfloat16])
def test_layernorm_fwd_bwd_fused_outputs(rows, d, dy_dtype):
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(rows + d)
    x = torch.randn(rows, d, generator=g, device="cuda") * 2 + 0.5
    gamma = torch.randn(d, generator=g, device="cuda")
    beta = torch.randn(d, generator=g, device="cuda")
    y = torch.empty(rows, d, device="cuda")
    mean = torch.empty(rows, device="cuda")
    rstd = torch.empty(rows, device="cuda")
    ops.layernorm_fwd(x, gamma, beta, y, mean, rstd, 1e-12)
    xr = x.clone().requires_grad_(True)
    gr, br = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    yr = torch.nn.functional.layer_norm(xr, (d,), gr, br, 1e-12)
    assert _close(y, yr, 1e-5)
    ylo = torch.empty(rows, d, device="cuda", dtype=torch.bfloat16)
    ops.layernorm_fwd(x, gamma, beta, ylo, None, None, 1e-12)
    assert _close(ylo, yr, 1e-2)
    dy = torch.randn(rows, d, generator=g, device="cuda").to(dy_dtype)
    yr.backward(dy.float())
    for accumulate in (False, True):
        base = torch.randn(rows, d, generator=g, device="cuda")
        dx = base.clone()
        dg, db = torch.zeros(d, device="cuda"), torch.zeros(d, device="cuda")
        cs = torch.ones(d, device="cuda")
        lo = torch.empty(rows, d, device="cuda", dtype=torch.bfloat16)
        ops.layernorm_bwd(dy, x, mean, rstd, gamma, dx, dg, db, accumulate, dx_lo=lo, colsum=cs, colsum_scale=0.5)
        ref = xr.grad + (base if accumulate else 0)
        assert _close(dx, ref, 1e-4)
        assert _close(lo, ref, 1e-2)
        assert _close(cs - 1.0, 0.5 * ref.sum(0), 1e-4)
        assert _close(dg, gr.grad, 1e-4) and _close(db, br.grad, 1e-4)
        # the plain call (no fused outputs) gives the same dx
        dx2 = base.clone()
        ops.layernorm_bwd(dy, x, mean, rstd, gamma, dx2, torch.zeros(d, device="cuda"), torch.zeros(d, device="cuda"), accumulate)
        assert torch.equal(dx, dx2)


def _conv_module_ref(y2, w, bias, gamma, beta, eps=1e-5):
    """GLU -> depthwise conv k=15 pad 7 -> BatchNorm (batch stats over all B*T frames) -> Swish, on (B,T,2d) input."""
    B, T, d2 = y2.shape
    d = d2 // 2
    u = torch.nn.functional.glu(y2.transpose(1, 2), dim=1)                      # (B,d,T)
    z = torch.nn.functional.conv1d(u, w.view(d, 1, -1), bias, padding=w.shape[1] // 2, groups=d)
    zn = torch.nn.functional.batch_norm(z, None, None, gamma, beta, True, 0.1, eps)
    a = zn * torch.sigmoid(zn)
    return z.transpose(1, 2), a.transpose(1, 2)


@pytest.mark.parametrize("B,T,d", [(3, 50, 64), (5, 299, 256), (2, 31, 128), (4, 97, 512), (2, 1, 64), (3, 64, 64), (2, 33, 192), (1, 7, 144)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_conv_module_middle_fwd_bwd(B, T, d, dtype):
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(B * T + d)
    y2 = torch.randn(B, T, 2 * d, generator=g, device="cuda").to(dtype)
    w = torch.randn(d, 15, generator=g, device="cuda") * 0.3
    bias = torch.randn(d, generator=g, device="cuda") * 0.1
    gamma = torch.rand(d, generator=g, device="cuda") + 0.5
    beta = torch.randn(d, generator=g, device="cuda") * 0.1
    rows = B * T
    y2f = y2.float().clone().requires_grad_(True)
    wr, br, gr, ber = (t.clone().requires_grad_(True) for t in (w, bias, gamma, beta))
    z_ref, a_ref = _conv_module_ref(y2f, wr, br, gr, ber)
    # forward
    z = torch.empty(rows, d, device="cuda")
    nblk = B * ((T + 31) // 32)
    partial = torch.empty(nblk, 2, d, device="cuda")
    ops.glu_dwconv_fwd(y2.view(rows, 2 * d), w, bias, z, partial, B, T, d)
    # bf16 operands: the streaming kernel's GLU uses sigmoid(x) = 0.5 tanh.approx(x / 2) + 0.5 (rel. error ~2^-11, below the 2^-9
    # resolution of the operands it multiplies)
    bf = dtype == torch.bfloat16
    assert _close(z, z_ref.reshape(rows, d), 2e-3 if bf else 1e-5)
    mean, rstd = torch.empty(d, device="cuda"), torch.empty(d, device="cuda")
    rm, rv = torch.zeros(d, device="cuda"), torch.ones(d, device="cuda")
    nbt = torch.zeros((), dtype=torch.int64, device="cuda")
    ops.bn_finalize(partial, nblk, d, rows, mean, rstd, rm, rv, nbt, True)
    zr = z_ref.detach().reshape(rows, d)
    assert _close(mean, zr.mean(0), 5e-4 if bf else 1e-5) and _close(rstd, (zr.var(0, unbiased=False) + 1e-5).rsqrt(), 1e-3 if bf else 1e-4)
    assert _close(rm, 0.1 * zr.mean(0), 5e-4 if bf else 1e-5) and _close(rv, 0.9 + 0.1 * zr.var(0, unbiased=True), 1e-3 if bf else 1e-4) and int(nbt) == 1
    zs = z.view(B, T, d).double()   # the statistics are exact for the z the kernel wrote
    assert _close(mean, zs.mean((0, 1)).float(), 1e-5) and _close(rstd, (zs.var((0, 1), unbiased=False) + 1e-5).rsqrt().float(), 1e-4)
    a = torch.empty(rows, d, device="cuda", dtype=dtype)
    ops.bn_swish_fwd(z, mean, rstd, gamma, beta, a)
    tol = 1e-4 if dtype == torch.float32 else 2e-2
    assert _close(a, a_ref.reshape(rows, d), tol)
    # backward
    da = torch.randn(rows, d, generator=g, device="cuda").to(dtype)
    a_ref.backward(da.float().view(B, T, d))
    part2 = torch.empty((rows + 31) // 32, 2, d, device="cuda")
    sums = torch.empty(2, d, device="cuda")
    dgam, dbet = torch.zeros(d, device="cuda"), torch.zeros(d, device="cuda")
    ops.bn_swish_bwd_stats(da, z, mean, rstd, gamma, beta, part2, sums, dgam, dbet)
    assert _close(dgam, gr.grad, 2e-4 if dtype == torch.float32 else 2e-2) and _close(dbet, ber.grad, 2e-4 if dtype == torch.float32 else 2e-2)
    dy2 = torch.empty(rows, 2 * d, device="cuda", dtype=dtype)
    dw, dbias = torch.zeros(d, 15, device="cuda"), torch.zeros(d, device="cuda")
    cs = torch.zeros(2 * d, device="cuda")
    ops.dwconv_glu_bwd(da, z, y2.view(rows, 2 * d), mean, rstd, gamma, beta, sums, w, dy2, dw, dbias, B, T, d, colsum=cs)
    # two-stage (deterministic) reduction of the same gradients
    dw2, dbias2, cs2 = torch.zeros(d, 15, device="cuda"), torch.zeros(d, device="cuda"), torch.zeros(2 * d, device="cuda")
    wpart = torch.empty(nblk, 18, d, device="cuda")
    ops.dwconv_glu_bwd(da, z, y2.view(rows, 2 * d), mean, rstd, gamma, beta, sums, w, torch.empty_like(dy2), dw2, dbias2, B, T, d,
                       colsum=cs2, wpartial=wpart)
    assert _close(dw2, dw, 1e-4) and _close(dbias2, dbias, 1e-4) and _close(cs2, cs, 1e-4)
    tolg = 2e-4 if dtype == torch.float32 else 3e-2
    assert _close(dy2, y2f.grad.reshape(rows, 2 * d), tolg)
    assert _close(dw, wr.grad, tolg) and _close(dbias, br.grad, tolg)
    assert _close(cs, dy2.float().sum(0), 1e-3 if dtype == torch.float32 else 3e-2)


# ---------------------------------------------------------------------------------------------------------------------------------
# attention softmax (csrc/attention.cu) against a float64 reference evaluated from the same rounded inputs the kernel reads
#
# Element-wise bounds (u = 2^-24, S = the largest |scaled logit| of the call):
#   forward, fp32 probs : |p - ref| <= ref * u * (6 S + 60)   (logit add / subtract, two expf at <= 2 ulp, 1/sum, the row sum over
#                                                             at most 2 NP + 5 sequential adds with NP <= 16)
#   forward, bf16 probs : one more rounding, + 2^-8 * ref
#   backward            : ds = p (dp - D) scale with D = sum_j p_j dp_j; the fp32 row dot product is off by at most
#                         (2 NP + 8) u sum_j |p_j dp_j|, the three roundings of the element by 2^-22 |p scale| (|dp| + |D|);
#                         bf16 outputs add 2^-8 |ref|.  dbd holds the same values moved through the inverse shift.
# Columns [Tk, ld) of probs / dscores / dbd must be exactly 0 (the buffers start as NaN).
# ---------------------------------------------------------------------------------------------------------------------------------
U32 = 2.0 ** -24
DTYPES = [(torch.float32, torch.float32), (torch.float32, torch.bfloat16), (torch.bfloat16, torch.bfloat16)]  # (scores, probs)


def _np_bucket(ld):
    return 1 if ld <= 64 else 2 if ld <= 128 else 5 if ld <= 320 else 7 if ld <= 448 else 16


def _key_len(lens, mode, B, Tk):
    if mode == 0:
        return torch.full((B,), Tk, dtype=torch.int64)
    k = lens.cpu() + (1 if mode == 2 else 0)
    if mode == 3:
        k = (lens.cpu() + 3) // 4
    return k.clamp(0, Tk)


def _softmax_case(B, H, Tq, Tk, ld, sdt, pdt, mode, causal, rel, lens, seed, scale=0.125):
    """Run lasr_attn_softmax_fwd and _bwd once (rel: with the legacy rel_shift of bd) and check every output element."""
    from liteasr_b200 import ops
    from oracle.u2_oracle import rel_shift
    g = torch.Generator(device="cuda").manual_seed(seed)
    nan = float("nan")
    ac = torch.full((B, H, Tq, ld), nan, device="cuda", dtype=sdt)   # padding columns are never read as scores
    ac[..., :Tk] = (torch.randn(B, H, Tq, Tk, generator=g, device="cuda") * 3).to(sdt)
    bd = None
    if rel:
        bd = torch.full((B, H, Tq, ld), nan, device="cuda", dtype=sdt)
        bd[..., :Tk] = (torch.randn(B, H, Tq, Tk, generator=g, device="cuda") * 3).to(sdt)
    probs = torch.full((B, H, Tq, ld), nan, device="cuda", dtype=pdt)
    ops.attn_softmax_fwd(ac, bd, probs, lens, mode, causal, scale, Tk)

    # float64 reference (masked_fill(-1e38) + softmax: a row without keys is uniform 1/Tk, quirk Q4)
    s = ac[..., :Tk].double().cpu()
    if rel:
        s = s + rel_shift(bd[..., :Tk].double().cpu())
    s = s * scale
    S = float(s.abs().max())
    j = torch.arange(Tk)
    mask = (j[None, :] >= _key_len(lens, mode, B, Tk)[:, None])[:, None, None, :]
    if causal:
        mask = mask | (j[None, :] > torch.arange(Tq)[:, None])[None, None]
    ref = torch.softmax(s.masked_fill(mask, -1e38), -1)
    got = probs.double().cpu()
    bound = ref * U32 * (6 * S + 60)
    if pdt == torch.bfloat16:
        bound = bound + 2.0 ** -8 * ref
    assert not torch.isnan(got).any(), "probs: element left unwritten or NaN"
    err = (got[..., :Tk] - ref).abs()
    assert (err <= bound).all(), f"probs: worst excess {float((err - bound).max()):.3g}"
    assert (got[..., Tk:] == 0).all(), "probs: padding columns not zeroed"

    # backward from the probabilities the kernel saved and dprobs of the score dtype
    dp = torch.full((B, H, Tq, ld), nan, device="cuda", dtype=sdt)
    dp[..., :Tk] = torch.randn(B, H, Tq, Tk, generator=g, device="cuda").to(sdt)
    dsc = torch.full((B, H, Tq, ld), nan, device="cuda", dtype=pdt)
    dbd = torch.full((B, H, Tq, ld), nan, device="cuda", dtype=pdt) if rel else None
    ops.attn_softmax_bwd(probs, dp, dsc, dbd, scale, Tk)
    p64, g64 = got[..., :Tk], dp[..., :Tk].double().cpu()
    D = (p64 * g64).sum(-1, keepdim=True)
    ds_ref = p64 * (g64 - D) * scale
    a = p64.abs() * abs(scale)
    ds_bound = a * ((2 * _np_bucket(ld) + 8) * U32 * (p64 * g64).abs().sum(-1, keepdim=True) + 2.0 ** -22 * (g64.abs() + D.abs()))
    if pdt == torch.bfloat16:
        ds_bound = ds_bound + 2.0 ** -8 * (ds_ref.abs() + ds_bound)
    outs = [("dscores", dsc, ds_ref, ds_bound)]
    if rel:
        x = torch.zeros(B, H, Tq, Tk, dtype=torch.float64, requires_grad=True)
        dbd_ref, dbd_bound = (torch.autograd.grad(rel_shift(x), x, t)[0] for t in (ds_ref, ds_bound))
        outs.append(("dbd", dbd, dbd_ref, dbd_bound))
    for name, out, r, bnd in outs:
        o = out.double().cpu()
        assert not torch.isnan(o).any(), f"{name}: element left unwritten or NaN"
        e = (o[..., :Tk] - r).abs()
        assert (e <= bnd).all(), f"{name}: worst excess {float((e - bnd).max()):.3g}"
        assert (o[..., Tk:] == 0).all(), f"{name}: padding columns not zeroed"
    return got


def test_attn_softmax_plain_causal_and_cross():
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(4)
    B, H, Tq, Tk = 3, 2, 9, 9
    ld = 16
    ac = torch.zeros(B, H, Tq, ld, device="cuda")
    ac[..., :Tk] = torch.randn(B, H, Tq, Tk, generator=g, device="cuda")
    ylens = torch.tensor([8, 5, 3], device="cuda")
    probs = torch.empty(B, H, Tq, ld, device="cuda")
    ops.attn_softmax_fwd(ac, None, probs, ylens, 2, 1, 0.5, Tk)   # decoder self-attention: keys j <= i and j < ylen+1
    j = torch.arange(Tk, device="cuda")
    mask = (j[None, None, :] > j[None, :, None]) | (j[None, None, :] >= (ylens + 1)[:, None, None])
    ref = torch.softmax((ac[..., :Tk] * 0.5).masked_fill(mask[:, None], -1e38), -1)
    assert _close(probs[..., :Tk], ref, 1e-5)


# T covers both sides of every NP bucket edge (64, 128, 320, 448) and the largest bucket (T' up to 1024)
@pytest.mark.parametrize("T", [7, 64, 65, 128, 129, 320, 321, 448, 449, 700, 1000])
@pytest.mark.parametrize("sdt,pdt", DTYPES)
@pytest.mark.parametrize("mode", [0, 1, 3])
def test_attn_softmax_relshift_fwd_bwd(T, sdt, pdt, mode):
    """Encoder self-attention (rel_shift of bd, Tq = Tk) at ld = ceil(T, 8) as the engine allocates it.  With a key mask the
    second utterance has no keys at all: every score of its rows is -1e38 and the softmax is uniform 1/Tk, like the reference."""
    B, H = 3, (2 if T <= 448 else 1)
    ld = (T + 7) // 8 * 8
    g = torch.Generator().manual_seed(T * 7 + mode)
    lens = None
    if mode == 1:
        lens = torch.tensor([T + 5, 0, int(torch.randint(1, T, (1,), generator=g)) if T > 1 else 1])
    elif mode == 3:                                           # raw frame counts: klen = ceil(l / 4)
        lens = torch.tensor([4 * T, 0, int(torch.randint(1, 4 * T - 3, (1,), generator=g))])
    lens = lens.cuda() if lens is not None else None
    probs = _softmax_case(B, H, T, T, ld, sdt, pdt, mode, 0, True, lens, seed=T + 100 * mode)
    if mode:
        assert torch.allclose(probs[1, ..., :T].double().cpu(), torch.full((H, T, T), 1.0 / T, dtype=torch.float64), rtol=2.0 ** -8, atol=0)


@pytest.mark.parametrize("sdt,pdt", DTYPES)
@pytest.mark.parametrize("Tq,Tk", [(1, 299), (41, 299), (1, 449), (41, 449)])
def test_attn_softmax_cross_attention(Tq, Tk, sdt, pdt):
    """Decoder source attention: Tq = L + 1 queries against T' encoder frames, encoder key mask (mode 3), no rel-pos term."""
    ld = (Tk + 7) // 8 * 8
    lens = torch.tensor([4 * Tk, 0, 4 * Tk - 13, 5], device="cuda")
    _softmax_case(4, 2, Tq, Tk, ld, sdt, pdt, 3, 0, False, lens, seed=Tq * Tk)


@pytest.mark.parametrize("sdt,pdt", DTYPES)
def test_attn_softmax_decoder_self_attention(sdt, pdt):
    """Decoder self-attention: causal and keys j < ylen + 1 (mode 2), Tq = Tk = 41, no rel-pos term."""
    lens = torch.tensor([40, 0, 17, 3], device="cuda")
    _softmax_case(4, 2, 41, 41, 48, sdt, pdt, 2, 1, False, lens, seed=41)


@pytest.mark.parametrize("sdt,pdt", DTYPES)
@pytest.mark.parametrize("Tk,ld", [(99, 100), (449, 450), (100, 128), (321, 384), (100, 200), (300, 512)])
def test_attn_softmax_padding_columns(Tk, ld, sdt, pdt):
    """include/lasr.h: columns [Tk, ld) of probs, dscores and dbd are zeroed for any even ld <= 1024, including a row buffer
    wider than the bucket that Tk alone would pick ((100, 200), (300, 512))."""
    lens = torch.tensor([4 * Tk, 4 * Tk - 9], device="cuda")
    _softmax_case(2, 2, Tk, Tk, ld, sdt, pdt, 3, 0, True, lens, seed=Tk + ld)


@pytest.mark.parametrize("rows,d", [(37674, 256), (1000, 512), (77, 64), (5166, 144)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_pos_bias_bwd(rows, d, dtype):
    """dq = dqu + dqv, du += colsum(dqu), dv += colsum(dqv), dq-bias += colsum(dq): the backward of q + pos_bias_u / q + pos_bias_v
    (nets/attention.py:135-139); bf16 with d % 8 == 0 takes the wide kernel, everything else the generic one."""
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(rows + d)
    wide = torch.randn(rows, 2 * d + 8, generator=g, device="cuda").to(dtype)   # strided views of a wider buffer
    dqu, dqv = wide[:, :d], wide[:, d:2 * d]
    out = torch.full((rows, 3 * d), float("nan"), device="cuda", dtype=dtype)
    du0, dv0, db0 = (torch.randn(d, generator=g, device="cuda") for _ in range(3))
    du, dv, db = du0.clone(), dv0.clone(), db0.clone()
    ops.pos_bias_bwd(dqu, dqv, out[:, :d], du, dv, db)
    torch.cuda.synchronize()
    want = (dqu.float() + dqv.float()).to(dtype)
    assert torch.equal(out[:, :d], want) and torch.isnan(out[:, d:]).all()
    su, sv = dqu.double().sum(0), dqv.double().sum(0)
    scale = max(1.0, float(su.abs().max()), float(sv.abs().max()))
    assert float((du.double() - du0.double() - su).abs().max()) <= 1e-4 * scale
    assert float((dv.double() - dv0.double() - sv).abs().max()) <= 1e-4 * scale
    assert float((db.double() - db0.double() - su - sv).abs().max()) <= 2e-4 * scale
