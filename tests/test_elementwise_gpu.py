"""GPU: the bandwidth kernels of csrc/elementwise.cu through the C ABI, element by element against float64 or bit-exact torch
references built from the same rounded inputs: activation backward + bias gradient, q + pos_bias, the weight relayouts and
their gradient scatters, the fp32 -> bf16 weight cast, the device-scalar scale and the decoder embedding.

Bounds (u = 2^-24):
  act_bwd dh   : none / relu one fp32 rounding (u |ref|); swish adds the fast-exp sigmoid, |scale da| 2^-19 (1 + |h|);
                 bf16 adds 2^-8 |ref|.  relu'(0) = 0 exactly.
  act_bwd dbias: per column, (ceil(rows/64) + 24) u sum_r |term_r| (16 rows per thread, 4-way shared reduce, one atomic per
                 64-row CTA) plus the per-term swish error.
  embed_fwd    : u (|e scale| + |ref|) (one or two roundings: nvcc may contract the multiply-add).
  embed_bwd    : (hits + 1) u (sum |terms| + |initial|) per element.
Everything else is bit-exact.
"""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

U32 = 2.0 ** -24
NAN = float("nan")


def _strided(rows, cols, dtype, fill=NAN):
    """A (rows, cols) view of a (rows, ceil(cols, 4) + 4) buffer filled with ``fill``: ld > cols, ld % 4 == 0."""
    ld = (cols + 3) // 4 * 4 + 4
    return torch.full((rows, ld), fill, device="cuda", dtype=dtype)[:, :cols]


# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rows,cols", [(1, 4), (63, 4233), (64, 256), (1000, 2048), (5166, 4233)])
@pytest.mark.parametrize("act", ["none", "relu", "swish"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_act_bwd(rows, cols, act, dtype):
    from liteasr_b200 import ops
    code = {"none": ops.ACT_NONE, "relu": ops.ACT_RELU, "swish": ops.ACT_SWISH}[act]
    g = torch.Generator(device="cuda").manual_seed(rows * 7 + cols + code)
    scale = 0.37
    da = _strided(rows, cols, dtype)
    da.copy_(torch.randn(rows, cols, generator=g, device="cuda").to(dtype))
    saved = None
    if act != "none":
        saved = _strided(rows, cols, dtype)
        h = torch.randn(rows, cols, generator=g, device="cuda") * 3
        if act == "relu":       # the activation output: >= 0 with exact zeros (and a few -0.0)
            h = h.clamp(min=0)
            h[::7, ::3] = -0.0
        saved.copy_(h.to(dtype))
    dh = _strided(rows, cols, dtype)
    dbias0 = torch.randn(cols, generator=g, device="cuda")
    dbias = dbias0.clone()
    ops.act_bwd(da, saved, dh, dbias, code, scale)

    d64 = da.double() * float(torch.tensor(scale, dtype=torch.float32))
    term_err = torch.zeros_like(d64)
    if act == "relu":
        ref = torch.where(saved.double() > 0, d64, torch.zeros_like(d64))
    elif act == "swish":
        x = saved.double()
        sg = torch.sigmoid(x)
        ref = d64 * sg * (1 + x * (1 - sg))
        term_err = d64.abs() * 2.0 ** -19 * (1 + x.abs())
    else:
        ref = d64
    bound = term_err + 2 * U32 * ref.abs()
    if dtype == torch.bfloat16:
        bound = bound + 2.0 ** -8 * (ref.abs() + bound)
    out = dh.double()
    assert not torch.isnan(out).any(), "dh: element left unwritten"
    err = (out - ref).abs()
    assert (err <= bound).all(), f"dh: worst excess {float((err - bound).max()):.3g}"
    if act == "relu":
        assert (out[saved.double() <= 0] == 0).all(), "relu'(0) must be 0"
    assert torch.isnan(dh._base[:, cols:]).all(), "columns past cols must keep their contents"

    colsum = ref.sum(0)
    cbound = (math.ceil(rows / 64) + 24) * U32 * (ref.abs().sum(0) + dbias0.double().abs()) + term_err.sum(0)
    cerr = (dbias.double() - dbias0.double() - colsum).abs()
    assert (cerr <= cbound).all(), f"dbias: worst excess {float((cerr - cbound).max()):.3g}"

    # dbias = None: the same dh; dh = None (bias gradient only, as the engine calls it for act = none): the same dbias
    dh2 = _strided(rows, cols, dtype)
    ops.act_bwd(da, saved, dh2, None, code, scale)
    assert torch.equal(dh2, dh)
    if act == "none":
        db2 = dbias0.clone()
        ops.act_bwd(da, None, None, db2, code, scale)
        cerr2 = (db2.double() - dbias0.double() - colsum).abs()
        assert (cerr2 <= cbound).all()


# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rows,d", [(77, 64), (1000, 144), (5166, 256)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_pos_bias_fwd(rows, d, dtype):
    """qu = q + pos_bias_u, qv = q + pos_bias_v with q the first third of a (rows, 3d) projection output, as the engine reads it."""
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(rows + d)
    qkv = torch.randn(rows, 3 * d, generator=g, device="cuda").to(dtype)
    q = qkv[:, :d]
    u, v = torch.randn(d, generator=g, device="cuda"), torch.randn(d, generator=g, device="cuda")
    out = torch.full((rows, 2 * d + 4), NAN, device="cuda", dtype=dtype)
    qu, qv = out[:, :d], out[:, d:2 * d]
    ops.pos_bias_fwd(q, u, v, qu, qv)
    assert torch.equal(qu, (q.float() + u).to(dtype)) and torch.equal(qv, (q.float() + v).to(dtype))
    assert torch.isnan(out[:, 2 * d:]).all()


# ---------------------------------------------------------------------------------------------------------------------------------
def _permute_calls(d, f2):
    """The engine's four calls (engine.py: _conv2_weight, _out_weight, embed_bwd): (src shape, dst shape, n, src strides,
    dst strides, accumulate, torch expression of dst from src)."""
    return [
        ("conv2_weight", (d, d, 3, 3), (d, 9 * d), (d, 3, 3, d), (9 * d, 3, 1, 9), (9 * d, 3 * d, d, 1), False,
         lambda s: s.permute(0, 2, 3, 1).reshape(d, 9 * d)),
        ("out_weight", (d, d * f2), (d, f2 * d), (d, f2, d, 1), (f2 * d, 1, f2, 0), (f2 * d, d, 1, 0), False,
         lambda s: s.view(d, d, f2).permute(0, 2, 1).reshape(d, f2 * d)),
        ("out_weight_grad", (d, f2 * d), (d, d * f2), (d, f2, d, 1), (f2 * d, d, 1, 0), (f2 * d, 1, f2, 0), True,
         lambda s: s.view(d, f2, d).permute(0, 2, 1).reshape(d, d * f2)),
        ("conv2_weight_grad", (d, 9 * d), (d, d, 3, 3), (d, 3, 3, d), (9 * d, 3 * d, d, 1), (9 * d, 3, 1, 9), True,
         lambda s: s.view(d, 3, 3, d).permute(0, 3, 1, 2)),
    ]


@pytest.mark.parametrize("call", range(4))
@pytest.mark.parametrize("sdt,ddt", [(torch.float32, torch.float32), (torch.float32, torch.bfloat16),
                                     (torch.bfloat16, torch.float32), (torch.bfloat16, torch.bfloat16)])
def test_permute4d(call, sdt, ddt):
    """conv.2 weight: d = 512 (2.36 M elements), out weight: d = 256, F2 = 19 (1.25 M): both above 148 * 16 * 256, so the
    grid-stride loop runs more than one trip."""
    from liteasr_b200 import ops
    d, f2 = (512, 19) if call in (0, 3) else (256, 19)
    name, ss, ds, n, sst, dst_st, acc, fn = _permute_calls(d, f2)[call]
    assert math.prod(n) > 148 * 16 * 256
    g = torch.Generator(device="cuda").manual_seed(call)
    src = torch.randn(ss, generator=g, device="cuda").to(sdt)
    dst0 = torch.randn(ds, generator=g, device="cuda").to(ddt) if acc else torch.full(ds, NAN, device="cuda", dtype=ddt)
    dst = dst0.clone()
    ops.permute4d(src, dst, n, sst, dst_st, accumulate=acc)
    moved = fn(src.float())
    want = (dst0.float() + moved).to(ddt) if acc else moved.to(ddt)
    assert torch.equal(dst, want), name


# ---------------------------------------------------------------------------------------------------------------------------------
def _special_f32():
    """Round-half-even ties (both parities), values just off a tie, +-0, subnormals, +-inf, values that round up to inf, NaN."""
    bits = [0x3F808000, 0x3F818000, 0xBF808000, 0xBF818000,   # ties: even mantissa stays, odd rounds up (both signs)
            0x3F808001, 0x3F807FFF, 0x00000000, 0x80000000,   # just above / below a tie, +0, -0
            0x00000001, 0x00008000, 0x00018000, 0x807FFFFF,   # subnormals (a tie among them too)
            0x7F800000, 0xFF800000, 0x7F7FFFFF, 0xFF7F8000,   # +-inf, FLT_MAX and a negative tie that round to inf
            0x7F7F7FFF, 0x7FC00000, 0x7F800001, 0x4B7F8000]   # largest finite bf16 after rounding, qNaN, sNaN, a large tie
    return torch.from_numpy(np.array(bits, dtype=np.uint32).view(np.float32))


@pytest.mark.parametrize("n", [1, 3, 4, 5, 1023, 1025, 4 * 2 ** 20 + 3])
def test_cast_bf16(n):
    """Bit-exact against torch's round-half-even conversion over the vector body and every tail length."""
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(n)
    x = torch.randn(n, generator=g, device="cuda") * 10
    sp = _special_f32().cuda()
    k = min(n, sp.numel())
    x[:k] = sp[:k]
    x[-k:] = sp[-k:]   # the specials land in the scalar tail as well
    dst = torch.full((n,), NAN, device="cuda", dtype=torch.bfloat16)
    ops.cast_bf16(x, dst)
    want = x.to(torch.bfloat16)
    nan = torch.isnan(want)
    assert torch.equal(torch.isnan(dst), nan)
    assert torch.equal(dst.view(torch.int16)[~nan], want.view(torch.int16)[~nan])


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_scale_by_scalar(dtype):
    """x *= *s with n above the grid cap (148 * 16 CTAs of 256): every element gets exactly one multiply."""
    from liteasr_b200 import ops
    n = 2 * 148 * 16 * 256 + 7
    g = torch.Generator(device="cuda").manual_seed(3)
    x = torch.randn(n, generator=g, device="cuda").to(dtype)
    s = torch.tensor([0.7123], device="cuda")
    want = (x.float() * s).to(dtype)
    ops.scale_by_scalar(x, s)
    assert torch.equal(x, want)


# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,L,d,vocab", [(3, 17, 256, 5000), (1, 1, 4, 3), (5, 40, 144, 37)])
def test_embed_fwd_bwd(B, L, d, vocab):
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(B * L + d)
    tokens = torch.randint(0, vocab, (B, L), generator=g, device="cuda")
    tokens[-1] = vocab - 1                                   # one batch row in which every token is the same: all atomics hit one row
    emb = torch.randn(vocab, d, generator=g, device="cuda")
    pe = torch.randn(L + 3, d, generator=g, device="cuda")
    scale = math.sqrt(d)
    out = torch.full((B, L, d), NAN, device="cuda")
    ops.embed_fwd(tokens, emb, pe, out, scale)
    s32 = float(torch.tensor(scale, dtype=torch.float32))
    es = emb.double()[tokens] * s32
    ref = es + pe.double()[:L]
    err = (out.double() - ref).abs()
    assert (err <= U32 * (1 + 2.0 ** -20) * (es.abs() + ref.abs())).all()

    dout = torch.randn(B, L, d, generator=g, device="cuda")
    demb0 = torch.randn(vocab, d, generator=g, device="cuda")
    demb = demb0.clone()
    ops.embed_bwd(tokens, dout, demb, scale)
    flat = tokens.reshape(-1)
    terms = dout.double().reshape(-1, d) * s32
    want = demb0.double().index_add(0, flat, terms)
    hits = torch.bincount(flat, minlength=vocab).double()[:, None]
    absum = torch.zeros(vocab, d, dtype=torch.float64, device="cuda").index_add(0, flat, terms.abs())
    bound = (hits + 1) * U32 * (absum + demb0.double().abs())
    assert ((demb.double() - want).abs() <= bound).all()
