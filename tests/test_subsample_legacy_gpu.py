"""GPU: the im2col front end (nets/subsampling.py:32-35,42-46) that runs in fp32 mode and, in bf16 mode, whenever the parity-plane
path is not supported (d not in {64, 128, 256, 512, 1024} or T/F < 7): conv1_fwd -> im2col_s2 -> (conv2 as a matmul on the
column matrix) -> col2im_s2_relu -> conv1_bwd, each step against float64 F.conv2d and its autograd evaluated from the tensors
the kernels actually read.

Bounds (u = 2^-24):
  conv1_fwd : 10 u (|b| + sum |w x|) per pre-activation (a chain of 9 fma), relu is 1-Lipschitz; bf16 adds 2^-8 |ref|
  im2col    : a gather, bit-exact
  col2im    : at most 4 terms per element, 3 u sum |terms|; bf16 adds 2^-8 |ref|; exactly 0 where h1 == 0 and on the last conv1
              row / column when T1 / F1 is even (it feeds no conv2 output)
  conv1_bwd : (16 F1 + ceil(B T1 / 16) + 4) u sum |terms| per weight / bias element (16 rows x F1 columns per thread, one
              atomic per CTA)
"""
import math

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

U32 = 2.0 ** -24
NAN = float("nan")


# T1 = (T-3)//2 + 1 and F1 take both parities: (3,3) (32,39) (49,40) (20,40); d = 144, 384 and 1024 are not plane shapes for
# bf16 (144, 384) or run here in fp32 as well, and (7, 7) is the minimum with T2 = F2 = 1
@pytest.mark.parametrize("B,T,Fq,d", [(2, 7, 7, 64), (3, 66, 80, 144), (2, 100, 82, 384), (1, 41, 81, 1024)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_subsample_legacy_chain(B, T, Fq, d, dtype):
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(B * T + Fq + d)
    T1, F1 = (T - 3) // 2 + 1, (Fq - 3) // 2 + 1
    T2, F2 = (T1 - 3) // 2 + 1, (F1 - 3) // 2 + 1
    x = torch.randn(B, T, Fq, generator=g, device="cuda")
    w = torch.randn(d, 9, generator=g, device="cuda") * 0.4
    bias = torch.randn(d, generator=g, device="cuda") * 0.3

    # conv1 + ReLU
    h1 = torch.full((B, T1, F1, d), NAN, device="cuda", dtype=dtype)
    ops.conv1_fwd(x, w, bias, h1)
    x64, w64, b64 = x.double()[:, None], w.double().view(d, 1, 3, 3), bias.double()
    pre = F.conv2d(x64, w64, b64, stride=2).permute(0, 2, 3, 1)
    ref = pre.clamp(min=0)
    mag = F.conv2d(x64.abs(), w64.abs(), b64.abs(), stride=2).permute(0, 2, 3, 1)
    bound = 10 * U32 * mag
    if dtype == torch.bfloat16:
        bound = bound + 2.0 ** -8 * (ref + bound)
    h = h1.double()
    assert not torch.isnan(h).any()
    assert ((h - ref).abs() <= bound).all(), "conv1_fwd"
    assert (h >= 0).all() and (h == 0).any() and (h > 0).any()

    # im2col: col[(b, t2, f2), (kh, kw, c)] = h1[b, 2 t2 + kh, 2 f2 + kw, c]
    col = torch.full((B * T2 * F2, 9 * d), NAN, device="cuda", dtype=dtype)
    ops.im2col_s2(h1, col)
    want = h1.unfold(1, 3, 2).unfold(2, 3, 2)                       # (B, T2, F2, d, kh, kw)
    want = want.permute(0, 1, 2, 4, 5, 3).reshape(B * T2 * F2, 9 * d)
    assert torch.equal(col, want), "im2col_s2 must be a pure gather"

    # conv2 as a float64 matmul on the column matrix equals F.conv2d on h1 with the (o, kh, kw, i) weight layout
    w2 = torch.randn(d, d, 3, 3, generator=g, device="cuda", dtype=torch.float64) / (3 * math.sqrt(d))
    w2k = w2.permute(0, 2, 3, 1).reshape(d, 9 * d)
    y_col = col.double() @ w2k.t()
    y_ref = F.conv2d(h.permute(0, 3, 1, 2), w2, stride=2).permute(0, 2, 3, 1).reshape(B * T2 * F2, d)
    assert torch.allclose(y_col, y_ref, rtol=1e-12, atol=1e-12)

    # col2im + conv1's ReLU mask, from a gradient of the column matrix in the operand dtype
    dcol = torch.randn(B * T2 * F2, 9 * d, generator=g, device="cuda").to(dtype)
    dh1 = torch.full((B, T1, F1, d), NAN, device="cuda", dtype=dtype)
    ops.col2im_s2_relu(dcol, h1, dh1)
    hx = h.permute(0, 3, 1, 2).clone().requires_grad_(True)         # (B, d, T1, F1)
    patches = hx.unfold(2, 3, 2).unfold(3, 3, 2).permute(0, 2, 3, 4, 5, 1).reshape(B * T2 * F2, 9 * d)
    (gath,) = torch.autograd.grad(patches, hx, dcol.double())
    (gabs,) = torch.autograd.grad(patches, hx, dcol.double().abs())
    mask = (h > 0).double()
    dref = gath.permute(0, 2, 3, 1) * mask
    dbound = 3 * U32 * gabs.permute(0, 2, 3, 1) * mask
    if dtype == torch.bfloat16:
        dbound = dbound + 2.0 ** -8 * (dref.abs() + dbound)
    dh = dh1.double()
    assert not torch.isnan(dh).any()
    assert ((dh - dref).abs() <= dbound).all(), "col2im_s2_relu"
    assert (dh[h == 0] == 0).all(), "relu'(0) must be 0"
    if T1 % 2 == 0:
        assert (dh[:, T1 - 1] == 0).all(), "the last conv1 row feeds no conv2 output"
    if F1 % 2 == 0:
        assert (dh[:, :, F1 - 1] == 0).all(), "the last conv1 column feeds no conv2 output"

    # conv1 weight / bias gradient from the masked dh1 the kernel wrote (accumulated into non-zero buffers)
    dw0 = torch.randn(d, 9, generator=g, device="cuda")
    db0 = torch.randn(d, generator=g, device="cuda")
    dw, db = dw0.clone(), db0.clone()
    ops.conv1_bwd(x, dh1, dw, db)
    wv = w64.clone().requires_grad_(True)
    bv = b64.clone().requires_grad_(True)
    gw, gb = torch.autograd.grad(F.conv2d(x64, wv, bv, stride=2), (wv, bv), dh.permute(0, 3, 1, 2))
    gwa, gba = torch.autograd.grad(F.conv2d(x64.abs(), wv, bv, stride=2), (wv, bv), dh.abs().permute(0, 3, 1, 2))
    depth = (16 * F1 + math.ceil(B * T1 / 16) + 4) * U32
    ew = (dw.double() - dw0.double() - gw.view(d, 9)).abs()
    eb = (db.double() - db0.double() - gb).abs()
    assert (ew <= depth * (gwa.view(d, 9) + dw0.double().abs())).all(), "conv1_bwd weight"
    assert (eb <= depth * (gba + db0.double().abs())).all(), "conv1_bwd bias"
