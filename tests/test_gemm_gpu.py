"""GPU: tcgen05 bf16 GEMM and SIMT fp32 GEMM through the C ABI vs a plain fp32 torch reference."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _ref(a, b, ta, tb):
    A = a.float().transpose(-1, -2) if ta else a.float()
    B = b.float().transpose(-1, -2) if tb else b.float()
    return A @ B.transpose(-1, -2)  # (M,K) @ (N,K)^T


def _mk(rows, cols, dtype, g):
    """(rows, cols) view of a buffer whose row stride is padded to 8 elements (TMA needs 16-byte strides)."""
    ld = (cols + 7) // 8 * 8
    buf = (torch.randn(rows, ld, generator=g, device="cuda") * 0.5).to(dtype)
    return buf[:, :cols]


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("ta,tb", [(False, False), (False, True), (True, False), (True, True)])
@pytest.mark.parametrize("m,n,k", [(128, 128, 64), (300, 200, 136), (1000, 256, 2048), (64, 520, 72), (257, 64, 256)])
def test_gemm_plain(dtype, ta, tb, m, n, k):
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(m * 7 + n * 3 + k)
    a = _mk(k, m, dtype, g) if ta else _mk(m, k, dtype, g)
    b = _mk(k, n, dtype, g) if tb else _mk(n, k, dtype, g)
    c = torch.full((m, n), float("nan"), device="cuda")
    ops.gemm(a, b, c, m, n, k, lda=a.stride(0), ldb=b.stride(0), ldc=n, ta=ta, tb=tb)
    ref = _ref(a, b, ta, tb)
    tol = 2e-2 if dtype == torch.bfloat16 else 1e-4
    assert torch.isfinite(c).all()
    err = (c - ref).abs().max().item()
    assert err <= tol * max(1.0, ref.abs().max().item()), err


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_gemm_epilogue_bias_act_res_aux(dtype):
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(5)
    m, n, k = 333, 320, 256
    x, w = _mk(m, k, dtype, g), _mk(n, k, dtype, g)
    bias = torch.randn(n, generator=g, device="cuda")
    res = torch.randn(m, n, generator=g, device="cuda")
    for act, fn in ((ops.ACT_NONE, lambda v: v), (ops.ACT_RELU, torch.relu), (ops.ACT_SWISH, lambda v: v * torch.sigmoid(v))):
        for cdt in ([torch.float32, torch.bfloat16] if dtype == torch.bfloat16 else [torch.float32]):
            out = torch.empty(m, n, device="cuda", dtype=cdt)
            aux = torch.empty(m, n, device="cuda", dtype=cdt)
            r = res if cdt == torch.float32 else None  # the residual stream is fp32: a residual needs an fp32 C
            ops.linear(x, w, out, bias=bias, res=r, aux=aux, alpha=0.5, act=act)
            pre = x.float() @ w.float().t() + bias
            ref = 0.5 * fn(pre) + (res if r is not None else 0.0)
            tol = 3e-2 if (dtype == torch.bfloat16 or cdt == torch.bfloat16) else 1e-4
            assert (out.float() - ref).abs().max().item() <= tol * ref.abs().max().item()
            assert (aux.float() - pre).abs().max().item() <= tol * pre.abs().max().item()


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_gemm_batched_head_interleaved(dtype):
    """Attention-style: A = Q (B,T,H,dk) per (b,h), B = K (B,T,H,dk); C (B,H,T,Tp) fp32."""
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(9)
    B, T, H, dk = 3, 77, 2, 64
    Tp = 80
    q = (torch.randn(B, T, H, dk, generator=g, device="cuda") * 0.3).to(dtype)
    kk = (torch.randn(B, T, H, dk, generator=g, device="cuda") * 0.3).to(dtype)
    c = torch.zeros(B, H, T, Tp, device="cuda")
    d = H * dk
    ops.gemm(q, kk, c, T, T, dk, lda=d, ldb=d, ldc=Tp, batch=(B, H), sa=(T * d, dk), sb=(T * d, dk), sc=(H * T * Tp, T * Tp))
    ref = torch.einsum("bihd,bjhd->bhij", q.float(), kk.float())
    tol = 2e-2 if dtype == torch.bfloat16 else 1e-4
    assert (c[..., :T] - ref).abs().max().item() <= tol * ref.abs().max().item()
    assert (c[..., T:] == 0).all()
    # P.V: A = probs (B,H,T,Tp) K-major, B = V (B,T,H,dk) MN-major (rows = keys); out (B,T,H,dk)
    probs = torch.softmax(ref, -1).to(dtype)
    pp = torch.zeros(B, H, T, Tp, device="cuda", dtype=dtype)
    pp[..., :T] = probs
    v = (torch.randn(B, T, H, dk, generator=g, device="cuda") * 0.3).to(dtype)
    o = torch.empty(B, T, H, dk, device="cuda", dtype=dtype)
    ops.gemm(pp, v, o, T, dk, T, lda=Tp, ldb=d, ldc=d, tb=True, batch=(B, H), sa=(H * T * Tp, T * Tp), sb=(T * d, dk), sc=(T * d, dk))
    ref_o = torch.einsum("bhij,bjhd->bihd", probs.float(), v.float())
    assert (o.float() - ref_o).abs().max().item() <= tol * max(1.0, ref_o.abs().max().item())
    # dV = probs^T . dO : A MN-major (rows = queries), B MN-major; broadcast operand (stride 0) + batch-reduce accumulate
    do = (torch.randn(B, T, H, dk, generator=g, device="cuda") * 0.3).to(dtype)
    dv = torch.empty(B, T, H, dk, device="cuda", dtype=dtype)
    ops.gemm(pp, do, dv, T, dk, T, lda=Tp, ldb=d, ldc=d, ta=True, tb=True, batch=(B, H), sa=(H * T * Tp, T * Tp), sb=(T * d, dk), sc=(T * d, dk))
    ref_dv = torch.einsum("bhij,bihd->bjhd", probs.float(), do.float())
    assert (dv.float() - ref_dv).abs().max().item() <= tol * max(1.0, ref_dv.abs().max().item())
    acc = torch.zeros(H, T, dk, device="cuda")
    ops.gemm(pp, do, acc, T, dk, T, lda=Tp, ldb=d, ldc=dk, ta=True, tb=True, batch=(B, H), sa=(H * T * Tp, T * Tp), sb=(T * d, dk),
             sc=(0, T * dk), accumulate=True)
    ref_acc = torch.einsum("bhij,bihd->hjd", probs.float(), do.float())
    assert (acc - ref_acc).abs().max().item() <= tol * max(1.0, ref_acc.abs().max().item())


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_gemm_wgrad_split_k(dtype):
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(11)
    rows, n, k = 3001, 256, 520
    dy, x = _mk(rows, n, dtype, g), _mk(rows, k, dtype, g)
    dw = torch.zeros(n, k, device="cuda")
    ops.gemm(dy, x, dw, n, k, rows, lda=dy.stride(0), ldb=x.stride(0), ldc=k, ta=True, tb=True, accumulate=True, split_k=5, alpha=2.0)
    ref = 2.0 * dy.float().t() @ x.float()
    tol = 2e-2 if dtype == torch.bfloat16 else 2e-4
    assert (dw - ref).abs().max().item() <= tol * ref.abs().max().item()


@pytest.mark.parametrize("cdt", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("m,n,k,tb", [(9568, 299, 64, False), (1000, 4233, 256, False), (2000, 4233, 320, True), (5000, 2048, 256, False),
                                      (41, 299, 64, False), (777, 152, 192, False), (640, 72, 128, True)])
def test_gemm_persistent_tiles_and_tails(cdt, m, n, k, tb):
    """More work units than SMs (persistent loop + both TMEM accumulator buffers), run-time BN, ragged N with a padded ld."""
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(m + n + k)
    a = _mk(m, k, torch.bfloat16, g)
    b = _mk(k, n, torch.bfloat16, g) if tb else _mk(n, k, torch.bfloat16, g)
    bias = torch.randn(n, generator=g, device="cuda")
    ld = (n + 7) // 8 * 8
    buf = torch.full((m, ld), 7.0, device="cuda", dtype=cdt)
    ops.gemm(a, b, buf[:, :n], m, n, k, lda=a.stride(0), ldb=b.stride(0), ldc=ld, tb=tb, bias=bias, act=ops.ACT_RELU)
    ref = torch.relu(_ref(a, b, False, tb) + bias)
    assert (buf[:, :n].float() - ref).abs().max().item() <= 2e-2 * max(1.0, ref.abs().max().item())
    assert (buf[:, n:] == 7.0).all()  # padding columns untouched


def test_gemm_many_small_batches_short_k():
    """Attention-score shape: 128 batches x (299 x 299 x 64) -> thousands of one-k-block work units."""
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(3)
    B, H, T, dk, ld = 8, 4, 299, 64, 304
    d = H * dk
    q = (torch.randn(B, T, H, dk, generator=g, device="cuda") * 0.3).to(torch.bfloat16)
    kk = (torch.randn(B, T, H, dk, generator=g, device="cuda") * 0.3).to(torch.bfloat16)
    c = torch.zeros(B, H, T, ld, device="cuda")
    ops.gemm(q, kk, c, T, T, dk, lda=d, ldb=d, ldc=ld, batch=(B, H), sa=(T * d, dk), sb=(T * d, dk), sc=(H * T * ld, T * ld))
    ref = torch.einsum("bihd,bjhd->bhij", q.float(), kk.float())
    assert (c[..., :T] - ref).abs().max().item() <= 2e-2 * ref.abs().max().item()
    assert (c[..., T:] == 0).all()


def test_gemm_bad_args_raise():
    from liteasr_b200 import ops
    a = torch.zeros(8, 8, device="cuda", dtype=torch.bfloat16)
    c = torch.zeros(8, 8, device="cuda")
    with pytest.raises(RuntimeError):
        ops.gemm(a, a, c, 8, 8, 8, lda=8, ldb=8, ldc=8, split_k=2)  # split_k without accumulate
    with pytest.raises(RuntimeError):
        ops.gemm(a, a, c, 8, 8, 8, lda=9, ldb=8, ldc=8)  # unaligned TMA stride


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("act", ["swish", "relu"])
@pytest.mark.parametrize("m,n,k", [(333, 320, 256), (1000, 2048, 256), (77, 100, 64)])
def test_gemm_fused_activation_backward_and_colsum(dtype, act, m, n, k):
    """dgrad epilogue: C = alpha * (dy @ W) * act'(saved), colsum += sum_rows C (bias gradient) -- nets/feed_forward.py:18-19 backward."""
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(m + n)
    dy, w = _mk(m, k, dtype, g), _mk(k, n, dtype, g)   # W stored (N_out=k, K_in=n): dx = dy @ W
    saved = _mk(m, n, dtype, g)
    cs = torch.randn(n, generator=g, device="cuda")
    cs0 = cs.clone()
    ld = (n + 7) // 8 * 8
    out = torch.empty(m, ld, device="cuda", dtype=dtype)[:, :n]
    code = ops.ACT_SWISH if act == "swish" else ops.ACT_RELU
    ops.gemm(dy, w, out, m, n, k, lda=dy.stride(0), ldb=w.stride(0), ldc=ld, tb=True, alpha=0.5, dact=saved, act=code, colsum=cs)
    sv = saved.float()
    sg = torch.sigmoid(sv)
    dact = sg * (1 + sv * (1 - sg)) if act == "swish" else (sv > 0).float()
    ref = 0.5 * (dy.float() @ w.float()) * dact
    tol = 3e-2 if dtype == torch.bfloat16 else 1e-4
    assert (out.float() - ref).abs().max().item() <= tol * max(1.0, ref.abs().max().item())
    assert (cs - cs0 - ref.sum(0)).abs().max().item() <= tol * max(1.0, ref.sum(0).abs().max().item())


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_gemm_batched_colsum_per_head(dtype):
    """dK-style GEMM: C (B,T,H,dk) head-interleaved; colsum[h*dk + c] += sum over batch and rows (k-projection bias gradient)."""
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(21)
    B, T, H, dk, Tp = 3, 77, 2, 64, 80
    d = H * dk
    ds = torch.zeros(B, H, T, Tp, device="cuda", dtype=dtype)
    ds[..., :T] = (torch.randn(B, H, T, T, generator=g, device="cuda") * 0.3).to(dtype)
    q = (torch.randn(B, T, H, dk, generator=g, device="cuda") * 0.3).to(dtype)
    dkk = torch.empty(B, T, H, dk, device="cuda", dtype=dtype)
    cs = torch.zeros(d, device="cuda")
    ops.gemm(ds, q, dkk, T, dk, T, lda=Tp, ldb=d, ldc=d, ta=True, tb=True, batch=(B, H), sa=(H * T * Tp, T * Tp), sb=(T * d, dk),
             sc=(T * d, dk), colsum=cs, cs=(0, dk))
    ref = torch.einsum("bhij,bihd->bjhd", ds[..., :T].float(), q.float())
    tol = 2e-2 if dtype == torch.bfloat16 else 1e-4
    assert (dkk.float() - ref).abs().max().item() <= tol * max(1.0, ref.abs().max().item())
    assert (cs - ref.sum((0, 1)).reshape(-1)).abs().max().item() <= tol * max(1.0, ref.sum((0, 1)).abs().max().item())


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_gemm_n_store_pads_with_zeros(dtype):
    """Attention-score call: N = 299 keys in a 304-wide buffer, n_store = 304 -> padding columns written as zeros."""
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(31)
    B, H, T, dk, ld = 2, 2, 299, 64, 304
    d = H * dk
    q = (torch.randn(B, T, H, dk, generator=g, device="cuda") * 0.3).to(dtype)
    kk = (torch.randn(B, T, H, dk, generator=g, device="cuda") * 0.3).to(dtype)
    c = torch.full((B, H, T, ld), 5.0, device="cuda")
    ops.gemm(q, kk, c, T, T, dk, lda=d, ldb=d, ldc=ld, batch=(B, H), sa=(T * d, dk), sb=(T * d, dk), sc=(H * T * ld, T * ld), n_store=ld)
    ref = torch.einsum("bihd,bjhd->bhij", q.float(), kk.float())
    tol = 2e-2 if dtype == torch.bfloat16 else 1e-4
    assert (c[..., :T] - ref).abs().max().item() <= tol * ref.abs().max().item()
    assert (c[..., T:] == 0).all()


def _swish(v):
    return v * torch.sigmoid(v)


def _dswish(v):
    s = torch.sigmoid(v)
    return s * (1 + v * (1 - s))


# The row count of the C2 FFN GEMMs at B = 126 (m = 37 674) with K <= 256: many M tiles per CTA, for every fused epilogue.
@pytest.mark.parametrize("m,n,k", [(37674, 256, 256), (37674, 2048, 256), (37674, 512, 200), (56000, 256, 64), (37674, 4233, 256)])
@pytest.mark.parametrize("tb", [False, True])
def test_gemm_c2_rows_plain_bias_bf16_and_f32(m, n, k, tb):
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(m + n + k)
    x = _mk(m, k, torch.bfloat16, g)
    w = _mk(k, n, torch.bfloat16, g) if tb else _mk(n, k, torch.bfloat16, g)
    bias = torch.randn(n, generator=g, device="cuda")
    ref = x.float() @ (w.float() if tb else w.float().t())
    ldn = (n + 7) // 8 * 8
    for cdt in (torch.bfloat16, torch.float32):
        use_bias = not tb
        c = torch.full((m, ldn), float("nan"), device="cuda", dtype=cdt)[:, :n]
        ops.gemm(x, w, c, m, n, k, lda=x.stride(0), ldb=w.stride(0), ldc=c.stride(0), tb=tb, bias=bias if use_bias else None, alpha=0.5)
        want = 0.5 * (ref + (bias if use_bias else 0.0))
        assert torch.isfinite(c.float()).all()
        err = (c.float() - want).abs().max().item()
        assert err <= (3e-2 if cdt == torch.bfloat16 else 2e-3) * max(1.0, want.abs().max().item()), (cdt, err)


def test_gemm_c2_rows_swish_aux_relu_res():
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(11)
    m, n, k = 37674, 2048, 256
    x, w = _mk(m, k, torch.bfloat16, g), _mk(n, k, torch.bfloat16, g)
    bias = torch.randn(n, generator=g, device="cuda")
    pre = x.float() @ w.float().t() + bias
    out = torch.empty(m, n, device="cuda", dtype=torch.bfloat16)
    aux = torch.empty(m, n, device="cuda", dtype=torch.bfloat16)
    ops.linear(x, w, out, bias=bias, aux=aux, act=ops.ACT_SWISH)
    assert (aux.float() - pre).abs().max().item() <= 3e-2 * pre.abs().max().item()
    assert (out.float() - _swish(pre)).abs().max().item() <= 3e-2 * pre.abs().max().item()
    ops.linear(x, w, out, bias=bias, act=ops.ACT_RELU, alpha=2.0)
    assert (out.float() - 2.0 * torch.relu(pre)).abs().max().item() <= 3e-2 * 2 * pre.abs().max().item()
    # fp32 C with residual (N = 256: one N tile)
    n2 = 256
    w2 = _mk(n2, k, torch.bfloat16, g)
    res = torch.randn(m, n2, generator=g, device="cuda")
    o32 = torch.empty(m, n2, device="cuda")
    ops.linear(x, w2, o32, bias=bias[:n2].contiguous(), res=res, alpha=0.5)
    want = 0.5 * (x.float() @ w2.float().t() + bias[:n2]) + res
    assert (o32 - want).abs().max().item() <= 2e-2 * want.abs().max().item()


@pytest.mark.parametrize("act", ["swish", "relu"])
def test_gemm_c2_rows_fused_activation_backward_and_colsum(act):
    from liteasr_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(13)
    m, n, k = 37674, 2048, 256
    dy = _mk(m, k, torch.bfloat16, g)
    w = _mk(k, n, torch.bfloat16, g)  # (N_out = k, K_in = n) weight, MN-major B
    saved = _mk(m, n, torch.bfloat16, g)
    dx = torch.empty(m, n, device="cuda", dtype=torch.bfloat16)
    cs = torch.zeros(n, device="cuda")
    ops.gemm(dy, w, dx, m, n, k, lda=dy.stride(0), ldb=w.stride(0), ldc=n, tb=True, alpha=0.5, dact=saved,
             act=ops.ACT_SWISH if act == "swish" else ops.ACT_RELU, colsum=cs)
    d = _dswish(saved.float()) if act == "swish" else (saved.float() > 0).float()
    want = 0.5 * (dy.float() @ w.float()) * d
    assert (dx.float() - want).abs().max().item() <= 3e-2 * max(1.0, want.abs().max().item())
    ref_cs = want.sum(0)
    assert (cs - ref_cs).abs().max().item() <= 2e-2 * max(1.0, ref_cs.abs().max().item()) + 0.5
