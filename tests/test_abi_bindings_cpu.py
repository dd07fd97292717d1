"""CPU: every ctypes call the Python side makes passes arguments whose C kinds match the prototype in include/lasr.h.

liteasr_b200/_lib.py sets no ``argtypes``, so ctypes converts whatever it is handed: a ``c_int`` where the C side takes an
``int64_t``, or a Python float where it takes a ``float``, is silently wrong.  Here the loaded library is replaced by a recorder,
every wrapper in ops.py (and the SpecAugment launch) is called once with small CPU tensors, and each recorded call is compared
position by position with the prototype.  A guard asserts that every declared entry point was exercised, so a new one cannot
skip the check.
"""
import ctypes as C
import re

import numpy as np
import pytest
import torch

# declared in include/lasr.h but never called from Python with arguments: the version / arch / error / counter queries, the two
# developer trace hooks (tools/*_trace.py) and the plain LayerNorm backward (ops.py calls lasr_layernorm_bwd_drop)
SKIPPED = {"lasr_version", "lasr_arch", "lasr_last_error", "lasr_launch_count", "lasr_spec_augment_npar",
           "lasr_ffn_bwd_set_trace", "lasr_rel_attn_fwd_set_trace", "lasr_layernorm_bwd"}

_C_KIND = {"int": "i32", "int32_t": "i32", "int64_t": "i64", "long": "i64", "size_t": "i64", "uint32_t": "u32",
           "unsigned": "u32", "float": "f32"}


def _prototypes():
    from liteasr_b200 import _lib
    src = re.sub(r"/\*.*?\*/", "", open(_lib.HEADER_PATH).read(), flags=re.S)
    src = re.sub(r"#.*", "", src)
    protos = {}
    for m in re.finditer(r"\b(lasr_[a-z0-9_]+)\s*\(([^()]*)\)\s*;", src):
        name, params = m.group(1), " ".join(m.group(2).split())
        kinds = []
        if params not in ("", "void"):
            for p in params.split(","):
                p = p.strip()
                if "*" in p:
                    kinds.append("ptr")
                else:
                    ctype = " ".join(p.replace("const ", "").split()[:-1])
                    assert ctype in _C_KIND, f"{name}: unknown parameter type {p!r}"
                    kinds.append(_C_KIND[ctype])
        protos[name] = kinds
    return protos


def _kind(a):
    if a is None or isinstance(a, (C.c_void_p, C.Array, bytes, C._Pointer)) or type(a).__name__ == "CArgObject":
        return "ptr"
    for t, k in ((C.c_int32, "i32"), (C.c_int64, "i64"), (C.c_size_t, "i64"), (C.c_uint32, "u32"), (C.c_float, "f32"),
                 (C.c_double, "f64")):
        if type(a) is t:
            return k
    if isinstance(a, bool) or isinstance(a, int):
        return "i32"       # what ctypes passes a bare Python int as
    if isinstance(a, float):
        return "f64"       # ... and a bare Python float
    return type(a).__name__


class _Recorder:
    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        if not name.startswith("lasr_"):
            raise AttributeError(name)

        def call(*args):
            self.calls.append((name, [_kind(a) for a in args]))
            return 37 if name == "lasr_spec_augment_npar" else 0   # 5 + 2 x 8 + 2 x 8 ints per utterance
        return call


class _FakeCuda(torch.Tensor):
    @property
    def is_cuda(self):
        return True


@pytest.fixture
def recorder(monkeypatch):
    from liteasr_b200 import _lib, ops
    rec = _Recorder()
    monkeypatch.setattr(_lib, "_lib", rec)
    monkeypatch.setattr(ops, "_require_cuda", lambda *ts: None)
    monkeypatch.setattr(ops, "_stream", lambda: C.c_void_p(0))
    monkeypatch.setattr(torch.cuda, "current_stream", lambda *a, **k: type("S", (), {"cuda_stream": 0})())
    return rec


def _call_every_wrapper():
    from liteasr_b200 import ops
    f32, bf = torch.float32, torch.bfloat16
    z = lambda *s, dt=f32: torch.zeros(*s, dtype=dt)  # noqa: E731
    i64 = lambda *s: torch.zeros(*s, dtype=torch.int64)  # noqa: E731
    state = i64(2)
    drop = ops.Drop(state, 3, 0.1)

    a, b = z(128, 64, dt=bf), z(64, 64, dt=bf)
    ops.gemm(a, b, z(128, 64), 128, 64, 64, lda=64, ldb=64, ldc=64, bias=z(64), drop=drop)
    ops.linear(a, b, z(128, 64, dt=bf))
    ops.wgrad2_supported(256, 256)
    ops.wgrad2(z(64, 256, dt=bf), z(64, 256, dt=bf), z(256, 256), 0.5, 2)
    ops.ffn_bwd_supported(64, 256)
    ops.ffn_bwd(z(8, 64, dt=bf), z(8, 256, dt=bf), z(64, 256, dt=bf), z(256, 64, dt=bf), z(8, 256, dt=bf), z(8, 64, dt=bf),
                colsum=z(256), alpha=0.5)
    ops.ffn_fwd_supported(64, 256)
    ops.ffn_fwd(z(8, 64, dt=bf), z(256, 64, dt=bf), z(256), z(64, 256, dt=bf), z(64), z(8, 64), z(8, 256, dt=bf),
                z(8, 256, dt=bf), z(8, 64), 0.5, drop, drop)
    ops.ctc_fwdbwd(z(5, 2, 7), i64(2, 3), i64(2), i64(2), time_major=True, upstream=z(1))
    ops.zero_(z(8))
    ops.cast_bf16(z(8), z(8, dt=bf))
    ops.permute4d(z(2, 3), z(3, 2, dt=bf), (1, 2, 3, 1), (0, 3, 1, 0), (0, 1, 2, 0), accumulate=True)
    ops.layernorm_fwd(z(4, 8), z(8), z(8), z(4, 8), z(4), z(4))
    ops.layernorm_bwd(z(4, 8, dt=bf), z(4, 8), z(4), z(4), z(8), z(4, 8), z(8), z(8), True, dx_lo=z(4, 8, dt=bf), colsum=z(8),
                      drop=drop)
    ops.rng_advance(state)
    ops.philox_raw(torch.zeros(6, dtype=torch.int32), 7)
    ops.dropout(z(4, 8), z(4, 8, dt=bf), drop)
    ops.act_bwd(z(4, 8), z(4, 8), z(4, 8), z(8), ops.ACT_SWISH, 0.5)
    ops.pos_bias_fwd(z(4, 8), z(8), z(8), z(4, 8), z(4, 8))
    ops.pos_bias_bwd(z(4, 8), z(4, 8), z(4, 8), z(8), z(8), z(8))
    ops.embed_fwd(i64(2, 3), z(5, 8), z(3, 8), z(2, 3, 8), 2.0)
    ops.embed_bwd(i64(2, 3), z(2, 3, 8), z(5, 8), 2.0)
    ops.scale_by_scalar(z(8), z(1))
    ops.glu_dwconv_fwd(z(6, 16), z(8, 15), z(8), z(6, 8), z(2, 2, 8), 2, 3, 8)
    ops.glu_dwconv_fwd_lens(z(6, 16), z(8, 15), z(8), z(6, 8), z(2, 2, 8), 2, 3, 8, i64(2))
    ops.bn_finalize(z(2, 2, 8), 2, 8, 6, z(8), z(8), z(8), z(8), i64(1), True)
    ops.bn_swish_fwd(z(6, 8), z(8), z(8), z(8), z(8), z(6, 8, dt=bf))
    ops.bn_swish_bwd_stats(z(6, 8), z(6, 8), z(8), z(8), z(8), z(8), z(1, 2, 8), z(2, 8), z(8), z(8))
    ops.dwconv_glu_bwd(z(6, 8), z(6, 8), z(6, 16), z(8), z(8), z(8), z(8), z(2, 8), z(8, 15), z(6, 16), z(8, 15), z(8), 2, 3, 8,
                       colsum=z(16), wpartial=z(2, 18, 8))
    ops.conv1_fwd(z(2, 9, 9), z(8, 9), z(8), z(2, 4, 4, 8))
    ops.conv1_bwd(z(2, 9, 9), z(2, 4, 4, 8), z(8, 9), z(8))
    ops.im2col_s2(z(2, 4, 4, 8), z(2, 72))
    ops.col2im_s2_relu(z(2, 72), z(2, 4, 4, 8), z(2, 4, 4, 8))
    ops.plane_dims(9, 9)
    ops.planes_supported(64, 9, 9)
    ops.conv1_fwd_planes(z(2, 9, 9), z(64, 9), z(64), z(2, 4, 4, 64, dt=bf))
    ops.conv1_bwd_planes(z(2, 9, 9), z(2, 4, 4, 64, dt=bf), z(64, 9), z(64))
    ops.conv2_fwd(z(2, 4, 4, 64, dt=bf), z(64, 576, dt=bf), z(64), z(2, 3, 64, dt=bf), 2, 9, 9)
    ops.conv2_dgrad(z(2, 3, 64, dt=bf), z(64, 576, dt=bf), z(2, 4, 4, 64, dt=bf), z(2, 4, 4, 64, dt=bf), 2, 9, 9)
    ops.conv2_wgrad(z(2, 3, 64, dt=bf), z(2, 4, 4, 64, dt=bf), z(64, 576), 2, 9, 9)
    ops.attn_softmax_fwd(z(2, 2, 5, 8), z(2, 2, 5, 8), z(2, 2, 5, 8, dt=bf), i64(2), 3, 0, 0.125, 5)
    ops.attn_softmax_bwd(z(2, 2, 5, 8, dt=bf), z(2, 2, 5, 8), z(2, 2, 5, 8, dt=bf), z(2, 2, 5, 8, dt=bf), 0.125, 5)
    ops.rel_attn_fwd_supported(5, 64)
    q = z(10, 128, dt=bf)
    ops.rel_attn_fwd(q, q, q, q, z(5, 128, dt=bf), z(2, 2, 5, 8, dt=bf), q, i64(2), 3, 0.125, 2, 2, 5, 64)
    ops.attn_bwd_pair_supported(5, 64)
    ops.attn_bwd_pair(z(2, 2, 5, 8, dt=bf), q, q, q, z(5, 128), 2, 2, 5, 5, 64, r_batched=False, reduce_b=True)
    ops.attn_bwd_pair(z(2, 2, 5, 8, dt=bf), q, q, q, q, 2, 2, 5, 5, 64, colsum=z(128))
    ops.lsmooth_kl_fwdbwd(z(8, 16), i64(2, 3), i64(2), 13, 0.1, 0.5, z(1), z(8), z(8, 16))
    ops.hybrid_combine(z(2), z(8), 0.3, z(3))
    ops.clip_adam_step(z(8), z(8), z(8), z(8), z(8), z(1024), lr=1e-3)
    ops.logsoftmax_topk(z(4, 16), 3, vocab=13, want_lse=True, want_full=True)
    ops.gather_logp(z(4, 16), z(4), i64(4), 13)
    ops.ctc_prefix_beam_search_host(np.zeros((4, 3), np.float32), np.zeros((4, 3), np.int32), beam=2)
    ops.ctc_prefix_beam_search_batch(z(8, 3), torch.zeros(8, 3, dtype=torch.int32), i64(2), 4, beam=2)

    from liteasr_b200.utils.transform.spec_augment import SpecAugment
    xs = torch.Tensor._make_subclass(_FakeCuda, z(2, 6, 5))   # apply_batch refuses tensors that are not on the GPU
    sa = SpecAugment.__new__(SpecAugment)
    sa.cfg = type("Cfg", (), {"replace_with_zero": False})()
    sa.apply_batch(xs, [dict(t=6, center=-1, warped=-1, freq=[(0, 1)], time=[(1, 2)])] * 2)


def test_every_ctypes_call_matches_the_header(recorder):
    protos = _prototypes()
    assert len(protos) >= 60 and "lasr_attn_softmax_fwd" in protos
    _call_every_wrapper()
    seen = set()
    for name, kinds in recorder.calls:
        assert name in protos, f"{name} is called but not declared in include/lasr.h"
        assert kinds == protos[name], f"{name}: passed {kinds}, declared {protos[name]}"
        seen.add(name)
    missing = set(protos) - SKIPPED - seen
    assert not missing, f"declared entry points no wrapper call exercised: {sorted(missing)}"
    assert not (SKIPPED - set(protos)), "skip list names a symbol the header no longer declares"


def test_kind_classifier_tells_the_widths_apart():
    assert [_kind(v) for v in (C.c_int(1), C.c_int64(1), C.c_size_t(1), C.c_uint32(1), C.c_float(1), 1, 1.0, None,
                               C.c_void_p(0), (C.c_int64 * 4)(), C.byref(C.c_int32(0)))] == \
        ["i32", "i64", "i64", "u32", "f32", "i32", "f64", "ptr", "ptr", "ptr", "ptr"]
