"""ctypes binding of liblasr.so (the C ABI in include/lasr.h).  No CPU fallback: a missing library or a
failing call raises ``RuntimeError``."""
from __future__ import annotations

import ctypes as C
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LASR_LIB_PATH") or os.path.join(_HERE, "liblasr.so")  # LASR_LIB_PATH: developer A/B builds
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "lasr.h")
ALIGN_HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "lasr_align.h")
FBANK_HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "lasr_fbank.h")

F32, BF16 = 0, 1
I16 = 2  # int16 samples (include/lasr_fbank.h: LASR_I16)
ACT_NONE, ACT_RELU, ACT_SWISH, ACT_MUL = 0, 1, 2, 3


class GemmArgs(C.Structure):
    _fields_ = [
        ("a", C.c_void_p), ("b", C.c_void_p), ("c", C.c_void_p),
        ("bias", C.c_void_p), ("res", C.c_void_p), ("aux", C.c_void_p),
        ("m", C.c_int32), ("n", C.c_int32), ("k", C.c_int32),
        ("ab_dtype", C.c_int32), ("c_dtype", C.c_int32),
        ("trans_a", C.c_int32), ("trans_b", C.c_int32),
        ("lda", C.c_int64), ("ldb", C.c_int64), ("ldc", C.c_int64), ("ldres", C.c_int64),
        ("batch1", C.c_int32), ("batch2", C.c_int32),
        ("sa1", C.c_int64), ("sa2", C.c_int64), ("sb1", C.c_int64), ("sb2", C.c_int64),
        ("sc1", C.c_int64), ("sc2", C.c_int64),
        ("alpha", C.c_float), ("act", C.c_int32), ("accumulate", C.c_int32), ("split_k", C.c_int32),
        ("dact", C.c_void_p), ("lddact", C.c_int64), ("colsum", C.c_void_p), ("cs1", C.c_int64), ("cs2", C.c_int64),
        ("n_store", C.c_int32),
        ("drop_state", C.c_void_p), ("drop_site", C.c_uint32), ("drop_thr", C.c_uint32), ("drop_scale", C.c_float),
        ("drop_mark_aux", C.c_int32), ("aux_deriv", C.c_int32),
    ]


_lib = None


def declared_symbols(header: str = HEADER_PATH) -> list:
    """Every function name declared in include/lasr.h, or in ``header`` (used by the symbol-export tests)."""
    with open(header) as f:
        src = f.read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(lasr_[a-z0-9_]+)\s*\(", src)))


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m liteasr_b200.build` "
                "(liteasr_b200 has no CPU fallback)")
        _lib = C.CDLL(LIB_PATH)
        _lib.lasr_last_error.restype = C.c_char_p
        _lib.lasr_ctc_workspace_bytes.restype = C.c_size_t
        _lib.lasr_ctc_prefix_beam_search_batch_workspace.restype = C.c_size_t
        _lib.lasr_ctc_forced_align_workspace.restype = C.c_size_t
        _lib.lasr_launch_count.restype = C.c_ulonglong
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().lasr_last_error().decode(errors="replace")
        raise RuntimeError(f"liblasr {what} failed (rc={rc}): {msg}")


def launch_count() -> int:
    return int(lib().lasr_launch_count())
