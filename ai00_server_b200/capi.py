"""ctypes binding of include/b200rwkv.h (the C-ABI shared library is the product; this file is
only the Python-side loader used by tests/ and bench.py).

The library is loaded from the package directory (built in-tree by ai00_server_b200.build);
loading fails loudly if it is missing — there is no CPU or eager fallback for any entry point.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200rwkv.so")

OK = 0
ERR_INVALID, ERR_UNSUPPORTED, ERR_CUDA, ERR_STATE = -1, -2, -3, -4
OPTION_LAST, OPTION_FULL, OPTION_NONE = 0, 1, 2
OPTION_SCORE, OPTION_SCORE_KEPT = 3, 4      # b200rwkv_infer_score only
TP_HANDLE_BYTES = 128
PLAN_INTS = 48            # B200RWKV_PLAN_INTS: one b200rwkv_debug_plan record


class Info(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "version", "num_layer", "num_emb", "num_hidden", "num_vocab", "num_head", "head_size",
        "time_mix_adapter", "time_decay_adapter")]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


MAX_LORA = 4


class Options(C.Structure):
    """b200rwkv_options (include/b200rwkv.h)."""
    _fields_ = [("struct_bytes", C.c_uint32), ("max_batch", C.c_int32), ("token_chunk_size", C.c_int32), ("precision", C.c_int32),
                ("num_devices", C.c_int32), ("devices", C.c_int32 * 8), ("num_lora", C.c_int32),
                ("lora_st", C.c_void_p * MAX_LORA), ("lora_len", C.c_size_t * MAX_LORA), ("lora_alpha", C.c_float * MAX_LORA),
                ("quant_layers", C.c_int32), ("quant_type", C.c_int32)]


QUANT_NONE, QUANT_INT8, QUANT_NF4 = 0, 1, 2


class B200Error(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"b200rwkv error {code}: {msg}")
        self.code = code


# every symbol include/b200rwkv.h declares: (name, restype, argtypes)
_P = C.c_void_p
SYMBOLS = [
    ("b200rwkv_info_from_st", C.c_int32, [_P, C.c_size_t, C.POINTER(Info)]),
    ("b200rwkv_create", C.c_int32, [_P, C.c_size_t, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(_P)]),
    ("b200rwkv_create_ex", C.c_int32, [_P, C.c_size_t, C.POINTER(Options), C.POINTER(_P)]),
    ("b200rwkv_create_tp", C.c_int32, [_P, C.c_size_t, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(_P)]),
    ("b200rwkv_tp_export", C.c_int32, [_P, _P]),
    ("b200rwkv_tp_connect", C.c_int32, [_P, _P]),
    ("b200rwkv_tp_connect_local", C.c_int32, [C.POINTER(_P), C.c_int32]),
    ("b200rwkv_destroy", None, [_P]),
    ("b200rwkv_get_info", C.c_int32, [_P, C.POINTER(Info)]),
    ("b200rwkv_infer", C.c_int32, [_P, C.c_int32, _P, _P, _P, _P, _P, C.c_size_t, _P]),
    ("b200rwkv_infer_score", C.c_int32, [_P, C.c_int32, _P, _P, _P, _P, _P, C.c_size_t, _P, _P, C.c_size_t]),
    ("b200rwkv_state_shape", C.c_int32, [_P, C.POINTER(C.c_int64 * 4)]),
    ("b200rwkv_state_init", C.c_int32, [_P, _P]),
    ("b200rwkv_state_load", C.c_int32, [_P, C.c_int32, _P]),
    ("b200rwkv_state_back", C.c_int32, [_P, C.c_int32, _P]),
    ("b200rwkv_state_read", C.c_int32, [_P, C.c_int32, C.POINTER(C.c_uint64)]),
    ("b200rwkv_state_write", C.c_int32, [_P, C.c_int32, C.c_uint64]),
    ("b200rwkv_state_free", C.c_int32, [_P, C.c_uint64]),
    ("b200rwkv_snapshot_back", C.c_int32, [_P, C.c_uint64, _P, _P]),
    ("b200rwkv_snapshot_load", C.c_int32, [_P, _P, _P, C.POINTER(C.c_uint64)]),
    ("b200rwkv_cache_stats", C.c_int32, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    ("b200rwkv_read_state", C.c_int32, [C.POINTER(Info), _P, C.c_size_t, _P]),
    ("b200rwkv_softmax", C.c_int32, [_P, C.c_int32, _P, _P]),
    ("b200rwkv_sample_topk", C.c_int32, [_P, C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int32, _P, _P]),
    ("b200rwkv_host_alloc", C.c_int32, [C.c_size_t, C.POINTER(_P)]),
    ("b200rwkv_host_free", None, [_P]),
    ("b200rwkv_bench_decode", C.c_int32, [_P, C.c_int32, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_int64), _P]),
    ("b200rwkv_profile_step", C.c_int32, [_P, C.c_int32, _P, _P, C.POINTER(C.c_float * 4), C.POINTER(C.c_int32 * 4), C.POINTER(C.c_int64)]),
    ("b200rwkv_profile_insitu", C.c_int32, [_P, C.c_int32, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, C.POINTER(C.c_double)]),
    ("b200rwkv_op_quantize", C.c_int32, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    ("b200rwkv_op_wkv", C.c_int32, [C.c_int32, C.c_int32, C.c_int32, C.c_int32] + [_P] * 14),
    ("b200rwkv_launch_count", C.c_int32, [_P, C.POINTER(C.c_int64)]),
    ("b200rwkv_keep_hidden", C.c_int32, [_P, C.c_int32]),
    ("b200rwkv_last_hidden", C.c_int32, [_P, _P, C.c_size_t]),
    ("b200rwkv_debug_read", C.c_int32, [_P, C.c_char_p, _P, C.c_size_t, C.POINTER(C.c_int32)]),
    ("b200rwkv_debug_plan", C.c_int32, [_P, C.c_int32, C.c_int32, _P, C.c_size_t]),
    ("b200rwkv_debug_trace", C.c_int32, [_P, _P, C.c_size_t, _P, _P]),
    ("b200rwkv_debug_gemm_time", C.c_int32, [_P, C.c_int32, C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_int64), _P]),
    ("b200rwkv_last_error", C.c_char_p, [_P]),
]

# debug build only (libb200rwkv_dbg.so): micro-benchmarks; the B200RWKV_* environment switches are honoured there
DEBUG_SYMBOLS = [
    ("b200rwkv_debug_stream", C.c_int32, [C.c_int32, C.c_int32, C.c_double, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_float)]),
    ("b200rwkv_debug_mma_rate", C.c_int32, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int64)]),
    ("b200rwkv_debug_prefetch", C.c_int32, [C.c_int32, C.c_double, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_int32, C.POINTER(C.c_float)]),
]
DEBUG_LIB_PATH = os.path.join(_HERE, "libb200rwkv_dbg.so")

_lib = None


def debug_lib() -> C.CDLL:
    """The debug build (python -m ai00_server_b200.build --debug); scripts/ only."""
    l = C.CDLL(DEBUG_LIB_PATH)
    for name, res, args in SYMBOLS + DEBUG_SYMBOLS:
        fn = getattr(l, name)
        fn.restype = res
        fn.argtypes = args
    return l


def lib() -> C.CDLL:
    """Load libb200rwkv.so; raises if the CUDA extension has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: run `python -m ai00_server_b200.build` "
                              "(there is no CPU fallback for the RWKV engine)")
        l = C.CDLL(LIB_PATH)
        for name, res, args in SYMBOLS:
            fn = getattr(l, name)          # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(code: int, engine=None):
    if code < 0:
        msg = lib().b200rwkv_last_error(engine)
        raise B200Error(code, msg.decode("utf-8", "replace") if msg else "")
    return code


def ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def info_from_st(st: np.ndarray) -> dict:
    st = np.ascontiguousarray(st, dtype=np.uint8)
    out = Info()
    check(lib().b200rwkv_info_from_st(ptr(st), st.size, C.byref(out)))
    return out.as_dict()


def op_quantize(quant_type: int, w16, device: int = 0):
    """The load-time quantiser on one [N, K] f16 matrix (b200rwkv_op_quantize).  Int8: (codes u8 [N, K], min f16 [N, K/128],
    scale f16 [N, K/128]); NF4: (level indices u8 [N, K], absmax f16 [N, K/64])."""
    w16 = np.ascontiguousarray(w16, np.float16)
    N, K = w16.shape
    nb = K // (128 if quant_type == QUANT_INT8 else 64)
    codes = np.empty((N, K), np.uint8)
    p0 = np.empty((N, nb), np.float16)
    p1 = np.empty((N, nb), np.float16)
    check(lib().b200rwkv_op_quantize(device, quant_type, N, K, ptr(w16), ptr(codes), ptr(p0), ptr(p1) if quant_type == QUANT_INT8 else None))
    return (codes, p0, p1) if quant_type == QUANT_INT8 else (codes, p0)


def op_wkv(version: int, r, k, v, w, state, u=None, a=None, k_k=None, k_a=None, r_k=None, g=None, lnx_w=None, lnx_b=None, device: int = 0):
    """One launch of the WKV kernel (b200rwkv_op_wkv).  r, k, v: [T, H, 64]; state [H, 64, 64] = M[value][key] (updated copy
    returned).  Returns (out [T, H, 64] f32, state)."""
    r = np.ascontiguousarray(r, np.float32)
    T, H, _ = r.shape
    f = lambda x: None if x is None else np.ascontiguousarray(x, np.float32)
    k, v, w, u, a, k_k, k_a, r_k, g, lnx_w, lnx_b = map(f, (k, v, w, u, a, k_k, k_a, r_k, g, lnx_w, lnx_b))
    st = np.array(state, np.float32, copy=True, order="C")
    out = np.empty((T, H, 64), np.float32)
    p = lambda x: None if x is None else ptr(x)
    check(lib().b200rwkv_op_wkv(device, version, T, H, p(r), p(k), p(v), p(w), p(u), p(a), p(k_k), p(k_a), p(r_k), p(g), p(lnx_w),
                                p(lnx_b), p(st), p(out)))
    return out, st
