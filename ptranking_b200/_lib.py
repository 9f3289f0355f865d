"""ctypes binding of libptranking_b200.so (the C ABI declared in include/ptranking_b200.h).

There is no CPU fallback: if the shared library is missing or the device is not
sm_100, loading raises -- the product path never routes around the CUDA kernels.
"""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "lib", "libptranking_b200.so")

MAX_FF_LAYERS = 16
MAX_CUTOFFS = 32
MAX_LIST_LEN = 4096

AF_CODES = {None: 0, "R": 1, "GE": 2, "S": 3, "T": 4, "CE": 5, "E": 6, "LR": 7, "SE": 8}
NORM_CODES = {None: 0, "BN": 1, "BN2": 2}
MATH_MODES = {"simt": 0, "3xtf32": 1, "tf32": 2, "bf16": 3}
LAMBDALOSS_TYPES = {"NDCG_Loss1": 0, "NDCG_Loss2": 1, "NDCG_Loss2++": 2}
WASS_COST_TYPES = {"eg": 0, "p1": 1, "p2": 2, "dg": 3, "ddg": 4}
WASS_SMOOTH_TYPES = {"ST": 0, "NG": 1}

_fp = C.c_void_p   # device pointers travel as integers


class FFNetDesc(C.Structure):
    """struct ptrb200_ffnet"""
    _fields_ = [
        ("num_linear", C.c_int),
        ("dims", C.c_int * (MAX_FF_LAYERS + 1)),
        ("act_hidden", C.c_int),
        ("act_tail", C.c_int),
        ("norm", C.c_int),
        ("norm_affine", C.c_int),
        ("dropout_p", C.c_float),
        ("math_mode", C.c_int),
        ("sync_bn", C.c_int),
        ("weight", _fp * MAX_FF_LAYERS),
        ("bias", _fp * MAX_FF_LAYERS),
        ("gamma", _fp * MAX_FF_LAYERS),
        ("beta", _fp * MAX_FF_LAYERS),
        ("aff_w", _fp * MAX_FF_LAYERS),
        ("aff_b", _fp * MAX_FF_LAYERS),
    ]


class FFNetGrads(C.Structure):
    """struct ptrb200_ffnet_grads"""
    _fields_ = [(name, _fp * MAX_FF_LAYERS) for name in ("weight", "bias", "gamma", "beta", "aff_w", "aff_b")]


# name -> (restype, argtypes); mirrors include/ptranking_b200.h one to one
_I, _F, _U64, _I64 = C.c_int, C.c_float, C.c_uint64, C.c_int64
SIGNATURES = {
    "ptrb200_version": (_I, []),
    "ptrb200_last_error": (C.c_char_p, []),
    "ptrb200_launch_count": (C.c_ulonglong, []),
    "ptrb200_device_ok": (_I, []),
    "ptrb200_timing_enable": (_I, [_I]),
    "ptrb200_timing_report": (_I, [C.c_char_p, _I]),
    "ptrb200_ranknet_fwd_bwd": (_I, [_fp, _fp, _fp, _fp, _fp, _I, _I, _F, _fp]),
    "ptrb200_lambdarank_fwd_bwd": (_I, [_fp, _fp, _fp, _fp, _fp, _I, _I, _F, _fp]),
    "ptrb200_lambdaloss_fwd_bwd": (_I, [_fp, _fp, _fp, _fp, _fp, _I, _I, _I, _F, _F, _I, _I, _fp]),
    "ptrb200_listnet_fwd_bwd": (_I, [_fp, _fp, _fp, _fp, _fp, _I, _I, _fp]),
    "ptrb200_listmle_fwd_bwd": (_I, [_fp, _fp, _fp, _fp, _fp, _I, _I, _fp]),
    "ptrb200_shuffle_ties_perm": (_I, [_fp, _fp, _fp, _I, _I, _U64, _U64, _fp]),
    "ptrb200_approxndcg_fwd_bwd": (_I, [_fp, _fp, _fp, _fp, _fp, _fp, _I, _I, _F, _I, _I, _fp]),
    "ptrb200_rankmse_fwd_bwd": (_I, [_fp, _fp, _fp, _fp, _fp, _I, _I, _fp]),
    "ptrb200_rankcosine_fwd_bwd": (_I, [_fp, _fp, _fp, _fp, _fp, _I, _I, _fp]),
    "ptrb200_stlistnet_fwd_bwd": (_I, [_fp, _fp, _fp, _fp, _fp, _fp, _I, _I, _F, _U64, _U64, _fp]),
    "ptrb200_softrank_fwd_bwd": (_I, [_fp, _fp, _fp, _fp, _fp, _I, _I, _F, _I, _fp]),
    "ptrb200_sinkstep": (_I, [_fp, _fp, _fp, _fp, _I, _I, _I, _F, _fp]),
    "ptrb200_wassrank_fwd_bwd": (_I, [_fp, _fp, _fp, _fp, _fp, _I, _I, _I, _I, _I, _F, _I, _F, _F, _F, _fp]),
    "ptrb200_standard_scale": (_I, [_fp, _fp, _fp, _I, _I, _I, _I, _F, _fp]),
    "ptrb200_sum_f32": (_I, [_fp, _fp, _I, _fp]),
    "ptrb200_ndcg_at_ks": (_I, [_fp, _fp, _fp, C.POINTER(C.c_int32), _I, _fp, _fp, _I, _I, _I, _fp]),
    "ptrb200_adhoc_metrics_at_ks": (_I, [_fp, _fp, _fp, C.POINTER(C.c_int32), _I, _fp, _I, _I, _I, _F, _fp]),
    "ptrb200_attention_fwd": (_I, [_fp, _fp, _fp, _fp, _fp, _I, _I, _I, _I, _F, _U64, _U64, _fp]),
    "ptrb200_adam_step": (_I, [_fp, _fp, _fp, _fp, _I64, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, _I, _fp]),
    "ptrb200_adagrad_step": (_I, [_fp, _fp, _fp, _I64, C.c_double, C.c_double, C.c_double, C.c_double, _I, _fp]),
    "ptrb200_rmsprop_step": (_I, [_fp, _fp, _fp, _I64, C.c_double, C.c_double, C.c_double, C.c_double, _fp]),
    "ptrb200_attention_tc_workspace_floats": (_I64, [_I, _I, _I, _I, _I]),
    "ptrb200_attention_tc_fwd": (_I, [_fp] * 6 + [_I, _I, _I, _I, _F, _U64, _U64, _I, _fp]),
    "ptrb200_attention_tc_bwd": (_I, [_fp] * 9 + [_I, _I, _I, _I, _F, _U64, _U64, _I, _fp]),
    "ptrb200_attention_tc_fwd_ld": (_I, [_fp] * 6 + [_I, _I, _I, _I, _I, _I, _fp, _F, _U64, _U64, _I, _fp]),
    "ptrb200_pad_lists": (_I, [_fp, _fp, _fp, _I, _I, _I, _fp]),
    "ptrb200_unpad_lists": (_I, [_fp, _fp, _fp, _I, _I, _I, _fp]),
    "ptrb200_attention_tc_bwd_ld": (_I, [_fp] * 9 + [_I, _I, _I, _I, _I, _I, _F, _U64, _U64, _I, _fp]),
    "ptrb200_attention_bwd": (_I, [_fp] * 10 + [_I, _I, _I, _I, _F, _U64, _U64, _fp]),
    "ptrb200_layernorm_fwd": (_I, [_fp, _fp, _fp, _fp, _fp, _fp, _I, _I, _F, _fp]),
    "ptrb200_layernorm_bwd": (_I, [_fp] * 9 + [_I, _I, _F, _fp]),
    "ptrb200_elementwise": (_I, [_I, _fp, _fp, _fp, _I64, _F, _U64, _U64, _fp]),
    "ptrb200_tc_gemm_nt": (_I, [_fp, _fp, _fp, _I, _I, _I, _I, _fp]),
    "ptrb200_tc_wgrad": (_I, [_fp, _fp, _fp, _fp, _I, _I, _I, _I, _fp]),
    "ptrb200_ffnet_workspace_bytes": (_I64, [C.POINTER(FFNetDesc), _I, _I, _I]),
    "ptrb200_ffnet_forward": (_I, [C.POINTER(FFNetDesc), _fp, _fp, _fp, _I64, _I, _I, _fp, _I, _I, _U64, _U64, _fp]),
    "ptrb200_ffnet_backward": (_I, [C.POINTER(FFNetDesc), C.POINTER(FFNetGrads), _fp, _fp, _fp, _fp, _I64,
                                    _I, _I, _fp, _I, _I, _U64, _U64, _fp]),
}

MAX_PEERS = 16


class PeerGroup(C.Structure):
    """struct ptrb200_peer_group"""
    _fields_ = [("world", C.c_int), ("rank", C.c_int), ("grads", _fp * MAX_PEERS), ("flags", _fp * MAX_PEERS),
                ("epoch", C.c_uint32), ("error", _fp)]


_D = C.c_double
_PG = C.POINTER(PeerGroup)
SIGNATURES.update({
    "ptrb200_peer_alloc": (_I, [_I64, C.POINTER(C.c_void_p), C.c_char_p]),
    "ptrb200_peer_open": (_I, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "ptrb200_peer_close": (_I, [_fp]),
    "ptrb200_peer_free": (_I, [_fp]),
    "ptrb200_peer_allreduce_sum": (_I, [_PG, _fp, _I64, _fp]),
    "ptrb200_adam_step_peer": (_I, [_PG, _fp, _fp, _fp, _I64, _D, _D, _D, _D, _D, _I, _fp]),
    "ptrb200_adagrad_step_peer": (_I, [_PG, _fp, _fp, _I64, _D, _D, _D, _D, _I, _fp]),
    "ptrb200_rmsprop_step_peer": (_I, [_PG, _fp, _fp, _I64, _D, _D, _D, _D, _fp]),
})


def peer_alloc(nbytes: int):
    """-> (device pointer, 64-byte CUDA IPC handle) of a zeroed allocation on the current device."""
    ptr, handle = C.c_void_p(), C.create_string_buffer(64)
    check(load().ptrb200_peer_alloc(int(nbytes), C.byref(ptr), handle), "peer_alloc")
    return int(ptr.value), handle.raw


def peer_open(handle: bytes) -> int:
    ptr = C.c_void_p()
    check(load().ptrb200_peer_open(C.create_string_buffer(bytes(handle), 64), C.byref(ptr)), "peer_open")
    return int(ptr.value)


HOOK_ALLREDUCE_F64, HOOK_LAYER_GRADS_READY = 1, 2
# int hook(int what, int layer, void* ptr, int64_t count, void* stream, void* user)
HOOK_T = C.CFUNCTYPE(C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p)
SIGNATURES["ptrb200_set_hook"] = (_I, [HOOK_T, C.c_void_p])

_lib = None
_hook_keepalive = None


def set_hook(pyfunc):
    """Install ``pyfunc(what, layer, ptr, count, stream) -> int`` as the library's host hook (None removes it)."""
    global _hook_keepalive
    lib = load()
    if pyfunc is None:
        _hook_keepalive = None
        check(lib.ptrb200_set_hook(C.cast(None, HOOK_T), None), "set_hook")
        return
    cb = HOOK_T(lambda what, layer, ptr, count, stream, user: int(pyfunc(what, layer, ptr or 0, count, stream or 0)))
    _hook_keepalive = cb          # ctypes callbacks must outlive their registration
    check(lib.ptrb200_set_hook(cb, None), "set_hook")


class B200LibraryError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the shared library once and attach the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m ptranking_b200.build` "
            "(nvcc, sm_100a).  ptranking_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().ptrb200_last_error()
        raise B200LibraryError(f"{what} failed with code {rc}: {msg.decode() if msg else ''}")


def launch_count() -> int:
    return int(load().ptrb200_launch_count())


def kernel_timings(enable=None):
    """enable=True/False switches per-launch event timing; enable=None drains the record ->
    {kernel name: (launches, total_ms)}."""
    lib = load()
    if enable is not None:
        check(lib.ptrb200_timing_enable(int(bool(enable))), "timing_enable")
        return None
    buf = C.create_string_buffer(1 << 16)
    check(lib.ptrb200_timing_report(buf, len(buf)), "timing_report")
    out = {}
    for line in buf.value.decode().splitlines():
        name, cnt, ms = line.split("\t")
        out[name] = (int(cnt), float(ms))
    return out
