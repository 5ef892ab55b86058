"""ctypes binding of the C ABI in include/pli_attention.h (libpli_attention.so).

There is no CPU fallback: if the library is missing or a call fails, the caller gets an exception.
The library is built in-tree by `physics_llm_inference_b200.build` / `__graft_entry__.build()`.
"""
from __future__ import annotations

import ctypes as C
import os
import re

_PKG = os.path.dirname(os.path.abspath(__file__))
# PLI_LIB_PATH: load another build of the same ABI (kernel tuning experiments); never a fallback
LIB_PATH = os.environ.get("PLI_LIB_PATH") or os.path.join(_PKG, "libpli_attention.so")
HEADER_PATH = os.path.join(os.path.dirname(_PKG), "include", "pli_attention.h")

PLI_BF16, PLI_F16, PLI_F32 = 0, 1, 2
PLI_KIND_NONE, PLI_KIND_TCGEN05, PLI_KIND_SIMT, PLI_KIND_MMA_TMA = 0, 1, 2, 3
KIND_NAMES = {0: "none", 1: "tcgen05", 2: "simt", 3: "mma_tma"}

_I64P = C.POINTER(C.c_int64)
_VP = C.c_void_p

PLI_MAX_PEERS = 8


class PeerScatter(C.Structure):
    """`pli_peer_scatter` of include/pli_attention.h."""
    _fields_ = [("n_peers", C.c_int32), ("rank", C.c_int32), ("peer_o", C.c_void_p * PLI_MAX_PEERS),
                ("peer_flags", C.c_void_p * PLI_MAX_PEERS), ("epoch", C.c_void_p),
                ("buffer_stride", C.c_int64), ("slice_offset", C.c_int64),
                ("peer_ready", C.c_void_p * PLI_MAX_PEERS), ("cta_counter", C.c_void_p)]


_SIGNATURES = {
    "pli_abi_version": (C.c_int, []),
    "pli_last_error": (C.c_char_p, []),
    "pli_set_device": (C.c_int, [C.c_int]),
    "pli_launch_count": (C.c_uint64, []),
    "pli_reset_launch_count": (None, []),
    "pli_prefill_fwd": (C.c_int, [_VP, _VP, _VP, _VP, _VP, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                  _I64P, _I64P, _I64P, _I64P, C.c_float, C.c_int, C.c_int, _VP]),
    "pli_prefill_paged_fwd": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, _VP, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                        C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64, _I64P, _I64P, _I64P, C.c_float,
                                        C.c_int, _VP]),
    "pli_prefill_varlen_paged_fwd": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, C.c_int, C.c_int, C.c_int, C.c_int64,
                                               C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64, _I64P,
                                               _I64P, _I64P, C.c_float, C.c_int, _VP]),
    "pli_prefill_kernel_kind": (C.c_int, [C.c_int, C.c_int, _I64P, _I64P, _I64P, _I64P, _VP, _VP, _VP, _VP]),
    "pli_decode_num_splits": (C.c_int, [C.c_int, C.c_int, C.c_int]),
    "pli_decode_num_splits_multi": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "pli_decode_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "pli_decode_splitkv": (C.c_int, [_VP, _VP, _VP, _VP, _VP, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.c_int, C.c_int, C.c_int64, _I64P, _I64P, C.c_float, C.c_int, C.c_int, _VP,
                                     C.c_size_t, _VP]),
    "pli_decode_combine": (C.c_int, [_VP, _VP, _VP, C.c_int, C.c_int, C.c_int, C.c_int, _I64P, C.c_int, _VP]),
    "pli_decode_fwd": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, _VP, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                 C.c_int, C.c_int, C.c_int, C.c_int64, _I64P, _I64P, _I64P, C.c_float, C.c_int,
                                 C.c_int, _VP, C.c_size_t, _VP]),
    "pli_decode_fwd_multi": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, _VP, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64, _I64P, _I64P, _I64P, C.c_float,
                                       C.c_int, C.c_int, _VP, C.c_size_t, _VP]),
    "pli_decode_kernel_kind": (C.c_int, [C.c_int, C.c_int, C.c_int, _I64P, _VP, _VP]),
    "pli_decode_fwd_scatter": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.c_int, C.c_int, C.c_int, C.c_int64, _I64P, _I64P, _I64P, C.c_float, C.c_int,
                                         C.c_int, _VP, C.c_size_t, C.POINTER(PeerScatter), _VP]),
    "pli_decode_fwd_gather": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                        C.c_int, C.c_int, C.c_int, C.c_int64, _I64P, _I64P, _I64P, C.c_float, C.c_int,
                                        C.c_int, _VP, C.c_size_t, C.POINTER(PeerScatter), _VP]),
    "pli_prefill_fwd_scatter": (C.c_int, [_VP, _VP, _VP, _VP, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                          _I64P, _I64P, _I64P, _I64P, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int,
                                          C.c_int, C.c_int, C.POINTER(PeerScatter), _VP]),
    "pli_peer_publish_wait": (C.c_int, [C.POINTER(PeerScatter), _VP]),
    "pli_peer_select_copy": (C.c_int, [C.POINTER(PeerScatter), _VP, C.c_int64, C.c_int, _VP]),
    "pli_set_peer_timeout_ms": (C.c_int, [C.c_int64]),
    "pli_device_status": (C.c_int, [C.POINTER(C.c_uint64), C.c_int]),
    "pli_kv_append": (C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                C.c_int, _I64P, _I64P, C.c_int, _VP]),
    "pli_paged_gather": (C.c_int, [_VP, _VP, _VP, _VP, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                   _I64P, C.c_int, _VP]),
    "pli_online_softmax": (C.c_int, [_VP, _VP, C.c_int64, C.c_int, C.c_int64, C.c_int64, C.c_int, _VP]),
    "pli_online_softmax_with_output": (C.c_int, [_VP, _VP, _VP, _VP, C.c_int64, C.c_int, C.c_int, C.c_int64, C.c_int64,
                                                 C.c_int64, C.c_int64, C.c_int, _VP]),
    # debug aid, not declared in the public header
    "pli_debug_umma_selftest": (C.c_int, [_VP, _VP, _VP, _VP, _VP, C.c_int, C.c_int, _VP]),
    "pli_debug_prefill_trace": (C.c_int, [_VP, C.c_int, C.c_int]),
    "pli_debug_decode_trace": (C.c_int, [_VP, C.c_int]),
}

_lib = None


class PliError(RuntimeError):
    """A C-ABI call returned a non-zero code."""


def header_symbols() -> list[str]:
    """Every function name declared in include/pli_attention.h."""
    with open(HEADER_PATH) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    return sorted(set(re.findall(r"\b(pli_[a-z0-9_]+)\s*\(", text)))


def load() -> C.CDLL:
    """Load libpli_attention.so (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PliError(
            f"{LIB_PATH} is missing: build it with `python -m physics_llm_inference_b200.build` "
            "(there is no CPU fallback for the attention path)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.pli_abi_version() != 1:
        raise PliError(f"ABI version mismatch: library reports {lib.pli_abi_version()}, binding expects 1")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().pli_last_error().decode("utf-8", "replace")
        if rc == -1:
            raise ValueError(f"pli: {msg}")
        raise PliError(f"pli error {rc}: {msg}")


FAULT_NAMES = {0: "none", 1: "mbarrier wait timed out inside a kernel (protocol bug; the kernel trapped)",
               2: "a peer rank's output slice did not arrive within the peer timeout"}


def device_status(clear: bool = False) -> dict:
    """The library's host-visible fault record (include/pli_attention.h: pli_device_status)."""
    buf = (C.c_uint64 * 8)()
    check(load().pli_device_status(buf, int(clear)))
    code = int(buf[0])
    rec = {"code": code, "what": FAULT_NAMES.get(code, "unknown"), "timer_ns": int(buf[3])}
    if code == 1:
        rec.update(block=int(buf[1]) >> 32, thread=int(buf[1]) & 0xFFFFFFFF, barrier_smem_addr=int(buf[2]) & 0xFFFFFFFF,
                   parity=int(buf[2]) >> 32)
    elif code == 2:
        rec.update(waiting_rank=int(buf[1]) >> 32, missing_rank=int(buf[1]) & 0xFFFFFFFF, step=int(buf[2]))
    return rec


def raise_on_device_fault() -> None:
    rec = device_status()
    if rec["code"] != 0:
        device_status(clear=True)
        raise PliError(f"device fault recorded: {rec}")


def set_peer_timeout_ms(ms: int) -> None:
    check(load().pli_set_peer_timeout_ms(int(ms)))


def i64(*vals) -> C.Array:
    return (C.c_int64 * len(vals))(*[int(v) for v in vals])


def dtype_code(dtype) -> int:
    import torch
    if dtype == torch.bfloat16:
        return PLI_BF16
    if dtype == torch.float16:
        return PLI_F16
    if dtype == torch.float32:
        return PLI_F32
    raise TypeError(f"unsupported dtype {dtype}: the attention path takes bfloat16, float16 or float32")


def current_stream_ptr(device) -> int:
    import torch
    return torch.cuda.current_stream(device).cuda_stream


_device_set = -1


class on_device:
    """`with on_device(t.device):` — make the tensor's device current for torch AND for the library's own CUDA
    runtime.  When it already is (the common case) this costs one integer compare instead of a
    torch.cuda.device() guard plus a cudaSetDevice per call (the wrappers were ~28 us of host time per call)."""
    __slots__ = ("idx", "guard")

    def __init__(self, device):
        self.idx = device.index if device.index is not None else 0
        self.guard = None

    def __enter__(self):
        global _device_set
        import torch
        if torch.cuda.current_device() != self.idx:
            self.guard = torch.cuda.device(self.idx)
            self.guard.__enter__()
            check(load().pli_set_device(self.idx))
            _device_set = -1                       # our runtime's current device must be re-asserted afterwards
        elif _device_set != self.idx:
            check(load().pli_set_device(self.idx))
            _device_set = self.idx
        return self

    def __exit__(self, *exc):
        if self.guard is not None:
            self.guard.__exit__(*exc)
            self.guard = None
        return False


def launch_count() -> int:
    return int(load().pli_launch_count())


def reset_launch_count() -> None:
    load().pli_reset_launch_count()
