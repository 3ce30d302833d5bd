"""ctypes binding of ``libtsgu_b200.so`` (the C ABI declared in ``include/tsgu_b200.h``).

There is deliberately no fallback: if the shared library is missing or a kernel launch fails the
caller gets an exception (the reference documents ``RuntimeError`` for kernel failures,
``torchsparsegradutils/sparse_matmul.py:62-63``).
"""
from __future__ import annotations

import ctypes
import os
import threading
from ctypes import c_char_p, c_int, c_int64, c_size_t, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TSGU_B200_LIB") or os.path.join(_HERE, "libtsgu_b200.so")  # env override: kernel-variant experiments only

# enums of include/tsgu_b200.h
F32, F64, BF16 = 0, 1, 2
I32, I64 = 0, 1
ALGO_AUTO, ALGO_ROWSPLIT, ALGO_MERGE = 0, 1, 2
ALGO_FLAG_KSLICE = 0x100  # OR-ed into algo for tsgu_spmm_csr: uniform rows, K may be cut into L2-resident slices

VAL_DTYPES = {torch.float32: F32, torch.float64: F64, torch.bfloat16: BF16}
IDX_DTYPES = {torch.int32: I32, torch.int64: I64}
IDX_TORCH = {I32: torch.int32, I64: torch.int64}

_P, _L, _I, _Z = c_void_p, c_int64, c_int, c_size_t
_SIGNATURES = {
    "tsgu_version": (c_int, []),
    "tsgu_error_string": (c_char_p, [_I]),
    "tsgu_launch_count": (_L, []),
    "tsgu_set_sm_margin": (_I, [_I]),
    "tsgu_mailbox_create": (_I, [_Z, ctypes.POINTER(_P), ctypes.POINTER(_P)]),
    "tsgu_mailbox_destroy": (_I, [_P]),
    "tsgu_publish": (_I, [_P, _P, _Z, _P]),
    "tsgu_fingerprint": (_I, [_P, _L, _I, _P, _P]),
    "tsgu_spmm_csr": (_I, [_P, _P, _P, _P, _P, _P, _L, _L, _L, _L, _L, _L, _L, _L, _L, _L, _L, _L, _I, _I, _I, _P, _Z, _P]),
    "tsgu_spmm_csr_rowmap": (_I, [_P, _P, _P, _P, _P, _P, _P, _L, _L, _L, _L, _L, _L, _L, _L, _L, _L, _L, _L, _I, _I, _I, _P]),
    "tsgu_spmm_workspace_bytes": (_Z, [_L, _L, _L, _L, _I, _I]),
    "tsgu_sddmm_csr": (_I, [_P, _P, _P, _P, _P, _P, _L, _L, _L, _L, _L, _L, _L, _L, _L, _L, _L, _L, _L, _I, _I, _I, _P, _Z, _P]),
    "tsgu_sddmm_workspace_bytes": (_Z, [_L, _L, _L, _I]),
    "tsgu_sddmm_coo": (_I, [_P, _P, _P, _P, _P, _L, _L, _L, _L, _L, _L, _I, _P]),
    "tsgu_coo_sort": (_I, [_P, _I, _L, _L, _P, _I, _P, _P, _I, _P, _Z, _P]),
    "tsgu_coo_sort_workspace_bytes": (_Z, [_I, _L, _I]),
    "tsgu_coo_to_csr": (_I, [_P, _I, _L, _L, _L, _L, _P, _P, _P, _I, _P]),
    "tsgu_compress_rows": (_I, [_P, _L, _L, _P, _I, _P, _Z, _P]),
    "tsgu_compress_rows_workspace_bytes": (_Z, [_L, _I]),
    "tsgu_decompress_crow": (_I, [_P, _L, _L, _P, _I, _P]),
    "tsgu_csr_transpose": (_I, [_P, _P, _L, _L, _L, _L, _L, _L, _I, _P, _P, _P, _I, _P, _Z, _P]),
    "tsgu_csr_transpose_workspace_bytes": (_Z, [_L, _L, _L, _I]),
    "tsgu_gather_values": (_I, [_P, _P, _P, _L, _I, _I, _P]),
    "tsgu_scatter_values": (_I, [_P, _P, _P, _L, _L, _I, _I, _P]),
    "tsgu_block_diag_csr": (_I, [_P, _P, _L, _L, _L, _L, _P, _P, _I, _P]),
    "tsgu_segment_sum_values": (_I, [_P, _P, _P, _P, _L, _I, _I, _P]),
    "tsgu_pack_dense": (_I, [_P, _P, _L, _L, _L, _L, _L, _L, _L, _L, _L, _I, _P]),
    "tsgu_pack_dense_add": (_I, [_P, _P, _P, _P, _L, _L, _L, _L, _L, _L, _L, _L, _L, _L, _L, _I, _P]),
    "tsgu_window_limits": (_I, [_P, _P, _P, _P]),
    "tsgu_window_plan": (_I, [_P, _P, _L, _L, _L, _L, _I, _I, _P, _P, _P, _P]),
    "tsgu_spmm_window": (_I, [_P, _P, _P, _P, _P, _P, _L, _L, _L, _L, _L, _L, _I, _L, _L, _L, _L, _L, _I, _I, _P]),
    "tsgu_sddmm_window": (_I, [_P, _P, _P, _P, _P, _P, _P, _L, _L, _L, _L, _L, _L, _I, _L, _L, _L, _L, _I, _I, _P]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None
_lock = threading.Lock()


class NativeLibraryError(RuntimeError):
    pass


def lib() -> ctypes.CDLL:
    """Load the shared library once; raise loudly if it has not been built."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise NativeLibraryError(
                        f"{LIB_PATH} not found: build it with `python -m torchsparsegradutils_b200.csrc.build` "
                        "(torchsparsegradutils_b200 has no CPU / PyTorch fallback)")
                handle = ctypes.CDLL(LIB_PATH)
                for name, (res, args) in _SIGNATURES.items():
                    fn = getattr(handle, name)  # AttributeError if the ABI and the binding drift apart
                    fn.restype, fn.argtypes = res, args
                _lib = handle
    return _lib


def check(code: int, what: str) -> None:
    if code != 0:
        msg = lib().tsgu_error_string(code)
        raise RuntimeError(f"{what} failed: {msg.decode() if msg else code} (code {code})")


class sm_margin:
    """``with sm_margin(16): ...`` -- persistent kernels launched inside leave that many SMs to concurrent kernels."""

    def __init__(self, sms: int):
        self.sms = int(sms)

    def __enter__(self):
        self.prev = lib().tsgu_set_sm_margin(self.sms)
        return self

    def __exit__(self, *exc):
        lib().tsgu_set_sm_margin(self.prev)
        return False


def launch_count() -> int:
    return int(lib().tsgu_launch_count())


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def stream_ptr(device: torch.device) -> int:
    """cudaStream_t of torch's current stream on `device` (the raw getter is ~30x cheaper than building a
    torch.cuda.Stream object: 11 us -> 0.3 us of host time per launch)."""
    if _raw_stream is not None and device.index is not None:
        return _raw_stream(device.index)
    return torch.cuda.current_stream(device).cuda_stream


_MAILBOX_WORDS = 64  # int64 slots per host read
_mailboxes = threading.local()


def host_read(t: torch.Tensor) -> list:
    """The values of a small integer CUDA tensor on the host: one publish kernel into this thread's mapped-memory
    mailbox plus a stream synchronise (``tsgu_publish``) -- not ``.tolist()``, whose cudaMemcpy would wait behind any
    bulk D2H traffic of the application."""
    if not t.is_cuda:  # host-side unit tests of the pattern logic
        return t.reshape(-1).long().tolist()
    if t.dtype != torch.int64:
        t = t.long()
    t = t.contiguous().reshape(-1)
    count = t.numel()
    if count == 0:
        return []
    if count > _MAILBOX_WORDS:
        raise ValueError(f"host_read carries at most {_MAILBOX_WORDS} values")
    box = getattr(_mailboxes, "box", None)
    if box is None:
        host, dev = _P(), _P()
        check(lib().tsgu_mailbox_create(_MAILBOX_WORDS * 8, ctypes.byref(host), ctypes.byref(dev)), "tsgu_mailbox_create")
        view = (c_int64 * _MAILBOX_WORDS).from_address(host.value)
        box = _mailboxes.box = (view, dev.value)  # lives as long as the thread (mapped memory is never recycled)
    view, dev = box
    with torch.cuda.device(t.device):
        check(lib().tsgu_publish(t.data_ptr(), dev, count * 8, stream_ptr(t.device)), "tsgu_publish")
        torch.cuda.current_stream(t.device).synchronize()
    return list(view[:count])


def ptr(t) -> int | None:
    return None if t is None else t.data_ptr()


def val_enum(dtype: torch.dtype) -> int:
    try:
        return VAL_DTYPES[dtype]
    except KeyError:
        raise RuntimeError(f"sparse_mm: unsupported value dtype {dtype}; supported: float32, float64, bfloat16") from None


def idx_enum(dtype: torch.dtype) -> int:
    try:
        return IDX_DTYPES[dtype]
    except KeyError:
        raise RuntimeError(f"sparse_mm: unsupported index dtype {dtype}") from None


def workspace(nbytes: int, device: torch.device) -> torch.Tensor:
    """Caller-owned scratch (torch caching allocator); the library never allocates."""
    return torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=device)
