"""ctypes binding of libb200lops.so (the C ABI declared in include/b200lops.h).

The product path has NO fallback: if the shared library is missing or cannot be
loaded, importing this module raises, and every compute entry point of the
package goes through it.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import torch  # noqa: F401  (loads the NCCL / CUDA runtime libraries libb200lops links against)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200lops.so")

# dtype codes (include/b200lops.h)
F32, F64, C64, C128, BF16, I64 = 0, 1, 2, 3, 4, 5
SUM, MAX, MIN = 0, 1, 2
NRM_COUNT_NONZERO, NRM_SUM_ABS, NRM_SUM_SQ, NRM_MAX_ABS, NRM_MIN_ABS, NRM_SUM_POW = range(6)
FD_FORWARD, FD_BACKWARD, FD_CENTERED = 0, 1, 2
OP_N, OP_T, OP_H = 0, 1, 2
THRESH_NONE, THRESH_SOFT, THRESH_HARD, THRESH_HALF = 0, 1, 2, 3

_TORCH2CODE = {torch.float32: F32, torch.float64: F64, torch.complex64: C64,
               torch.complex128: C128, torch.bfloat16: BF16, torch.int64: I64}
_NP2TORCH = {np.dtype(np.float32): torch.float32, np.dtype(np.float64): torch.float64,
             np.dtype(np.complex64): torch.complex64, np.dtype(np.complex128): torch.complex128,
             np.dtype(np.int64): torch.int64, np.dtype(np.int32): torch.int32}
_TORCH2NP = {v: k for k, v in _NP2TORCH.items()}


def torch_dtype(dtype) -> torch.dtype:
    """numpy-or-torch dtype spec -> torch.dtype"""
    if isinstance(dtype, torch.dtype):
        return dtype
    if isinstance(dtype, str) and dtype in ("bfloat16", "bf16"):
        return torch.bfloat16
    return _NP2TORCH[np.dtype(dtype)]


def numpy_dtype(dtype):
    """torch-or-numpy dtype spec -> numpy dtype (bfloat16 has none: returned as torch.bfloat16)"""
    if isinstance(dtype, torch.dtype):
        return _TORCH2NP.get(dtype, dtype)
    if isinstance(dtype, str) and dtype in ("bfloat16", "bf16"):
        return torch.bfloat16
    return np.dtype(dtype)


def code(t: torch.dtype) -> int:
    try:
        return _TORCH2CODE[t]
    except KeyError:
        raise TypeError(f"dtype {t} is not supported by libb200lops") from None


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: the CUDA extension is mandatory (no CPU fallback). "
            "Build it with `python -m pylops_mpi_b200.build` (needs nvcc, sm_100a).")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    vp, sz, i, d, dp = C.c_void_p, C.c_size_t, C.c_int, C.c_double, C.POINTER(C.c_double)
    sigs = {
        "b2_version": ([], i),
        "b2_strerror": ([i], C.c_char_p),
        "b2_ctx_create": ([i, C.POINTER(vp)], i),
        "b2_ctx_destroy": ([vp], i),
        "b2_ctx_sm_count": ([vp, C.POINTER(i)], i),
        "b2_lincomb": ([vp, vp, dp, vp, dp, vp, sz, i, i, vp], i),
        "b2_lincomb_dev": ([vp, vp, vp, d, vp, vp, d, vp, sz, i, vp], i),
        "b2_lincomb_dev_norm2": ([vp, vp, vp, d, vp, vp, d, vp, sz, i, vp, vp], i),
        "b2_mul": ([vp, vp, vp, vp, sz, i, i, vp], i),
        "b2_fill": ([vp, vp, dp, sz, i, vp], i),
        "b2_dot": ([vp, vp, vp, sz, i, i, vp, vp], i),
        "b2_norm_partial": ([vp, vp, sz, i, i, d, vp, vp], i),
        "b2_norm_axis": ([vp, vp, sz, sz, sz, i, i, d, vp, vp], i),
        "b2_dot_multi": ([vp, i, C.POINTER(vp), C.POINTER(vp), sz, i, i, vp, vp], i),
        "b2_scalar_div": ([vp, vp, vp, vp, d, vp], i),
        "b2_history_push": ([vp, i, i, vp, vp, sz, vp, vp, vp], i),
        "b2_sparse_update": ([vp, vp, vp, d, vp, d, i, vp, vp, d, vp, sz, i, vp], i),
        "b2_first_derivative": ([vp, vp, vp, vp, i, vp, i, sz, sz, sz, sz, i, i, i, d, i, i, vp], i),
        "b2_first_derivative_halo": ([i, i, i, C.POINTER(i), C.POINTER(i)], i),
        "b2_second_derivative": ([vp, vp, vp, vp, i, vp, i, sz, sz, sz, sz, i, i, d, i, i, vp], i),
        "b2_second_derivative_halo": ([i, i, i, C.POINTER(i), C.POINTER(i)], i),
        "b2_derivative_axis": ([vp, vp, vp, sz, sz, sz, i, i, i, i, d, i, i, vp], i),
        "b2_convolve1d": ([vp, vp, vp, sz, sz, sz, vp, i, C.c_longlong, i, i, vp], i),
        "b2_halo_bytes": ([sz], sz),
        "b2_halo_create": ([i, i, C.POINTER(vp), sz, C.POINTER(vp)], i),
        "b2_halo_destroy": ([vp], i),
        "b2_derivative_peer": ([vp, vp, vp, vp, sz, sz, sz, sz, i, i, i, i, d, i, i, vp], i),
        "b2_first_derivative_host": ([vp, vp, vp, sz, sz, sz, sz, i, i, i, d, i, i], i),
        "b2_gemv": ([vp, vp, sz, sz, sz, vp, vp, i, i, i, vp], i),
        "b2_gemm_bf16": ([vp, vp, sz, vp, sz, vp, sz, sz, sz, sz, i, i, vp], i),
        "b2_gemm": ([vp, vp, sz, vp, sz, vp, sz, sz, sz, sz, i, i, i, vp], i),
        "b2_cast_bf16_multi": ([vp, vp, sz, sz, sz, C.POINTER(vp), i, sz, vp], i),
        "b2_gemm_bf16_seg": ([vp, vp, sz, vp, sz, C.POINTER(vp), i, sz, sz, sz, sz, sz, i, vp], i),
        "b2_sum_slots": ([vp, vp, sz, i, sz, vp, sz, sz, vp], i),
        "b2_batched_gemm": ([vp, vp, vp, vp, sz, sz, sz, sz, i, i, vp], i),
        "b2_batched_gemm_allgather": ([vp, vp, vp, vp, C.POINTER(vp), i, sz, sz, sz, sz, i, i, vp], i),
        "b2_fredholm_plan_create": ([vp, vp, sz, sz, sz, sz, i, C.POINTER(vp)], i),
        "b2_fredholm_plan_destroy": ([vp], i),
        "b2_fredholm_apply": ([vp, vp, vp, C.POINTER(vp), i, i, vp], i),
        "b2_fredholm_apply_parts": ([vp, vp, vp, i, i, vp], i),
        "b2_symm_alloc": ([sz, C.POINTER(vp)], i),
        "b2_symm_free": ([vp], i),
        "b2_ipc_get_handle": ([vp, vp], i),
        "b2_ipc_open_handle": ([vp, C.POINTER(vp)], i),
        "b2_ipc_close_handle": ([vp], i),
        "b2_peer_slots_bytes": ([], sz),
        "b2_peer_create": ([i, i, C.POINTER(vp), C.POINTER(vp)], i),
        "b2_peer_destroy": ([vp], i),
        "b2_peer_allreduce": ([vp, vp, i, i, vp], i),
        "b2_peer_vec_bytes": ([], sz),
        "b2_peer_vec_max_bytes": ([], sz),
        "b2_peer_vec_create": ([i, i, C.POINTER(vp), C.POINTER(vp)], i),
        "b2_peer_vec_destroy": ([vp], i),
        "b2_peer_vec_allreduce": ([vp, vp, sz, i, vp], i),
        "b2_peer_vec_allgatherv": ([vp, vp, vp, C.POINTER(sz), i, vp], i),
        "b2_get_unique_id": ([vp], i),
        "b2_comm_create": ([i, i, vp, i, C.POINTER(vp)], i),
        "b2_comm_split": ([vp, i, i, C.POINTER(vp)], i),
        "b2_comm_destroy": ([vp], i),
        "b2_comm_rank": ([vp, C.POINTER(i), C.POINTER(i)], i),
        "b2_allreduce": ([vp, vp, vp, sz, i, i, vp], i),
        "b2_allgather": ([vp, vp, vp, sz, i, vp], i),
        "b2_allgatherv": ([vp, vp, vp, C.POINTER(sz), i, vp], i),
        "b2_allgatherv_at": ([vp, vp, vp, C.POINTER(sz), C.POINTER(sz), i, vp], i),
        "b2_bcast": ([vp, vp, sz, i, i, vp], i),
        "b2_send": ([vp, vp, sz, i, i, vp], i),
        "b2_recv": ([vp, vp, sz, i, i, vp], i),
        "b2_group_start": ([], i),
        "b2_group_end": ([], i),
    }
    for name, (args, res) in sigs.items():
        fn = getattr(lib, name)  # AttributeError if the ABI and the header disagree
        fn.argtypes = args
        fn.restype = res
    return lib, tuple(sigs)


lib, EXPORTS = _load()


class B200Error(RuntimeError):
    pass


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib.b2_strerror(rc).decode()
        raise B200Error(f"libb200lops {what} failed: [{rc}] {msg}")


def ptr(t) -> int:
    """raw device (or host) pointer of a torch tensor / None"""
    if t is None:
        return None
    return t.data_ptr()


_RAW_STREAM = getattr(torch._C, "_cuda_getCurrentRawStream", None)
_GET_DEVICE = getattr(torch._C, "_cuda_getDevice", None)


def stream() -> int:
    """raw ``cudaStream_t`` of torch's current stream on the current device (hot enqueue path: the private C
    accessors avoid building a ``torch.cuda.Stream`` object, ~6 us per launch)"""
    if _RAW_STREAM is not None and _GET_DEVICE is not None:
        return _RAW_STREAM(_GET_DEVICE())
    return torch.cuda.current_stream().cuda_stream


def cpair(z):
    z = complex(z)
    return (C.c_double * 2)(z.real, z.imag)


_CTX = {}
_CUDA_OK = False


def ctx(device=None):
    """per-device b2_ctx handle (created on first use; needs a CUDA device)"""
    global _CUDA_OK
    if not _CUDA_OK:            # checked until it succeeds once (the check costs microseconds on a hot enqueue path)
        if not torch.cuda.is_available():
            raise B200Error("pylops_mpi_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        _CUDA_OK = True
    dev = torch.cuda.current_device() if device is None else int(device)
    h = _CTX.get(dev)
    if h is None:
        out = C.c_void_p()
        check(lib.b2_ctx_create(dev, C.byref(out)), "b2_ctx_create")
        h = _CTX[dev] = out
    return h
