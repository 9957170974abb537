"""ctypes binding of libfpa_b200.so (C ABI declared in include/fpa_b200.h).

The library is built in-tree by `__graft_entry__.build()` (nvcc, sm_100a).  There is no
CPU implementation behind these calls: when the shared object is missing, or no CUDA
device is visible, every compute call raises.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import os
from pathlib import Path

import numpy as np

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "libfpa_b200.so"

# status codes / flags (include/fpa_b200.h)
OK, ERR_INVALID, ERR_CUDA, ERR_NO_DEVICE, ERR_UNSUPPORTED = 0, 1, 2, 3, 4
OUT_TRACE, OUT_END, OUT_PMAX, CHECK_NAN, PHASE_EXACT, UNIFORM_PHYSICS, NWAVE_TABLE, NWAVE_COMB = 1, 2, 4, 8, 16, 32, 64, 128
NWAVE_PLAIN = 256
POINT_OK = -1
PM_GENERAL_TAYLOR, PM_SYMMETRIC_EVEN, PM_PROVIDED = 0, 1, 2
MAX_TAYLOR_ORDER = 12

c_dp = C.POINTER(C.c_double)


class Yaman4Desc(C.Structure):
    _fields_ = [
        ("n_points", C.c_int64),
        ("dbeta", C.c_void_p),
        ("gamma", C.c_void_p), ("gamma_stride", C.c_int64),
        ("alpha", C.c_void_p), ("alpha_stride", C.c_int64),
        ("A0", C.c_void_p), ("A0_stride", C.c_int64),
        ("z0", C.c_double), ("z_max", C.c_double),
        ("n_steps", C.c_int64), ("save_every", C.c_int64),
        ("z_grid", C.c_void_p),
        ("flags", C.c_uint32), ("reserved", C.c_uint32),
        ("A_trace", C.c_void_p), ("A_end", C.c_void_p), ("Pmax", C.c_void_p),
        ("status", C.c_void_p),
        ("gamma_uniform", C.c_double), ("alpha_uniform", C.c_double),
        ("scratch", C.c_void_p), ("scratch_bytes", C.c_int64),
    ]


class PlanDesc(C.Structure):
    _fields_ = [
        ("n1", C.c_int64), ("n3", C.c_int64),
        ("lambda1", C.c_void_p), ("lambda2", C.c_void_p), ("lambda2_stride", C.c_int64),
        ("lambda3", C.c_void_p),
        ("method", C.c_int32), ("max_order", C.c_int32), ("n_even", C.c_int32),
        ("even_orders", C.c_int32 * MAX_TAYLOR_ORDER),
        ("beta", C.c_double * (MAX_TAYLOR_ORDER + 1)),
        ("omega_ref", C.c_double), ("atol", C.c_double), ("rtol", C.c_double),
        ("provided", C.c_double),
        ("omega", C.c_void_p), ("dbeta", C.c_void_p), ("valid", C.c_void_p),
    ]


class SweepDesc(C.Structure):
    _fields_ = [
        ("plan", PlanDesc),
        ("A0", C.c_double * 8),
        ("p_signal", C.c_double),
        ("gamma", C.c_double), ("alpha", C.c_double),
        ("z_max", C.c_double), ("dz", C.c_double),
        ("length_scale", C.c_double),
        ("save_every", C.c_int64),
        ("flags", C.c_uint32), ("reserved", C.c_uint32),
        ("gain_lin", C.c_void_p), ("Pmax", C.c_void_p), ("A_end", C.c_void_p),
        ("status", C.c_void_p),
        ("first_point", C.c_int64), ("n_sub_points", C.c_int64),
        ("n_peers", C.c_int32), ("reserved3", C.c_int32), ("peer_gain", C.c_void_p * 8),
    ]


GAIN_MAX_SAVED, GAIN_LAST_SAVED = 0, 1
MAX_PHASES = 65536


class PhaseSweepDesc(C.Structure):
    _fields_ = [
        ("sweep", SweepDesc),
        ("n_phases", C.c_int64),
        ("A0_table", C.c_void_p),
        ("metric", C.c_int32), ("reserved", C.c_int32),
        ("gain_max", C.c_void_p), ("gain_min", C.c_void_p),
        ("idx_max", C.c_void_p), ("idx_min", C.c_void_p), ("n_finite", C.c_void_p),
    ]


class TransferOut(C.Structure):
    _fields_ = [("columns", C.c_uint32), ("reserved", C.c_uint32), ("jac", C.c_void_p)]


class Triplet(C.Structure):
    _fields_ = [("k", C.c_int16), ("l", C.c_int16), ("m", C.c_int16), ("weight", C.c_int16)]


TRIPLET_DTYPE = np.dtype([("k", "<i2"), ("l", "<i2"), ("m", "<i2"), ("weight", "<i2")])


class NwaveDesc(C.Structure):
    _fields_ = [
        ("n_points", C.c_int64),
        ("n_waves", C.c_int32), ("reserved0", C.c_int32),
        ("beta", C.c_void_p), ("beta_stride", C.c_int64),
        ("gamma", C.c_void_p), ("gamma_stride", C.c_int64),
        ("alpha", C.c_void_p), ("alpha_stride", C.c_int64),
        ("A0", C.c_void_p), ("A0_stride", C.c_int64),
        ("triplets", C.c_void_p), ("row_ptr", C.c_void_p), ("n_triplets", C.c_int64),
        ("z0", C.c_double), ("z_max", C.c_double),
        ("n_steps", C.c_int64), ("save_every", C.c_int64),
        ("flags", C.c_uint32), ("reserved1", C.c_uint32),
        ("A_trace", C.c_void_p), ("A_end", C.c_void_p), ("Pmax", C.c_void_p),
        ("status", C.c_void_p),
        ("grid_slot", C.c_void_p), ("grid_span", C.c_int32), ("n_classes", C.c_int32),
        ("factored", C.c_void_p),
    ]


# name -> (restype, argtypes); this table is also what tests check against the header
SIGNATURES = {
    "fpa_last_error": (C.c_char_p, []),
    "fpa_version": (C.c_char_p, []),
    "fpa_device_count": (C.c_int, []),
    "fpa_device_info": (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_char_p, C.c_int]),
    "fpa_set_device": (C.c_int, [C.c_int]),
    "fpa_n_saved": (C.c_int64, [C.c_int64, C.c_int64]),
    "fpa_interval_steps": (C.c_int64, [C.c_double, C.c_double]),
    "fpa_yaman4_rk4_batch_dev": (C.c_int, [C.POINTER(Yaman4Desc), C.c_void_p]),
    "fpa_yaman4_rk4_batch_host": (C.c_int, [C.POINTER(Yaman4Desc), C.c_int]),
    "fpa_yaman4_rk4_batch_multi_host": (C.c_int, [C.POINTER(Yaman4Desc), C.c_int, C.POINTER(C.c_int)]),
    "fpa_yaman4_scratch_bytes": (C.c_int64, [C.c_int64]),
    "fpa_yaman4_rhs_host": (C.c_int, [C.c_int64] + [C.c_void_p] * 6 + [C.c_int]),
    "fpa_dbeta_table_dev": (C.c_int, [C.POINTER(PlanDesc), C.c_void_p]),
    "fpa_dbeta_table_host": (C.c_int, [C.POINTER(PlanDesc), C.c_int]),
    "fpa_yaman4_sweep_host": (C.c_int, [C.POINTER(SweepDesc), C.c_int]),
    "fpa_yaman4_sweep_multi_host": (C.c_int, [C.POINTER(SweepDesc), C.c_int, C.POINTER(C.c_int)]),
    "fpa_yaman4_sweep_scratch_bytes": (C.c_int64, [C.c_int64]),
    "fpa_yaman4_sweep_dev": (C.c_int, [C.POINTER(SweepDesc), C.c_void_p, C.c_int64, C.c_void_p]),
    "fpa_yaman4_phase_sweep_host": (C.c_int, [C.POINTER(PhaseSweepDesc), C.c_int]),
    "fpa_yaman4_phase_sweep_multi_host": (C.c_int, [C.POINTER(PhaseSweepDesc), C.c_int, C.POINTER(C.c_int)]),
    "fpa_yaman4_phase_sweep_scratch_bytes": (C.c_int64, [C.c_int64]),
    "fpa_yaman4_phase_sweep_dev": (C.c_int, [C.POINTER(PhaseSweepDesc), C.c_void_p, C.c_int64, C.c_void_p]),
    "fpa_yaman4_transfer_batch_dev": (C.c_int, [C.POINTER(Yaman4Desc), C.POINTER(TransferOut), C.c_void_p]),
    "fpa_yaman4_transfer_batch_host": (C.c_int, [C.POINTER(Yaman4Desc), C.POINTER(TransferOut), C.c_int]),
    "fpa_yaman4_transfer_batch_multi_host": (C.c_int, [C.POINTER(Yaman4Desc), C.POINTER(TransferOut), C.c_int,
                                                       C.POINTER(C.c_int)]),
    "fpa_yaman4_transfer_sweep_dev": (C.c_int, [C.POINTER(SweepDesc), C.POINTER(TransferOut), C.c_void_p]),
    "fpa_yaman4_transfer_sweep_host": (C.c_int, [C.POINTER(SweepDesc), C.POINTER(TransferOut), C.c_int]),
    "fpa_yaman4_transfer_sweep_multi_host": (C.c_int, [C.POINTER(SweepDesc), C.POINTER(TransferOut), C.c_int,
                                                       C.POINTER(C.c_int)]),
    "fpa_linear_rk4_batch_host": (C.c_int, [C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_double,
                                            C.c_double, C.c_int64, C.c_int64, C.c_void_p, C.c_uint32,
                                            C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "fpa_enumerate_triplets": (C.c_int64, [C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "fpa_nwave_factor_table": (C.c_int64, [C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]),
    "fpa_enumerate_triplets_omega": (C.c_int64, [C.c_int32, C.c_void_p, C.c_double, C.c_double, C.c_void_p, C.c_int64,
                                                 C.c_void_p]),
    "fpa_nwave_rk4_batch_multi_host": (C.c_int, [C.POINTER(NwaveDesc), C.c_int, C.POINTER(C.c_int)]),
    "fpa_nwave_rk4_batch_dev": (C.c_int, [C.POINTER(NwaveDesc), C.c_void_p]),
    "fpa_nwave_rk4_batch_host": (C.c_int, [C.POINTER(NwaveDesc), C.c_int]),
    "fpa_nwave_flops_per_step": (C.c_double, [C.c_int32, C.c_int64, C.c_int64]),
    "fpa_nwave_factored_flops_per_step": (C.c_double, [C.c_void_p]),
    "fpa_nwave_comb_flops_per_step": (C.c_double, [C.c_int32, C.c_int32]),
    "fpa_fp64_peak_probe": (C.c_int, [C.c_int, C.c_int, c_dp, c_dp]),
    "fpa_yaman4_flops_per_step": (C.c_double, []),
    "fpa_host_alloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_int64]),
    "fpa_host_free": (C.c_int, [C.c_void_p]),
    "fpa_dev_alloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_int64, C.c_int]),
    "fpa_dev_free": (C.c_int, [C.c_void_p]),
    "fpa_ipc_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "fpa_ipc_open": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "fpa_ipc_close": (C.c_int, [C.c_void_p]),
    "fpa_host_register": (C.c_int, [C.c_void_p, C.c_int64]),
    "fpa_host_unregister": (C.c_int, [C.c_void_p]),
}

_lib = None


class FpaError(RuntimeError):
    """CUDA / device failure reported by libfpa_b200."""


def _load(path: Path):
    handle = C.CDLL(str(path))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(handle, name)
        fn.restype = res
        fn.argtypes = args
    return handle


def lib():
    """Load (once) and return the shared library; raises if it has not been built."""
    global _lib
    if _lib is None:
        path = Path(os.environ.get("FPA_B200_LIB", LIB_PATH))
        if not path.exists():
            raise ImportError(
                f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  This package has no CPU fallback."
            )
        _lib = _load(path)
    return _lib


@contextlib.contextmanager
def use_library(path):
    """Route every call of this package through another build of the same C ABI for the duration
    of the block (tests: the library with ptxas' own instruction schedule, build/libfpa_b200_ref.so,
    must give bit-identical results)."""
    global _lib
    saved = lib()
    _lib = _load(Path(path))
    try:
        yield _lib
    finally:
        _lib = saved


def last_error() -> str:
    return lib().fpa_last_error().decode("utf-8", "replace")


def check(rc: int) -> None:
    """Translate an FPA_* status into the exception the reference would raise."""
    if rc == OK:
        return
    msg = last_error()
    if rc == ERR_INVALID:
        raise ValueError(msg)
    if rc == ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    if rc == ERR_NO_DEVICE:
        raise FpaError(f"{msg} [no CUDA device; there is no CPU fallback]")
    raise FpaError(msg)


def device_count() -> int:
    return int(lib().fpa_device_count())


_default_device = 0


def set_device(device: int) -> None:
    """CUDA ordinal used by the host-pointer entry points of this process."""
    global _default_device
    _default_device = int(device)


def get_device() -> int:
    return _default_device


def ptr(a) -> int | None:
    """Address of a C-contiguous numpy array (None -> NULL)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data


def f64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float64)


def c128(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.complex128)


# Page-locked result pool.  cudaHostAlloc costs ~0.3 ms per MB, far more than a sweep launch, so blocks
# are recycled: when the array handed to the caller is garbage-collected its block goes back to the
# free list (up to _POOL_CAP bytes are kept; the rest is released with fpa_host_free).
_POOL_CAP = 1 << 30
_pool_free: dict[int, list[int]] = {}      # block size -> addresses
_pool_bytes = 0


def _pool_release(addr: int, size: int) -> None:
    global _pool_bytes
    if _lib is None:
        return
    if _pool_bytes + size <= _POOL_CAP:
        _pool_free.setdefault(size, []).append(addr)
        _pool_bytes += size
    else:
        _lib.fpa_host_free(C.c_void_p(addr))


def pinned_empty(shape, dtype) -> np.ndarray:
    """Page-locked host array (`fpa_host_alloc`) from the recycling pool.  Result buffers of this kind
    are written by the kernels directly, with no staging copy.  The block returns to the pool when
    the array (and every view of it) is garbage-collected."""
    import weakref

    global _pool_bytes
    shape = (int(shape),) if np.isscalar(shape) else tuple(int(v) for v in shape)
    count = int(np.prod(shape))
    nbytes = max(count * np.dtype(dtype).itemsize, 1)
    size = 1 << max(12, (nbytes - 1).bit_length())          # power-of-two size classes, >= one page
    free = _pool_free.get(size)
    if free:
        addr = free.pop()
        _pool_bytes -= size
    else:
        p = C.c_void_p()
        check(lib().fpa_host_alloc(C.byref(p), size))
        addr = p.value
    buf = (C.c_char * size).from_address(addr)
    weakref.finalize(buf, _pool_release, addr, size)         # buf lives as long as any view of it
    return np.frombuffer(buf, dtype=dtype, count=count).reshape(shape)


def register_host(arr: np.ndarray) -> None:
    """Page-lock memory the caller owns (`fpa_host_register`), e.g. a shared-memory segment that several
    ranks map: each rank's kernels then store their shard straight into the one host array."""
    check(lib().fpa_host_register(arr.ctypes.data, arr.nbytes))


def unregister_host(arr: np.ndarray) -> None:
    check(lib().fpa_host_unregister(arr.ctypes.data))
