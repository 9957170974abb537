"""numpy-facing wrappers over the host-pointer entry points of libfpa_b200 (one call = H2D,
one kernel launch, D2H).  Nothing here computes: arrays are shaped, the C-ABI is called and
FPA_* codes become exceptions (`_lib.check`).  The reference-named modules of this package
(integrators, yaman_model, simulation, scan_mismtach, nwave) are built on these.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _lib
from ._lib import c128, f64, ptr


def n_saved(n_steps: int, save_every: int) -> int:
    return int(n_steps) // int(save_every) + 1


def interval_steps(z_max: float, dz: float) -> int:
    """int(round(z_max/dz)) exactly as integrators.py:194 (round-half-even)."""
    return int(round(float(z_max) / float(dz)))


def _flags(trace, end, pmax, check_nan, phase_exact) -> int:
    return ((_lib.OUT_TRACE if trace else 0) | (_lib.OUT_END if end else 0) |
            (_lib.OUT_PMAX if pmax else 0) | (_lib.CHECK_NAN if check_nan else 0) |
            (_lib.PHASE_EXACT if phase_exact else 0))


def _per_point(a, B: int, width: int, name: str, conv=f64):
    """(array, stride): `a` is scalar / shape (width,) -> broadcast, or [B(,width)] -> per point."""
    arr = conv(a)
    flat = arr.reshape(-1)
    if flat.size == width:
        return flat, 0
    if flat.size == B * width:
        return flat, 1
    raise ValueError(f"{name} must broadcast to {B} points x {width}, got shape {arr.shape}")


def result_array(shape, dtype, pinned: bool = True) -> np.ndarray:
    """Result buffer handed back to the caller.  By default it comes from the library's page-locked
    pool (`_lib.pinned_empty`): the kernels store into it directly, so the reference-named calls
    (which never pass `out=`) get the same zero-copy delivery as a caller with its own pinned
    buffers.  Falls back to pageable memory when page-locking fails (e.g. the locked-memory limit)."""
    if pinned and int(np.prod(shape)) > 0:
        try:
            return _lib.pinned_empty(shape, dtype)
        except _lib.FpaError:
            pass
    return np.empty(shape, dtype=dtype)


def _run_host(host, multi_host, desc, device, devices) -> None:
    """`multi_host` over `devices` when they are several, else `host` on `device` (or the one entry of
    `devices`, or the process default)."""
    if devices is not None and len(devices) > 1:
        ids = (C.c_int * len(devices))(*[int(v) for v in devices])
        _lib.check(multi_host(C.byref(desc), len(devices), ids))
        return
    dev = _lib.get_device() if device is None else int(device)
    if devices is not None and len(devices) == 1:
        dev = int(devices[0])
    _lib.check(host(C.byref(desc), dev))


def yaman4_batch(dbeta, gamma, alpha, A0, *, z0=0.0, z_max, n_steps, save_every=1, z_grid=None,
                 trace=False, end=True, pmax=False, check_nan=True, phase_exact=False,
                 device: Optional[int] = None, devices=None) -> dict:
    """B scan points through `fpa_yaman4_rk4_batch_host` (`devices=[...]`: split over several GPUs
    of the box by `fpa_yaman4_rk4_batch_multi_host`, bit-identical).  Returns a dict with the requested
    outputs: A_trace [B,n_saved,4] c128, A_end [B,4] c128, Pmax [B,4] f64, status [B] i32."""
    dbeta = f64(dbeta).reshape(-1)
    B = dbeta.size
    gam, gs = _per_point(gamma, B, 1, "gamma")
    alp, as_ = _per_point(alpha, B, 1, "alpha")
    a0, a0s = _per_point(A0, B, 4, "A0", c128)
    n_steps, save_every = int(n_steps), int(save_every)
    if n_steps < 1:
        raise ValueError("n_steps must be >= 1")
    if save_every <= 0:
        raise ValueError("save_every must be a positive integer")
    ns = n_saved(n_steps, save_every)
    grid = None
    if z_grid is not None:
        grid = f64(z_grid).reshape(-1)
        if grid.size != n_steps + 1:
            raise ValueError("z_grid must hold n_steps+1 values")
    big = B >= 4096            # single runs and small batches: not worth page-locking
    out = {"status": result_array(B, np.int32, big)}
    if trace:
        out["A_trace"] = result_array((B, ns, 4), np.complex128, big and B * ns * 64 <= (1 << 30))
    if end:
        out["A_end"] = result_array((B, 4), np.complex128, big)
    if pmax:
        out["Pmax"] = result_array((B, 4), np.float64, big)
    d = _lib.Yaman4Desc()
    d.n_points = B
    d.dbeta = ptr(dbeta)
    d.gamma, d.gamma_stride = ptr(gam), gs
    d.alpha, d.alpha_stride = ptr(alp), as_
    d.A0, d.A0_stride = ptr(a0), a0s
    d.z0, d.z_max = float(z0), float(z_max)
    d.n_steps, d.save_every = n_steps, save_every
    d.z_grid = ptr(grid)
    d.flags = _flags(trace, end, pmax, check_nan, phase_exact)
    d.A_trace = ptr(out.get("A_trace"))
    d.A_end = ptr(out.get("A_end"))
    d.Pmax = ptr(out.get("Pmax"))
    d.status = ptr(out["status"])
    L = _lib.lib()
    _run_host(L.fpa_yaman4_rk4_batch_host, L.fpa_yaman4_rk4_batch_multi_host, d, device, devices)
    return out


def yaman4_rhs(z, A, gamma, alpha, dbeta, *, device: Optional[int] = None) -> np.ndarray:
    """dA[b,:] for B (z, A) pairs through `fpa_yaman4_rhs_host`."""
    A = c128(A).reshape(-1, 4)
    B = A.shape[0]
    z, gamma, alpha, dbeta = (np.ascontiguousarray(np.broadcast_to(f64(v).reshape(-1), (B,)))
                              for v in (z, gamma, alpha, dbeta))
    dA = np.empty_like(A)
    dev = _lib.get_device() if device is None else int(device)
    _lib.check(_lib.lib().fpa_yaman4_rhs_host(B, ptr(z), ptr(A), ptr(gamma), ptr(alpha), ptr(dbeta),
                                              ptr(dA), dev))
    return dA


def linear_batch(y0, lam, *, z0=0.0, z_max, n_steps, save_every=1, z_grid=None, trace=True, end=True,
                 check_nan=True, device: Optional[int] = None) -> dict:
    """y_j' = lam_j y_j for y0 [B,dim] through `fpa_linear_rk4_batch_host`."""
    y0 = c128(y0)
    if y0.ndim == 1:
        y0 = y0.reshape(1, -1)
    B, dim = y0.shape
    lam = c128(np.broadcast_to(c128(lam).reshape(-1), (dim,)))
    n_steps, save_every = int(n_steps), int(save_every)
    ns = n_saved(n_steps, save_every)
    grid = None if z_grid is None else f64(z_grid).reshape(-1)
    out = {"status": np.empty(B, dtype=np.int32)}
    if trace:
        out["y_trace"] = np.empty((B, ns, dim), dtype=np.complex128)
    if end:
        out["y_end"] = np.empty((B, dim), dtype=np.complex128)
    dev = _lib.get_device() if device is None else int(device)
    _lib.check(_lib.lib().fpa_linear_rk4_batch_host(
        B, dim, ptr(y0), ptr(lam), float(z0), float(z_max), n_steps, save_every, ptr(grid),
        _flags(trace, end, False, check_nan, False), ptr(out.get("y_trace")), ptr(out.get("y_end")),
        ptr(out["status"]), dev))
    return out


def new_plan_desc(lambda1, lambda2, lambda3):
    """PlanDesc over host wavelength axes; returns (desc, keepalive arrays)."""
    l1 = f64(lambda1).reshape(-1)
    l3 = f64(lambda3).reshape(-1)
    l2 = f64(lambda2).reshape(-1)
    if l2.size not in (1, l1.size):
        raise ValueError("lambda2 must be a scalar or match lambda1")
    p = _lib.PlanDesc()
    p.n1, p.n3 = l1.size, l3.size
    p.lambda1, p.lambda2, p.lambda3 = ptr(l1), ptr(l2), ptr(l3)
    p.lambda2_stride = 1 if (l2.size == l1.size and l1.size > 1) else 0
    return p, (l1, l2, l3)


def dbeta_table(plan, *, want_omega=False, device: Optional[int] = None) -> dict:
    """Run `fpa_dbeta_table_host` on a filled PlanDesc; returns dbeta [n1,n3], valid, omega."""
    B = plan.n1 * plan.n3
    out = {"dbeta": np.empty((plan.n1, plan.n3)), "valid": np.empty((plan.n1, plan.n3), dtype=np.int32)}
    if want_omega:
        out["omega"] = np.empty((plan.n1, plan.n3, 4))
    plan.dbeta, plan.valid, plan.omega = ptr(out["dbeta"]), ptr(out["valid"]), ptr(out.get("omega"))
    dev = _lib.get_device() if device is None else int(device)
    if B:
        _lib.check(_lib.lib().fpa_dbeta_table_host(C.byref(plan), dev))
    return out


def sweep(desc, *, want_pmax=False, want_end=False, device: Optional[int] = None,
          out: Optional[dict] = None, devices=None) -> dict:
    """Run `fpa_yaman4_sweep_host` on a SweepDesc whose plan axes / physics are filled.
    `out` may supply preallocated result arrays gain_lin / dbeta / valid / status; without it they
    come from the library's page-locked pool (`result_array`), so either way the kernel delivers
    its results straight into host memory.
    `devices`: CUDA ordinals to split the flattened grid over from this one process
    (`fpa_yaman4_sweep_multi_host`)."""
    n1, n3 = desc.plan.n1, desc.plan.n3
    given = out or {}
    out = {}
    for key, dtype in (("gain_lin", np.float64), ("dbeta", np.float64), ("valid", np.int32),
                       ("status", np.int32)):
        arr = given.get(key)
        if arr is None:
            arr = result_array((n1, n3), dtype, n1 * n3 >= 4096)
        elif arr.shape != (n1, n3) or arr.dtype != dtype or not arr.flags["C_CONTIGUOUS"]:
            raise ValueError(f"out[{key!r}] must be a C-contiguous {np.dtype(dtype)} array of shape {(n1, n3)}")
        out[key] = arr
    if want_pmax:
        out["Pmax"] = np.empty((n1, n3, 4))
    if want_end:
        out["A_end"] = np.empty((n1, n3, 4), dtype=np.complex128)
    desc.plan.dbeta, desc.plan.valid, desc.plan.omega = ptr(out["dbeta"]), ptr(out["valid"]), None
    desc.gain_lin, desc.status = ptr(out["gain_lin"]), ptr(out["status"])
    desc.Pmax, desc.A_end = ptr(out.get("Pmax")), ptr(out.get("A_end"))
    if n1 * n3 == 0:
        return out
    L = _lib.lib()
    _run_host(L.fpa_yaman4_sweep_host, L.fpa_yaman4_sweep_multi_host, desc, device, devices)
    return out


def phase_sweep(desc, *, want_map: bool = True, device: Optional[int] = None, devices=None) -> dict:
    """Run `fpa_yaman4_phase_sweep_host` on a PhaseSweepDesc whose plan axes, physics, n_phases, A0_table and
    metric are filled.  Returns gain_lin / status [n1,n3,K], dbeta / valid and the reductions gain_max,
    gain_min, idx_max, idx_min, n_finite [n1,n3].  `want_map=False` leaves the gain map in the library's
    workspace (no gain_lin in the result).  `devices`: split the grid over several GPUs
    (`fpa_yaman4_phase_sweep_multi_host`)."""
    n1, n3, K = desc.sweep.plan.n1, desc.sweep.plan.n3, int(desc.n_phases)
    big = n1 * n3 * K >= 4096
    out = {"dbeta": result_array((n1, n3), np.float64, big), "valid": result_array((n1, n3), np.int32, big),
           "status": result_array((n1, n3, K), np.int32, big)}
    if want_map:
        out["gain_lin"] = result_array((n1, n3, K), np.float64, big)
    for key, dtype in (("gain_max", np.float64), ("gain_min", np.float64), ("idx_max", np.int32),
                       ("idx_min", np.int32), ("n_finite", np.int32)):
        out[key] = result_array((n1, n3), dtype, big)
        setattr(desc, key, ptr(out[key]))
    w = desc.sweep
    w.plan.dbeta, w.plan.valid, w.plan.omega = ptr(out["dbeta"]), ptr(out["valid"]), None
    w.gain_lin, w.status, w.Pmax, w.A_end = ptr(out.get("gain_lin")), ptr(out["status"]), None, None
    if n1 * n3 == 0:
        return out
    L = _lib.lib()
    _run_host(L.fpa_yaman4_phase_sweep_host, L.fpa_yaman4_phase_sweep_multi_host, desc, device, devices)
    return out


def enumerate_triplets(grid_index) -> tuple[np.ndarray, np.ndarray]:
    """(table[T] of (k,l,m,weight) int16, row_ptr[N+1] int64) on an integer frequency grid."""
    g = np.ascontiguousarray(grid_index, dtype=np.int32).reshape(-1)
    N = g.size
    L = _lib.lib()
    count = L.fpa_enumerate_triplets(N, ptr(g), None, 0, None)
    if count < 0:
        raise ValueError(_lib.last_error())
    table = np.empty(count, dtype=_lib.TRIPLET_DTYPE)
    rows = np.empty(N + 1, dtype=np.int64)
    got = L.fpa_enumerate_triplets(N, ptr(g), ptr(table) if count else None, count, ptr(rows))
    if got != count:
        raise ValueError(_lib.last_error())
    return table, rows


def enumerate_triplets_omega(omega, atol: float = 0.0, rtol: float = 1e-12) -> tuple[np.ndarray, np.ndarray]:
    """(table, row_ptr) of a plan that is not on an integer grid: photon-energy matching with the reference's
    tolerance rule (`fpa_enumerate_triplets_omega`)."""
    w = f64(omega).reshape(-1)
    N = w.size
    L = _lib.lib()
    count = L.fpa_enumerate_triplets_omega(N, ptr(w), float(atol), float(rtol), None, 0, None)
    if count < 0:
        raise ValueError(_lib.last_error())
    table = np.empty(count, dtype=_lib.TRIPLET_DTYPE)
    rows = np.empty(N + 1, dtype=np.int64)
    got = L.fpa_enumerate_triplets_omega(N, ptr(w), float(atol), float(rtol), ptr(table) if count else None, count, ptr(rows))
    if got != count:
        raise ValueError(_lib.last_error())
    return table, rows


def factor_table(n_waves: int, table, row_ptr) -> tuple[np.ndarray, int]:
    """(blob, n_classes) of `fpa_nwave_factor_table`: the factored form of a triplet table the table kernel
    integrates from (pair products once per RHS, one cell per (n, m)); `fpa_nwave_rk4_batch_host` builds it
    itself, callers of the `_dev` entry upload the blob and point `fpa_nwave_desc.factored` at it."""
    table = np.ascontiguousarray(table, dtype=_lib.TRIPLET_DTYPE)
    rows = np.ascontiguousarray(row_ptr, dtype=np.int64)
    L = _lib.lib()
    nc = C.c_int32()
    nb = L.fpa_nwave_factor_table(int(n_waves), ptr(table) if table.size else None, ptr(rows), table.size, None, 0, C.byref(nc))
    if nb < 0:
        raise ValueError(_lib.last_error())
    blob = np.zeros(nb, dtype=np.uint8)
    if L.fpa_nwave_factor_table(int(n_waves), ptr(table) if table.size else None, ptr(rows), table.size, ptr(blob), nb, C.byref(nc)) != nb:
        raise ValueError(_lib.last_error())
    return blob, int(nc.value)


def nwave_batch(beta, gamma, alpha, A0, table, row_ptr, *, z0=0.0, z_max, n_steps, save_every=1,
                trace=False, end=True, pmax=False, check_nan=True, n_points: Optional[int] = None,
                grid_index=None, force_table: bool = False, force_comb: bool = False, plain_table: bool = False,
                device: Optional[int] = None, devices=None) -> dict:
    """B points of the N-wave model through `fpa_nwave_rk4_batch_host` (`devices=[...]`:
    `fpa_nwave_rk4_batch_multi_host`).  With `grid_index` (integer grid position of every wave) the
    library may integrate the convolution form of the same ODE (O(span^2) per RHS): it does so for plans
    within that kernel's limits unless they are sparse; `force_table` / `force_comb` override the choice.
    The table kernel integrates from the factored table (`factor_table`); `plain_table` makes it walk the entry
    list instead (the round-1 kernel, kept as the independent check)."""
    A0 = c128(A0)
    N = A0.shape[-1]
    beta = f64(beta)
    sizes = [A0.size // N, beta.size // N, f64(gamma).size, f64(alpha).size]
    B = int(n_points) if n_points is not None else max(sizes)
    bet, bs = _per_point(beta, B, N, "beta")
    gam, gs = _per_point(gamma, B, 1, "gamma")
    alp, as_ = _per_point(alpha, B, 1, "alpha")
    a0, a0s = _per_point(A0, B, N, "A0", c128)
    table = np.ascontiguousarray(table, dtype=_lib.TRIPLET_DTYPE)
    rows = np.ascontiguousarray(row_ptr, dtype=np.int64)
    n_steps, save_every = int(n_steps), int(save_every)
    ns = n_saved(n_steps, save_every)
    out = {"status": np.empty(B, dtype=np.int32)}
    if trace:
        out["A_trace"] = np.empty((B, ns, N), dtype=np.complex128)
    if end:
        out["A_end"] = np.empty((B, N), dtype=np.complex128)
    if pmax:
        out["Pmax"] = np.empty((B, N), dtype=np.float64)
    d = _lib.NwaveDesc()
    d.n_points, d.n_waves = B, N
    d.beta, d.beta_stride = ptr(bet), bs
    d.gamma, d.gamma_stride = ptr(gam), gs
    d.alpha, d.alpha_stride = ptr(alp), as_
    d.A0, d.A0_stride = ptr(a0), a0s
    d.triplets, d.row_ptr, d.n_triplets = (ptr(table) if table.size else None), ptr(rows), table.size
    d.z0, d.z_max, d.n_steps, d.save_every = float(z0), float(z_max), n_steps, save_every
    d.flags = (_flags(trace, end, pmax, check_nan, False) | (_lib.NWAVE_TABLE if force_table else 0) |
               (_lib.NWAVE_COMB if force_comb else 0) | (_lib.NWAVE_PLAIN if plain_table else 0))
    d.A_trace, d.A_end, d.Pmax = ptr(out.get("A_trace")), ptr(out.get("A_end")), ptr(out.get("Pmax"))
    d.status = ptr(out["status"])
    slots = None
    if grid_index is not None:
        g = np.asarray(grid_index, dtype=np.int64).reshape(-1)
        if g.size != N:
            raise ValueError("grid_index must hold one entry per wave")
        slots = np.ascontiguousarray(g - g.min(), dtype=np.int32)
        d.grid_slot, d.grid_span = ptr(slots), int(g.max() - g.min() + 1)
    L = _lib.lib()
    _run_host(L.fpa_nwave_rk4_batch_host, L.fpa_nwave_rk4_batch_multi_host, d, device, devices)
    return out


def fp64_peak(iters: int = 4096, device: Optional[int] = None) -> tuple[float, float]:
    """(TFLOP/s, ms) of the DFMA probe kernel."""
    tf, ms = C.c_double(), C.c_double()
    dev = _lib.get_device() if device is None else int(device)
    _lib.check(_lib.lib().fpa_fp64_peak_probe(dev, int(iters), C.byref(tf), C.byref(ms)))
    return tf.value, ms.value
