"""CPU (with or without a device): every host-pointer entry point refuses a malformed descriptor with FPA_ERR_INVALID
and names the fault in fpa_last_error(), before it selects a device or stages anything."""
import ctypes as C

import numpy as np
import pytest

BIG_STEPS = 1 << 31


def _batch(L, keep):
    B = 3
    arrs = dict(dbeta=np.zeros(B), gamma=np.full(1, 0.01), alpha=np.zeros(1), A0=np.ones(4, np.complex128),
                A_trace=np.empty((B, 3, 4), np.complex128), A_end=np.empty((B, 4), np.complex128),
                Pmax=np.empty((B, 4)), status=np.empty(B, np.int32))
    keep.append(arrs)
    d = L.Yaman4Desc()
    d.n_points, d.z_max, d.n_steps, d.save_every = B, 1.0, 2, 1
    for k, a in arrs.items():
        setattr(d, k, L.ptr(a))
    d.flags = L.OUT_TRACE | L.OUT_END | L.OUT_PMAX | L.CHECK_NAN
    return d


def _sweep(L, keep, d=None):
    lam1, lam2, lam3 = np.array([1550e-9, 1551e-9]), np.array([1558e-9]), np.linspace(1540e-9, 1565e-9, 4)
    out = dict(gain_lin=np.empty(8), status=np.empty(8, np.int32), db=np.empty(8), va=np.empty(8, np.int32))
    keep += [lam1, lam2, lam3, out]
    d = L.SweepDesc() if d is None else d
    d.plan.n1, d.plan.n3 = 2, 4
    d.plan.lambda1, d.plan.lambda2, d.plan.lambda3 = L.ptr(lam1), L.ptr(lam2), L.ptr(lam3)
    d.plan.dbeta, d.plan.valid = L.ptr(out["db"]), L.ptr(out["va"])
    d.plan.method = L.PM_PROVIDED
    d.p_signal, d.gamma, d.z_max, d.dz, d.length_scale, d.save_every = 1.0, 0.01, 1.0, 0.1, 1.0, 1
    d.gain_lin, d.status = L.ptr(out["gain_lin"]), L.ptr(out["status"])
    return d


def _phase(L, keep):
    d = L.PhaseSweepDesc()
    _sweep(L, keep, d.sweep)
    table, gmax = np.ones((2, 4), np.complex128), np.empty(8)
    keep += [table, gmax]
    d.n_phases, d.A0_table, d.metric, d.gain_max = 2, L.ptr(table), L.GAIN_MAX_SAVED, L.ptr(gmax)
    return d


def _nwave(L, keep):
    B, N = 3, 4
    slots = np.array([0, 1, 2, 3], np.int32)
    arrs = dict(beta=np.zeros(N), gamma=np.full(1, 0.01), alpha=np.zeros(1), A0=np.ones(N, np.complex128),
                A_trace=np.empty((B, 3, N), np.complex128), A_end=np.empty((B, N), np.complex128),
                Pmax=np.empty((B, N)), status=np.empty(B, np.int32))
    keep += [arrs, slots]
    d = L.NwaveDesc()
    d.n_points, d.n_waves, d.z_max, d.n_steps, d.save_every = B, N, 1.0, 2, 1
    for k, a in arrs.items():
        setattr(d, k, L.ptr(a))
    d.grid_slot, d.grid_span = L.ptr(slots), 4
    d.flags = L.OUT_TRACE | L.OUT_END | L.OUT_PMAX | L.CHECK_NAN
    return d, slots


def _host_and_multi(lib, host, multi):
    ids = (C.c_int * 2)(0, 0)
    return [lambda d: getattr(lib, host)(d, 0), lambda d: getattr(lib, multi)(d, 2, ids)]


def _refused(L, rc, word):
    assert rc == L.ERR_INVALID, (rc, L.last_error())
    assert word in L.last_error(), L.last_error()


BATCH_CASES = [
    ("n_points", -1, "n_points"), ("n_steps", 0, "n_steps"), ("n_steps", BIG_STEPS, "n_steps"),
    ("save_every", 0, "save_every"), ("dbeta", None, "must be set"), ("A0", None, "must be set"),
    ("gamma_stride", 2, "strides"), ("A0_stride", 2, "strides"),
    ("A_trace", None, "FPA_OUT_TRACE"), ("Pmax", None, "FPA_OUT_PMAX"), ("A_end", None, "FPA_OUT_END"),
]


@pytest.mark.parametrize("field, value, word", BATCH_CASES)
@pytest.mark.parametrize("multi", [False, True])
def test_batch_refusals(fpa, field, value, word, multi):
    L, keep = fpa._lib, []
    d = _batch(L, keep)
    setattr(d, field, value)
    call = _host_and_multi(L.lib(), "fpa_yaman4_rk4_batch_host", "fpa_yaman4_rk4_batch_multi_host")[multi]
    _refused(L, call(C.byref(d)), word)


SWEEP_CASES = [
    ("plan.n1", -1, "grid sizes"), ("plan.lambda3", None, "wavelength axes"),
]


def _set(d, path, value):
    *head, last = path.split(".")
    for part in head:
        d = getattr(d, part)
    setattr(d, last, value)


@pytest.mark.parametrize("field, value, word", SWEEP_CASES)
@pytest.mark.parametrize("multi", [False, True])
def test_sweep_refusals(fpa, field, value, word, multi):
    L, keep = fpa._lib, []
    d = _sweep(L, keep)
    _set(d, field, value)
    call = _host_and_multi(L.lib(), "fpa_yaman4_sweep_host", "fpa_yaman4_sweep_multi_host")[multi]
    _refused(L, call(C.byref(d)), word)


@pytest.mark.parametrize("first, count", [(7, 2), (-1, 1), (0, 9), (9, 0)])
def test_sweep_sub_range_outside_the_grid(fpa, first, count):
    """Checked before the device is selected: the host entry sizes its buffers from this range."""
    L, keep = fpa._lib, []
    for d, entry in ((_sweep(L, keep), "fpa_yaman4_sweep_host"), (_phase(L, keep), "fpa_yaman4_phase_sweep_host")):
        w = getattr(d, "sweep", d)
        w.first_point, w.n_sub_points = first, count
        _refused(L, getattr(L.lib(), entry)(C.byref(d), 0), "first_point")


PHASE_CASES = [
    ("n_phases", 0, "n_phases"), ("n_phases", 65537, "n_phases"), ("A0_table", None, "A0_table"),
    ("metric", 7, "metric"), ("sweep.n_peers", 1, "n_peers"), ("sweep.plan.n3", -1, "grid sizes"),
    ("sweep.plan.lambda1", None, "wavelength axes"),
]


@pytest.mark.parametrize("field, value, word", PHASE_CASES)
def test_phase_sweep_refusals(fpa, field, value, word):
    L, keep = fpa._lib, []
    d = _phase(L, keep)
    _set(d, field, value)
    _refused(L, L.lib().fpa_yaman4_phase_sweep_host(C.byref(d), 0), word)


@pytest.mark.parametrize("n_devices, word", [(0, "device ordinals"), (65, "device ordinals")])
def test_multi_host_device_lists(fpa, n_devices, word):
    L, keep, lib = fpa._lib, [], fpa._lib.lib()
    ids = (C.c_int * 65)()
    d, _ = _nwave(L, keep)
    for entry, desc in (("fpa_yaman4_rk4_batch_multi_host", _batch(L, keep)),
                        ("fpa_yaman4_sweep_multi_host", _sweep(L, keep)),
                        ("fpa_yaman4_phase_sweep_multi_host", _phase(L, keep)),
                        ("fpa_nwave_rk4_batch_multi_host", d)):
        _refused(L, getattr(lib, entry)(C.byref(desc), n_devices, ids), word)
        _refused(L, getattr(lib, entry)(C.byref(desc), 2, None), word)


def test_multi_host_sweeps_split_the_whole_grid(fpa):
    L, keep, lib = fpa._lib, [], fpa._lib.lib()
    ids = (C.c_int * 2)(0, 0)
    d, p = _sweep(L, keep), _phase(L, keep)
    d.first_point = p.sweep.first_point = 1
    _refused(L, lib.fpa_yaman4_sweep_multi_host(C.byref(d), 2, ids), "whole grid")
    _refused(L, lib.fpa_yaman4_phase_sweep_multi_host(C.byref(p), 2, ids), "whole grid")


def test_null_descriptors(fpa):
    L, lib = fpa._lib, fpa._lib.lib()
    ids = (C.c_int * 2)(0, 0)
    for entry in ("fpa_yaman4_rk4_batch_host", "fpa_yaman4_sweep_host", "fpa_yaman4_phase_sweep_host",
                  "fpa_nwave_rk4_batch_host", "fpa_dbeta_table_host"):
        _refused(L, getattr(lib, entry)(None, 0), "descriptor is NULL")
    for entry in ("fpa_yaman4_rk4_batch_multi_host", "fpa_yaman4_sweep_multi_host",
                  "fpa_yaman4_phase_sweep_multi_host", "fpa_nwave_rk4_batch_multi_host"):
        _refused(L, getattr(lib, entry)(None, 2, ids), "descriptor is NULL")


NWAVE_CASES = [
    ("n_points", -1, "n_points"), ("n_waves", 0, "n_waves"), ("n_steps", 0, "n_steps"),
    ("n_steps", BIG_STEPS, "n_steps"), ("save_every", 0, "save_every"), ("beta", None, "must be set"),
    ("gamma", None, "must be set"), ("beta_stride", 2, "strides"), ("alpha_stride", 2, "strides"),
    ("A_trace", None, "FPA_OUT_TRACE"), ("Pmax", None, "FPA_OUT_PMAX"), ("A_end", None, "FPA_OUT_END"),
    ("flags", "table|comb", "exclude"), ("grid_slot", None, "triplet table"), ("grid_span", 0, "grid_span"),
    ("slot", (0, 4), "outside"), ("slot", (2, -1), "outside"), ("slot", (3, 1), "distinct"),
]


@pytest.mark.parametrize("field, value, word", NWAVE_CASES)
@pytest.mark.parametrize("multi", [False, True])
def test_nwave_refusals(fpa, field, value, word, multi):
    L, keep = fpa._lib, []
    d, slots = _nwave(L, keep)
    if field == "flags":
        d.flags |= L.NWAVE_TABLE | L.NWAVE_COMB
    elif field == "slot":
        slots[value[0]] = value[1]
    else:
        setattr(d, field, value)
    call = _host_and_multi(L.lib(), "fpa_nwave_rk4_batch_host", "fpa_nwave_rk4_batch_multi_host")[multi]
    _refused(L, call(C.byref(d)), word)


def test_nwave_forced_comb_needs_grid_slot(fpa):
    L, keep = fpa._lib, []
    d, _ = _nwave(L, keep)
    d.grid_slot, d.flags = None, d.flags | L.NWAVE_COMB
    _refused(L, L.lib().fpa_nwave_rk4_batch_host(C.byref(d), 0), "needs grid_slot")


def test_linear_rhs_and_dbeta_table_refusals(fpa):
    L, lib = fpa._lib, fpa._lib.lib()
    y0, lam = np.ones((2, 3), np.complex128), np.ones(3, np.complex128)
    yt, ye, st = np.empty((2, 2, 3), np.complex128), np.empty((2, 3), np.complex128), np.empty(2, np.int32)
    base = dict(B=2, dim=3, y0=L.ptr(y0), lam=L.ptr(lam), n_steps=1, save_every=1, flags=L.OUT_TRACE | L.OUT_END,
                y_trace=L.ptr(yt), y_end=L.ptr(ye))

    def linear(**change):
        a = {**base, **change}
        return lib.fpa_linear_rk4_batch_host(a["B"], a["dim"], a["y0"], a["lam"], 0.0, 1.0, a["n_steps"],
                                             a["save_every"], None, a["flags"], a["y_trace"], a["y_end"],
                                             L.ptr(st), 0)

    for change, word in (({"B": -1}, "dim"), ({"dim": 0}, "dim"), ({"n_steps": 0}, "n_steps"),
                         ({"save_every": 0}, "save_every"), ({"y0": None}, "y0"),
                         ({"y_trace": None}, "FPA_OUT_TRACE"), ({"y_end": None}, "FPA_OUT_END")):
        _refused(L, linear(**change), word)

    z, A, dA = np.zeros(2), np.ones((2, 4), np.complex128), np.empty((2, 4), np.complex128)
    _refused(L, lib.fpa_yaman4_rhs_host(-1, L.ptr(z), L.ptr(A), L.ptr(z), L.ptr(z), L.ptr(z), L.ptr(dA), 0), "B must")
    _refused(L, lib.fpa_yaman4_rhs_host(2, L.ptr(z), L.ptr(A), L.ptr(z), L.ptr(z), L.ptr(z), None, 0), "NULL")

    keep = []
    for field, value, word in (("n1", -1, "grid sizes"), ("lambda2", None, "wavelength axes"),
                               ("dbeta", None, "dbeta output")):
        d = _sweep(L, keep).plan
        setattr(d, field, value)
        _refused(L, lib.fpa_dbeta_table_host(C.byref(d), 0), word)
