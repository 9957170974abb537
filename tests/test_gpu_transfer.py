"""GPU: small-signal transfer matrices (fpa_yaman4_transfer_*).  J against the CPU tangent model
(tools/transfer_model.py) and against finite differences of the library's own batch integrator; the base outputs
bit for bit those of the plain batch / sweep; every entry, column mask, device split and the ptxas-schedule build
giving the same bits; NaN J for failed points; refusals; undepleted-pump theory; and the ties to the phase sweep
and to the batch integrator's pump-power response."""
import ctypes as C
import os
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tools"))
import transfer_model as TM  # noqa: E402
from test_transfer_ld_cpu import assert_blocks, assert_waves  # noqa: E402

pytestmark = pytest.mark.gpu
P_IN = [0.3, 0.2, 1e-4, 2e-5]
PHASE_IN = [0.1, -0.2, 0.3, 0.05]


@pytest.fixture(autouse=True)
def _clean_env():
    yield
    os.environ.pop("FPA_SWEEP_SYM", None)


def _rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / np.max(np.abs(b)))


def _disp(fpa, golden, scale=1.0):
    b2, b3, b4, wref = golden["b4_beta"]
    return fpa.dispersion.DispersionParams(omega_ref=wref, beta2=b2 * scale, beta3=b3 * scale, beta4=b4 * scale)


def _sweep_kw(gpu, golden, unit="m", alpha=1e-4, n1=6, n3=50, z_max=20.0, wide=True, p_in=P_IN, save_every=7):
    s = 1.0 if unit == "m" else 1e-3
    cfg = gpu.config.custom_simulation_config(z_max=z_max * s, dz=0.2 * s, save_every=save_every)
    lam3 = np.linspace(600e-9, 1700e-9, n3) if wide else np.linspace(1540e-9, 1565e-9, n3)  # wide: invalid plans
    return dict(cfg=cfg, lambda_p1_m=np.linspace(1545e-9, 1555e-9, n1), lambda_signal_m=lam3, lambda_p2_m=1558e-9,
                gamma=11.5e-3 / s, alpha=alpha / s, p_in=p_in, phase_in=PHASE_IN, dispersion=_disp(gpu, golden, 1.0 / s),
                length_unit=unit)


def _sweep_desc(gpu, kw):
    """The SweepDesc sweep_gain_2d / sweep_transfer_2d build for `kw` (and the arrays it points to)."""
    sm = gpu.scan_mismtach
    cfg = kw["cfg"]
    s = 1.0 if kw["length_unit"] == "m" else 1000.0
    pm = sm._default_phase_matching_cfg(dispersion=kw["dispersion"], beta_legacy=None)
    d = gpu._lib.SweepDesc()
    plan, keep = gpu._device.new_plan_desc(np.atleast_1d(kw["lambda_p1_m"]), np.atleast_1d(kw["lambda_p2_m"]),
                                           np.asarray(kw["lambda_signal_m"]))
    gpu.phase_matching.fill_plan_desc(plan, kw["dispersion"], pm)
    d.plan = plan
    A0 = gpu.simulation.make_initial_amplitudes(kw["p_in"], kw["phase_in"])
    for j in range(4):
        d.A0[2 * j], d.A0[2 * j + 1] = A0[j].real, A0[j].imag
    d.p_signal = float(kw["p_in"][2])
    d.gamma, d.alpha = float(kw["gamma"]), float(kw["alpha"])
    d.z_max, d.dz, d.length_scale = float(cfg.z_max), float(cfg.dz), s
    d.save_every = int(cfg.save_every)
    d.flags = gpu._lib.CHECK_NAN if cfg.check_nan else 0
    return d, keep


def _batch_inputs(B=24, seed=3):
    rng = np.random.default_rng(seed)
    A0 = np.sqrt(np.array(P_IN)) * np.exp(1j * np.array(PHASE_IN)) * (1.0 + 0.05 * rng.standard_normal((B, 4)))
    return rng.uniform(-0.5, 0.5, B), A0, rng.uniform(0.01, 0.02, B), rng.uniform(0.0, 2e-3, B)


# ------------------------------------------------------------------ J against the CPU tangent model
@pytest.mark.parametrize("case", ["lossy_uniform", "lossless_uniform", "per_point", "z0"])
def test_batch_jac_matches_cpu_model(gpu, case):
    db, A0, gam, alp = _batch_inputs(B=6)
    n_steps, z_max, z0 = 70, 30.0, 0.0
    if case == "lossy_uniform":
        gam, alp = 0.015, 1e-3
    elif case == "lossless_uniform":
        gam, alp = 0.015, 0.0
    elif case == "z0":
        gam, alp, z0, z_max = 0.015, 1e-3, 7.5, 37.5
    r = gpu._device.yaman4_transfer(db, gam, alp, A0, 0xFF, z0=z0, z_max=z_max, n_steps=n_steps)
    worst = 0.0
    for b in range(db.size):
        g = gam if np.isscalar(gam) else gam[b]
        a = alp if np.isscalar(alp) else alp[b]
        A_end, J = TM.integrate(A0[b], g, a, db[b], z_max, n_steps, z0=z0)
        worst = max(worst, assert_blocks(r["jac"][b], J, 1e-13, f"{case} point {b}")[0])
        assert_waves(r["A_end"][b], A_end, 1e-13, f"{case} point {b}")
    assert np.all(r["status"] == -1)
    print(f"\n{case}: kernel vs the FP64 model, largest per-block error {worst:.1e}")


def test_sweep_jac_matches_cpu_model_km(gpu, golden):
    kw = _sweep_kw(gpu, golden, unit="km", n1=2, n3=6, wide=False, z_max=10.0)
    r = gpu.scan_mismtach.sweep_transfer_2d(waves=(0, 1, 2, 3), **kw)
    L = 10.0
    A0 = gpu.simulation.make_initial_amplitudes(P_IN, PHASE_IN)
    n_steps = r["n_steps"]
    # the integration uses dbeta / 1000 per metre; the reported dbeta is per km
    worst = 0.0
    for i1 in range(2):
        for i3 in range(6):
            _, J = TM.integrate(A0, 11.5e-3, 1e-4, r["dbeta"][i1, i3] / 1000.0, L, n_steps)
            worst = max(worst, assert_blocks(r["jac"][i1, i3], J, 1e-13, f"point ({i1}, {i3})")[0])
    print(f"\nkm sweep: kernel vs the FP64 model, largest per-block error {worst:.1e}")


# ------------------------------------------------------------------ J against finite differences of the batch integrator
def test_batch_jac_matches_finite_differences_of_the_integrator(gpu):
    db, A0, gam, alp = _batch_inputs(B=4, seed=7)
    n_steps, z_max = 200, 60.0
    r = gpu._device.yaman4_transfer(db, gam, alp, A0, 0xFF, z_max=z_max, n_steps=n_steps)
    for b in range(db.size):
        y0 = A0[b].view(np.float64).copy()
        eps = 1e-6 * np.max(np.abs(y0))
        pert = []
        for c in range(8):
            for sgn in (1.0, -1.0):
                y = y0.copy()
                y[c] += sgn * eps
                pert.append(y.view(np.complex128))
        out = gpu._device.yaman4_batch(np.full(16, db[b]), gam[b], alp[b], np.array(pert), z_max=z_max,
                                       n_steps=n_steps)["A_end"].view(np.float64).reshape(8, 2, 8)
        Jfd = ((out[:, 0] - out[:, 1]) / (2 * eps)).T
        assert _rel(r["jac"][b], Jfd) <= 1e-6


# ------------------------------------------------------------------ bit identity
def test_batch_base_outputs_bit_identical_to_the_integrator(gpu):
    db, A0, gam, alp = _batch_inputs(B=300)
    for g, a in ((gam, alp), (0.015, 1e-3), (0.015, 0.0)):
        r = gpu._device.yaman4_transfer(db, g, a, A0, 0x30, z_max=40.0, n_steps=160, pmax=True)
        ref = gpu._device.yaman4_batch(db, g, a, A0, z_max=40.0, n_steps=160, pmax=True)
        for k in ("A_end", "status", "Pmax"):
            assert r[k].tobytes() == ref[k].tobytes(), k


def test_column_subsets_equal_the_full_mask(gpu):
    db, A0, gam, alp = _batch_inputs(B=37)
    full = gpu._device.yaman4_transfer(db, gam, alp, A0, 0xFF, z_max=20.0, n_steps=96)["jac"]
    for mask in (0x01, 0x80, 0x30, 0xC0, 0x5A, 0x07, 0x7F):
        cols = [c for c in range(8) if mask >> c & 1]
        sub = gpu._device.yaman4_transfer(db, gam, alp, A0, mask, z_max=20.0, n_steps=96)["jac"]
        assert sub.tobytes() == np.ascontiguousarray(full[:, :, cols]).tobytes(), hex(mask)


@pytest.mark.parametrize("sym", ["0", "1"])
def test_sweep_base_outputs_bit_identical_to_the_sweep(gpu, golden, sym):
    os.environ["FPA_SWEEP_SYM"] = sym
    for p_in, phase_in, alpha in ((P_IN, PHASE_IN, 1e-4), ([0.1, 0.1, 1e-7, 1e-7], None, 1e-4),
                                  ([0.1, 0.1, 1e-7, 1e-7], None, 0.0)):
        kw = _sweep_kw(gpu, golden, alpha=alpha, p_in=p_in)
        kw["phase_in"] = phase_in
        r = gpu.scan_mismtach.sweep_transfer_2d(**kw)
        d, keep = _sweep_desc(gpu, kw)
        ref = gpu._device.sweep(d, want_end=True)
        for k in ("gain_lin", "dbeta", "valid", "status", "A_end"):
            assert r[k].tobytes() == ref[k].tobytes(), (sym, k)


def test_entries_and_device_splits_agree(gpu, golden):
    import torch
    kw = _sweep_kw(gpu, golden, n1=5, n3=41)
    ref = gpu.scan_mismtach.sweep_transfer_2d(**kw)
    for devs in ([0, 0], [0, 0, 0], [0] * 7):
        r = gpu.scan_mismtach.sweep_transfer_2d(devices=devs, **kw)
        for k in ("jac", "gain_lin", "dbeta", "valid", "status", "A_end"):
            assert r[k].tobytes() == ref[k].tobytes(), (devs, k)
    L = gpu._lib
    G = 5 * 41
    nc = ref["jac"].shape[-1]
    # host sub-ranges of the flattened grid
    for lo, n in ((0, 1), (13, 57), (G - 9, 9)):
        d, keep = _sweep_desc(gpu, kw)
        jac = np.full((n, 8, nc), 7.0)
        gain, status = np.empty(n), np.empty(n, np.int32)
        dbeta, valid = np.empty(n), np.empty(n, np.int32)
        d.first_point, d.n_sub_points = lo, n
        d.gain_lin, d.status, d.plan.dbeta, d.plan.valid = gain.ctypes.data, status.ctypes.data, dbeta.ctypes.data, valid.ctypes.data
        t = L.TransferOut(columns=0xF0, jac=jac.ctypes.data)
        L.check(L.lib().fpa_yaman4_transfer_sweep_host(C.byref(d), C.byref(t), 0))
        assert jac.tobytes() == ref["jac"].reshape(G, 8, nc)[lo:lo + n].tobytes()
        assert gain.tobytes() == ref["gain_lin"].reshape(-1)[lo:lo + n].tobytes()
        assert status.tobytes() == ref["status"].reshape(-1)[lo:lo + n].tobytes()
    # the _dev entry
    d, keep = _sweep_desc(gpu, kw)
    dev = "cuda:0"
    ax = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in keep]
    d.plan.lambda1, d.plan.lambda2, d.plan.lambda3 = (a.data_ptr() for a in ax)
    o = {"jac": torch.empty((G, 8, nc), dtype=torch.float64, device=dev),
         "gain_lin": torch.empty(G, dtype=torch.float64, device=dev),
         "status": torch.empty(G, dtype=torch.int32, device=dev), "dbeta": torch.empty(G, dtype=torch.float64, device=dev),
         "valid": torch.empty(G, dtype=torch.int32, device=dev)}
    d.gain_lin, d.status = o["gain_lin"].data_ptr(), o["status"].data_ptr()
    d.plan.dbeta, d.plan.valid = o["dbeta"].data_ptr(), o["valid"].data_ptr()
    t = L.TransferOut(columns=0xF0, jac=o["jac"].data_ptr())
    L.check(L.lib().fpa_yaman4_transfer_sweep_dev(C.byref(d), C.byref(t), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    assert o["jac"].cpu().numpy().tobytes() == ref["jac"].reshape(G, 8, nc).tobytes()
    for k in ("gain_lin", "status", "dbeta", "valid"):
        assert o[k].cpu().numpy().tobytes() == ref[k].reshape(-1).tobytes(), k
    # batch: host against _dev
    db, A0, gam, alp = _batch_inputs(B=50)
    rb = gpu._device.yaman4_transfer(db, gam, alp, A0, 0xFF, z_max=20.0, n_steps=64)
    for devs in [[0, 0, 0]] + ([[0, 1]] if L.device_count() > 1 else []):
        rb2 = gpu._device.yaman4_transfer(db, gam, alp, A0, 0xFF, z_max=20.0, n_steps=64, devices=devs)
        assert rb["jac"].tobytes() == rb2["jac"].tobytes(), devs
    bd = L.Yaman4Desc()
    ins = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in
           (("db", db), ("gam", gam), ("alp", alp), ("A0", A0.astype(np.complex128)))}
    bd.n_points, bd.z_max, bd.n_steps, bd.save_every = 50, 20.0, 64, 1
    bd.dbeta, bd.gamma, bd.alpha, bd.A0 = (ins[k].data_ptr() for k in ("db", "gam", "alp", "A0"))
    bd.gamma_stride = bd.alpha_stride = bd.A0_stride = 1
    jac = torch.empty((50, 8, 8), dtype=torch.float64, device=dev)
    st = torch.empty(50, dtype=torch.int32, device=dev)
    bd.status, bd.flags = st.data_ptr(), L.CHECK_NAN
    t = L.TransferOut(columns=0xFF, jac=jac.data_ptr())
    L.check(L.lib().fpa_yaman4_transfer_batch_dev(C.byref(bd), C.byref(t), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    assert jac.cpu().numpy().tobytes() == rb["jac"].tobytes()


def test_shipped_library_equals_ptxas_schedule_library(gpu, golden):
    import __graft_entry__ as entry
    kw = _sweep_kw(gpu, golden)
    db, A0, gam, alp = _batch_inputs(B=40)
    a = gpu.scan_mismtach.sweep_transfer_2d(waves=(0, 1, 2, 3), **kw)
    b = gpu._device.yaman4_transfer(db, gam, alp, A0, 0xFF, z_max=20.0, n_steps=100)
    c = gpu._device.yaman4_transfer(db, 0.015, 0.0, A0, 0xFF, z_max=20.0, n_steps=100)
    with gpu._lib.use_library(entry.REF_LIB):
        a2 = gpu.scan_mismtach.sweep_transfer_2d(waves=(0, 1, 2, 3), **kw)
        b2 = gpu._device.yaman4_transfer(db, gam, alp, A0, 0xFF, z_max=20.0, n_steps=100)
        c2 = gpu._device.yaman4_transfer(db, 0.015, 0.0, A0, 0xFF, z_max=20.0, n_steps=100)
    for x, y in ((a, a2), (b, b2), (c, c2)):
        for k in x:
            if isinstance(x[k], np.ndarray):
                assert x[k].tobytes() == y[k].tobytes(), k


# ------------------------------------------------------------------ failed points
def test_invalid_and_overflowing_points_get_nan_jac(gpu, golden):
    kw = _sweep_kw(gpu, golden)                     # the wide signal axis has invalid plans
    r = gpu.scan_mismtach.sweep_transfer_2d(**kw)
    bad = r["valid"] == 0
    assert bad.any() and (~bad).any()
    assert np.all(np.isnan(r["jac"][bad])) and np.all(np.isfinite(r["jac"][~bad]))
    # overflow under check_nan: huge powers and gamma
    db, A0, _, _ = _batch_inputs(B=8)
    A0 = A0 * 1e3
    r = gpu._device.yaman4_transfer(db, 50.0, 0.0, A0, 0xFF, z_max=500.0, n_steps=200)
    ref = gpu._device.yaman4_batch(db, 50.0, 0.0, A0, z_max=500.0, n_steps=200)
    assert r["status"].tobytes() == ref["status"].tobytes()
    failed = r["status"] != -1
    assert failed.any()
    assert np.all(np.isnan(r["jac"][failed])) and np.all(np.isfinite(r["jac"][~failed]))
    # NaN dbeta in a batch
    db[2] = np.nan
    r = gpu._device.yaman4_transfer(db, 0.015, 1e-3, A0 / 1e3, 0xFF, z_max=5.0, n_steps=20)
    assert np.all(np.isnan(r["jac"][2])) and r["status"][2] == 0 and np.all(np.isfinite(r["jac"][3]))


# ------------------------------------------------------------------ refusals
def test_refusals_leave_outputs_untouched(gpu, golden):
    import torch
    L = gpu._lib
    lib = L.lib()
    db, A0, gam, alp = _batch_inputs(B=4)
    jac = np.full((4, 8, 8), 7.0)
    st = np.full(4, 5, np.int32)
    a_end = np.full((4, 4), 3.0 + 0j)

    def desc(**kv):
        d = L.Yaman4Desc()
        d.n_points, d.z_max, d.n_steps, d.save_every = 4, 5.0, 10, 1
        d.dbeta, d.gamma, d.alpha, d.A0 = db.ctypes.data, gam.ctypes.data, alp.ctypes.data, A0.ctypes.data
        d.gamma_stride = d.alpha_stride = d.A0_stride = 1
        d.status, d.A_end, d.flags = st.ctypes.data, a_end.ctypes.data, L.OUT_END | L.CHECK_NAN
        for k, v in kv.items():
            setattr(d, k, v)
        return d

    grid = np.linspace(0.0, 5.0, 11)
    trace = np.empty((4, 11, 4), np.complex128)
    t = L.TransferOut(columns=0xFF, jac=jac.ctypes.data)
    cases = [(desc(flags=L.OUT_TRACE | L.OUT_END, A_trace=trace.ctypes.data), t, L.ERR_UNSUPPORTED),
             (desc(z_grid=grid.ctypes.data), t, L.ERR_UNSUPPORTED),
             (desc(flags=L.PHASE_EXACT | L.OUT_END), t, L.ERR_UNSUPPORTED),
             (desc(), L.TransferOut(columns=0, jac=jac.ctypes.data), L.ERR_INVALID)]
    for d, tt, rc in cases:
        assert lib.fpa_yaman4_transfer_batch_host(C.byref(d), C.byref(tt), 0) == rc
    assert np.all(jac == 7.0) and np.all(st == 5) and np.all(a_end == 3.0)
    # sweeps
    kw = _sweep_kw(gpu, golden, n1=2, n3=5)
    G = 10
    sj = np.full((G, 8, 2), 7.0)
    gain = np.full(G, 9.0)
    d, keep = _sweep_desc(gpu, kw)
    d.gain_lin = gain.ctypes.data
    d.n_peers = 1
    assert lib.fpa_yaman4_transfer_sweep_host(C.byref(d), C.byref(L.TransferOut(columns=0x30, jac=sj.ctypes.data)), 0) == L.ERR_INVALID
    d.n_peers = 0
    assert lib.fpa_yaman4_transfer_sweep_host(C.byref(d), C.byref(L.TransferOut(columns=0, jac=sj.ctypes.data)), 0) == L.ERR_INVALID
    d.p_signal = 0.0
    assert lib.fpa_yaman4_transfer_sweep_host(C.byref(d), C.byref(L.TransferOut(columns=0x30, jac=sj.ctypes.data)), 0) == L.ERR_INVALID
    d.p_signal = P_IN[2]
    d.flags |= L.PHASE_EXACT
    assert lib.fpa_yaman4_transfer_sweep_host(C.byref(d), C.byref(L.TransferOut(columns=0x30, jac=sj.ctypes.data)), 0) == L.ERR_UNSUPPORTED
    assert np.all(sj == 7.0) and np.all(gain == 9.0)
    # a _dev jac that is not 8-byte aligned
    dev = "cuda:0"
    raw = torch.full((4 * 64 * 8 + 8,), 0xA5, dtype=torch.uint8, device=dev)
    ins = {k: torch.from_numpy(np.ascontiguousarray(v)).to(dev) for k, v in
           (("db", db), ("gam", gam), ("alp", alp), ("A0", A0))}
    bd = desc()
    bd.dbeta, bd.gamma, bd.alpha, bd.A0 = (ins[k].data_ptr() for k in ("db", "gam", "alp", "A0"))
    bd.A_end, bd.flags = None, L.CHECK_NAN
    sdev = torch.full((4,), 5, dtype=torch.int32, device=dev)
    bd.status = sdev.data_ptr()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = lib.fpa_yaman4_transfer_batch_dev(C.byref(bd), C.byref(L.TransferOut(columns=0xFF, jac=raw.data_ptr() + 4)), stream)
    assert rc == L.ERR_INVALID and "aligned" in L.last_error()
    torch.cuda.synchronize()
    assert bool((raw == 0xA5).all()) and bool((sdev == 5).all())


# ------------------------------------------------------------------ theory and ties to the existing features
@pytest.mark.parametrize("kappa", [0.0, 0.006, 0.03])
def test_undepleted_pump_theory(gpu, kappa):
    g, P, L_, n = 0.01, 0.5, 500.0, 2000
    db = kappa - g * 2 * P
    cfg = gpu.config.custom_simulation_config(z_max=L_, dz=L_ / n, save_every=n)
    A0 = np.sqrt([P, P, 0.0, 0.0]).astype(np.complex128)
    r = gpu.simulation.run_batch_transfer(cfg, gamma=g, alpha=0.0, delta_beta=[db], A0=A0, waves=(0, 1, 2, 3))
    ss = gpu.small_signal
    rr = 2 * g * P
    g2 = rr ** 2 - kappa ** 2 / 4
    s2 = np.sinh(np.sqrt(g2) * L_) ** 2 / g2 if g2 > 0 else np.sin(np.sqrt(-g2) * L_) ** 2 / -g2
    mu2 = 1 + rr ** 2 * s2
    mu, nu = ss.mu_nu(r["jac"][0], r["columns"], 2, 2)
    mi, ni = ss.mu_nu(r["jac"][0], r["columns"], 3, 2)
    assert abs(abs(mu) ** 2 / mu2 - 1) <= 1e-8 and abs(nu) ** 2 <= 1e-8 * mu2
    assert abs(abs(ni) ** 2 / (mu2 - 1) - 1) <= 1e-8 and abs(mi) ** 2 <= 1e-8 * mu2
    J = r["jac"][0]
    assert abs(np.linalg.det(J[4:, 4:]) - 1.0) <= 1e-9
    a = 2e-4
    r = gpu.simulation.run_batch_transfer(cfg, gamma=g, alpha=a, delta_beta=[db], A0=A0, waves=(0, 1, 2, 3))
    J = r["jac"][0]
    assert abs(np.linalg.det(J[4:, 4:]) / np.exp(-2 * a * L_) - 1.0) <= 1e-9
    assert abs(np.linalg.det(J) / np.exp(-4 * a * L_) - 1.0) <= 1e-6


def test_phase_gain_matches_the_phase_sweep_at_small_seeds(gpu, golden):
    kw = _sweep_kw(gpu, golden, n1=3, n3=12, wide=False, z_max=40.0, save_every=10, alpha=1e-4)
    pumps = [0.3, 0.2, 0.0, 0.0]
    ax = np.linspace(0.0, 2 * np.pi, 16, endpoint=False)
    kw_t = dict(kw, p_in=pumps, phase_in=[0.1, -0.2, 0.0, 0.0])
    r = gpu.scan_mismtach.sweep_transfer_2d(**kw_t)
    seeds = [0.3, 0.2, 1e-12, 1e-12]
    pg = gpu.small_signal.phase_gain(r["jac"], r["columns"], seeds, [0.1, -0.2, 0.0, 0.0], ax)
    kw_p = dict(kw, p_in=seeds, phase_in=[0.1, -0.2, 0.0, 0.0])
    ref = gpu.scan_mismtach.sweep_phase_gain_2d(phase_axis=ax, gain_metric="end", gain_unit="linear", **kw_p)
    assert ref["n_steps"] % 10 == 0
    assert np.nanmax(np.abs(pg["gain_lin"] / ref["gain_lin"] - 1)) <= 1e-6
    assert np.nanmin(ref["gain_lin"]) < 1.0                    # de-amplified phases are covered
    assert np.array_equal(pg["n_finite"], ref["n_finite"])


def test_pump_power_sensitivity_matches_the_batch_integrator(gpu):
    cfg = gpu.config.custom_simulation_config(z_max=300.0, dz=0.25, save_every=1200)
    p_in = np.array([0.1, 0.1, 1e-7, 1e-7])
    db = [-0.0005, 0.0, 0.001, 0.003]
    r = gpu.simulation.run_batch_transfer(cfg, gamma=11.5e-3, alpha=1e-4, delta_beta=db, p_in=p_in,
                                          waves=(0, 1, 2, 3))
    A0 = gpu.simulation.make_initial_amplitudes(p_in)
    for pump in (0, 1, (0, 1)):
        sens = gpu.small_signal.pump_power_sensitivity(r["jac"], r["columns"], A0, r["A_end"], pump)
        P3 = []
        for f in (1 + 1e-6, 1 - 1e-6):
            p = p_in.copy()
            p[list(np.atleast_1d(pump))] *= f
            e = gpu.simulation.run_batch_simulation(cfg, gamma=11.5e-3, alpha=1e-4, delta_beta=db, p_in=p,
                                                    outputs=("end",))["A_end"]
            P3.append(np.abs(e[:, 2]) ** 2)
        fd = (P3[0] - P3[1]) / (2e-6 * np.abs(r["A_end"][:, 2]) ** 2)
        assert np.max(np.abs(sens / fd - 1)) <= 1e-5, pump
