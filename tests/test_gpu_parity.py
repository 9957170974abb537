"""GPU: parity of the CUDA path (through the C ABI) with the reference.

Three anchors: (1) golden vectors produced by the live reference (tests/golden/), (2) the CPU
oracle on seeded inputs at sizes it finishes in seconds, (3) size-independent properties at
BASELINE's full sizes.  Tolerance (north star): 1e-10 relative on |A|^2 at fiber output; the
Delta-beta table 1e-12 relative (it is evaluated without FMA contraction in the reference's
operation order); trace samples 1e-10 relative to the largest power of the run.
"""
import numpy as np
import pytest

from conftest import rel_err

pytestmark = pytest.mark.gpu
TOL = 1e-10
# beta_6 .. beta_12 [s^n/m] about 1552 nm, orders 5, 9 and 11 zero: each order adds ~1e-2 1/m to Delta-beta
# (beta_n * dw^n / n! with dw = 4e13 rad/s), far from underflow (beta_12 * dw^12 > 1e-30 for dw >= 1e11)
TAYLOR_HIGH = {6: 1.8e-81, 7: -3.1e-94, 8: 6.2e-107, 10: -3.5e-132, 12: 2.9e-157}
EVEN_12 = (2, 4, 6, 8, 10, 12)


def _disp(fpa, b2, b3, b4, wref):
    return fpa.dispersion.DispersionParams(omega_ref=wref, beta2=b2, beta3=b3, beta4=b4)


# ------------------------------------------------------------------ RHS and single steps
def test_rhs_matches_oracle(gpu, oracle):
    rng = np.random.default_rng(11)
    B = 512
    A = rng.normal(size=(B, 4)) + 1j * rng.normal(size=(B, 4))
    z, g = rng.uniform(0, 1000, B), rng.uniform(1e-3, 12, B)
    a, db = rng.uniform(0, 1e-3, B) * (rng.random(B) < 0.5), rng.normal(size=B) * 0.05
    got = gpu._device.yaman4_rhs(z, A, g, a, db)
    ref = np.array([oracle.yaman_rhs(z[i], A[i], g[i], a[i], db[i]) for i in range(B)])
    assert np.max(np.abs(got - ref) / np.max(np.abs(ref), axis=1, keepdims=True)) < 1e-14
    # through the reference-named callable, with a ModelParams-like object
    P = gpu.parameters
    mp = P.make_model_params(waves=P.WavesParams.from_wavelengths(1550e-9, 1560e-9, 1555e-9),
                             fiber=P.FiberParams(length_m=1.0, gamma_W_m=g[0], alpha_1_m=a[0]),
                             grid=P.SimulationGrid(dz_m=0.1))
    mp.cache.set_phase_mismatch(db[0])
    one = gpu.yaman_model.rhs_yaman_simplified(z[0], A[0], mp)
    assert one.shape == (4,) and one.dtype == np.complex128 and np.array_equal(one, got[0])
    with pytest.raises(ValueError):
        gpu.yaman_model.rhs_yaman_simplified(0.0, np.ones(3), mp)


def test_rk4_step_matches_oracle(gpu, oracle):
    P = gpu.parameters
    rng = np.random.default_rng(12)
    for _ in range(8):
        A = rng.normal(size=4) + 1j * rng.normal(size=4)
        g, a, db, z, h = rng.uniform(0.01, 5), rng.uniform(0, 1e-3), rng.normal() * 0.1, rng.uniform(0, 64), 0.125
        mp = P.make_model_params(waves=P.WavesParams(omega=np.full(4, 1.2e15)),
                                 fiber=P.FiberParams(length_m=1.0, gamma_W_m=g, alpha_1_m=a),
                                 grid=P.SimulationGrid(dz_m=h))
        mp.cache.set_phase_mismatch(db)
        got = gpu.integrators.rk4_step(gpu.yaman_model.rhs_yaman_simplified, z, A, h, mp)
        ref = oracle.rk4_advance(oracle.yaman_rhs_p, z, A, h, oracle.YamanPoint(g, a, db))
        assert rel_err(got, ref) < 1e-13


# ------------------------------------------------------------------ reference integrator tests, on device
def test_reference_integrator_tests_replayed(gpu):
    """tests.py:146-226 of the reference: y' = y on a real state of dimension 1."""
    I = gpu.integrators
    f = I.LinearRHS(1.0)
    y1 = I.rk4_step(f, 0.0, np.array([1.0]), 0.1, None)
    assert y1.shape == (1,) and np.allclose(y1, np.exp(0.1), rtol=1e-7)
    z, y = I.integrate_interval(f, 1.0, 0.1, np.array([1.0]), None, save_every=2)
    assert z.shape == (6,) and y.shape == (6, 1) and y.dtype == np.float64
    assert np.allclose(z, [0.0, 0.2, 0.4, 0.6, 0.8, 1.0], atol=1e-15)
    assert np.allclose(y[:, 0], np.exp(z), atol=3e-6)
    z, y = I.integrate_fixed_step(f, np.linspace(0, 1, 11), np.array([1.0]), None)
    assert z.shape == (11,) and np.allclose(y[:, 0], np.exp(z), atol=3e-6)
    # Q1: effective step is z_max/round(z_max/dz); end state not saved when n % save_every != 0
    z, y = I.integrate_interval(f, 1.0, 0.3, np.array([1.0]), None)
    assert z.size == 4 and z[-1] == 1.0
    z, y = I.integrate_interval(f, 1.0, 0.1, np.array([1.0]), None, save_every=3)
    assert z.size == 4 and abs(z[-1] - 0.9) < 1e-15
    # NaN RHS -> FloatingPointError with the reference's text; NaNs returned when check is off
    nan_rhs = I.LinearRHS(float("nan"))
    with pytest.raises(FloatingPointError, match=r"NaN or Inf detected at step 0, z = 0.0"):
        I.integrate_interval(nan_rhs, 1.0, 0.5, np.array([1.0]), None, check_nan=True)
    z, y = I.integrate_interval(nan_rhs, 1.0, 0.5, np.array([1.0]), None, check_nan=False)
    assert y[0, 0] == 1.0 and np.isnan(y[1:]).all()
    # complex lambda, several components, against the exact exponential
    lam = np.array([-0.3 + 2j, 0.1j, -1.0])
    z, y = I.integrate_interval(I.LinearRHS(lam), 2.0, 0.01, np.array([1.0 + 0j, 2.0, -1j]), None, save_every=50)
    assert y.dtype == np.complex128
    assert np.allclose(y, np.array([1.0, 2.0, -1j]) * np.exp(np.outer(z, lam)), rtol=1e-8)


def test_overflow_detected_at_the_reference_step(gpu, oracle):
    """A run that blows up: the first non-finite step index and message match the oracle's."""
    P = gpu.parameters
    mp = P.make_model_params(waves=P.WavesParams(omega=np.full(4, 1.2e15)),
                             fiber=P.FiberParams(length_m=1.0, gamma_W_m=5.0), grid=P.SimulationGrid(dz_m=0.1))
    mp.cache.set_phase_mismatch(0.0)
    A0 = np.array([1e60, 1e60, 1e10, 0], dtype=complex)
    with pytest.raises(FloatingPointError) as ref:
        oracle.march_interval(oracle.yaman_rhs_p, 1.0, 0.125, A0, oracle.YamanPoint(5.0, 0.0, 0.0))
    with pytest.raises(FloatingPointError) as got:
        gpu.integrators.integrate_interval(gpu.yaman_model.rhs_yaman_simplified, 1.0, 0.125, A0, mp)
    assert str(got.value) == str(ref.value)


# ------------------------------------------------------------------ golden single runs
def _check_trace(A, A_ref, tol=TOL):
    P, P_ref = np.abs(A) ** 2, np.abs(A_ref) ** 2
    assert A.shape == A_ref.shape
    assert rel_err(P[-1][P_ref[-1] > 0], P_ref[-1][P_ref[-1] > 0]) < tol      # north-star metric
    assert np.max(np.abs(P - P_ref)) / np.max(P_ref) < tol
    assert np.max(np.abs(A - A_ref)) / np.max(np.abs(A_ref)) < tol


def test_golden_b1_main_single_run(gpu, golden):
    fp, sim = gpu.frequency_plan, gpu.simulation
    om = fp.plan_from_wavelengths(1550e-9, 1560e-9, 1555e-9)
    disp = _disp(gpu, *golden["b1_beta"], golden["b1_sym"][0])
    cfg = gpu.config.custom_simulation_config(z_max=1000.0, dz=0.1, save_every=10)
    gamma, alpha = golden["b1_gamma_alpha"]
    z, A = sim.run_single_simulation(cfg, gamma=gamma, alpha=alpha, omega=om, p_in=golden["b1_p_in"],
                                     dispersion=disp, length_unit="m")
    assert np.array_equal(z, golden["b1_z"])
    _check_trace(A, golden["b1_A"])
    # per-sample relative error on the signal (45 dB of gain across the trace)
    assert rel_err(np.abs(A[:, 2]) ** 2, np.abs(golden["b1_A"][:, 2]) ** 2) < TOL
    # exact-phase mode (sincos at every abscissa) agrees too
    r = sim.run_batch_simulation(cfg, gamma=gamma, alpha=alpha, delta_beta=[golden["b1_dbeta"][1]],
                                 p_in=golden["b1_p_in"], outputs=("trace", "end", "pmax"), phase_exact=True)
    _check_trace(r["A_trace"][0], golden["b1_A"])
    assert np.array_equal(r["A_end"][0], r["A_trace"][0, -1])
    assert rel_err(r["Pmax"][0], (np.abs(r["A_trace"][0]) ** 2).max(axis=0)) < 1e-15
    assert np.array_equal(r["z"], golden["b1_z"])


def test_golden_b2_b3_examples(gpu, golden):
    z, A = gpu.simulation.example_zero_signal()
    assert A.shape == (51, 4) and z[-1] == 0.5 and np.all(A[:, 2:] == 0)       # tests.py:318-323
    assert np.allclose(z, golden["b2_z"], rtol=0, atol=1e-15)
    assert rel_err(A[:, :2], golden["b2_A"][:, :2]) < TOL
    z, A = gpu.simulation.custom_seeded_signal()
    assert A.shape == (501, 4)
    _check_trace(A, golden["b3_A"])


def test_golden_random_runs(gpu, golden):
    fp, sim, pm = gpu.frequency_plan, gpu.simulation, gpu.phase_matching
    for row, A_last, P_max in zip(golden["rand_in"], golden["rand_A_last"], golden["rand_P_max"]):
        l1, l2, l3, b2, b3, b4, wref, mi, prov, zmax, dz, se, g_, a_ = row[:14]
        p, ph, n_saved, z_last = row[14:18], row[18:22], int(row[22]), row[23]
        method = ("general_taylor", "symmetric_even", "provided")[int(mi)]
        pmc = pm.PhaseMatchingConfig(method=method, provided_delta_beta=prov if method == "provided" else None)
        cfg = gpu.config.custom_simulation_config(z_max=zmax, dz=dz, save_every=int(se))
        z, A = sim.run_single_simulation(cfg, gamma=g_, alpha=a_, omega=fp.plan_from_wavelengths(l1, l2, l3),
                                         p_in=p, phase_in=ph, dispersion=_disp(gpu, b2, b3, b4, wref),
                                         phase_matching_cfg=pmc)
        assert z.size == n_saved and z[-1] == z_last
        assert rel_err(np.abs(A[-1]) ** 2, np.abs(A_last) ** 2) < TOL
        assert rel_err(A[-1], A_last) < TOL
        assert rel_err((np.abs(A) ** 2).max(axis=0), P_max) < TOL


def test_explicit_grid_and_units_vs_oracle(gpu, oracle):
    """integrate_fixed_step on a NON-uniform grid, and a km-unit run, against the oracle."""
    P = gpu.parameters
    rng = np.random.default_rng(21)
    grid = np.concatenate(([0.0], np.cumsum(rng.uniform(0.05, 0.4, 300))))
    mp = P.make_model_params(waves=P.WavesParams(omega=np.full(4, 1.2e15)),
                             fiber=P.FiberParams(length_m=grid[-1], gamma_W_m=0.02, alpha_1_m=3e-4),
                             grid=P.SimulationGrid(dz_m=0.1))
    mp.cache.set_phase_mismatch(-0.03)
    A0 = oracle.initial_amplitudes([0.3, 0.5, 1e-4, 1e-6], [0.0, 0.4, -1.0, 2.0])
    z, A = gpu.integrators.integrate_fixed_step(gpu.yaman_model.rhs_yaman_simplified, grid, A0, mp, save_every=7)
    z_ref, A_ref = oracle.march_grid(oracle.yaman_rhs_p, grid, A0, oracle.YamanPoint(0.02, 3e-4, -0.03), save_every=7)
    assert np.array_equal(z, z_ref)
    _check_trace(A, A_ref)
    # km units with dispersion given per km
    fp = gpu.frequency_plan
    om = fp.plan_from_wavelengths(1550e-9, 1559e-9, 1553e-9)
    disp_km = gpu.dispersion.DispersionParams(omega_ref=0.5 * (om[0] + om[1]), beta2=-2.5e-26, beta3=3e-38, beta4=-1.6e-52)
    cfg = gpu.config.custom_simulation_config(z_max=0.2, dz=2.5e-4, save_every=16)
    for method in ("general_taylor", "symmetric_even"):
        z, A = gpu.simulation.run_single_simulation(
            cfg, gamma=11.5, alpha=0.2, omega=om, p_in=[0.4, 0.4, 1e-6, 0.0], dispersion=disp_km,
            phase_matching_cfg=gpu.phase_matching.PhaseMatchingConfig(method=method), length_unit="km")
        z_ref, A_ref, _ = oracle.single_run(
            z_max=0.2, dz=2.5e-4, save_every=16, check_nan=True, gamma=11.5, alpha=0.2, omega=om,
            p_in=[0.4, 0.4, 1e-6, 0.0], disp=oracle.Taylor(disp_km.omega_ref, 0, 0, -2.5e-26, 3e-38, -1.6e-52),
            method=method, length_unit="km")
        assert np.array_equal(z, z_ref)
        _check_trace(A, A_ref)


# ------------------------------------------------------------------ sweeps
def test_golden_b4_main_sweep(gpu, golden):
    """`python main.py` default: 30-point lambda3 sweep (main.py:206-279)."""
    b2, b3, b4, wref = golden["b4_beta"]
    cfg = gpu.config.custom_simulation_config(z_max=500.0, dz=0.2, save_every=10)
    kw = dict(cfg=cfg, lambda_p1_m=1550e-9, lambda_p2_m=1558e-9, lambda_signal_m=golden["b4_lam"], gamma=11.5e-3,
              alpha=float(golden["b4_alpha"][0]), p_in=golden["b4_p_in"], dispersion=_disp(gpu, b2, b3, b4, wref),
              show=False, show_progress=False)
    x, g, d = gpu.scan_mismtach.plot_max_gain_and_dbeta_vs_lambda_signal(**kw)
    assert np.array_equal(x, golden["b4_x"]) and not np.isnan(g).any()
    assert rel_err(d, golden["b4_dbeta"]) < 1e-12
    lin, lin_ref = 10 ** (g / 10), 10 ** (golden["b4_gain_db"] / 10)
    assert rel_err(lin, lin_ref) < TOL
    assert g[0] == golden["b4_gain_db"][0] == 9.643274665532869e-16          # quirk Q6, bit for bit
    x2, g2 = gpu.scan_mismtach.plot_max_signal_gain_vs_lambda_signal(
        **kw, phase_matching_cfg=gpu.phase_matching.PhaseMatchingConfig(method="general_taylor"), gain_unit="linear")
    assert rel_err(g2, golden["b4_gain_lin_general"]) < TOL


def test_best_point_rerun_with_trace(gpu, golden):
    """Reduce-mode sweep -> peak -> full trace of the best point: the trace's max equals the sweep's gain."""
    b2, b3, b4, wref = golden["b4_beta"]
    cfg = gpu.config.custom_simulation_config(z_max=500.0, dz=0.2, save_every=10)
    kw = dict(cfg=cfg, lambda_p1_m=1550e-9, lambda_p2_m=1558e-9, gamma=11.5e-3, alpha=float(golden["b4_alpha"][0]),
              p_in=golden["b4_p_in"], dispersion=_disp(gpu, b2, b3, b4, wref))
    x, g, d = gpu.scan_mismtach.plot_max_gain_and_dbeta_vs_lambda_signal(
        lambda_signal_m=golden["b4_lam"], gain_unit="linear", show=False, **kw)
    pk = gpu.scan_mismtach.sweep_peak(x, g)
    assert pk["index"] == int(np.nanargmax(golden["b4_gain_db"]))
    z, A = gpu.scan_mismtach.rerun_point_with_trace(lambda_signal_m=golden["b4_lam"][pk["index"]], **kw)
    assert A.shape == (251, 4) and z[-1] == 500.0
    assert rel_err((np.abs(A[:, 2]) ** 2).max() / golden["b4_p_in"][2], pk["gain"]) < 1e-12


def test_dbeta_only_sweep(gpu, oracle, golden):
    """plot_dbeta_vs_lambda_signal: the reference's helper convention (minus the project dbeta)."""
    b2, b3, b4, wref = golden["b4_beta"]
    lam3 = np.concatenate((golden["b4_lam"], [3e-7]))
    x, d = gpu.scan_mismtach.plot_dbeta_vs_lambda_signal(
        gamma=11.5e-3, lambda_p1_m=1550e-9, lambda_p2_m=1558e-9, lambda_signal_m=lam3, p_in=golden["b4_p_in"],
        dispersion=_disp(gpu, b2, b3, b4, wref), show=False)
    ref = [-oracle.phase_mismatch(oracle.plan_from_wavelengths(1550e-9, 1558e-9, l), oracle.Taylor(wref, 0, 0, b2, b3, b4),
                                  oracle.GENERAL_TAYLOR) for l in golden["b4_lam"]]
    assert np.array_equal(x[:-1], golden["b4_x"]) and np.isnan(d[-1])
    assert rel_err(d[:-1], ref) < 1e-12


def test_golden_config4_grid_nan_semantics(gpu, golden):
    b2, b3, b4, wref = golden["b4_beta"]
    cfg = gpu.config.custom_simulation_config(z_max=500.0, dz=0.2, save_every=10)
    r = gpu.scan_mismtach.sweep_gain_2d(
        cfg=cfg, lambda_p1_m=golden["c4_lam1"], lambda_p2_m=1558e-9, lambda_signal_m=golden["c4_lam3"],
        gamma=11.5e-3, alpha=float(golden["b4_alpha"][0]), p_in=golden["b4_p_in"],
        dispersion=_disp(gpu, b2, b3, b4, wref),
        phase_matching_cfg=gpu.phase_matching.PhaseMatchingConfig(method="general_taylor"), gain_unit="linear")
    G, D = golden["c4_gain_lin"], golden["c4_dbeta"]
    assert np.array_equal(np.isnan(r["gain"]), np.isnan(G)) and np.isnan(G[:, -1]).all()
    assert np.array_equal(np.isnan(r["dbeta"]), np.isnan(D))
    ok = ~np.isnan(G)
    assert rel_err(r["gain"][ok], G[ok]) < TOL and rel_err(r["dbeta"][ok], D[ok]) < 1e-12
    assert (r["valid"][:, -1] == 0).all() and (r["valid"][:, :-1] == 1).all()
    # a config the reference rejects inside its per-point try -> every gain NaN, dbeta still reported
    bad = gpu.config.custom_simulation_config(z_max=1.0, dz=2.0)
    rb = gpu.scan_mismtach.sweep_gain_2d(
        cfg=bad, lambda_p1_m=golden["c4_lam1"], lambda_p2_m=1558e-9, lambda_signal_m=golden["c4_lam3"],
        gamma=11.5e-3, alpha=0.0, p_in=golden["b4_p_in"], dispersion=_disp(gpu, b2, b3, b4, wref),
        phase_matching_cfg=gpu.phase_matching.PhaseMatchingConfig(method="general_taylor"))
    assert np.isnan(rb["gain"]).all() and rel_err(rb["dbeta"][ok], D[ok]) < 1e-12


def test_golden_config3_dbeta_sweep(gpu, golden):
    cfg = gpu.config.custom_simulation_config(z_max=0.5, dz=1e-3, save_every=10)
    for mode, key in (("end", "c3_P_end"), ("max", "c3_P_max")):
        r = gpu.scan_mismtach.sweep_dbeta_gain(cfg=cfg, delta_beta=golden["c3_dbeta"], gamma=10.0, alpha=0.0,
                                               p_in=[0.1, 0.1, 1e-5, 0.0], length_unit="km", gain_mode=mode)
        ref = golden[key]
        assert rel_err(r["Gs"], ref[:, 2] / (1e-5 + 1e-30)) < TOL
        assert np.max(np.abs(r["Gi"] - ref[:, 3] / (1e-5 + 1e-30))) < TOL * np.max(ref[:, 3] / 1e-5)
        assert (r["status"] == -1).all()
    d, Gs, Gi = gpu.scan_mismtach.scan_mismatch_seeded_signal("max", n_points=9, verbose=False)
    assert np.array_equal(d, golden["c3_dbeta"]) and rel_err(Gs, golden["c3_P_max"][:, 2] / 1e-5) < TOL


def test_dbeta_table_vs_oracle_all_methods(gpu, oracle):
    """The device front-end against the per-point oracle on a 2-D grid incl. invalid points.
    (a) beta0 = beta1 = 0: agreement 1e-12 on the scale of the Taylor terms and >= 90 % of the
    entries bit-equal; (b) beta0 ~ 6e6, beta1 ~ 5e-9 (general Taylor cancels 10 digits): within
    8 ulp of the largest beta(omega).  Up to the supported Taylor order 12: every order from 6 on
    adds ~1e-2 1/m at the 90th percentile of the grid (1e16 at the far outliers), orders 5, 9 and 11
    are zero."""
    rng = np.random.default_rng(31)
    lam1 = rng.uniform(1540e-9, 1560e-9, 7)
    lam2 = rng.uniform(1540e-9, 1560e-9, 7)
    lam3 = np.concatenate((rng.uniform(1500e-9, 1600e-9, 40), [700e-9, 780e-9, 3e-6]))
    wref = oracle.omega_from_lambda(1552e-9)
    PM = gpu.phase_matching.PhaseMatchingConfig
    low, high = {6: 2e-85}, TAYLOR_HIGH
    cases = ((PM(method="general_taylor", max_order=6), oracle.GENERAL_TAYLOR, dict(max_order=6), low),
             (PM(method="general_taylor", max_order=3), oracle.GENERAL_TAYLOR, dict(max_order=3), low),
             (PM(method="symmetric_even", even_orders=(2, 4, 6)), oracle.SYMMETRIC_EVEN, dict(even_orders=(2, 4, 6)),
              low),
             (PM(method="provided", provided_delta_beta=0.125), oracle.PROVIDED, dict(provided=0.125), low),
             (PM(method="general_taylor", max_order=12), oracle.GENERAL_TAYLOR, dict(max_order=12), high),
             (PM(method="symmetric_even", even_orders=EVEN_12), oracle.SYMMETRIC_EVEN, dict(even_orders=EVEN_12), high))
    for b0, b1, abs_tol in ((0.0, 0.0, None), (5.8e6, 4.9e-9, 8 * np.spacing(5.9e6))):
        for cfg, ometh, okw, extra in cases:
            disp = gpu.dispersion.DispersionParams(omega_ref=wref, beta0=b0, beta1=b1, beta2=-2.6e-29, beta3=3.3e-41,
                                                   beta4=-1.6e-55, extra=extra)
            odisp = oracle.Taylor(wref, b0, b1, -2.6e-29, 3.3e-41, -1.6e-55, extra=extra)
            plan, keep = gpu._device.new_plan_desc(lam1, lam2, lam3)
            gpu.phase_matching.fill_plan_desc(plan, disp, cfg)
            out = gpu._device.dbeta_table(plan, want_omega=True)
            n_bad = n_ok = n_equal = 0
            for i in range(lam1.size):
                for j in range(lam3.size):
                    try:
                        om = oracle.plan_from_wavelengths(lam1[i], lam2[i], lam3[j])
                        ref = oracle.phase_mismatch(om, odisp, ometh, **okw)
                    except ValueError:
                        assert out["valid"][i, j] == 0 and np.isnan(out["dbeta"][i, j])
                        n_bad += 1
                        continue
                    assert out["valid"][i, j] == 1
                    assert np.array_equal(out["omega"][i, j], om)               # omegas bit-exact
                    got = out["dbeta"][i, j]
                    n_ok += 1
                    n_equal += int(got == ref)
                    if abs_tol is None or ometh != oracle.GENERAL_TAYLOR:
                        assert abs(got - ref) <= 1e-12 * max(abs(ref), 1e-3)
                    elif extra is low:
                        assert abs(got - ref) <= abs_tol
                    else:   # the high orders make beta(omega) of the far outliers ~1e16: 8 ulp of that point's largest
                        big = max(abs(oracle.beta_taylor(w, odisp, okw["max_order"])) for w in om)
                        assert abs(got - ref) <= max(abs_tol, 8 * np.spacing(big))
            assert n_bad >= 7
            if abs_tol is None:
                assert n_equal >= 0.9 * n_ok, f"only {n_equal}/{n_ok} dbeta entries bit-equal"


@pytest.mark.parametrize("unit", ["m", "km"])
def test_sweep_at_taylor_order_12_vs_oracle(gpu, oracle, unit):
    """The fused sweep with general Taylor to order 12 (the same coefficients as above): the reported dbeta uses
    beta_n as given, the integration beta_n / 1000 in km -- every coefficient of the table is rescaled.  Order 12
    moves the gain of the outer signal wavelengths by up to 1 %."""
    s = 1.0 if unit == "m" else 1e3
    wref = oracle.omega_from_lambda(1552e-9)
    lam1, lam3 = np.array([1549e-9, 1551e-9]), np.linspace(1500e-9, 1600e-9, 7)
    extra = {n: v * s for n, v in TAYLOR_HIGH.items()}
    disp = gpu.dispersion.DispersionParams(omega_ref=wref, beta2=-2.6e-29 * s, beta3=3.3e-41 * s, beta4=-1.6e-55 * s,
                                           extra=extra)
    odisp = oracle.Taylor(wref, 0.0, 0.0, -2.6e-29 * s, 3.3e-41 * s, -1.6e-55 * s, extra=extra)
    p_in = [0.3, 0.3, 1e-4, 0.0]
    cfg = gpu.config.custom_simulation_config(z_max=300.0 / s, dz=1.0 / s, save_every=10)
    r = gpu.scan_mismtach.sweep_gain_2d(
        cfg=cfg, lambda_p1_m=lam1, lambda_p2_m=1558e-9, lambda_signal_m=lam3, gamma=11.5e-3 * s, alpha=2e-4 * s,
        p_in=p_in, dispersion=disp, length_unit=unit, gain_unit="linear",
        phase_matching_cfg=gpu.phase_matching.PhaseMatchingConfig(method="general_taylor", max_order=12))
    for i in range(lam1.size):
        g_ref, d_ref = oracle.sweep_lambda3_gain(
            lam1=lam1[i], lam2=1558e-9, lam3_arr=lam3, z_max=300.0 / s, dz=1.0 / s, save_every=10, check_nan=True,
            gamma=11.5e-3 * s, alpha=2e-4 * s, p_in=p_in, disp=odisp, method=oracle.GENERAL_TAYLOR, max_order=12,
            length_unit=unit, gain_unit="linear")
        assert np.isfinite(g_ref).all()
        assert rel_err(r["gain"][i], g_ref) < TOL
        assert np.max(np.abs(r["dbeta"][i] - d_ref)) <= 1e-12 * np.max(np.abs(d_ref))


# ------------------------------------------------------------------ properties at full size
def test_full_size_partition_invariance_and_symmetry(gpu):
    """BASELINE config 3 at full size (1e5 points x 500 steps): any partition of the batch gives
    bit-identical results (points are independent); exact-phase and recurrence modes agree to
    1e-11; with alpha = 0 and equal pumps the invariants P1-P2 and P3-P4 hold."""
    cfg = gpu.config.custom_simulation_config(z_max=0.5, dz=1e-3, save_every=10)
    db = np.linspace(-40.0, 40.0, 100_000)
    run = lambda d, **kw: gpu.simulation.run_batch_simulation(          # noqa: E731
        cfg, gamma=10.0, alpha=0.0, delta_beta=d, p_in=[0.1, 0.1, 1e-5, 0.0], length_unit="km", **kw)
    full = run(db)
    parts = [run(db[a:b]) for a, b in ((0, 12_345), (12_345, 50_001), (50_001, 100_000))]
    for key in ("A_end", "Pmax", "status"):
        assert np.array_equal(full[key], np.concatenate([p[key] for p in parts]))
    assert (full["status"] == -1).all()
    exact = run(db[::97], phase_exact=True)
    assert rel_err(np.abs(exact["A_end"]) ** 2, np.abs(full["A_end"][::97]) ** 2) < 1e-11
    P = np.abs(full["A_end"]) ** 2
    assert np.max(np.abs(P[:, 0] - P[:, 1])) < 1e-15
    assert np.max(np.abs((P[:, 2] - P[:, 3]) - 1e-5)) < 1e-15
    assert np.max(np.abs(P.sum(axis=1) - (0.2 + 1e-5))) < 1e-13
    # mirror symmetry of the physics is NOT exact (Kerr shifts the peak): the peak sits at
    # dbeta = -gamma (P1 + P2) = -2 /km; check the location instead
    peak = db[np.argmax(full["Pmax"][:, 2])]
    assert abs(peak + 2.0) < 0.5


def test_full_size_2d_sweep_rows_equal_1d_sweeps(gpu, golden):
    """BASELINE config 4 shape (1000 x 1000 grid; shortened fiber so the test stays fast): rows of
    the 2-D launch are bit-identical to independent 1-D launches, and the gain is NaN exactly
    where the plan is invalid."""
    b2, b3, b4, wref = golden["b4_beta"]
    cfg = gpu.config.custom_simulation_config(z_max=20.0, dz=0.2, save_every=10)
    lam1 = np.linspace(1545e-9, 1555e-9, 1000)
    lam3 = np.linspace(1540e-9, 1565e-9, 1000)
    kw = dict(cfg=cfg, lambda_p2_m=1558e-9, gamma=11.5e-3, alpha=float(golden["b4_alpha"][0]),
              p_in=golden["b4_p_in"], dispersion=_disp(gpu, b2, b3, b4, wref), gain_unit="linear")
    full = gpu.scan_mismtach.sweep_gain_2d(lambda_p1_m=lam1, lambda_signal_m=lam3, **kw)
    assert full["gain"].shape == (1000, 1000) and not np.isnan(full["gain"]).any()
    for i in (0, 137, 999):
        row = gpu.scan_mismtach.sweep_gain_2d(lambda_p1_m=[lam1[i]], lambda_signal_m=lam3, **kw)
        assert np.array_equal(row["gain"][0], full["gain"][i]) and np.array_equal(row["dbeta"][0], full["dbeta"][i])
    assert (full["gain"] >= 1.0 - 1e-12).all()
