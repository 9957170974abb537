"""GPU: edge cases of the C-ABI entry points -- empty and ragged batches, degenerate step counts,
per-point versus broadcast physics, invalid points inside a batch, long runs."""
import numpy as np
import pytest

from conftest import rel_err

pytestmark = pytest.mark.gpu


def _A0(oracle, p=(0.3, 0.4, 1e-5, 1e-6), ph=None):
    return oracle.initial_amplitudes(list(p), ph)


def test_empty_batches(gpu, oracle):
    D = gpu._device
    r = D.yaman4_batch(np.zeros(0), 0.01, 0.0, _A0(oracle), z_max=1.0, n_steps=10, trace=True, pmax=True)
    assert r["A_trace"].shape == (0, 11, 4) and r["A_end"].shape == (0, 4) and r["status"].shape == (0,)
    assert D.yaman4_rhs(np.zeros(0), np.zeros((0, 4)), np.zeros(0), np.zeros(0), np.zeros(0)).shape == (0, 4)
    cfg = gpu.config.custom_simulation_config(z_max=10.0, dz=0.1)
    disp = gpu.dispersion.DispersionParams(1.2e15, beta2=-1e-28)
    r = gpu.scan_mismtach.sweep_gain_2d(cfg=cfg, lambda_p1_m=np.zeros(0), lambda_p2_m=1558e-9,
                                        lambda_signal_m=[1554e-9], gamma=0.01, alpha=0.0,
                                        p_in=[0.1, 0.1, 1e-6, 0.0], dispersion=disp)
    assert r["gain"].shape == (0, 1) and r["dbeta"].shape == (0, 1)


def test_degenerate_step_counts(gpu, oracle):
    D = gpu._device
    A0 = _A0(oracle)
    pt = oracle.YamanPoint(0.02, 1e-4, 0.03)
    # one step; save_every larger than n_steps (only the initial sample is kept, integrators.py:115)
    for n_steps, save_every in ((1, 1), (7, 10), (10, 3), (9, 9)):
        r = D.yaman4_batch([0.03], 0.02, 1e-4, A0, z_max=2.0, n_steps=n_steps, save_every=save_every, trace=True,
                           pmax=True)
        z_ref, A_ref = oracle.march_grid(oracle.yaman_rhs_p, np.linspace(0.0, 2.0, n_steps + 1), A0, pt,
                                         save_every=save_every)
        assert r["A_trace"].shape == (1, n_steps // save_every + 1, 4) == (1,) + A_ref.shape
        assert np.max(np.abs(r["A_trace"][0] - A_ref)) < 1e-13
        # A_end is the state after the LAST step even when that step is not a saved sample
        z_all, A_all = oracle.march_grid(oracle.yaman_rhs_p, np.linspace(0.0, 2.0, n_steps + 1), A0, pt)
        assert np.max(np.abs(r["A_end"][0] - A_all[-1])) < 1e-13
        assert rel_err(r["Pmax"][0], (np.abs(A_ref) ** 2).max(axis=0)) < 1e-13
    with pytest.raises(ValueError):
        D.yaman4_batch([0.0], 0.02, 0.0, A0, z_max=1.0, n_steps=0)
    with pytest.raises(ValueError):
        D.yaman4_batch([0.0], 0.02, 0.0, A0, z_max=1.0, n_steps=4, save_every=0)


def test_per_point_physics_equals_broadcast_bit_for_bit(gpu, oracle):
    """gamma / alpha / A0 given per point (registers) or broadcast (constant bank): same bits, also for runs
    that start at z0 != 0 (dbeta*z0 up to ~50 rad), lossless and on the exact kernel; a ragged batch (not a
    multiple of the block size) with distinct physics per point matches the oracle."""
    D = gpu._device
    rng = np.random.default_rng(5)
    B = 301
    db = rng.normal(size=B) * 0.02
    A0 = _A0(oracle, ph=[0.2, -0.1, 0.5, 1.0])
    kw = dict(z_max=30.0, n_steps=150, save_every=7, pmax=True)
    for z0, alpha, exact in ((0.0, 2e-4, False), (5.0, 2e-4, False), (2000.0, 2e-4, False), (2000.0, 0.0, False),
                             (2000.0, 2e-4, True)):
        run = dict(kw, z0=z0, z_max=z0 + 30.0, trace=z0 != 0.0, phase_exact=exact)
        a = D.yaman4_batch(db, 0.015, alpha, A0, **run)
        b = D.yaman4_batch(db, np.full(B, 0.015), np.full(B, alpha), np.tile(A0, (B, 1)), **run)
        for k in a:
            assert np.array_equal(a[k], b[k]), (k, z0, alpha, exact)
    g = rng.uniform(0.005, 0.03, B)
    al = rng.uniform(0, 5e-4, B) * (rng.random(B) < 0.7)
    A0s = np.sqrt(rng.uniform(1e-6, 0.5, (B, 4))) * np.exp(1j * rng.uniform(-3, 3, (B, 4)))
    r = D.yaman4_batch(db, g, al, A0s, **kw)
    for i in (0, 77, 300):
        pt = oracle.YamanPoint(g[i], al[i], db[i])
        z, A = oracle.march_interval(oracle.yaman_rhs_p, 30.0, 0.2, A0s[i], pt, save_every=7)
        A_last = oracle.march_interval(oracle.yaman_rhs_p, 30.0, 0.2, A0s[i], pt)[1][-1]   # 150 % 7 != 0
        assert rel_err(r["A_end"][i], A_last) < 1e-11
        assert rel_err(r["Pmax"][i], (np.abs(A) ** 2).max(axis=0)) < 1e-11


def test_invalid_points_inside_a_batch(gpu, oracle):
    D = gpu._device
    db = np.array([0.01, np.nan, -0.02, np.inf, 0.0])
    for exact in (False, True):
        r = D.yaman4_batch(db, 0.02, 0.0, _A0(oracle), z_max=5.0, n_steps=50, save_every=10, trace=True, pmax=True,
                           phase_exact=exact)
        assert r["status"].tolist() == [-1, 0, -1, 0, -1]
        for i in (1, 3):
            assert np.array_equal(r["A_trace"][i, 0], _A0(oracle)) and np.isnan(r["A_trace"][i, 1:]).all()
            assert np.isnan(r["A_end"][i]).all() and np.isnan(r["Pmax"][i]).all()
        assert np.isfinite(r["A_trace"][[0, 2, 4]]).all()
    # check_nan off: same numbers, no status
    r = D.yaman4_batch(db, 0.02, 0.0, _A0(oracle), z_max=5.0, n_steps=50, check_nan=False)
    assert (r["status"] == -1).all() and np.isnan(r["A_end"][1]).all()


def test_sweep_with_per_row_second_pump_and_km_units(gpu, oracle):
    """lambda_p2 given per pump row; dispersion / gamma / alpha / lengths per km: reported dbeta per km,
    integration per metre (simulation.py:126-175, scan_mismtach.py:700-706)."""
    lam1 = np.array([1549e-9, 1550e-9, 1551e-9])
    lam2 = np.array([1559e-9, 1558e-9, 1557e-9])
    lam3 = np.linspace(1545e-9, 1562e-9, 6)
    wref = oracle.omega_from_lambda(1554e-9)
    disp_km = gpu.dispersion.DispersionParams(omega_ref=wref, beta2=-1.2e-25, beta3=3.3e-38, beta4=-1.6e-52)
    odisp = oracle.Taylor(wref, 0, 0, -1.2e-25, 3.3e-38, -1.6e-52)
    cfg = gpu.config.custom_simulation_config(z_max=0.3, dz=1e-3, save_every=10)
    for method, ometh in (("general_taylor", oracle.GENERAL_TAYLOR), ("symmetric_even", oracle.SYMMETRIC_EVEN)):
        r = gpu.scan_mismtach.sweep_gain_2d(
            cfg=cfg, lambda_p1_m=lam1, lambda_p2_m=lam2, lambda_signal_m=lam3, gamma=11.5, alpha=0.1,
            p_in=[0.2, 0.2, 1e-6, 0.0], dispersion=disp_km,
            phase_matching_cfg=gpu.phase_matching.PhaseMatchingConfig(method=method), length_unit="km",
            gain_unit="linear")
        for i in range(3):
            g_ref, d_ref = oracle.sweep_lambda3_gain(
                lam1=lam1[i], lam2=lam2[i], lam3_arr=lam3, z_max=0.3, dz=1e-3, save_every=10, check_nan=True,
                gamma=11.5, alpha=0.1, p_in=[0.2, 0.2, 1e-6, 0.0], disp=odisp, method=ometh, length_unit="km",
                gain_unit="linear")
            assert rel_err(r["gain"][i], g_ref) < 1e-10
            assert np.max(np.abs(r["dbeta"][i] - d_ref)) <= 1e-12 * np.max(np.abs(d_ref))


def test_long_single_run_keeps_phase_in_sync(gpu, oracle):
    """2e5 steps of one point: the phase recurrence (re-synchronised every 32 steps) against the exact
    kernel and, on a 2e4-step prefix, against the oracle."""
    D = gpu._device
    A0 = _A0(oracle, p=(0.5, 0.5, 1e-8, 1e-8))
    kw = dict(z_max=2000.0, n_steps=200_000, save_every=1000, trace=True, end=False)
    fast = D.yaman4_batch([4e-4], 11.5e-3, 2e-4, A0, **kw)["A_trace"][0]
    exact = D.yaman4_batch([4e-4], 11.5e-3, 2e-4, A0, phase_exact=True, **kw)["A_trace"][0]
    assert np.max(np.abs(fast - exact)) / np.max(np.abs(exact)) < 1e-10
    P, Pe = np.abs(fast) ** 2, np.abs(exact) ** 2
    assert rel_err(P[-1], Pe[-1]) < 1e-10
    z, A = oracle.march_interval(oracle.yaman_rhs_p, 200.0, 0.01, A0, oracle.YamanPoint(11.5e-3, 2e-4, 4e-4),
                                 save_every=1000)
    assert np.max(np.abs(fast[:21] - A)) / np.max(np.abs(A)) < 1e-11


def test_sweep_results_written_into_pinned_host_buffers(gpu, golden):
    """`fpa_yaman4_sweep_host` lets the kernel store into pinned result buffers (zero-copy); with
    pageable buffers it stages through device memory.  Same bits either way, NaN placement included."""
    b2, b3, b4, wref = golden["b4_beta"]
    disp = gpu.dispersion.DispersionParams(omega_ref=wref, beta2=b2, beta3=b3, beta4=b4)
    cfg = gpu.config.custom_simulation_config(z_max=30.0, dz=0.2, save_every=10)
    lam1 = np.linspace(1545e-9, 1555e-9, 37)
    lam3 = np.linspace(1400e-9, 1700e-9, 501)          # wide enough to hold invalid plans
    kw = dict(cfg=cfg, lambda_p1_m=lam1, lambda_signal_m=lam3, lambda_p2_m=1558e-9, gamma=11.5e-3, alpha=1e-4,
              p_in=golden["b4_p_in"], dispersion=disp, gain_unit="dB")
    plain = {k: np.full((37, 501), -9, dt) for k, dt in
             (("gain_lin", np.float64), ("dbeta", np.float64), ("valid", np.int32), ("status", np.int32))}
    pageable = gpu.scan_mismtach.sweep_gain_2d(out=plain, **kw)       # pageable memory: staged + copied
    default = gpu.scan_mismtach.sweep_gain_2d(**kw)                   # library-owned page-locked pool
    for k in ("gain", "gain_lin", "dbeta", "valid", "status"):
        assert np.array_equal(default[k], pageable[k], equal_nan=True), k
    bufs = {k: gpu._lib.pinned_empty((37, 501), dt) for k, dt in
            (("gain_lin", np.float64), ("dbeta", np.float64), ("valid", np.int32), ("status", np.int32))}
    for v in bufs.values():
        v.fill(-7)
    pinned = gpu.scan_mismtach.sweep_gain_2d(out=bufs, **kw)
    assert pinned["gain_lin"] is bufs["gain_lin"]
    for k in ("gain", "gain_lin", "dbeta", "valid", "status"):
        assert np.array_equal(pinned[k], pageable[k], equal_nan=True), k
    assert np.isfinite(pinned["gain"]).any()


@pytest.mark.parametrize("pinned", [False, True])
def test_multi_device_sweep_equals_single_device(gpu, golden, pinned):
    """`fpa_yaman4_sweep_multi_host`: pump rows split over devices from one process; same bits as one
    device for any split (ragged row counts, more devices than rows).  On a one-GPU box the device
    list repeats device 0, which still exercises the partitioning and the per-part pointer offsets."""
    b2, b3, b4, wref = golden["b4_beta"]
    disp = gpu.dispersion.DispersionParams(omega_ref=wref, beta2=b2, beta3=b3, beta4=b4)
    cfg = gpu.config.custom_simulation_config(z_max=20.0, dz=0.2, save_every=10)
    lam1 = np.linspace(1545e-9, 1555e-9, 13)
    lam2 = np.linspace(1557e-9, 1559e-9, 13)           # per-row second pump: lambda2 pointer must move too
    lam3 = np.linspace(1400e-9, 1700e-9, 257)
    kw = dict(cfg=cfg, lambda_p1_m=lam1, lambda_signal_m=lam3, lambda_p2_m=lam2, gamma=11.5e-3, alpha=1e-4,
              p_in=golden["b4_p_in"], dispersion=disp, gain_unit="linear", want_pmax=True)
    one = gpu.scan_mismtach.sweep_gain_2d(**kw)
    n_dev = gpu._lib.device_count()
    for count in (2, 5, 16):
        devices = [k % n_dev for k in range(count)]
        out = None
        if pinned:
            out = {k: gpu._lib.pinned_empty((13, 257), dt) for k, dt in
                   (("gain_lin", np.float64), ("dbeta", np.float64), ("valid", np.int32), ("status", np.int32))}
        many = gpu.scan_mismtach.sweep_gain_2d(devices=devices, out=out, **kw)
        for k in ("gain", "dbeta", "valid", "status", "Pmax"):
            assert np.array_equal(one[k], many[k], equal_nan=True), (k, count)

