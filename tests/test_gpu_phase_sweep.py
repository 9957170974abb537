"""GPU: the phase-sensitive sweep (`sweep_phase_gain_2d`, fpa_yaman4_phase_sweep_*) -- a pump x signal
wavelength grid x input-phase axis in one sweep-kernel launch plus one reduction launch.

Run (g, k) must be bit-identical to the plain sweep of grid point g with phase_in + phase_axis[k] * weights, on
both launch paths (whole-run kernel, z-segment scheduler), over several devices and in both library builds;
both gain metrics must match the CPU oracle; and the physics of a phase-sensitive amplifier must come out:
no phase dependence without an idler seed, and the small-signal PSA relations G_max = (sqrt(G) + sqrt(G-1))^2,
G_max * G_min = 1 against the phase-insensitive gain G."""
import ctypes as C
import os
import warnings

import numpy as np
import pytest

import __graft_entry__ as entry

pytestmark = pytest.mark.gpu
ONE_WAVE = 148 * 16 * 32          # points that fill every resident warp of a B200 once
P_IN = [0.3, 0.2, 1e-4, 2e-5]
PHASE_IN = [0.1, -0.2, 0.3, 0.05]


@pytest.fixture(autouse=True)
def _clean_env():
    yield
    for k in ("FPA_SWEEP_SEG", "FPA_SWEEP_SEG_STEPS"):
        os.environ.pop(k, None)


def _disp(fpa, golden, scale=1.0):
    b2, b3, b4, wref = golden["b4_beta"]
    return fpa.dispersion.DispersionParams(omega_ref=wref, beta2=b2 * scale, beta3=b3 * scale, beta4=b4 * scale)


def _kw(gpu, golden, unit="m", alpha=1e-4, n1=16, n3=200, save_every=7, z_max=20.0, wide=True):
    s = 1.0 if unit == "m" else 1e-3
    cfg = gpu.config.custom_simulation_config(z_max=z_max * s, dz=0.2 * s, save_every=save_every)
    lam3 = np.linspace(600e-9, 1700e-9, n3) if wide else np.linspace(1540e-9, 1565e-9, n3)  # wide: invalid plans
    return dict(cfg=cfg, lambda_p1_m=np.linspace(1545e-9, 1555e-9, n1), lambda_signal_m=lam3, lambda_p2_m=1558e-9,
                gamma=11.5e-3 / s, alpha=alpha / s, p_in=P_IN, dispersion=_disp(gpu, golden, 1.0 / s),
                gain_unit="linear", length_unit=unit)


def _nan_reductions(gl):
    """numpy's nan-reductions over the phase axis, -1 / NaN / 0 for all-NaN rows."""
    fin = ~np.isnan(gl)
    n = fin.sum(axis=-1).astype(np.int32)
    empty = n == 0
    filled = np.where(empty[..., None], 0.0, gl)        # nanarg* raise on all-NaN rows
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)
        gmax, gmin = np.nanmax(gl, axis=-1), np.nanmin(gl, axis=-1)
    imax = np.where(empty, -1, np.nanargmax(filled, axis=-1)).astype(np.int32)
    imin = np.where(empty, -1, np.nanargmin(filled, axis=-1)).astype(np.int32)
    return {"gain_max": gmax, "gain_min": gmin, "idx_max": imax, "idx_min": imin, "n_finite": n}


def _check_reductions(r):
    want = _nan_reductions(r["gain_lin"])
    for k, v in want.items():
        assert r[k].dtype == v.dtype and r[k].tobytes() == v.tobytes(), k


def _check_against_plain_sweep(gpu, r, kw, ax, w):
    base = np.asarray(PHASE_IN, dtype=float)
    for k in range(ax.size):
        ref = gpu.scan_mismtach.sweep_gain_2d(phase_in=base + ax[k] * w, **kw)
        assert r["gain_lin"][:, :, k].tobytes() == ref["gain_lin"].tobytes(), k
        assert r["status"][:, :, k].tobytes() == ref["status"].tobytes(), k
        if k == 0:
            assert r["dbeta"].tobytes() == ref["dbeta"].tobytes() and r["valid"].tobytes() == ref["valid"].tobytes()


@pytest.mark.parametrize("K", [5, 33])
@pytest.mark.parametrize("alpha", [0.0, 1e-4])
@pytest.mark.parametrize("unit", ["m", "km"])
def test_each_phase_is_the_plain_sweep_bit_for_bit(gpu, golden, K, alpha, unit):
    """16 x 200 grid with invalid plans: K = 5 runs the whole-run kernel (16 000 points), K = 33 the z-segment
    scheduler (105 600 points, 1.4 waves).  Every slice k equals sweep_gain_2d at that phase_in."""
    kw = _kw(gpu, golden, unit, alpha)
    ax = np.linspace(0.0, 2 * np.pi, K, endpoint=False) + 0.01
    w = np.array([0.0, 0.0, 1.0, 0.0]) if K == 5 else np.array([0.5, 0.0, 1.0, -0.25])
    r = gpu.scan_mismtach.sweep_phase_gain_2d(phase_in=PHASE_IN, phase_axis=ax, phase_weights=w, gain_metric="max", **kw)
    assert r["gain_lin"].shape == (16, 200, K) and r["status"].shape == (16, 200, K) and r["dbeta"].shape == (16, 200)
    assert np.isnan(r["gain_lin"]).any() and np.isfinite(r["gain_lin"]).any()
    assert (16 * 200 * K >= ONE_WAVE) == (K == 33)
    _check_against_plain_sweep(gpu, r, kw, ax, w)
    _check_reductions(r)
    theta = (np.asarray(PHASE_IN) + ax[:, None] * w) @ np.array([1.0, 1.0, -1.0, -1.0])
    assert np.allclose(r["relative_phase"], theta, rtol=0, atol=1e-15)


@pytest.mark.parametrize("metric", ["end", "max"])
def test_gains_match_the_oracle(gpu, golden, oracle, metric):
    """48 random (grid point, phase) runs against oracle.single_run; 150 steps with save_every = 7, so the
    'end' metric is step 147, not the fiber end."""
    kw = _kw(gpu, golden, "m", 1e-4, n1=8, n3=50, save_every=7, z_max=30.0, wide=False)
    K = 8
    ax = np.linspace(0.0, 2 * np.pi, K, endpoint=False)
    r = gpu.scan_mismtach.sweep_phase_gain_2d(phase_in=PHASE_IN, phase_axis=ax, gain_metric=metric, **kw)
    d = kw["dispersion"]
    od = oracle.Taylor(d.omega_ref, 0.0, 0.0, d.beta2, d.beta3, d.beta4)
    rng = np.random.default_rng(11)
    for i, j, k in zip(rng.integers(0, 8, 48), rng.integers(0, 50, 48), rng.integers(0, K, 48)):
        om = oracle.plan_from_wavelengths(kw["lambda_p1_m"][i], 1558e-9, kw["lambda_signal_m"][j])
        ph = np.asarray(PHASE_IN) + ax[k] * np.array([0.0, 0.0, 1.0, 0.0])
        _, A, _ = oracle.single_run(z_max=30.0, dz=0.2, save_every=7, check_nan=True, gamma=11.5e-3, alpha=1e-4,
                                    omega=om, p_in=P_IN, phase_in=ph, disp=od)
        P3 = np.abs(A[:, 2]) ** 2
        want = (P3.max() if metric == "max" else P3[-1]) / P_IN[2]
        assert abs(r["gain_lin"][i, j, k] - want) <= 1e-10 * want, (i, j, k)
    _check_reductions(r)


def test_no_idler_seed_means_no_phase_dependence(gpu, golden):
    kw = _kw(gpu, golden, "m", 1e-4, n1=6, n3=40, save_every=10, z_max=60.0, wide=False)
    kw["p_in"] = [0.3, 0.2, 1e-4, 0.0]
    ax = np.linspace(0.0, 2 * np.pi, 8, endpoint=False)
    r = gpu.scan_mismtach.sweep_phase_gain_2d(phase_in=None, phase_axis=ax, gain_metric="end", **kw)
    g = r["gain_lin"]
    assert np.isfinite(g).all() and g.max() > 1.05
    assert np.max(np.abs(g - g[:, :, :1]) / g[:, :, :1]) <= 1e-12
    assert (r["n_finite"] == 8).all()


def test_small_signal_psa_relations(gpu, golden):
    """Undepleted pumps, equal signal and idler seeds: G(phi) = C + a cos(phi) + b sin(phi) with
    C + D = (sqrt(G_PIA) + sqrt(G_PIA - 1))^2 and (C + D)(C - D) = 1, D = hypot(a, b), G_PIA the gain of the same
    grid point without an idler seed."""
    cfg = gpu.config.custom_simulation_config(z_max=100.0, dz=0.5, save_every=10)
    kw = dict(cfg=cfg, lambda_p1_m=np.linspace(1549e-9, 1551e-9, 4), lambda_signal_m=np.linspace(1552e-9, 1556e-9, 24),
              lambda_p2_m=1558e-9, gamma=11.5e-3, alpha=0.0, dispersion=_disp(gpu, golden), gain_unit="linear")
    K = 8
    phi = 2 * np.pi * np.arange(K) / K
    psa = gpu.scan_mismtach.sweep_phase_gain_2d(p_in=[0.5, 0.5, 1e-12, 1e-12], phase_axis=phi, gain_metric="end", **kw)
    pia = gpu.scan_mismtach.sweep_phase_gain_2d(p_in=[0.5, 0.5, 1e-12, 0.0], phase_axis=[0.0], gain_metric="end", **kw)
    g = psa["gain_lin"]
    C_ = g.mean(axis=-1)
    a = 2 * (g * np.cos(phi)).mean(axis=-1)
    b = 2 * (g * np.sin(phi)).mean(axis=-1)
    D = np.hypot(a, b)
    G = pia["gain_lin"][:, :, 0]
    sel = G <= 4.0
    assert sel.sum() >= 48 and G[sel].max() > 1.5
    pred = (np.sqrt(G) + np.sqrt(np.maximum(G - 1.0, 0.0))) ** 2
    assert np.max(np.abs((C_ + D)[sel] / pred[sel] - 1.0)) <= 1e-8
    assert np.max(np.abs(((C_ + D) * (C_ - D))[sel] - 1.0)) <= 1e-8
    assert np.allclose(psa["gain_max"], g.max(axis=-1), rtol=0, atol=0)
    assert np.all(psa["extinction_db"][sel] > 0.0)


def _phase_desc(gpu, golden, kw, ax, metric):
    """A PhaseSweepDesc over host axes, as sweep_phase_gain_2d fills it; returns (desc, keepalive)."""
    L = gpu._lib
    table, _, _ = gpu.scan_mismtach.phase_sweep_inputs(P_IN, PHASE_IN, ax)
    plan, keep = gpu._device.new_plan_desc(kw["lambda_p1_m"], kw["lambda_p2_m"], kw["lambda_signal_m"])
    gpu.phase_matching.fill_plan_desc(plan, kw["dispersion"], gpu.phase_matching.PhaseMatchingConfig())
    d = L.PhaseSweepDesc()
    d.sweep.plan = plan
    d.sweep.p_signal, d.sweep.gamma, d.sweep.alpha = P_IN[2], kw["gamma"], kw["alpha"]
    d.sweep.z_max, d.sweep.dz, d.sweep.length_scale = kw["cfg"].z_max, kw["cfg"].dz, 1.0
    d.sweep.save_every, d.sweep.flags = kw["cfg"].save_every, L.CHECK_NAN
    d.n_phases, d.A0_table, d.metric = ax.size, L.ptr(table), (L.GAIN_LAST_SAVED if metric == "end" else L.GAIN_MAX_SAVED)
    return d, (keep, table)


def test_reductions_without_the_map_and_all_nan_rows(gpu, golden):
    """gain_lin = NULL on the host entry: the map stays in the workspace, the reductions are the same bits."""
    kw = _kw(gpu, golden, "m", 1e-4, n1=16, n3=200, save_every=7)
    ax = np.linspace(0.0, 2 * np.pi, 9, endpoint=False)
    r = gpu.scan_mismtach.sweep_phase_gain_2d(phase_in=PHASE_IN, phase_axis=ax, gain_metric="end", **kw)
    _check_reductions(r)
    assert (r["idx_max"] == -1).any() and (r["n_finite"] == 0).any() and (r["n_finite"] == 9).any()
    d, keep = _phase_desc(gpu, golden, kw, ax, "end")
    got = gpu._device.phase_sweep(d, want_map=False)
    assert "gain_lin" not in got
    for k in ("gain_max", "gain_min", "idx_max", "idx_min", "n_finite", "dbeta", "valid", "status"):
        assert got[k].tobytes() == r[k].tobytes(), k


def test_segment_scheduler_and_dev_entry(gpu, golden):
    """~90 000 runs (1.2 waves): the z-segment scheduler equals the whole-run kernel; the _dev entry with scratch
    and with NULL scratch equals the host entry, reductions included."""
    import torch
    kw = _kw(gpu, golden, "m", 1e-4, n1=90, n3=200, save_every=7, z_max=40.0)
    ax = np.linspace(0.0, 2 * np.pi, 5, endpoint=False)
    G, K = 90 * 200, 5
    assert ONE_WAVE < G * K < 8 * ONE_WAVE
    for metric in ("end", "max"):
        seg = gpu.scan_mismtach.sweep_phase_gain_2d(phase_in=PHASE_IN, phase_axis=ax, gain_metric=metric, **kw)
        os.environ["FPA_SWEEP_SEG"] = "0"
        whole = gpu.scan_mismtach.sweep_phase_gain_2d(phase_in=PHASE_IN, phase_axis=ax, gain_metric=metric, **kw)
        os.environ.pop("FPA_SWEEP_SEG")
        for k in ("gain_lin", "status", "dbeta", "valid", "gain_max", "gain_min", "idx_max", "idx_min", "n_finite"):
            assert seg[k].tobytes() == whole[k].tobytes(), (metric, k)
    _check_against_plain_sweep(gpu, seg, kw, ax, np.array([0.0, 0.0, 1.0, 0.0]))

    L, lib = gpu._lib, gpu._lib.lib()
    dev = torch.device("cuda", 0)
    L.check(lib.fpa_set_device(0))
    table, _, _ = gpu.scan_mismtach.phase_sweep_inputs(P_IN, PHASE_IN, ax)
    t = {"l1": torch.from_numpy(kw["lambda_p1_m"]).to(dev), "l2": torch.tensor([1558e-9], dtype=torch.float64, device=dev),
         "l3": torch.from_numpy(kw["lambda_signal_m"]).to(dev),
         "tab": torch.from_numpy(table.view(np.float64).copy()).to(dev)}
    nb = int(lib.fpa_yaman4_phase_sweep_scratch_bytes(G * K))
    assert nb > int(lib.fpa_yaman4_scratch_bytes(G * K))

    def run(scratch):
        o = {"gain_lin": torch.empty(G * K, dtype=torch.float64, device=dev),
             "status": torch.empty(G * K, dtype=torch.int32, device=dev),
             "dbeta": torch.empty(G, dtype=torch.float64, device=dev), "valid": torch.empty(G, dtype=torch.int32, device=dev),
             "gain_max": torch.empty(G, dtype=torch.float64, device=dev),
             "gain_min": torch.empty(G, dtype=torch.float64, device=dev),
             "idx_max": torch.empty(G, dtype=torch.int32, device=dev), "idx_min": torch.empty(G, dtype=torch.int32, device=dev),
             "n_finite": torch.empty(G, dtype=torch.int32, device=dev)}
        d, keep = _phase_desc(gpu, golden, kw, ax, "end")
        d.sweep.plan.lambda1, d.sweep.plan.lambda2 = t["l1"].data_ptr(), t["l2"].data_ptr()
        d.sweep.plan.lambda3, d.sweep.plan.lambda2_stride = t["l3"].data_ptr(), 0
        d.sweep.plan.dbeta, d.sweep.plan.valid = o["dbeta"].data_ptr(), o["valid"].data_ptr()
        d.sweep.gain_lin, d.sweep.status = o["gain_lin"].data_ptr(), o["status"].data_ptr()
        d.A0_table = t["tab"].data_ptr()
        for k in ("gain_max", "gain_min", "idx_max", "idx_min", "n_finite"):
            setattr(d, k, o[k].data_ptr())
        scr = torch.empty(max(nb, 16), dtype=torch.uint8, device=dev) if scratch else None
        L.check(lib.fpa_yaman4_phase_sweep_dev(C.byref(d), scr.data_ptr() if scratch else None, nb if scratch else 0,
                                               torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        return {k: v.cpu().numpy() for k, v in o.items()}

    with_scr, without = run(True), run(False)
    os.environ["FPA_SWEEP_SEG"] = "0"
    host_end = gpu.scan_mismtach.sweep_phase_gain_2d(phase_in=PHASE_IN, phase_axis=ax, gain_metric="end", **kw)
    for k in with_scr:
        assert with_scr[k].tobytes() == without[k].tobytes(), k
        assert with_scr[k].tobytes() == host_end[k].reshape(-1).tobytes(), k


def test_multi_device_equals_one_device(gpu, golden):
    """devices=[0, 0, 0] with a grid of 3 * 1067 + 1 points: ragged shares, bit-identical results."""
    kw = _kw(gpu, golden, "m", 1e-4, n1=1, n3=3202, save_every=7)
    ax = np.linspace(0.0, 2 * np.pi, 6, endpoint=False)
    one = gpu.scan_mismtach.sweep_phase_gain_2d(phase_in=PHASE_IN, phase_axis=ax, gain_metric="end", **kw)
    many = gpu.scan_mismtach.sweep_phase_gain_2d(phase_in=PHASE_IN, phase_axis=ax, gain_metric="end", devices=[0, 0, 0],
                                                 **kw)
    assert 3202 % 3 != 0
    for k in ("gain_lin", "status", "dbeta", "valid", "gain_max", "gain_min", "idx_max", "idx_min", "n_finite"):
        assert one[k].tobytes() == many[k].tobytes(), k


def _both(gpu, fn):
    out = fn()
    if not entry.REF_LIB.exists():
        pytest.fail("build/libfpa_b200_ref.so missing: build() did not produce the reference-schedule library")
    with gpu._lib.use_library(entry.REF_LIB) as ref:
        assert gpu._lib.lib() is ref and b"ptxas schedule" in gpu._lib.lib().fpa_version()
        out_ref = fn()
    assert b"re-scheduled" in gpu._lib.lib().fpa_version()
    return out, out_ref


@pytest.mark.parametrize("alpha", [0.0, 1e-4])
@pytest.mark.parametrize("n1", [16, 90])            # whole-run kernel / z-segment scheduler
def test_sass_pass_bit_identical(gpu, golden, alpha, n1):
    """The phase-sweep instantiations go through the SASS pass like every kernel of yaman4.cu: bit-identical to the
    ptxas-schedule build on both launch paths, lossy and lossless, both metrics."""
    kw = _kw(gpu, golden, "m", alpha, n1=n1, n3=200, save_every=7, z_max=40.0)
    ax = np.linspace(0.0, 2 * np.pi, 5, endpoint=False)
    for metric in ("end", "max"):
        a, b = _both(gpu, lambda: gpu.scan_mismtach.sweep_phase_gain_2d(  # noqa: E731
            phase_in=PHASE_IN, phase_axis=ax, gain_metric=metric, **kw))
        for k in a:
            if isinstance(a[k], np.ndarray):
                assert a[k].tobytes() == b[k].tobytes(), (metric, k)
