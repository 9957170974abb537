"""CPU: the host side of the phase-sensitive sweep -- descriptor layout against the compiled header, the entry points
without a device, argument checking of `sweep_phase_gain_2d`, and the host-built table of initial states."""
import ctypes as C
import shutil
import subprocess
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def test_phase_sweep_desc_matches_the_compiled_header(fpa, tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    L = fpa._lib
    prog = ('#include <stdio.h>\n#include <stddef.h>\n#include "fpa_b200.h"\nint main(void) {\n'
            '  printf("%zu %zu %zu %zu %d %d %d %d\\n", sizeof(fpa_phase_sweep_desc), '
            'offsetof(fpa_phase_sweep_desc, n_finite), offsetof(fpa_phase_sweep_desc, n_phases), '
            'offsetof(fpa_phase_sweep_desc, metric), FPA_GAIN_MAX_SAVED, FPA_GAIN_LAST_SAVED, FPA_MAX_PHASES, 0);\n'
            '  return 0;\n}\n')
    src, exe = tmp_path / "sizes.c", tmp_path / "sizes"
    src.write_text(prog)
    subprocess.run(["gcc", "-I", str(ROOT / "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    D = L.PhaseSweepDesc
    assert got[:4] == [C.sizeof(D), D.n_finite.offset, D.n_phases.offset, D.metric.offset]
    assert D.n_phases.offset == C.sizeof(L.SweepDesc)
    assert got[4:7] == [L.GAIN_MAX_SAVED, L.GAIN_LAST_SAVED, L.MAX_PHASES]


def _desc(fpa, keep):
    L = fpa._lib
    lam1, lam3 = np.array([1550e-9]), np.linspace(1540e-9, 1565e-9, 8)
    lam2 = np.array([1558e-9])
    table = np.ones((3, 4), dtype=np.complex128)
    out = {k: np.empty(n, dt) for k, n, dt in (("g", 24, np.float64), ("st", 24, np.int32), ("db", 8, np.float64),
                                               ("va", 8, np.int32), ("gmax", 8, np.float64))}
    keep += [lam1, lam2, lam3, table, out]
    d = L.PhaseSweepDesc()
    w = d.sweep
    w.plan.n1, w.plan.n3 = 1, 8
    w.plan.lambda1, w.plan.lambda2, w.plan.lambda3 = L.ptr(lam1), L.ptr(lam2), L.ptr(lam3)
    w.plan.dbeta, w.plan.valid = L.ptr(out["db"]), L.ptr(out["va"])
    w.plan.method, w.plan.provided = L.PM_PROVIDED, 0.0
    w.p_signal, w.gamma, w.z_max, w.dz, w.length_scale, w.save_every = 1.0, 0.01, 1.0, 0.1, 1.0, 1
    w.gain_lin, w.status = L.ptr(out["g"]), L.ptr(out["st"])
    d.n_phases, d.A0_table, d.metric, d.gain_max = 3, L.ptr(table), L.GAIN_LAST_SAVED, L.ptr(out["gmax"])
    return d


def test_entry_points_need_a_device(fpa):
    if fpa._lib.device_count() > 0:
        pytest.skip("a CUDA device is present")
    L, lib = fpa._lib, fpa._lib.lib()
    keep = []
    d = _desc(fpa, keep)
    assert lib.fpa_yaman4_phase_sweep_host(C.byref(d), 0) == L.ERR_NO_DEVICE
    assert lib.fpa_yaman4_phase_sweep_dev(C.byref(d), None, 0, None) == L.ERR_NO_DEVICE
    ids = (C.c_int * 2)(0, 1)
    assert lib.fpa_yaman4_phase_sweep_multi_host(C.byref(d), 2, ids) == L.ERR_NO_DEVICE
    with pytest.raises(L.FpaError, match="no CPU"):
        fpa._device.phase_sweep(d)


def test_scratch_holds_one_more_double_per_run(fpa):
    lib = fpa._lib.lib()
    assert lib.fpa_yaman4_phase_sweep_scratch_bytes(0) == 0
    for n in (1, 31, 32, 33, 90_000, 10**7):
        n_pad = (n + 31) // 32 * 32
        extra = lib.fpa_yaman4_phase_sweep_scratch_bytes(n) - lib.fpa_yaman4_scratch_bytes(n)
        assert n_pad * 8 <= extra <= n_pad * 8 + 256, n


def test_bad_descriptors_are_refused_before_any_device_work(fpa):
    """n_phases outside [1, 65536], a NULL table and peer maps are argument errors of the host entry."""
    L, lib = fpa._lib, fpa._lib.lib()
    keep = []
    for field, value in (("n_phases", 0), ("n_phases", 65537), ("A0_table", None)):
        d = _desc(fpa, keep)
        setattr(d, field, value)
        assert lib.fpa_yaman4_phase_sweep_host(C.byref(d), 0) == L.ERR_INVALID, field
    d = _desc(fpa, keep)
    d.sweep.n_peers = 1
    assert lib.fpa_yaman4_phase_sweep_host(C.byref(d), 0) == L.ERR_INVALID
    assert "n_peers" in L.last_error()


def _kw(fpa):
    cfg = fpa.config.custom_simulation_config(z_max=10.0, dz=0.2, save_every=10)
    return dict(cfg=cfg, lambda_p1_m=[1550e-9], lambda_p2_m=1558e-9, lambda_signal_m=[1554e-9], gamma=11.5e-3,
                alpha=0.0, p_in=[0.1, 0.1, 1e-6, 1e-6], phase_axis=[0.0, 1.0])


@pytest.mark.parametrize("change, match", [
    ({"lambda_signal_m": []}, "lambda_signal_m"),
    ({"lambda_signal_m": [-1.0]}, "lambda_signal_m"),
    ({"p_in": [0.1, 0.1, 1e-6]}, "p_in"),
    ({"p_in": [0.1, 0.1, 0.0, 1e-6]}, "signal seed"),
    ({"p_in": [0.1, -0.1, 1e-6, 1e-6]}, "non-negative"),
    ({"phase_in": [0.0, 0.0, 0.0]}, "phase_in"),
    ({"phase_in": [0.0, 0.0, np.nan, 0.0]}, "phase_in"),
    ({"gain_unit": "neper"}, "gain_unit"),
    ({"phase_axis": []}, "phase_axis"),
    ({"phase_axis": [[0.0, 1.0]]}, "phase_axis"),
    ({"phase_axis": [0.0, np.inf]}, "phase_axis"),
    ({"phase_axis": np.zeros(65537)}, "at most"),
    ({"phase_weights": (0.0, 1.0)}, "phase_weights"),
    ({"phase_weights": (0.0, 0.0, np.nan, 0.0)}, "phase_weights"),
    ({"gain_metric": "mean"}, "gain_metric"),
])
def test_argument_errors_raise(fpa, change, match):
    kw = _kw(fpa)
    kw.update(change)
    with pytest.raises(ValueError, match=match):
        fpa.scan_mismtach.sweep_phase_gain_2d(**kw)


def test_same_argument_errors_as_sweep_gain_2d(fpa):
    """Every wavelength / power / phase / unit error of sweep_gain_2d is raised by the phase sweep as well."""
    for change in ({"lambda_signal_m": []}, {"p_in": [0.1, 0.1, 0.0, 1e-6]}, {"phase_in": [0.0]}, {"gain_unit": "x"}):
        kw = _kw(fpa)
        kw.update(change)
        with pytest.raises(ValueError) as plain:
            fpa.scan_mismtach.sweep_gain_2d(**{k: v for k, v in kw.items() if k != "phase_axis"})
        with pytest.raises(ValueError) as phased:
            fpa.scan_mismtach.sweep_phase_gain_2d(**kw)
        assert str(plain.value) == str(phased.value)


def test_every_run_would_raise_gives_all_nan(fpa):
    """No dispersion and no phase-matching config: the reference raises in every run, so every gain is NaN, every
    reduction empty -- without touching a device."""
    kw = _kw(fpa)
    kw.update(lambda_p1_m=[1549e-9, 1550e-9], lambda_signal_m=[1553e-9, 1554e-9, 1555e-9], phase_axis=np.arange(4.0))
    r = fpa.scan_mismtach.sweep_phase_gain_2d(**kw)
    assert r["gain_lin"].shape == (2, 3, 4) and np.isnan(r["gain_lin"]).all() and np.isnan(r["gain"]).all()
    assert np.isnan(r["gain_max"]).all() and np.isnan(r["gain_min"]).all() and np.isnan(r["extinction_db"]).all()
    assert (r["idx_max"] == -1).all() and (r["idx_min"] == -1).all() and (r["n_finite"] == 0).all()
    assert np.isnan(r["phase_at_max"]).all() and r["status"].shape == (2, 3, 4) and r["n_steps"] == 0
    assert np.array_equal(r["relative_phase"], -np.arange(4.0))


@pytest.mark.parametrize("phase_in", [None, [0.1, -0.2, 0.3, 0.05]])
@pytest.mark.parametrize("weights", [(0.0, 0.0, 1.0, 0.0), (0.5, 0.5, -1.0, 0.25)])
def test_initial_state_table_is_make_initial_amplitudes(fpa, phase_in, weights):
    p_in = [0.3, 0.2, 1e-4, 2e-5]
    ax = np.linspace(-np.pi, np.pi, 17)
    table, phases, theta = fpa.scan_mismtach.phase_sweep_inputs(p_in, phase_in, ax, weights)
    base = np.zeros(4) if phase_in is None else np.asarray(phase_in, dtype=float)
    w = np.asarray(weights, dtype=float)
    assert table.shape == (17, 4) and table.dtype == np.complex128 and table.flags["C_CONTIGUOUS"]
    for k in range(ax.size):
        want = fpa.simulation.make_initial_amplitudes(p_in, base + ax[k] * w)
        assert table[k].tobytes() == want.tobytes(), k
        ph = base + ax[k] * w
        assert theta[k] == ph[0] + ph[1] - ph[2] - ph[3]
