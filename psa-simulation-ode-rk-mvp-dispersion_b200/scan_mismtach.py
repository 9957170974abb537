"""Sweep drivers (the data-parallel dimension of the hot path), batched on the device.

Module name keeps the reference's spelling (`scan_mismtach.py`, imported as such by its main.py:17).
Public functions keep the reference's keyword signatures and return tuples:

    plot_max_signal_gain_vs_lambda_signal(...)     -> (x, gain_max)          scan_mismtach.py:262-430
    plot_max_gain_and_dbeta_vs_lambda_signal(...)  -> (x, gain_max, dbeta)   scan_mismtach.py:588-783
    scan_mismatch_seeded_signal(gain_mode)         -> 1-D dbeta sweep        scan_mismtach.py:43-259
    plot_dbeta_vs_lambda_signal(...)               -> (x, dbeta)             scan_mismtach.py:473-585

The reference runs `plan_from_wavelengths` + `compute_phase_mismatch` + `run_single_simulation`
per point in a Python loop (:357-392, :694-738).  Here only the wavelength axes go to the GPU:
`fpa_yaman4_sweep_host` runs ONE kernel that builds each point's frequency plan, validity flag and
Delta-beta, integrates it with the fused RK4 loop and reduces to max_saved |A3|^2 / p_in[2];
gain / dbeta / status come back.  Per-point failures become NaN exactly where the reference's `except Exception`
leaves NaN; argument errors raised before the reference's loop are raised here too.

`sweep_gain_2d` extends the same call to a pump x signal wavelength grid (BASELINE config 4).
Plotting is presentation only: it runs when matplotlib is importable and a figure is asked for.
"""
from __future__ import annotations

import time
from typing import Literal, Optional, Sequence, Tuple

import numpy as np

from . import _device, _lib
from .config import SimulationConfig, custom_simulation_config, validate_config
from .dispersion import DispersionParams
from .parameters import FiberParams, SimulationGrid
from .phase_matching import PhaseMatchingConfig, PhaseMatchingMethod, fill_plan_desc
from .simulation import (_default_phase_matching_cfg, _length_scale_to_m, make_initial_amplitudes,
                         run_batch_simulation)

GainMode = Literal["end", "max"]


def _select_power_metric(Pz: np.ndarray, mode: GainMode) -> float:
    """'end' -> P(z_max); 'max' -> max over the saved samples."""
    if Pz.ndim != 1:
        raise ValueError("Pz must be a 1D array of power versus z.")
    if mode == "end":
        return float(Pz[-1])
    if mode == "max":
        return float(np.max(Pz))
    raise ValueError(f"Unknown gain_mode={mode!r}. Use 'end' or 'max'.")


# ------------------------------------------------------------------ shared argument handling
def _signal_axis(lambda_signal_m) -> np.ndarray:
    lam3 = np.asarray(list(lambda_signal_m), dtype=float)
    if lam3.ndim != 1 or lam3.size == 0:
        raise ValueError("lambda_signal_m must be a non-empty 1D sequence")
    if not np.all(np.isfinite(lam3)) or np.any(lam3 <= 0.0):
        raise ValueError("lambda_signal_m must contain finite positive wavelengths (m)")
    return lam3


def _powers_and_phases(p_in, phase_in):
    p0 = np.asarray(list(p_in), dtype=float)
    if p0.shape != (4,):
        raise ValueError(f"p_in must have shape (4,), got {p0.shape}")
    if not np.all(np.isfinite(p0)) or np.any(p0 < 0.0):
        raise ValueError("p_in must contain finite non-negative powers")
    if p0[2] <= 0.0:
        raise ValueError("p_in[2] (signal seed power) must be > 0 to define gain")
    ph0 = None
    if phase_in is not None:
        ph0 = np.asarray(list(phase_in), dtype=float)
        if ph0.shape != (4,):
            raise ValueError(f"phase_in must have shape (4,), got {ph0.shape}")
        if not np.all(np.isfinite(ph0)):
            raise ValueError("phase_in must contain finite values")
    return p0, ph0


def _norm_choice(value, allowed, text):
    v = str(value).strip().lower()
    if v not in allowed:
        raise ValueError(text)
    return v


def _x_axis(lam3, unit):
    u = unit.strip().lower()
    if u == "nm":
        return lam3 * 1e9, r"Signal wavelength $\lambda_3$ (nm)"
    if u == "m":
        return lam3, r"Signal wavelength $\lambda_3$ (m)"
    raise ValueError("return_wavelength_unit must be 'm' or 'nm'")


def _run_constants_ok(cfg, gamma, alpha, dispersion, pm_cfg, length_unit) -> bool:
    """The per-run checks of run_single_simulation that do not depend on the scan point
    (simulation.py:277-336).  In the reference a failure here raises inside the per-point
    `try` and therefore turns EVERY point into NaN; same here."""
    try:
        validate_config(cfg)
        s = _length_scale_to_m(length_unit)
        if dispersion is not None and not isinstance(dispersion, DispersionParams):
            raise TypeError("dispersion must be DispersionParams or None")
        if not isinstance(pm_cfg, PhaseMatchingConfig):
            raise TypeError("phase_matching_cfg must be PhaseMatchingConfig or None")
        FiberParams(length_m=float(cfg.z_max) * s, gamma_W_m=float(gamma) / s, alpha_1_m=float(alpha) / s)
        SimulationGrid(dz_m=float(cfg.dz) * s)
        if pm_cfg.method != PhaseMatchingMethod.PROVIDED and dispersion is None:
            raise ValueError("disp must be provided unless method == 'provided'")
        return True
    except Exception:
        return False


def sweep_gain_2d(*, cfg: SimulationConfig, lambda_p1_m, lambda_p2_m, lambda_signal_m, gamma: float,
                  alpha: float, p_in, phase_in=None, dispersion: Optional[DispersionParams] = None,
                  phase_matching_cfg: Optional[PhaseMatchingConfig] = None, length_unit: str = "m",
                  gain_unit: str = "dB", want_pmax: bool = False,
                  device: Optional[int] = None, out: Optional[dict] = None, devices=None) -> dict:
    """max-over-saved signal gain and dbeta on the grid lambda_p1[n1] x lambda_signal[n3]
    (lambda_p2 scalar or [n1]).  Returns dict(gain[n1,n3] in gain_unit, gain_lin, dbeta, valid,
    status, n_steps).  One C-ABI call: axes up, results down.  `out` may hold preallocated
    (pinned) arrays for gain_lin / dbeta / valid / status.  `devices=[0, 1, ...]` splits the pump
    rows over several GPUs of the box from this one process (bit-identical results)."""
    lam3 = _signal_axis(lambda_signal_m)
    lam1 = np.atleast_1d(np.asarray(lambda_p1_m, dtype=float))
    lam2 = np.atleast_1d(np.asarray(lambda_p2_m, dtype=float))
    p0, ph0 = _powers_and_phases(p_in, phase_in)
    unit = _norm_choice(gain_unit, ("db", "linear"), "gain_unit must be 'dB' or 'linear'")

    pm_cfg = phase_matching_cfg
    if pm_cfg is None:
        try:
            pm_cfg = _default_phase_matching_cfg(dispersion=dispersion, beta_legacy=None)
        except ValueError:
            pm_cfg = None
    n1, n3 = lam1.size, lam3.size
    if pm_cfg is None or not _run_constants_ok(cfg, gamma, alpha, dispersion, pm_cfg, length_unit):
        # every run would raise -> all NaN; dbeta is still reported when it can be computed
        nan = np.full((n1, n3), np.nan)
        out = {"gain": nan, "gain_lin": nan.copy(), "dbeta": nan.copy(),
               "valid": np.zeros((n1, n3), np.int32), "status": np.full((n1, n3), -1, np.int32),
               "n_steps": 0}
        if isinstance(pm_cfg, PhaseMatchingConfig) and (dispersion is not None or
                                                        pm_cfg.method == PhaseMatchingMethod.PROVIDED):
            plan, keep = _device.new_plan_desc(lam1, lam2, lam3)
            fill_plan_desc(plan, dispersion, pm_cfg)
            out["dbeta"] = _device.dbeta_table(plan, device=device)["dbeta"]
        return out

    s = _length_scale_to_m(length_unit)
    d = _lib.SweepDesc()
    plan, keep = _device.new_plan_desc(lam1, lam2, lam3)
    fill_plan_desc(plan, dispersion, pm_cfg)
    d.plan = plan
    A0 = make_initial_amplitudes(p0, ph0)
    for j in range(4):
        d.A0[2 * j], d.A0[2 * j + 1] = A0[j].real, A0[j].imag
    d.p_signal = float(p0[2])
    d.gamma, d.alpha = float(gamma), float(alpha)
    d.z_max, d.dz = float(cfg.z_max), float(cfg.dz)
    d.length_scale = s
    d.save_every = int(cfg.save_every)
    d.flags = _lib.CHECK_NAN if cfg.check_nan else 0
    out = _device.sweep(d, want_pmax=want_pmax, device=device, out=out, devices=devices)
    g = out["gain_lin"]
    with np.errstate(invalid="ignore", divide="ignore"):
        out["gain"] = g if unit == "linear" else 10.0 * np.log10(g)
    out["n_steps"] = int(round(float(cfg.z_max) * s / (float(cfg.dz) * s)))
    return out


def _phase_axis(phase_axis, phase_weights):
    ax = np.asarray(phase_axis, dtype=float)
    if ax.ndim != 1 or ax.size == 0:
        raise ValueError("phase_axis must be a non-empty 1D sequence of phases (rad)")
    if ax.size > _lib.MAX_PHASES:
        raise ValueError(f"phase_axis may hold at most {_lib.MAX_PHASES} phases, got {ax.size}")
    if not np.all(np.isfinite(ax)):
        raise ValueError("phase_axis must contain finite values")
    w = np.asarray(list(phase_weights), dtype=float)
    if w.shape != (4,):
        raise ValueError(f"phase_weights must have shape (4,), got {w.shape}")
    if not np.all(np.isfinite(w)):
        raise ValueError("phase_weights must contain finite values")
    return ax, w


def phase_sweep_inputs(p_in, phase_in, phase_axis, phase_weights=(0.0, 0.0, 1.0, 0.0)):
    """(A0_table [K,4] complex128, phases [K,4], relative_phase [K]) of a phase sweep: phase index k starts from
    make_initial_amplitudes(p_in, phase_in + phase_axis[k] * phase_weights); its relative phase is
    theta_k = phi_p1 + phi_p2 - phi_s - phi_i of that input phase."""
    p0, ph0 = _powers_and_phases(p_in, phase_in)
    ax, w = _phase_axis(phase_axis, phase_weights)
    base = np.zeros(4) if ph0 is None else ph0
    phases = np.stack([base + ax[k] * w for k in range(ax.size)])
    table = np.stack([make_initial_amplitudes(p0, phases[k]) for k in range(ax.size)])
    theta = phases[:, 0] + phases[:, 1] - phases[:, 2] - phases[:, 3]
    return np.ascontiguousarray(table, dtype=np.complex128), phases, theta


def sweep_phase_gain_2d(*, cfg: SimulationConfig, lambda_p1_m, lambda_p2_m, lambda_signal_m, gamma: float,
                        alpha: float, p_in, phase_in=None, phase_axis, phase_weights=(0.0, 0.0, 1.0, 0.0),
                        gain_metric: GainMode = "end", dispersion: Optional[DispersionParams] = None,
                        phase_matching_cfg: Optional[PhaseMatchingConfig] = None, length_unit: str = "m",
                        gain_unit: str = "dB", device: Optional[int] = None, devices=None) -> dict:
    """Phase-sensitive gain on the grid lambda_p1[n1] x lambda_signal[n3] x phase_axis[K]: the wavelength grid of
    `sweep_gain_2d`, and for every grid point K runs, run k starting from the input phase
    phase_in + phase_axis[k] * phase_weights (default weights sweep the signal phase).  One kernel launch per GPU
    plus one reduction launch.

    gain_metric: 'end' = |A3|^2 of the last saved sample / p_in[2] (the reference's Pz[-1]), 'max' = max over the
    saved samples (the metric of `sweep_gain_2d`); NaN for failed, non-finite or <= 0 runs.

    Returns dict(gain [n1,n3,K] in gain_unit, gain_lin [n1,n3,K], status [n1,n3,K]; per grid point [n1,n3]:
    gain_max / gain_min (linear; numpy nanmax / nanmin over the K phases), idx_max / idx_min (nanargmax /
    nanargmin, -1 where all K are NaN), phase_at_max / phase_at_min (phase_axis at those indices, NaN there),
    n_finite, extinction_db = 10 log10(gain_max / gain_min), dbeta, valid; relative_phase [K] = the theta_k of
    each phase index; n_steps).  A single plan (n1 = n3 = 1) is the G(theta) curve of one amplifier."""
    lam3 = _signal_axis(lambda_signal_m)
    lam1 = np.atleast_1d(np.asarray(lambda_p1_m, dtype=float))
    lam2 = np.atleast_1d(np.asarray(lambda_p2_m, dtype=float))
    p0, _ = _powers_and_phases(p_in, phase_in)
    table, _, theta = phase_sweep_inputs(p_in, phase_in, phase_axis, phase_weights)
    ax = np.asarray(phase_axis, dtype=float)
    K = ax.size
    unit = _norm_choice(gain_unit, ("db", "linear"), "gain_unit must be 'dB' or 'linear'")
    if gain_metric not in ("end", "max"):
        raise ValueError(f"Unknown gain_metric={gain_metric!r}. Use 'end' or 'max'.")

    pm_cfg = phase_matching_cfg
    if pm_cfg is None:
        try:
            pm_cfg = _default_phase_matching_cfg(dispersion=dispersion, beta_legacy=None)
        except ValueError:
            pm_cfg = None
    n1, n3 = lam1.size, lam3.size
    if pm_cfg is None or not _run_constants_ok(cfg, gamma, alpha, dispersion, pm_cfg, length_unit):
        # every run would raise -> all NaN; dbeta is still reported when it can be computed
        nan = np.full((n1, n3), np.nan)
        out = {"gain_lin": np.full((n1, n3, K), np.nan), "gain_max": nan, "gain_min": nan.copy(),
               "idx_max": np.full((n1, n3), -1, np.int32), "idx_min": np.full((n1, n3), -1, np.int32),
               "n_finite": np.zeros((n1, n3), np.int32), "dbeta": nan.copy(),
               "valid": np.zeros((n1, n3), np.int32), "status": np.full((n1, n3, K), -1, np.int32), "n_steps": 0}
        if isinstance(pm_cfg, PhaseMatchingConfig) and (dispersion is not None or
                                                        pm_cfg.method == PhaseMatchingMethod.PROVIDED):
            plan, keep = _device.new_plan_desc(lam1, lam2, lam3)
            fill_plan_desc(plan, dispersion, pm_cfg)
            out["dbeta"] = _device.dbeta_table(plan, device=device)["dbeta"]
    else:
        s = _length_scale_to_m(length_unit)
        d = _lib.PhaseSweepDesc()
        plan, keep = _device.new_plan_desc(lam1, lam2, lam3)
        fill_plan_desc(plan, dispersion, pm_cfg)
        w = d.sweep
        w.plan = plan
        w.p_signal = float(p0[2])
        w.gamma, w.alpha = float(gamma), float(alpha)
        w.z_max, w.dz = float(cfg.z_max), float(cfg.dz)
        w.length_scale = s
        w.save_every = int(cfg.save_every)
        w.flags = _lib.CHECK_NAN if cfg.check_nan else 0
        d.n_phases = K
        d.A0_table = _lib.ptr(table)
        d.metric = _lib.GAIN_LAST_SAVED if gain_metric == "end" else _lib.GAIN_MAX_SAVED
        out = _device.phase_sweep(d, device=device, devices=devices)
        out["n_steps"] = int(round(float(cfg.z_max) * s / (float(cfg.dz) * s)))
    g = out["gain_lin"]
    with np.errstate(invalid="ignore", divide="ignore"):
        out["gain"] = g if unit == "linear" else 10.0 * np.log10(g)
        out["extinction_db"] = 10.0 * np.log10(out["gain_max"] / out["gain_min"])
    for key in ("max", "min"):
        idx = out[f"idx_{key}"]
        out[f"phase_at_{key}"] = np.where(idx >= 0, ax[np.maximum(idx, 0)], np.nan)
    out["relative_phase"] = theta
    return out


def _sweep_1d(cfg, lambda_p1_m, lambda_p2_m, lam3, gamma, alpha, p_in, phase_in, dispersion,
              phase_matching_cfg, length_unit, gain_unit):
    r = sweep_gain_2d(cfg=cfg, lambda_p1_m=[float(lambda_p1_m)], lambda_p2_m=[float(lambda_p2_m)],
                      lambda_signal_m=lam3, gamma=gamma, alpha=alpha, p_in=p_in, phase_in=phase_in,
                      dispersion=dispersion, phase_matching_cfg=phase_matching_cfg,
                      length_unit=length_unit, gain_unit=gain_unit)
    return r["gain"][0].copy(), r["dbeta"][0].copy()


def _figure(make, save_path, show):
    """Presentation tail; silently skipped when matplotlib is not installed."""
    if not show and save_path is None:
        return
    try:
        import matplotlib.pyplot as plt
    except ImportError:
        return
    fig = make(plt)
    if save_path is not None:
        fig.savefig(save_path, dpi=200, bbox_inches="tight")
    if show:
        plt.show()
    else:
        plt.close(fig)


def plot_max_signal_gain_vs_lambda_signal(
        *, cfg: SimulationConfig, lambda_p1_m: float, lambda_p2_m: float,
        lambda_signal_m: Sequence[float], gamma: float, alpha: float, p_in: Sequence[float],
        phase_in: Optional[Sequence[float]] = None, dispersion: Optional[DispersionParams] = None,
        phase_matching_cfg: Optional[PhaseMatchingConfig] = None, length_unit: str = "m",
        return_wavelength_unit: str = "nm", gain_unit: str = "dB", xscale: str = "linear",
        yscale: str = "linear", show_progress: bool = True, tqdm_desc: str = "Sweeping λ3",
        save_path: Optional[str] = None, show: bool = True) -> Tuple[np.ndarray, np.ndarray]:
    """Max (over saved z samples) signal gain versus signal wavelength; NaN where a run fails.
    `show_progress` / `tqdm_desc` are accepted for compatibility (one kernel launch: no bar)."""
    lam3 = _signal_axis(lambda_signal_m)
    _powers_and_phases(p_in, phase_in)
    unit = _norm_choice(gain_unit, ("db", "linear"), "gain_unit must be 'dB' or 'linear'")
    xs = _norm_choice(xscale, ("linear", "log"), "xscale must be 'linear' or 'log'")
    ys = _norm_choice(yscale, ("linear", "log"), "yscale must be 'linear' or 'log'")
    if ys == "log" and unit == "db":
        raise ValueError("yscale='log' is not supported with gain_unit='dB'. Use gain_unit='linear'.")
    gain_max, _ = _sweep_1d(cfg, float(lambda_p1_m), float(lambda_p2_m), lam3, gamma, alpha, p_in,
                            phase_in, dispersion, phase_matching_cfg, length_unit, gain_unit)
    x, x_label = _x_axis(lam3, return_wavelength_unit)

    def make(plt):
        fig = plt.figure()
        plt.plot(x, gain_max, marker="o")
        plt.xlabel(x_label)
        plt.ylabel("Max signal gain (linear)" if unit == "linear" else "Max signal gain (dB)")
        plt.title("Maximum signal gain vs signal wavelength")
        plt.grid(True, which="both")
        plt.xscale(xs)
        plt.yscale(ys)
        return fig

    _figure(make, save_path, show)
    return x, gain_max


def plot_max_gain_and_dbeta_vs_lambda_signal(
        *, cfg: SimulationConfig, lambda_p1_m: float, lambda_p2_m: float,
        lambda_signal_m: Sequence[float], gamma: float, alpha: float, p_in: Sequence[float],
        phase_in: Optional[Sequence[float]] = None, dispersion: DispersionParams,
        phase_matching_cfg: Optional[PhaseMatchingConfig] = None, length_unit: str = "m",
        return_wavelength_unit: str = "nm", gain_unit: str = "dB", xscale: str = "linear",
        yscale_gain: str = "linear", yscale_dbeta: str = "linear", show_progress: bool = True,
        tqdm_desc: str = "Sweeping λ3 (gain + dBeta)", save_path: Optional[str] = None,
        show: bool = True) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """One sweep over lambda3 returning max signal gain AND dbeta(lambda3) (per length_unit)."""
    lam3 = _signal_axis(lambda_signal_m)
    p0, _ = _powers_and_phases(p_in, phase_in)
    if dispersion is None:
        raise ValueError("dispersion must be provided to compute dBeta(λ3)")
    unit = _norm_choice(gain_unit, ("db", "linear"), "gain_unit must be 'dB' or 'linear'")
    xs = _norm_choice(xscale, ("linear", "log"), "xscale must be 'linear' or 'log'")
    yg = _norm_choice(yscale_gain, ("linear", "log"), "yscale_gain must be 'linear' or 'log'")
    yd = _norm_choice(yscale_dbeta, ("linear", "log"), "yscale_dbeta must be 'linear' or 'log'")
    if yg == "log" and unit == "db":
        raise ValueError("yscale_gain='log' is not supported with gain_unit='dB'. Use gain_unit='linear'.")
    gain_max, dbeta = _sweep_1d(cfg, float(lambda_p1_m), float(lambda_p2_m), lam3, gamma, alpha, p_in,
                                phase_in, dispersion, phase_matching_cfg, length_unit, gain_unit)
    x, x_label = _x_axis(lam3, return_wavelength_unit)
    ref_line = -float(gamma) * float(p0[0] + p0[1])

    def make(plt):
        fig, (top, bottom) = plt.subplots(2, 1, sharex=True, figsize=(9, 7))
        top.plot(x, gain_max, marker="o")
        top.set_ylabel("Max signal gain (linear)" if unit == "linear" else "Max signal gain (dB)")
        top.grid(True, which="both", alpha=0.3)
        top.set_yscale(yg)
        bottom.plot(x, dbeta, marker="o", label=r"$\Delta\beta(\lambda_3)$")
        bottom.axhline(ref_line, ls="--", lw=2, label=r"$\gamma(P_1+P_2)$")
        bottom.set_xlabel(x_label)
        bottom.set_ylabel(rf"$\Delta\beta$  [1/{length_unit}]")
        bottom.grid(True, which="both", alpha=0.3)
        bottom.set_xscale(xs)
        bottom.set_yscale(yd)
        bottom.legend()
        fig.suptitle("Max signal gain and phase mismatch vs signal wavelength")
        fig.tight_layout()
        return fig

    _figure(make, save_path, show)
    return x, gain_max, dbeta


def plot_dbeta_vs_lambda_signal(
        *, gamma: float, lambda_p1_m: float, lambda_p2_m: float, lambda_signal_m: Sequence[float],
        p_in: Sequence[float], dispersion: DispersionParams, return_wavelength_unit: str = "nm",
        xscale: str = "linear", yscale: str = "linear", length_unit: str = "m", show_progress: bool = True,
        tqdm_desc: str = "Scanning dBeta(λ3)", title: Optional[str] = None, save_path: Optional[str] = None,
        show: bool = True) -> Tuple[np.ndarray, np.ndarray]:
    """dBeta(lambda3) with the sign convention of the reference's private helper
    (scan_mismtach.py:462-470): beta(w1)+beta(w2)-beta(w3)-beta(w4), Taylor to 4th order about the
    dispersion's reference frequency -- i.e. MINUS the project-wide dbeta (dispersion.py:318).
    NOTE: the reference's version returns all-NaN today (it looks for `disp.omega0`, which
    DispersionParams does not have, and swallows the AttributeError, :433-438, :531-535); this is
    what it computes once that lookup is pointed at `omega_ref`.  The table is built on the device
    (`fpa_dbeta_table_host`); invalid points are NaN."""
    lam3 = _signal_axis(lambda_signal_m)
    p0 = np.asarray(list(p_in), dtype=float)
    if p0.shape != (4,):
        raise ValueError(f"p_in must have shape (4,), got {p0.shape}")
    if not np.all(np.isfinite(p0)) or np.any(p0 < 0.0):
        raise ValueError("p_in must contain finite non-negative powers")
    xs = _norm_choice(xscale, ("linear", "log"), "xscale must be 'linear' or 'log'")
    ys = _norm_choice(yscale, ("linear", "log"), "yscale must be 'linear' or 'log'")
    plan, keep = _device.new_plan_desc([float(lambda_p1_m)], [float(lambda_p2_m)], lam3)
    fill_plan_desc(plan, dispersion, PhaseMatchingConfig(method=PhaseMatchingMethod.GENERAL_TAYLOR, max_order=4))
    dbeta = -_device.dbeta_table(plan)["dbeta"][0]
    x, x_label = _x_axis(lam3, return_wavelength_unit)
    ref = float(gamma) * float(p0[0] + p0[1])
    if ys == "log" and (np.nanmin(dbeta) <= 0.0 or ref <= 0.0):
        raise ValueError("yscale='log' requires dBeta and gamma*(P1+P2) to be strictly > 0.")
    y_unit = "1/km" if str(length_unit).strip().lower() == "km" else "1/m"

    def make(plt):
        fig = plt.figure(figsize=(8.0, 5.0))
        plt.plot(x, dbeta, label=r"$d\beta(\lambda_3)$")
        plt.axhline(ref, linestyle="--", label=r"$\gamma(P_1+P_2)$")
        plt.xlabel(x_label)
        plt.ylabel(rf"$d\beta$ [{y_unit}]")
        plt.xscale(xs)
        plt.yscale(ys)
        if title is not None:
            plt.title(title)
        plt.grid(True, which="both", linestyle="--", alpha=0.5)
        plt.legend()
        plt.tight_layout()
        return fig

    _figure(make, save_path, show)
    return x, dbeta


def sweep_peak(x, gain) -> dict:
    """Location of the best scan point (the reference prints it after its dbeta scan,
    scan_mismtach.py:183-199): index (unravelled for 2-D maps), abscissa and gain; NaNs ignored."""
    g = np.asarray(gain, dtype=float)
    if g.size == 0 or np.all(np.isnan(g)):
        raise ValueError("no finite gain in the sweep")
    flat = int(np.nanargmax(g))
    idx = np.unravel_index(flat, g.shape)
    xs = np.asarray(x)
    return {"index": idx if g.ndim > 1 else idx[0], "gain": float(g[idx]),
            "x": xs[idx[-1]].item() if xs.ndim == 1 else xs[idx].item()}


def rerun_point_with_trace(*, cfg: SimulationConfig, lambda_p1_m: float, lambda_p2_m: float,
                           lambda_signal_m: float, gamma: float, alpha: float, p_in, phase_in=None,
                           dispersion: Optional[DispersionParams] = None,
                           phase_matching_cfg: Optional[PhaseMatchingConfig] = None, length_unit: str = "m"):
    """Full (z, A[n_saved, 4]) trace of ONE scan point of a wavelength sweep -- what a user runs on the
    best point of a reduce-mode sweep to look at the evolution (the (z, A) layout plotting.py consumes)."""
    from .frequency_plan import plan_from_wavelengths
    from .simulation import run_single_simulation
    omega = plan_from_wavelengths(float(lambda_p1_m), float(lambda_p2_m), float(lambda_signal_m))
    return run_single_simulation(cfg, gamma=gamma, alpha=alpha, omega=omega, p_in=p_in, phase_in=phase_in,
                                 dispersion=dispersion, phase_matching_cfg=phase_matching_cfg,
                                 length_unit=length_unit)


def sweep_dbeta_gain(*, cfg: SimulationConfig, delta_beta, gamma: float, alpha: float, p_in,
                     phase_in=None, length_unit: str = "km", gain_mode: GainMode = "end",
                     device: Optional[int] = None, devices=None) -> dict:
    """1-D phase-mismatch sweep with PROVIDED dbeta (BASELINE config 3): for each dbeta_k
    Gs = metric(P3)/(P3(0)+1e-30), Gi = metric(P4)/(p_in[2]+1e-30) with metric = end | max over
    saved samples (scan_mismtach.py:139-156; the idler is normalised by the SIGNAL seed, :82-83).
    'end' is the LAST SAVED sample, Pz[-1] (scan_mismtach.py:33-34): when save_every does not divide
    the step count that is not the end of the fiber, and the (rare) case is served from the trace.
    `devices=[...]` splits the points over several GPUs of the box."""
    if gain_mode not in ("end", "max"):
        raise ValueError(f"Unknown gain_mode={gain_mode!r}. Use 'end' or 'max'.")
    p0 = np.asarray(list(p_in), dtype=float)
    A0 = make_initial_amplitudes(p0, phase_in)
    s = _length_scale_to_m(length_unit)
    n_steps = int(round(float(cfg.z_max) * s / (float(cfg.dz) * s)))
    ragged = gain_mode == "end" and n_steps % int(cfg.save_every) != 0
    r = run_batch_simulation(cfg, gamma=gamma, alpha=alpha, delta_beta=delta_beta, A0=A0,
                             length_unit=length_unit, outputs=("trace",) if ragged else ("end", "pmax"),
                             device=device, devices=devices)
    if ragged:
        P_metric = np.abs(r["A_trace"][:, -1, :]) ** 2
    else:
        P_metric = np.abs(r["A_end"]) ** 2 if gain_mode == "end" else r["Pmax"]
    eps = 1e-30
    Ps0 = float(np.abs(A0[2]) ** 2)
    return {"Gs": P_metric[:, 2] / (Ps0 + eps), "Gi": P_metric[:, 3] / (float(p0[2]) + eps),
            "Ps_metric": P_metric[:, 2], "Pi_metric": P_metric[:, 3], "status": r["status"],
            "n_steps": r["n_steps"]}


def scan_mismatch_seeded_signal(gain_mode: GainMode = "end", *, n_points: int = 200,
                                verbose: bool = True):
    """The reference's 200-point dbeta scan (scan_mismtach.py:43-259; gamma = 10 /W/km,
    P = [0.1, 0.1, 1e-5, 0] W, 0.5 km, dz = 1e-3 km, dbeta in [-40, 40] 1/km).  The reference
    version no longer runs (it passes a removed `beta=` keyword); this one expresses the same
    scan through PROVIDED dbeta and returns (delta_list, Gs, Gi) besides printing its timing
    summary (elapsed, s/pt, pt/s as in :172-180)."""
    cfg = custom_simulation_config(z_max=0.5, dz=1e-3)
    delta_list = np.linspace(-40.0, 40.0, int(n_points))
    t0 = time.perf_counter()
    r = sweep_dbeta_gain(cfg=cfg, delta_beta=delta_list, gamma=10.0, alpha=0.0,
                         p_in=[0.1, 0.1, 1e-5, 0.0], length_unit="km", gain_mode=gain_mode)
    elapsed = time.perf_counter() - t0
    if verbose:
        best = int(np.nanargmax(r["Gs"]))
        print("=== Mismatch scan finished ===")
        print(f"n_points = {delta_list.size}; gain metric mode = {gain_mode!r}")
        print(f"elapsed = {elapsed:.3f} s; {elapsed / delta_list.size:.3e} s/pt; "
              f"{delta_list.size / max(elapsed, 1e-12):.3e} pt/s")
        print(f"best signal gain {r['Gs'][best]:.6g} at delta = {delta_list[best]:.6g} 1/km")
    return delta_list, r["Gs"], r["Gi"]
