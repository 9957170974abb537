"""Single-run and batched runners of the 4-wave FWM model.

`run_single_simulation` keeps the reference's signature, unit handling and validation order
(simulation.py:220-364: validate cfg :277, km->m scale :279, A0 :282-284, dispersion / PROVIDED
dbeta scaling :287-313, dataclass assembly :316-336, dbeta once :340-346, march :349-357, z
back-conversion :360-364); the march itself is one launch of the fused CUDA integrator.

`run_batch_simulation` is the batched analogue (NOT in the reference, which loops in Python):
B scan points that differ in dbeta (and optionally gamma / alpha / A0) go through ONE kernel
launch and come back either as reductions (end state, max over saved samples) or as traces.
"""
from __future__ import annotations

from typing import Optional, Sequence

import numpy as np

from . import _device, constants
from ._checks import four
from .config import (SimulationConfig, custom_simulation_config, default_simulation_config,
                     validate_config)
from .dispersion import DispersionParams
from .integrators import integrate_interval
from .parameters import FiberParams, PhaseMatchingParams, SimulationGrid, WavesParams, make_model_params
from .phase_matching import (PhaseMatchingConfig, PhaseMatchingMethod, PhaseMatchingResult,
                             compute_phase_mismatch)
from .yaman_model import rhs_yaman_simplified


def _length_scale_to_m(length_unit: str) -> float:
    unit = str(length_unit).strip().lower()
    if unit == "m":
        return 1.0
    if unit == "km":
        return 1000.0
    raise ValueError(f"Unsupported length_unit={length_unit!r}. Use 'm' or 'km'.")


def _n_steps(cfg: SimulationConfig, s: float) -> int:
    """RK4 steps of a run over cfg.z_max in steps of cfg.dz, both per length unit with `s` metres each: both are
    scaled to metres before they are divided, so the count is the one the runner's metre-valued z_max and dz give
    (z_max / dz unscaled can round differently when s != 1)."""
    return int(round(float(cfg.z_max) * s / (float(cfg.dz) * s)))


def _to_omega_array(omega) -> np.ndarray:
    return four(omega, "omega", positive_only=True)


def _to_power_array(p_in) -> np.ndarray:
    return four(p_in, "p_in", nonneg_only=True)


def _to_phase_array(phase_in) -> np.ndarray:
    return np.zeros(4, dtype=float) if phase_in is None else four(phase_in, "phase_in")


def make_initial_amplitudes(p_in: Sequence[float], phase_in: Optional[Sequence[float]] = None) -> np.ndarray:
    """A0 = sqrt(P) as complex128; multiplied by exp(i phi) only when some phi != 0."""
    amp = np.sqrt(_to_power_array(p_in)).astype(np.complex128, copy=False)
    ph = _to_phase_array(phase_in)
    if np.any(ph != 0.0):
        amp *= np.exp(1j * ph)
    return amp


def _scale_dispersion_to_m(disp: DispersionParams, length_scale_to_m: float) -> DispersionParams:
    """beta_n per length_unit -> per metre (every order divided by the scale)."""
    s = float(length_scale_to_m)
    if s == 1.0:
        return disp
    extra = None if disp.extra is None else {int(k): float(v) / s for k, v in disp.extra.items()}
    return DispersionParams(disp.omega_ref, *(float(getattr(disp, f"beta{n}")) / s for n in range(5)),
                            extra=extra)


def _scale_phase_matching_cfg_to_m(cfg: PhaseMatchingConfig, length_scale_to_m: float) -> PhaseMatchingConfig:
    """Only a PROVIDED dbeta carries a length unit."""
    if cfg.method != PhaseMatchingMethod.PROVIDED:
        return cfg
    if cfg.provided_delta_beta is None:
        raise ValueError("PhaseMatchingConfig.PROVIDED requires provided_delta_beta")
    s = float(length_scale_to_m)
    if s == 1.0:
        return cfg
    return PhaseMatchingConfig(method=PhaseMatchingMethod.PROVIDED, max_order=cfg.max_order,
                               even_orders=cfg.even_orders, atol=cfg.atol, rtol=cfg.rtol,
                               provided_delta_beta=float(cfg.provided_delta_beta) / s)


def _default_phase_matching_cfg(*, dispersion, beta_legacy) -> PhaseMatchingConfig:
    """dispersion given -> SYMMETRIC_EVEN (2,4); only legacy betas -> PROVIDED (b3+b4)-(b1+b2)."""
    if dispersion is not None:
        return PhaseMatchingConfig(method=PhaseMatchingMethod.SYMMETRIC_EVEN, max_order=4,
                                   even_orders=(2, 4), atol=0.0, rtol=1e-12)
    if beta_legacy is not None:
        b = np.asarray(beta_legacy, dtype=float)
        if b.shape != (4,):
            raise ValueError("beta_legacy must have shape (4,)")
        return PhaseMatchingConfig(method=PhaseMatchingMethod.PROVIDED, max_order=0, even_orders=(2,),
                                   atol=0.0, rtol=1e-12,
                                   provided_delta_beta=float((b[2] + b[3]) - (b[0] + b[1])))
    raise ValueError("Provide either dispersion or beta_legacy (or an explicit phase_matching_cfg).")


def _assemble(cfg, *, gamma, alpha, omega, p_in, phase_in, dispersion, phase_matching_cfg,
              beta_legacy, length_unit):
    """Everything run_single_simulation does before the march: returns (params, A0)."""
    validate_config(cfg)
    s = _length_scale_to_m(length_unit)
    om = _to_omega_array(omega)
    A0 = make_initial_amplitudes(_to_power_array(p_in), phase_in)

    legacy_m = None
    if beta_legacy is not None:
        b = np.asarray(list(beta_legacy), dtype=float)
        if b.shape != (4,):
            raise ValueError(f"beta_legacy must have shape (4,), got {b.shape}")
        if not np.all(np.isfinite(b)):
            raise ValueError("beta_legacy must be finite")
        legacy_m = b / s
    disp_m = None
    if dispersion is not None:
        if not isinstance(dispersion, DispersionParams):
            raise TypeError("dispersion must be DispersionParams or None")
        disp_m = _scale_dispersion_to_m(dispersion, s)
    pm_cfg = phase_matching_cfg
    if pm_cfg is None:
        pm_cfg = _default_phase_matching_cfg(dispersion=disp_m, beta_legacy=legacy_m)
    if not isinstance(pm_cfg, PhaseMatchingConfig):
        raise TypeError("phase_matching_cfg must be PhaseMatchingConfig or None")
    pm_cfg = _scale_phase_matching_cfg_to_m(pm_cfg, s)

    params = make_model_params(
        waves=WavesParams(omega=om, symmetric=None),
        fiber=FiberParams(length_m=float(cfg.z_max) * s, gamma_W_m=float(gamma) / s,
                          alpha_1_m=float(alpha) / s, dispersion=disp_m, beta_legacy_1_m=legacy_m),
        grid=SimulationGrid(dz_m=float(cfg.dz) * s, z0_m=0.0),
        phase_matching=PhaseMatchingParams(config=pm_cfg),
    )
    res: PhaseMatchingResult = compute_phase_mismatch(
        params.waves.omega, params.fiber.dispersion, params.phase_matching.config,
        symmetric_hint=params.waves.symmetric)
    params.cache.set_phase_mismatch(res.delta_beta, symmetric=res.symmetric)
    return params, A0


def run_single_simulation(cfg: SimulationConfig, *, gamma: float, alpha: float,
                          omega: Sequence[float], p_in: Sequence[float],
                          phase_in: Optional[Sequence[float]] = None,
                          dispersion: Optional[DispersionParams] = None,
                          phase_matching_cfg: Optional[PhaseMatchingConfig] = None,
                          beta_legacy: Optional[Sequence[float]] = None, length_unit: str = "m",
                          return_length_unit: Optional[str] = None) -> tuple[np.ndarray, np.ndarray]:
    """One scalar 4-wave run -> (z_out[n_saved], A[n_saved, 4] complex128).  gamma, alpha,
    cfg.z_max/dz, dispersion and a PROVIDED dbeta are per `length_unit` ('m' | 'km')."""
    params, A0 = _assemble(cfg, gamma=gamma, alpha=alpha, omega=omega, p_in=p_in, phase_in=phase_in,
                           dispersion=dispersion, phase_matching_cfg=phase_matching_cfg,
                           beta_legacy=beta_legacy, length_unit=length_unit)
    z_m, A = integrate_interval(rhs_yaman_simplified, params.fiber.length_m, params.grid.dz_m, A0,
                                params, save_every=cfg.save_every, check_nan=cfg.check_nan)
    out_unit = length_unit if return_length_unit is None else return_length_unit
    return z_m / _length_scale_to_m(out_unit), A


def _batch_inputs(cfg, gamma, alpha, delta_beta, p_in, phase_in, A0, length_unit):
    """The checks and unit scaling both batch runners start with: (s, A0, dbeta [B], gamma, alpha, z_max, n_steps),
    dbeta / gamma / alpha per metre, z_max in metres, s = metres per length_unit."""
    validate_config(cfg)
    s = _length_scale_to_m(length_unit)
    if A0 is None:
        A0 = make_initial_amplitudes(p_in, phase_in)
    db = np.asarray(delta_beta, dtype=float).reshape(-1) / s
    return (s, A0, db, np.asarray(gamma, dtype=float) / s, np.asarray(alpha, dtype=float) / s,
            float(cfg.z_max) * s, _n_steps(cfg, s))


def run_batch_simulation(cfg: SimulationConfig, *, gamma, alpha, delta_beta, p_in=None, phase_in=None,
                         A0=None, length_unit: str = "m", outputs: Sequence[str] = ("end", "pmax"),
                         phase_exact: bool = False, device: Optional[int] = None, devices=None) -> dict:
    """B runs in one kernel launch (`devices=[0, 1, ...]`: one launch per listed GPU, each on its own
    contiguous share of the points, bit-identical results).  `delta_beta` [B] (per length_unit); gamma / alpha scalars
    or [B]; initial state from (p_in, phase_in) shared by all points, or explicit A0 [B,4] / [4].
    outputs: any of 'end' (A_end[B,4]), 'pmax' (max over SAVED samples of |A|^2, [B,4]),
    'trace' (A[B,n_saved,4] and z[n_saved]).  `status[B]` = first non-finite step or -1; with
    cfg.check_nan nothing is raised here -- bad points are the caller's to mask (the sweeps
    turn them into NaN like the reference, scan_mismtach.py:736-738)."""
    s, A0, db, gam, alp, z_max, n_steps = _batch_inputs(cfg, gamma, alpha, delta_beta, p_in, phase_in, A0, length_unit)
    want = {str(o).lower() for o in outputs}
    r = _device.yaman4_batch(db, gam, alp, A0, z_max=z_max, n_steps=n_steps, save_every=cfg.save_every,
                             trace="trace" in want, end="end" in want, pmax="pmax" in want,
                             check_nan=cfg.check_nan, phase_exact=phase_exact, device=device, devices=devices)
    if "trace" in want:
        grid = np.linspace(0.0, z_max, n_steps + 1)
        r["z"] = np.concatenate((grid[:1], grid[cfg.save_every::cfg.save_every])) / s
    r["n_steps"] = n_steps
    return r


def waves_to_columns(waves) -> int:
    """Column mask of the transfer kernels for whole waves: wave w -> columns 2w (Re A_w(0)) and 2w+1 (Im)."""
    mask = 0
    for w in np.atleast_1d(np.asarray(waves, dtype=int)).tolist():
        if not 0 <= w < 4:
            raise ValueError(f"waves must be indices in 0..3, got {w}")
        mask |= 3 << (2 * w)
    if mask == 0:
        raise ValueError("waves must name at least one wave")
    return mask


def run_batch_transfer(cfg: SimulationConfig, *, gamma, alpha, delta_beta, p_in=None, phase_in=None, A0=None,
                       waves=(2, 3), length_unit: str = "m", device: Optional[int] = None, devices=None) -> dict:
    """Small-signal transfer matrices of B runs (arguments as `run_batch_simulation`): J = dA(L)/dA(0), the exact
    derivative of the RK4 map the batch integrator computes, one tangent column per real input component.

    Returns dict(jac [B,8,nc], columns, A_end [B,4], status [B], n_steps).  Row r of jac is Re (r even) or Im
    (r odd) of A_{r//2}(L); column k is the derivative with respect to input component columns[k] (2w: Re A_w(0),
    2w+1: Im A_w(0)); `waves` selects whole waves (both quadratures).  J is dimensionless, the same in m and km.
    A run that fails under cfg.check_nan, or whose dbeta is not finite, gets an all-NaN J."""
    s, A0, db, gam, alp, z_max, n_steps = _batch_inputs(cfg, gamma, alpha, delta_beta, p_in, phase_in, A0, length_unit)
    mask = waves_to_columns(waves)
    r = _device.yaman4_transfer(db, gam, alp, A0, mask, z_max=z_max, n_steps=n_steps, check_nan=cfg.check_nan,
                                device=device, devices=devices)
    r["columns"] = tuple(c for c in range(8) if mask >> c & 1)
    r["n_steps"] = n_steps
    return r


def example_zero_signal() -> tuple[np.ndarray, np.ndarray]:
    """Two 0.5 W pumps, no signal/idler, dbeta = 0 PROVIDED, km units (simulation.py:371-405)."""
    w0 = 2.0 * np.pi * constants.c / 1.55e-6
    return run_single_simulation(
        default_simulation_config(), gamma=1.3, alpha=0.0, omega=np.full(4, w0),
        p_in=np.array([0.5, 0.5, 0.0, 0.0]), phase_in=None, dispersion=None,
        phase_matching_cfg=PhaseMatchingConfig(method=PhaseMatchingMethod.PROVIDED, provided_delta_beta=0.0),
        beta_legacy=None, length_unit="km", return_length_unit="km")


def custom_seeded_signal() -> tuple[np.ndarray, np.ndarray]:
    """Seeded signal + idler, dbeta = 0 PROVIDED, 5000 steps (simulation.py:408-447)."""
    w0 = 2.0 * np.pi * constants.c / 1.55e-6
    return run_single_simulation(
        custom_simulation_config(z_max=0.5, dz=1e-4), gamma=10.0, alpha=0.0, omega=np.full(4, w0),
        p_in=np.array([1e-1, 1e-1, 1e-4, 1e-6]), phase_in=np.zeros(4), dispersion=None,
        phase_matching_cfg=PhaseMatchingConfig(method=PhaseMatchingMethod.PROVIDED, provided_delta_beta=0.0),
        beta_legacy=None, length_unit="km", return_length_unit="km")
