"""Small-signal quantities from the transfer matrices of `simulation.run_batch_transfer` and
`scan_mismtach.sweep_transfer_2d` (pure numpy on the host, a few FLOPs per point).

A transfer matrix J = dA(L)/dA(0) comes as jac [..., 8, nc] with the tuple `columns`: row r is Re (r even) or
Im (r odd) of A_{r//2}(L), column k the derivative with respect to input component columns[k] (2w: Re A_w(0),
2w + 1: Im A_w(0)).  Wave order [pump1, pump2, signal, idler] = 0, 1, 2, 3.

The real 2x2 block of output wave o and input wave w,

    M = [[a, b], [c, d]] = [[dRe A_o/dRe A_w, dRe A_o/dIm A_w], [dIm A_o/dRe A_w, dIm A_o/dIm A_w]],

acts on a complex perturbation as  dA_o(L) = mu dA_w(0) + nu conj(dA_w(0))  with

    mu = ((a + d) + i (c - b)) / 2      (complex-linear part)
    nu = ((a - d) + i (c + b)) / 2      (antilinear part).
"""
from __future__ import annotations

import numpy as np

from .scan_mismtach import phase_sweep_inputs


def _col(columns, c):
    columns = tuple(int(v) for v in columns)
    if c not in columns:
        raise ValueError(f"jac has no column {c} (columns {columns}): compute it with that wave in `waves`")
    return columns.index(c)


def mu_nu(jac, columns, out_wave: int, in_wave: int):
    """(mu, nu) of the block (out_wave <- in_wave): mu = ((a + d) + i(c - b))/2, nu = ((a - d) + i(c + b))/2 with
    M = [[a, b], [c, d]] the real 2x2 block (module docstring).  Arrays of the leading shape of jac."""
    J = np.asarray(jac, dtype=float)
    kr, ki = _col(columns, 2 * in_wave), _col(columns, 2 * in_wave + 1)
    a, b = J[..., 2 * out_wave, kr], J[..., 2 * out_wave, ki]
    c, d = J[..., 2 * out_wave + 1, kr], J[..., 2 * out_wave + 1, ki]
    return 0.5 * ((a + d) + 1j * (c - b)), 0.5 * ((a - d) + 1j * (c + b))


def signal_gain(jac, columns):
    """Phase-averaged small-signal gain of the signal, |mu|^2 + |nu|^2 (= ||M||_F^2 / 2) of the block
    (signal <- signal): the output signal power per unit input signal power, averaged over the input phase."""
    mu, nu = mu_nu(jac, columns, 2, 2)
    return np.abs(mu) ** 2 + np.abs(nu) ** 2


def idler_conversion(jac, columns):
    """Phase-averaged idler conversion, |mu|^2 + |nu|^2 of the block (idler <- signal): the output idler power per
    unit input signal power, averaged over the input phase."""
    mu, nu = mu_nu(jac, columns, 3, 2)
    return np.abs(mu) ** 2 + np.abs(nu) ** 2


def linear_response(jac, columns, dA0):
    """dA(L) = sum_w mu_{o,w} dA_w(0) + nu_{o,w} conj(dA_w(0)) for complex input perturbations dA0 [..., 4] (or [4],
    broadcast over the points).  A wave whose columns jac lacks must have dA0 = 0 there."""
    J = np.asarray(jac, dtype=float)
    dA0 = np.asarray(dA0, dtype=np.complex128)
    lead = J.shape[:-2]
    out = np.zeros(lead + (4,), dtype=np.complex128)
    cols = tuple(int(v) for v in columns)
    for w in range(4):
        x = dA0[..., w]
        if 2 * w not in cols or 2 * w + 1 not in cols:
            if np.any(x != 0):
                raise ValueError(f"dA0 perturbs wave {w}, whose columns jac does not have (columns {cols})")
            continue
        for o in range(4):
            mu, nu = mu_nu(J, cols, o, w)
            out[..., o] += mu * x + nu * np.conj(x)
    return out


def phase_gain(jac, columns, p_in, phase_in=None, phase_axis=(0.0,), phase_weights=(0.0, 0.0, 1.0, 0.0)):
    """Small-signal counterpart of `sweep_phase_gain_2d`'s gain: the inputs are `phase_sweep_inputs(p_in, phase_in,
    phase_axis, phase_weights)`, of which the signal and idler components are the perturbation dA(0)_k (the pumps
    are the operating point J was taken at, normally with zero seeds), and

        gain_lin[..., k] = |dA_3(L)_k|^2 / p_in[2],   dA(L)_k = linear_response(jac, columns, dA(0)_k).

    Returns dict(gain_lin [..., K], and over the phase axis numpy's nan-reductions gain_max = nanmax, gain_min =
    nanmin, idx_max / idx_min = nanargmax / nanargmin (-1 where all K are NaN), n_finite).  A J taken with zero
    seeds reproduces the full runs' gain in the limit of small seeds."""
    p0 = np.asarray(p_in, dtype=float)
    table, _, _ = phase_sweep_inputs(p0, phase_in, phase_axis, phase_weights)
    dA0 = table.copy()
    dA0[:, :2] = 0.0
    J = np.asarray(jac, dtype=float)
    lead = J.shape[:-2]
    K = dA0.shape[0]
    gain = np.empty(lead + (K,))
    for k in range(K):
        gain[..., k] = np.abs(linear_response(J, columns, dA0[k])[..., 2]) ** 2 / p0[2]
    fin = ~np.isnan(gain)
    n_fin = fin.sum(axis=-1).astype(np.int32)
    any_fin = n_fin > 0
    with np.errstate(invalid="ignore"):
        gmax = np.where(any_fin, np.max(np.where(fin, gain, -np.inf), axis=-1), np.nan)
        gmin = np.where(any_fin, np.min(np.where(fin, gain, np.inf), axis=-1), np.nan)
    imax = np.where(any_fin, np.argmax(np.where(fin, gain, -np.inf), axis=-1), -1).astype(np.int32)
    imin = np.where(any_fin, np.argmin(np.where(fin, gain, np.inf), axis=-1), -1).astype(np.int32)
    return {"gain_lin": gain, "gain_max": gmax, "gain_min": gmin, "idx_max": imax, "idx_min": imin,
            "n_finite": n_fin}


def pump_power_sensitivity(jac, columns, A0, A_end, pump=0):
    """d ln P3(L) / d ln P_pump(0): the relative change of the output signal power per relative change of the input
    power of pump `pump` (0, 1, or a sequence of both: scaled together).  Scaling P_pump(0) by (1 + e) scales
    A_pump(0) by (1 + e/2), so dA(0) = A_pump(0)/2 on that wave and

        d ln P3 / d ln P_pump = 2 Re(conj(A_3(L)) dA_3(L)) / |A_3(L)|^2,   dA(L) = linear_response(jac, columns, dA(0)).

    A0 [..., 4] or [4] is the input J was taken at, A_end [..., 4] its output.  Needs non-zero seeds (P3(L) > 0);
    it is the fiber-end power, not the sweep's max-over-samples metric."""
    A0 = np.asarray(A0, dtype=np.complex128)
    A_end = np.asarray(A_end, dtype=np.complex128)
    lead = np.asarray(jac).shape[:-2]
    dA0 = np.zeros(lead + (4,), dtype=np.complex128)
    for w in np.atleast_1d(pump).tolist():
        if w not in (0, 1):
            raise ValueError(f"pump must be 0, 1 or both, got {w}")
        dA0[..., w] = np.broadcast_to(A0[..., w], lead) / 2.0
    dA3 = linear_response(jac, columns, dA0)[..., 2]
    A3 = A_end[..., 2]
    with np.errstate(invalid="ignore", divide="ignore"):
        return 2.0 * np.real(np.conj(A3) * dA3) / np.abs(A3) ** 2
