"""oracle/transfer_ld.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Long-double reference for the small-signal transfer matrices J = dA(L)/dA(z0) of the 4-wave system: textbook RK4 of
the ODE of `yaman_model.rhs_yaman_simplified`, with its forward-mode tangent carried beside it, vectorised over a
batch of points.  It is written from the ODE and shares nothing with the kernels' tangent (`stage_tan()`) or with the
CPU models of it (tools/transfer_model.py, oracle/fast_kernel_model.py), so a wrong derivative term in those shows
up as a difference from it.

    dA_j/dz = f_j(A, z) = -(alpha/2) A_j + i gamma (2S - P_j) A_j + 2i gamma conj(A_m) C_j,    P_j = |A_j|^2, S = sum P,
    C_1 = C_2 = e A_3 A_4,  C_3 = C_4 = conj(e) A_1 A_2,  e = exp(i dbeta z),  m = partner of j (1<->2, 3<->4).

f is not complex-analytic, so its derivative along a complex tangent t is Df(A) t = (df/dA) t + (df/dconj(A)) conj(t)
with the Wirtinger derivatives (P_k = A_k conj(A_k))

    df_j/dA_k     = -(alpha/2) d_jk + i gamma [(2 - d_jk) conj(A_k) A_j + (2S - P_j) d_jk] + 2i gamma conj(A_m) dC_j/dA_k
    df_j/dconj(A_k) =                 i gamma (2 - d_jk) A_k A_j                       + 2i gamma d_km C_j.

The discrete map is the one the kernels are specified to compute: the FP64 inputs promoted as they are, the FP64 step
h = (z_max - z0) / n_steps, the abscissae z0 + i h (+ h/2, + h) formed in long double, and exp(i dbeta z) from
long-double cos / sin at every abscissa.  (The kernels realise the same phase factors in FP64 by a rotation
recurrence, re-synchronised every 32 steps.)

Needs numpy's longdouble to carry at least 63 mantissa bits (x86-64 Linux: the x87 80-bit format); anywhere else it
raises instead of silently computing in FP64."""
from __future__ import annotations

import numpy as np

from oracle.nwave_oracle import _require_extended_precision

_PARTNER = np.array([1, 0, 3, 2])


def _rhs_and_tangent(A, T, z, gamma, alpha, dbeta):
    """f(A, z) [B,4] and Df(A, z) T [B,4,nc] in long double."""
    LD = np.longdouble
    ph = dbeta * z
    e = np.empty(ph.shape, dtype=np.clongdouble)
    e.real, e.imag = np.cos(ph), np.sin(ph)
    ig = 1j * gamma[:, None]                                              # [B,1]
    P = A.real * A.real + A.imag * A.imag
    S = P.sum(axis=1, keepdims=True)
    Ac = np.conj(A)
    a1, a2, a3, a4 = A[:, 0], A[:, 1], A[:, 2], A[:, 3]
    C = np.stack([e * a3 * a4, e * a3 * a4, np.conj(e) * a1 * a2, np.conj(e) * a1 * a2], axis=1)
    Am = Ac[:, _PARTNER]                                                  # conj(A_m)
    f = (-alpha[:, None] / 2) * A + ig * ((2 * S - P) * A) + 2 * ig * (Am * C)

    B = A.shape[0]
    eye = np.eye(4, dtype=LD)
    own = 2 - eye                                                         # 2 - d_jk
    # dC_j/dA_k: C_1,2 = e A3 A4, C_3,4 = conj(e) A1 A2
    dC = np.zeros((B, 4, 4), dtype=np.clongdouble)
    dC[:, 0:2, 2] = (e * a4)[:, None]
    dC[:, 0:2, 3] = (e * a3)[:, None]
    dC[:, 2:4, 0] = (np.conj(e) * a2)[:, None]
    dC[:, 2:4, 1] = (np.conj(e) * a1)[:, None]
    Fa = (-alpha[:, None, None] / 2) * eye \
        + ig[:, :, None] * (own * (A[:, :, None] * Ac[:, None, :]) + (2 * S - P)[:, :, None] * eye) \
        + 2 * ig[:, :, None] * (Am[:, :, None] * dC)
    Fb = ig[:, :, None] * (own * (A[:, :, None] * A[:, None, :])) \
        + 2 * ig[:, :, None] * (C[:, :, None] * eye[_PARTNER][None, :, :])
    return f, Fa @ T + Fb @ np.conj(T)


def transfer_ld(A0, gamma, alpha, dbeta, *, z0=0.0, z_max, n_steps, columns=range(8)):
    """RK4 from z0 to z_max in n_steps equal steps for B points, with the tangent of each input component in `columns`.

    A0 complex [B,4] (or [4]): FP64 is promoted, clongdouble taken as it is (central differences of the map in long
    double); columns may be empty (the base map alone).  gamma, alpha, dbeta scalars or [B].  Returns (A_end clongdouble [B,4],
    J longdouble [B,8,nc]) in the conventions of fpa_transfer_out: J[b, r, k] = d y_r(z_max) / d y_{columns[k]}(z0),
    y = (Re A1, Im A1, ..., Re A4, Im A4)."""
    _require_extended_precision()
    LD = np.longdouble
    A0 = np.atleast_2d(np.asarray(A0))
    A0 = A0 if A0.dtype == np.clongdouble else A0.astype(np.complex128)
    B = A0.shape[0]
    gamma, alpha, dbeta = (np.broadcast_to(np.asarray(v, dtype=float), (B,)).astype(LD) for v in (gamma, alpha, dbeta))
    cols = [int(c) for c in columns]
    if any(c < 0 or c > 7 for c in cols) or len(set(cols)) != len(cols):
        raise ValueError(f"columns must be distinct integers in [0, 8), got {cols}")
    h = LD(float((z_max - z0) / n_steps))                                # the FP64 step, promoted
    z0 = LD(float(z0))
    half, sixth = LD(1) / 2, LD(1) / 6
    A = A0.astype(np.clongdouble)
    T = np.zeros((B, 4, len(cols)), dtype=np.clongdouble)
    for k, c in enumerate(cols):
        T[:, c // 2, k] = 1 if c % 2 == 0 else 1j

    def f(z, A, T):
        return _rhs_and_tangent(A, T, np.full(B, z, dtype=LD), gamma, alpha, dbeta)

    for i in range(n_steps):
        z = z0 + i * h
        k1, K1 = f(z, A, T)
        k2, K2 = f(z + half * h, A + (half * h) * k1, T + (half * h) * K1)
        k3, K3 = f(z + half * h, A + (half * h) * k2, T + (half * h) * K2)
        k4, K4 = f(z + h, A + h * k3, T + h * K3)
        A = A + (h * sixth) * (k1 + 2 * k2 + 2 * k3 + k4)
        T = T + (h * sixth) * (K1 + 2 * K2 + 2 * K3 + K4)
    J = np.empty((B, 8, len(cols)), dtype=LD)
    J[:, 0::2], J[:, 1::2] = T.real, T.imag
    return A, J
