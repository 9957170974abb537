"""tools/transfer_model.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

CPU model of the transfer kernels (csrc/yaman4.cu: `stage_tan()`, `Tangent` and the z-loop of `fast_integrate`):
the exact-FMA tangent of oracle/fast_kernel_model.py, in stage_tan()'s operation order.  The base trajectory is
fast_kernel_model's own (its `stage` and `fma`), the tangent columns are carried beside it with the base run's
phase factors and the same RK4 combination weights, so the result is the exact derivative of the discrete map the
library integrates.  Pure-Python loops: small cases only.
"""
from __future__ import annotations

import math
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

from oracle.fast_kernel_model import RESYNC, fma, stage, weights  # noqa: E402


def _wave(xj, yj, dxj, dyj, xm, ym, dxm, dym, G, dG, Cr, Ci, dCr, dCi, cn, tbr, tbi, loss):
    r = fma(cn, dxj, tbr) if loss else tbr
    i = fma(cn, dyj, tbi) if loss else tbi
    r = fma(-G, dyj, fma(-dG, yj, fma(ym, dCr, fma(dym, Cr, fma(-xm, dCi, fma(-dxm, Ci, r))))))
    i = fma(G, dxj, fma(dG, xj, fma(xm, dCr, fma(dxm, Cr, fma(ym, dCi, fma(dym, Ci, i))))))
    return r, i


def stage_tan(inn, t, tbase, qr, qi, cg, c2g, cn, loss=True):
    """tout = tbase + c*Df(in)*t -- the operation order of `stage_tan()` in csrc/yaman4.cu."""
    x1, y1, x2, y2, x3, y3, x4, y4 = inn
    dx1, dy1, dx2, dy2, dx3, dy3, dx4, dy4 = t
    P1, P2, P3, P4 = fma(y1, y1, x1 * x1), fma(y2, y2, x2 * x2), fma(y3, y3, x3 * x3), fma(y4, y4, x4 * x4)
    S = (P1 + P2) + (P3 + P4)
    c2 = c2g * S
    G1, G2, G3, G4 = (fma(-cg, P, c2) for P in (P1, P2, P3, P4))
    Ur, Ui = fma(-y3, y4, x3 * x4), fma(x3, y4, y3 * x4)
    Vr, Vi = fma(-y1, y2, x1 * x2), fma(x1, y2, y1 * x2)
    Wr, Wi = fma(-qi, Ui, qr * Ur), fma(qr, Ui, qi * Ur)
    Zr, Zi = fma(qi, Vi, qr * Vr), fma(qr, Vi, -(qi * Vr))
    h1, h2 = fma(y1, dy1, x1 * dx1), fma(y2, dy2, x2 * dx2)
    h3, h4 = fma(y3, dy3, x3 * dx3), fma(y4, dy4, x4 * dx4)
    hS = (h1 + h2) + (h3 + h4)
    d2 = (c2g + c2g) * hS
    dG1, dG2, dG3, dG4 = (fma(-c2g, h, d2) for h in (h1, h2, h3, h4))
    dUr = fma(x3, dx4, fma(-y3, dy4, fma(-dy3, y4, dx3 * x4)))
    dUi = fma(x3, dy4, fma(y3, dx4, fma(dy3, x4, dx3 * y4)))
    dVr = fma(x1, dx2, fma(-y1, dy2, fma(-dy1, y2, dx1 * x2)))
    dVi = fma(x1, dy2, fma(y1, dx2, fma(dy1, x2, dx1 * y2)))
    dWr, dWi = fma(-qi, dUi, qr * dUr), fma(qr, dUi, qi * dUr)
    dZr, dZi = fma(qi, dVi, qr * dVr), fma(qr, dVi, -(qi * dVr))
    out = []
    out += _wave(x1, y1, dx1, dy1, x2, y2, dx2, dy2, G1, dG1, Wr, Wi, dWr, dWi, cn, tbase[0], tbase[1], loss)
    out += _wave(x2, y2, dx2, dy2, x1, y1, dx1, dy1, G2, dG2, Wr, Wi, dWr, dWi, cn, tbase[2], tbase[3], loss)
    out += _wave(x3, y3, dx3, dy3, x4, y4, dx4, dy4, G3, dG3, Zr, Zi, dZr, dZi, cn, tbase[4], tbase[5], loss)
    out += _wave(x4, y4, dx4, dy4, x3, y3, dx3, dy3, G4, dG4, Zr, Zi, dZr, dZi, cn, tbase[6], tbase[7], loss)
    return out


def integrate(A0, gamma, alpha, dbeta, z_max, n_steps, *, z0=0.0, columns=range(8)):
    """The transfer kernel's z-loop for one point from z0 to z_max: returns (A_end complex[4], J [8, nc]) with
    J[r, k] = d y_r(L) / d y_{columns[k]}(z0), y = (Re A1, Im A1, ..., Re A4, Im A4).  alpha == 0 takes the
    lossless stage (no loss FMAs), as the kernels do for uniform lossless physics."""
    loss = alpha != 0.0
    h = (z_max - z0) / n_steps
    w = [0.5 * h, h, h * (1.0 / 6.0)]
    nha = -0.5 * alpha
    cg = [wi * gamma for wi in w]
    c2g = [c + c for c in cg]
    cn = [wi * nha for wi in w]
    q0 = c2g[0]
    third, two_thirds, third_c = weights("shipped")
    y = []
    for a in np.asarray(A0, dtype=np.complex128):
        y += [float(a.real), float(a.imag)]
    cols = list(columns)
    T = [[1.0 if j == c else 0.0 for j in range(8)] for c in cols]
    rr, ri = math.cos(dbeta * (0.5 * h)), math.sin(dbeta * (0.5 * h))
    qr, qi = q0, 0.0
    for i in range(n_steps):
        if i % RESYNC == 0:
            ang = dbeta * fma(float(i), h, z0)
            qr, qi = q0 * math.cos(ang), q0 * math.sin(ang)
        qhr, qhi = fma(-qi, ri, qr * rr), fma(qr, ri, qi * rr)
        q2r, q2i = qhr + qhr, qhi + qhi
        qfr, qfi = fma(-qhi, ri, qhr * rr), fma(qhr, ri, qhi * rr)
        q6r, q6i = qfr * third, qfi * third
        ys = _stage(y, y, qr, qi, cg[0], c2g[0], cn[0], loss)
        acc = [fma(third, ys[j], y[j] * (-third)) for j in range(8)]
        yt = _stage(ys, y, qhr, qhi, cg[0], c2g[0], cn[0], loss)
        acc = [fma(two_thirds, yt[j], acc[j]) for j in range(8)]
        ys2 = _stage(yt, y, q2r, q2i, cg[1], c2g[1], cn[1], loss)
        acc = [fma(third_c, ys2[j], acc[j]) for j in range(8)]
        yn = _stage(ys2, acc, q6r, q6i, cg[2], c2g[2], cn[2], loss)
        for k, t in enumerate(T):
            ts = stage_tan(y, t, t, qr, qi, cg[0], c2g[0], cn[0], loss)
            ta = [fma(third, ts[j], t[j] * (-third)) for j in range(8)]
            tt = stage_tan(ys, ts, t, qhr, qhi, cg[0], c2g[0], cn[0], loss)
            ta = [fma(two_thirds, tt[j], ta[j]) for j in range(8)]
            ts = stage_tan(yt, tt, t, q2r, q2i, cg[1], c2g[1], cn[1], loss)
            ta = [fma(third_c, ts[j], ta[j]) for j in range(8)]
            T[k] = stage_tan(ys2, ts, ta, q6r, q6i, cg[2], c2g[2], cn[2], loss)
        y = yn
        qr, qi = qfr, qfi
    A_end = np.array([complex(y[2 * j], y[2 * j + 1]) for j in range(4)])
    return A_end, np.array(T).T


def _stage(inn, base, qr, qi, cg, c2g, cn, loss):
    """fast_kernel_model.stage, or its lossless form (cn == 0 adds exact zeros: same bits either way)."""
    return stage(inn, base, qr, qi, cg, c2g, cn if loss else 0.0)
