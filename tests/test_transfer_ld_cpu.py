"""CPU: the long-double transfer reference (oracle/transfer_ld.py) and the FP64 tangent model of the transfer kernels
(tools/transfer_model.py) against it, block by block.

A user reads single blocks of J: signal <- pump (pump_power_sensitivity), the seed blocks (signal_gain,
idler_conversion), the de-amplified quadrature (phase_gain).  Blocks span many decades: with a 1e-13 W seed the
signal <- pump block is ~1e-6 of the signal <- signal one.  A check of |got - ref| against max|J| says nothing about
the weak blocks, so every comparison here is per block: for output wave o and input wave w, (mu, nu) as
small_signal.mu_nu forms them, and |d mu| + |d nu| <= tol (|mu_ref| + |nu_ref|).

The cases of tests/test_gpu_transfer_ld.py are defined here: the bench's fiber (gamma = 11.5e-3 /W/m, 0.5 + 0.5 W pumps,
dz = 0.2 m, 500 m, 2 500 steps), kappa = dbeta + gamma (P1 + P2) across the gain band (|kappa| < 2r = 0.023 /m:
0 to ~45 dB), signal seeds of 1e-4, 1e-9, 1e-13 W and 0, idlers seeded on some points."""
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tools"))
import transfer_model as TM  # noqa: E402
from oracle import fast_kernel_model as FKM  # noqa: E402
from oracle import fwm_oracle as FO  # noqa: E402
from oracle import transfer_ld as TL  # noqa: E402

GAMMA, P_PUMP, DZ, L = 11.5e-3, 0.5, 0.2, 500.0
ALPHA = float(np.log(10) / 10 * 0.5 / 1000)             # 0.5 dB/km, the bench's loss
FLOOR = 1e-30         # |mu| + |nu| below which a non-zero block is not checked (no case has one)
# (kappa, signal seed W, idler seed W) of the batch points; point 0 is the depleted one (43 dB small-signal gain, a
# 1e-4 W seed: |nu_ss| / |mu_ss| = 0.98), points 3 and 8 have zero seeds (8 exactly-zero pump <-> seed blocks)
POINTS = [(0.0, 1e-4, 0.0), (0.0, 1e-9, 2e-10), (0.0, 1e-13, 0.0), (0.0, 0.0, 0.0), (0.0, 1e-13, 1e-13),
          (0.012, 1e-4, 1e-5), (0.012, 1e-9, 0.0), (0.02, 1e-13, 2e-14), (0.02, 0.0, 0.0), (-0.01, 1e-9, 1e-9),
          (0.05, 1e-4, 0.0), (0.05, 1e-13, 0.0)]
Z0 = 2000.0
KAPPA_FAR = 0.5       # the last point of the z0 case: dbeta z0 ~ 1e3 rad (outside the gain band)


def batch_case(case, n_steps=int(L / DZ)):
    """(A0 [B,4], dbeta [B], gamma, alpha, z0, z_max) of a batch case.  case: 'lossy' (UNIFORM 1), 'lossless'
    (UNIFORM 2), 'per_point' (UNIFORM 0: gamma and alpha per point, alpha = 0 on some), 'z0' (z0 = 2000 m, lossy)."""
    B = len(POINTS)
    b = np.arange(B)
    kappa = np.array([p[0] for p in POINTS])
    if case == "z0":
        kappa[-1] = KAPPA_FAR
    P = np.array([[P_PUMP, P_PUMP, ps, pi] for _, ps, pi in POINTS])
    ph = np.stack([0.1 + 0.3 * b, -0.2 - 0.5 * b, 0.3 + 0.7 * b, 0.05 - 0.4 * b], axis=1)
    A0 = np.sqrt(P) * np.exp(1j * ph)
    gamma, alpha = GAMMA, ALPHA
    if case == "lossless":
        alpha = 0.0
    elif case == "per_point":
        gamma = GAMMA * (1.0 + 0.04 * np.sin(b))
        alpha = ALPHA * (b % 3)
    dbeta = kappa - np.asarray(gamma) * 2 * P_PUMP
    z0 = Z0 if case == "z0" else 0.0
    return A0, dbeta, gamma, alpha, z0, z0 + n_steps * DZ


def _ld(x):
    return np.asarray(x).astype(np.longdouble)


def mu_nu_ld(J, o, w, columns=range(8)):
    """(mu, nu) of block (o <- w) of J [..., 8, nc] in long double, the formula of small_signal.mu_nu."""
    cols = list(columns)
    J = _ld(J)
    kr, ki = cols.index(2 * w), cols.index(2 * w + 1)
    a, b = J[..., 2 * o, kr], J[..., 2 * o, ki]
    c, d = J[..., 2 * o + 1, kr], J[..., 2 * o + 1, ki]
    return ((a + d) + 1j * (c - b)) / 2, ((a - d) + 1j * (c + b)) / 2


def block_errors(got, ref, columns=range(8)):
    """(err [B,4,nw], mag [B,4,nw], waves): per block |d mu| + |d nu| / (|mu_ref| + |nu_ref|) and |mu_ref| + |nu_ref|,
    output wave o, input wave waves[i] (the waves both of whose columns J has)."""
    cols = list(columns)
    waves = [w for w in range(4) if 2 * w in cols and 2 * w + 1 in cols]
    got, ref = np.asarray(got).reshape(-1, 8, len(cols)), _ld(ref).reshape(-1, 8, len(cols))
    err = np.zeros((got.shape[0], 4, len(waves)))
    mag = np.zeros((got.shape[0], 4, len(waves)), dtype=np.longdouble)
    for o in range(4):
        for i, w in enumerate(waves):
            mr, nr = mu_nu_ld(ref, o, w, cols)
            mg, ng = mu_nu_ld(got, o, w, cols)
            m = np.abs(mr) + np.abs(nr)
            mag[:, o, i] = m
            with np.errstate(invalid="ignore", divide="ignore"):
                err[:, o, i] = ((np.abs(mg - mr) + np.abs(ng - nr)) / m).astype(float)
    return err, mag, waves


def assert_blocks(got, ref, tol, what, floor=FLOOR, columns=range(8)):
    """J `got` [B,8,nc] (or [8,nc]) against the long-double `ref`, block by block: |d mu| + |d nu| <= tol (|mu_ref| +
    |nu_ref|) wherever |mu_ref| + |nu_ref| >= floor; the 2x2 blocks that are exactly 0 in ref are exactly 0 in got;
    got is finite.  A miss names the block, the point and the error.  Returns (largest error, weakest |mu| + |nu|
    checked)."""
    got = np.asarray(got, dtype=float)
    cols = list(columns)
    g3 = got.reshape(-1, 8, len(cols))
    r3 = _ld(ref).reshape(-1, 8, len(cols))
    assert g3.shape == r3.shape, (what, got.shape, np.shape(ref))
    if not np.isfinite(g3).all():
        raise AssertionError(f"{what}: non-finite J at point {int(np.argwhere(~np.isfinite(g3))[0, 0])}")
    err, mag, waves = block_errors(g3, r3, cols)
    for b in range(g3.shape[0]):
        for o in range(4):
            for i, w in enumerate(waves):
                rows = slice(2 * o, 2 * o + 2)
                k = [cols.index(2 * w), cols.index(2 * w + 1)]
                if mag[b, o, i] == 0:
                    if np.any(g3[b, rows][:, k] != 0):
                        raise AssertionError(f"{what}: block ({o} <- {w}) of point {b} is exactly 0 in the reference, "
                                             f"got {g3[b, rows][:, k].tolist()}")
                elif mag[b, o, i] >= floor and not err[b, o, i] <= tol:
                    raise AssertionError(f"{what}: block ({o} <- {w}) of point {b}: |d mu| + |d nu| = {err[b, o, i]:.3e} "
                                         f"of |mu| + |nu| = {float(mag[b, o, i]):.3e}, above {tol:g}")
    checked = mag >= floor
    return float(err[checked].max()), float(mag[checked].min())


def assert_waves(got, ref, tol, what):
    """A_end `got` [B,4] against the long-double `ref` per wave: |d A_j| <= tol |A_j|, exactly 0 where ref is."""
    got, ref = np.atleast_2d(got), np.atleast_2d(np.asarray(ref, dtype=np.clongdouble))
    a = np.abs(ref)
    zero = a == 0
    if np.any(got[zero] != 0):
        raise AssertionError(f"{what}: A_end not 0 where the reference is, at {np.argwhere(zero & (got != 0))[0]}")
    err = np.zeros(ref.shape)
    err[~zero] = (np.abs(got.astype(np.clongdouble) - ref)[~zero] / a[~zero]).astype(float)
    if not err.max() <= tol:
        b, j = np.argwhere(err == err.max())[0]
        raise AssertionError(f"{what}: A_end of wave {j} at point {b} off by {err[b, j]:.3e} of |A|, above {tol:g}")
    return float(err.max())


def model(A0, dbeta, gamma, alpha, z0, z_max, n_steps, pts, columns=range(8)):
    """tools/transfer_model.py on the points `pts` of a case: (A_end [n,4], J [n,8,nc])."""
    out = [TM.integrate(A0[b], np.broadcast_to(gamma, (len(A0),))[b], np.broadcast_to(alpha, (len(A0),))[b],
                        dbeta[b], z_max, n_steps, z0=z0, columns=columns) for b in pts]
    return np.array([o[0] for o in out]), np.array([o[1] for o in out])


def reference(A0, dbeta, gamma, alpha, z0, z_max, n_steps, pts=None, columns=range(8)):
    pts = slice(None) if pts is None else list(pts)
    g, a = (np.broadcast_to(v, (len(A0),))[pts] for v in (gamma, alpha))
    return TL.transfer_ld(A0[pts], g, a, dbeta[pts], z0=z0, z_max=z_max, n_steps=n_steps, columns=columns)


# ------------------------------------------------------------------ the reference itself
def test_transfer_ld_refuses_without_extended_precision(monkeypatch):
    """No silent fall-back: where numpy's longdouble is FP64, transfer_ld raises."""
    real = np.finfo

    class _F:
        nmant = 52

    monkeypatch.setattr(TL.np, "finfo", lambda t: _F() if t is np.longdouble else real(t))
    with pytest.raises(RuntimeError, match="mantissa bits"):
        TL.transfer_ld(np.ones(4, complex), 0.01, 0.0, 0.0, z_max=1.0, n_steps=2)


def test_reference_derivative_matches_its_own_central_differences():
    """The tangent of transfer_ld against fourth-order central differences of its own long-double base map (steps of
    1e-3 sqrt(W) on each input component): every block to 1e-8 of itself.  Measured 1.2e-11 (x86-64); a
    missing or wrong derivative term moves its blocks by far more."""
    A0, db, g, a, z0, _ = batch_case("lossy")
    pts = [0, 1, 3, 5, 9]
    A0, db, n, zm = A0[pts], db[pts], 100, 20.0
    A_end, J = TL.transfer_ld(A0, g, a, db, z_max=zm, n_steps=n)
    assert A_end.dtype == np.clongdouble and J.dtype == np.longdouble and J.shape == (5, 8, 8)
    eps = np.longdouble(1e-3)
    y0 = A0.astype(np.clongdouble)
    shifts = []
    for c in range(8):
        d = np.zeros(4, np.clongdouble)
        d[c // 2] = eps * (1 if c % 2 == 0 else 1j)
        shifts += [y0 + s * d for s in (2, 1, -1, -2)]
    B = len(pts)
    r, _ = TL.transfer_ld(np.concatenate(shifts), g, a, np.tile(db, 32), z_max=zm, n_steps=n, columns=())
    r = r.reshape(8, 4, B, 4)
    D = (8 * (r[:, 1] - r[:, 2]) - (r[:, 0] - r[:, 3])) / (12 * eps)        # [8 columns, B, 4]
    Jfd = np.empty_like(J)
    Jfd[:, 0::2], Jfd[:, 1::2] = D.real.transpose(1, 2, 0), D.imag.transpose(1, 2, 0)
    err, mag, _ = block_errors(Jfd, J)
    assert np.all(mag[1] > 0) and np.sum(mag[2] == 0) == 8                # point 3 (zero seeds): 8 zero blocks
    worst = float(err[mag > 0].max())
    assert worst <= 1e-8
    assert np.all(Jfd.astype(float)[mag.repeat(2, 1).repeat(2, 2) == 0] == 0)
    print(f"transfer_ld vs its own central differences: largest per-block error {worst:.1e}")


def test_reference_end_state_matches_the_fp64_oracle():
    """A_end of transfer_ld against the FP64 oracle's RK4 (oracle/fwm_oracle.py) on the same abscissae, per wave.
    Measured 4e-14 over 600 steps (the FP64 oracle's own rounding); 1e-12."""
    A0, db, g, a, z0, _ = batch_case("per_point")
    n, zm = 600, 120.0
    A_end, _ = reference(A0, db, g, a, z0, zm, n, columns=())
    h = (zm - z0) / n
    worst = 0.0
    for b in range(len(A0)):
        p = FO.YamanPoint(np.broadcast_to(g, (len(A0),))[b], np.broadcast_to(a, (len(A0),))[b], db[b])
        _, ys = FO.march_grid(FO.yaman_rhs_p, z0 + h * np.arange(n + 1), A0[b], p)
        worst = max(worst, assert_waves(ys[-1][None], A_end[b][None], 1e-12, f"point {b}"))
    print(f"transfer_ld A_end vs the FP64 oracle: largest per-wave error {worst:.1e}")


# ------------------------------------------------------------------ the FP64 model against the reference
# (case, steps, points, columns): the shortened GPU cases, and at the full 2 500 steps the depleted point and the point
# whose weak pump <- signal block (|mu| + |nu| ~ 1e-2) is the model's worst at that length (columns of the blocks only)
MODEL_RUNS = [("lossy", 100, [1, 4, 7, 10], range(8)), ("lossless", 100, [2, 9], range(8)),
              ("per_point", 100, [0, 5], range(8)), ("z0", 100, [6, 11], range(8)),
              ("lossy", 2500, [0], (0, 1)), ("per_point", 2500, [2], (4, 5))]


@pytest.mark.parametrize("case, n_steps, pts, columns", MODEL_RUNS, ids=[f"{c}-{n}-{p[0]}" for c, n, p, _ in MODEL_RUNS])
def test_fp64_model_matches_the_reference_block_by_block(case, n_steps, pts, columns):
    """tools/transfer_model.py (the kernels' operation order in FP64) against transfer_ld, per block and A_end per
    wave, to 1e-12.  Measured (x86-64) at the full 2 500 steps, every point of the per-point and z0 cases: at most
    7.4e-13 (point 2, the 1e-13 W seed at 43 dB, on pump 1 <- signal, |mu| + |nu| = 9e-3), 1.4e-13 on the depleted
    point; 5.2e-13 over 10 000 steps (the GPU file's long run).  The GPU file holds the kernels to 2e-10, two decades
    above the largest."""
    A0, db, g, a, z0, zm = batch_case(case, n_steps)
    Ae, J = model(A0, db, g, a, z0, zm, n_steps, pts, columns)
    Al, Jl = reference(A0, db, g, a, z0, zm, n_steps, pts, columns)
    worst, weakest = assert_blocks(J, Jl, 1e-12, f"{case} {n_steps} steps", columns=columns)
    we = assert_waves(Ae, Al, 1e-12, f"{case} {n_steps} steps")
    print(f"{case} {n_steps} steps, points {pts}: model vs long double, largest per-block error {worst:.1e}, "
          f"weakest block |mu| + |nu| = {weakest:.1e}; A_end {we:.1e}")


# ------------------------------------------------------------------ what the old criteria cannot see
def _stage_tan_cut(cut):
    """tools/transfer_model.stage_tan with one term of the tangent removed (cut = None: all terms, the same bits).
    Terms: loss cn A_j'; own Kerr G_j A_j'; Kerr derivative G_j' A_j (everywhere, or on the signal and idler rows
    only); the halves A3' A4 / A3 A4' of U' and A1' A2 / A1 A2' of V'; the q_r and q_i halves of W' = q U' and
    Z' = conj(q) V'; the conjugate-partner terms conj(A_m') {W|Z}."""
    def k(*names):
        return 0.0 if cut in names else 1.0

    def stage_tan(inn, t, tbase, qr, qi, cg, c2g, cn, loss=True):
        fma = FKM.fma
        x1, y1, x2, y2, x3, y3, x4, y4 = inn
        dx1, dy1, dx2, dy2, dx3, dy3, dx4, dy4 = t
        P1, P2, P3, P4 = fma(y1, y1, x1 * x1), fma(y2, y2, x2 * x2), fma(y3, y3, x3 * x3), fma(y4, y4, x4 * x4)
        S = (P1 + P2) + (P3 + P4)
        c2 = c2g * S
        G = [fma(-cg, P, c2) * k("own_kerr") for P in (P1, P2, P3, P4)]
        Ur, Ui = fma(-y3, y4, x3 * x4), fma(x3, y4, y3 * x4)
        Vr, Vi = fma(-y1, y2, x1 * x2), fma(x1, y2, y1 * x2)
        Wr, Wi = fma(-qi, Ui, qr * Ur), fma(qr, Ui, qi * Ur)
        Zr, Zi = fma(qi, Vi, qr * Vr), fma(qr, Vi, -(qi * Vr))
        h1, h2 = fma(y1, dy1, x1 * dx1), fma(y2, dy2, x2 * dx2)
        h3, h4 = fma(y3, dy3, x3 * dx3), fma(y4, dy4, x4 * dx4)
        hS = (h1 + h2) + (h3 + h4)
        d2 = (c2g + c2g) * hS
        kd = k("kerr_derivative")
        dG = [fma(-c2g, h, d2) * kd * (k("kerr_derivative_seed_rows") if j >= 2 else 1.0)
              for j, h in enumerate((h1, h2, h3, h4))]
        a, b = k("dU_A3'A4"), k("dU_A3A4'")
        dUr = fma(x3, b * dx4, fma(-y3, b * dy4, fma(-a * dy3, y4, (a * dx3) * x4)))
        dUi = fma(x3, b * dy4, fma(y3, b * dx4, fma(a * dy3, x4, (a * dx3) * y4)))
        a, b = k("dV_A1'A2"), k("dV_A1A2'")
        dVr = fma(x1, b * dx2, fma(-y1, b * dy2, fma(-a * dy1, y2, (a * dx1) * x2)))
        dVi = fma(x1, b * dy2, fma(y1, b * dx2, fma(a * dy1, x2, (a * dx1) * y2)))
        r, i = k("dW_qr"), k("dW_qi")
        dWr, dWi = fma(-qi * i, dUi, (qr * r) * dUr), fma(qr * r, dUi, (qi * i) * dUr)
        r, i = k("dZ_qr"), k("dZ_qi")
        dZr, dZi = fma(qi * i, dVi, (qr * r) * dVr), fma(qr * r, dVi, -((qi * i) * dVr))
        cn = cn * k("loss")
        p = k("conj_partner")
        out = []
        out += TM._wave(x1, y1, dx1, dy1, x2, y2, p * dx2, p * dy2, G[0], dG[0], Wr, Wi, dWr, dWi, cn, tbase[0], tbase[1], loss)
        out += TM._wave(x2, y2, dx2, dy2, x1, y1, p * dx1, p * dy1, G[1], dG[1], Wr, Wi, dWr, dWi, cn, tbase[2], tbase[3], loss)
        out += TM._wave(x3, y3, dx3, dy3, x4, y4, p * dx4, p * dy4, G[2], dG[2], Zr, Zi, dZr, dZi, cn, tbase[4], tbase[5], loss)
        out += TM._wave(x4, y4, dx4, dy4, x3, y3, p * dx3, p * dy3, G[3], dG[3], Zr, Zi, dZr, dZi, cn, tbase[6], tbase[7], loss)
        return out

    return stage_tan


CUTS = ["loss", "own_kerr", "kerr_derivative", "kerr_derivative_seed_rows", "dU_A3'A4", "dU_A3A4'", "dV_A1'A2",
        "dV_A1A2'", "dW_qr", "dW_qi", "dZ_qr", "dZ_qi", "conj_partner"]


def test_per_block_criterion_catches_a_planted_bug(monkeypatch):
    """The model with i G_j' A_j dropped from the signal and idler rows: the signal <- pump-1 block is wrong by tens of
    percent, yet with a 1e-16 W seed J moves by ~2e-8 of max|J|, inside both finite-difference criteria of the old
    tests (1e-7 of max|J| on the CPU, 1e-6 on the GPU).  The per-block check against transfer_ld fails, on that block."""
    A0 = np.sqrt([0.4, 0.3, 1e-16, 2e-17]) * np.exp(1j * np.array([0.1, 0.3, -0.2, 0.7]))
    g, al, db, zm, n = 0.02, 2e-3, 0.004, 80.0, 70
    _, J = TM.integrate(A0, g, al, db, zm, n)
    monkeypatch.setattr(TM, "stage_tan", _stage_tan_cut("kerr_derivative_seed_rows"))
    _, Jb = TM.integrate(A0, g, al, db, zm, n)
    monkeypatch.undo()
    y0 = A0.view(np.float64)
    Jfd = np.empty((8, 8))
    for c in range(8):
        eps = 1e-6 * abs(y0[c])                                            # the CPU file's step
        yp, ym = y0.copy(), y0.copy()
        yp[c] += eps
        ym[c] -= eps
        Jfd[:, c] = (FKM.integrate(yp.view(np.complex128), g, al, db, zm, n)[-1].view(np.float64) -
                     FKM.integrate(ym.view(np.complex128), g, al, db, zm, n)[-1].view(np.float64)) / (2 * eps)
    M = np.max(np.abs(J))
    old = np.max(np.abs(Jb - Jfd)) / M
    assert old <= 1e-7 and np.max(np.abs(Jb - J)) / M <= 1e-7              # the old criteria pass
    _, Jl = TL.transfer_ld(A0, g, al, db, z_max=zm, n_steps=n)
    assert_blocks(J, Jl, 1e-12, "the model")
    err, _, _ = block_errors(Jb, Jl)
    assert err[0, 2, 0] > 0.1 and err[0, 2, 0] == err.max()
    with pytest.raises(AssertionError, match=r"block \(2 <- 0\) of point 0"):
        assert_blocks(Jb, Jl, 2e-10, "planted bug")
    print(f"planted bug: {old:.1e} of max|J| against finite differences; per block {err[0, 2, 0]:.2f} on signal <- pump 1")


def test_every_tangent_term_is_needed(monkeypatch):
    """Remove each term of stage_tan in turn: every removal fails the per-block check against transfer_ld (at the GPU
    file's 2e-10) on at least one point of the GPU file's lossy case, shortened to 20 steps.  The points include seeded
    idlers: the A3' A4 / A3 A4' halves of U' differ only when both seeds are non-zero."""
    pts = [1, 5, 9]
    n = 20
    A0, db, g, a, z0, zm = batch_case("lossy", n)
    _, Jl = reference(A0, db, g, a, z0, zm, n, pts)
    _, J = model(A0, db, g, a, z0, zm, n, pts)
    monkeypatch.setattr(TM, "stage_tan", _stage_tan_cut(None))
    _, J_same = model(A0, db, g, a, z0, zm, n, pts)
    assert J_same.tobytes() == J.tobytes()
    assert_blocks(J, Jl, 1e-12, "the model")
    missed, seen = [], {}
    for cut in CUTS:
        monkeypatch.setattr(TM, "stage_tan", _stage_tan_cut(cut))
        _, Jc = model(A0, db, g, a, z0, zm, n, pts)
        err, mag, _ = block_errors(Jc, Jl)
        seen[cut] = float(np.nan_to_num(err[mag > 0], nan=np.inf).max())
        try:
            assert_blocks(Jc, Jl, 2e-10, cut)
            missed.append(cut)
        except AssertionError:
            pass
    print("largest per-block error with the term removed: " + ", ".join(f"{c} {e:.1e}" for c, e in seen.items()))
    assert not missed, f"removing {missed} passes the per-block check"
