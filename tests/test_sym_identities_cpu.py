"""CPU: the guarded symmetric z-loop of csrc/yaman4.cu (stage_sym_fast, fast_integrate<..., SYM, GUARD>).

stage_sym_fast() replaces two expressions of stage_sym() with exactly equal ones:
  1. c2g * S, S = (P1 + P1) + (P3 + P3), by c4g * T with T = P1 + P3 and c4g = c2g + c2g;
  2. in stage 2, Ui = fma(x3, y3, m3) (m3 = y3 x3) times the phase qh by m3 times q2 = qh + qh (the same for Vi).
Both can fail only when a doubling overflows, i.e. T >= 2^1023; the kernel folds the high word of every stage's T
into a guard and replays the run with stage_sym() when it reaches 0x7FE00000.  Checked here:
  * on a large sampled set and on edge cases (+-0, subnormals, components near 2^511, inf, NaN), with an exact FMA,
    every state where either identity differs raises the guard;
  * on the exact-FMA model of the kernel (oracle/fast_kernel_model.py), the guarded loop reproduces the stage_sym()
    loop bit for bit over runs that span phase re-synchronisations, lossy and lossless, without raising the guard;
  * a run driven to overflow raises the guard no later than the step whose finite check fires in the stage_sym() loop
    (so dropping that check from the guarded loop loses nothing: such runs are replayed)."""
import math
import random
import struct
from fractions import Fraction

import numpy as np
import pytest

from oracle import fast_kernel_model as M

GUARD_LIMIT = 0x7FE00000


def hi_word(v):
    """The high 32 bits of a double's pattern, as an unsigned number (the kernel's __double2hiint, cast)."""
    return struct.unpack("<Q", struct.pack("<d", v))[0] >> 32


def same_bits(a, b):
    return struct.pack("<d", a) == struct.pack("<d", b)


def fma_exact(a, b, c):
    """a*b + c with one rounding, exactly (rational arithmetic; float(Fraction) rounds to nearest even, subnormals
    included).  Non-finite operands follow IEEE through the unfused expression, which agrees with an FMA there."""
    if not (math.isfinite(a) and math.isfinite(b) and math.isfinite(c)):
        return a * b + c
    r = Fraction(a) * Fraction(b) + Fraction(c)
    if r == 0:                                   # the sign of an exact zero sum, as IEEE defines it
        return (a * b) + c if a * b != 0 else c + 0.0 if c != 0 else (a * b) + c
    try:
        return float(r)
    except OverflowError:
        return math.inf if r > 0 else -math.inf


# ------------------------------------------------------------------ the two stages, operation for operation
def stage_sym(inn, base, qr, qi, cg, c2g, cn, fma, loss=True):
    """stage_sym() of csrc/yaman4.cu; also returns S."""
    x1, y1, x3, y3 = inn
    P1 = fma(y1, y1, x1 * x1)
    P3 = fma(y3, y3, x3 * x3)
    S = (P1 + P1) + (P3 + P3)
    c2 = c2g * S
    G1, G3 = fma(-cg, P1, c2), fma(-cg, P3, c2)
    Ur, Ui = fma(-y3, y3, x3 * x3), fma(x3, y3, y3 * x3)
    Vr, Vi = fma(-y1, y1, x1 * x1), fma(x1, y1, y1 * x1)
    Wr, Wi = fma(-qi, Ui, qr * Ur), fma(qr, Ui, qi * Ur)
    Zr, Zi = fma(qi, Vi, qr * Vr), fma(qr, Vi, -(qi * Vr))
    b = [fma(cn, v, bb) for v, bb in zip(inn, base)] if loss else list(base)
    return [
        fma(-G1, y1, fma(y1, Wr, fma(-x1, Wi, b[0]))),
        fma(G1, x1, fma(x1, Wr, fma(y1, Wi, b[1]))),
        fma(-G3, y3, fma(y3, Zr, fma(-x3, Zi, b[2]))),
        fma(G3, x3, fma(x3, Zr, fma(y3, Zi, b[3]))),
    ], S


def stage_sym_fast(inn, base, qr, qi, q2r, q2i, cg, c4g, cn, dbl, fma, loss=True):
    """stage_sym_fast() of csrc/yaman4.cu; returns (out, high word of T)."""
    x1, y1, x3, y3 = inn
    P1 = fma(y1, y1, x1 * x1)
    P3 = fma(y3, y3, x3 * x3)
    T = P1 + P3
    c2 = c4g * T
    G1, G3 = fma(-cg, P1, c2), fma(-cg, P3, c2)
    Ur, m3 = fma(-y3, y3, x3 * x3), y3 * x3
    Vr, m1 = fma(-y1, y1, x1 * x1), y1 * x1
    if dbl:
        Wr, Wi = fma(-q2i, m3, qr * Ur), fma(q2r, m3, qi * Ur)
        Zr, Zi = fma(q2i, m1, qr * Vr), fma(q2r, m1, -(qi * Vr))
    else:
        Ui, Vi = fma(x3, y3, m3), fma(x1, y1, m1)
        Wr, Wi = fma(-qi, Ui, qr * Ur), fma(qr, Ui, qi * Ur)
        Zr, Zi = fma(qi, Vi, qr * Vr), fma(qr, Vi, -(qi * Vr))
    b = [fma(cn, v, bb) for v, bb in zip(inn, base)] if loss else list(base)
    return [
        fma(-G1, y1, fma(y1, Wr, fma(-x1, Wi, b[0]))),
        fma(G1, x1, fma(x1, Wr, fma(y1, Wi, b[1]))),
        fma(-G3, y3, fma(y3, Zr, fma(-x3, Zi, b[2]))),
        fma(G3, x3, fma(x3, Zr, fma(y3, Zi, b[3]))),
    ], hi_word(T)


# ------------------------------------------------------------------ the identities against the guard
def _component(rng):
    k = rng.random()
    if k < 0.15:
        e = rng.uniform(505, 513)                # squares near the overflow of T and of 2T
    elif k < 0.3:
        e = rng.uniform(-1074, -1000)            # subnormal squares and products
    elif k < 0.35:
        e = rng.uniform(-540, -520)              # products at the bottom of the normal range
    else:
        e = rng.uniform(-60, 60)
    return rng.choice((-1.0, 1.0)) * 2.0 ** e * rng.uniform(1.0, 2.0)


EDGE = [0.0, -0.0, 5e-324, -5e-324, 2.2250738585072014e-308, 1.4916681462400413e-154, 2.0 ** 511,
        2.0 ** 511 * (1 + 2 ** -52), 1.3407807929942596e154, -1.3407807929942596e154, 2.0 ** 512, math.inf,
        -math.inf, math.nan]


def _check_identities(x1, y1, x3, y3, c2g, qi, t):
    """(identity 1 differs, identity 2 differs, guard raised) for one state, both waves' pair products."""
    P1 = fma_exact(y1, y1, x1 * x1)
    P3 = fma_exact(y3, y3, x3 * x3)
    S, T = (P1 + P1) + (P3 + P3), P1 + P3
    c4g = c2g + c2g
    bad1 = not same_bits(c2g * S, c4g * T) and not (math.isnan(c2g * S) and math.isnan(c4g * T))
    bad2 = False
    for x, y in ((x3, y3), (x1, y1)):
        m = y * x
        U = fma_exact(x, y, m)
        o, n = fma_exact(-qi, U, t), fma_exact(-(qi + qi), m, t)
        bad2 |= not same_bits(o, n) and not (math.isnan(o) and math.isnan(n))
    return bad1, bad2, hi_word(T) >= GUARD_LIMIT


def test_every_state_where_an_identity_differs_raises_the_guard():
    rng = random.Random(20261021)
    cases = []
    for _ in range(60000):
        cases.append((_component(rng), _component(rng), _component(rng), _component(rng)))
    for a in EDGE:
        for b in EDGE:
            cases.append((a, b, _component(rng), _component(rng)))
            cases.append((_component(rng), _component(rng), a, b))
            cases.append((a, b, a, b))
    n1 = n2 = 0
    for x1, y1, x3, y3 in cases:
        c2g = 2.0 ** rng.uniform(-40, 0) * rng.uniform(1, 2)
        qi = rng.uniform(-1e-3, 1e-3)
        t = rng.uniform(-1.0, 1.0) * 2.0 ** rng.choice((-1070, 0, 500))
        bad1, bad2, flag = _check_identities(x1, y1, x3, y3, c2g, qi, t)
        assert flag or not (bad1 or bad2), (x1, y1, x3, y3, c2g, qi, t, bad1, bad2)
        n1 += bad1
        n2 += bad2
    # the sample reaches the states where the identities fail, so the guard is what keeps the bits
    assert n1 > 100 and n2 > 10, (n1, n2)


def test_guard_limit_is_where_doubling_T_overflows():
    below = np.nextafter(2.0 ** 1023, 0.0)
    assert math.isfinite(below + below) and hi_word(below) < GUARD_LIMIT
    assert math.isinf(2.0 ** 1023 + 2.0 ** 1023) and hi_word(2.0 ** 1023) == GUARD_LIMIT
    # a NaN of either sign, and inf, raise the guard as unsigned high words
    for v in (math.inf, math.nan, -math.nan, struct.unpack("<d", struct.pack("<Q", 0xFFF8000000000001))[0]):
        assert hi_word(v) >= GUARD_LIMIT


# ------------------------------------------------------------------ the z-loop, guarded against stage_sym()
def _loops(A1, A3, gamma, alpha, dbeta, z_max, n_steps):
    """The stage_sym() loop and the guarded loop on the exact-FMA model; per step: both states, the first bad step
    of the stage_sym() loop's finite check, and whether the guard has been raised."""
    fma = M.fma
    loss = alpha != 0.0
    h = z_max / n_steps
    w = [0.5 * h, h, h * (1.0 / 6.0)]
    cg = [wi * gamma for wi in w]
    c2g = [c + c for c in cg]
    c4g = [c + c for c in c2g]
    cn = [wi * (-0.5 * alpha) for wi in w]
    q0 = c2g[0]
    third, two_thirds, third_c = M.weights("shipped")
    rr, ri = math.cos(dbeta * (0.5 * h)), math.sin(dbeta * (0.5 * h))
    y = [A1.real, A1.imag, A3.real, A3.imag]
    g = list(y)
    qr, qi = q0, 0.0
    bad, guard, steps = -1, 0, []
    for i in range(n_steps):
        if i % M.RESYNC == 0:
            ang = dbeta * fma(float(i), h, 0.0)
            qr, qi = q0 * math.cos(ang), q0 * math.sin(ang)
        qhr, qhi = fma(-qi, ri, qr * rr), fma(qr, ri, qi * rr)
        q2r, q2i = qhr + qhr, qhi + qhi
        qfr, qfi = fma(-qhi, ri, qhr * rr), fma(qhr, ri, qhi * rr)
        q6r, q6i = qfr * third, qfi * third
        # stage_sym() loop, with the finite check
        ys, S = stage_sym(y, y, qr, qi, cg[0], c2g[0], cn[0], fma, loss)
        if not math.isfinite(S) and bad == -1 and i > 0 and not all(math.isfinite(v) for v in y):
            bad = i - 1
        acc = [fma(third, ys[j], y[j] * (-third)) for j in range(4)]
        yt, _ = stage_sym(ys, y, qhr, qhi, cg[0], c2g[0], cn[0], fma, loss)
        acc = [fma(two_thirds, yt[j], acc[j]) for j in range(4)]
        ys, _ = stage_sym(yt, y, q2r, q2i, cg[1], c2g[1], cn[1], fma, loss)
        acc = [fma(third_c, ys[j], acc[j]) for j in range(4)]
        y, _ = stage_sym(ys, acc, q6r, q6i, cg[2], c2g[2], cn[2], fma, loss)
        # the guarded loop
        gs, h1 = stage_sym_fast(g, g, qr, qi, q2r, q2i, cg[0], c4g[0], cn[0], False, fma, loss)
        acc = [fma(third, gs[j], g[j] * (-third)) for j in range(4)]
        gt, h2 = stage_sym_fast(gs, g, qhr, qhi, q2r, q2i, cg[0], c4g[0], cn[0], True, fma, loss)
        acc = [fma(two_thirds, gt[j], acc[j]) for j in range(4)]
        gs, h3 = stage_sym_fast(gt, g, q2r, q2i, q2r, q2i, cg[1], c4g[1], cn[1], False, fma, loss)
        acc = [fma(third_c, gs[j], acc[j]) for j in range(4)]
        g, h4 = stage_sym_fast(gs, acc, q6r, q6i, q2r, q2i, cg[2], c4g[2], cn[2], False, fma, loss)
        guard = max(guard, h1, h2, h3, h4)
        qr, qi = qfr, qfi
        steps.append((list(y), list(g), bad, guard >= GUARD_LIMIT))
    return steps


A1 = 0.5 ** 0.5 * np.exp(0.4j)
A3 = 1e-3 * np.exp(-1.1j)


@pytest.mark.parametrize("alpha", [1.15e-4, 0.0], ids=["lossy", "lossless"])
def test_guarded_loop_reproduces_stage_sym_bit_for_bit(alpha):
    # strong coupling (~25 dB of gain), 200 steps: six phase re-synchronisations
    steps = _loops(A1, A3, 11.5e-3, alpha, -2.1e-3, 2000.0, 200)
    assert abs(complex(*steps[-1][0][2:])) ** 2 / abs(A3) ** 2 > 10.0
    for y, g, bad, tripped in steps:
        assert not tripped and bad == -1
        assert all(same_bits(a, b) for a, b in zip(y, g))


def test_overflowing_run_raises_the_guard_before_the_finite_check_fires():
    """Negative loss drives the state to overflow, with the Kerr term and without it (gamma = 0, where T passes 2^1023
    with finite components).  Up to the step where the guard is raised the loops agree bit for bit."""
    for gamma, alpha, n_steps in ((11.5e-3, -40.0, 120), (0.0, -22.0, 120), (0.0, -40.0, 120)):
        steps = _loops(A1, A3, gamma, alpha, -2.1e-3, 37.4, n_steps)
        first_trip = next(i for i, s in enumerate(steps) if s[3])
        first_bad = next((i for i, s in enumerate(steps) if s[2] != -1), None)
        assert first_bad is None or first_trip <= first_bad + 1, (gamma, alpha, first_trip, first_bad)
        for y, g, _, tripped in steps[:first_trip]:
            assert all(same_bits(a, b) for a, b in zip(y, g))
