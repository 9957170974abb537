"""CPU: the N-wave oracle line by line, down to cascaded sidebands 40 decades below the pumps.

A comb user reads the weak lines: sidebands that start at exactly 0 and end 10 to 40 decades below the pumps.  A check
of |got - ref| against the strongest line of the run says nothing about them.  Here the FP64 oracle (`march`) is
compared per line with its long-double restatement (`march_ld`), which is what tests/test_gpu_nwave_lines.py holds the
kernels to; and a test shows that the per-line criterion catches an error the trace-maximum criterion does not.

The plans (also used by the GPU file):
  (a) BASELINE config 2, lines -10..10: pumps +-5 at 0.5 W, signal +1 at 1e-5 W, the rest 0.  Every seed is on an odd
      line and k + l - m of odd lines is odd, so the 11 even lines stay exactly 0.
  (b) BASELINE config 5, lines -32..31: pumps +-4 at 1 W, signal +1 at 1e-6 W, the rest 0.
  (c) lines 0, 2, .., 126 (span 127): pumps at 56 and 72 (1 W), signal at 66 (1e-6 W), the rest 0.  Two ADJACENT
      pumps alone make the lines below ~1e-15 ill-conditioned: a 1e-15 change of one pump moves them by 14 % in the
      long-double march, and the FP64 oracle misses that march by up to a factor 460 there -- no FP64 implementation
      can meet a per-line bound on such a case.
  (d) lines 0..23 and 168..191 (span 192): pumps at 8 and 16 (0.5 W), signal at 11 (1e-6 W).  k + l - m of the low
      cluster never reaches the high one: its 24 lines stay exactly 0.
"""
import numpy as np
import pytest

from oracle import nwave_oracle as O

W5, DW5 = 2 * np.pi * 299792458.0 / 1550e-9, 2 * np.pi * 100e9
BETA5 = (-2.57e-29, 3.30e-41, -1.63e-55)
N_STEPS, DZ = 40, 0.1
FLOOR = 1e-100        # below it a product of three amplitudes leaves the FP64 normal range: out of scope

PLANS = {   # lines, centre line of the dispersion expansion, seeded lines {index: W}
    "a": (list(range(-10, 11)), None, {5: 0.5, 15: 0.5, 11: 1e-5}),
    "b": (list(range(-32, 32)), 0, {28: 1.0, 36: 1.0, 33: 1e-6}),
    "c": (list(range(0, 127, 2)), 63, {28: 1.0, 36: 1.0, 33: 1e-6}),
    "d": (list(range(0, 24)) + list(range(168, 192)), 96, {8: 0.5, 16: 0.5, 11: 1e-6}),
}
ZERO_LINES = {"a": list(range(0, 21, 2)), "d": list(range(24, 48))}    # exactly 0 for the whole run


def plan_case(fpa, golden, name):
    """(plan, beta, A0, gamma, alpha) of plan `name`; A0 real (the phases of a batch are the caller's)."""
    nw = fpa.nwave
    lines, centre, seeds = PLANS[name]
    if name == "a":
        wc, wd = golden["b1_sym"][0], golden["b1_sym"][1]
        plan = nw.uniform_comb_plan(wc, wd / 5.0, lines)
        disp = fpa.dispersion.DispersionParams(omega_ref=wc, beta2=golden["b1_beta"][0], beta3=golden["b1_beta"][1],
                                               beta4=golden["b1_beta"][2])
        gamma, alpha = (float(v) for v in golden["b1_gamma_alpha"])
    else:
        plan = nw.uniform_comb_plan(W5 - centre * DW5, DW5, lines)
        disp = fpa.dispersion.DispersionParams(omega_ref=W5, beta2=BETA5[0], beta3=BETA5[1], beta4=BETA5[2])
        gamma, alpha = 11.5e-3, 2e-4
    p = np.zeros(plan.n_waves)
    for j, w in seeds.items():
        p[j] = w
    return plan, nw.beta_per_wave(plan, disp), np.sqrt(p).astype(complex), gamma, alpha


def table_list(plan):
    t = plan.table
    return np.stack([t["k"], t["l"], t["m"], t["weight"]], axis=1).astype(np.int64), plan.row_ptr.tolist()


def line_errors(got, ref, floor=FLOOR):
    """Per-line relative error |got - ref| / |ref| of a kernel or FP64 result `got` against the long-double `ref`
    (same shape, [..., N]), where |ref| >= floor.  Returns (err, checked): err is 0 where not checked."""
    ref = np.asarray(ref, dtype=np.clongdouble)
    a = np.abs(ref)
    checked = a >= floor
    err = np.zeros(ref.shape)
    d = np.abs(np.asarray(got).astype(np.clongdouble) - ref)
    err[checked] = (d[checked] / a[checked]).astype(float)
    return err, checked


def assert_lines(got, ref, tol, what, floor=FLOOR):
    """got [S, N] (samples x lines) or [N] against the long-double ref: the per-line relative error is <= tol wherever
    |ref| >= floor, got == 0 exactly where ref == 0 and got != 0 wherever |ref| >= floor.  A miss names the line and
    the first sample where it occurs.  Returns (largest error, weakest |ref| checked)."""
    got, ref = np.atleast_2d(got), np.atleast_2d(np.asarray(ref, dtype=np.clongdouble))
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    err, checked = line_errors(got, ref, floor)
    for bad, kind in ((err > tol, f"relative error above {tol:g}"), ((ref == 0) & (got != 0), "not 0 where ref == 0"),
                      (checked & (got == 0), "0 where |ref| >= floor")):
        if bad.any():
            s, n = np.argwhere(bad)[np.argmin(np.argwhere(bad)[:, 0])]
            raise AssertionError(f"{what}: {kind} -- line {n}, first at sample {s}: got {got[s, n]!r}, "
                                 f"ref {complex(ref[s, n])!r}, rel err {err[s, n]:.3e}; {int(bad.sum())} misses in all")
    return float(err.max()), float(np.abs(ref[checked]).min()) if checked.any() else float("nan")


@pytest.fixture(scope="module")
def refs(fpa, golden):
    """Per plan (a), (b): case, FP64 march and long-double march, 40 steps of 0.1 m, every step saved."""
    out = {}
    for name in ("a", "b"):
        plan, beta, A0, gamma, alpha = plan_case(fpa, golden, name)
        tab, rows = table_list(plan)
        kw = dict(z_max=N_STEPS * DZ, n_steps=N_STEPS)
        out[name] = (plan, beta, A0, gamma, alpha, O.march(A0, gamma, alpha, beta, tab, rows, **kw)[1],
                     O.march_ld(A0, gamma, alpha, beta, tab, rows, **kw)[1])
    return out


def test_march_ld_is_extended_precision_and_matches_march_on_a_strong_run(fpa, golden):
    """march_ld returns long-double states on march's abscissae, and on a run with every line seeded (no weak lines)
    agrees with the FP64 march to its rounding."""
    assert np.finfo(np.longdouble).nmant >= 63
    table, rows = O.enumerate_triplets(list(range(-6, 7)))
    rng = np.random.default_rng(7)
    A0 = np.sqrt(rng.uniform(1e-3, 0.3, 13)) * np.exp(1j * rng.uniform(0, 2 * np.pi, 13))
    beta = rng.uniform(-2.0, 2.0, 13)
    kw = dict(z0=0.3, z_max=2.3, n_steps=20, save_every=3)
    z, A = O.march(A0, 0.02, 1e-4, beta, table, rows, **kw)
    zl, Al = O.march_ld(A0, 0.02, 1e-4, beta, table, rows, **kw)
    assert Al.dtype == np.clongdouble and Al.shape == A.shape == (7, 13)
    assert zl.tobytes() == z.tobytes()
    assert np.array_equal(Al[0], A0)
    err, checked = line_errors(A, Al)
    assert checked.all() and err.max() < 1e-13
    _, _, st = O.march_ld(A0, 0.02, 1e-4, beta, table, rows, check=True, **kw)
    assert st == -1


@pytest.mark.parametrize("name", ["a", "b"])
def test_fp64_oracle_is_accurate_line_by_line(refs, name):
    """The FP64 oracle against the long-double march, every line at every step, zero-seeded lines included.

    Measured (x86-64, numpy 2.3): plan (b) 8.2e-14 at step 2 on line +29 (the first steps of the cascade: lines
    near 1e-24, made by the RK4 stages out of nothing), 1.2e-14 at the end; plan (a) 8e-16.  Hence 1e-12 on every
    sample and 1e-13 on the end state.  Plan (b) spans 40 decades of line power at the end (7e-41 .. 1 W); plan (a)
    spans 23 over the run (5e-24 .. 0.5 W) and keeps its 11 even lines at exactly 0."""
    plan, beta, A0, gamma, alpha, A, Al = refs[name]
    assert Al.shape == (N_STEPS + 1, plan.n_waves)
    worst, _ = assert_lines(A, Al, 1e-12, f"plan ({name}) FP64 oracle")
    end, weakest = assert_lines(A[-1], Al[-1], 1e-13, f"plan ({name}) FP64 oracle, end state")
    P = np.abs(Al.astype(np.complex128)) ** 2
    if name == "b":
        assert (Al[-1] != 0).all() and P[-1].max() / P[-1].min() > 1e35
    else:
        assert (Al[:, ZERO_LINES["a"]] == 0).all() and (Al[1:, 1::2] != 0).all()
        assert P.max() / P[P > 0].min() > 1e20
    print(f"plan ({name}): FP64 oracle vs long double, largest per-line error {worst:.1e} (end {end:.1e}); "
          f"weakest line at the end {weakest ** 2:.1e} W")


def test_per_line_criterion_catches_what_the_trace_maximum_does_not(refs):
    """The oracle with the entry (n; k, l, m) = (-32; -24, -4, +4) of plan (b) removed -- the main source of the
    outermost line -- passes the old criterion, |got - ref| <= 1e-12 max|ref| over the trace, and fails the per-line
    one on that line by many orders of magnitude."""
    plan, beta, A0, gamma, alpha, _, Al = refs["b"]
    tab, rows = table_list(plan)
    g = np.asarray(PLANS["b"][0])
    row0 = np.arange(rows[0], rows[1])
    hit = [e for e in row0 if sorted(g[tab[e, :2]].tolist()) == [-24, -4] and g[tab[e, 2]] == 4]
    assert len(hit) == 1 and g[0] == -32
    cut = np.delete(tab, hit[0], axis=0)
    cut_rows = [0] + [r - 1 for r in rows[1:]]
    A = O.march(A0, gamma, alpha, beta, cut, cut_rows, z_max=N_STEPS * DZ, n_steps=N_STEPS)[1]
    ref = Al.astype(np.complex128)
    assert np.abs(A - ref).max() < 1e-12 * np.abs(ref).max()              # the old criterion passes
    err, checked = line_errors(A, Al)
    assert checked[1:].all()                                               # every line lit from step 1 on
    assert err[-1, 0] > 1e-2 and np.argmax(err.max(axis=0)) == 0           # the new one fails, on line -32
    with pytest.raises(AssertionError, match="line 0,"):
        assert_lines(A, Al, 1e-11, "dropped entry")
    print(f"dropped entry: old criterion {np.abs(A - ref).max() / np.abs(ref).max():.1e} of the trace maximum, "
          f"per-line error on line -32 at the end {err[-1, 0]:.1e}")


def test_march_ld_refuses_without_extended_precision(monkeypatch):
    """No silent fall-back: where numpy's longdouble is FP64, march_ld raises."""
    real = np.finfo

    class _F:
        nmant = 52

    monkeypatch.setattr(O.np, "finfo", lambda t: _F() if t is np.longdouble else real(t))
    with pytest.raises(RuntimeError, match="mantissa bits"):
        O.march_ld(np.ones(3, complex), 0.01, 0.0, np.zeros(3), [], [0, 0, 0, 0], z_max=1.0, n_steps=2)
