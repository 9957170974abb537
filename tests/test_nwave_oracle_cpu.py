"""CPU: the N-wave oracle's z0 start and status (oracle/nwave_oracle.py), and the oracle itself at the shapes the GPU
coverage tests (tests/test_gpu_nwave_coverage.py) trust it with: spans beyond 128, a random table."""
import warnings

import numpy as np
import pytest

from oracle import nwave_oracle as O


def _old_march(A0, gamma, alpha, beta, table, rows, *, z_max, n_steps, save_every=1, fast=True):
    """march() as it was before it took z0 and check: existing callers must keep these bits."""
    beta = np.asarray(beta, dtype=float)
    rows = np.asarray(rows)
    tab_arr = np.asarray(table, dtype=np.int64).reshape(-1, 4)
    f = (lambda z, y: O.nwave_rhs_fast(z, y, gamma, alpha, beta, tab_arr, rows)) if fast else \
        (lambda z, y: O.nwave_rhs(z, y, gamma, alpha, beta, table, rows))
    grid = np.linspace(0.0, z_max, n_steps + 1)
    y = np.asarray(A0, dtype=np.complex128).copy()
    zs, ys = [grid[0]], [y.copy()]
    for i in range(n_steps):
        z, h = grid[i], grid[i + 1] - grid[i]
        k1 = f(z, y)
        k2 = f(z + 0.5 * h, y + 0.5 * h * k1)
        k3 = f(z + 0.5 * h, y + 0.5 * h * k2)
        k4 = f(z + h, y + h * k3)
        y = y + (h / 6.0) * (k1 + 2.0 * k2 + 2.0 * k3 + k4)
        if (i + 1) % save_every == 0:
            zs.append(grid[i + 1])
            ys.append(y.copy())
    return np.array(zs), np.array(ys)


def _case(lines, seed, lo=1e-3, hi=1e-1):
    table, rows = O.enumerate_triplets(lines)
    N = len(lines)
    rng = np.random.default_rng(seed)
    A0 = np.sqrt(rng.uniform(lo, hi, N)) * np.exp(1j * rng.uniform(0, 2 * np.pi, N))
    beta = rng.uniform(-20.0, 20.0, N)
    return A0, beta, table, rows


def test_default_march_keeps_its_bits():
    A0, beta, table, rows = _case(list(range(-10, 11)), 1)
    for fast in (True, False):
        for save_every in (1, 7):
            old = _old_march(A0, 0.02, 1e-4, beta, table, rows, z_max=3.0, n_steps=30, save_every=save_every, fast=fast)
            new = O.march(A0, 0.02, 1e-4, beta, table, rows, z_max=3.0, n_steps=30, save_every=save_every, fast=fast)
            explicit = O.march(A0, 0.02, 1e-4, beta, table, rows, z_max=3.0, n_steps=30, save_every=save_every, fast=fast,
                               z0=0.0, check=True)
            for a, b in ((old, new), (old, explicit[:2])):
                assert a[0].tobytes() == b[0].tobytes() and a[1].tobytes() == b[1].tobytes()
            assert explicit[2] == -1


def test_z0_enters_the_phases():
    """beta = 0: the system is autonomous, a march from z0 = 5 is the march from 0 (to the rounding of the grid);
    beta != 0: the two differ by far more than the GPU tests' 1e-12 tolerance."""
    A0, beta, table, rows = _case(list(range(0, 24)) + list(range(40, 48)), 2)
    kw = dict(n_steps=40, save_every=5)
    z5, a5 = O.march(A0, 0.02, 1e-4, np.zeros_like(beta), table, rows, z0=5.0, z_max=9.0, **kw)
    z0, a0 = O.march(A0, 0.02, 1e-4, np.zeros_like(beta), table, rows, z_max=4.0, **kw)
    assert np.allclose(z5 - 5.0, z0, rtol=0, atol=1e-14) and z5[0] == 5.0 and z5[-1] == 9.0
    scale = np.abs(a0).max()
    assert np.abs(a5 - a0).max() < 1e-13 * scale
    b5 = O.march(A0, 0.02, 1e-4, beta, table, rows, z0=5.0, z_max=9.0, **kw)[1]
    b0 = O.march(A0, 0.02, 1e-4, beta, table, rows, z_max=4.0, **kw)[1]
    assert np.abs(b5 - b0).max() > 1e-6 * scale


@pytest.mark.parametrize("lines, expect", [
    (list(range(0, 129, 2)), (65, 129, 88384)),
    (list(range(0, 24)) + list(range(168, 192)), (48, 192, 25656)),
    (list(range(0, 256, 2)), (128, 255, 686784)),
    (list(range(0, 257, 4)), (65, 257, 88384)),
    (list(range(0, 512, 7)), (74, 512, 130980)),
    (list(range(0, 508, 4)) + [511], (128, 512, 670719)),
])
def test_wide_plan_counts(lines, expect):
    """(N, span, T) of the GPU coverage tests' wide plans, and that each passes the density rule for the comb form."""
    table, rows = O.enumerate_triplets(lines)
    N, M, T = len(lines), max(lines) - min(lines) + 1, len(table)
    assert (N, M, T) == expect and rows[-1] == T
    assert M * M <= 5 * T


def test_fast_rhs_equals_per_term_rhs_beyond_span_128():
    """nwave_rhs_fast (vectorised, used by march) against the per-term statement on a span-257 grid plan and on a
    random table with repeats, k > l, negative weights and empty rows; at z != 0 so the phases matter."""
    rng = np.random.default_rng(3)
    A0, beta, table, rows = _case(list(range(0, 257, 4)), 4)
    tab = np.asarray(table, dtype=np.int64)
    for z in (0.0, 3.7):
        slow = O.nwave_rhs(z, A0, 0.02, 1e-4, beta, table, rows)
        fast = O.nwave_rhs_fast(z, A0, 0.02, 1e-4, beta, tab, np.asarray(rows))
        assert np.abs(fast - slow).max() < 1e-13 * np.abs(slow).max()
    N = 9
    ent = sorted((int(rng.integers(0, N - 2)),) + tuple(int(v) for v in rng.integers(0, N, 3)) + (int(rng.integers(-3, 4)),)
                 for _ in range(60))
    rnd = [e[1:] for e in ent]
    rrows = np.searchsorted(np.array([e[0] for e in ent]), np.arange(N + 1)).tolist()
    assert rrows[-1] == 60 and rrows[N - 1] == rrows[N]          # the last rows are empty
    A = np.sqrt(rng.uniform(1e-3, 0.3, N)) * np.exp(1j * rng.uniform(0, 6.28, N))
    b = rng.uniform(-2.0, 2.0, N)
    slow = O.nwave_rhs(1.3, A, 0.02, 1e-4, b, rnd, rrows)
    fast = O.nwave_rhs_fast(1.3, A, 0.02, 1e-4, b, np.asarray(rnd, dtype=np.int64), np.asarray(rrows))
    assert np.abs(fast - slow).max() < 1e-13 * np.abs(slow).max()


def test_status_is_the_first_nonfinite_step():
    """check=True: -1 for a healthy run, 0 for NaN in A0 or in beta, a mid-run index for a run that overflows (a gain
    of 1e30 per step from a tiny A0: the last finite state is about 1e171, the next step overflows outright).  The
    march stops there, without numpy warnings."""
    A0, beta, table, rows = _case(list(range(-10, 11)), 5)
    kw = dict(z_max=1.2, n_steps=12, save_every=5, check=True)
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        z, A, st = O.march(A0, 0.02, 1e-4, beta, table, rows, **kw)
        assert st == -1 and A.shape == (3, 21) and np.isfinite(A).all()
        bad = A0.copy()
        bad[3] = np.nan
        assert O.march(bad, 0.02, 1e-4, beta, table, rows, **kw)[2] == 0
        nb = beta.copy()
        nb[7] = np.nan
        assert O.march(A0, 0.02, 1e-4, nb, table, rows, **kw)[2] == 0
        for k in (1, 2, 3, 4):
            z, A, st = O.march(A0 * 10.0 ** (-30 * (k - 1)), 0.02, -1.4e9, beta, table, rows, **kw)
            assert st == k
            assert len(z) == len(A) == 1 + (k + 1) // 5      # stopped after step k: the samples saved up to it
            _, every, st1 = O.march(A0 * 10.0 ** (-30 * (k - 1)), 0.02, -1.4e9, beta, table, rows,
                                    z_max=1.2, n_steps=12, check=True)
            assert st1 == k and len(every) == k + 2 and not np.isfinite(every[-1]).all()
            assert 1e150 < np.abs(every[-2]).max() < 1e200      # wide margin on both sides of the overflow
            # a perturbation far above the rounding does not move the step
            for d in (1e-9, -1e-9):
                assert O.march(A0 * 10.0 ** (-30 * (k - 1)) * (1 + d), 0.02, -1.4e9, beta * (1 + d), table, rows, **kw)[2] == k
