"""
oracle/nwave_oracle.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

CPU statement (numpy) of the N-wave generalisation defined in SURVEY.md Appendix C.  The
reference has NO N-wave model (every layer checks shape == (4,)), so this file is the
specification's executable form rather than a restatement of reference lines; it is anchored
to the reference in one way only: at N = 4 with the fixed process table it must reproduce
yaman_model.rhs_yaman_simplified (yaman_model.py:10-52, :123-186), which
`oracle/pin_against_reference.py` and tests/test_oracle_cpu.py check.

Parity status: the N = 4 reduction is PINNED against the live reference; for N > 4 parity is
UNPINNED (no reference exists) -- the GPU kernel is checked against this file only.

Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may import this module.
"""
from __future__ import annotations

import contextlib

import numpy as np


def enumerate_triplets(grid_index):
    """Entries (n; k <= l, m not in {k, l}) with g[k] + g[l] - g[m] == g[n], canonical order
    n, k, l, m; weight 1 for k == l else 2.  Returns (list of (k, l, m, weight), row_ptr)."""
    g = [int(v) for v in grid_index]
    N = len(g)
    where = {}
    for idx, v in enumerate(g):
        where.setdefault(v, []).append(idx)
    table, rows = [], [0]
    for n in range(N):
        for k in range(N):
            for l in range(k, N):
                target = g[k] + g[l] - g[n]
                for m in where.get(target, ()):
                    if m == k or m == l:
                        continue
                    table.append((k, l, m, 1 if k == l else 2))
        rows.append(len(table))
    return table, rows


def enumerate_triplets_omega(omega, atol=0.0, rtol=1e-12):
    """Entries (n; k <= l, m not in {k, l}) whose photon energies match under the reference's own rule for its
    four-wave plan, numpy.isclose(w_k + w_l, w_m + w_n, atol=atol, rtol=rtol)
    (frequency_plan.enforce_energy_conservation, frequency_plan.py:112-131).  Canonical order n, k, l, m."""
    w = np.asarray(omega, dtype=float).reshape(-1)
    N = w.size
    table, rows = [], [0]
    for n in range(N):
        for k in range(N):
            lhs = w[k] + w[k:]                      # l = k .. N-1
            rhs = w + w[n]                          # m = 0 .. N-1
            ok = np.isclose(lhs[:, None], rhs[None, :], atol=atol, rtol=rtol)
            for dl, m in zip(*np.nonzero(ok)):
                l = k + int(dl)
                if m == k or m == l:
                    continue
                table.append((k, l, int(m), 1 if k == l else 2))
        rows.append(len(table))
    return table, rows


def count_ordered(grid_index):
    """(ordered combinations incl. Kerr, non-Kerr ordered, distinct (k,l) pairs) -- the known
    answers quoted in SURVEY App. C (N=4 uniform: 44 / 16 / 6 pairs, 10 table entries)."""
    g = [int(v) for v in grid_index]
    N = len(g)
    pos = {v: i for i, v in enumerate(g)}
    total = nonkerr = 0
    for n in range(N):
        for k in range(N):
            for l in range(N):
                m = pos.get(g[k] + g[l] - g[n])
                if m is None:
                    continue
                total += 1
                if m != k and m != l:
                    nonkerr += 1
    table, _ = enumerate_triplets(g)
    pairs = len({(k, l) for k, l, _, _ in table})
    return total, nonkerr, pairs


FOUR_WAVE_TABLE = [(2, 3, 1, 2), (2, 3, 0, 2), (0, 1, 3, 2), (0, 1, 2, 2)]
FOUR_WAVE_ROWS = [0, 1, 2, 3, 4]


def nwave_rhs(z, A, gamma, alpha, beta, table, rows):
    """dA/dz of the N-wave system (App. C), straightforward per-term evaluation."""
    A = np.asarray(A, dtype=np.complex128)
    N = A.size
    P = np.abs(A) ** 2
    S = P.sum()
    out = (-0.5 * alpha) * A + 1j * gamma * (2.0 * S - P) * A
    for n in range(N):
        acc = 0.0 + 0.0j
        for e in range(rows[n], rows[n + 1]):
            k, l, m, w = table[e]
            dphi = (beta[k] + beta[l] - beta[m] - beta[n]) * z
            acc += w * A[k] * A[l] * np.conj(A[m]) * np.exp(1j * dphi)
        out[n] += 1j * gamma * acc
    return out


def nwave_rhs_fast(z, A, gamma, alpha, beta, tab_arr, rows):
    """Same sum, vectorised over the table (tab_arr: int array [T,4]); used for long runs."""
    A = np.asarray(A, dtype=np.complex128)
    P = np.abs(A) ** 2
    S = P.sum()
    out = (-0.5 * alpha) * A + 1j * gamma * (2.0 * S - P) * A
    if tab_arr.shape[0]:
        k, l, m, w = tab_arr[:, 0], tab_arr[:, 1], tab_arr[:, 2], tab_arr[:, 3]
        n_of = np.repeat(np.arange(A.size), np.diff(rows))
        dphi = (beta[k] + beta[l] - beta[m] - beta[n_of]) * z
        terms = w * A[k] * A[l] * np.conj(A[m]) * np.exp(1j * dphi)
        acc = np.zeros(A.size, dtype=np.complex128)
        np.add.at(acc, n_of, terms)
        out = out + 1j * gamma * acc
    return out


def march(A0, gamma, alpha, beta, table, rows, *, z_max, n_steps, save_every=1, fast=True, z0=0.0, check=False):
    """Classical RK4 on linspace(z0, z_max, n_steps+1) with the reference's saving rule
    (integrators.py:111-142).  Returns (z_saved, A_saved[n_saved, N]).

    check=True: also return the status the kernels report -- the index of the first step whose result
    has a non-finite component, or -1 (integrators.py:132-135) -- as (z_saved, A_saved, status).  The
    march stops after that step; the samples saved up to and including it are returned."""
    beta = np.asarray(beta, dtype=float)
    rows = np.asarray(rows)
    tab_arr = np.asarray(table, dtype=np.int64).reshape(-1, 4)
    f = (lambda z, y: nwave_rhs_fast(z, y, gamma, alpha, beta, tab_arr, rows)) if fast else \
        (lambda z, y: nwave_rhs(z, y, gamma, alpha, beta, table, rows))
    grid = np.linspace(z0, z_max, n_steps + 1)
    y = np.asarray(A0, dtype=np.complex128).copy()
    zs, ys = [grid[0]], [y.copy()]
    status = -1
    # a run that blows up overflows inside the stages; with check=True that is an expected outcome
    with np.errstate(over="ignore", invalid="ignore") if check else contextlib.nullcontext():
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
            if check and not np.all(np.isfinite(y)):
                status = i
                break
    if check:
        return np.array(zs), np.array(ys), status
    return np.array(zs), np.array(ys)

