"""CPU: the symmetric sweep path of csrc/yaman4.cu (stage_sym, fast_integrate<..., SYM>).

The argument it rests on, checked on the exact-FMA model of the kernel (oracle/fast_kernel_model.py): from an
initial state with A1 == A2 and A3 == A4 bit for bit, the 4-wave z-loop keeps the state bitwise on that subspace
(lossy and lossless, across the phase re-synchronisations), and a reduced z-loop on (x1, y1, x3, y3) with the
operations of stage_sym() reproduces it bit for bit.  A one-ulp asymmetry leaves the subspace, so the launcher
must compare A0's bit patterns, not test a tolerance.  Plus: the SASS pass re-orders the new kernels' hot blocks
and they still compute what ptxas' schedule computes."""
import math
import sys

import numpy as np
import pytest

import __graft_entry__ as entry
from oracle import fast_kernel_model as M

fma = M.fma


def stage_sym(inn, base, qr, qi, cg, c2g, cn):
    """stage_sym() of csrc/yaman4.cu: M.stage with x2 -> x1, y2 -> y1, x4 -> x3, y4 -> y3, on 4 doubles."""
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
    return [
        fma(-G1, y1, fma(y1, Wr, fma(-x1, Wi, fma(cn, x1, base[0])))),
        fma(G1, x1, fma(x1, Wr, fma(y1, Wi, fma(cn, y1, base[1])))),
        fma(-G3, y3, fma(y3, Zr, fma(-x3, Zi, fma(cn, x3, base[2])))),
        fma(G3, x3, fma(x3, Zr, fma(y3, Zi, fma(cn, y3, base[3])))),
    ]


def integrate_sym(A0, gamma, alpha, dbeta, z_max, n_steps, save_every):
    """M.integrate's z-loop on the symmetric half (x1, y1, x3, y3); saved states expanded to complex[4]."""
    h = z_max / n_steps
    w = [0.5 * h, h, h * (1.0 / 6.0)]
    cg = [wi * gamma for wi in w]
    c2g = [c + c for c in cg]
    cn = [wi * (-0.5 * alpha) for wi in w]
    q0 = c2g[0]
    third, two_thirds, third_c = M.weights("shipped")
    a1, a3 = complex(A0[0]), complex(A0[2])
    y = [a1.real, a1.imag, a3.real, a3.imag]
    rr, ri = math.cos(dbeta * (0.5 * h)), math.sin(dbeta * (0.5 * h))
    qr, qi = q0, 0.0
    full = lambda y: np.array([complex(y[0], y[1]), complex(y[0], y[1]), complex(y[2], y[3]), complex(y[2], y[3])])  # noqa: E731
    saved = [full(y)]
    for i in range(n_steps):
        if i % M.RESYNC == 0:
            ang = dbeta * fma(float(i), h, 0.0)
            qr, qi = q0 * math.cos(ang), q0 * math.sin(ang)
        qhr, qhi = fma(-qi, ri, qr * rr), fma(qr, ri, qi * rr)
        q2r, q2i = qhr + qhr, qhi + qhi
        qfr, qfi = fma(-qhi, ri, qhr * rr), fma(qhr, ri, qhi * rr)
        q6r, q6i = qfr * third, qfi * third
        ys = stage_sym(y, y, qr, qi, cg[0], c2g[0], cn[0])
        acc = [fma(third, ys[j], y[j] * (-third)) for j in range(4)]
        yt = stage_sym(ys, y, qhr, qhi, cg[0], c2g[0], cn[0])
        acc = [fma(two_thirds, yt[j], acc[j]) for j in range(4)]
        ys = stage_sym(yt, y, q2r, q2i, cg[1], c2g[1], cn[1])
        acc = [fma(third_c, ys[j], acc[j]) for j in range(4)]
        y = stage_sym(ys, acc, q6r, q6i, cg[2], c2g[2], cn[2])
        qr, qi = qfr, qfi
        if (i + 1) % save_every == 0:
            saved.append(full(y))
    return saved


# strong coupling (0.5 W pumps, ~25 dB of gain over the run) so that every term of the RHS matters; 200 steps span
# six phase re-synchronisations (every 32 steps)
A1 = 0.5 ** 0.5 * np.exp(0.4j)
A3 = 1e-3 * np.exp(-1.1j)
PHYS = dict(gamma=11.5e-3, dbeta=-2.1e-3, z_max=2000.0, n_steps=200)


def bits(a):
    return np.asarray(a, dtype=np.complex128).tobytes()


@pytest.mark.parametrize("alpha", [1.15e-4, 0.0], ids=["lossy", "lossless"])
def test_symmetric_state_stays_symmetric_and_the_reduced_loop_reproduces_it(alpha):
    A0 = np.array([A1, A1, A3, A3])
    full = M.integrate(A0, PHYS["gamma"], alpha, PHYS["dbeta"], PHYS["z_max"], PHYS["n_steps"], save_every=1)
    assert len(full) == PHYS["n_steps"] + 1
    for s in full:
        assert bits(s[0]) == bits(s[1]) and bits(s[2]) == bits(s[3])
    g = abs(full[-1][2]) ** 2 / abs(A3) ** 2
    assert g > 10.0                                          # the signal grew: the coupling terms are exercised
    red = integrate_sym(A0, PHYS["gamma"], alpha, PHYS["dbeta"], PHYS["z_max"], PHYS["n_steps"], save_every=1)
    assert len(red) == len(full)
    for a, b in zip(full, red):
        assert bits(a) == bits(b)


def test_one_ulp_asymmetry_leaves_the_subspace():
    """A2 one ulp off A1: the 4-wave run is not symmetric, so only bit-equal A0 may take the reduced loop."""
    A2 = complex(np.nextafter(A1.real, 1.0), A1.imag)
    A0 = np.array([A1, A2, A3, A3])
    assert A0[0] != A0[1]
    full = M.integrate(A0, PHYS["gamma"], 1.15e-4, PHYS["dbeta"], PHYS["z_max"], 64, save_every=1)
    assert any(bits(s[0]) != bits(s[1]) for s in full[1:])
    # and the symmetric run from A1 differs from it
    sym = M.integrate(np.array([A1, A1, A3, A3]), PHYS["gamma"], 1.15e-4, PHYS["dbeta"], PHYS["z_max"], 64, save_every=1)
    assert bits(sym[-1]) != bits(full[-1])


# ------------------------------------------------------------------ the SASS pass on the symmetric kernels
SYM_KERNELS = ("yaman4_sweep_kernelILb1ELi128ELi{mb}ENS_10SweepExtraELb1E", "yaman4_sweep_kernelILb0ELi128ELi{mb}ENS_10SweepExtraELb1E",
               "yaman4_sweep_seg_kernelILb1ELi128ELi{mb}ENS_10SweepExtraELb1E",
               "yaman4_sweep_seg_kernelILb0ELi128ELi{mb}ENS_10SweepExtraELb1E")


@pytest.fixture(scope="module")
def libs(fpa):
    sys.path.insert(0, str(entry.ROOT / "tools"))
    import sass_sched as S
    assert entry.LIB.exists() and entry.REF_LIB.exists()
    return S, S.disassemble_all(str(entry.LIB)), S.disassemble_all(str(entry.REF_LIB))


def test_symmetric_kernels_are_rescheduled_and_compute_the_same_values(libs):
    S, new_f, ref_f = libs
    if b"re-scheduled" not in entry.load_package()._lib.lib().fpa_version():
        pytest.skip("library built with ptxas' own schedule (SASS pass not applied)")
    for pat in SYM_KERNELS:
        names = [k for k in ref_f if any(pat.format(mb=mb) in k for mb in range(1, 9))]
        assert len(names) == 1, (pat, names)
        new, ref = new_f[names[0]], ref_f[names[0]]
        assert len(new) == len(ref)
        blocks = S.hot_blocks(ref)
        assert blocks
        hot = set()
        for b in blocks:
            hot |= set(b)
            assert S.symbolic([ref[i] for i in b]) == S.symbolic([new[i] for i in b])
        for i, (x, y) in enumerate(zip(ref, new)):
            if i not in hot:
                assert (x.lo, x.hi) == (y.lo, y.hi)
        # the pass changed something: fewer three-register fetches than ptxas left
        m_new = sum(S.cost([new[i] for i in b])[1] for b in blocks)
        m_ref = sum(S.cost_ptxas([ref[i] for i in b])[1] for b in blocks)
        assert m_new < m_ref, (names[0], m_ref, m_new)
