"""CPU: the tangent model of the transfer kernels (tools/transfer_model.py) against central finite differences of
oracle/fast_kernel_model.py and against undepleted-pump theory; the fpa_transfer_out layout against the compiled
header; the argument refusals that need no device; the small_signal helpers on hand-built matrices."""
import ctypes as C
import shutil
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tools"))
import transfer_model as TM  # noqa: E402
from oracle import fast_kernel_model as FKM  # noqa: E402

A0 = np.sqrt([0.4, 0.3, 1e-3, 2e-4]) * np.exp(1j * np.array([0.1, 0.3, -0.2, 0.7]))


def _end(a, gamma, alpha, dbeta, z_max, n):
    return FKM.integrate(a, gamma, alpha, dbeta, z_max, n)[-1].view(np.float64)


@pytest.mark.parametrize("alpha", [2e-3, 0.0])
def test_model_matches_finite_differences(alpha):
    g, db, z_max, n = 0.02, 0.004, 80.0, 70             # 70 steps: across two re-synchronisations of the phase
    A_end, J = TM.integrate(A0, g, alpha, db, z_max, n)
    assert A_end.tobytes() == FKM.integrate(A0, g, alpha, db, z_max, n)[-1].tobytes()
    y0 = A0.view(np.float64)
    Jfd = np.empty((8, 8))
    for c in range(8):
        eps = 1e-6 * abs(y0[c])
        yp, ym = y0.copy(), y0.copy()
        yp[c] += eps
        ym[c] -= eps
        Jfd[:, c] = (_end(yp.view(np.complex128), g, alpha, db, z_max, n) -
                     _end(ym.view(np.complex128), g, alpha, db, z_max, n)) / (2 * eps)
    assert np.max(np.abs(J - Jfd)) <= 1e-7 * np.max(np.abs(J))


@pytest.mark.parametrize("kappa", [0.0, 0.006, 0.03])
def test_model_matches_undepleted_pump_theory(kappa):
    """Zero seeds, alpha = 0: kappa = dbeta + gamma(P1 + P2), r = 2 gamma sqrt(P1 P2), g^2 = r^2 - kappa^2/4;
    signal <- signal is complex-linear with |mu|^2 = 1 + (r/g)^2 sinh^2(gL) (sin where g^2 < 0), idler <- signal
    antilinear with |nu|^2 = |mu|^2 - 1, and the signal/idler block has det 1."""
    gam, P, L, n = 0.01, 0.5, 500.0, 2000
    a0 = np.sqrt([P, P, 0.0, 0.0]).astype(np.complex128)
    _, J = TM.integrate(a0, gam, 0.0, kappa - 2 * gam * P, L, n, columns=range(4, 8))
    r = 2 * gam * P
    g2 = r ** 2 - kappa ** 2 / 4
    s2 = np.sinh(np.sqrt(g2) * L) ** 2 / g2 if g2 > 0 else np.sin(np.sqrt(-g2) * L) ** 2 / -g2
    mu2 = 1 + r ** 2 * s2
    from importlib import import_module
    ss = import_module("psa-simulation-ode-rk-mvp-dispersion_b200.small_signal")
    cols = tuple(range(4, 8))
    mu, nu = ss.mu_nu(J, cols, 2, 2)
    mi, ni = ss.mu_nu(J, cols, 3, 2)
    assert abs(abs(mu) ** 2 / mu2 - 1) <= 1e-8 and abs(nu) ** 2 <= 1e-8 * mu2
    assert abs(abs(ni) ** 2 / (mu2 - 1) - 1) <= 1e-8 and abs(mi) ** 2 <= 1e-8 * mu2
    assert abs(np.linalg.det(J[4:, :]) - 1.0) <= 1e-9


def test_model_determinants_with_loss():
    """det of the signal/idler block e^{-2 alpha L}, det of the full J e^{-4 alpha L}."""
    gam, P, L, n, a = 0.01, 0.5, 500.0, 2000, 2e-4
    a0 = np.sqrt([P, P, 0.0, 0.0]).astype(np.complex128)
    _, J = TM.integrate(a0, gam, a, -2 * gam * P, L, n)
    assert abs(np.linalg.det(J[4:, 4:]) / np.exp(-2 * a * L) - 1) <= 1e-9
    assert abs(np.linalg.det(J) / np.exp(-4 * a * L) - 1) <= 1e-6


def test_transfer_out_layout_matches_the_compiled_header(fpa, tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    L = fpa._lib
    prog = ('#include <stdio.h>\n#include <stddef.h>\n#include "fpa_b200.h"\nint main(void) {\n'
            '  printf("%zu %zu %zu\\n", sizeof(fpa_transfer_out), offsetof(fpa_transfer_out, reserved), '
            'offsetof(fpa_transfer_out, jac));\n  return 0;\n}\n')
    src, exe = tmp_path / "t.c", tmp_path / "t"
    src.write_text(prog)
    subprocess.run(["gcc", "-I", str(ROOT / "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert got == [C.sizeof(L.TransferOut), L.TransferOut.reserved.offset, L.TransferOut.jac.offset]


def test_refusals_that_need_no_device(fpa):
    L = fpa._lib
    lib = L.lib()
    db, g, a = np.zeros(2), np.array([0.01]), np.array([0.0])
    a0 = np.tile(A0, (2, 1))
    jac = np.full((2, 8, 8), 7.0)
    st = np.full(2, 5, np.int32)

    def desc(**kv):
        d = L.Yaman4Desc()
        d.n_points, d.z_max, d.n_steps, d.save_every = 2, 1.0, 4, 1
        d.dbeta, d.gamma, d.alpha, d.A0, d.A0_stride = db.ctypes.data, g.ctypes.data, a.ctypes.data, a0.ctypes.data, 1
        d.status = st.ctypes.data
        for k, v in kv.items():
            setattr(d, k, v)
        return d

    t = L.TransferOut(columns=0xFF, jac=jac.ctypes.data)
    grid = np.linspace(0.0, 1.0, 5)
    tr = np.empty((2, 5, 4), np.complex128)
    assert lib.fpa_yaman4_transfer_batch_host(C.byref(desc(flags=L.OUT_TRACE, A_trace=tr.ctypes.data)), C.byref(t), 0) == L.ERR_UNSUPPORTED
    assert lib.fpa_yaman4_transfer_batch_host(C.byref(desc(z_grid=grid.ctypes.data)), C.byref(t), 0) == L.ERR_UNSUPPORTED
    assert lib.fpa_yaman4_transfer_batch_host(C.byref(desc(flags=L.PHASE_EXACT)), C.byref(t), 0) == L.ERR_UNSUPPORTED
    for cols in (0, 0x100):
        tt = L.TransferOut(columns=cols, jac=jac.ctypes.data)
        assert lib.fpa_yaman4_transfer_batch_host(C.byref(desc()), C.byref(tt), 0) == L.ERR_INVALID
        assert "columns" in L.last_error()
    assert lib.fpa_yaman4_transfer_batch_host(C.byref(desc()), None, 0) == L.ERR_INVALID
    assert lib.fpa_yaman4_transfer_sweep_host(C.byref(L.SweepDesc()), None, 0) == L.ERR_INVALID
    sd = L.SweepDesc()
    assert lib.fpa_yaman4_transfer_sweep_host(C.byref(sd), C.byref(L.TransferOut(columns=0, jac=jac.ctypes.data)), 0) == L.ERR_INVALID
    assert lib.fpa_yaman4_transfer_sweep_multi_host(C.byref(sd), None, 1, (C.c_int * 1)(0)) == L.ERR_INVALID
    assert np.all(jac == 7.0) and np.all(st == 5)
    cfg = fpa.config.custom_simulation_config(z_max=1.0, dz=0.25, save_every=1)
    for waves in ((4,), (), (-1,)):
        with pytest.raises(ValueError):
            fpa.simulation.run_batch_transfer(cfg, gamma=0.01, alpha=0.0, delta_beta=[0.0], p_in=[1, 1, 0, 0],
                                              waves=waves)
    with pytest.raises(ValueError):
        fpa.scan_mismtach.sweep_transfer_2d(cfg=cfg, lambda_p1_m=1550e-9, lambda_p2_m=1558e-9,
                                            lambda_signal_m=[1554e-9], gamma=0.01, alpha=0.0, p_in=[1, 1, -1e-3, 0])


def _block(mu, nu):
    """The real 2x2 block of dA_out = mu dA + nu conj(dA)."""
    return np.array([[(mu + nu).real, -(mu - nu).imag], [(mu + nu).imag, (mu - nu).real]])


def test_small_signal_helpers_on_hand_built_matrices(fpa):
    ss = fpa.small_signal
    rng = np.random.default_rng(5)
    mus = rng.standard_normal((4, 4)) + 1j * rng.standard_normal((4, 4))
    nus = rng.standard_normal((4, 4)) + 1j * rng.standard_normal((4, 4))
    J = np.zeros((8, 8))
    for o in range(4):
        for w in range(4):
            J[2 * o:2 * o + 2, 2 * w:2 * w + 2] = _block(mus[o, w], nus[o, w])
    cols = tuple(range(8))
    for o in range(4):
        for w in range(4):
            mu, nu = ss.mu_nu(J, cols, o, w)
            assert np.isclose(mu, mus[o, w], rtol=0, atol=1e-14) and np.isclose(nu, nus[o, w], rtol=0, atol=1e-14)
    assert np.isclose(ss.signal_gain(J, cols), abs(mus[2, 2]) ** 2 + abs(nus[2, 2]) ** 2)
    assert np.isclose(ss.signal_gain(J, cols), 0.5 * np.sum(J[4:6, 4:6] ** 2))
    assert np.isclose(ss.idler_conversion(J, cols), abs(mus[3, 2]) ** 2 + abs(nus[3, 2]) ** 2)
    dA0 = rng.standard_normal(4) + 1j * rng.standard_normal(4)
    direct = (J @ dA0.view(np.float64)).view(np.complex128)
    assert np.allclose(ss.linear_response(J, cols, dA0), direct, rtol=0, atol=1e-13)
    # a column subset: only waves 2, 3; a perturbation of a missing wave is refused
    sub = np.ascontiguousarray(J[:, 4:])
    d2 = dA0.copy()
    d2[:2] = 0
    assert np.allclose(ss.linear_response(sub, (4, 5, 6, 7), d2), (J @ d2.view(np.float64)).view(np.complex128))
    with pytest.raises(ValueError):
        ss.linear_response(sub, (4, 5, 6, 7), dA0)
    with pytest.raises(ValueError):
        ss.mu_nu(sub, (4, 5, 6, 7), 2, 0)
    # phase-sensitive amplifier: signal <- signal mu = cosh r, idler <- signal nu = sinh r (and the mirror image):
    # with equal signal and idler seeds the gain is |cosh r e^{i phi} + sinh r|^2 against the signal phase phi
    r = 0.7
    psa = np.zeros((4, 8, 4))
    psa[0, 4:6, 0:2] = _block(np.cosh(r), 0)
    psa[0, 4:6, 2:4] = _block(0, np.sinh(r))
    psa[0, 6:8, 2:4] = _block(np.cosh(r), 0)
    psa[0, 6:8, 0:2] = _block(0, np.sinh(r))
    psa[1:] = np.nan
    ax = np.linspace(0, 2 * np.pi, 8, endpoint=False)
    pg = ss.phase_gain(psa, (4, 5, 6, 7), [1.0, 1.0, 1e-6, 1e-6], None, ax)
    assert np.allclose(pg["gain_lin"][0], np.abs(np.cosh(r) * np.exp(1j * ax) + np.sinh(r)) ** 2)
    assert pg["idx_max"][0] == 0 and pg["idx_min"][0] == 4 and pg["n_finite"][0] == 8
    assert np.all(pg["idx_max"][1:] == -1) and np.all(np.isnan(pg["gain_max"][1:])) and np.all(pg["n_finite"][1:] == 0)
    # pump sensitivity by hand: dA3(L) = 0.5 * A1(0) * (mu + nu) for a real pump amplitude
    A_in = np.array([2.0, 1.0, 0.1, 0.0], dtype=np.complex128)
    A_out = np.array([1.0, 1.0, 0.3 + 0.4j, 0.0])
    s = ss.pump_power_sensitivity(J, cols, A_in, A_out, 0)
    dA3 = 0.5 * 2.0 * (mus[2, 0] + nus[2, 0])
    assert np.isclose(s, 2 * np.real(np.conj(A_out[2]) * dA3) / abs(A_out[2]) ** 2)
