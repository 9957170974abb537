"""GPU: parity at the fiber lengths of the BASELINE configurations (not shortened).

The N-wave comb kernels advance exp(i*beta_j*z) by a rotation per half step and re-synchronise it with an
exact sincos every 32 steps; the enumerated-triplet kernel evaluates sincos(beta_j * z) at every RK4
abscissa and shares no phase or indexing code with them.  Agreement of the two over 1e4 (config 2) and
2e4+ (config 5 plan) steps bounds the drift of the recurrence; an oracle prefix ties both to the CPU
statement of SURVEY App. C.  For N > 4 the oracle is UNPINNED (the reference has no N-wave model).
The last test is the full-length config-4 sweep against the (pinned) 4-wave oracle on a sample of points.
"""
import numpy as np
import pytest

from test_nwave_lines_cpu import assert_lines

pytestmark = pytest.mark.gpu


def _table_as_list(plan):
    t = plan.table
    return [(int(a), int(b), int(c), int(d)) for a, b, c, d in zip(t["k"], t["l"], t["m"], t["weight"])]


def _config2(gpu, golden):
    nw = gpu.nwave
    wc, wd = golden["b1_sym"][0], golden["b1_sym"][1]
    plan = nw.uniform_comb_plan(wc, wd / 5.0, range(-10, 11))
    b2, b3, b4 = golden["b1_beta"]
    beta = nw.beta_per_wave(plan, gpu.dispersion.DispersionParams(omega_ref=wc, beta2=b2, beta3=b3, beta4=b4))
    p_in = np.zeros(21)
    p_in[[5, 15]] = 0.5
    p_in[[9, 11]] = 1e-5
    gamma, alpha = golden["b1_gamma_alpha"]
    return plan, beta, p_in, float(gamma), float(alpha)


def _config5(gpu, n_points, p_lo=0.1, p_hi=1.0, seed=0):
    nw = gpu.nwave
    w0 = 2 * np.pi * 299792458.0 / 1550e-9
    plan = nw.uniform_comb_plan(w0, 2 * np.pi * 100e9, range(-32, 32))
    beta = nw.beta_per_wave(plan, gpu.dispersion.DispersionParams(omega_ref=w0, beta2=-2.57e-29, beta3=3.30e-41,
                                                                   beta4=-1.63e-55))
    phases = np.random.default_rng(seed).uniform(0, 2 * np.pi, 64)
    A0 = np.empty((n_points, 64), dtype=complex)
    for b, pw in enumerate(np.linspace(p_lo, p_hi, n_points)):
        p = np.full(64, 1e-12)
        p[33] = 1e-6
        p[[28, 36]] = pw
        A0[b] = np.sqrt(p) * np.exp(1j * phases)
    return plan, beta, A0


def test_config2_full_length_comb_vs_table_vs_oracle(gpu, nw_oracle, golden):
    """BASELINE config 2 at its own length: N = 21, 10 000 steps (z = 1 km), full trace [1001, 21]."""
    nw = gpu.nwave
    plan, beta, p_in, gamma, alpha = _config2(gpu, golden)
    cfg = gpu.config.custom_simulation_config(z_max=1000.0, dz=0.1, save_every=10)
    t = nw.run_nwave_simulation(cfg, plan, gamma=gamma, alpha=alpha, p_in=p_in, beta=beta, form="table")
    c = nw.run_nwave_simulation(cfg, plan, gamma=gamma, alpha=alpha, p_in=p_in, beta=beta, form="comb")
    At, Ac = t["A_trace"][0], c["A_trace"][0]
    assert At.shape == (1001, 21) and (t["status"] == -1).all() and (c["status"] == -1).all()
    scale = np.max(np.abs(At))
    assert np.max(np.abs(Ac - At)) <= 1e-10 * scale                    # whole trace, recurrence vs exact phases
    assert_lines(Ac[-1], At[-1], 1e-10, "config 2 end state, comb vs table")     # every line on its own scale
    # oracle prefix: the first 3 000 steps (301 samples)
    z_ref, A_ref = nw_oracle.march(np.sqrt(p_in).astype(complex), gamma, alpha, beta, _table_as_list(plan),
                                   plan.row_ptr.tolist(), z_max=300.0, n_steps=3000, save_every=10)
    assert np.allclose(t["z"][:301], z_ref, rtol=0, atol=1e-9)
    for A in (At, Ac):
        assert np.max(np.abs(A[:301] - A_ref)) <= 1e-10 * np.max(np.abs(A_ref))
    # the batch kernel (warp per point) on the same run, replicated: 600 copies, every one equal to the single run's physics
    many = nw.run_nwave_simulation(cfg, plan, gamma=gamma, alpha=alpha, A0=np.tile(np.sqrt(p_in).astype(complex), (600, 1)),
                                   beta=beta, form="comb", outputs=("end",))
    assert np.max(np.abs(many["A_end"] - At[-1])) <= 1e-10 * scale
    assert np.array_equal(many["A_end"][0], many["A_end"][599])


def test_config5_plan_long_fiber_comb_vs_table_vs_oracle(gpu, nw_oracle):
    """BASELINE config 5 plan (N = 64, 100 GHz grid, beta2..beta4, dz = 0.1 m): 24 000 steps.  Batch kernel
    (608 points, warp per point), single-run kernel (CTA per point) and the triplet-table kernel.
    Pump powers 0.02 .. 0.09 W: the system amplifies any perturbation -- a rounding difference between two
    summation orders included -- by about exp(2 gamma P_total z); at the config's upper powers (1 W over
    kilometres) that factor exceeds 1e16 and NO two evaluation orders agree, so a drift test has to stay
    where it is ~1e4 (here: exp(2 * 0.0115 * 0.18 * 2400) = 2e4)."""
    nw = gpu.nwave
    n_steps = 24_000
    plan, beta, A0 = _config5(gpu, 608, 0.02, 0.09)
    cfg = gpu.config.custom_simulation_config(z_max=0.1 * n_steps, dz=0.1, save_every=2000)
    kw = dict(gamma=11.5e-3, alpha=2e-4, beta=beta, outputs=("trace",))
    batch = nw.run_nwave_simulation(cfg, plan, A0=A0, form="comb", **kw)
    assert batch["A_trace"].shape == (608, 13, 64) and (batch["status"] == -1).all()
    for b in (0, 607):
        table = nw.run_nwave_simulation(cfg, plan, A0=A0[b:b + 1], form="table", **kw)["A_trace"][0]
        single = nw.run_nwave_simulation(cfg, plan, A0=A0[b:b + 1], form="comb", **kw)["A_trace"][0]
        scale = np.max(np.abs(table))
        assert np.max(np.abs(batch["A_trace"][b] - table)) <= 1e-10 * scale, b
        assert np.max(np.abs(single - table)) <= 1e-10 * scale, b
        strong = np.abs(table[-1]) ** 2 > 1e-9
        rel = np.abs(np.abs(batch["A_trace"][b][-1, strong]) ** 2 - np.abs(table[-1, strong]) ** 2) / np.abs(table[-1, strong]) ** 2
        assert rel.max() < 1e-10, b
    # oracle prefix (1 000 steps) for the strongest-pump point
    cfg_p = gpu.config.custom_simulation_config(z_max=100.0, dz=0.1, save_every=500)
    z_ref, A_ref = nw_oracle.march(A0[607], 11.5e-3, 2e-4, beta, _table_as_list(plan), plan.row_ptr.tolist(), z_max=100.0,
                                   n_steps=1000, save_every=500)
    pre = nw.run_nwave_simulation(cfg_p, plan, A0=A0[592:], form="comb", **kw)      # 16 points: CTA-per-point kernel
    pre_b = nw.run_nwave_simulation(cfg_p, plan, A0=A0, form="comb", **kw)          # 608 points: batch kernel
    for A in (pre["A_trace"][15], pre_b["A_trace"][607]):
        assert np.max(np.abs(A - A_ref)) <= 1e-11 * np.max(np.abs(A_ref))


def test_config5_full_size_invariants(gpu):
    """BASELINE config 5 at its FULL size -- N = 64, B = 1024 pump powers, 1e5 z-steps of 0.1 m -- through
    size-independent properties (no CPU statement finishes this in test time): (i) lossless fiber: the total power of
    every point is conserved (Manley-Rowe) to RK4 accuracy over the 10 km; (ii) the same point at two positions of
    the batch gives the same bits; (iii) with loss the total power follows exp(-alpha z) (the Kerr and mixing terms
    conserve it, so dP/dz = -alpha P whatever the lines exchange among themselves)."""
    nw = gpu.nwave
    n_steps = 100_000
    plan, beta, A0 = _config5(gpu, 512, 0.1, 1.0)
    A0 = np.concatenate((A0, A0))                       # 1 024 points: every point twice, 512 positions apart
    cfg = gpu.config.custom_simulation_config(z_max=0.1 * n_steps, dz=0.1, save_every=10_000)
    r = nw.run_nwave_simulation(cfg, plan, A0=A0, gamma=11.5e-3, alpha=0.0, beta=beta, outputs=("trace", "pmax"), form="comb")
    assert r["A_trace"].shape == (1024, 11, 64) and (r["status"] == -1).all()
    P = (np.abs(r["A_trace"]) ** 2).sum(axis=2)         # [B, saved]
    assert np.max(np.abs(P / P[:, :1] - 1.0)) < 1e-8
    assert r["A_trace"][:512].tobytes() == r["A_trace"][512:].tobytes()
    assert r["Pmax"][:512].tobytes() == r["Pmax"][512:].tobytes()
    # cascaded mixing did happen: lines that started at 1e-12 W carry power at the end
    assert (np.abs(r["A_trace"][:, -1, :]) ** 2 > 1e-6).sum(axis=1).min() >= 8
    lossy = nw.run_nwave_simulation(cfg, plan, A0=A0[:64], gamma=11.5e-3, alpha=2e-4, beta=beta, outputs=("trace",), form="comb")
    Pl = (np.abs(lossy["A_trace"]) ** 2).sum(axis=2)
    z = lossy["z"]
    assert np.max(np.abs(Pl / (Pl[:, :1] * np.exp(-2e-4 * z)[None, :]) - 1.0)) < 1e-8


def test_config4_full_length_sample_vs_oracle(gpu, oracle, golden):
    """BASELINE config 4 at full size -- 1000 x 1000 grid, 2 500 steps -- against the pinned 4-wave oracle on 48
    random grid points: gain to 1e-10, dbeta to 1e-12 (what bench.py also reports as parity_max_rel_err_vs_gpu)."""
    b2, b3, b4, wref = golden["b4_beta"]
    disp = gpu.dispersion.DispersionParams(omega_ref=wref, beta2=b2, beta3=b3, beta4=b4)
    alpha = float(golden["b4_alpha"][0])
    cfg = gpu.config.custom_simulation_config(z_max=500.0, dz=0.2, save_every=10)
    lam1 = np.linspace(1545e-9, 1555e-9, 1000)
    lam3 = np.linspace(1540e-9, 1565e-9, 1000)
    r = gpu.scan_mismtach.sweep_gain_2d(cfg=cfg, lambda_p1_m=lam1, lambda_p2_m=1558e-9, lambda_signal_m=lam3, gamma=11.5e-3,
                                        alpha=alpha, p_in=golden["b4_p_in"], dispersion=disp, gain_unit="linear")
    assert r["gain"].shape == (1000, 1000) and (r["status"] == -1).all() and (r["valid"] == 1).all()
    od = oracle.Taylor(wref, 0.0, 0.0, b2, b3, b4)
    rng = np.random.default_rng(2024)
    worst = 0.0
    for i, j in zip(rng.integers(0, 1000, 48), rng.integers(0, 1000, 48)):
        g, db = oracle.sweep_lambda3_gain(lam1=lam1[i], lam2=1558e-9, lam3_arr=[lam3[j]], z_max=500.0, dz=0.2, save_every=10,
                                          check_nan=True, gamma=11.5e-3, alpha=alpha, p_in=golden["b4_p_in"], disp=od,
                                          gain_unit="linear")
        worst = max(worst, abs(r["gain"][i, j] - g[0]) / abs(g[0]))
        assert abs(r["dbeta"][i, j] - db[0]) <= 1e-12 * max(abs(db[0]), 1e-3)
    assert worst < 1e-10, worst
