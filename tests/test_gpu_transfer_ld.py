"""GPU: the transfer matrices of the batch and sweep transfer kernels block by block against the long-double reference
(oracle/transfer_ld.py), at the bench's fiber and gains up to ~45 dB.

Cases (tests/test_transfer_ld_cpu.py defines the batch points): gamma = 11.5e-3 /W/m, 0.5 + 0.5 W pumps, 500 m in
2 500 steps of 0.2 m; signal seeds of 1e-4, 1e-9, 1e-13 W and 0, idlers seeded on some points; kappa across the gain
band and beyond it; one depleted point (1e-4 W at 43 dB).
  - batch: UNIFORM 1 (lossy), 2 (lossless), 0 (per-point gamma / alpha), and z0 = 2000 m (one point at dbeta z0 ~ 1e3 rad);
  - sweep: a 3 x 4 grid around the gain peak in m and in km units, asymmetric and symmetric [P, P, Ps, Ps] inputs;
  - one run of 10 000 steps (2 000 m) at 0.125 + 0.125 W pumps, so that the gain stays at ~43 dB.

Checks: every 2x2 block of J within TOL of itself (|d mu| + |d nu| <= TOL (|mu| + |nu|)), the blocks that are exactly 0
in the reference exactly 0, A_end within TOL per wave, status -1; J of a symmetric input invariant under swapping
(1 <-> 2, 3 <-> 4); and signal_gain, idler_conversion, pump_power_sensitivity and phase_gain's max and min against the
same functions of the reference J, each within the bound TOL and its condition number give it (`_check_small_signal`).

TOL: the FP64 model of the kernels (tools/transfer_model.py) meets the reference per block to 7.4e-13 at 2 500 steps
and 5.2e-13 at 10 000 steps (x86-64; the CPU file and DESIGN section 4.1d), and the kernels to 1.1e-12 (NVIDIA B200,
1 000 W power limit: batch z0 case), so TOL = 2e-10 is two decades above either."""
import os

import numpy as np
import pytest
from scipy.optimize import minimize_scalar

from test_transfer_ld_cpu import (ALPHA, DZ, GAMMA, L, P_PUMP, POINTS, assert_blocks, assert_waves, batch_case,
                                  block_errors, mu_nu_ld, reference)
from oracle import transfer_ld as TL

pytestmark = pytest.mark.gpu

TOL = 2e-10
N_STEPS = int(round(L / DZ))
LAM_P1 = np.array([1551e-9, 1552e-9, 1553e-9])            # kappa -0.006 .. 0.006 on the signal axis below: 40-45 dB
LAM_S = np.linspace(1540.5e-9, 1544.5e-9, 4)
LAM_P2 = 1558e-9
PHASE_IN = [0.1, -0.2, 0.3, 0.05]
SWEEPS = {   # unit, p_in, phase_in
    "m-1e-9": ("m", [P_PUMP, P_PUMP, 1e-9, 2e-10], PHASE_IN),
    "m-1e-13": ("m", [P_PUMP, P_PUMP, 1e-13, 0.0], PHASE_IN),
    "km-1e-4": ("km", [P_PUMP, P_PUMP, 1e-4, 0.0], PHASE_IN),
    "km-0": ("km", [P_PUMP, P_PUMP, 0.0, 0.0], PHASE_IN),
    "m-sym-1e-9": ("m", [P_PUMP, P_PUMP, 1e-9, 1e-9], None),
    "km-sym-1e-13": ("km", [P_PUMP, P_PUMP, 1e-13, 1e-13], None),
}
SWAP = [2, 3, 0, 1, 6, 7, 4, 5]        # component r of A1 <-> A2, A3 <-> A4


@pytest.fixture(autouse=True)
def _clean_env():
    yield
    os.environ.pop("FPA_SWEEP_SYM", None)


@pytest.fixture(scope="module")
def refs():
    """Long-double references, each computed once per module."""
    cache = {}

    def get(key, make):
        if key not in cache:
            cache[key] = make()
        return cache[key]
    return get


def _bench_dispersion(gpu, scale=1.0):
    """The bench's fiber (D = 0.1 ps/nm/km, S = 0.02 ps/nm^2/km at the pumps' centre), per metre * scale."""
    import bench
    from oracle import fwm_oracle as O
    d = bench.fiber_dispersion(O)
    return gpu.dispersion.DispersionParams(omega_ref=d.omega_ref, beta2=d.b[2] * scale, beta3=d.b[3] * scale,
                                           beta4=d.b[4] * scale)


# ------------------------------------------------------------------ small-signal quantities
def _check_small_signal(gpu, jac, ref, A0, A_end, A_end_ref, what):
    """The small_signal helpers on the kernel's J against the same helpers on the reference J, per point, each within
    what the per-block bound implies.  With |d mu| + |d nu| <= TOL (|mu| + |nu|) on every block:

    - signal_gain / idler_conversion G = |mu|^2 + |nu|^2 of one block: |dG| <= 2 (|mu| |d mu| + |nu| |d nu|) + (d)^2
      <= (2 TOL + TOL^2) (|mu| + |nu|)^2, and (|mu| + |nu|)^2 / G <= 2: at most ~4 TOL relative.
    - pump_power_sensitivity s = 2 Re(conj(A3) dA3) / |A3|^2 with dA3 = sum_p mu_p x_p + nu_p conj(x_p), x_p = A_p(0)/2:
      |d dA3| <= TOL M, M = sum_p (|mu_p| + |nu_p|) |x_p|, and |dA3| <= M; with |d A3| <= TOL |A3| (A_end per wave),
      |ds| <= 2 TOL M / |A3| + 2 TOL M / |A3| + 2 TOL |s| = TOL (4 M / |A3| + 2 |s|): the condition number M / |A3| is
      large where the seed is weak against the pump's pull on it.
    - phase_gain with equal seeds x2, x3 of power p: out_k = sum_{w=2,3} mu_w x_w + nu_w conj(x_w), G_k = |out_k|^2 / p,
      |d out_k| <= TOL sqrt(p) M2, M2 = sum_{w=2,3} |mu_{2w}| + |nu_{2w}| (blocks signal <- signal, signal <- idler);
      |dG_k| <= 2 TOL M2 sqrt(G_k) + TOL^2 M2^2.  Relative to G_min this is 2 TOL M2 / sqrt(G_min) ~ 2 TOL
      (|mu| + |nu|)^2 since G_min ~ 1 / (|mu| + |nu|)^2: the de-amplified quadrature is the most sensitive quantity J
      gives.  The axis holds 16 phases and the exact minimiser of the reference's G, so G_min is the deep minimum.
    Every bound gets 1e-13 relative on top for the FP64 arithmetic of the helpers."""
    ss = gpu.small_signal
    cols = tuple(range(8))
    J, Jr = np.asarray(jac, dtype=float), np.asarray(ref, dtype=np.longdouble)
    Jf = Jr.astype(float)
    B = J.shape[0]
    slack = 1e-13
    # gains of the seed blocks
    for fn, (o, w) in ((ss.signal_gain, (2, 2)), (ss.idler_conversion, (3, 2))):
        mu, nu = mu_nu_ld(Jr, o, w)
        cond = ((np.abs(mu) + np.abs(nu)) ** 2).astype(float)
        g, gr = fn(J, cols), fn(Jf, cols)
        bound = (2 * TOL + TOL ** 2) * cond + slack * gr
        assert np.all(np.abs(g - gr) <= bound), (what, fn.__name__, np.max(np.abs(g - gr) / bound))
    # pump sensitivity where the signal is non-zero at the end
    A_end_ref = np.asarray(A_end_ref, dtype=np.clongdouble).astype(complex)
    live = np.abs(A_end_ref[:, 2]) > 0
    n_sens = 0
    for pump in (0, 1, (0, 1)):
        s = ss.pump_power_sensitivity(J, cols, A0, A_end, pump)
        sr = ss.pump_power_sensitivity(Jf, cols, A0, A_end_ref, pump)
        M = np.zeros(B)
        for p in np.atleast_1d(pump):
            mu, nu = mu_nu_ld(Jr, 2, int(p))
            M += (np.abs(mu) + np.abs(nu)).astype(float) * np.abs(np.broadcast_to(A0, (B, 4))[:, p]) / 2
        with np.errstate(divide="ignore", invalid="ignore"):
            bound = TOL * (4 * M / np.abs(A_end_ref[:, 2]) + 2 * np.abs(sr)) + slack * (1 + np.abs(sr))
        assert np.all(np.abs(s - sr)[live] <= bound[live]), (what, pump, np.max((np.abs(s - sr) / bound)[live]))
        n_sens += int(live.sum())
    # phase-sensitive gain: max and min over the input phase, equal seeds
    p_in = [P_PUMP, P_PUMP, 1e-6, 1e-6]
    deep = 0
    for b in range(B):
        m22, n22 = (v.astype(complex) for v in mu_nu_ld(Jr[b], 2, 2))
        m23, n23 = (v.astype(complex) for v in mu_nu_ld(Jr[b], 2, 3))
        c = m23 + n23                                    # the idler seed's contribution (phase 0)
        f = lambda x: abs(m22 * np.exp(1j * x) + n22 * np.exp(-1j * x) + c) ** 2  # noqa: E731
        phi = np.linspace(0, 2 * np.pi, 4097)
        k = int(np.argmin([f(x) for x in phi]))
        opt = minimize_scalar(f, bounds=(phi[k] - 2 * np.pi / 4096, phi[k] + 2 * np.pi / 4096), method="bounded",
                              options={"xatol": 1e-13})
        ax = np.concatenate([np.linspace(0, 2 * np.pi, 16, endpoint=False), [opt.x]])
        pg = ss.phase_gain(J[b], cols, p_in, None, ax)
        pr = ss.phase_gain(Jf[b], cols, p_in, None, ax)
        M2 = float(sum(abs(v) for v in (m22, n22, m23, n23)))
        bound = 2 * TOL * M2 * np.sqrt(pr["gain_lin"]) + (TOL * M2) ** 2 + slack * pr["gain_lin"]
        assert np.all(np.abs(pg["gain_lin"] - pr["gain_lin"]) <= bound), (what, b)
        for key, idx in (("gain_max", "idx_max"), ("gain_min", "idx_min")):
            assert pg[idx] == pr[idx], (what, b, key)
            assert abs(pg[key] - pr[key]) <= bound[pr[idx]], (what, b, key, pg[key], pr[key], bound[pr[idx]])
        if pr["gain_max"] >= 1e3 and pr["gain_min"] <= 1e-2:
            deep += 1
    return n_sens, deep


def _check_run(gpu, r, A0, ref, what, zero_blocks=None):
    """J, A_end and status of a run ([B, ...] flattened) against the reference (A_end, J)."""
    A_end_ref, J_ref = ref
    jac, A_end = r["jac"].reshape(-1, 8, 8), r["A_end"].reshape(-1, 4)
    assert np.all(r["status"] == -1), what
    worst, weakest = assert_blocks(jac, J_ref, TOL, what)
    we = assert_waves(A_end, A_end_ref, TOL, what)
    _, mag, _ = block_errors(jac, J_ref)
    if zero_blocks is not None:
        assert int(np.sum(mag == 0)) == zero_blocks, (what, int(np.sum(mag == 0)))
    n_sens, deep = _check_small_signal(gpu, jac, J_ref, A0, A_end, A_end_ref, what)
    G = np.max(gpu.small_signal.signal_gain(J_ref.astype(float), tuple(range(8))))
    print(f"\n{what}: largest per-block error {worst:.1e}, weakest block checked |mu| + |nu| = {weakest:.1e}, A_end "
          f"{we:.1e}; largest signal gain {10 * np.log10(G):.1f} dB, {n_sens} pump sensitivities, {deep} points with "
          f"G_max >= 1e3 and G_min <= 1e-2")
    return G, deep


# ------------------------------------------------------------------ batch
@pytest.mark.parametrize("case", ["lossy", "lossless", "per_point", "z0"])
def test_batch_every_block_vs_long_double(gpu, refs, case):
    A0, db, g, a, z0, zm = batch_case(case)
    r = gpu._device.yaman4_transfer(db, g, a, A0, 0xFF, z0=z0, z_max=zm, n_steps=N_STEPS)
    ref = refs(("batch", case), lambda: reference(A0, db, g, a, z0, zm, N_STEPS))
    n_zero = 8 * sum(1 for _, ps, pi in POINTS if ps == pi == 0)
    G, deep = _check_run(gpu, r, A0, ref, f"batch {case}", zero_blocks=n_zero)
    assert G >= 1e4 and deep >= 1
    if case == "z0":
        assert abs(db[-1] * z0) > 900


def test_long_run_every_block_vs_long_double(gpu, refs):
    """10 000 steps over 2 000 m at 0.125 + 0.125 W: the same 2 r L as the 500 m cases, 37.5 dB at the peak once the
    pumps' loss over 2 000 m (1 dB) is taken."""
    P, n = 0.125, 10000
    pts = [(0.0, 1e-4, 0.0), (0.0, 1e-13, 1e-13), (0.004, 1e-9, 0.0), (0.0, 0.0, 0.0), (-0.003, 1e-9, 1e-10)]
    b = np.arange(len(pts))
    A0 = np.sqrt([[P, P, ps, pi] for _, ps, pi in pts]) * \
        np.exp(1j * np.stack([0.1 + 0.3 * b, -0.2 - 0.5 * b, 0.3 + 0.7 * b, 0.05 - 0.4 * b], axis=1))
    db = np.array([k for k, _, _ in pts]) - GAMMA * 2 * P
    r = gpu._device.yaman4_transfer(db, GAMMA, ALPHA, A0, 0xFF, z_max=n * DZ, n_steps=n)
    ref = refs("long", lambda: TL.transfer_ld(A0, GAMMA, ALPHA, db, z_max=n * DZ, n_steps=n))
    G, _ = _check_run(gpu, r, A0, ref, "batch 10 000 steps", zero_blocks=8)
    assert 10 ** 3.5 <= G <= 10 ** 4.5


# ------------------------------------------------------------------ sweeps
def _sweep(gpu, name):
    unit, p_in, phase_in = SWEEPS[name]
    s = 1.0 if unit == "m" else 1e-3
    cfg = gpu.config.custom_simulation_config(z_max=L * s, dz=DZ * s, save_every=10)
    kw = dict(cfg=cfg, lambda_p1_m=LAM_P1, lambda_p2_m=LAM_P2, lambda_signal_m=LAM_S, gamma=GAMMA / s, alpha=ALPHA / s,
              p_in=p_in, phase_in=phase_in, dispersion=_bench_dispersion(gpu, 1.0 / s), length_unit=unit)
    return kw, gpu.scan_mismtach.sweep_transfer_2d(waves=(0, 1, 2, 3), **kw)


def _run_dbeta(gpu, kw):
    """The FP64 dbeta the sweep kernel integrates: the reported one in m units; in km units the plan's dbeta with every
    beta_n divided by 1000, computed by the same device code (fpa_dbeta_table_host)."""
    sm = gpu.scan_mismtach
    plan, keep = gpu._device.new_plan_desc(kw["lambda_p1_m"], kw["lambda_p2_m"], kw["lambda_signal_m"])
    gpu.phase_matching.fill_plan_desc(plan, kw["dispersion"], sm._default_phase_matching_cfg(
        dispersion=kw["dispersion"], beta_legacy=None))
    sc = 1.0 if kw["length_unit"] == "m" else 1000.0
    for n in range(len(plan.beta)):
        plan.beta[n] = plan.beta[n] / sc
    plan.provided = plan.provided / sc
    return gpu._device.dbeta_table(plan)["dbeta"]


@pytest.mark.parametrize("name", list(SWEEPS))
def test_sweep_every_block_vs_long_double(gpu, refs, name):
    kw, r = _sweep(gpu, name)
    unit = kw["length_unit"]
    sc = 1.0 if unit == "m" else 1000.0
    assert r["n_steps"] == N_STEPS and np.all(r["valid"] == 1)
    # the run's constants per metre, formed as the kernel forms them
    gam, alp, z_run = kw["gamma"] / sc, kw["alpha"] / sc, kw["cfg"].z_max * sc
    db = _run_dbeta(gpu, kw)
    if unit == "m":
        assert db.tobytes() == r["dbeta"].tobytes()
    # the run dbeta is the one integrated: the batch integrator from it gives the sweep's A_end bit for bit
    A0 = gpu.simulation.make_initial_amplitudes(kw["p_in"], kw["phase_in"])
    B = db.size
    e = gpu._device.yaman4_batch(db.reshape(-1), gam, alp, np.tile(A0, (B, 1)), z_max=z_run,
                                n_steps=N_STEPS)["A_end"]
    assert e.tobytes() == r["A_end"].reshape(B, 4).tobytes(), name
    n_off = int(np.sum(db != r["dbeta"] / sc))
    ref = refs(("sweep", name), lambda: TL.transfer_ld(np.tile(A0, (B, 1)), gam, alp, db.reshape(-1),
                                                        z_max=z_run, n_steps=N_STEPS))
    zero = 8 * B if kw["p_in"][2] == kw["p_in"][3] == 0 else 0
    G, _ = _check_run(gpu, r, np.tile(A0, (B, 1)), ref, f"sweep {name}", zero_blocks=zero)
    assert G >= (1e3 if kw["p_in"][2] >= 1e-4 else 1e4)          # a 1e-4 W seed saturates the gain (32.6 dB)
    print(f"sweep {name}: integration dbeta differs from reported / {sc:g} on {n_off} of {B} points")
    if "sym" in name:
        # A1 = A2, A3 = A4: J commutes with the swap, to rounding (the kernel integrates the 4-wave system)
        jac = r["jac"].reshape(B, 8, 8)
        assert np.all(A0[0] == A0[1]) and np.all(A0[2] == A0[3])
        Jr = np.asarray(ref[1])
        assert_blocks(Jr[:, SWAP][:, :, SWAP], Jr, 1e-15, f"sweep {name} reference swap")
        worst, _ = assert_blocks(jac[:, SWAP][:, :, SWAP], jac, TOL, f"sweep {name} swap")
        print(f"sweep {name}: swap (1 <-> 2, 3 <-> 4) changes J by at most {worst:.1e} per block")
