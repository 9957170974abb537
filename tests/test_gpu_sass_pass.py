"""GPU: the library whose FP64 hot loops were re-scheduled after ptxas (tools/sass_sched.py) must
give results BIT-IDENTICAL to the same sources with ptxas' own schedule
(build/libfpa_b200_ref.so).  The pass only re-orders instructions, swaps commutative operands and
sets operand-reuse flags, so any differing bit is a scheduling hazard."""
import numpy as np
import pytest

import __graft_entry__ as entry

pytestmark = pytest.mark.gpu


def _both(gpu, fn):
    out = fn()
    if not entry.REF_LIB.exists():
        pytest.fail("build/libfpa_b200_ref.so missing: build() did not produce the reference-schedule library")
    with gpu._lib.use_library(entry.REF_LIB) as ref:
        # every call of the package now goes through the reference-schedule build
        assert gpu._lib.lib() is ref and b"ptxas schedule" in gpu._lib.lib().fpa_version()
        out_ref = fn()
    assert b"re-scheduled" in gpu._lib.lib().fpa_version()
    return out, out_ref


def _same(a, b):
    for k in a:
        if isinstance(a[k], np.ndarray):
            assert a[k].tobytes() == b[k].tobytes(), f"{k} differs between the two schedules"


def test_shipped_library_carries_the_pass(gpu):
    assert b"re-scheduled after ptxas" in gpu._lib.lib().fpa_version()


@pytest.mark.parametrize("alpha", [0.0, 1.15e-4])
def test_fused_sweep_bit_identical(gpu, golden, alpha):
    b2, b3, b4, wref = golden["b4_beta"]
    cfg = gpu.config.custom_simulation_config(z_max=100.0, dz=0.2, save_every=10)
    lam1 = np.linspace(1545e-9, 1555e-9, 64)
    lam3 = np.linspace(1540e-9, 1565e-9, 1000)
    disp = gpu.dispersion.DispersionParams(omega_ref=wref, beta2=b2, beta3=b3, beta4=b4)
    run = lambda: gpu.scan_mismtach.sweep_gain_2d(  # noqa: E731
        cfg=cfg, lambda_p1_m=lam1, lambda_signal_m=lam3, lambda_p2_m=1558e-9, gamma=11.5e-3, alpha=alpha,
        p_in=golden["b4_p_in"], dispersion=disp, gain_unit="linear")
    a, b = _both(gpu, run)
    _same(a, b)
    assert np.isfinite(a["gain"]).all()


@pytest.mark.parametrize("outputs", [("end", "pmax"), ("trace",), ("end",), ("trace", "end", "pmax")])
@pytest.mark.parametrize("uniform", [True, False])
@pytest.mark.parametrize("alpha", [0.0, 2e-4])
def test_batch_integrator_bit_identical(gpu, outputs, uniform, alpha):
    """Every instantiation of the fast kernel: TRACE/PMAX x {uniform, lossless, per-point physics}."""
    cfg = gpu.config.custom_simulation_config(z_max=300.0, dz=0.25, save_every=7)
    rng = np.random.default_rng(5)
    B = 20_000
    db = rng.normal(size=B) * 0.02
    gamma = 11.5e-3 if uniform else rng.uniform(5e-3, 2e-2, B)
    al = alpha if uniform else np.full(B, alpha)
    run = lambda: gpu.simulation.run_batch_simulation(  # noqa: E731
        cfg, gamma=gamma, alpha=al, delta_beta=db, p_in=[0.3, 0.2, 1e-4, 1e-6], outputs=outputs)
    a, b = _both(gpu, run)
    _same(a, b)


@pytest.mark.parametrize("grid", [False, True])
def test_exact_phase_kernel_bit_identical(gpu, grid):
    rng = np.random.default_rng(6)
    B = 4096
    db = rng.normal(size=B) * 0.05
    if grid:
        z = np.cumsum(np.concatenate(([0.0], rng.uniform(0.05, 0.3, 400))))
        A0 = np.tile(np.sqrt(np.array([0.3, 0.2, 1e-4, 1e-6])).astype(complex), (B, 1))
        run = lambda: gpu._device.yaman4_batch(  # noqa: E731
            db, np.asarray(11.5e-3), np.asarray(2e-4), A0, z_max=float(z[-1]), n_steps=z.size - 1, z_grid=z,
            save_every=5, trace=True, end=True,
            pmax=True, check_nan=True, phase_exact=True)
    else:
        cfg = gpu.config.custom_simulation_config(z_max=100.0, dz=0.25, save_every=5)
        run = lambda: gpu.simulation.run_batch_simulation(  # noqa: E731
            cfg, gamma=11.5e-3, alpha=2e-4, delta_beta=db, p_in=[0.3, 0.2, 1e-4, 1e-6],
            outputs=("end", "pmax", "trace"), phase_exact=True)
    a, b = _both(gpu, run)
    _same(a, b)


def test_segment_scheduler_kernels_bit_identical(gpu, golden):
    """The persistent (z-segment scheduler) instantiations go through the pass too; they only run for batches of
    one wave of the resident warps or more, so they need their own comparison with the ptxas-schedule build:
    the fused sweep (lossy and lossless) and the batch integrator in every output mode."""
    b2, b3, b4, wref = golden["b4_beta"]
    disp = gpu.dispersion.DispersionParams(omega_ref=wref, beta2=b2, beta3=b3, beta4=b4)
    cfg = gpu.config.custom_simulation_config(z_max=40.0, dz=0.2, save_every=7)
    lam1 = np.linspace(1545e-9, 1555e-9, 90)
    lam3 = np.linspace(1540e-9, 1565e-9, 1000)          # 90 000 points = 1.19 waves
    for alpha in (0.0, 1.15e-4):
        run = lambda: gpu.scan_mismtach.sweep_gain_2d(  # noqa: E731
            cfg=cfg, lambda_p1_m=lam1, lambda_signal_m=lam3, lambda_p2_m=1558e-9, gamma=11.5e-3, alpha=alpha,
            p_in=golden["b4_p_in"], dispersion=disp, gain_unit="linear", want_pmax=True)
        a, b = _both(gpu, run)
        _same(a, b)
    db = np.linspace(-40.0, 40.0, 80_000)
    cfg3 = gpu.config.custom_simulation_config(z_max=0.13, dz=1e-3, save_every=10)
    for outputs in (("end", "pmax"), ("trace",), ("end",), ("trace", "end", "pmax")):
        for alpha in (0.0, 0.2):
            run = lambda: gpu.simulation.run_batch_simulation(      # noqa: E731
                cfg3, gamma=10.0, alpha=alpha, delta_beta=db, p_in=[0.1, 0.1, 1e-5, 0.0], length_unit="km", outputs=outputs)
            a, b = _both(gpu, run)
            _same(a, b)


def test_comb_batch_kernel_bit_identical(gpu):
    """`nwave_comb8_kernel` goes through the pass in flags-only mode (ptxas' order kept, yield hints cleared,
    operand-reuse flags set): it must agree bit for bit with the ptxas-schedule build."""
    batch = 640
    nw = gpu.nwave
    w0 = 2 * np.pi * 299792458.0 / 1550e-9
    for lines in (range(-32, 32), range(-10, 11), [0, 1, 2, 3, 5, 8, 13, 21, 34, 55, 89]):
        plan = nw.uniform_comb_plan(w0, 2 * np.pi * 100e9, lines)
        N = plan.n_waves
        beta = nw.beta_per_wave(plan, gpu.dispersion.DispersionParams(omega_ref=w0, beta2=-2.57e-29, beta3=3.30e-41,
                                                                       beta4=-1.63e-55))
        rng = np.random.default_rng(N)
        A0 = np.sqrt(rng.uniform(1e-6, 0.2, (batch, N))) * np.exp(1j * rng.uniform(0, 6.28, (batch, N)))
        cfg = gpu.config.custom_simulation_config(z_max=15.0, dz=0.1, save_every=50)
        run = lambda: nw.run_nwave_simulation(cfg, plan, gamma=11.5e-3, alpha=2e-4, A0=A0, beta=beta,   # noqa: E731
                                              outputs=("trace", "end", "pmax"), form="comb")
        a, b = _both(gpu, run)
        _same(a, b)
