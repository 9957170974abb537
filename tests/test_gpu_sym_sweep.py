"""GPU: the symmetric sweep kernels (stage_sym, csrc/yaman4.cu) against the 4-wave kernels.

With A0 = [A1, A1, A3, A3] bit for bit, the launcher integrates only (A1, A3); the results must be the 4-wave
kernels' bits on every output (gain, dbeta, valid, status, Pmax, A_end): whole-run kernel and z-segment scheduler
at 1, 1.65 and 8+ waves, m and km, lossy and lossless, every Delta-beta method, invalid plans, overflowing points,
sub-range launches, the host / device / multi-device entries and the ptxas-schedule build.  An A0 one ulp off
symmetric must take the 4-wave kernels.  `FPA_SWEEP_SYM=0` forces the 4-wave kernels.
"""
import ctypes as C
import os

import numpy as np
import pytest

import __graft_entry__ as entry

pytestmark = pytest.mark.gpu
WAVE = 148 * 6 * 4 * 32            # points that fill every resident warp once at 6 blocks of 128 threads per SM
OUT_KEYS = ("gain_lin", "dbeta", "valid", "status", "Pmax", "A_end")
A1 = 0.1 ** 0.5 + 0j
A3 = 1e-7 ** 0.5 + 0j


def _env(**kw):
    for k in ("FPA_SWEEP_SYM", "FPA_SWEEP_SEG", "FPA_SWEEP_SEG_STEPS"):
        os.environ.pop(k, None)
    os.environ.update({k: str(v) for k, v in kw.items()})


@pytest.fixture(autouse=True)
def _clean_env():
    yield
    _env()


def _desc(gpu, golden, n1, lam3, *, unit="m", alpha=1.15e-4, method="symmetric_even", A0=(A1, A1, A3, A3),
          gamma=11.5e-3, z_max=37.4, dz=0.2, save_every=10):
    s = 1.0 if unit == "m" else 1e-3
    b2, b3, b4, wref = golden["b4_beta"]
    k = 1.0 if unit == "m" else 1e3
    disp = gpu.dispersion.DispersionParams(omega_ref=wref, beta2=b2 * k, beta3=b3 * k, beta4=b4 * k)
    PM = gpu.phase_matching
    cfg = PM.PhaseMatchingConfig(method=PM.PhaseMatchingMethod(method),
                                 provided_delta_beta=(-2.5e-3 * k if method == "provided" else None))
    lam1 = np.linspace(1545e-9, 1555e-9, n1)
    plan, keep = gpu._device.new_plan_desc(lam1, np.array([1558e-9]), np.asarray(lam3, dtype=float))
    PM.fill_plan_desc(plan, disp, cfg)
    d = gpu._lib.SweepDesc()
    d.plan = plan
    for j in range(4):
        d.A0[2 * j], d.A0[2 * j + 1] = complex(A0[j]).real, complex(A0[j]).imag
    d.p_signal = abs(complex(A0[2])) ** 2
    d.gamma, d.alpha = gamma / s, alpha / s
    d.z_max, d.dz, d.length_scale, d.save_every = z_max * s, dz * s, 1000.0 if unit == "km" else 1.0, save_every
    d.flags = gpu._lib.CHECK_NAN
    return d, keep


def _run(gpu, d, devices=None, **env):
    _env(**env)
    return gpu._device.sweep(d, want_pmax=True, want_end=True, devices=devices)


def _same(a, b, what):
    for k in OUT_KEYS:
        assert a[k].tobytes() == b[k].tobytes(), (what, k)


WIDE = np.linspace(600e-9, 1700e-9, 1000)        # w4 <= 0 below ~775 nm: invalid plans (NaN, valid 0)


@pytest.mark.parametrize("n1, seg_env", [(3, {}), (114, {"FPA_SWEEP_SEG_STEPS": 32}), (190, {"FPA_SWEEP_SEG_STEPS": 32}),
                                         (1000, {"FPA_SWEEP_SEG": 2, "FPA_SWEEP_SEG_STEPS": 32})],
                         ids=["whole-run", "seg-1.0-wave", "seg-1.65-waves", "seg-8+-waves"])
def test_sym_paths_are_bit_identical_to_4wave(gpu, golden, n1, seg_env):
    d, keep = _desc(gpu, golden, n1, WIDE)
    assert n1 < 100 or n1 * 1000 >= WAVE
    sym = _run(gpu, d, FPA_SWEEP_SYM=1, **seg_env)
    ref = _run(gpu, d, FPA_SWEEP_SYM=0, **seg_env)
    assert np.isnan(ref["gain_lin"]).any() and np.isfinite(ref["gain_lin"]).any()
    assert (ref["valid"] == 0).any()
    _same(sym, ref, n1)
    # the scheduler computes what the whole-run kernel computes
    _same(sym, _run(gpu, d, FPA_SWEEP_SYM=1, FPA_SWEEP_SEG=0), "whole-run")


@pytest.mark.parametrize("unit", ["m", "km"])
@pytest.mark.parametrize("alpha", [1.15e-4, 0.0], ids=["lossy", "lossless"])
@pytest.mark.parametrize("method", ["symmetric_even", "general_taylor", "provided"])
def test_sym_physics_variants(gpu, golden, unit, alpha, method):
    for n1, env in ((2, {}), (120, {"FPA_SWEEP_SEG_STEPS": 64})):
        d, keep = _desc(gpu, golden, n1, WIDE if method != "provided" else np.linspace(1540e-9, 1565e-9, 1000),
                        unit=unit, alpha=alpha, method=method, save_every=7)
        _same(_run(gpu, d, FPA_SWEEP_SYM=1, **env), _run(gpu, d, FPA_SWEEP_SYM=0, **env), (unit, alpha, method, n1))


def test_overflowing_points_report_the_same_status(gpu, golden):
    """Negative loss (exponential growth) drives every state to overflow mid-run: same first non-finite step."""
    for n1, env in ((2, {}), (120, {"FPA_SWEEP_SEG_STEPS": 32})):
        d, keep = _desc(gpu, golden, n1, np.linspace(1540e-9, 1565e-9, 1000), alpha=-40.0)
        sym, ref = _run(gpu, d, FPA_SWEEP_SYM=1, **env), _run(gpu, d, FPA_SWEEP_SYM=0, **env)
        assert (ref["status"] > 0).all() and (ref["status"] < 187).all()
        _same(sym, ref, n1)


def test_sym_multi_device_entry(gpu, golden):
    n_dev = gpu._lib.device_count()
    d, keep = _desc(gpu, golden, 7, WIDE)
    ref = _run(gpu, d, FPA_SWEEP_SYM=0)
    for devices in ([0, n_dev - 1], [k % n_dev for k in range(3)]):
        _same(_run(gpu, d, devices=devices, FPA_SWEEP_SYM=1), ref, devices)


def test_sym_device_entry_sub_range(gpu, golden):
    """`fpa_yaman4_sweep_dev` with first_point / n_sub_points: the two halves equal the single launch."""
    import torch
    L, lib = gpu._lib, gpu._lib.lib()
    dev = torch.device("cuda", 0)
    L.check(lib.fpa_set_device(0))
    n1 = 130
    B = n1 * 1000

    def launch(first, count, sym):
        d, keep = _desc(gpu, golden, n1, WIDE)
        # the device entry reads the wavelength axes from device memory
        axes = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in keep]
        d.plan.lambda1, d.plan.lambda2, d.plan.lambda3 = (a.data_ptr() for a in axes)
        t = {k: torch.full((count * m,), -3, dtype=dt, device=dev)
             for k, dt, m in (("gain_lin", torch.float64, 1), ("dbeta", torch.float64, 1), ("valid", torch.int32, 1),
                              ("status", torch.int32, 1), ("Pmax", torch.float64, 4), ("A_end", torch.float64, 8))}
        nb = int(lib.fpa_yaman4_sweep_scratch_bytes(count))
        scr = torch.empty(max(nb, 16), dtype=torch.uint8, device=dev)
        d.plan.dbeta, d.plan.valid, d.plan.omega = t["dbeta"].data_ptr(), t["valid"].data_ptr(), None
        d.gain_lin, d.status, d.Pmax, d.A_end = (t["gain_lin"].data_ptr(), t["status"].data_ptr(), t["Pmax"].data_ptr(),
                                                 t["A_end"].data_ptr())
        if count != B:
            d.first_point, d.n_sub_points = first, count
        _env(FPA_SWEEP_SYM=int(sym), FPA_SWEEP_SEG_STEPS=32)
        L.check(lib.fpa_yaman4_sweep_dev(C.byref(d), scr.data_ptr(), nb, torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        return {k: v.cpu().numpy() for k, v in t.items()}

    whole = launch(0, B, False)
    cut = 97_001                                     # two ragged sub-ranges
    a, b = launch(0, cut, True), launch(cut, B - cut, True)
    for k in OUT_KEYS:
        assert np.concatenate([a[k], b[k]]).tobytes() == whole[k].tobytes(), k


def test_sym_sass_pass_build_matches_ptxas_schedule(gpu, golden):
    if b"re-scheduled" not in gpu._lib.lib().fpa_version():
        pytest.skip("library built with ptxas' own schedule")
    for n1, env in ((3, {}), (120, {"FPA_SWEEP_SEG_STEPS": 32})):
        for alpha in (1.15e-4, 0.0):
            d, keep = _desc(gpu, golden, n1, WIDE, alpha=alpha)
            new = _run(gpu, d, FPA_SWEEP_SYM=1, **env)
            with gpu._lib.use_library(entry.REF_LIB):
                ref = _run(gpu, d, FPA_SWEEP_SYM=1, **env)
            _same(new, ref, (n1, alpha))


def test_one_ulp_off_symmetric_takes_the_4wave_kernels(gpu, golden):
    """A2 one ulp off A1, or A4 = conj(A3) with a -0.0 imaginary part (equal in value, not in bits): FPA_SWEEP_SYM
    has no effect, the 4-wave kernels run either way."""
    A2 = complex(np.nextafter(A1.real, 1.0), 0.0)
    for A0 in ((A1, A2, A3, A3), (A1, A1, A3, complex(A3.real, -0.0))):
        for n1, env in ((3, {}), (120, {"FPA_SWEEP_SEG_STEPS": 32})):
            d, keep = _desc(gpu, golden, n1, WIDE, A0=A0)
            on, off = _run(gpu, d, FPA_SWEEP_SYM=1, **env), _run(gpu, d, FPA_SWEEP_SYM=0, **env)
            _same(on, off, (A0, n1))
            if A0[1] != A0[0]:                       # waves 2 of the 4-wave result are not copies of waves 1
                e = on["A_end"].reshape(-1, 4)
                ok = np.isfinite(e[:, 0])
                assert e[ok][:, 0].tobytes() != e[ok][:, 1].tobytes()
