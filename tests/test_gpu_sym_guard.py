"""GPU: the guard of the symmetric sweep kernels (stage_sym_fast, csrc/yaman4.cu).

The guarded z-loop computes stage_sym()'s bits while every stage's T = |A1|^2 + |A3|^2 stays below 2^1023; a run or
z-segment where it reached 2^1023 (or inf, or NaN) is replayed with stage_sym().  Negative loss makes T cross 2^1023
at a step set by alpha: with gamma = 0 while the components are still finite (where c2g * S and c4g * T can part:
c2g * inf against c4g * T), with gamma != 0 after the Kerr term has overflowed.
Each run must give the 4-wave kernels' bytes (FPA_SWEEP_SYM=0) on every output, on the whole-run kernel and on the
z-segment scheduler (the crossing falls in a middle segment and is replayed from the record).  The lambda3 grid puts
invalid scan points (not integrated) and integrated ones into the same warps."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
OUT_KEYS = ("gain_lin", "dbeta", "valid", "status", "Pmax", "A_end")
A1 = 0.1 ** 0.5 + 0j
A3 = 1e-7 ** 0.5 + 0j
WIDE = np.linspace(600e-9, 1700e-9, 1000)        # invalid plans below ~775 nm


def _env(**kw):
    for k in ("FPA_SWEEP_SYM", "FPA_SWEEP_SEG", "FPA_SWEEP_SEG_STEPS"):
        os.environ.pop(k, None)
    os.environ.update({k: str(v) for k, v in kw.items()})


@pytest.fixture(autouse=True)
def _clean_env():
    yield
    _env()


def _sweep(gpu, golden, n1, gamma, alpha, **env):
    b2, b3, b4, wref = golden["b4_beta"]
    disp = gpu.dispersion.DispersionParams(omega_ref=wref, beta2=b2, beta3=b3, beta4=b4)
    PM = gpu.phase_matching
    plan, keep = gpu._device.new_plan_desc(np.linspace(1545e-9, 1555e-9, n1), np.array([1558e-9]), WIDE)
    PM.fill_plan_desc(plan, disp, PM.PhaseMatchingConfig(method=PM.PhaseMatchingMethod("symmetric_even")))
    d = gpu._lib.SweepDesc()
    d.plan = plan
    for j, a in enumerate((A1, A1, A3, A3)):
        d.A0[2 * j], d.A0[2 * j + 1] = a.real, a.imag
    d.p_signal = abs(A3) ** 2
    d.gamma, d.alpha = gamma, alpha
    d.z_max, d.dz, d.length_scale, d.save_every = 37.4, 0.2, 1.0, 10
    d.flags = gpu._lib.CHECK_NAN
    _env(**env)
    return gpu._device.sweep(d, want_pmax=True, want_end=True)


# alpha: T stays below 2^1023 (-19.5, values near 1e307), or crosses it at steps ~182, ~167, ~144, ~127 of 187
@pytest.mark.parametrize("gamma", [0.0, 11.5e-3], ids=["gamma0", "kerr"])
@pytest.mark.parametrize("alpha", [-19.5, -20.0, -22.0, -26.0, -30.0])
@pytest.mark.parametrize("n1, seg_env", [(3, {}), (120, {"FPA_SWEEP_SEG_STEPS": 32})], ids=["whole-run", "segments"])
def test_runs_crossing_the_guard_give_the_4wave_bytes(gpu, golden, gamma, alpha, n1, seg_env):
    sym = _sweep(gpu, golden, n1, gamma, alpha, FPA_SWEEP_SYM=1, **seg_env)
    ref = _sweep(gpu, golden, n1, gamma, alpha, FPA_SWEEP_SYM=0, **seg_env)
    assert (ref["valid"] == 0).any() and (ref["valid"] == 1).any()
    if gamma == 0.0 and alpha == -19.5:
        assert (ref["status"][ref["valid"] == 1] == -1).all()      # healthy: no point failed
    if alpha <= -22.0:
        assert (ref["status"][ref["valid"] == 1] > 0).all()        # every integrated point failed mid-run
    for k in OUT_KEYS:
        assert sym[k].tobytes() == ref[k].tobytes(), (k, gamma, alpha, n1)
