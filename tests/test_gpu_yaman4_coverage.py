"""GPU: the 4-wave integrator started at z0 != 0, and its trace rows stored 16 bytes at a time.

Every integration path takes the phase exp(i*dbeta*z) from the absolute position z: the whole-run kernel re-syncs
it with sincos(dbeta * (i*h + z0)), the z-segment kernel does the same per segment, the exact kernel forms
z_i = i*step + z0.  A path that dropped z0 would still pass every run that starts at 0, so here the runs start at
z0 = 5 m and at z0 = 2000 m, where dbeta*z0 is ~1e3 rad and dropping z0 moves the signal and idler by 1-30 %:
  * against the oracle on numpy.linspace(z0, z_max, n+1), per-point and broadcast gamma / alpha, lossless and
    lossy, every output mode, a save period that does not divide the step count, fast and exact kernels;
  * bit for bit: the z-segment kernel against the whole-run kernel, the grid-free exact kernel against the exact
    kernel on the linspace grid (per-point against broadcast physics from z0: tests/test_gpu_edges.py).
save_sample writes a trace row as two 32-byte stores when A_trace is 32-byte aligned and as four 16-byte stores
otherwise; `_dev` runs with A_trace 16 bytes past a 32-byte boundary must give the aligned run's bytes on the
whole-run, z-segment and exact kernels.
"""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import rel_err

pytestmark = pytest.mark.gpu
ONE_WAVE = 148 * 16 * 32          # points that fill every resident warp of a B200 once (as in test_gpu_segments.py)
P_IN, PHASE_IN = [0.3, 0.4, 1e-3, 1e-4], [0.2, -0.1, 0.5, 1.0]
DBETA = np.array([0.5, -0.45, 0.31, 0.52, -0.6])     # 1/m: dbeta*z0 of -1200 .. 1040 rad at z0 = 2000 m
SAVE = 7                                             # divides neither step count below
STARTS = [(5.0, 105.0, 400), (2000.0, 2200.0, 500)]   # (z0, z_max, n_steps)
MODES = [("trace",), ("end", "pmax"), ("trace", "end", "pmax"), ("end",)]


def _env(**kw):
    for k in ("FPA_SWEEP_SEG", "FPA_SWEEP_SEG_STEPS"):
        os.environ.pop(k, None)
    os.environ.update({k: str(v) for k, v in kw.items()})


@pytest.fixture(autouse=True)
def _clean_env():
    yield
    _env()


@pytest.fixture(scope="module")
def A0(oracle):
    return oracle.initial_amplitudes(P_IN, PHASE_IN)


def _physics(per_point, lossy, B):
    """(gamma, alpha) broadcast scalars or per-point arrays."""
    if not per_point:
        return 0.02, (3e-4 if lossy else 0.0)
    rng = np.random.default_rng(7)
    return rng.uniform(0.01, 0.03, B), (rng.uniform(1e-4, 5e-4, B) if lossy else np.zeros(B))


def _run(gpu, modes, *args, **kw):
    return gpu._device.yaman4_batch(*args, trace="trace" in modes, end="end" in modes, pmax="pmax" in modes, **kw)


@pytest.mark.parametrize("per_point", [False, True], ids=["broadcast", "per_point"])
@pytest.mark.parametrize("lossy", [False, True], ids=["lossless", "lossy"])
@pytest.mark.parametrize("z0, z_max, n", STARTS)
def test_run_from_z0_matches_oracle(gpu, oracle, A0, z0, z_max, n, lossy, per_point):
    B = DBETA.size
    gamma, alpha = _physics(per_point, lossy, B)
    g, a = np.broadcast_to(gamma, B), np.broadcast_to(alpha, B)
    grid = np.linspace(z0, z_max, n + 1)
    ref = []
    for i in range(B):
        pt = oracle.YamanPoint(g[i], a[i], DBETA[i])
        A_all = oracle.march_grid(oracle.yaman_rhs_p, grid, A0, pt)[1]
        ref.append((A_all[::SAVE], A_all[-1]))
    # the oracle itself: a run from 0 over the same length differs far beyond the tolerances below
    shifted = oracle.march_grid(oracle.yaman_rhs_p, grid - z0, A0, oracle.YamanPoint(g[0], a[0], DBETA[0]))[1][-1]
    assert rel_err(shifted[2:], ref[0][1][2:]) > 1e-3
    kernels = {"fast": {}, "exact": dict(phase_exact=True), "grid": dict(z_grid=grid)}
    for name, extra in kernels.items():
        for modes in MODES:
            r = _run(gpu, modes, DBETA, gamma, alpha, A0, z0=z0, z_max=z_max, n_steps=n, save_every=SAVE, **extra)
            assert (r["status"] == -1).all(), (name, modes)
            for i, (tr, end) in enumerate(ref):
                if "trace" in modes:
                    assert r["A_trace"].shape[1] == n // SAVE + 1
                    assert np.max(np.abs(r["A_trace"][i] - tr)) / np.max(np.abs(tr)) < 1e-11, (name, modes, i)
                if "end" in modes:
                    assert rel_err(r["A_end"][i], end) < 1e-10, (name, modes, i)
                if "pmax" in modes:
                    assert rel_err(r["Pmax"][i], (np.abs(tr) ** 2).max(axis=0)) < 1e-10, (name, modes, i)


@pytest.mark.parametrize("modes", [("end", "pmax"), ("trace",), ("trace", "end", "pmax")])
def test_segmented_run_from_z0_is_bit_identical_to_whole_run(gpu, A0, modes):
    """Broadcast physics (per-point physics never segments), 1.06 waves, ragged, lossless and lossy."""
    B = ONE_WAVE + 4321
    db = np.linspace(-0.6, 0.6, B)
    for alpha in (0.0, 3e-4):
        kw = dict(z0=2000.0, z_max=2040.0, n_steps=160, save_every=SAVE)
        _env(FPA_SWEEP_SEG=0)
        whole = _run(gpu, modes, db, 0.02, alpha, A0, **kw)
        _env(FPA_SWEEP_SEG_STEPS=32)
        segd = _run(gpu, modes, db, 0.02, alpha, A0, **kw)
        assert (whole["status"] == -1).all()
        for k, v in whole.items():
            assert v.tobytes() == segd[k].tobytes(), (k, alpha)


@pytest.mark.parametrize("per_point", [False, True], ids=["broadcast", "per_point"])
def test_grid_free_exact_run_from_z0_equals_linspace_grid(gpu, A0, per_point):
    """numpy.linspace forms i*step + z0 with two roundings and sets the last point to z_max; so does the grid-free
    exact kernel: the same abscissae, the same bits."""
    B = DBETA.size
    gamma, alpha = _physics(per_point, True, B)
    for z0, z_max, n in STARTS + [(0.37, 1000.1, 777), (-12.5, 3.3, 101)]:
        grid = np.linspace(z0, z_max, n + 1)
        assert np.array_equal(grid[:-1], np.arange(n) * ((z_max - z0) / n) + z0) and grid[-1] == z_max
        kw = dict(z0=z0, z_max=z_max, n_steps=n, save_every=SAVE)
        free = _run(gpu, MODES[2], DBETA, gamma, alpha, A0, phase_exact=True, **kw)
        on_grid = _run(gpu, MODES[2], DBETA, gamma, alpha, A0, z_grid=grid, **kw)
        for k in ("A_trace", "A_end", "Pmax", "status"):
            assert free[k].tobytes() == on_grid[k].tobytes(), (k, z0)


# ------------------------------------------------------------------ the 16-byte trace store branch
def _dev_batch(gpu, A0, db, *, shift, uniform, exact, scratch, n_steps, save_every, z0, z_max):
    """fpa_yaman4_rk4_batch_dev on torch tensors, A_trace and A_end starting `shift` bytes past their allocations;
    returns the bytes of every output."""
    import torch
    L, lib, dev = gpu._lib, gpu._lib.lib(), torch.device("cuda", 0)
    L.check(lib.fpa_set_device(0))
    B = db.size
    ns = n_steps // save_every + 1
    t_db = torch.from_numpy(db).to(dev)
    t_g = torch.full((B if not uniform else 1,), 0.02, dtype=torch.float64, device=dev)
    t_a = torch.full((B if not uniform else 1,), 3e-4, dtype=torch.float64, device=dev)
    t_A0 = torch.from_numpy(np.tile(A0, (B, 1)).view(np.float64).copy()).to(dev)
    out = {"A_trace": torch.empty(B * ns * 64 + shift, dtype=torch.uint8, device=dev)[shift:],
           "A_end": torch.empty(B * 64 + shift, dtype=torch.uint8, device=dev)[shift:],
           "Pmax": torch.empty(B * 32, dtype=torch.uint8, device=dev),
           "status": torch.empty(B * 4, dtype=torch.uint8, device=dev)}
    d = L.Yaman4Desc()
    d.n_points, d.z0, d.z_max, d.n_steps, d.save_every = B, z0, z_max, n_steps, save_every
    d.dbeta, d.gamma, d.alpha, d.A0 = (t.data_ptr() for t in (t_db, t_g, t_a, t_A0))
    d.gamma_stride = d.alpha_stride = 0 if uniform else 1
    d.A0_stride = 1
    d.flags = L.CHECK_NAN | L.OUT_TRACE | L.OUT_END | L.OUT_PMAX | (L.PHASE_EXACT if exact else 0)
    if uniform:
        d.flags |= L.UNIFORM_PHYSICS
        d.gamma_uniform, d.alpha_uniform = 0.02, 3e-4
    d.A_trace, d.A_end, d.Pmax, d.status = (out[k].data_ptr() for k in ("A_trace", "A_end", "Pmax", "status"))
    if scratch:
        nb = int(lib.fpa_yaman4_scratch_bytes(B))
        t_scr = torch.empty(nb, dtype=torch.uint8, device=dev)
        d.scratch, d.scratch_bytes = t_scr.data_ptr(), nb
    L.check(lib.fpa_yaman4_rk4_batch_dev(C.byref(d), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return {k: v.cpu().numpy().tobytes() for k, v in out.items()}


@pytest.mark.parametrize("kernel", ["whole_run", "whole_run_per_point", "z_segment", "exact"])
def test_trace_rows_off_a_32_byte_boundary_equal_aligned_rows(gpu, A0, kernel):
    seg = kernel == "z_segment"
    B = ONE_WAVE + 4321 if seg else 1000
    db = np.linspace(-0.6, 0.6, B)
    kw = dict(uniform=kernel in ("whole_run", "z_segment"), exact=kernel == "exact", scratch=seg, n_steps=96,
              save_every=SAVE, z0=5.0, z_max=25.0)
    if seg:
        _env(FPA_SWEEP_SEG_STEPS=32)
    aligned = _dev_batch(gpu, A0, db, shift=0, **kw)
    off = _dev_batch(gpu, A0, db, shift=16, **kw)
    assert np.frombuffer(aligned["status"], np.int32).tolist() == [-1] * B
    for k in aligned:
        assert off[k] == aligned[k], k
