"""GPU: the `_dev` entries refuse a device pointer that a kernel reads or writes with 16-byte vector accesses when it
is only 8-byte aligned (a complex128 tensor view at an odd element offset, say).  Such an access is a misaligned
address on the GPU, which would end the process's CUDA context; the launchers check the pointers first.  For every
entry and every such pointer, moved 8 bytes past its allocation one at a time: FPA_ERR_INVALID, an error text that
names the pointer and says "aligned", and every output keeps its sentinel bytes (nothing was queued).  The same
descriptor with every pointer aligned runs and writes every output."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
SENTINEL = 0xA5
P_IN, PHASE_IN = [0.1, 0.1, 1e-4, 2e-5], [0.1, -0.2, 0.3, 0.05]
GRID = np.array([0, 1, 3, 4, 6, 7])       # N-wave plan: six lines of an integer grid
N = GRID.size


class Bufs:
    """Device buffers of one call.  The one named k in `shift` starts shift[k] bytes past its (256-byte aligned)
    allocation; outputs are filled with the sentinel byte."""

    def __init__(self, shift):
        import torch
        self.torch, self.shift, self.keep, self.outs = torch, shift, [], {}

    def _alloc(self, name, nbytes):
        s = self.shift.get(name, 0)
        t = self.torch.empty(nbytes + s, dtype=self.torch.uint8, device="cuda:0")[s:]
        self.keep.append(t)
        return t

    def inp(self, name, arr):
        raw = np.ascontiguousarray(arr).reshape(-1).view(np.uint8)
        t = self._alloc(name, raw.size)
        t.copy_(self.torch.from_numpy(raw.copy()))
        return t.data_ptr()

    def out(self, name, nbytes):
        t = self._alloc(name, nbytes)
        t.fill_(SENTINEL)
        self.outs[name] = t
        return t.data_ptr()


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def _batch(gpu, golden, b):
    L = gpu._lib
    B, steps, save = 300, 40, 7
    ns = steps // save + 1
    rng = np.random.default_rng(1)
    A0 = (np.sqrt(np.array(P_IN)) * np.exp(1j * np.array(PHASE_IN)) * (1.0 + 0.01 * rng.standard_normal((B, 1))))
    d = L.Yaman4Desc()
    d.n_points, d.z_max, d.n_steps, d.save_every = B, 5.0, steps, save
    d.dbeta = b.inp("dbeta", rng.uniform(-1.0, 1.0, B))
    d.gamma, d.alpha = b.inp("gamma", np.array([0.02])), b.inp("alpha", np.array([1e-3]))
    d.A0, d.A0_stride = b.inp("A0", A0.astype(np.complex128)), 1
    d.flags = L.CHECK_NAN | L.OUT_TRACE | L.OUT_END | L.OUT_PMAX
    d.A_trace, d.A_end = b.out("A_trace", B * ns * 64), b.out("A_end", B * 64)
    d.Pmax, d.status = b.out("Pmax", B * 32), b.out("status", B * 4)
    return lambda: L.lib().fpa_yaman4_rk4_batch_dev(C.byref(d), _stream())


def _plan(gpu, golden, b, n1=2, n3=16):
    b2, b3, b4, wref = golden["b4_beta"]
    disp = gpu.dispersion.DispersionParams(omega_ref=wref, beta2=b2, beta3=b3, beta4=b4)
    plan, (l1, l2, l3) = gpu._device.new_plan_desc(np.linspace(1545e-9, 1555e-9, n1), 1558e-9,
                                                   np.linspace(1540e-9, 1565e-9, n3))
    gpu.phase_matching.fill_plan_desc(plan, disp, gpu.phase_matching.PhaseMatchingConfig())
    plan.lambda1, plan.lambda2, plan.lambda3 = b.inp("lambda1", l1), b.inp("lambda2", l2), b.inp("lambda3", l3)
    G = n1 * n3
    plan.dbeta, plan.valid, plan.omega = b.out("dbeta", G * 8), b.out("valid", G * 4), b.out("omega", G * 32)
    return plan, G


def _fill_sweep(gpu, golden, b, w, K):
    L = gpu._lib
    w.plan, G = _plan(gpu, golden, b)
    A0 = gpu.simulation.make_initial_amplitudes(P_IN, PHASE_IN)
    for j in range(4):
        w.A0[2 * j], w.A0[2 * j + 1] = A0[j].real, A0[j].imag
    w.p_signal, w.gamma, w.alpha = P_IN[2], 11.5e-3, 1e-4
    w.z_max, w.dz, w.length_scale, w.save_every = 4.0, 0.2, 1.0, 7
    w.flags = L.CHECK_NAN
    w.gain_lin, w.status = b.out("gain_lin", G * K * 8), b.out("status", G * K * 4)
    w.Pmax, w.A_end = b.out("Pmax", G * K * 32), b.out("A_end", G * K * 64)
    return G


def _sweep(gpu, golden, b):
    d = gpu._lib.SweepDesc()
    _fill_sweep(gpu, golden, b, d, 1)
    return lambda: gpu._lib.lib().fpa_yaman4_sweep_dev(C.byref(d), None, 0, _stream())


def _phase_sweep(gpu, golden, b):
    L, K = gpu._lib, 3
    table, _, _ = gpu.scan_mismtach.phase_sweep_inputs(P_IN, PHASE_IN, np.linspace(0.0, 2.0, K))
    d = L.PhaseSweepDesc()
    G = _fill_sweep(gpu, golden, b, d.sweep, K)
    d.n_phases, d.A0_table, d.metric = K, b.inp("A0_table", table), L.GAIN_MAX_SAVED
    for k, size in (("gain_max", 8), ("gain_min", 8), ("idx_max", 4), ("idx_min", 4), ("n_finite", 4)):
        setattr(d, k, b.out(k, G * size))
    return lambda: L.lib().fpa_yaman4_phase_sweep_dev(C.byref(d), None, 0, _stream())


def _dbeta_table(gpu, golden, b):
    plan, _ = _plan(gpu, golden, b)
    return lambda: gpu._lib.lib().fpa_dbeta_table_dev(C.byref(plan), _stream())


def _nwave(form):
    def setup(gpu, golden, b):
        L = gpu._lib
        B, steps, save = 40, 30, 7
        ns = steps // save + 1
        rng = np.random.default_rng(2)
        A0 = np.sqrt(rng.uniform(1e-4, 0.1, (B, N))) * np.exp(1j * rng.uniform(0.0, 6.28, (B, N)))
        d = L.NwaveDesc()
        d.n_points, d.n_waves, d.z_max, d.n_steps, d.save_every = B, N, 10.0, steps, save
        d.beta, d.beta_stride = b.inp("beta", rng.uniform(-1.0, 1.0, (B, N))), 1
        d.gamma, d.alpha = b.inp("gamma", np.array([11.5e-3])), b.inp("alpha", np.array([1e-4]))
        d.A0, d.A0_stride = b.inp("A0", A0.astype(np.complex128)), 1
        d.flags = L.CHECK_NAN | L.OUT_TRACE | L.OUT_END | L.OUT_PMAX
        d.A_trace, d.A_end = b.out("A_trace", B * ns * N * 16), b.out("A_end", B * N * 16)
        d.Pmax, d.status = b.out("Pmax", B * N * 8), b.out("status", B * 4)
        if form == "comb":
            slots = np.ascontiguousarray(GRID - GRID.min(), dtype=np.int32)
            d.grid_slot, d.grid_span = b.inp("grid_slot", slots), int(slots.max() + 1)
            d.flags |= L.NWAVE_COMB
        else:
            table, rows = gpu._device.enumerate_triplets(GRID)
            blob, n_classes = gpu._device.factor_table(N, table, rows)
            d.triplets, d.row_ptr, d.n_triplets = b.inp("triplets", table), b.inp("row_ptr", rows), table.size
            d.factored, d.n_classes = b.inp("factored", blob), n_classes
            d.flags |= L.NWAVE_TABLE
        return lambda: L.lib().fpa_nwave_rk4_batch_dev(C.byref(d), _stream())
    return setup


# entry -> (descriptor builder, {buffer: the name the error text gives it}) for every pointer a kernel of the entry
# reads or writes 16 bytes at a time
CASES = {
    "batch": (_batch, {"A0": "A0", "A_trace": "A_trace", "A_end": "A_end", "Pmax": "Pmax"}),
    "sweep": (_sweep, {"omega": "plan.omega", "A_end": "A_end", "Pmax": "Pmax"}),
    "phase_sweep": (_phase_sweep, {"A0_table": "A0_table", "omega": "plan.omega", "A_end": "A_end", "Pmax": "Pmax"}),
    "dbeta_table": (_dbeta_table, {"omega": "omega"}),
    "nwave_comb": (_nwave("comb"), {"A0": "A0", "A_trace": "A_trace", "A_end": "A_end"}),
    "nwave_table": (_nwave("table"), {"A0": "A0", "A_trace": "A_trace", "A_end": "A_end", "factored": "factored"}),
}


@pytest.mark.parametrize("entry", list(CASES))
def test_dev_entry_refuses_pointers_its_kernels_cannot_access(gpu, golden, entry):
    import torch
    L = gpu._lib
    L.check(L.lib().fpa_set_device(0))
    setup, names = CASES[entry]
    b = Bufs({})
    L.check(setup(gpu, golden, b)())
    torch.cuda.synchronize()
    for k, t in b.outs.items():
        assert (t != SENTINEL).any(), (entry, k)
    for buf, text in names.items():
        b = Bufs({buf: 8})
        rc = setup(gpu, golden, b)()
        err = L.last_error()
        torch.cuda.synchronize()
        assert rc == L.ERR_INVALID and f"{text} must be 16-byte aligned" in err, (entry, buf, rc, err)
        for k, t in b.outs.items():
            assert (t == SENTINEL).all(), (entry, buf, k)
