"""GPU: the staging of the host-pointer entry points.  Which result buffers the kernels write directly (page-locked
memory) and which go through the device workspace and a copy must not change what a caller gets: every output is
byte-equal whether it lives in pageable, pinned (`_lib.pinned_empty`), registered (`fpa_host_register`) or mixed
memory, and whether the optional outputs are requested or NULL.  The batch, sweep, phase-sweep and N-wave entries
also equal their `_dev` entry on torch tensors given the descriptor the host entry builds, the *_multi_host entries
with devices=[0, 0, 0] equal the single-device call, and a large call after a small one (the grow-only workspace)
repeats its bytes."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
KINDS = ("pageable", "pinned", "registered", "mixed", "null")
P_IN, PHASE_IN = [0.1, 0.1, 1e-4, 2e-5], [0.1, -0.2, 0.3, 0.05]
PAGE = 4096


class Mem:
    """Result arrays of one memory kind, filled with a sentinel byte; `optional` arrays are None for kind 'null'."""

    def __init__(self, L, kind):
        self.L, self.kind, self.n, self.registered = L, kind, 0, []

    def __call__(self, shape, dtype, optional=False):
        if optional and self.kind == "null":
            return None
        self.n += 1
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        if self.kind == "pinned" or (self.kind == "mixed" and self.n % 2):
            a = self.L.pinned_empty(shape, dtype)
        elif self.kind == "registered":
            # whole pages of its own: two registrations never share a page
            span = -(-nbytes // PAGE) * PAGE
            buf = np.empty(span + PAGE, np.uint8)
            off = -buf.ctypes.data % PAGE
            self.L.register_host(buf[off:off + span])
            self.registered.append(buf[off:off + span])
            a = buf[off:off + nbytes].view(dtype).reshape(shape)
        else:
            a = np.empty(shape, dtype)
        a.view(np.uint8)[...] = 0xA5
        return a

    def release(self):
        for a in self.registered:
            self.L.unregister_host(a)


def _ptr(L, a):
    return None if a is None else L.ptr(a)


def _run_kinds(gpu, build, size):
    """{kind: {output: bytes}} of build(mem, size) run once per memory kind; all agree with 'pageable'."""
    L, got = gpu._lib, {}
    for kind in KINDS:
        mem = Mem(L, kind)
        try:
            outs = build(mem, size)
            got[kind] = {k: v.tobytes() for k, v in outs.items() if v is not None}
        finally:
            mem.release()
    ref = got["pageable"]
    for kind, outs in got.items():
        assert outs.keys() <= ref.keys() and outs, kind
        for k, v in outs.items():
            assert v == ref[k], (kind, k)
    assert got["null"].keys() < ref.keys()
    return ref


def _dev_tensors(arrays):
    import torch
    dev = torch.device("cuda", 0)
    return {k: torch.from_numpy(np.ascontiguousarray(v).reshape(-1).view(np.uint8).copy()).to(dev)
            for k, v in arrays.items()}


def _dev_out(template):
    """Device buffers shaped like the host outputs (by bytes)."""
    import torch
    return {k: torch.empty(len(v), dtype=torch.uint8, device="cuda:0") for k, v in template.items()}


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def _sync_bytes(t):
    import torch
    torch.cuda.synchronize()
    return {k: v.cpu().numpy().tobytes() for k, v in t.items()}


def _check_sizes(gpu, build, sizes, dev=None, multi_size=None):
    """Large, small, large: each size agrees across memory kinds (and with `dev`); the repeated size repeats."""
    seen = {}
    for s in sizes:
        ref = _run_kinds(gpu, build, s)
        if s in seen:
            assert ref == seen[s]
        seen[s] = ref
        if dev is not None:
            want = dev(s, ref)
            for k, v in want.items():
                assert v == ref[k], (s, k)
    if multi_size is not None:
        one = _run_kinds(gpu, build, multi_size)
        mem = Mem(gpu._lib, "pageable")
        many = {k: v.tobytes() for k, v in build(mem, multi_size, devices=[0, 0, 0]).items()}
        assert many == one


# ----------------------------------------------------------------- 4-wave batch
def _batch_inputs(B):
    rng = np.random.default_rng(B)
    A0 = np.sqrt(np.array(P_IN)) * np.exp(1j * np.array(PHASE_IN))
    A0 = (A0 * (1.0 + 0.01 * rng.standard_normal((B, 1)))).astype(np.complex128)
    return {"dbeta": rng.uniform(-3.0, 3.0, B), "gamma": np.array([11.5e-3]), "alpha": np.array([1e-4]), "A0": A0}


STEPS, SAVE = 300, 7


def _batch_desc(L, B, inp, out):
    d = L.Yaman4Desc()
    d.n_points, d.z_max, d.n_steps, d.save_every = B, 150.0, STEPS, SAVE
    for k in ("dbeta", "gamma", "alpha", "A0"):
        setattr(d, k, inp[k] if isinstance(inp[k], int) else L.ptr(inp[k]))
    d.A0_stride = 1
    d.flags = L.CHECK_NAN
    for key, flag in (("A_trace", L.OUT_TRACE), ("A_end", L.OUT_END), ("Pmax", L.OUT_PMAX)):
        if out.get(key) is not None:
            d.flags |= flag
    return d


def test_batch(gpu):
    L, lib = gpu._lib, gpu._lib.lib()
    ns = STEPS // SAVE + 1

    def build(mem, B, devices=None):
        inp = _batch_inputs(B)
        out = {"A_trace": mem((B, ns, 4), np.complex128, True), "A_end": mem((B, 4), np.complex128),
               "Pmax": mem((B, 4), np.float64, True), "status": mem(B, np.int32, True)}
        d = _batch_desc(L, B, inp, out)
        for k, v in out.items():
            setattr(d, k, _ptr(L, v))
        gpu._device._run_host(lib.fpa_yaman4_rk4_batch_host, lib.fpa_yaman4_rk4_batch_multi_host, d, 0, devices)
        return out

    def dev(B, ref):
        inp = _batch_inputs(B)
        t, o = _dev_tensors(inp), _dev_out(ref)
        d = _batch_desc(L, B, {k: v.data_ptr() for k, v in t.items()}, o)
        for k, v in o.items():
            setattr(d, k, v.data_ptr())
        d.flags |= L.UNIFORM_PHYSICS
        d.gamma_uniform, d.alpha_uniform = float(inp["gamma"][0]), float(inp["alpha"][0])
        nb = int(lib.fpa_yaman4_scratch_bytes(B))
        scr = _dev_out({"s": bytes(nb)})["s"]
        d.scratch, d.scratch_bytes = scr.data_ptr(), nb
        L.check(lib.fpa_yaman4_rk4_batch_dev(C.byref(d), _stream()))
        return _sync_bytes(o)

    _check_sizes(gpu, build, [40_000, 1_000, 40_000], dev, multi_size=3 * 3_001 + 1)


# ----------------------------------------------------------------- sweeps
def _plan(gpu, golden, n1, n3):
    b2, b3, b4, wref = golden["b4_beta"]
    disp = gpu.dispersion.DispersionParams(omega_ref=wref, beta2=b2, beta3=b3, beta4=b4)
    pm = gpu.scan_mismtach._default_phase_matching_cfg(dispersion=disp, beta_legacy=None)
    plan, keep = gpu._device.new_plan_desc(np.linspace(1545e-9, 1555e-9, n1), 1558e-9,
                                           np.linspace(700e-9, 1700e-9, n3))   # wide: invalid plans too
    gpu.phase_matching.fill_plan_desc(plan, disp, pm)
    return plan, keep


def _fill_sweep(gpu, w, plan):
    w.plan = plan
    w.p_signal, w.gamma, w.alpha = P_IN[2], 11.5e-3, 1e-4
    w.z_max, w.dz, w.length_scale, w.save_every = 60.0, 0.2, 1.0, 7
    w.flags = gpu._lib.CHECK_NAN


def _sweep_outputs(mem, G, K, gain_optional):
    return {"gain_lin": mem(G * K, np.float64, gain_optional), "status": mem(G * K, np.int32, True),
            "Pmax": mem((G * K, 4), np.float64, True), "A_end": mem((G * K, 4), np.complex128, True),
            "dbeta": mem(G, np.float64, True), "valid": mem(G, np.int32, True), "omega": mem((G, 4), np.float64, True)}


def _point_sweep(w, out, ptr):
    w.gain_lin, w.status, w.Pmax, w.A_end = (ptr(out[k]) for k in ("gain_lin", "status", "Pmax", "A_end"))
    w.plan.dbeta, w.plan.valid, w.plan.omega = (ptr(out[k]) for k in ("dbeta", "valid", "omega"))


def _sweep_axes_on_device(w, plan, keep):
    l1, l2, l3 = keep
    t = _dev_tensors({"l1": l1, "l2": l2, "l3": l3})
    w.plan.lambda1, w.plan.lambda2, w.plan.lambda3 = (t[k].data_ptr() for k in ("l1", "l2", "l3"))
    return t


def test_sweep(gpu, golden):
    L, lib = gpu._lib, gpu._lib.lib()
    A0 = gpu.simulation.make_initial_amplitudes(P_IN, PHASE_IN)

    def desc(G):
        plan, keep = _plan(gpu, golden, 4, G // 4)
        d = L.SweepDesc()
        _fill_sweep(gpu, d, plan)
        for j in range(4):
            d.A0[2 * j], d.A0[2 * j + 1] = A0[j].real, A0[j].imag
        return d, keep

    def build(mem, G, devices=None):
        d, keep = desc(G)
        out = _sweep_outputs(mem, G, 1, False)
        _point_sweep(d, out, lambda a: _ptr(L, a))
        gpu._device._run_host(lib.fpa_yaman4_sweep_host, lib.fpa_yaman4_sweep_multi_host, d, 0, devices)
        return out

    def dev(G, ref):
        d, keep = desc(G)
        t, o = _sweep_axes_on_device(d, d.plan, keep), _dev_out(ref)
        _point_sweep(d, o, lambda a: a.data_ptr())
        nb = int(lib.fpa_yaman4_sweep_scratch_bytes(G))
        scr = _dev_out({"s": bytes(nb)})["s"]
        L.check(lib.fpa_yaman4_sweep_dev(C.byref(d), scr.data_ptr(), nb, _stream()))
        return _sync_bytes(o)

    _check_sizes(gpu, build, [4 * 20_000, 4 * 500, 4 * 20_000], dev, multi_size=4 * 2_501)


def test_phase_sweep(gpu, golden):
    L, lib = gpu._lib, gpu._lib.lib()
    K = 3
    table, _, _ = gpu.scan_mismtach.phase_sweep_inputs(P_IN, PHASE_IN, np.linspace(0.0, 2.0, K))
    red = (("gain_max", np.float64), ("gain_min", np.float64), ("idx_max", np.int32), ("idx_min", np.int32),
           ("n_finite", np.int32))

    def desc(G):
        plan, keep = _plan(gpu, golden, 2, G // 2)
        d = L.PhaseSweepDesc()
        _fill_sweep(gpu, d.sweep, plan)
        d.n_phases, d.A0_table, d.metric = K, L.ptr(table), L.GAIN_LAST_SAVED
        return d, keep

    def point(d, out, ptr):
        _point_sweep(d.sweep, out, ptr)
        for k, _ in red:
            setattr(d, k, ptr(out[k]))

    def build(mem, G, devices=None):
        d, keep = desc(G)
        out = _sweep_outputs(mem, G, K, True)
        out.update({k: mem(G, dt, k != "gain_max") for k, dt in red})
        point(d, out, lambda a: _ptr(L, a))
        gpu._device._run_host(lib.fpa_yaman4_phase_sweep_host, lib.fpa_yaman4_phase_sweep_multi_host, d, 0, devices)
        return out

    def dev(G, ref):
        d, keep = desc(G)
        t, o = _sweep_axes_on_device(d.sweep, d.sweep.plan, keep), _dev_out(ref)
        tab = _dev_tensors({"tab": table})["tab"]
        d.A0_table = tab.data_ptr()
        point(d, o, lambda a: a.data_ptr())
        nb = int(lib.fpa_yaman4_phase_sweep_scratch_bytes(G * K))
        scr = _dev_out({"s": bytes(nb)})["s"]
        L.check(lib.fpa_yaman4_phase_sweep_dev(C.byref(d), scr.data_ptr(), nb, _stream()))
        return _sync_bytes(o)

    _check_sizes(gpu, build, [2 * 10_000, 2 * 300, 2 * 10_000], dev, multi_size=2 * 1_501)


# ----------------------------------------------------------------- N-wave
GRID = np.array([0, 1, 3, 4, 6, 7])
N = GRID.size


def _nwave_inputs(B):
    rng = np.random.default_rng(B)
    A0 = (np.sqrt(rng.uniform(1e-4, 0.1, (B, N))) * np.exp(1j * rng.uniform(0, 6.28, (B, N)))).astype(np.complex128)
    return {"beta": rng.uniform(-1.0, 1.0, (B, N)), "gamma": np.array([11.5e-3]), "alpha": np.array([1e-4]), "A0": A0}


@pytest.mark.parametrize("form", ["comb", "table"])
def test_nwave(gpu, form):
    L, lib = gpu._lib, gpu._lib.lib()
    table, rows = gpu._device.enumerate_triplets(GRID)
    blob, n_classes = gpu._device.factor_table(N, table, rows)
    slots = np.ascontiguousarray(GRID - GRID.min(), dtype=np.int32)
    steps, save = 200, 9
    ns = steps // save + 1

    def desc(B, inp, out, ptr):
        d = L.NwaveDesc()
        d.n_points, d.n_waves, d.z_max, d.n_steps, d.save_every = B, N, 40.0, steps, save
        for k in ("beta", "gamma", "alpha", "A0"):
            setattr(d, k, ptr(inp[k]))
        d.beta_stride, d.A0_stride = 1, 1
        d.flags = L.CHECK_NAN
        for key, flag in (("A_trace", L.OUT_TRACE), ("A_end", L.OUT_END), ("Pmax", L.OUT_PMAX)):
            if out.get(key) is not None:
                d.flags |= flag
            setattr(d, key, ptr(out.get(key)))
        d.status = ptr(out.get("status"))
        if form == "comb":
            d.grid_slot, d.grid_span = ptr(inp["slots"]), int(slots.max() + 1)
        else:
            d.triplets, d.row_ptr, d.n_triplets = ptr(inp["table"]), ptr(inp["rows"]), table.size
        return d

    def build(mem, B, devices=None):
        inp = dict(_nwave_inputs(B), slots=slots, table=table, rows=rows)
        out = {"A_trace": mem((B, ns, N), np.complex128, True), "A_end": mem((B, N), np.complex128),
               "Pmax": mem((B, N), np.float64, True), "status": mem(B, np.int32, True)}
        d = desc(B, inp, out, lambda a: _ptr(L, a))
        gpu._device._run_host(lib.fpa_nwave_rk4_batch_host, lib.fpa_nwave_rk4_batch_multi_host, d, 0, devices)
        return out

    def dev(B, ref):
        t = _dev_tensors(dict(_nwave_inputs(B), slots=slots, table=table, rows=rows, blob=blob))
        o = _dev_out(ref)
        d = desc(B, t, o, lambda a: None if a is None else a.data_ptr())
        if form == "comb":
            d.flags |= L.NWAVE_COMB
        else:
            d.flags |= L.NWAVE_TABLE
            d.factored, d.n_classes = t["blob"].data_ptr(), n_classes
        L.check(lib.fpa_nwave_rk4_batch_dev(C.byref(d), _stream()))
        return _sync_bytes(o)

    # the comb kernel's thread mapping depends on the batch size (one warp per point from 4 * SM count points on):
    # the whole batch and its three shards stay below that threshold, so they run the same mapping
    _check_sizes(gpu, build, [3_000, 50, 3_000], dev, multi_size=3 * 100 + 2)


# ----------------------------------------------------------------- linear, RHS, Delta-beta table
def test_linear(gpu):
    L, lib = gpu._lib, gpu._lib.lib()
    dim, steps, save = 3, 50, 4
    ns = steps // save + 1
    lam = np.array([1.0 + 0.5j, -0.3 + 2.0j, 0.1 - 1.0j])

    def build(mem, B, devices=None):
        y0 = np.random.default_rng(B).standard_normal((B, dim)).astype(np.complex128)
        out = {"y_trace": mem((B, ns, dim), np.complex128, True), "y_end": mem((B, dim), np.complex128),
               "status": mem(B, np.int32, True)}
        flags = L.CHECK_NAN | (L.OUT_TRACE if out["y_trace"] is not None else 0) | \
            (L.OUT_END if out["y_end"] is not None else 0)
        L.check(lib.fpa_linear_rk4_batch_host(B, dim, L.ptr(y0), L.ptr(lam), 0.0, 1.0, steps, save, None, flags,
                                              _ptr(L, out["y_trace"]), _ptr(L, out["y_end"]),
                                              _ptr(L, out["status"]), 0))
        return out

    _check_sizes(gpu, build, [5_000, 7, 5_000])


def test_rhs(gpu):
    L, lib = gpu._lib, gpu._lib.lib()

    def build(mem, B, devices=None):
        rng = np.random.default_rng(B)
        z, g, a, db = (rng.uniform(0.0, 1.0, B) for _ in range(4))
        A = (rng.standard_normal((B, 4)) + 1j * rng.standard_normal((B, 4))).astype(np.complex128)
        out = {"dA": mem((B, 4), np.complex128)}
        L.check(lib.fpa_yaman4_rhs_host(B, L.ptr(z), L.ptr(A), L.ptr(g), L.ptr(a), L.ptr(db), L.ptr(out["dA"]), 0))
        return out

    for B in (20_000, 3, 20_000):
        for kind in KINDS[:4]:
            mem = Mem(L, kind)
            try:
                got = build(mem, B)["dA"].tobytes()
            finally:
                mem.release()
            if kind == "pageable":
                ref = got
            assert got == ref, (B, kind)


def test_dbeta_table(gpu, golden):
    L, lib = gpu._lib, gpu._lib.lib()

    def build(mem, G, devices=None):
        plan, keep = _plan(gpu, golden, 4, G // 4)
        out = {"dbeta": mem(G, np.float64), "valid": mem(G, np.int32, True), "omega": mem((G, 4), np.float64, True)}
        plan.dbeta, plan.valid, plan.omega = (_ptr(L, out[k]) for k in ("dbeta", "valid", "omega"))
        L.check(lib.fpa_dbeta_table_host(C.byref(plan), 0))
        return out

    _check_sizes(gpu, build, [4 * 10_000, 4 * 3, 4 * 10_000])
