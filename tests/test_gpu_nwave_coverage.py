"""GPU: the N-wave kernels (csrc/nwave_comb.cu, csrc/nwave.cu) against the CPU oracle (oracle/nwave_oracle.py) on
the paths the library selects by itself that the comb-versus-table comparisons cannot vouch for, because both kernels
share the launch plumbing, the stride handling and the z0 handling:

- grid spans 129 .. 512 (the generic reduce-scatter of the batch kernel, two rounds of tiles from span 257 on,
  3 .. 8 rounds in the single-run kernel), N = 128 and span 512 together, and span 513 past the limit;
- beta given per point, in every kernel form;
- a start at z0 != 0 (initial phase, resync abscissae, the table kernel's z);
- batch-kernel launches whose last CTA is partly filled, on both sides of the 4 x SM threshold, with one and with
  half a warp per point, and nothing stored past the batch;
- overflow and NaN inside a launch: the status of every point and the isolation of its neighbours.

Tolerances as in test_gpu_nwave.py: 1e-12 of the trace maximum against the oracle and between comb and table,
1e-13 between the factored table and the entry list."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

W0, DW = 1.2125e15, 6.28e11
TOL_ORACLE, TOL_FORMS, TOL_ENTRIES = 1e-12, 1e-12, 1e-13

# grid plans with span > 128 that pass the density rule (span^2 <= 5 T): (N, span, T) from the oracle's enumerator
WIDE = {
    "span129": (list(range(0, 129, 2)), (65, 129, 88384)),            # first span past the PLOG = 1 instantiation
    "gap192": (list(range(0, 24)) + list(range(168, 192)), (48, 192, 25656)),   # two clusters, wide gap
    "n128": (list(range(0, 256, 2)), (128, 255, 686784)),           # N at its limit
    "span257": (list(range(0, 257, 4)), (65, 257, 88384)),          # two rounds of tiles in the batch kernel
    "span512": (list(range(0, 512, 7)), (74, 512, 130980)),         # span at its limit
    "both": (list(range(0, 508, 4)) + [511], (128, 512, 670719)),   # both limits together
}


@pytest.fixture(scope="module")
def sm4(gpu):
    """The batch (warp-per-point) kernel threshold: 4 x the SM count of the device the tests run on."""
    L = gpu._lib
    n, khz = C.c_int(), C.c_int()
    name = C.create_string_buffer(128)
    L.check(L.lib().fpa_device_info(L.get_device(), C.byref(n), C.byref(khz), name, 128))
    assert n.value > 0
    return 4 * n.value


def _disp(gpu):
    return gpu.dispersion.DispersionParams(W0, beta2=-2.6e-29, beta3=3.3e-41, beta4=-1.6e-55)


def _plan(gpu, lines):
    return gpu.nwave.uniform_comb_plan(W0, DW, list(lines))


def _tab(plan):
    t = plan.table
    return np.stack([t["k"], t["l"], t["m"], t["weight"]], axis=1).astype(np.int64), plan.row_ptr.tolist()


def _amps(rng, B, N, lo=1e-4, hi=2e-2):
    return np.sqrt(rng.uniform(lo, hi, (B, N))) * np.exp(1j * rng.uniform(0, 2 * np.pi, (B, N)))


def _oracle_steps(nw_oracle, plan, A0, gamma, alpha, beta, *, z0=0.0, z_max, n_steps):
    """The oracle's state after every step (row 0: A0)."""
    tab, rows = _tab(plan)
    return nw_oracle.march(A0, gamma, alpha, beta, tab, rows, z0=z0, z_max=z_max, n_steps=n_steps)[1]


def _batch(gpu, plan, form, beta, gamma, alpha, A0, *, z0=0.0, z_max, n_steps, save_every, check_nan=True):
    """One launch of the library's host entry with the kernel form chosen as nwave.run_nwave_simulation does."""
    return gpu._device.nwave_batch(beta, gamma, alpha, A0, plan.table, plan.row_ptr, z0=z0, z_max=z_max, n_steps=n_steps,
                                   save_every=save_every, trace=True, end=True, pmax=True, check_nan=check_nan,
                                   grid_index=plan.grid_index if form in ("auto", "comb") else None,
                                   force_comb=form == "comb", force_table=form in ("table", "entries"),
                                   plain_table=form == "entries")


def _check_vs_oracle(r, b, ref, save_every, what):
    """Point b of a launch (trace, A_end, Pmax) against the oracle's per-step states `ref`."""
    n_saved = r["A_trace"].shape[1]
    ref_tr = ref[::save_every][:n_saved]
    scale = np.abs(ref).max()
    assert np.abs(r["A_trace"][b] - ref_tr).max() < TOL_ORACLE * scale, (what, b, "trace")
    assert np.abs(r["A_end"][b] - ref[-1]).max() < TOL_ORACLE * scale, (what, b, "end")
    assert np.abs(r["Pmax"][b] - (np.abs(ref_tr) ** 2).max(axis=0)).max() < TOL_ORACLE * scale ** 2, (what, b, "pmax")
    assert r["status"][b] == -1, (what, b)


def _check_close(a, b, tol, what):
    scale = np.abs(b["A_trace"]).max()
    for key, pw in (("A_trace", 1), ("A_end", 1), ("Pmax", 2)):
        assert np.abs(a[key] - b[key]).max() < tol * scale ** pw, (what, key)
    assert np.array_equal(a["status"], b["status"]), what


def _same_bits(a, b, what):
    for key in ("A_trace", "A_end", "Pmax", "status"):
        assert a[key].tobytes() == b[key].tobytes(), (what, key)


# ------------------------------------------------------------------------------------------------ 1. wide spans
@pytest.mark.parametrize("name", list(WIDE))
def test_wide_span_comb_vs_oracle_and_table(gpu, nw_oracle, sm4, name):
    """Both mappings (B = 2: one CTA per point; B = 4 SM + 1: warp per point, last CTA partly filled) of the comb
    kernel at spans 129 .. 512 against the oracle (first, middle, last point; N = 128: first and last over 16 steps)
    and, for the whole batch, against the table kernel; form='auto' takes the comb kernel for all these plans."""
    nw = gpu.nwave
    lines, (N_, M_, T_) = WIDE[name]
    plan = _plan(gpu, lines)
    N, M, T = plan.n_waves, plan.grid_span, plan.n_triplets
    assert (N, M, T) == (N_, M_, T_)
    assert M > 128 and M * M <= 5 * T and N <= 128 and M <= 512
    beta = nw.beta_per_wave(plan, _disp(gpu))
    n_steps, save_every = (16, 6) if N > 100 else (40, 7)          # ragged: the last steps are not saved
    dz = 0.1
    cfg = gpu.config.custom_simulation_config(z_max=dz * n_steps, dz=dz, save_every=save_every)
    gamma, alpha = 0.02, 1e-4
    rng = np.random.default_rng(M)
    big = _amps(rng, sm4 + 1, N)
    checked = [0, sm4] if N > 100 else [0, (sm4 + 1) // 2, sm4]
    refs = {b: _oracle_steps(nw_oracle, plan, big[b], gamma, alpha, beta, z_max=cfg.z_max, n_steps=n_steps) for b in checked}
    outs = ("trace", "end", "pmax")
    for A0, at in ((big[[0, sm4]], {0: 0, 1: sm4}), (big, {b: b for b in checked})):
        run = lambda form: nw.run_nwave_simulation(cfg, plan, gamma=gamma, alpha=alpha, A0=A0, beta=beta, outputs=outs, form=form)
        c = run("comb")
        assert c["n_steps"] == n_steps and c["A_trace"].shape == (A0.shape[0], n_steps // save_every + 1, N)
        for i, b in at.items():
            _check_vs_oracle(c, i, refs[b], save_every, (name, A0.shape[0]))
        _same_bits(run("auto"), c, (name, "auto"))
        t = run("table")
        _check_close(c, t, TOL_FORMS, (name, A0.shape[0], "comb vs table"))
        if N <= 48:
            _check_close(run("entries"), t, TOL_ENTRIES, (name, A0.shape[0], "entries vs table"))


def test_span_513_goes_to_the_table_kernel(gpu, nw_oracle):
    """One slot past the comb kernel's span limit: 'auto' integrates through the table kernel (same bits as
    form='table', and the oracle's numbers), an explicit form='comb' is refused."""
    nw = gpu.nwave
    plan = _plan(gpu, range(0, 513, 8))
    assert (plan.n_waves, plan.grid_span) == (65, 513)
    beta = nw.beta_per_wave(plan, _disp(gpu))
    cfg = gpu.config.custom_simulation_config(z_max=2.0, dz=0.1, save_every=6)
    A0 = _amps(np.random.default_rng(513), 3, 65)
    run = lambda form: nw.run_nwave_simulation(cfg, plan, gamma=0.02, alpha=1e-4, A0=A0, beta=beta,
                                               outputs=("trace", "end", "pmax"), form=form)
    a, t = run("auto"), run("table")
    _same_bits(a, t, "span 513")
    ref = _oracle_steps(nw_oracle, plan, A0[2], 0.02, 1e-4, beta, z_max=2.0, n_steps=20)
    _check_vs_oracle(a, 2, ref, 6, "span 513")
    with pytest.raises(NotImplementedError):
        run("comb")


# ------------------------------------------------------------------------------------------------ 2. per-point parameters
def test_per_point_beta_gamma_alpha_A0_in_every_form(gpu, nw_oracle, sm4):
    """beta [B, N] with distinct rows (and per-point gamma, alpha, A0) in the comb kernel at both mappings, the table
    kernel and the entry list, three points against the oracle; and stride 0 / stride 1 do the same arithmetic: rows
    that all equal row k give the bits of the same batch with beta[k] broadcast as [N]."""
    nw = gpu.nwave
    plan = _plan(gpu, WIDE["gap192"][0])
    N = plan.n_waves
    base = nw.beta_per_wave(plan, _disp(gpu))
    n_steps, save_every, z_max = 40, 7, 4.0
    for B in (3, sm4 + 1):
        rng = np.random.default_rng(B)
        beta = base * rng.uniform(0.5, 1.5, (B, N)) + rng.uniform(-2.0, 2.0, (B, N))
        gam = rng.uniform(5e-3, 3e-2, B)
        alp = rng.uniform(0.0, 1e-3, B)
        A0 = _amps(rng, B, N)
        checked = (0, B // 2, B - 1)
        refs = {b: _oracle_steps(nw_oracle, plan, A0[b], gam[b], alp[b], beta[b], z_max=z_max, n_steps=n_steps)
                for b in checked}
        kw = dict(z_max=z_max, n_steps=n_steps, save_every=save_every)
        res = {form: _batch(gpu, plan, form, beta, gam, alp, A0, **kw) for form in ("comb", "table", "entries")}
        for form, r in res.items():
            for b in checked:
                _check_vs_oracle(r, b, refs[b], save_every, (form, B))
        _check_close(res["comb"], res["table"], TOL_FORMS, ("comb vs table", B))
        _check_close(res["entries"], res["table"], TOL_ENTRIES, ("entries vs table", B))
        k = B // 2
        for form in ("comb", "table", "entries"):
            rows = _batch(gpu, plan, form, np.tile(beta[k], (B, 1)), gam, alp, A0, **kw)
            bc = _batch(gpu, plan, form, beta[k], gam, alp, A0, **kw)
            _same_bits(rows, bc, (form, B, "beta stride 1 vs 0"))


# ------------------------------------------------------------------------------------------------ 3. z0 != 0
def test_start_at_nonzero_z0(gpu, nw_oracle, sm4):
    """A march on [z0, z1] with dbeta * z0 of many radians: the reference-shaped integrators (integrate_fixed_step,
    rk4_step) with the comb and the table kernel, the entry list, and batches in both comb mappings, all against
    the oracle's march from z0 -- and far from the same march started at 0."""
    nw, I = gpu.nwave, gpu.integrators
    plan = _plan(gpu, WIDE["span257"][0])
    N = plan.n_waves
    beta = nw.beta_per_wave(plan, _disp(gpu))
    z0, n, save_every = 5.0, 30, 7
    z1 = z0 + 0.1 * n
    assert np.ptp(beta) * z0 > 20.0
    gamma, alpha = 0.02, 1e-4
    rng = np.random.default_rng(50)
    A0 = _amps(rng, sm4 + 1, N)
    ref = _oracle_steps(nw_oracle, plan, A0[0], gamma, alpha, beta, z0=z0, z_max=z1, n_steps=n)
    ref_last = _oracle_steps(nw_oracle, plan, A0[sm4], gamma, alpha, beta, z0=z0, z_max=z1, n_steps=n)
    ref_at0 = _oracle_steps(nw_oracle, plan, A0[0], gamma, alpha, beta, z_max=z1 - z0, n_steps=n)
    scale = np.abs(ref).max()
    assert np.abs(ref - ref_at0).max() > 1e3 * TOL_ORACLE * scale      # z0 really enters the phases
    grid = np.linspace(z0, z1, n + 1)
    ref_tr = ref[::save_every]
    results = []
    for form in ("comb", "table"):
        rhs = nw.NWaveRHS(plan, beta, gamma, alpha, form=form)
        z, A = I.integrate_fixed_step(rhs, grid, A0[0], None, save_every=save_every)
        assert np.array_equal(z, grid[::save_every])
        assert np.abs(A - ref_tr).max() < TOL_ORACLE * scale, form
        results.append(A)
        # one step from z != 0
        y1 = I.rk4_step(rhs, grid[3], ref[3], grid[4] - grid[3], None)
        one = _oracle_steps(nw_oracle, plan, ref[3], gamma, alpha, beta, z0=grid[3], z_max=grid[4], n_steps=1)[1]
        assert np.abs(y1 - one).max() < TOL_ORACLE * scale, form
    e = gpu._device.nwave_batch(beta, gamma, alpha, A0[:1], plan.table, plan.row_ptr, z0=z0, z_max=z1, n_steps=n,
                                save_every=save_every, trace=True, plain_table=True, force_table=True)
    assert np.abs(e["A_trace"][0] - ref_tr).max() < TOL_ORACLE * scale
    for A in results + [e["A_trace"][0]]:
        assert np.abs(A - ref_at0[::save_every]).max() > 1e3 * TOL_ORACLE * scale
    for A in (A0[[0, sm4]], A0):
        r = _batch(gpu, plan, "comb", beta, gamma, alpha, A, z0=z0, z_max=z1, n_steps=n, save_every=save_every)
        _check_vs_oracle(r, 0, ref, save_every, ("z0 batch", A.shape[0]))
        _check_vs_oracle(r, A.shape[0] - 1, ref_last, save_every, ("z0 batch", A.shape[0]))
        _check_close(r, _batch(gpu, plan, "table", beta, gamma, alpha, A, z0=z0, z_max=z1, n_steps=n, save_every=save_every),
                     TOL_FORMS, ("z0 comb vs table", A.shape[0]))
        assert np.abs(r["A_trace"][0] - ref_at0[::save_every]).max() > 1e3 * TOL_ORACLE * scale


# ------------------------------------------------------------------------------------------------ 4. ragged batches
def _config2(gpu):
    """BASELINE config 2's grid (21 lines, span 21): small enough for 8 points in a CTA of the batch kernel."""
    plan = _plan(gpu, range(-10, 11))
    return plan, gpu.nwave.beta_per_wave(plan, _disp(gpu))


def test_ragged_batch_kernel_launches(gpu, nw_oracle, sm4):
    """Batch sizes on both sides of the 4 x SM threshold and 16 x SM + 3 (eight points per CTA: the last CTA holds
    three).  First and last point against the oracle, the batch against the table."""
    plan, beta = _config2(gpu)
    N = plan.n_waves
    sms = sm4 // 4
    sizes = (sm4 - 1, sm4, sm4 + 1, 16 * sms + 3)
    n_steps, save_every, z_max = 40, 7, 4.0
    rng = np.random.default_rng(32)
    A0 = _amps(rng, 16 * sms + 3, N, 1e-3, 0.1)
    gam = rng.uniform(5e-3, 3e-2, A0.shape[0])
    ref0 = _oracle_steps(nw_oracle, plan, A0[0], gam[0], 1e-4, beta, z_max=z_max, n_steps=n_steps)
    kw = dict(z_max=z_max, n_steps=n_steps, save_every=save_every)
    for B in sizes:
        A, g = A0[:B], gam[:B]
        refB = _oracle_steps(nw_oracle, plan, A[B - 1], g[B - 1], 1e-4, beta, z_max=z_max, n_steps=n_steps)
        c = _batch(gpu, plan, "auto", beta, g, 1e-4, A, **kw)
        _check_vs_oracle(c, 0, ref0, save_every, B)
        _check_vs_oracle(c, B - 1, refB, save_every, B)
        _check_close(c, _batch(gpu, plan, "table", beta, g, 1e-4, A, **kw), TOL_FORMS, (B, "comb vs table"))


def test_nothing_is_stored_past_the_batch(gpu, sm4):
    """Through `fpa_nwave_rk4_batch_dev` with every output buffer one point longer than the batch and filled with a
    sentinel: the comb kernel (odd batches in both kernels, 16 x SM + 3) and the table kernel write the batch's
    results -- the bits the host entry gives -- and leave the extra point untouched."""
    import torch
    L, lib = gpu._lib, gpu._lib.lib()
    dev = torch.device("cuda", L.get_device())
    plan, beta = _config2(gpu)
    N = plan.n_waves
    n_steps, save_every = 12, 5
    ns = n_steps // save_every + 1
    rng = np.random.default_rng(7)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    blob, nc = gpu._device.factor_table(N, plan.table, plan.row_ptr)
    t_tab, t_rows, t_blob = t(np.ascontiguousarray(plan.table).view(np.int16)), t(plan.row_ptr.astype(np.int64)), t(blob)
    t_slot = t((plan.grid_index - plan.grid_index.min()).astype(np.int32))
    t_beta = t(beta)
    for B in (3, sm4 + 1, 16 * (sm4 // 4) + 3):
        A0 = _amps(rng, B, N, 1e-3, 0.1)
        for form in ("comb", "table", "entries"):
            host = _batch(gpu, plan, form, beta, 0.02, 1e-4, A0, z_max=1.2, n_steps=n_steps, save_every=save_every)
            t_A0, t_ga = t(A0.view(np.float64)), t(np.array([0.02, 1e-4]))
            t_tr = torch.full(((B + 1) * ns * N * 2,), -7.25, dtype=torch.float64, device=dev)
            t_end = torch.full(((B + 1) * N * 2,), -7.25, dtype=torch.float64, device=dev)
            t_pm = torch.full(((B + 1) * N,), -7.25, dtype=torch.float64, device=dev)
            t_st = torch.full((B + 1,), 12345, dtype=torch.int32, device=dev)
            d = L.NwaveDesc()
            d.n_points, d.n_waves = B, N
            d.beta, d.gamma, d.alpha, d.A0 = t_beta.data_ptr(), t_ga.data_ptr(), t_ga.data_ptr() + 8, t_A0.data_ptr()
            d.A0_stride = 1
            d.z0, d.z_max, d.n_steps, d.save_every = 0.0, 1.2, n_steps, save_every
            d.flags = L.OUT_TRACE | L.OUT_END | L.OUT_PMAX | L.CHECK_NAN
            d.A_trace, d.A_end, d.Pmax, d.status = t_tr.data_ptr(), t_end.data_ptr(), t_pm.data_ptr(), t_st.data_ptr()
            if form == "comb":
                d.flags |= L.NWAVE_COMB
                d.grid_slot, d.grid_span = t_slot.data_ptr(), plan.grid_span
            else:
                d.flags |= L.NWAVE_TABLE
                d.triplets, d.row_ptr, d.n_triplets = t_tab.data_ptr(), t_rows.data_ptr(), plan.n_triplets
                if form == "table":
                    d.factored, d.n_classes = t_blob.data_ptr(), nc
            L.check(lib.fpa_nwave_rk4_batch_dev(C.byref(d), torch.cuda.current_stream().cuda_stream))
            torch.cuda.synchronize()
            tr, end, pm, st = t_tr.cpu().numpy(), t_end.cpu().numpy(), t_pm.cpu().numpy(), t_st.cpu().numpy()
            what = (B, form)
            assert (tr[B * ns * N * 2:] == -7.25).all() and (end[B * N * 2:] == -7.25).all(), what
            assert (pm[B * N:] == -7.25).all() and st[B] == 12345, what
            assert tr[:B * ns * N * 2].tobytes() == host["A_trace"].tobytes(), what
            assert end[:B * N * 2].tobytes() == host["A_end"].tobytes(), what
            assert pm[:B * N].tobytes() == host["Pmax"].tobytes(), what
            assert st[:B].tobytes() == host["status"].tobytes() and (st[:B] == -1).all(), what


# ------------------------------------------------------------------------------------------------ 5. overflow and NaN
def _bad_batch(B, N, beta, bad_at, rng):
    """A healthy batch (A0, alpha, beta [B, N]) and the same batch with the points `bad_at` made to fail: four points
    with a gain of 1e30 per step whose A0 is scaled so that they overflow at steps 1 .. 4 (the last finite state is
    about 1e171, the next step overflows by hundreds of decades), one with NaN in A0, one with a NaN beta row."""
    A0 = _amps(rng, B, N, 1e-3, 0.1)
    alp = np.full(B, 1e-4)
    bet = np.tile(beta, (B, 1)) + rng.uniform(-0.5, 0.5, (B, N))
    A0b, alpb, betb = A0.copy(), alp.copy(), bet.copy()
    for k, b in enumerate(bad_at[:4]):
        A0b[b] = A0[b] * 10.0 ** (-30 * k)
        alpb[b] = -1.4e9
    A0b[bad_at[4], 3] = np.nan
    betb[bad_at[5], 7] = np.nan
    return (A0, alp, bet), (A0b, alpb, betb)


def test_overflow_and_nan_inside_a_launch(gpu, nw_oracle, sm4):
    """Points that overflow at different steps, a NaN in A0 and a NaN beta row, some of them sharing a CTA of the
    batch kernel, in the batch kernel, the single-run comb kernel and the table kernel: each reports the oracle's
    first non-finite step, its Pmax is the NaN-propagating maximum of |A|^2 over its saved samples, every other point
    has the bits of the same batch without the bad points, and with check_nan off all statuses are -1 and the
    numbers are the same."""
    plan, beta = _config2(gpu)
    N = plan.n_waves
    tab, rows = _tab(plan)
    n_steps, save_every, z_max = 12, 5, 1.2
    kw = dict(z_max=z_max, n_steps=n_steps, save_every=save_every)
    for B, bad_at, forms in ((sm4 + 1, [5, 6, 7, 100, 101, sm4], ("auto", "table")), (8, [1, 2, 3, 4, 5, 6], ("comb", "table"))):
        rng = np.random.default_rng(B)
        good, bad = _bad_batch(B, N, beta, bad_at, rng)
        A0b, alpb, betb = bad
        expect = np.full(B, -1)
        for b in bad_at:
            st = nw_oracle.march(A0b[b], 0.02, alpb[b], betb[b], tab, rows, z_max=z_max, n_steps=n_steps, check=True)[2]
            expect[b] = st
        assert sorted(expect[bad_at].tolist()) == [0, 0, 1, 2, 3, 4]
        healthy = np.setdiff1d(np.arange(B), bad_at)
        for form in forms:
            what = (B, form)
            rg = _batch(gpu, plan, form, good[2], 0.02, good[1], good[0], **kw)
            rb = _batch(gpu, plan, form, betb, 0.02, alpb, A0b, **kw)
            assert np.array_equal(rb["status"], expect), (what, rb["status"][bad_at], expect[bad_at])
            for key in ("A_trace", "A_end", "Pmax"):
                assert rb[key][healthy].tobytes() == rg[key][healthy].tobytes(), (what, key)
            tr = rb["A_trace"][bad_at]
            pmax_ref = np.max(tr.real * tr.real + tr.imag * tr.imag, axis=1)     # np.max propagates NaN
            assert np.isnan(pmax_ref).any()
            np.testing.assert_allclose(rb["Pmax"][bad_at], pmax_ref, rtol=1e-15, equal_nan=True, err_msg=str(what))
            assert not np.isfinite(rb["A_end"][bad_at]).all(axis=1).any(), what
            off = _batch(gpu, plan, form, betb, 0.02, alpb, A0b, check_nan=False, **kw)
            assert (off["status"] == -1).all(), what
            for key in ("A_trace", "A_end", "Pmax"):
                assert off[key].tobytes() == rb[key].tobytes(), (what, key, "check_nan off")
