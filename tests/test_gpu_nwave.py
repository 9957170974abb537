"""GPU: the N-wave kernel (csrc/nwave.cu) against the CPU statement of SURVEY App. C
(oracle/nwave_oracle.py) and, at N = 4 with the fixed process table, against the reference model
(golden B1 trace).  No reference exists for N > 4: parity there is to the oracle only."""
import numpy as np
import pytest

from conftest import rel_err

pytestmark = pytest.mark.gpu


def _table_as_list(plan):
    t = plan.table
    return [(int(a), int(b), int(c), int(d)) for a, b, c, d in zip(t["k"], t["l"], t["m"], t["weight"])]


def test_n4_fixed_table_reproduces_reference_trace(gpu, golden):
    """beta = [0,0,0,dbeta] + the fixed 4-entry table == yaman_model (golden B1, main.py:27-96)."""
    nw = gpu.nwave
    plan = nw.four_wave_plan(golden["b1_omega"])
    cfg = gpu.config.custom_simulation_config(z_max=1000.0, dz=0.1, save_every=10)
    gamma, alpha = golden["b1_gamma_alpha"]
    r = nw.run_nwave_simulation(cfg, plan, gamma=gamma, alpha=alpha, p_in=golden["b1_p_in"],
                                beta=[0.0, 0.0, 0.0, golden["b1_dbeta"][1]], outputs=("trace", "end", "pmax"))
    A, A_ref = r["A_trace"][0], golden["b1_A"]
    assert np.array_equal(r["z"], golden["b1_z"]) and A.shape == A_ref.shape
    assert rel_err(np.abs(A[-1]) ** 2, np.abs(A_ref[-1]) ** 2) < 1e-10
    assert np.max(np.abs(A - A_ref)) / np.max(np.abs(A_ref)) < 1e-10
    assert np.array_equal(r["A_end"][0], A[-1]) and r["status"][0] == -1
    assert rel_err(r["Pmax"][0], (np.abs(A) ** 2).max(axis=0)) < 1e-15


def test_n21_dual_pump_plan_vs_oracle(gpu, nw_oracle, golden):
    """BASELINE config 2 (21 lines, pumps at +-5, signal/idler at +-1), shortened to 400 steps."""
    nw, fp = gpu.nwave, gpu.frequency_plan
    wc, wd = golden["b1_sym"][0], golden["b1_sym"][1]
    plan = nw.uniform_comb_plan(wc, wd / 5.0, range(-10, 11))
    assert plan.n_waves == 21 and plan.n_triplets == 2760
    b2, b3, b4 = golden["b1_beta"]
    disp = gpu.dispersion.DispersionParams(omega_ref=wc, beta2=b2, beta3=b3, beta4=b4)
    beta = nw.beta_per_wave(plan, disp)
    p_in = np.zeros(21)
    p_in[[5, 15]] = 0.5
    p_in[[9, 11]] = 1e-5
    gamma, alpha = golden["b1_gamma_alpha"]
    cfg = gpu.config.custom_simulation_config(z_max=40.0, dz=0.1, save_every=10)
    z_ref, A_ref = nw_oracle.march(np.sqrt(p_in).astype(complex), gamma, alpha, beta, _table_as_list(plan),
                                   plan.row_ptr.tolist(), z_max=40.0, n_steps=400, save_every=10)
    seeded = p_in > 0
    for form in ("table", "comb"):       # enumerated triplets and the O(N^2) convolution form: same ODE
        r = nw.run_nwave_simulation(cfg, plan, gamma=gamma, alpha=alpha, p_in=p_in, beta=beta,
                                    outputs=("trace", "end"), form=form)
        assert np.array_equal(r["z"], z_ref)
        A = r["A_trace"][0]
        assert A.shape == (41, 21)
        assert np.max(np.abs(A - A_ref)) / np.max(np.abs(A_ref)) < 1e-11, form
        assert rel_err(np.abs(A[-1, seeded]) ** 2, np.abs(A_ref[-1, seeded]) ** 2) < 1e-10, form
        assert np.array_equal(r["A_end"][0], A[-1])
    # cascaded FWM populated lines that started empty
    assert (np.abs(A[-1, ~seeded]) ** 2).max() > 1e-12
    # through the reference-shaped integrator API as a registered RHS kind
    rhs = nw.NWaveRHS(plan, beta, gamma, alpha)
    z2, A2 = gpu.integrators.integrate_interval(rhs, 40.0, 0.1, np.sqrt(p_in).astype(complex), None, save_every=10)
    assert np.array_equal(z2, z_ref) and np.array_equal(A2, A)


def test_n64_comb_batch_vs_oracle(gpu, nw_oracle):
    """BASELINE config 5 plan (64 lines, 100 GHz, beta2..beta4), 40 steps, a batch of 3 pump powers:
    one CTA per scan point, each checked against the oracle."""
    nw = gpu.nwave
    w0 = 2 * np.pi * 299792458.0 / 1550e-9
    plan = nw.uniform_comb_plan(w0, 2 * np.pi * 100e9, range(-32, 32))
    assert plan.n_triplets == 84320 and plan.n_pairs() == 2076
    disp = gpu.dispersion.DispersionParams(omega_ref=w0, beta2=-2.57e-29, beta3=3.30e-41, beta4=-1.63e-55)
    beta = nw.beta_per_wave(plan, disp)
    rng = np.random.default_rng(0)
    base = np.full(64, 1e-12)
    base[32 + 1] = 1e-6
    phases = rng.uniform(0, 2 * np.pi, 64)
    pumps = np.array([0.1, 0.5, 1.0])
    A0 = np.empty((3, 64), dtype=complex)
    for b, pw in enumerate(pumps):
        p = base.copy()
        p[[32 - 4, 32 + 4]] = pw
        A0[b] = np.sqrt(p) * np.exp(1j * phases)
    cfg = gpu.config.custom_simulation_config(z_max=4.0, dz=0.1, save_every=20)
    table = _table_as_list(plan)
    refs = [nw_oracle.march(A0[b], 11.5e-3, 2e-4, beta, table, plan.row_ptr.tolist(), z_max=4.0, n_steps=40,
                            save_every=20)[1] for b in range(3)]
    for form in ("table", "comb"):
        r = nw.run_nwave_simulation(cfg, plan, gamma=11.5e-3, alpha=2e-4, A0=A0, beta=beta,
                                    outputs=("trace", "end", "pmax"), form=form)
        assert r["A_trace"].shape == (3, 3, 64) and (r["status"] == -1).all()
        for b in range(3):
            A_ref = refs[b]
            assert np.max(np.abs(r["A_trace"][b] - A_ref)) / np.max(np.abs(A_ref)) < 1e-12, form
            # the 1e-12 W lines sit 12 decades below the pumps: their power is compared on the scale
            # of the sum they are a small difference of (|A_pump|^3 * gamma * z)
            strong = np.abs(A_ref[-1]) ** 2 > 1e-9
            assert rel_err(np.abs(r["A_end"][b][strong]) ** 2, np.abs(A_ref[-1][strong]) ** 2) < 1e-10, form
    assert plan.flops_per_step("comb") < plan.flops_per_step("entries") / 10
    # per-point gamma: a batch equals the single runs, bit for bit
    g = np.array([5e-3, 11.5e-3, 2e-2])
    rb = nw.run_nwave_simulation(cfg, plan, gamma=g, alpha=2e-4, A0=A0, beta=beta, outputs=("end",))
    for b in range(3):
        one = nw.run_nwave_simulation(cfg, plan, gamma=g[b], alpha=2e-4, A0=A0[b:b + 1], beta=beta, outputs=("end",))
        assert np.array_equal(one["A_end"][0], rb["A_end"][b])


def test_nwave_invariants(gpu):
    """alpha = 0: total power is conserved by the N-wave system (Manley-Rowe), here to RK4 accuracy."""
    nw = gpu.nwave
    w0 = 1.2e15
    plan = nw.uniform_comb_plan(w0, 2 * np.pi * 200e9, range(-4, 5))
    disp = gpu.dispersion.DispersionParams(omega_ref=w0, beta2=-5e-28)
    p_in = np.array([0, 0, 0.3, 1e-4, 0, 0, 0.4, 0, 1e-6], dtype=float)
    cfg = gpu.config.custom_simulation_config(z_max=100.0, dz=0.05, save_every=100)
    for form in ("table", "comb"):
        r = nw.run_nwave_simulation(cfg, plan, gamma=0.02, alpha=0.0, p_in=p_in, dispersion=disp, form=form)
        P = (np.abs(r["A_trace"][0]) ** 2).sum(axis=1)
        assert np.ptp(P) < 1e-11 * P[0]
    # a grid with gaps (missing lines never get populated) and a NaN run reported at the oracle's step
    gap = nw.uniform_comb_plan(w0, 2 * np.pi * 200e9, [-6, -3, -1, 0, 1, 2, 5, 9])
    p8 = np.array([0.2, 1e-5, 0.0, 0.3, 1e-4, 0.0, 0.0, 1e-6])
    bt = nw.beta_per_wave(gap, disp)
    a = nw.run_nwave_simulation(cfg, gap, gamma=0.02, alpha=1e-4, p_in=p8, beta=bt, form="table", outputs=("end",))
    c = nw.run_nwave_simulation(cfg, gap, gamma=0.02, alpha=1e-4, p_in=p8, beta=bt, form="comb", outputs=("end",))
    assert np.max(np.abs(a["A_end"] - c["A_end"])) < 1e-13 * np.max(np.abs(a["A_end"]))
    boom = np.full(8, 1e120)
    for form in ("table", "comb"):
        r = nw.run_nwave_simulation(gpu.config.custom_simulation_config(z_max=1.0, dz=0.125, save_every=1), gap,
                                    gamma=1.0, alpha=0.0, p_in=boom, beta=bt, form=form, outputs=("end",))
        assert r["status"][0] == 0


@pytest.mark.parametrize("lines", [[0], [0, 1], list(range(-3, 4)), list(range(-16, 17)), [0, 1, 2, 100],
                                   list(range(-40, 41)), list(range(0, 127, 2)), list(range(-64, 64)),
                                   list(range(0, 129, 2)), list(range(0, 24)) + list(range(168, 192)),
                                   list(range(0, 257, 4)), list(range(0, 512, 7))])
@pytest.mark.parametrize("batch", [2, 640])          # CTA-per-point and warp-per-point mappings
def test_comb_equals_table_on_odd_shapes(gpu, lines, batch):
    """Grid spans that are not multiples of the kernel's tile (2, 4) or block (8) sizes, one and two
    lines, wide gaps, spans above 64 (several rounds of tiles) and up to the limit of 512 (the generic
    reduce-scatter; two rounds of tiles in the batch kernel from 257 on): the correlation form must reproduce
    the enumerated-triplet kernel, which shares no indexing code with it."""
    nw = gpu.nwave
    plan = nw.uniform_comb_plan(1.2125e15, 6.28e11, lines)
    N = plan.n_waves
    disp = gpu.dispersion.DispersionParams(1.2125e15, beta2=-2.6e-29, beta3=3.3e-41, beta4=-1.6e-55)
    beta = nw.beta_per_wave(plan, disp)
    rng = np.random.default_rng(N + batch)
    A0 = np.sqrt(rng.uniform(1e-5, 2e-1, (batch, N))) * np.exp(1j * rng.uniform(0, 6.28, (batch, N)))
    cfg = gpu.config.custom_simulation_config(z_max=4.0, dz=0.1, save_every=8)
    t = nw.run_nwave_simulation(cfg, plan, gamma=0.02, alpha=1e-4, A0=A0, beta=beta, form="table", outputs=("end", "pmax"))
    c = nw.run_nwave_simulation(cfg, plan, gamma=0.02, alpha=1e-4, A0=A0, beta=beta, form="comb", outputs=("end", "pmax"))
    scale = np.max(np.abs(t["A_end"]))
    assert np.max(np.abs(t["A_end"] - c["A_end"])) < 1e-12 * scale
    assert np.max(np.abs(t["Pmax"] - c["Pmax"])) < 1e-12 * scale ** 2
    assert (c["status"] == -1).all()
    if N <= 48 or batch == 2:       # and the table kernel's two ways through the table (entry list: minutes beyond)
        e = nw.run_nwave_simulation(cfg, plan, gamma=0.02, alpha=1e-4, A0=A0, beta=beta, form="entries", outputs=("end", "pmax"))
        assert np.max(np.abs(t["A_end"] - e["A_end"])) < 1e-13 * scale
        assert np.max(np.abs(t["Pmax"] - e["Pmax"])) < 1e-13 * scale ** 2


def test_factored_table_equals_entry_list(gpu, nw_oracle):
    """The table kernel integrates from `fpa_nwave_factor_table`'s form of the table (pair products once per RHS);
    FPA_NWAVE_PLAIN walks the entry list as round 1 did.  Same ODE, different summation order: 1e-13 of the
    state's scale -- on tables from plans (comb, off-grid, the reference's fixed four-wave table) and on one no
    plan would give (repeats, k > l, negative weights, empty rows), the latter against the oracle's march too."""
    nw, D = gpu.nwave, gpu._device
    rng = np.random.default_rng(11)
    w0, dw = 1.2125e15, 6.28e11
    disp = gpu.dispersion.DispersionParams(w0, beta2=-2.6e-29, beta3=3.3e-41, beta4=-1.6e-55)
    cases = []
    for lines in (range(-10, 11), range(-32, 32)):
        plan = nw.uniform_comb_plan(w0, dw, lines)
        cases.append((plan.n_waves, plan.table, plan.row_ptr, nw.beta_per_wave(plan, disp)))
    off = nw.irregular_plan(w0 + dw * np.array([-5.0, 5.0, 1.3, -1.3, 2.77, -7.41, 0.0, 3.7, -3.7]))
    cases.append((off.n_waves, off.table, off.row_ptr, nw.beta_per_wave(off, disp)))
    ent = [(0, 3, 2, 1, 5), (0, 2, 3, 1, -2), (0, 1, 1, 0, 3), (0, 6, 6, 0, 1), (2, 5, 4, 2, 7), (2, 0, 1, 3, 1), (6, 0, 0, 0, 1)]
    ragged = np.array([e[1:] for e in ent], dtype=gpu._lib.TRIPLET_DTYPE)
    rrows = np.searchsorted(np.array([e[0] for e in ent]), np.arange(8)).astype(np.int64)
    ragged_case = (7, ragged, rrows, rng.uniform(-2.0, 2.0, 7))
    cases.append(ragged_case)
    from test_cabi_cpu import comb_table_with_an_own_pair      # mode 1 of the factoriser: own-pair weight matrix
    own_t, own_r = comb_table_with_an_own_pair(gpu, 16)
    assert np.frombuffer(D.factor_table(16, own_t, own_r)[0][:48], dtype=np.int32)[4] == 1
    cases.append((16, own_t, own_r, rng.uniform(-0.5, 0.5, 16)))
    for N, table, rows, beta in cases:
        B = 3
        A0 = np.sqrt(rng.uniform(1e-4, 0.3, (B, N))) * np.exp(1j * rng.uniform(0, 6.28, (B, N)))
        kw = dict(z_max=6.0, n_steps=60, save_every=7, trace=True, end=True, pmax=True, force_table=True)
        f = D.nwave_batch(beta, 0.02, 1e-4, A0, table, rows, **kw)
        e = D.nwave_batch(beta, 0.02, 1e-4, A0, table, rows, plain_table=True, **kw)
        scale = np.abs(e["A_trace"]).max()
        assert (f["status"] == -1).all() and (e["status"] == -1).all()
        for key, pw in (("A_trace", 1), ("A_end", 1), ("Pmax", 2)):
            assert np.max(np.abs(f[key] - e[key])) < 1e-13 * scale ** pw, (N, key)
    # the ragged table against the CPU march
    N, table, rows, beta = ragged_case
    A0 = np.sqrt(rng.uniform(1e-4, 0.3, N)) * np.exp(1j * rng.uniform(0, 6.28, N))
    f = D.nwave_batch(beta, 0.02, 1e-4, A0[None, :], table, rows, z_max=6.0, n_steps=60, save_every=6, trace=True, force_table=True)
    tl = [(int(a), int(b), int(c), int(d)) for a, b, c, d in zip(table["k"], table["l"], table["m"], table["weight"])]
    _, A_ref = nw_oracle.march(A0, 0.02, 1e-4, beta, tl, rrows.tolist(), z_max=6.0, n_steps=60, save_every=6)
    assert np.max(np.abs(f["A_trace"][0] - A_ref)) < 1e-12 * np.max(np.abs(A_ref))


def test_foreign_factored_blob_gives_no_result(gpu):
    """`_dev` callers pass the blob themselves: one that does not belong to the plan (wrong class count / wave
    count) must not produce numbers -- status 0 and NaN."""
    import ctypes as C

    import torch
    L, lib, D = gpu._lib, gpu._lib.lib(), gpu._device
    dev = torch.device("cuda", 0)
    table, rows = D.enumerate_triplets(np.arange(8))
    blob, nc = D.factor_table(8, table, rows)
    t_blob = torch.from_numpy(blob).to(dev)
    t_A0 = torch.ones(16, dtype=torch.float64, device=dev)
    t_beta = torch.zeros(8, dtype=torch.float64, device=dev)
    t_ga = torch.tensor([0.01, 0.0], dtype=torch.float64, device=dev)
    t_out = torch.zeros(16, dtype=torch.float64, device=dev)
    t_st = torch.full((1,), 7, dtype=torch.int32, device=dev)
    d = L.NwaveDesc()
    d.n_points, d.n_waves = 1, 8
    d.beta, d.gamma, d.alpha, d.A0 = t_beta.data_ptr(), t_ga.data_ptr(), t_ga.data_ptr() + 8, t_A0.data_ptr()
    d.z0, d.z_max, d.n_steps, d.save_every = 0.0, 1.0, 10, 1
    d.flags = L.OUT_END | L.CHECK_NAN | L.NWAVE_TABLE
    d.A_end, d.status = t_out.data_ptr(), t_st.data_ptr()
    d.factored, d.n_classes = t_blob.data_ptr(), nc          # triplets / row_ptr left NULL: the blob is enough
    L.check(lib.fpa_nwave_rk4_batch_dev(C.byref(d), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert int(t_st[0]) == -1 and bool(torch.isfinite(t_out).all())
    good = t_out.clone()
    d.n_classes = nc + 1
    L.check(lib.fpa_nwave_rk4_batch_dev(C.byref(d), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert int(t_st[0]) == 0 and bool(torch.isnan(t_out).all())
    d.n_classes = nc
    L.check(lib.fpa_nwave_rk4_batch_dev(C.byref(d), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert torch.equal(t_out, good)



def test_irregular_and_sparse_plans_run_through_the_table_kernel(gpu, nw_oracle):
    """Plans the convolution form does not suit: (i) lines off any integer grid (tolerance-matched enumeration),
    (ii) a sparse wide grid, span 801 > 512 -- with form='auto' both integrate through the enumerated-triplet
    kernel (round 1 raised NotImplementedError for (ii)); an explicit form='comb' beyond the limits still raises."""
    nw = gpu.nwave
    w0, dw = 1.2125e15, 6.28e11
    disp = gpu.dispersion.DispersionParams(w0, beta2=-2.6e-29, beta3=3.3e-41, beta4=-1.6e-55)
    cfg = gpu.config.custom_simulation_config(z_max=20.0, dz=0.1, save_every=50)
    # (i) off-grid: two pumps, a signal and its idler, plus lines that match nothing
    om = w0 + dw * np.array([-5.0, 5.0, 1.3, -1.3, 2.77, -7.41])
    plan = nw.irregular_plan(om)
    assert plan.n_triplets > 0
    beta = nw.beta_per_wave(plan, disp)
    p_in = np.array([0.4, 0.4, 1e-4, 1e-4, 1e-5, 1e-5])
    r = nw.run_nwave_simulation(cfg, plan, gamma=0.0115, alpha=1e-4, p_in=p_in, beta=beta, outputs=("trace", "end"))
    table = [(int(a), int(b), int(c), int(d)) for a, b, c, d in zip(plan.table["k"], plan.table["l"], plan.table["m"],
                                                                      plan.table["weight"])]
    z_ref, A_ref = nw_oracle.march(np.sqrt(p_in).astype(complex), 0.0115, 1e-4, beta, table, plan.row_ptr.tolist(),
                                   z_max=20.0, n_steps=200, save_every=50)
    assert np.max(np.abs(r["A_trace"][0] - A_ref)) < 1e-12 * np.max(np.abs(A_ref))
    with pytest.raises(ValueError):
        nw.run_nwave_simulation(cfg, plan, gamma=0.0115, alpha=1e-4, p_in=p_in, beta=beta, form="comb")
    # (ii) sparse wide grid
    sparse = nw.uniform_comb_plan(w0, dw / 100.0, [-400, 0, 400])
    bs = nw.beta_per_wave(sparse, disp)
    p3 = np.array([1e-4, 0.5, 1e-4])
    a = nw.run_nwave_simulation(cfg, sparse, gamma=0.0115, alpha=1e-4, p_in=p3, beta=bs, outputs=("end",))      # auto
    b = nw.run_nwave_simulation(cfg, sparse, gamma=0.0115, alpha=1e-4, p_in=p3, beta=bs, outputs=("end",), form="table")
    assert np.array_equal(a["A_end"], b["A_end"]) and (a["status"] == -1).all()
    with pytest.raises(NotImplementedError):
        nw.run_nwave_simulation(cfg, sparse, gamma=0.0115, alpha=1e-4, p_in=p3, beta=bs, outputs=("end",), form="comb")
    # a moderately sparse grid inside the comb limits: 'auto' picks the table (span^2 > 5 T), both forms agree
    mid = nw.uniform_comb_plan(w0, dw, [-40, -3, 0, 3, 40])
    bm = nw.beta_per_wave(mid, disp)
    p5 = np.array([1e-5, 0.3, 0.4, 1e-4, 1e-5])
    t_ = nw.run_nwave_simulation(cfg, mid, gamma=0.0115, alpha=1e-4, p_in=p5, beta=bm, outputs=("end",), form="table")
    c_ = nw.run_nwave_simulation(cfg, mid, gamma=0.0115, alpha=1e-4, p_in=p5, beta=bm, outputs=("end",), form="comb")
    u_ = nw.run_nwave_simulation(cfg, mid, gamma=0.0115, alpha=1e-4, p_in=p5, beta=bm, outputs=("end",))
    assert np.array_equal(u_["A_end"], t_["A_end"])
    assert np.max(np.abs(c_["A_end"] - t_["A_end"])) < 1e-13 * np.max(np.abs(t_["A_end"]))


def test_bad_grid_slots_are_rejected(gpu):
    D = gpu._device
    table, rows = D.enumerate_triplets([0, 1, 2])
    A0 = np.ones((1, 3), dtype=complex)
    with pytest.raises(ValueError, match="distinct"):
        D.nwave_batch(np.zeros(3), 0.01, 0.0, A0, table, rows, z_max=1.0, n_steps=4, grid_index=[0, 1, 1])


def test_multi_device_nwave_batch_equals_single_device(gpu):
    """`fpa_nwave_rk4_batch_multi_host` (BASELINE config 5 shape: a batch of pump powers): contiguous balanced
    point ranges over the listed devices (a one-GPU box repeats device 0); every shard uses the same kernel as the
    whole batch here (CTA per point), so the results are bit-identical."""
    nw = gpu.nwave
    w0 = 2 * np.pi * 299792458.0 / 1550e-9
    plan = nw.uniform_comb_plan(w0, 2 * np.pi * 100e9, range(-16, 16))
    beta = nw.beta_per_wave(plan, gpu.dispersion.DispersionParams(omega_ref=w0, beta2=-2.57e-29, beta3=3.30e-41, beta4=-1.63e-55))
    rng = np.random.default_rng(4)
    B = 37
    A0 = np.sqrt(rng.uniform(1e-6, 0.3, (B, 32))) * np.exp(1j * rng.uniform(0, 6.28, (B, 32)))
    gam = rng.uniform(5e-3, 2e-2, B)
    cfg = gpu.config.custom_simulation_config(z_max=30.0, dz=0.1, save_every=100)
    n_dev = gpu._lib.device_count()
    for form in ("comb", "table"):
        one = nw.run_nwave_simulation(cfg, plan, gamma=gam, alpha=2e-4, A0=A0, beta=beta, outputs=("trace", "end", "pmax"), form=form)
        for count in (2, 5):
            many = nw.run_nwave_simulation(cfg, plan, gamma=gam, alpha=2e-4, A0=A0, beta=beta, outputs=("trace", "end", "pmax"),
                                           form=form, devices=[k % n_dev for k in range(count)])
            for k in ("A_trace", "A_end", "Pmax", "status"):
                assert one[k].tobytes() == many[k].tobytes(), (k, form, count)
