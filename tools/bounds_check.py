#!/usr/bin/env python
"""tools/bounds_check.py -- compute-sanitizer is closed on the B200 pool, so the kernels with
non-trivial shared-memory indexing carry their own bounds checks (-DFPA_BOUNDS_CHECK: device
asserts on every sequence access of csrc/nwave_comb.cu and on every offset the factored-table kernel of
csrc/nwave.cu takes from its blob).  This builds that variant of the library
into build/libfpa_b200_checked.so and runs the N-wave GPU tests and a sweep of odd shapes on it;
a failed assert aborts the kernel and the call returns a CUDA error.

usage (GPU box):  python tools/bounds_check.py
"""
import ctypes as C
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import __graft_entry__ as entry  # noqa: E402

out = entry.BUILD / "libfpa_b200_checked.so"
entry.BUILD.mkdir(exist_ok=True)
flags = [f for f in entry.NVCC_FLAGS] + ["-DFPA_BOUNDS_CHECK", "-DFPA_SASS_PASS=0", "-UNDEBUG"]
res = subprocess.run([entry._nvcc(), *flags, "-o", str(out), *[str(entry.CSRC / s) for s in entry.SOURCES]],
                     capture_output=True, text=True)
if res.returncode != 0:
    raise SystemExit(res.stderr)
fpa = entry.load_package()
nw = fpa.nwave
with fpa._lib.use_library(out):
    L = fpa._lib
    n_sm, khz, name = C.c_int(), C.c_int(), C.create_string_buffer(128)
    L.check(L.lib().fpa_device_info(L.get_device(), C.byref(n_sm), C.byref(khz), name, 128))
    sm4 = 4 * n_sm.value
    disp = fpa.dispersion.DispersionParams(1.2125e15, beta2=-2.6e-29, beta3=3.3e-41, beta4=-1.6e-55)
    rng = np.random.default_rng(3)
    n_cases = 0
    # spans that are not multiples of the tile / block sizes, gapped grids, spans 129 .. 512 (the generic
    # reduce-scatter, two rounds of tiles from 257 on), N = 128 with span 512; one CTA per point and the batch
    # mapping on both sides of its threshold (4 x SM), with a partly filled last CTA (16 x SM + 3: eight points per
    # CTA for small plans); beta per point
    wide = (range(0, 129, 2), list(range(0, 24)) + list(range(168, 192)), range(0, 256, 2), range(0, 257, 4),
            range(0, 512, 7), list(range(0, 508, 4)) + [511])
    for lines in ([0], [0, 1], range(-1, 2), range(-3, 4), [-6, -3, -1, 0, 1, 2, 5, 9], range(-10, 11),
                  range(-16, 17), range(-32, 32), range(-40, 41), [0, 1, 2, 100], range(0, 127)) + wide:
        plan = nw.uniform_comb_plan(1.2125e15, 6.28e11, list(lines))
        N = plan.n_waves
        beta = nw.beta_per_wave(plan, disp)
        sizes = (1, 3, 700, sm4 - 1, sm4 + 1) + (() if N > 100 else (16 * n_sm.value + 3,))
        for B in sizes:
            A0 = np.sqrt(rng.uniform(1e-6, 1e-2, (B, N))) * np.exp(1j * rng.uniform(0, 6.28, (B, N)))
            bet = beta * rng.uniform(0.9, 1.1, (B, N)) if B % 2 else beta
            cfg = fpa.config.custom_simulation_config(z_max=0.7, dz=0.1, save_every=3)
            r = nw.run_nwave_simulation(cfg, plan, gamma=0.02, alpha=1e-4, A0=A0, beta=bet, form="comb",
                                        outputs=("trace", "end", "pmax"))
            assert np.isfinite(r["A_end"]).all()
            n_cases += 1
    print(f"bounds-checked comb kernel: {n_cases} launches without a failed assert")
    # the factored-table kernel: every offset it takes from its blob, over plan sizes 1 .. 128, single runs (512 / 256
    # / 64 threads per point) and batches (64 / 128 threads), grid plans, an off-grid plan and tables no plan gives
    n_cases = 0
    sys.path.insert(0, str(ROOT / "tests"))
    from test_cabi_cpu import comb_table_with_an_own_pair
    tables = []
    for lines in ([0], [0, 1], range(3), range(-3, 4), [-6, -3, -1, 0, 1, 2, 5, 9], range(13), range(-10, 11), range(-16, 17),
                  range(-32, 32), range(-40, 41), [0, 1, 2, 100], range(0, 127, 2), range(-64, 64)) + wide:
        plan = nw.uniform_comb_plan(1.2125e15, 6.28e11, list(lines))
        tables.append((plan.n_waves, plan.table, plan.row_ptr))
    off = nw.irregular_plan(1.2125e15 + 6.28e11 * np.array([-5.0, 5.0, 1.3, -1.3, 2.77, -7.41, 0.0, 3.7, -3.7]))
    tables.append((off.n_waves, off.table, off.row_ptr))
    tables.append((16,) + comb_table_with_an_own_pair(fpa, 16))
    tables.append((5, np.empty(0, dtype=fpa._lib.TRIPLET_DTYPE), np.zeros(6, dtype=np.int64)))
    for N, table, rows in tables:
        for B in (1, 3, 700, 2500):
            if N > 100 and B > 700:
                continue
            A0 = np.sqrt(rng.uniform(1e-6, 1e-2, (B, N))) * np.exp(1j * rng.uniform(0, 6.28, (B, N)))
            r = fpa._device.nwave_batch(rng.uniform(-0.1, 0.1, N), 0.02, 1e-4, A0, table, rows, z_max=0.7, n_steps=7, save_every=3,
                                        trace=True, end=True, pmax=True, force_table=True)
            assert np.isfinite(r["A_end"]).all() and (r["status"] == -1).all()
            n_cases += 1
    print(f"bounds-checked factored-table kernel: {n_cases} launches without a failed assert")
