#!/usr/bin/env python
"""tools/profile_cases.py <case> -- one small launch sequence per secondary kernel, for ncu captures.
  trace : yaman4_fast_kernel<TRACE>, 2e5 points x 2500 steps, save_every = 1 (32 GB written)
  comb  : nwave_comb8_kernel<2> (warp per point), N = 64, B = 4736, 200 steps
  comb1024 : the same kernel at the batch of BASELINE config 5, B = 1024, 400 steps
  comb1 : nwave_comb_kernel (CTA per point), N = 64, B = 1, 2000 steps
  table : nwave_rk4_kernel<factored> (512 threads per point), N = 64, B = 148, 100 steps
  table4736 : the same kernel (64 threads per point) at B = 4736, 100 steps
"""
import ctypes as C
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import __graft_entry__ as entry  # noqa: E402

fpa = entry.load_package()
L, lib = fpa._lib, fpa._lib.lib()
case = sys.argv[1]
torch.cuda.set_device(0)
L.check(lib.fpa_set_device(0))
dev = torch.device("cuda", 0)
if case == "trace":
    B, n_steps = 200_000, 2500
    dbeta = torch.linspace(-0.015, 0.015, B, dtype=torch.float64, device=dev)
    A0 = np.sqrt(np.array([0.1, 0.1, 1e-7, 1e-7]))
    consts = torch.tensor([11.5e-3, 1.1512925464970228e-4] + [v for a in A0 for v in (a, 0.0)], dtype=torch.float64, device=dev)
    trace = torch.empty(B * (n_steps + 1) * 8, dtype=torch.float64, device=dev)
    status = torch.empty(B, dtype=torch.int32, device=dev)
    d = L.Yaman4Desc()
    d.n_points, d.dbeta = B, dbeta.data_ptr()
    d.gamma, d.alpha, d.A0 = consts.data_ptr(), consts.data_ptr() + 8, consts.data_ptr() + 16
    d.z0, d.z_max, d.n_steps, d.save_every = 0.0, 500.0, n_steps, 1
    d.flags = L.OUT_TRACE | L.CHECK_NAN | L.UNIFORM_PHYSICS
    d.gamma_uniform, d.alpha_uniform = 11.5e-3, 1.1512925464970228e-4
    d.A_trace, d.status = trace.data_ptr(), status.data_ptr()
    for _ in range(3):
        L.check(lib.fpa_yaman4_rk4_batch_dev(C.byref(d), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
else:
    nw, ds = fpa.nwave, fpa.dispersion
    w0 = 2 * np.pi * 299792458.0 / 1550e-9
    plan = nw.uniform_comb_plan(w0, 2 * np.pi * 100e9, range(-32, 32))
    disp = ds.DispersionParams(omega_ref=w0, beta2=-2.57e-29, beta3=3.30e-41, beta4=-1.63e-55)
    beta = nw.beta_per_wave(plan, disp)
    Bn, steps = {"comb": (4736, 200), "comb1024": (1024, 400), "comb1": (1, 2000),
                 "table": (148, 100), "table4736": (4736, 100)}[case]
    rng = np.random.default_rng(0)
    A0 = np.sqrt(np.full((Bn, 64), 1e-6)) * np.exp(1j * rng.uniform(0, 6.28, (Bn, 64)))
    A0[:, [28, 36]] = np.sqrt(np.linspace(0.1, 1.0, Bn))[:, None]
    cfg = fpa.config.custom_simulation_config(z_max=steps * 0.1, dz=0.1, save_every=100)
    for _ in range(3):
        nw.run_nwave_simulation(cfg, plan, gamma=11.5e-3, alpha=2e-4, A0=A0, beta=beta, outputs=("end",),
                                form="comb" if case.startswith("comb") else "table")
print("done", case)
