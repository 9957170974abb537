#!/usr/bin/env python
"""tools/comb_bench.py [B ...] -- N = 64 comb plan of BASELINE config 5 through fpa_nwave_rk4_batch_dev for
several batch sizes (device-resident, CUDA events): point.steps/s, credited TFLOP/s and the fraction of the
measured FP64 peak."""
import ctypes as C
import os
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import __graft_entry__ as entry  # noqa: E402

entry.build()
fpa = entry.load_package()
L, lib = fpa._lib, fpa._lib.lib()
dev = torch.device("cuda", 0)
torch.cuda.set_device(0)
L.check(lib.fpa_set_device(0))
nw, ds = fpa.nwave, fpa.dispersion
steps = int(os.environ.get("COMB_STEPS", "2000"))
sizes = [int(v) for v in sys.argv[1:]] or [592, 1024, 2368, 4736, 9472]
peak_tf, _ = fpa._device.fp64_peak(iters=2048)
w0 = 2 * np.pi * 299792458.0 / 1550e-9
plan = nw.uniform_comb_plan(w0, 2 * np.pi * 100e9, range(-32, 32))
beta = nw.beta_per_wave(plan, ds.DispersionParams(omega_ref=w0, beta2=-2.57e-29, beta3=3.30e-41, beta4=-1.63e-55))
phases = np.random.default_rng(0).uniform(0, 2 * np.pi, 64)
flops = plan.flops_per_step("comb")
print(f"{torch.cuda.get_device_name(0)}; FP64 peak {peak_tf:.2f} TF; N = 64, {steps} steps, {flops:.0f} credited flops per point.step")
for Bn in sizes:
    A0 = np.empty((Bn, 64), dtype=complex)
    for b, pw in enumerate(np.linspace(0.1, 1.0, Bn)):
        p = np.full(64, 1e-12)
        p[33] = 1e-6
        p[[28, 36]] = pw
        A0[b] = np.sqrt(p) * np.exp(1j * phases)
    t_beta = torch.from_numpy(beta.copy()).to(dev)
    t_ga = torch.tensor([11.5e-3, 2e-4], dtype=torch.float64, device=dev)
    t_A0 = torch.from_numpy(A0.view(np.float64)).to(dev)
    t_out = torch.empty(Bn * 128, dtype=torch.float64, device=dev)
    t_st = torch.empty(Bn, dtype=torch.int32, device=dev)
    g = plan.grid_index.astype(np.int64)
    t_slot = torch.from_numpy((g - g.min()).astype(np.int32)).to(dev)
    d = L.NwaveDesc()
    d.n_points, d.n_waves = Bn, 64
    d.beta, d.beta_stride = t_beta.data_ptr(), 0
    d.gamma, d.gamma_stride = t_ga.data_ptr(), 0
    d.alpha, d.alpha_stride = t_ga.data_ptr() + 8, 0
    d.A0, d.A0_stride = t_A0.data_ptr(), 1
    d.z0, d.z_max, d.n_steps, d.save_every = 0.0, 0.1 * steps, steps, 100
    d.flags = L.OUT_END | L.CHECK_NAN
    d.A_end, d.status = t_out.data_ptr(), t_st.data_ptr()
    d.grid_slot, d.grid_span = t_slot.data_ptr(), 64
    ts = []
    for r in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        L.check(lib.fpa_nwave_rk4_batch_dev(C.byref(d), torch.cuda.current_stream().cuda_stream))
        e1.record()
        torch.cuda.synchronize()
        if r:
            ts.append(e0.elapsed_time(e1))
    ms = float(np.median(ts))
    rate = Bn * steps / (ms * 1e-3)
    h = float(np.abs(t_out.cpu().numpy()).sum())
    print(f"B={Bn:6d}  {ms:9.3f} ms  {rate:10.4e} point.steps/s  {flops * rate / 1e12:6.2f} TF credited  "
          f"{100 * flops * rate / 1e12 / peak_tf:5.1f} % of peak   checksum {h:.12e}", flush=True)
