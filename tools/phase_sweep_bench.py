#!/usr/bin/env python
"""tools/phase_sweep_bench.py [--steps N] [--reps R] [--out FILE] -- the phase sweep (fpa_yaman4_phase_sweep_dev:
sweep kernel + reduction kernel) against the plain sweep (fpa_yaman4_sweep_dev) at the same number of runs:
250 x 250 x 16 phases against a 1000 x 1000 grid, and 1000 x 1000 x 16 phases against a 4000 x 4000 grid.  Same
wavelength ranges (every plan valid), same physics and step count, so the per-run work is identical.

Device-resident (torch buffers), CUDA events around each call, one warm-up call per arm, the 126 MB L2 overwritten
by a 512 MB fill before every timed call, the two arms alternated `reps` times; the spread is max/min - 1 per arm.
A second pass under torch.profiler gives the reduction kernel's share of the phase sweep's device time.  The card
name, power limit and SM clock are read in the same run."""
import argparse
import ctypes as C
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import __graft_entry__ as entry  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=500)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--out", default=None)
args = ap.parse_args()

entry.build()
fpa = entry.load_package()
L, lib = fpa._lib, fpa._lib.lib()
dev = torch.device("cuda", 0)
torch.cuda.set_device(0)
L.check(lib.fpa_set_device(0))
stream = torch.cuda.current_stream()


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def axes(n1, n3):
    return (torch.from_numpy(np.linspace(1545e-9, 1555e-9, n1)).to(dev),
            torch.tensor([1558e-9], dtype=torch.float64, device=dev),
            torch.from_numpy(np.linspace(1540e-9, 1565e-9, n3)).to(dev))


disp = fpa.dispersion.DispersionParams(omega_ref=2 * np.pi * 299792458.0 / 1553e-9, beta2=-2.0e-28, beta3=1.2e-40,
                                       beta4=-1.5e-55)
P_IN = [0.5, 0.5, 1e-6, 1e-6]
Z_MAX, DZ = 0.2 * args.steps, 0.2


def fill_sweep(w, n1, n3, ax):
    w.plan.n1, w.plan.n3 = n1, n3
    w.plan.lambda1, w.plan.lambda2, w.plan.lambda3 = (t.data_ptr() for t in ax)
    fpa.phase_matching.fill_plan_desc(w.plan, disp, fpa.phase_matching.PhaseMatchingConfig())
    w.p_signal, w.gamma, w.alpha = P_IN[2], 11.5e-3, 1e-4
    w.z_max, w.dz, w.length_scale, w.save_every = Z_MAX, DZ, 1.0, 10
    w.flags = L.CHECK_NAN


class Plain:
    def __init__(self, n1, n3):
        self.B = n1 * n3
        self.ax = axes(n1, n3)
        self.db = torch.empty(self.B, dtype=torch.float64, device=dev)
        self.va = torch.empty(self.B, dtype=torch.int32, device=dev)
        self.gain = torch.empty(self.B, dtype=torch.float64, device=dev)
        self.st = torch.empty(self.B, dtype=torch.int32, device=dev)
        self.nb = int(lib.fpa_yaman4_sweep_scratch_bytes(self.B))
        self.scr = torch.empty(max(self.nb, 16), dtype=torch.uint8, device=dev)
        self.d = L.SweepDesc()
        fill_sweep(self.d, n1, n3, self.ax)
        A0 = fpa.simulation.make_initial_amplitudes(P_IN)
        for j in range(4):
            self.d.A0[2 * j], self.d.A0[2 * j + 1] = A0[j].real, A0[j].imag
        self.d.plan.dbeta, self.d.plan.valid = self.db.data_ptr(), self.va.data_ptr()
        self.d.gain_lin, self.d.status = self.gain.data_ptr(), self.st.data_ptr()

    def __call__(self):
        L.check(lib.fpa_yaman4_sweep_dev(C.byref(self.d), self.scr.data_ptr(), self.nb, stream.cuda_stream))


class Phased:
    def __init__(self, n1, n3, K):
        G = n1 * n3
        self.B = G * K
        self.ax = axes(n1, n3)
        table, _, _ = fpa.scan_mismtach.phase_sweep_inputs(P_IN, None, np.linspace(0, 2 * np.pi, K, endpoint=False))
        self.tab = torch.from_numpy(table.view(np.float64).copy()).to(dev)
        self.db = torch.empty(G, dtype=torch.float64, device=dev)
        self.va = torch.empty(G, dtype=torch.int32, device=dev)
        self.gain = torch.empty(self.B, dtype=torch.float64, device=dev)
        self.st = torch.empty(self.B, dtype=torch.int32, device=dev)
        self.red = [torch.empty(G, dtype=dt, device=dev) for dt in (torch.float64, torch.float64, torch.int32,
                                                                     torch.int32, torch.int32)]
        self.nb = int(lib.fpa_yaman4_phase_sweep_scratch_bytes(self.B))
        self.scr = torch.empty(max(self.nb, 16), dtype=torch.uint8, device=dev)
        self.d = L.PhaseSweepDesc()
        fill_sweep(self.d.sweep, n1, n3, self.ax)
        self.d.sweep.plan.dbeta, self.d.sweep.plan.valid = self.db.data_ptr(), self.va.data_ptr()
        self.d.sweep.gain_lin, self.d.sweep.status = self.gain.data_ptr(), self.st.data_ptr()
        self.d.n_phases, self.d.A0_table, self.d.metric = K, self.tab.data_ptr(), L.GAIN_LAST_SAVED
        (self.d.gain_max, self.d.gain_min, self.d.idx_max, self.d.idx_min, self.d.n_finite) = (t.data_ptr()
                                                                                            for t in self.red)

    def __call__(self):
        L.check(lib.fpa_yaman4_phase_sweep_dev(C.byref(self.d), self.scr.data_ptr(), self.nb, stream.cuda_stream))


flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)


def timed(fn):
    flush.fill_(1)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e-3


def reduction_share(fn):
    """(reduction kernel time, sweep kernel time) of one call, from torch.profiler's CUDA activity."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    red = sweep = 0.0
    for e in prof.events():
        t = getattr(e, "device_time", None) or getattr(e, "cuda_time", 0.0)
        if "phase_reduce_kernel" in e.name:
            red += t
        elif "yaman4_sweep" in e.name:
            sweep += t
    return red * 1e-6, sweep * 1e-6


info = card()
print(f"# {info}; {args.steps} RK4 steps per run, save_every 10, lossy, CUDA events, L2 overwritten before each call",
      flush=True)
results = []
for (n1p, n3p, K), (n1, n3) in (((250, 250, 16), (1000, 1000)), ((1000, 1000, 16), (4000, 4000))):
    ph, pl = Phased(n1p, n3p, K), Plain(n1, n3)
    assert ph.B == pl.B
    ph(), pl()                                                     # warm-up: module load, first launch
    torch.cuda.synchronize()
    t_ph, t_pl = [], []
    for _ in range(args.reps):
        t_ph.append(timed(ph))
        t_pl.append(timed(pl))
    g_ph = ph.gain.cpu().numpy()
    fin = float(np.isfinite(g_ph).mean())
    red, swp = reduction_share(ph)
    rate = lambda ts: ph.B * args.steps / float(np.median(ts))  # noqa: E731
    row = {"phase_sweep": f"{n1p}x{n3p}x{K}", "plain_sweep": f"{n1}x{n3}", "runs": ph.B, "steps": args.steps,
           "phase_s": [round(v, 6) for v in t_ph], "plain_s": [round(v, 6) for v in t_pl],
           "phase_spread": round(max(t_ph) / min(t_ph) - 1, 4), "plain_spread": round(max(t_pl) / min(t_pl) - 1, 4),
           "phase_point_steps_per_s": rate(t_ph), "plain_point_steps_per_s": rate(t_pl),
           "phase_over_plain": rate(t_ph) / rate(t_pl), "finite_fraction": fin,
           "profiler_reduction_ms": red * 1e3, "profiler_sweep_ms": swp * 1e3,
           "reduction_share": red / swp if swp else None, "card": info}
    results.append(row)
    print(json.dumps(row), flush=True)
    del ph, pl
    torch.cuda.empty_cache()
if args.out:
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text("".join(json.dumps(r) + "\n" for r in results))
