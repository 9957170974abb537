#!/usr/bin/env python
"""tools/sym_sweep_bench.py -- the symmetric sweep kernels (stage_sym, csrc/yaman4.cu) against the 4-wave ones on one B200.

The bench's physics (BASELINE configs[3]: p_in = [0.1, 0.1, 1e-7, 1e-7], 2 500 RK4 steps, save_every 10) through
`fpa_yaman4_sweep_dev`, timed with FPA_SWEEP_SYM=1 and =0 alternately in one process (CUDA events, the L2 overwritten
before every launch, median of the repetitions), at 1e6 points (whole-run kernel), 250 000 and 125 000 points (the
4- and 8-GPU shards, z-segment scheduler) and at 1e6 points with GENERAL_TAYLOR Delta-beta.  Every pair of runs is
byte-compared on gain, Delta-beta, valid, status, Pmax and the end state.  --lib PATH adds other builds of the same
C ABI (launch-shape variants); each is timed against the shipped library's 4-wave kernels.

usage: python tools/sym_sweep_bench.py [--reps N] [--lib PATH ...] [--out profiles/r3_sym_sweep.txt]
"""
import argparse
import ctypes as C
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import __graft_entry__ as entry  # noqa: E402
import bench  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--lib", action="append", default=[], help="another build of libfpa_b200.so to time (SYM=1)")
ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_sym_sweep.txt"))
args = ap.parse_args()

entry.build()
fpa = entry.load_package()
L = fpa._lib
from oracle import fwm_oracle as O  # noqa: E402  (dispersion constants of the bench workload only)

dev = torch.device("cuda", 0)
torch.cuda.set_device(0)
L.check(L.lib().fpa_set_device(0))
N3 = 1000
n_steps = int(round(bench.Z_MAX / bench.DZ))
odisp = bench.fiber_dispersion(O)
disp = fpa.dispersion.DispersionParams(omega_ref=odisp.omega_ref, beta2=odisp.b[2], beta3=odisp.b[3], beta4=odisp.b[4])
t_flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
out_lines = []


def say(s=""):
    print(s, flush=True)
    out_lines.append(s)


def smi(q):
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "n/a"


def case(n1, method):
    """Buffers and descriptor of one sweep: n1 pump rows x N3 signal points."""
    B = n1 * N3
    lam1 = np.linspace(1545e-9, 1555e-9, 1000)[:n1].copy()
    lam3 = np.linspace(1540e-9, 1565e-9, N3)
    t = {"l1": torch.from_numpy(lam1).to(dev), "l3": torch.from_numpy(lam3).to(dev),
         "l2": torch.tensor([bench.LAM_P2], dtype=torch.float64, device=dev)}
    for k, dt, n in (("gain", torch.float64, B), ("dbeta", torch.float64, B), ("valid", torch.int32, B),
                     ("status", torch.int32, B), ("Pmax", torch.float64, 4 * B), ("A_end", torch.float64, 8 * B)):
        t[k] = torch.empty(n, dtype=dt, device=dev)
    d = L.SweepDesc()
    d.plan.n1, d.plan.n3 = n1, N3
    d.plan.lambda1, d.plan.lambda2, d.plan.lambda3 = t["l1"].data_ptr(), t["l2"].data_ptr(), t["l3"].data_ptr()
    d.plan.lambda2_stride = 0
    fpa.phase_matching.fill_plan_desc(d.plan, disp, fpa.phase_matching.PhaseMatchingConfig(method=method))
    d.plan.omega, d.plan.dbeta, d.plan.valid = None, t["dbeta"].data_ptr(), t["valid"].data_ptr()
    A0 = fpa.simulation.make_initial_amplitudes(bench.P_IN)
    for j in range(4):
        d.A0[2 * j], d.A0[2 * j + 1] = A0[j].real, A0[j].imag
    d.p_signal, d.gamma, d.alpha = bench.P_IN[2], bench.GAMMA, bench.ALPHA
    d.z_max, d.dz, d.length_scale, d.save_every = bench.Z_MAX, bench.DZ, 1.0, bench.SAVE_EVERY
    d.flags = L.CHECK_NAN
    d.gain_lin, d.status, d.Pmax, d.A_end = t["gain"].data_ptr(), t["status"].data_ptr(), t["Pmax"].data_ptr(), t["A_end"].data_ptr()
    nb = int(L.lib().fpa_yaman4_sweep_scratch_bytes(B))
    t["scratch"] = torch.empty(max(nb, 16), dtype=torch.uint8, device=dev)
    return d, t, nb


def run_once(d, t, nb, sym):
    os.environ["FPA_SWEEP_SYM"] = "1" if sym else "0"
    for k in ("gain", "dbeta", "valid", "status", "Pmax", "A_end"):
        t[k].fill_(-7)                                  # every output must be written by the launch
    t_flush.zero_()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    L.check(L.lib().fpa_yaman4_sweep_dev(C.byref(d), t["scratch"].data_ptr(), nb, torch.cuda.current_stream().cuda_stream))
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), b"".join(t[k].cpu().numpy().tobytes() for k in ("gain", "dbeta", "valid", "status", "Pmax", "A_end"))


def compare(label, n1, method, libs):
    """Alternate SYM=1 / SYM=0 (and the extra builds, SYM=1); median times, byte comparison."""
    d, t, nb = case(n1, method)
    B = n1 * N3
    arms = [("sym", None, True), ("4-wave", None, False)] + [(f"sym {Path(p).parent.name}/{Path(p).name}", p, True) for p in libs]
    times = {a[0]: [] for a in arms}
    ref = None
    same = True
    for r in range(args.reps + 1):
        for name, path, sym in arms:
            if path is None:
                ms, blob = run_once(d, t, nb, sym)
            else:
                with L.use_library(path):
                    ms, blob = run_once(d, t, nb, sym)
            if r == 0:                                  # warm-up round: module load, first launch
                if ref is None:
                    ref = blob
                same &= blob == ref
                continue
            times[name].append(ms)
            same &= blob == ref
    os.environ.pop("FPA_SWEEP_SYM", None)
    base = float(np.median(times["4-wave"]))
    say(f"{label}: {B} points x {n_steps} steps, outputs (gain, dbeta, valid, status, Pmax, A_end) "
        f"{'byte-identical' if same else 'DIFFERENT'} across all arms")
    for name, _, _ in arms:
        ms = float(np.median(times[name]))
        rate = B * n_steps / (ms * 1e-3)
        spread = (max(times[name]) - min(times[name])) / ms * 100
        say(f"  {name:<28s} {ms:9.2f} ms  {rate:.4e} point.steps/s  x{base / ms:5.3f} vs 4-wave  "
            f"(spread {spread:.2f} % over {len(times[name])})")
    return same


say(f"device {torch.cuda.get_device_name(0)}; power.limit {smi('power.limit')}; clocks.max.sm {smi('clocks.max.sm')}; "
    f"clocks.sm now {smi('clocks.sm')}; library {L.lib().fpa_version().decode()}")
say(f"bench physics: p_in {bench.P_IN}, gamma {bench.GAMMA}, alpha {bench.ALPHA:.6e} 1/m, dz {bench.DZ} m, "
    f"save_every {bench.SAVE_EVERY}; {args.reps} timed repetitions per arm, alternating, L2 overwritten before each")
PM = fpa.phase_matching.PhaseMatchingMethod
ok = True
ok &= compare("1e6 points, SYMMETRIC_EVEN (whole-run kernel)", 1000, PM.SYMMETRIC_EVEN, args.lib)
ok &= compare("1e6 points, GENERAL_TAYLOR (whole-run kernel)", 1000, PM.GENERAL_TAYLOR, [])
ok &= compare("250 000 points (4-GPU shard), SYMMETRIC_EVEN", 250, PM.SYMMETRIC_EVEN, args.lib)
ok &= compare("125 000 points (8-GPU shard), SYMMETRIC_EVEN", 125, PM.SYMMETRIC_EVEN, args.lib)
say(f"clocks.sm after {smi('clocks.sm')}; power.draw {smi('power.draw')}")
Path(args.out).parent.mkdir(parents=True, exist_ok=True)
Path(args.out).write_text("\n".join(out_lines) + "\n")
sys.exit(0 if ok else 1)
