#!/usr/bin/env python
"""tools/transfer_bench.py -- the transfer sweep (fpa_yaman4_transfer_sweep_dev) against the plain 4-wave sweep on one B200.

The bench's physics (BASELINE configs[3]: 1000 x 1000 grid, p_in = [0.1, 0.1, 1e-7, 1e-7], 2 500 RK4 steps) timed
in one process, alternating: the plain sweep with FPA_SWEEP_SYM=0 (4-wave kernels, z-segment scheduler scratch
given), the transfer sweep at waves (2, 3) (4 columns) and at all 8 columns; CUDA events, the L2 overwritten before
every launch, median of the repetitions.  The transfer runs' gain, Delta-beta, valid and status are byte-compared
with the plain sweep's.  Reports point.steps/s, column.point.steps/s and the FP64 instructions per RK4 step of one
lane, counted in the z-loop of each kernel in `cuobjdump -sass` of the shipped library; the card name, power limit
and SM clock are read in the same run.

usage: python tools/transfer_bench.py [--reps N] [--out profiles/r4_transfer_bench.txt]
"""
import argparse
import ctypes as C
import os
import re
import shutil
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
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--out", default=str(ROOT / "profiles" / "r4_transfer_bench.txt"))
args = ap.parse_args()

entry.build()
fpa = entry.load_package()
L = fpa._lib
from oracle import fwm_oracle as O  # noqa: E402  (dispersion constants of the bench workload only)

dev = torch.device("cuda", 0)
torch.cuda.set_device(0)
L.check(L.lib().fpa_set_device(0))
N1 = N3 = 1000
B = N1 * N3
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


def fp64_per_step(kernel_re):
    """FP64 instructions (D* opcodes) in the innermost loop with the most of them, in the first SASS function whose
    name matches kernel_re: one RK4 step of one lane."""
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    text = subprocess.run([exe, "-sass", str(entry.LIB)], capture_output=True, text=True).stdout
    funcs = re.split(r"\n\s+Function : ", text)
    for f in funcs[1:]:
        name = f.split("\n", 1)[0].strip()
        if not re.search(kernel_re, name):
            continue
        ins = []
        for m in re.finditer(r"/\*([0-9a-f]{4,})\*/\s+(@!?U?P\w+\s+)?([A-Z][A-Z0-9_.]*)([^;]*);", f):
            ins.append((int(m.group(1), 16), m.group(3), m.group(4)))
        best = 0
        for addr, op, rest in ins:
            if op.startswith("BRA"):
                t = re.search(r"0x([0-9a-f]+)", rest)
                if t and int(t.group(1), 16) < addr:
                    lo = int(t.group(1), 16)
                    n = sum(1 for a, o, _ in ins if lo <= a <= addr and re.match(r"D(FMA|MUL|ADD)", o))
                    best = max(best, n)
        return name, best
    return None, 0


def case(columns):
    """Buffers and descriptor of one sweep (columns None: the plain sweep)."""
    lam1 = np.linspace(1545e-9, 1555e-9, N1)
    lam3 = np.linspace(1540e-9, 1565e-9, N3)
    t = {"l1": torch.from_numpy(lam1).to(dev), "l3": torch.from_numpy(lam3).to(dev),
         "l2": torch.tensor([bench.LAM_P2], dtype=torch.float64, device=dev)}
    for k, dt, n in (("gain", torch.float64, B), ("dbeta", torch.float64, B), ("valid", torch.int32, B),
                     ("status", torch.int32, B)):
        t[k] = torch.empty(n, dtype=dt, device=dev)
    d = L.SweepDesc()
    d.plan.n1, d.plan.n3 = N1, N3
    d.plan.lambda1, d.plan.lambda2, d.plan.lambda3 = t["l1"].data_ptr(), t["l2"].data_ptr(), t["l3"].data_ptr()
    d.plan.lambda2_stride = 0
    fpa.phase_matching.fill_plan_desc(d.plan, disp, fpa.phase_matching.PhaseMatchingConfig(
        method=fpa.phase_matching.PhaseMatchingMethod.SYMMETRIC_EVEN))
    d.plan.omega, d.plan.dbeta, d.plan.valid = None, t["dbeta"].data_ptr(), t["valid"].data_ptr()
    A0 = fpa.simulation.make_initial_amplitudes(bench.P_IN)
    for j in range(4):
        d.A0[2 * j], d.A0[2 * j + 1] = A0[j].real, A0[j].imag
    d.p_signal, d.gamma, d.alpha = bench.P_IN[2], bench.GAMMA, bench.ALPHA
    d.z_max, d.dz, d.length_scale, d.save_every = bench.Z_MAX, bench.DZ, 1.0, bench.SAVE_EVERY
    d.flags = L.CHECK_NAN
    d.gain_lin, d.status = t["gain"].data_ptr(), t["status"].data_ptr()
    tout = None
    if columns is None:
        nb = int(L.lib().fpa_yaman4_sweep_scratch_bytes(B))
        t["scratch"] = torch.empty(max(nb, 16), dtype=torch.uint8, device=dev)
    else:
        nc = bin(columns).count("1")
        t["jac"] = torch.empty(B * 8 * nc, dtype=torch.float64, device=dev)
        tout = L.TransferOut(columns=columns, jac=t["jac"].data_ptr())
        nb = 0
    return d, t, nb, tout


def run_once(d, t, nb, tout):
    for k in ("gain", "dbeta", "valid", "status"):
        t[k].fill_(-7)
    t_flush.zero_()
    st = torch.cuda.current_stream().cuda_stream
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    if tout is None:
        L.check(L.lib().fpa_yaman4_sweep_dev(C.byref(d), t["scratch"].data_ptr(), nb, st))
    else:
        L.check(L.lib().fpa_yaman4_transfer_sweep_dev(C.byref(d), C.byref(tout), st))
    e1.record()
    torch.cuda.synchronize()
    blob = b"".join(t[k].cpu().numpy().tobytes() for k in ("gain", "dbeta", "valid", "status"))
    return e0.elapsed_time(e1), blob


say(f"device {torch.cuda.get_device_name(0)}; power.limit {smi('power.limit')}; clocks.max.sm {smi('clocks.max.sm')}; "
    f"clocks.sm now {smi('clocks.sm')}; library {L.lib().fpa_version().decode()}")
say(f"bench physics: {N1} x {N3} grid, {n_steps} steps, p_in {bench.P_IN}, gamma {bench.GAMMA}, alpha {bench.ALPHA:.6e} 1/m, "
    f"save_every {bench.SAVE_EVERY}; {args.reps} timed repetitions per arm, alternating, L2 overwritten before each")
os.environ["FPA_SWEEP_SYM"] = "0"
arms = [("plain 4-wave sweep", None, 1), ("transfer, 4 columns (2,3)", 0xF0, 4), ("transfer, 8 columns", 0xFF, 8)]
bufs = {name: case(cols) for name, cols, _ in arms}
times = {name: [] for name, _, _ in arms}
ref, same = None, True
for r in range(args.reps + 1):
    for name, _, _ in arms:
        ms, blob = run_once(*bufs[name])
        ref = blob if ref is None else ref
        same &= blob == ref
        if r > 0:
            times[name].append(ms)
os.environ.pop("FPA_SWEEP_SYM", None)
say(f"gain, dbeta, valid, status {'byte-identical' if same else 'DIFFERENT'} across the three arms")
base = float(np.median(times[arms[0][0]]))
for name, _, nc in arms:
    ms = float(np.median(times[name]))
    spread = (max(times[name]) - min(times[name])) / ms * 100
    rate = B * n_steps / (ms * 1e-3)
    extra = f"  {rate * nc if nc > 1 else rate:.4e} column.point.steps/s" if nc > 1 else ""
    say(f"  {name:<28s} {ms:10.2f} ms  {rate:.4e} point.steps/s{extra}  x{ms / base:6.2f} the plain sweep's time  "
        f"(spread {spread:.2f} % over {len(times[name])})")
for label, rex in (("plain 4-wave sweep kernel", r"yaman4_sweep_kernel.*ILb1ELi128ELi4ENS_10SweepExtraELb0E"),
                   ("transfer sweep kernel (lossy)", r"yaman4_transfer_kernelILi1ENS_10SweepExtra")):
    name, n = fp64_per_step(rex)
    say(f"FP64 instructions per RK4 step per lane, {label}: {n}  ({name})")
say(f"clocks.sm after {smi('clocks.sm')}; power.draw {smi('power.draw')}")
Path(args.out).parent.mkdir(parents=True, exist_ok=True)
Path(args.out).write_text("\n".join(out_lines) + "\n")
sys.exit(0 if same else 1)
