#!/usr/bin/env python
"""bench.py -- scan-points x RK4-steps / second of the batched FWM sweep on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[3], the configuration the metric is quoted on): the 2-D pump x signal
wavelength sweep, 1000 x 1000 = 1e6 scan points, 2 500 RK4 steps each (z_max = 500 m, dz = 0.2 m,
save_every = 10), physics of the reference's main.py:206-279.  A "step" of this benchmark is ONE full
sweep = ONE kernel launch per GPU: frequency plan + Delta-beta prologue, fused RK4 integration and gain
metric for every point = 2.5e9 point.RK4-steps.

  value     device-resident inputs (wavelength axes already in HBM), CUDA-event timed, max over ranks
  e2e       the same sweep through the public call (scan_mismtach.sweep_gain_2d -> fpa_yaman4_sweep_host)
            with HOST buffers: H2D of the axes and delivery of gain / dbeta / valid / status into host
            memory inside the timed region; at N > 1 every rank's kernel stores its shard into ONE
            shared host array (the assembled map), timed to the last rank
  roofline  FP64 FMA pipe: 568 algorithmic flops per point.step / integrator-kernel time, against the
            DFMA peak measured live on this GPU (MEASURED_PEAKS.json has no FP64 figure) and against the
            nominal 148 SM x 64 lanes x 2 x clock
  cpu_baseline  the reference's numpy path on the host cores (bounded sample): the byte-compiled
            reference itself (oracle/_ref, kind "reference") when present, else the bit-equal oracle port
  secondary the other BASELINE configurations (1a, 2, 3 short + long, 4 with GENERAL_TAYLOR, 5 at
            B = 1 and 1024, trace write-out), N = 1 only

N > 1 (torchrun, one rank per GPU): the headline is STRONG scaling -- the fixed 1e6-point grid of the
config is split into N contiguous point ranges, one kernel per GPU; the final gather of the gain map is
done by the sweep kernel itself (NVLink peer stores into the full-size map of every GPU, opened over CUDA
IPC; `--gather nccl` or a box without peer access: an NCCL all-gather after the kernel); the weak-scaling
figure (1e6 points per GPU, NCCL all-gather) is reported alongside under "weak".
`--impl reference` times the CPU arm with all host cores; only rank 0 works.

`--dump-outputs DIR` writes what the last timed step computed as DIR/<name>.npy.  The inputs are fixed
(linspace axes, seeded samples), so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "scan-points*RK4-steps/sec (FP64)"
UNIT = "point-steps/s"
N1, N3 = 1000, 1000
Z_MAX, DZ, SAVE_EVERY = 500.0, 0.2, 10
GAMMA = 11.5e-3
ALPHA = float(np.log(10) / 10 * 0.5 / 1000)
P_IN = [0.1, 0.1, 1e-7, 1e-7]
LAM_P2 = 1558e-9
FLOPS_PER_POINT_STEP = 568.0
FLOPS_LOSSLESS = 504.0       # alpha == 0: the 4 x 8 loss FMAs of a step are not executed, so not credited
FLUSH_BYTES = 136 << 20      # 142.6e6 B > the 126 MB L2, written between steps
RESULT_OUT = sys.stdout      # main() replaces it with a private duplicate of the original stdout
WORKLOAD = ("sweep2d_1000x1000_x2500steps (BASELINE configs[3]: pump x signal wavelength sweep, 1e6 scan points, "
            "z_max=500 m, dz=0.2 m, save_every=10, SYMMETRIC_EVEN(2,4) dbeta, max-over-saved signal gain)")


def grid_axes(rows: int = N1):
    """Wavelength axes of the sweep: `rows` pump wavelengths x 1000 signal wavelengths."""
    return np.linspace(1545e-9, 1555e-9, rows), np.linspace(1540e-9, 1565e-9, N3)


def balanced_range(n: int, world: int, rank: int):
    base, extra = divmod(int(n), int(world))
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def fiber_dispersion(O):
    """Dispersion of the reference's main.py sweep: D = 0.1, S = 0.02 at lambda_c of (1550, 1558) nm."""
    om = O.plan_from_wavelengths(1550e-9, LAM_P2, 1540e-9)
    oc, _, _ = O.symmetric_vars(om)
    return O.taylor_from_D_S(O.TWO_PI * O.C_LIGHT / oc, 0.1, 0.02, 0.0, omega_ref=oc)


def ncu_traffic_bytes(seg: bool):
    """dram read + write bytes per launch of the sweep kernel that ran -- the whole-run kernel or the
    z-segment scheduler -- from the newest committed ncu summary of that kernel
    (profiles/r*_ncu_yaman4_sweep_kernel*.csv / r*_ncu_yaman4_sweep_seg_kernel*.csv); (None, None) when there is none."""
    best = None
    for path in sorted((ROOT / "profiles").glob(f"r*_ncu_yaman4_sweep_{'seg_' if seg else ''}kernel*.csv")):
        vals = {}
        for line in path.read_text().splitlines():
            parts = line.split(",")
            if len(parts) >= 3 and parts[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(parts[1])
                if scale is not None:
                    vals[parts[0]] = float(parts[2]) * scale
        if len(vals) == 2:
            best = (sum(vals.values()), path.name)
    return best if best else (None, None)


def dump_outputs(out_dir, arrays: dict) -> None:
    """Write the results of the last timed step as <out_dir>/<name>.npy: a map of the whole grid as [N1, N3],
    anything smaller (a shard, a sample of points) flat."""
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out_dir / f"{name}.npy", a.reshape(N1, N3) if a.size == N1 * N3 else a)


# ----------------------------------------------------------------------------- CPU arm
_REF = None


def cpu_kind() -> str:
    from oracle import build_ref
    return "reference" if build_ref.available() else "port"


def _cpu_points(args):
    """Worker: the reference's per-point sweep body (scan_mismtach.py:694-738) over a handful of
    (lam1, lam3) points -- the byte-compiled reference itself, or the oracle port.  Returns gains."""
    global _REF
    pts, disp_tuple, kind = args
    out = []
    if kind == "reference":
        if _REF is None:
            from oracle import build_ref
            _REF = build_ref.load()
        R = _REF
        disp = R.dispersion.DispersionParams(omega_ref=disp_tuple[0], beta0=disp_tuple[1], beta1=disp_tuple[2],
                                             beta2=disp_tuple[3], beta3=disp_tuple[4], beta4=disp_tuple[5])
        cfg = R.config.custom_simulation_config(z_max=Z_MAX, dz=DZ, save_every=SAVE_EVERY)
        for l1, l3 in pts:
            _, g, _ = R.scan_mismtach.plot_max_gain_and_dbeta_vs_lambda_signal(
                cfg=cfg, lambda_p1_m=l1, lambda_p2_m=LAM_P2, lambda_signal_m=[l3], gamma=GAMMA, alpha=ALPHA,
                p_in=P_IN, dispersion=disp, gain_unit="linear", show_progress=False, show=False)
            out.append(float(g[0]))
        return out
    from oracle import fwm_oracle as O
    disp = O.Taylor(*disp_tuple)
    for l1, l3 in pts:
        g, _ = O.sweep_lambda3_gain(lam1=l1, lam2=LAM_P2, lam3_arr=[l3], z_max=Z_MAX, dz=DZ,
                                    save_every=SAVE_EVERY, check_nan=True, gamma=GAMMA, alpha=ALPHA,
                                    p_in=P_IN, disp=disp, gain_unit="linear")
        out.append(float(g[0]))
    return out


def cpu_sample(n_points: int, cores: int, seed: int = 0, kind: str = "port"):
    """Time the CPU arm on `n_points` random grid points with `cores` processes.
    Returns (points*steps/s, wall seconds, sample indices, gains)."""
    import multiprocessing as mp
    from oracle import fwm_oracle as O
    disp = fiber_dispersion(O)
    lam1, lam3 = grid_axes()
    rng = np.random.default_rng(seed)
    idx = rng.choice(N1 * N3, size=n_points, replace=False)
    pts = [(float(lam1[i // N3]), float(lam3[i % N3])) for i in idx]
    chunks = [pts[c::cores] for c in range(cores)]
    dt = (disp.omega_ref, *disp.b)
    n_steps = int(round(Z_MAX / DZ))
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        pool.map(_cpu_points, [([pts[0]], dt, kind)] * cores)          # spin the workers up (untimed)
        t0 = time.perf_counter()
        res = pool.map(_cpu_points, [(c, dt, kind) for c in chunks])
        wall = time.perf_counter() - t0
    gains = np.empty(n_points)
    for c, r in enumerate(res):
        gains[c::cores] = r
    return n_points * n_steps / wall, wall, idx, gains


CPU_NOTE = {
    "reference": "the UNMODIFIED reference (byte-compiled by oracle/build_ref.py from /root/reference into oracle/_ref, "
                 "imported sourceless): scan_mismtach.plot_max_gain_and_dbeta_vs_lambda_signal per point, one process per host core",
    "port": "oracle/fwm_oracle.py (bit-equal restatement of the reference's numpy RK4, pinned by "
            "oracle/pin_against_reference.py; oracle/_ref is absent here), one process per host core",
}


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    kind = cpu_kind()
    cores = os.cpu_count() or 1
    per_core = 16 if kind == "port" else 6     # a few seconds of all-core work per bench step
    n_points = per_core * cores
    n_steps = int(round(Z_MAX / DZ))
    for _ in range(max(args.warmup, 0)):
        cpu_sample(cores, cores, seed=99, kind=kind)
    t_total = 0.0
    for k in range(args.steps):
        _, wall, idx, gains = cpu_sample(n_points, cores, seed=k, kind=kind)
        t_total += wall
    if args.dump_outputs:       # the sampled points of the last step: flat indices into the N1 x N3 grid
        dump_outputs(args.dump_outputs, {"gain_lin": gains, "point_index": idx.astype(np.float64)})
    value = n_points * n_steps * args.steps / t_total
    sample = f"{n_points} random points of the 1000x1000 grid x {n_steps} RK4 steps per bench step"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": WORKLOAD + ", bounded sample", "points_per_step": n_points, "rk4_steps": n_steps},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "timed arm: " + CPU_NOTE[kind],
    }), file=RESULT_OUT, flush=True)


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def summary(self, t0: float = 0.0, t1: float = float("inf")) -> dict:
        """Summary of the samples taken inside [t0, t1]."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm, smax, power, reasons = [], [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        inside = [r for t, r in list(self.rows) if t0 <= t <= t1 + 0.15]
        for r in inside:
            try:
                sm.append(float(r[0])); smax.append(float(r[1])); power.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, flag in zip(names, r[3:7]):
                if flag.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(smax)), "power_w_max": max(power),
                "samples": len(sm), "reasons": sorted(reasons)}

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()


# ----------------------------------------------------------------------------- GPU arm helpers
class PeerMaps:
    """One full-size gain map per GPU of the box, each opened in every rank (CUDA IPC through the C ABI): the
    sweep kernel stores each point's gain into all of them (`fpa_sweep_desc.peer_gain`), which IS the final
    gather -- no collective after the kernel.  `setup` returns None (on every rank alike) when any rank cannot
    allocate, export or open a map; every rank takes part in every collective of the set-up whatever happened
    locally, so a failure on one rank cannot leave the others waiting."""

    @classmethod
    def setup(cls, fpa, dist, torch, world, rank, local, n_points):
        self = cls()
        L, lib = fpa._lib, fpa._lib.lib()
        self.lib, self.n, self.torch, self.dev = lib, n_points, torch, torch.device("cuda", local)
        self.own, self.ptrs, self.opened = C.c_void_p(), [], []
        handle, why = None, ""
        try:
            L.check(lib.fpa_dev_alloc(C.byref(self.own), n_points * 8, local))
            buf = (C.c_char * 64)()
            L.check(lib.fpa_ipc_export(self.own, buf))
            handle = bytes(buf.raw)
        except Exception as exc:                      # noqa: BLE001
            why = repr(exc)
        handles = [None] * world
        dist.all_gather_object(handles, handle)
        ok = all(h is not None for h in handles)
        if ok:
            try:
                for r in range(world):
                    if r == rank:
                        self.ptrs.append(self.own.value)
                        continue
                    q = C.c_void_p()
                    L.check(lib.fpa_ipc_open(handles[r], C.byref(q)))
                    self.ptrs.append(q.value)
                    self.opened.append(q)
            except Exception as exc:                  # noqa: BLE001
                ok, why = False, repr(exc)
        flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=self.dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 1:
            return self
        if why:
            print(f"rank {rank}: peer maps unavailable ({why}); falling back to the NCCL all-gather", file=sys.stderr)
        self.close(dist)
        return None

    def own_map(self):
        """This rank's map as a torch tensor (no copy)."""
        class _View:
            pass
        v = _View()
        v.__cuda_array_interface__ = {"shape": (self.n,), "typestr": "<f8", "data": (self.own.value, False), "version": 3}
        return self.torch.as_tensor(v, device=self.dev)

    def close(self, dist):
        for q in self.opened:
            self.lib.fpa_ipc_close(q)
        self.opened = []
        dist.barrier()              # nobody still has this rank's map open
        if self.own.value:
            self.lib.fpa_dev_free(self.own)
            self.own = C.c_void_p()


class DeviceSweep:
    """Device-resident descriptor of one rank's share of a sweep: points [first, first + count) of the
    flattened rows x 1000 grid; the wavelength axes already live in HBM."""

    def __init__(self, fpa, torch, dev, rows, first, count, disp, pm_cfg, peer_maps=None):
        L, lib = fpa._lib, fpa._lib.lib()
        lam1, lam3 = grid_axes(rows)
        self.count = count
        self.t_l1 = torch.from_numpy(lam1).to(dev)
        self.t_l2 = torch.tensor([LAM_P2], dtype=torch.float64, device=dev)
        self.t_l3 = torch.from_numpy(lam3).to(dev)
        self.t_gain = torch.empty(count, dtype=torch.float64, device=dev)
        self.t_dbeta = torch.empty(count, dtype=torch.float64, device=dev)
        self.t_valid = torch.empty(count, dtype=torch.int32, device=dev)
        self.t_status = torch.empty(count, dtype=torch.int32, device=dev)
        self.scratch_bytes = int(lib.fpa_yaman4_sweep_scratch_bytes(count))   # z-segment scheduler state
        self.t_scratch = torch.empty(max(self.scratch_bytes, 16), dtype=torch.uint8, device=dev)
        d = L.SweepDesc()
        d.plan.n1, d.plan.n3 = rows, N3
        d.plan.lambda1, d.plan.lambda2, d.plan.lambda3 = self.t_l1.data_ptr(), self.t_l2.data_ptr(), self.t_l3.data_ptr()
        d.plan.lambda2_stride = 0
        fpa.phase_matching.fill_plan_desc(d.plan, disp, pm_cfg)
        d.plan.omega, d.plan.dbeta, d.plan.valid = None, self.t_dbeta.data_ptr(), self.t_valid.data_ptr()
        A0 = fpa.simulation.make_initial_amplitudes(P_IN)
        for j in range(4):
            d.A0[2 * j], d.A0[2 * j + 1] = A0[j].real, A0[j].imag
        d.p_signal, d.gamma, d.alpha = P_IN[2], GAMMA, ALPHA
        d.z_max, d.dz, d.length_scale, d.save_every = Z_MAX, DZ, 1.0, SAVE_EVERY
        d.flags = L.CHECK_NAN
        d.gain_lin, d.status, d.Pmax, d.A_end = self.t_gain.data_ptr(), self.t_status.data_ptr(), None, None
        if not (first == 0 and count == rows * N3):
            d.first_point, d.n_sub_points = first, count
        if peer_maps:       # the kernel stores every gain into the full-size map of every GPU of the box as well
            d.n_peers = len(peer_maps)
            for r, ptr in enumerate(peer_maps):
                d.peer_gain[r] = ptr
        self.desc, self.L, self.lib = d, L, lib

    def launch(self, stream):
        self.L.check(self.lib.fpa_yaman4_sweep_dev(C.byref(self.desc), self.t_scratch.data_ptr(), self.scratch_bytes, stream))


def timed_sweeps(torch, dist, sweep, gather, world, steps, warmup, t_flush, dev):
    """W warm-up steps, then exactly K timed steps between barrier + synchronize pairs.  A step = L2
    flush, one sweep launch (CUDA events around it, on its stream), the result gather.  Returns
    (ms_total max over ranks, per-launch kernel ms of the timed steps, wall-clock window)."""
    k_events = []

    def step():
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        t_flush.zero_()                                                    # L2 flush between steps
        stream = torch.cuda.current_stream().cuda_stream
        ev[1].record()
        sweep.launch(stream)
        ev[2].record()
        gather()
        ev[3].record()
        k_events.append(ev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warmup):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_begin = time.time()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    barrier()
    t_end = time.time()
    ms_total = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    k_ms = [ev[1].elapsed_time(ev[2]) for ev in k_events[-steps:]]
    parts = {"l2_flush_ms": float(np.mean([ev[0].elapsed_time(ev[1]) for ev in k_events[-steps:]])),
             "sweep_kernel_ms": float(np.mean(k_ms)),
             "gather_ms": float(np.mean([ev[2].elapsed_time(ev[3]) for ev in k_events[-steps:]])),
             "step_ms_this_rank": e0.elapsed_time(e1) / steps}
    return ms_total, k_ms, (t_begin, t_end), parts


def run_ours(args) -> None:
    import torch
    import torch.distributed as dist

    import __graft_entry__ as entry
    entry.build()
    fpa = entry.load_package()
    L, lib = fpa._lib, fpa._lib.lib()
    from oracle import fwm_oracle as O          # cpu_baseline leg and the workload's dispersion constants only

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("launch N > 1 with torchrun (one rank per GPU)")
    # The CPU leg forks worker processes: do it BEFORE this process creates a CUDA context (a forked
    # child of a CUDA process is fragile even when it never touches the GPU).  The sample is compared
    # with the GPU results further down.
    cpu_leg = None
    if world == 1 and not args.no_cpu_baseline and args.shard_of <= 1:
        kind = cpu_kind()
        cores = os.cpu_count() or 1
        n_pts = max(64, (40 if kind == "port" else 14) * cores)      # ~10-20 s of wall time on the box's cores
        cpu_value, wall, idx, cpu_gain = cpu_sample(n_pts, cores, seed=0, kind=kind)
        one_core, _, _, _ = cpu_sample(8 if kind == "port" else 4, 1, seed=1, kind=kind)   # the reference as shipped: one thread
        cpu_leg = (cores, n_pts, cpu_value, wall, idx, cpu_gain, one_core, kind)
    if not torch.cuda.is_available() or lib.fpa_device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    L.check(lib.fpa_set_device(local))
    L.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    odisp = fiber_dispersion(O)
    disp = fpa.dispersion.DispersionParams(omega_ref=odisp.omega_ref, beta2=odisp.b[2], beta3=odisp.b[3],
                                           beta4=odisp.b[4])
    pm_cfg = fpa.phase_matching.PhaseMatchingConfig()        # SYMMETRIC_EVEN (2,4): the reference default
    cfg = fpa.config.custom_simulation_config(z_max=Z_MAX, dz=DZ, save_every=SAVE_EVERY)
    n_steps = int(round(Z_MAX / DZ))
    t_flush = torch.empty(FLUSH_BYTES, dtype=torch.uint8, device=dev)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                 # nvidia-smi needs a few hundred ms to deliver its first sample

    # ---- headline: the fixed 1e6-point grid, split into `world` contiguous point ranges (strong scaling)
    total_points = N1 * N3
    lo, hi = balanced_range(total_points, world, rank)
    if args.shard_of > 1:       # profiling aid: rank 0's share of an N-way split, on this one GPU
        lo, hi = balanced_range(total_points, args.shard_of, 0)
    # the final gather: peer stores by the sweep kernel itself (default), or an NCCL all-gather after it
    peers, gather_how = None, "none (one GPU)"
    if world > 1:
        if args.gather == "peer":
            peers = PeerMaps.setup(fpa, dist, torch, world, rank, local, total_points)
        gather_how = ("kernel: NVLink peer stores into the full-size map of every GPU (fpa_sweep_desc.peer_gain)"
                      if peers is not None else "NCCL all_gather_into_tensor after the kernel")
    sweep = DeviceSweep(fpa, torch, dev, N1, lo, hi - lo, disp, pm_cfg, peer_maps=peers.ptrs if peers else None)
    B = hi - lo
    even = total_points % world == 0
    tall = -(-total_points // world)
    t_all = torch.empty(world * tall, dtype=torch.float64, device=dev) if world > 1 else None
    t_pad = torch.zeros(tall, dtype=torch.float64, device=dev) if (world > 1 and not even) else None

    def gather_strong():
        if world == 1 or peers is not None:
            return
        if even:
            dist.all_gather_into_tensor(t_all, sweep.t_gain)               # the final result gather
        else:
            t_pad[:B] = sweep.t_gain
            dist.all_gather_into_tensor(t_all, t_pad)

    ms_total, k_ms, window, parts = timed_sweeps(torch, dist, sweep, gather_strong, world, args.steps, args.warmup, t_flush, dev)
    clocks = sampler.summary(*window) if rank == 0 else None
    value = (hi - lo if args.shard_of > 1 else total_points) * n_steps * args.steps / (ms_total * 1e-3)
    kernel_ms = float(np.mean(k_ms))
    achieved_tf = FLOPS_PER_POINT_STEP * B * n_steps / (kernel_ms * 1e-3) / 1e12
    gain_dev = sweep.t_gain.cpu().numpy()
    if world > 1:       # every rank holds the gathered map; rank 0 later checks it against the assembled host map
        if peers is not None:   # untimed NCCL gather of the same results: the kernel-built map must equal it bit for bit
            if even:
                dist.all_gather_into_tensor(t_all, sweep.t_gain)
            else:
                t_pad[:B] = sweep.t_gain
                dist.all_gather_into_tensor(t_all, t_pad)
            torch.cuda.synchronize()
        shards = t_all.view(world, tall).cpu().numpy()
        sizes = [balanced_range(total_points, world, r) for r in range(world)]
        full_dev = np.concatenate([shards[r, :b - a] for r, (a, b) in enumerate(sizes)])
        if peers is not None:
            built = peers.own_map().cpu().numpy()
            assert built.tobytes() == full_dev.tobytes(), f"rank {rank}: the map built by peer stores differs from the NCCL gather"
            peers.close(dist)
    else:
        full_dev = gain_dev
    if args.dump_outputs and rank == 0:
        outputs = {"gain_lin": full_dev}
        if world == 1:      # the per-point outputs of a shard are not gathered at N > 1
            outputs.update(dbeta=sweep.t_dbeta.cpu().numpy(), valid=sweep.t_valid.cpu().numpy().astype(np.float32),
                           status=sweep.t_status.cpu().numpy().astype(np.float32))
        dump_outputs(args.dump_outputs, outputs)

    # ---- weak scaling alongside (N > 1): 1e6 points per GPU on a (1000 N) x 1000 grid
    weak = None
    if world > 1 and args.scaling in ("both", "weak"):
        wsweep = DeviceSweep(fpa, torch, dev, N1 * world, rank * N1 * N3, N1 * N3, disp, pm_cfg)
        w_all = torch.empty(world * N1 * N3, dtype=torch.float64, device=dev)
        w_ms, w_k, _, _ = timed_sweeps(torch, dist, wsweep, lambda: dist.all_gather_into_tensor(w_all, wsweep.t_gain),
                                    world, args.steps, args.warmup, t_flush, dev)
        weak = {"value": world * N1 * N3 * n_steps * args.steps / (w_ms * 1e-3), "unit": UNIT, "ms_per_step": w_ms / args.steps,
                "points_total": world * N1 * N3, "kernel_ms": float(np.mean(w_k)),
                "note": "1e6 points per GPU on a (1000 N) x 1000 grid + all-gather of the gain map"}
        del wsweep, w_all
        torch.cuda.empty_cache()

    # ---- e2e through the public call with HOST buffers
    lam1, lam3 = grid_axes()

    def public_call(rows, out=None, **kw):
        return fpa.scan_mismtach.sweep_gain_2d(
            cfg=cfg, lambda_p1_m=rows, lambda_p2_m=LAM_P2, lambda_signal_m=lam3, gamma=GAMMA, alpha=ALPHA,
            p_in=P_IN, dispersion=disp, phase_matching_cfg=pm_cfg, gain_unit="linear", device=local, out=out, **kw)

    def time_calls(fn, reps):
        res, res2 = fn(), fn()                      # warm: workspace, and two result sets in the page-locked pool
        del res, res2                               # (a caller rebinding `r = call()` holds two for a moment)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            res = fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()                          # every rank's shard has landed in the host array
        sec = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([sec], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sec = float(t.item())
        return sec, res

    e2e_steps = max(2, min(args.steps, 5))
    e2e_variants = {}
    if args.shard_of > 1:
        e2e_value, e2e_api, h2d, d2h = None, "not measured with --shard-of", 0, 0
    elif world == 1:
        sec_a, res = time_calls(lambda: public_call(lam1), e2e_steps)
        e2e_value = total_points * n_steps * e2e_steps / sec_a
        assert res["gain_lin"].tobytes() == full_dev.reshape(N1, N3).tobytes(), "e2e and device-resident sweeps differ"
        del res
        bufs = {k: L.pinned_empty((N1, N3), dt) for k, dt in
                (("gain_lin", np.float64), ("dbeta", np.float64), ("valid", np.int32), ("status", np.int32))}
        h_l1 = L.pinned_empty((N1,), np.float64)
        h_l1[:] = lam1
        sec_b, _ = time_calls(lambda: public_call(h_l1, out=bufs), e2e_steps)
        plain = {k: np.empty((N1, N3), v.dtype) for k, v in bufs.items()}
        sec_c, _ = time_calls(lambda: public_call(lam1, out=plain), e2e_steps)
        # the reference-NAMED call is one-dimensional (one pump pair per call, scan_mismtach.py:588-611):
        # a 2-D map through it is a Python loop over pump rows, each a 1 000-point launch (1.3 % of a wave)
        rows_1d = 24
        def named_rows():
            for i in range(rows_1d):
                x, g, db = fpa.scan_mismtach.plot_max_gain_and_dbeta_vs_lambda_signal(
                    cfg=cfg, lambda_p1_m=float(lam1[i * 40]), lambda_p2_m=LAM_P2, lambda_signal_m=lam3, gamma=GAMMA,
                    alpha=ALPHA, p_in=P_IN, dispersion=disp, phase_matching_cfg=pm_cfg, gain_unit="linear",
                    show=False, show_progress=False)
            return g
        sec_d, g_last = time_calls(named_rows, 1)
        assert g_last.tobytes() == full_dev.reshape(N1, N3)[(rows_1d - 1) * 40].tobytes()
        e2e_variants = {
            "default_buffers": {"value": e2e_value, "api": "sweep_gain_2d(...) with no out=: results land in the library's page-locked pool"},
            "pinned_out": {"value": total_points * n_steps * e2e_steps / sec_b, "api": "sweep_gain_2d(..., out=caller's page-locked arrays)"},
            "pageable_out": {"value": total_points * n_steps * e2e_steps / sec_c,
                             "api": "sweep_gain_2d(..., out=np.empty arrays): device staging + 4 pageable D2H copies"},
            "reference_named_1d_rows": {"value": rows_1d * N3 * n_steps / sec_d, "rows": rows_1d,
                                        "api": "plot_max_gain_and_dbeta_vs_lambda_signal per pump row (1 000 points per launch: "
                                               "latency-bound, the reference's own call shape)"},
        }
        e2e_api = ("scan_mismtach.sweep_gain_2d -> fpa_yaman4_sweep_host, default buffers: axes copied up, the kernel writes its "
                   "24 B per point straight into page-locked host result arrays owned by the library")
        h2d, d2h = (N1 + 1 + N3) * 8, total_points * 24
    else:
        # one assembled map in ONE host array: a shared-memory segment every rank page-locks; each rank's
        # kernel stores its pump rows straight into it
        from multiprocessing import shared_memory
        r_lo, r_hi = balanced_range(N1, world, rank)
        name = [None]
        shm = None
        if rank == 0:
            shm = shared_memory.SharedMemory(create=True, size=total_points * 24)
            name[0] = shm.name
        dist.broadcast_object_list(name, src=0)
        if rank != 0:
            shm = shared_memory.SharedMemory(name=name[0])
        seg = np.ndarray(total_points * 24, dtype=np.uint8, buffer=shm.buf)
        L.register_host(seg)
        full = {"gain_lin": np.ndarray((N1, N3), np.float64, shm.buf, 0),
                "dbeta": np.ndarray((N1, N3), np.float64, shm.buf, 8 * total_points),
                "valid": np.ndarray((N1, N3), np.int32, shm.buf, 16 * total_points),
                "status": np.ndarray((N1, N3), np.int32, shm.buf, 20 * total_points)}
        mine = {k: v[r_lo:r_hi] for k, v in full.items()}
        rows_mine = lam1[r_lo:r_hi].copy()
        sec_a, _ = time_calls(lambda: public_call(rows_mine, out=mine), e2e_steps)
        e2e_value = total_points * n_steps * e2e_steps / sec_a
        if rank == 0:
            assert full["gain_lin"].tobytes() == full_dev.tobytes(), "assembled host map and gathered device map differ"
        dist.barrier()
        L.unregister_host(seg)
        del full, mine, seg
        shm.close()
        if rank == 0:
            shm.unlink()
        e2e_api = ("every rank: scan_mismtach.sweep_gain_2d(its pump rows, out=its rows of ONE shared host map) -> fpa_yaman4_sweep_host; "
                   "the segment is page-locked by each rank (fpa_host_register), kernels store into it directly; timed to the last rank")
        h2d, d2h = (N1 + 1 + N3) * 8 + (world - 1) * (1 + N3) * 8, total_points * 24

    # ---- secondary configurations (N = 1)
    secondary, sec_window = None, None
    if world == 1 and not args.no_secondary and args.shard_of <= 1:
        peak_tf, _ = fpa._device.fp64_peak(iters=2048, device=local)
        t_a = time.time()
        secondary = run_secondary(fpa, torch, dev, local, disp, peak_tf, t_flush)
        sec_window = (t_a, time.time())

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- rank 0: FP64 peak probe, JSON line
    peak_tf, _ = fpa._device.fp64_peak(iters=2048, device=local)
    sm_count, khz = C.c_int(), C.c_int()
    name = C.create_string_buffer(128)
    lib.fpa_device_info(local, C.byref(sm_count), C.byref(khz), name, 128)
    nominal_tf = sm_count.value * 64 * 2 * khz.value * 1e3 / 1e12
    seg_on = os.environ.get("FPA_SWEEP_SEG", "1") != "0" and 148 * 16 <= (B + 31) // 32 < 8 * 148 * 16
    traffic, traffic_src = ncu_traffic_bytes(seg_on)
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD + (f" -- ONLY the first of {args.shard_of} shards (profiling aid)" if args.shard_of > 1 else ""),
                   "points_total": total_points, "points_per_gpu": B, "rk4_steps": n_steps,
                   "parallelism": f"flattened point range split x{world}; final gather: {gather_how}" if world > 1 else "one GPU",
                   "l2": f"{FLUSH_BYTES >> 20} MiB buffer written between steps (inside the timed region); "
                         "the kernel keeps its state in registers"},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": e2e_steps, "api": e2e_api, "variants": e2e_variants},
        "gpu_launches": args.steps,              # one sweep kernel per step on every rank
        "step_breakdown": {**parts, "note": "rank 0, CUDA events between the pieces of a step; gather_ms is the NCCL all-gather incl. "
                                            "waiting for the slowest rank (~0 when the sweep kernel gathers by peer stores); the "
                                            "rest of a step is launch gaps"},
        "clocks": clocks,
        "roofline": {"bound": "fp64_fma", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                     "frac": achieved_tf / peak_tf, "frac_of_nominal": achieved_tf / nominal_tf,
                     "traffic": traffic,
                     "traffic_unit": f"bytes per launch (dram read+write, ncu --set full, profiles/{traffic_src})",
                     "kernel": ("yaman4_sweep_seg_kernel<LOSS,128,4> (persistent, z-segment scheduler: plan + dbeta prologue, fused RK4 "
                                "z-loop, gain epilogue" if seg_on else "yaman4_sweep_kernel<LOSS,128,4> (plan + dbeta prologue, fused RK4 z-loop, gain epilogue") +
                               "; every launch of the timed region, CUDA events on the launching stream)",
                     "kernel_ms": kernel_ms, "library": lib.fpa_version().decode(),
                     "kernel_share_of_step": kernel_ms / (ms_total / args.steps),
                     "flops_per_point_step": FLOPS_PER_POINT_STEP, "points_per_launch": B,
                     "peak_source": "DFMA probe measured live on this GPU (fpa_fp64_peak_probe); "
                                    "MEASURED_PEAKS.json holds no FP64 figure",
                     "nominal_peak": nominal_tf,
                     "hbm_note": "reduce-mode sweep: 24 B per point per launch + scheduler state through L2, HBM is idle"},
        "device": name.value.decode(),
    }
    if weak is not None:
        out["weak"] = weak
    if cpu_leg is not None:
        cores, n_pts, cpu_value, wall, idx, cpu_gain, one_core, kind = cpu_leg
        gpu_gain = full_dev.reshape(-1)[idx]
        out["cpu_baseline"] = {
            "value": cpu_value, "unit": UNIT, "cores": cores, "value_1core": one_core, "kind": kind,
            "sample": f"{n_pts} random points (default_rng(0)) of the 1e6-point grid x {n_steps} steps, "
                      f"{wall:.1f} s wall; " + CPU_NOTE[kind],
            "parity_max_rel_err_vs_gpu": float(np.max(np.abs(gpu_gain - cpu_gain) / np.abs(cpu_gain))),
        }
    if secondary is not None:
        secondary["clocks"] = sampler.summary(*sec_window)
        out["secondary"] = secondary
    sampler.stop()
    print(json.dumps(out), file=RESULT_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------- secondary configurations
def run_secondary(fpa, torch, dev, local, disp4, peak_tf, t_flush) -> dict:
    """The other BASELINE configurations on one GPU, device-resident, CUDA events around each launch
    (median of 3 after one warm-up, L2 flushed before each).  `frac` = credited flops / measured FP64 peak."""
    L, lib = fpa._lib, fpa._lib.lib()
    nw, fp, ds = fpa.nwave, fpa.frequency_plan, fpa.dispersion
    res = {"peak_tflops": peak_tf}
    stream = lambda: torch.cuda.current_stream().cuda_stream      # noqa: E731

    def timed(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            t_flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return float(np.median(ts))

    def entry(points, steps, ms, flops_per_step, **extra):
        rate = points * steps / (ms * 1e-3)
        tf = flops_per_step * rate / 1e12
        return {"points": points, "steps": steps, "kernel_ms": ms, "point_steps_per_s": rate,
                "flops_per_point_step": flops_per_step, "tflops": tf, "frac": tf / peak_tf, **extra}

    def yaman_desc(B, dbeta, consts, z_max, n_steps, save_every, flags, trace=None, end=None, pmax=None, status=None):
        d = L.Yaman4Desc()
        d.n_points = B
        d.dbeta = dbeta.data_ptr()
        d.gamma, d.gamma_stride = consts.data_ptr(), 0
        d.alpha, d.alpha_stride = consts.data_ptr() + 8, 0
        d.A0, d.A0_stride = consts.data_ptr() + 16, 0
        d.z0, d.z_max, d.n_steps, d.save_every = 0.0, z_max, n_steps, save_every
        d.flags = flags | L.UNIFORM_PHYSICS
        d.gamma_uniform, d.alpha_uniform = float(consts[0]), float(consts[1])
        d.A_trace = trace.data_ptr() if trace is not None else None
        d.A_end = end.data_ptr() if end is not None else None
        d.Pmax = pmax.data_ptr() if pmax is not None else None
        d.status = status.data_ptr() if status is not None else None
        nb = int(lib.fpa_yaman4_scratch_bytes(B))
        scr = torch.empty(max(nb, 16), dtype=torch.uint8, device=dev)
        d.scratch, d.scratch_bytes = scr.data_ptr(), nb
        return d, scr

    # ---- config 1a: one run, 10 000 steps, full trace, through the reference-shaped host call
    om = fp.plan_from_wavelengths(1550e-9, 1560e-9, 1555e-9)
    sp = fp.infer_symmetry_from_omegas(*om)
    disp1 = ds.dispersion_params_from_D_S(fp.lambda_from_omega(sp.omega_c), 0.02, 0.02, 0.0, D_units="ps/nm/km",
                                          S_units="ps/nm^2/km", dSdlmbd_units="ps/nm^3/km", omega_ref=sp.omega_c)
    cfg1 = fpa.config.custom_simulation_config(z_max=1000.0, dz=0.1, save_every=10)
    alpha1 = float(np.log(10) / 10 * 0.9 / 1000)
    kw1 = dict(gamma=11.5e-3, alpha=alpha1, omega=om, p_in=[0.5, 0.5, 1e-5, 1e-5], dispersion=disp1)
    fpa.simulation.run_single_simulation(cfg1, **kw1)
    t0 = time.perf_counter()
    for _ in range(5):
        z, A = fpa.simulation.run_single_simulation(cfg1, **kw1)
    dt = (time.perf_counter() - t0) / 5
    res["config1a_single_run"] = entry(1, 10000, 1e3 * dt, FLOPS_PER_POINT_STEP, saved=int(z.size),
                                       note="wall time of run_single_simulation (B = 1: one thread, latency-bound; H2D/D2H included)")

    # ---- config 3: 1e5-point dbeta sweep, reduce mode (A_end + Pmax), short and long fiber
    B = 100_000
    dbeta = torch.linspace(-40.0, 40.0, B, dtype=torch.float64, device=dev) / 1000.0
    A0 = np.sqrt(np.array([0.1, 0.1, 1e-5, 0.0]))
    consts = torch.tensor([10.0 / 1000, 0.0] + [v for a in A0 for v in (a, 0.0)], dtype=torch.float64, device=dev)
    end = torch.empty(B * 8, dtype=torch.float64, device=dev)
    pmax = torch.empty(B * 4, dtype=torch.float64, device=dev)
    status = torch.empty(B, dtype=torch.int32, device=dev)
    for name, n_steps in (("config3_1e5x500", 500), ("config3_long_1e5x50000", 50000)):
        d, scr = yaman_desc(B, dbeta, consts, 500.0, n_steps, 10, L.OUT_END | L.OUT_PMAX | L.CHECK_NAN, end=end, pmax=pmax,
                            status=status)
        ms = timed(lambda: L.check(lib.fpa_yaman4_rk4_batch_dev(C.byref(d), stream())))
        res[name] = entry(B, n_steps, ms, FLOPS_LOSSLESS, waves=round(B / 32 / (148 * 16), 2),
                          note="alpha = 0: credited with the 504 flops per step the lossless kernel executes")
    del end, pmax

    # ---- trace-mode write-out: 2e5 points x 2 500 steps, every 10th and every step
    B = 200_000
    dbeta = torch.linspace(-0.015, 0.015, B, dtype=torch.float64, device=dev)
    A0 = np.sqrt(np.array(P_IN))
    consts = torch.tensor([GAMMA, ALPHA] + [v for a in A0 for v in (a, 0.0)], dtype=torch.float64, device=dev)
    status = torch.empty(B, dtype=torch.int32, device=dev)
    for save_every in (10, 1):
        n_saved = 2500 // save_every + 1
        trace = torch.empty(B * n_saved * 8, dtype=torch.float64, device=dev)
        d, scr = yaman_desc(B, dbeta, consts, 500.0, 2500, save_every, L.OUT_TRACE | L.CHECK_NAN, trace=trace, status=status)
        ms = timed(lambda: L.check(lib.fpa_yaman4_rk4_batch_dev(C.byref(d), stream())))
        res[f"trace_save_every_{save_every}"] = entry(B, 2500, ms, FLOPS_PER_POINT_STEP, n_saved=n_saved,
                                                      trace_bytes=B * n_saved * 64,
                                                      hbm_write_GBps=B * n_saved * 64 / (ms * 1e-3) / 1e9)
        del trace, d, scr
        torch.cuda.empty_cache()

    # ---- config 4 with GENERAL_TAYLOR (max_order 4) instead of SYMMETRIC_EVEN
    pm_gt = fpa.phase_matching.PhaseMatchingConfig(method=fpa.phase_matching.PhaseMatchingMethod.GENERAL_TAYLOR, max_order=4)
    sw = DeviceSweep(fpa, torch, dev, N1, 0, N1 * N3, disp4, pm_gt)
    ms = timed(lambda: sw.launch(stream()))
    res["config4_general_taylor"] = entry(N1 * N3, 2500, ms, FLOPS_PER_POINT_STEP,
                                          nan_points=int(torch.isnan(sw.t_gain).sum().item()))
    del sw

    # ---- N-wave descriptors (device-resident)
    def nwave_dev(plan, beta, A0n, gamma, alpha, z_max, n_steps, save_every, form, trace):
        Bn, N = A0n.shape
        t_beta = torch.from_numpy(np.ascontiguousarray(beta, dtype=np.float64)).to(dev)
        t_ga = torch.tensor([gamma, alpha], dtype=torch.float64, device=dev)
        t_A0 = torch.from_numpy(np.ascontiguousarray(A0n).view(np.float64)).to(dev)
        n_saved = n_steps // save_every + 1
        t_out = torch.empty(Bn * (n_saved if trace else 1) * N * 2, dtype=torch.float64, device=dev)
        t_st = torch.empty(Bn, dtype=torch.int32, device=dev)
        keep = [t_beta, t_ga, t_A0, t_out, t_st]
        d = L.NwaveDesc()
        d.n_points, d.n_waves = Bn, N
        d.beta, d.beta_stride = t_beta.data_ptr(), 0
        d.gamma, d.gamma_stride = t_ga.data_ptr(), 0
        d.alpha, d.alpha_stride = t_ga.data_ptr() + 8, 0
        d.A0, d.A0_stride = t_A0.data_ptr(), 1
        d.z0, d.z_max, d.n_steps, d.save_every = 0.0, z_max, n_steps, save_every
        d.flags = (L.OUT_TRACE if trace else L.OUT_END) | L.CHECK_NAN | (L.NWAVE_TABLE if form in ("table", "entries") else 0)
        if trace:
            d.A_trace = t_out.data_ptr()
        else:
            d.A_end = t_out.data_ptr()
        d.status = t_st.data_ptr()
        if form in ("table", "entries"):
            t_tab = torch.from_numpy(plan.table.view(np.int16).copy()).to(dev)
            t_rows = torch.from_numpy(plan.row_ptr.copy()).to(dev)
            keep += [t_tab, t_rows]
            d.triplets, d.row_ptr, d.n_triplets = t_tab.data_ptr(), t_rows.data_ptr(), plan.n_triplets
            if form == "table":     # the table kernel integrates from the factored table; "entries": the entry list
                blob, n_classes = fpa._device.factor_table(N, plan.table, plan.row_ptr)
                t_blob = torch.from_numpy(blob).to(dev)
                keep.append(t_blob)
                d.factored, d.n_classes = t_blob.data_ptr(), n_classes
            else:
                d.flags |= L.NWAVE_PLAIN
        else:
            g = plan.grid_index.astype(np.int64)
            t_slot = torch.from_numpy((g - g.min()).astype(np.int32)).to(dev)
            keep.append(t_slot)
            d.grid_slot, d.grid_span = t_slot.data_ptr(), int(g.max() - g.min() + 1)
        return d, keep

    # ---- config 2: N = 21 dual-pump plan, single run, 10 000 steps, full trace
    plan21 = nw.uniform_comb_plan(sp.omega_c, sp.omega_d / 5.0, range(-10, 11))
    beta21 = nw.beta_per_wave(plan21, disp1)
    p21 = np.zeros(21)
    p21[[5, 15]] = 0.5
    p21[[9, 11]] = 1e-5
    for form in ("comb", "table"):
        d, keep = nwave_dev(plan21, beta21, np.sqrt(p21).astype(np.complex128).reshape(1, 21), 11.5e-3, alpha1, 1000.0, 10000,
                            10, form, True)
        ms = timed(lambda: L.check(lib.fpa_nwave_rk4_batch_dev(C.byref(d), stream())), reps=3)
        res[f"config2_n21_single_run_{form}"] = entry(1, 10000, ms, plan21.flops_per_step(form), waves=21,
                                                      note="N > 4: oracle parity unpinned (no reference exists)")

    # ---- config 5: N = 64 comb, 1e5 z-steps, B = 1 and B = 1024 (pump power linspace 0.1 .. 1 W)
    w0 = 2 * np.pi * 299792458.0 / 1550e-9
    plan64 = nw.uniform_comb_plan(w0, 2 * np.pi * 100e9, range(-32, 32))
    disp64 = ds.DispersionParams(omega_ref=w0, beta2=-2.57e-29, beta3=3.30e-41, beta4=-1.63e-55)
    beta64 = nw.beta_per_wave(plan64, disp64)
    phases = np.random.default_rng(0).uniform(0, 2 * np.pi, 64)

    def comb_A0(Bn):
        A0n = np.empty((Bn, 64), dtype=complex)
        for b, pw in enumerate(np.linspace(0.1, 1.0, Bn)):
            p = np.full(64, 1e-12)
            p[33] = 1e-6
            p[[28, 36]] = pw
            A0n[b] = np.sqrt(p) * np.exp(1j * phases)
        return A0n

    for Bn, form, steps in ((1, "comb", 100_000), (1024, "comb", 100_000), (148, "table", 2_000), (148, "entries", 400)):
        d, keep = nwave_dev(plan64, beta64, comb_A0(Bn), 11.5e-3, 2e-4, 1e4 * steps / 1e5, steps, 100, form, False)
        ms = timed(lambda: L.check(lib.fpa_nwave_rk4_batch_dev(C.byref(d), stream())), reps=1 if steps > 10_000 else 3)
        res[f"config5_n64_B{Bn}_{form}"] = entry(Bn, steps, ms, plan64.flops_per_step(form), waves=64,
                                                 note="N > 4: oracle parity unpinned (no reference exists)" +
                                                      ("" if steps == 100_000 else f"; {steps} of the 1e5 steps (rate is constant in z)"))
    return res


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scaling", default="both", choices=["both", "strong", "weak"],
                    help="N > 1: the headline is always strong scaling (the fixed 1e6-point grid split over the ranks); "
                         "'both' (default) and 'weak' also time 1e6 points per GPU and report it under \"weak\"")
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"],
                    help="N > 1: how the gain map is gathered -- by the sweep kernel (peer stores over NVLink, default) "
                         "or by an NCCL all-gather after it")
    ap.add_argument("--no-cpu-baseline", action="store_true",
                    help="skip the CPU leg (profiling runs under ncu)")
    ap.add_argument("--shard-of", type=int, default=1,
                    help="profiling aid (one GPU): run only rank 0's share of an N-way split of the grid, e.g. 8 -> 125 000 points")
    ap.add_argument("--no-secondary", action="store_true",
                    help="skip the secondary configurations (profiling runs under ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed sweep computed as DIR/<name>.npy (24 MB at N = 1): gain_lin and "
                         "dbeta in float64, valid and status in float32; at N > 1 rank 0 writes the gathered gain_lin map")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    # stdout carries ONE JSON line.  Anything else written to file descriptor 1 -- NCCL prints its
    # version banner there with NCCL_DEBUG >= VERSION, libraries may print -- is sent to stderr; the
    # result line goes to a duplicate of the original stdout.
    global RESULT_OUT
    sys.stdout.flush()
    RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
