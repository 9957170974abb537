"""GPU: every N-wave kernel form line by line against the long-double march (oracle/nwave_oracle.py::march_ld), down
to cascaded sidebands 40 decades below the pumps.

The plans (a)-(d) and the seeds are those of tests/test_nwave_lines_cpu.py, chosen so that each instantiation of the
batch comb kernel runs: span 21 (generic reduce-scatter), 64 (PLOG 2), 127 (PLOG 1), 192 (generic, beyond 128).
Plans (a) and (d) hold lines that stay exactly 0 for the whole run; the comb kernels still multiply across the whole
span, so those lines check the padding and the empty slots bit for bit.

Forms: `comb` at B = 1 (nwave_comb_kernel, a CTA per point) and at B = 4 SM + 1 (nwave_comb8_kernel, warp per point,
last CTA partly filled); `table` (factored table; a different number of threads per point at the two sizes) at both;
`entries` at B = 1 where N <= 48.  A batch gives its points different pump phases; points 0, middle and last are
checked.  40 steps of 0.1 m, every step saved, and plan (a) over 2 000 steps.

On every saved sample, A_end and Pmax, line by line: |got - ref| / |ref| <= 1e-11 wherever |ref| >= 1e-100 (Pmax:
against the reference's max of |A|^2 over the saved samples, where that is >= 1e-200), got == 0 exactly where
ref == 0, got != 0 wherever |ref| >= 1e-100, status -1 for every point.  The FP64 oracle meets this per line to
8e-14 (the CPU file), so 1e-11 leaves two decades for the kernels' own summation orders.

Measured on an NVIDIA B200 (1 000 W power limit), largest per-line error over the checked points: plan (a) comb 1.1e-14,
table 3.2e-15, entries 2.1e-15, 2 000 steps 5.9e-14; plan (b) comb 8.2e-14, table 3.6e-14; plan (c) comb 1.5e-13,
table 4.1e-14; plan (d) comb 4.4e-14, table 7.4e-15, entries 4.4e-15.  Weakest lines checked: 5.5e-24 W (a), 2.0e-55 W
(b), 2.2e-55 W (c), 8.0e-45 W (d), all in the first steps of the cascade."""
import ctypes as C

import numpy as np
import pytest

from oracle import nwave_oracle as O
from test_nwave_lines_cpu import DZ, N_STEPS, ZERO_LINES, assert_lines, plan_case, table_list

pytestmark = pytest.mark.gpu

TOL = 1e-11
FORMS = [("comb", "one"), ("comb", "batch"), ("table", "one"), ("table", "batch"), ("entries", "one")]
# the entry list only where N <= 48: at N = 64 one run of it takes minutes
CASES = [(name, form, size) for name in "abcd" for form, size in FORMS if form != "entries" or name in "ad"]


@pytest.fixture(scope="module")
def sm4(gpu):
    """The batch (warp-per-point) kernel threshold: 4 x the SM count of the device the tests run on."""
    L = gpu._lib
    n, khz = C.c_int(), C.c_int()
    name = C.create_string_buffer(128)
    L.check(L.lib().fpa_device_info(L.get_device(), C.byref(n), C.byref(khz), name, 128))
    assert n.value > 0
    return 4 * n.value


def _pump_phases(plan, A0, b, B):
    """Point b of a batch: line j of A0 turned by phi + g_j * theta (g_j its grid index), phi and theta growing with b
    (point 0: A0 itself).  k + l - m = n on the grid, so this maps the run of A0 onto an exactly rotated one: the
    pumps of the points have different phases, the conditioning of every line stays that of point 0.  (Turning the
    pumps alone changes the physics; a line that then passes near 0 has no per-line accuracy to check: with the pumps
    of plan (b) turned by 2 pi and -1.4 pi, the FP64 oracle itself misses the long-double march by 2.3e-11 there.)"""
    t = b / B
    return A0 * np.exp(1j * (2 * np.pi * t + 0.9 * t * plan.grid_index))


class _Refs:
    """Long-double references, each computed once per module: (plan, point) -> states after every saved step."""

    def __init__(self, gpu, golden):
        self.gpu, self.golden, self.cases, self.runs = gpu, golden, {}, {}

    def case(self, name):
        if name not in self.cases:
            self.cases[name] = plan_case(self.gpu, self.golden, name)
        return self.cases[name]

    def ref(self, name, A0, n_steps=N_STEPS, save_every=1):
        key = (name, A0.tobytes(), n_steps, save_every)
        if key not in self.runs:
            plan, beta, _, gamma, alpha = self.case(name)
            tab, rows = table_list(plan)
            self.runs[key] = O.march_ld(A0, gamma, alpha, beta, tab, rows, z_max=n_steps * DZ, n_steps=n_steps,
                                        save_every=save_every)[1]
        return self.runs[key]


@pytest.fixture(scope="module")
def refs(gpu, golden):
    return _Refs(gpu, golden)


def _run(gpu, plan, beta, gamma, alpha, A0, form, n_steps=N_STEPS, save_every=1):
    cfg = gpu.config.custom_simulation_config(z_max=n_steps * DZ, dz=DZ, save_every=save_every)
    return gpu.nwave.run_nwave_simulation(cfg, plan, gamma=gamma, alpha=alpha, A0=A0, beta=beta,
                                          outputs=("trace", "end", "pmax"), form=form)


def _check_point(r, b, ref, what):
    """Point b of a run (trace, A_end, Pmax) against the long-double states `ref` [n_saved, N], line by line."""
    e_tr, w_tr = assert_lines(r["A_trace"][b], ref, TOL, what + " trace")
    e_end, _ = assert_lines(r["A_end"][b], ref[-1], TOL, what + " A_end")
    P_ref = (ref.real * ref.real + ref.imag * ref.imag).max(axis=0)
    e_pm, _ = assert_lines(r["Pmax"][b], P_ref, TOL, what + " Pmax", floor=1e-200)
    return max(e_tr, e_end, e_pm), w_tr


@pytest.mark.parametrize("name, form, size", CASES, ids=[f"{n}-{f}-{s}" for n, f, s in CASES])
def test_every_line_vs_long_double(gpu, refs, sm4, name, form, size):
    plan, beta, A0, gamma, alpha = refs.case(name)
    N = plan.n_waves
    assert plan.grid_span == {"a": 21, "b": 64, "c": 127, "d": 192}[name]
    B = 1 if size == "one" else sm4 + 1
    batch = np.array([_pump_phases(plan, A0, b, B) for b in range(B)])
    r = _run(gpu, plan, beta, gamma, alpha, batch, form)
    assert r["A_trace"].shape == (B, N_STEPS + 1, N) and (r["status"] == -1).all()
    worst, weakest = 0.0, np.inf
    for b in sorted({0, B // 2, B - 1}):
        ref = refs.ref(name, batch[b])
        if name in ZERO_LINES:        # the case keeps its exact zeros (the checks then demand them of the kernel)
            assert (ref[:, ZERO_LINES[name]] == 0).all()
        e, w = _check_point(r, b, ref, f"plan ({name}) {form} B={B} point {b}")
        worst, weakest = max(worst, e), min(weakest, w)
    print(f"\nplan ({name}) N={N} span={plan.grid_span} {form:7s} B={B:4d}: largest per-line error {worst:.1e}, "
          f"weakest line checked |A| = {weakest:.1e} ({weakest ** 2:.1e} W)")


@pytest.mark.parametrize("form", ["comb", "table"])
def test_plan_a_long_run_every_line(gpu, refs, form):
    """Plan (a) over 2 000 steps (z = 200 m), every 10th state: the odd lines span 3e-11 .. 0.48 W at the end, the
    11 even ones are still exactly 0."""
    plan, beta, A0, gamma, alpha = refs.case("a")
    ref = refs.ref("a", A0, n_steps=2000, save_every=10)
    assert ref.shape == (201, 21) and (ref[:, ZERO_LINES["a"]] == 0).all() and (ref[1:, 1::2] != 0).all()
    r = _run(gpu, plan, beta, gamma, alpha, A0[None, :], form, n_steps=2000, save_every=10)
    assert (r["status"] == -1).all()
    worst, weakest = _check_point(r, 0, ref, f"plan (a) 2000 steps {form}")
    print(f"\nplan (a) 2000 steps {form:7s} B=   1: largest per-line error {worst:.1e}, "
          f"weakest line checked |A| = {weakest:.1e} ({weakest ** 2:.1e} W)")
