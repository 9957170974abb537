"""CPU: the host-side pieces of bench.py that need no device -- the point partition of the strong-scaling arm,
the roofline bookkeeping read from profiles/, and the reference arm (`--impl reference`), which must keep
producing its JSON line (the byte-compiled reference when oracle/_ref exists, else the oracle port)."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402


def test_balanced_range_partitions_the_grid():
    for n, world in ((1_000_000, 8), (1_000_000, 3), (7, 8), (1000, 1)):
        parts = [bench.balanced_range(n, world, r) for r in range(world)]
        assert parts[0][0] == 0 and parts[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(parts, parts[1:]))
        sizes = [b - a for a, b in parts]
        assert max(sizes) - min(sizes) <= 1


def test_roofline_traffic_comes_from_committed_ncu_summaries():
    whole, src = bench.ncu_traffic_bytes(False)
    seg, src_seg = bench.ncu_traffic_bytes(True)
    assert src and "sweep_kernel" in src and whole is not None and 0 < whole < 1e7        # the whole-run kernel: ~0.2 MB
    assert src_seg and "seg_kernel" in src_seg and seg is not None and seg > whole        # scheduler state hand-over
    assert (ROOT / "profiles" / src).exists() and (ROOT / "profiles" / src_seg).exists()


def test_reference_arm_prints_one_json_line(tmp_path):
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--dump-outputs", str(tmp_path / "out")], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == bench.UNIT and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    gain, idx = np.load(tmp_path / "out" / "gain_lin.npy"), np.load(tmp_path / "out" / "point_index.npy")
    n = d["config"]["points_per_step"]
    assert gain.shape == idx.shape == (n,) and gain.dtype == idx.dtype == np.float64 and np.all(gain > 0)
    assert np.array_equal(idx, np.random.default_rng(0).choice(bench.N1 * bench.N3, size=n, replace=False))
