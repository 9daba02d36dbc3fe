"""bench.py pieces that can be checked without a GPU: the synthetic problem of the measured arm is built
by the product's own host code (no oracle on that path) and equals what the oracle's builder gives, and
the reference arm prints the contract's JSON line."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_problem_inputs_match_oracle_builder():
    sys.path.insert(0, ROOT)
    import bench
    from oracle.api import create_plume_bcs
    batch, mconf, model = bench.make_problem(32)
    ref = {k: batch[k].copy() for k in ("pDiv", "UDiv", "flags", "density")}
    create_plume_bcs(ref, [1.0], 32 / 128.0, 0.15)
    for k in ("UBC", "UBCInvMask", "densityBC", "densityBCInvMask"):
        assert np.array_equal(batch[k], ref[k]), k
    assert mconf["simMethod"] == "convnet" and model["is3D"] is True


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--grid", "32",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
    d = json.loads(line)
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port")


def test_dump_outputs_float32_and_a_fixed_sample_above_the_limit(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    a = np.arange(3000, dtype=np.float64).reshape(3, 10, 100)
    bench.dump_outputs(str(tmp_path / "full"), {"U": a})
    got = np.load(tmp_path / "full" / "U.npy")
    assert got.dtype == np.float32 and np.array_equal(got, a.astype(np.float32))
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 4000)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), {"U": a, "p": a[0]})
    s1 = {k: np.load(tmp_path / "s1" / (k + ".npy")) for k in ("U", "p")}
    assert s1["U"].size == 750 and s1["p"].size == 250          # each array's share of the 4000 bytes
    for k, v in s1.items():
        assert np.array_equal(v, np.load(tmp_path / "s2" / (k + ".npy")))
        assert np.all(np.diff(v) >= 0) and np.isin(v, a).all()


def test_roofline_traffic_is_read_from_the_tracked_ncu_table():
    """bench.py's roofline.traffic comes from profiles/r02_advect_ncu_raw.csv (the ncu --set full capture of the
    current advection kernels), never from a literal: the parser finds the kernel and gives DRAM bytes per launch."""
    sys.path.insert(0, ROOT)
    import bench
    traffic, src = bench.ncu_traffic([r"k_advect_vel_tile"])
    assert src == os.path.join("profiles", "r02_advect_ncu_raw.csv")
    assert 5e6 < traffic < 2e8, traffic           # bytes per launch at 128^3 (algorithmic: 58.7 MB)
    assert bench.ncu_traffic([r"no_such_kernel"]) == (None, None)
