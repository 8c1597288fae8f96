"""CPU checks of bench.py's contract: the reference arm's JSON line (it runs without a GPU: the unmodified reference from
oracle/_ref, or the oracle port where that install is absent), the workload table, and the synthetic field generator."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "theta_rh_era5_f64", "--steps", "2",
                        "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "thermo grid-points/s" and line["unit"] == "grid-points/s"
    assert line["higher_is_better"] is True and line["steps"] == 2 and line["warmup"] == 1 and line["vs_baseline"] is None
    assert line["dtype"] == "f64" and line["config"]["workload"] == "theta_rh_era5_f64" and line["gpu_launches"] == 0
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == line["value"] > 0 and "sample" in cb
    assert line["e2e"] == {"value": line["value"], "unit": "grid-points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    if cb["kind"] == "reference":  # the installed reference passed its own thermo tests before it was timed
        assert line["reference_tests"].startswith("92 passed")


def test_other_ranks_of_the_reference_arm_exit_without_work():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"], capture_output=True,
                       text=True, timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_writes_all_points_or_a_fixed_sample(tmp_path, monkeypatch):
    import bench

    n = 50_000
    out = {"theta": torch.arange(n, dtype=torch.float64), "rh": -torch.arange(n, dtype=torch.float32)}
    bench.dump_outputs(str(tmp_path / "all"), out)
    assert np.array_equal(np.load(tmp_path / "all" / "theta.npy"), out["theta"].numpy())
    assert np.load(tmp_path / "all" / "rh.npy").dtype == np.float32
    monkeypatch.setattr(bench, "DUMP_BYTES", (64 << 10) + 8 * 2 * 1000)  # room for 1000 points of each output
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), out)
    theta, rh = np.load(tmp_path / "a" / "theta.npy"), np.load(tmp_path / "a" / "rh.npy")
    assert theta.size == rh.size == 1000 and theta.dtype == np.float64 and rh.dtype == np.float32
    assert np.all(np.diff(theta) > 0) and np.array_equal(rh, -theta.astype(np.float32))  # distinct points, the same for every output
    assert np.array_equal(np.load(tmp_path / "b" / "theta.npy"), theta)  # and the same from run to run


def test_workload_table_and_generator():
    import bench
    from synthetic import IfsField, sample_levels

    assert bench.DEFAULT_WORKLOAD == "suite_tqp_o1280x137_f64"
    wl = bench.WORKLOADS[bench.DEFAULT_WORKLOAD]
    assert wl["levels"] * wl["npl"] == 904_156_160 and wl["outputs"] == ("theta", "es", "rh", "td", "tv") and wl["dtype"] == "f64"
    assert bench.WORKLOADS["conv_ens_o640_f64"]["slabs"] == 51 * 137 and bench.WORKLOADS["conv_ens_o640_f64"]["sharded"]
    assert sample_levels(137, 8) == [8, 25, 42, 59, 77, 94, 111, 128] and sample_levels(1, 8) == [0]
    # every slab is reproducible on its own (its own seed), whatever was generated before it
    f1, f2 = IfsField("tqp", 1000, levels=137, seed=3), IfsField("tqp", 1000, levels=137, seed=3)
    a = [x.clone() for x in f1.slab(140)]  # member 1, level 3
    f2.slab(5), f2.slab(300)
    b = f2.slab(140)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    t, q, p = f1.slab(136)  # the lowest level: physical values, q below saturation
    assert 2.0e4 < float(p.min()) and float(p.max()) < 1.06e5 and 180.0 <= float(t.min()) and float(t.max()) <= 320.0 and float(q.min()) > 0
    t, q, p = f1.slab(0)  # the top level: about 1 Pa
    assert float(p.max()) < 3.0
    hy = IfsField("hybrid", 1000, levels=20, seed=3)
    assert hy.A_half.size == 21 and np.isclose(float(hy.slab(19)[2].mean()), float((hy.A_half[19:].mean() + hy.B_half[19:].mean() * hy.sp(0)).mean()), rtol=1e-12)
