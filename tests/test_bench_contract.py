"""bench.py on a machine without a GPU: the reference arm (the CPU oracle, the one place besides tests/ and smoke() that
may execute oracle/) prints one JSON line with the contract's keys; the product arm refuses to run (no CPU fallback);
workloads load."""
import json
import os
import subprocess
import sys

import pytest

from turbo_b200 import engine

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--workload", "simplified:accap_a3"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "propagations/sec" and d["unit"] == "propagations/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["nodes_per_sec"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload_arg"] == "simplified:accap_a3" and "benchmarks/accap_a3.fzn" in d["config"]["workload"]


def check_dump(out_dir, workload):
    """The files --dump-outputs writes, checked against the network: an assigned store at the network's fixpoint."""
    import numpy as np
    from oracle import oracle_py as orc
    from tests import golden_io
    out = {p.stem: np.load(p) for p in out_dir.glob("*.npy")}
    assert set(out) == {"lb", "ub", "has_solution", "exhaustive", "objective"}
    assert all(a.dtype == np.float64 for a in out.values())
    pb, info = golden_io.load_simplified_problem(workload)
    assert out["lb"].shape == out["ub"].shape == (pb.nvars,) and out["has_solution"] == 1
    assert np.array_equal(out["lb"], out["ub"]) and out["objective"] == out["lb"][pb.obj_var]
    lb, ub = out["lb"].astype(np.int32), out["ub"].astype(np.int32)
    r = orc.fixpoint(pb, lb, ub)
    assert not r["failed"] and np.array_equal(r["lb"], lb) and np.array_equal(r["ub"], ub)
    return golden_io.user_objective(info, lb, ub)


def test_reference_arm_dumps_its_last_step(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "0",
                        "--workload", "simplified:accap_a3", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert json.loads(r.stdout)["steps"] == 2
    check_dump(tmp_path, "accap_a3")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert r.returncode != 0 and "--steps" in r.stderr


@pytest.mark.gpu
def test_product_arm_dumps_its_last_step(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--workload", "simplified:accap_a3",
                        "--no-cpu-baseline", "--no-fixpoint-leg", "--strong-ms", "0", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    d = json.loads(r.stdout)
    assert d["steps"] == 2 and d["e2e"]["steps"] == 2
    assert check_dump(tmp_path, "accap_a3") == d["best_objective"]


def test_a_large_store_is_dumped_as_a_fixed_sample(tmp_path):
    """More variables than 64 MB of float64 holds: the same seeded sample of variables every time, its indices beside it."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    n = 5_000_000
    pb = type("Problem", (), {"obj_var": 7})
    res = dict(lb=np.arange(n, dtype=np.int32), ub=np.arange(n, dtype=np.int32) + 1, has_solution=True, exhaustive=False)
    bench.dump_outputs(str(tmp_path / "a"), pb, res)
    bench.dump_outputs(str(tmp_path / "b"), pb, res)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["exhaustive.npy", "has_solution.npy", "lb.npy", "objective.npy", "ub.npy", "var_index.npy"]
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= bench.DUMP_BUDGET_BYTES
    idx = np.load(tmp_path / "a" / "var_index.npy")
    assert np.array_equal(idx, np.load(tmp_path / "b" / "var_index.npy"))
    assert 0 < len(idx) < n and np.all(np.diff(idx) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "lb.npy"), idx) and np.array_equal(np.load(tmp_path / "a" / "ub.npy"), idx + 1)
    assert np.load(tmp_path / "a" / "objective.npy") == 7


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.skipif(engine.device_count() > 0, reason="a GPU is present")
def test_product_arm_has_no_cpu_fallback():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_workloads_load():
    sys.path.insert(0, ROOT)
    import bench
    pb, info = bench.load_workload("simplified:trains15")
    full, _ = bench.load_workload("trains15")
    assert 0 < pb.nvars < full.nvars and 0 < pb.nprops < full.nprops and info["objective_kind"] == 0
    assert "simplifier" in bench.data_description("simplified:trains15") and "disable_simplify" in bench.data_description("trains15")
