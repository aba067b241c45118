"""bench.py contract, CPU side: the reference arm prints exactly one JSON line with the agreed keys."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, OMP_NUM_THREADS="1")          # what torchrun exports; the arm must not honour it
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "batched NLP evals/s (g+sparse Jacobian)" and d["unit"] == "evals/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] == d["value"] > 0
    assert d["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0))
    assert d["e2e"] == {"value": d["value"], "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["gpu_launches"] == 0


def check_dump(path, Z, exact):
    """DIR holds f of the whole batch Z and grad / g / jac of the rows listed in rows.npy, as the oracle computes them
    (bit for bit when `exact`, else within the fp64 parity tolerance), in float64 files of at most 64 MB together."""
    import numpy as np
    from conftest import assert_parity
    from oracle.oracle import Oracle
    import quadruped_landing_b200 as ql
    files = sorted(os.listdir(path))
    assert files == ["f.npy", "g.npy", "grad.npy", "jac.npy", "rows.npy"]
    assert sum(os.path.getsize(os.path.join(path, f)) for f in files) <= 64 << 20
    got = {f[:-4]: np.load(os.path.join(path, f)) for f in files}
    assert all(v.dtype == np.float64 for v in got.values())
    rows = got.pop("rows").astype(np.int64)
    assert len(np.unique(rows)) == len(rows) == 128 and rows.min() >= 0 and rows.max() < Z.shape[0]
    o = Oracle(ql.default_problem())
    ref = o.eval_batch(Z[rows])
    ref["f"] = o.eval_batch(Z, want=("f",))["f"]
    for k, v in got.items():
        if exact:
            assert np.array_equal(v, ref[k]), k
        else:
            assert_parity(v, ref[k], k)


def test_reference_arm_dumps_its_last_step(tmp_path):
    import bench
    import quadruped_landing_b200 as ql
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "0",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout)["steps"] == 2
    check_dump(tmp_path, bench.make_inputs(ql.default_problem(), 0, 1)[0], exact=True)


def test_other_ranks_of_the_reference_arm_exit_silently():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                       capture_output=True, text=True, env=env, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""
