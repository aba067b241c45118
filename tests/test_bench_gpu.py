"""bench.py contract, GPU side: --steps sets the number of timed steps, and --dump-outputs writes what the timed
kernel computed in the last of them."""
import json
import os
import subprocess
import sys

import pytest

from test_bench_cpu import ROOT, check_dump

pytestmark = pytest.mark.gpu


def test_dump_outputs_are_the_last_timed_step(tmp_path):
    import bench
    import quadruped_landing_b200 as ql
    steps = 7                                        # the last step evaluates input set 2, not the first one
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1",
                        "--no-extras", "--no-cpu", "--dump-outputs", str(tmp_path)], capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads(r.stdout)
    assert d["steps"] == steps and d["gpu_launches"] == steps
    Z = bench.make_inputs(ql.default_problem(), 0, bench.N_INPUT_SETS)[(steps - 1) % bench.N_INPUT_SETS]
    check_dump(tmp_path, Z, exact=False)
