"""bench.py --dump-outputs: the headline run writes what its last timed step computed, within 64 MB, for a seeded sample
of the 4096 instances, and --steps sets the number of timed steps of every timed loop."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from cvxpylayers_b200 import problems as pr
from oracle import np_ref

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dumps_the_outputs_of_its_last_timed_step(cuda_device, tmp_path):
    out = tmp_path / "outputs"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--cpu-sample", "0",
                        "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-800:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["steps"] == 2 and d["e2e"]["pageable_inputs"]["steps"] == 2
    files = sorted(os.listdir(out))
    assert files == sorted(f"{k}.npy" for k in ("instances", "x", "y", "s", "status", "grad_A_eval", "grad_q_eval", "grad_P_eval"))
    assert sum(os.path.getsize(out / f) for f in files) <= 64 * 10**6
    z = {f[:-4]: np.load(out / f) for f in files}
    assert all(v.dtype == np.float64 for v in z.values())
    idx = z["instances"].astype(np.int64)
    k = idx.size
    assert 0 < k < 4096 and np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < 4096
    bt = pr.CONFIGS["C2"](B=4096, seed=0)   # bench.py's workload on a single GPU
    st = bt.structure
    assert z["x"].shape == (k, st.n) and z["y"].shape == (k, st.m) and z["s"].shape == (k, st.m)
    assert z["grad_A_eval"].shape == (st.nnzA + st.m, k) and z["grad_q_eval"].shape == (st.n + 1, k)
    assert z["grad_P_eval"].shape == (st.nnzP, k)
    assert (z["status"] == 1).all() and (z["grad_q_eval"][-1] == 0).all()
    assert np.isfinite(z["grad_A_eval"]).all() and np.abs(z["grad_A_eval"]).max() > 0
    eps = d["config"]["solver_args"]["eps"]
    for j in range(0, k, max(1, k // 16)):
        i = idx[j]
        res = np_ref.kkt_residuals(bt.A_dense(i), bt.P_dense(i), bt.b[i], bt.c[i], z["x"][j], z["y"][j], z["s"][j])
        assert np_ref.is_converged(res, eps, eps, 1.001), (i, res)
