"""`bench.py --dump-outputs`: what the last timed headline step returned, written as float64 .npy files, equals the
oracle's predict+grad over the same seeded rows and model."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench            # noqa: E402
from oracle.oracle import CSR  # noqa: E402
from helpers import max_rel  # noqa: E402

pytestmark = pytest.mark.gpu


def test_dump_outputs_are_the_timed_step(oracle, tmp_path):
    n, out = 20_000, tmp_path / "outputs"
    skip = "det,e2e,c4_adagrad,c3,c5,cd,seq,uniform"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--rows", str(n), "--steps", "2", "--warmup", "3",
                        "--no-cpu-baseline", "--skip", skip, "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.strip()][-1])
    assert line["steps"] == 2
    got = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert set(got) == {"loss_sum", "grad_intercept", "grad_w", "grad_P_sampled", "grad_P_sampled_features"}
    assert all(a.dtype == np.float64 for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    assert got["loss_sum"][0] == line["loss_sum"]

    data, indices, indptr, y = bench.gen_criteo_rows(n, 1000)
    P, w, b = bench.model_params(7)
    ref = oracle.fm_loss_grad(CSR(data, indices, indptr, n, bench.D_FEATURES), y, P, w, b, bench.DEGREE, "logistic")
    feats = got["grad_P_sampled_features"].astype(np.int64)
    assert len(feats) == bench.DUMP_FEATURES and np.all(np.diff(feats) > 0)
    assert abs(got["loss_sum"][0] - ref["loss"]) <= 1e-10 * abs(ref["loss"])
    assert abs(got["grad_intercept"][0] - ref["gb"]) <= 1e-10 * abs(ref["gb"])
    assert max_rel(got["grad_w"], ref["gw"]) <= 1e-9
    assert max_rel(got["grad_P_sampled"], ref["gP"][:, :, feats]) <= 1e-9
