"""The deterministic FM predict+grad route (NIMFM_DETERMINISTIC=1, csrc/fm_cols.cu) at shapes outside the tuned
kernels, against the RED route on the same step, on the C4 row shape (bench.gen_criteo_rows: 39 nonzeros per row,
13 always-present columns, Zipf categoricals, 1 M features):
  - degree 3 explicit, k = 30 (generic stash forward + generic column kernel);
  - degree 4 explicit, k = 16 (generic pair);
  - degree 3 explicit, k = 32: the tuned pair against the generic pair forced by NIMFM_ROW_KERNEL=generic, the cost of
    the generic kernels on a shape both run;
  - degree 3 explicit, k = 32 on rows of 1 000 nonzeros (one per slot of 1 000 id ranges; the generic pair).
Times are CUDA events around 3 blocking predict+grad calls after one warm call (which also builds the CSC twin).
Outputs are compared against the first arm: loss, gw and gP with helpers.sums_agree (bit equality where expected).
usage: python scratch/det_shapes_ab.py [rows]   -> JSON lines on stdout"""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench  # noqa: E402
import nimfm_b200 as nf  # noqa: E402
from nimfm_b200 import _lib  # noqa: E402
from helpers import sums_agree  # noqa: E402

lib, ctx = _lib.load(), _lib.ctx()
N = int(sys.argv[1]) if len(sys.argv) > 1 else 2_000_000
D = bench.D_FEATURES
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                      text=True).stdout.strip().splitlines()[0]
print(json.dumps({"card": card, "rows_c4": N, "d": D}), flush=True)

ARMS = {"red": {}, "det": {"NIMFM_DETERMINISTIC": "1"},
        "det_generic": {"NIMFM_DETERMINISTIC": "1", "NIMFM_ROW_KERNEL": "generic"}}


def long_rows(n, z=1000, seed=11):
    """z nonzeros per row, one in each of z id ranges (uniform inside the range), values U(0,1]"""
    rng = np.random.default_rng(seed)
    R = D // z
    idx = (rng.integers(0, R, size=(n, z)) + np.arange(z)[None, :] * R).astype(np.int64)
    data = 1.0 - rng.random((n, z))
    y = np.where(rng.random(n) < 0.5, -1.0, 1.0)
    return data.reshape(-1), idx.reshape(-1), np.arange(n + 1, dtype=np.int64) * z, y


def run(label, data, indices, indptr, y, degree, k, arms):
    n = len(indptr) - 1
    ds = nf.newCSRDataset(data, indices, indptr, n, D)
    ds.set_targets(y)
    ds.handle()
    rng = np.random.default_rng(7)
    P = rng.standard_normal((degree - 1, k, D)) * 0.01
    w = rng.standard_normal(D) * 0.01
    fm = nf.newFactorizationMachine(nf.classification, degree=degree, nComponents=k, fitLower=nf.explicit)
    fm.P, fm.w, fm.intercept, fm.isInitialized = P, w, 0.0, True
    h = fm._to_device(D)
    loss_kind = nf.Logistic().kind

    def step():
        ls = C.c_double()
        _lib.check(lib.nimfm_fm_loss_grad(ctx, h, ds.handle(), loss_kind, 1.0, 0, n, None, n, 1, 0, C.byref(ls)))
        return ls.value

    outs, ms_all = {}, {a: [] for a in arms}
    try:
        for rep in range(2):
            for arm in arms:
                for key in ("NIMFM_DETERMINISTIC", "NIMFM_ROW_KERNEL"):
                    os.environ.pop(key, None)
                os.environ.update(ARMS[arm])
                ls = step()                                     # warm (first det call builds the CSC twin)
                ms = C.c_float()
                _lib.check(lib.nimfm_timer_start(ctx))
                for _ in range(3):
                    step()
                _lib.check(lib.nimfm_timer_stop(ctx, C.byref(ms)))
                ms_all[arm].append(ms.value / 3)
                if rep == 0:
                    gP, gw, gb = np.zeros_like(P), np.zeros(D), C.c_double()
                    _lib.check(lib.nimfm_fm_get_grads(ctx, h, _lib.ptr(gP), _lib.ptr(gw), C.byref(gb)))
                    outs[arm] = (ls, gP, gw, gb.value)
    finally:
        for key in ("NIMFM_DETERMINISTIC", "NIMFM_ROW_KERNEL"):
            os.environ.pop(key, None)
        lib.nimfm_fm_free(ctx, h)
        ds.free()
    ref = arms[0]
    for arm in arms:
        ms = min(ms_all[arm])
        out = {"shape": label, "degree": degree, "k": k, "rows": n, "nnz_per_row": int(indptr[1] - indptr[0]),
               "route": arm, "Mrows_s": round(n / ms / 1e3, 3), "ms_per_step": round(ms, 3),
               "ms_all": [round(v, 3) for v in ms_all[arm]]}
        if arm != ref:
            l0, g0, w0, b0 = outs[ref]
            l1, g1, w1, b1 = outs[arm]
            out["loss_rel"] = abs(l1 - l0) / abs(l0)
            out["gb_abs"] = abs(b1 - b0)
            out["gP_err_vs_max"] = float(np.max(np.abs(g1 - g0)) / np.max(np.abs(g0)))
            out["gP_sums_agree"] = bool(sums_agree(g1, g0))
            out["gw_sums_agree"] = bool(sums_agree(w1, w0))
            out["gP_gw_bit_identical"] = bool(np.array_equal(g1, g0) and np.array_equal(w1, w0))
        print(json.dumps(out), flush=True)


c4 = bench.gen_criteo_rows(N, 1000)
run("c4", *c4, 3, 30, ["red", "det"])
run("c4", *c4, 4, 16, ["red", "det"])
run("c4", *c4, 3, 32, ["det", "det_generic", "red"])
del c4
run("rows_1000", *long_rows(max(N // 20, 1000)), 3, 32, ["red", "det"])
