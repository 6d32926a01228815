"""The deterministic FFM predict+grad route (NIMFM_DETERMINISTIC=1: forward kernel, then a column kernel over the CSC
twin, ffm_cols.cuh) against the RED route on the same step, on the C5 row shape (bench.gen_ffm_rows: 39 fields, one
nonzero each, Zipf ids; d = 100 000 so that k = 64 fits):
  - k = 10 (the default model), 20 and 64: the generic column kernel, which is the only one that runs there;
  - k = 8: the tuned column kernel against the generic one forced by NIMFM_FFM_COLS=generic, the cost of the generic
    kernel on a shape both run.
Times are CUDA events around 3 blocking predict+grad calls (nimfm_ffm_loss_grad) after one warm call (which also
builds the CSC twin); best of 2, arms alternating.  Outputs are compared against the first arm: loss, gw and gP with
helpers.sums_agree (bit equality where expected).
usage: python scratch/ffm_det_shapes_ab.py [rows]   -> JSON lines on stdout"""
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
D, NF = 100_000, 39
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                      text=True).stdout.strip().splitlines()[0]
print(json.dumps({"card": card, "rows_c5": N, "d": D}), flush=True)

ENV_KEYS = ("NIMFM_DETERMINISTIC", "NIMFM_FFM_COLS")
ARMS = {"red": {}, "det": {"NIMFM_DETERMINISTIC": "1"},
        "det_generic": {"NIMFM_DETERMINISTIC": "1", "NIMFM_FFM_COLS": "generic"}}


def set_arm(arm):
    for key in ENV_KEYS:
        os.environ.pop(key, None)
    os.environ.update(ARMS[arm])


def run(ds, n, k, arms):
    rng = np.random.default_rng(7)
    P = rng.standard_normal((NF, D, k)) * (0.3 / np.sqrt(NF * k))
    w = rng.standard_normal(D) * 0.01
    m = nf.newFieldAwareFactorizationMachine(nf.classification, nComponents=k, warmStart=True)
    m.P, m.w, m.intercept, m.isInitialized = P, w, 0.0, True
    h = m._to_device(ds)
    del P
    loss_kind = nf.Logistic().kind

    def step():
        ls = C.c_double()
        _lib.check(lib.nimfm_ffm_loss_grad(ctx, h, ds.handle(), loss_kind, 1.0, 0, n, None, n, 1, 0, C.byref(ls)))
        return ls.value

    ms_all, cmp = {a: [] for a in arms}, {}
    ref = None
    try:
        for rep in range(2):
            for arm in arms:
                set_arm(arm)
                ls = step()
                ms = C.c_float()
                _lib.check(lib.nimfm_timer_start(ctx))
                for _ in range(3):
                    step()
                _lib.check(lib.nimfm_timer_stop(ctx, C.byref(ms)))
                ms_all[arm].append(ms.value / 3)
                if rep == 0:
                    gP, gw, gb = np.zeros((NF, D, k)), np.zeros(D), C.c_double()
                    _lib.check(lib.nimfm_ffm_get_grads(ctx, h, _lib.ptr(gP), _lib.ptr(gw), C.byref(gb)))
                    if ref is None:
                        ref = (ls, gP, gw, gb.value)
                        continue
                    l0, g0, w0, b0 = ref
                    cmp[arm] = {"loss_rel": abs(ls - l0) / abs(l0), "gb_abs": abs(gb.value - b0),
                                "gP_err_vs_max": float(np.max(np.abs(gP - g0)) / np.max(np.abs(g0))),
                                "gP_sums_agree": bool(sums_agree(gP, g0)), "gw_sums_agree": bool(sums_agree(gw, w0)),
                                "bit_identical": bool(ls == l0 and gb.value == b0 and np.array_equal(gP, g0)
                                                      and np.array_equal(gw, w0))}
                    del gP, gw
    finally:
        for key in ENV_KEYS:
            os.environ.pop(key, None)
        lib.nimfm_ffm_free(ctx, h)
    for arm in arms:
        ms = min(ms_all[arm])
        out = {"shape": "c5", "k": k, "rows": n, "route": arm, "Mrows_s": round(n / ms / 1e3, 3),
               "ms_per_step": round(ms, 3), "ms_all": [round(v, 3) for v in ms_all[arm]]}
        out.update(cmp.get(arm, {}))
        print(json.dumps(out), flush=True)


data, idx, ptr, fields, y = bench.gen_ffm_rows(N, 6000, d=D)
ds = nf.newCSRFieldDataset(data, idx, ptr, fields, N, D, NF)
ds.set_targets(y)
ds.handle()
del data, idx, fields
run(ds, N, 10, ["red", "det"])
run(ds, N, 20, ["red", "det"])
run(ds, N, 64, ["red", "det"])
run(ds, N, 8, ["det", "det_generic", "red"])
ds.free()
