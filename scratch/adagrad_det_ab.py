"""Synchronous-minibatch AdaGrad under NIMFM_DETERMINISTIC=1 (a column index per minibatch, then the stash / FFM
forward and the AdaGrad column kernels) against the default RED route, one shuffled epoch each:
  - C4 AdaGrad: bench.gen_criteo_rows (39 nnz/row, 1 M hashed features), HOFM degree 3 explicit, rank 32, logistic,
    minibatch 524 288;
  - C5 FFM AdaGrad: bench.gen_ffm_rows (39 fields, one nonzero each), rank 8, logistic, minibatch 524 288, d = 100 000
    (P of 39 x d x 8 doubles).
Each arm starts from the same parameters and a reset AdaGrad state; an epoch is one blocking library call timed with
the host clock, arms alternating, best of 2 after a warm epoch.  The deterministic arm runs with NIMFM_TRACE=1, whose
per-phase CUDA events give the share of the epoch spent building the minibatch index ("det index": gather, sort,
segment table and the one device-to-host copy of four counts).  P after one epoch of each arm is compared at the
suite's AdaGrad bar (rtol 1e-8, atol 1e-13), and so are two runs of the same arm: two RED epochs show how far the
RED route's own summation-order noise carries over an epoch, two deterministic epochs must be bit-identical.
usage: python scratch/adagrad_det_ab.py [c4_rows] [c5_rows]   -> JSON lines on stdout"""
import ctypes as C
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ["NIMFM_TRACE"] = "1"          # read once per context: spans exist only in the deterministic epochs
import bench  # noqa: E402
import nimfm_b200 as nf  # noqa: E402
from nimfm_b200 import _lib  # noqa: E402

N4 = int(sys.argv[1]) if len(sys.argv) > 1 else 10_000_000
N5 = int(sys.argv[2]) if len(sys.argv) > 2 else 4_000_000
MB = 524_288
D5 = 100_000
lib, ctx = _lib.load(), _lib.ctx()
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                      text=True).stdout.strip().splitlines()[0]
print(json.dumps({"card": card, "c4_rows": N4, "c5_rows": N5, "miniBatchSize": MB}), flush=True)

# the library's trace lines go to fd 2: keep them in a file to read the index share back
trace_file = tempfile.TemporaryFile(mode="w+")
saved_err = os.dup(2)
os.dup2(trace_file.fileno(), 2)


def trace_lines():
    sys.stderr.flush()
    trace_file.seek(0)
    text = trace_file.read()
    trace_file.seek(0)
    trace_file.truncate()
    return [ln for ln in text.splitlines() if "deterministic adagrad epoch" in ln]


def index_share(lines):
    per = {}
    for ln in lines:
        for tag, us, cnt in re.findall(r"  (det \w+) ([0-9.]+) us x (\d+)", ln):
            per.setdefault(tag, []).append(float(us) * int(cnt))
    idx, passes = sum(per.get("det index", [])), sum(per.get("det passes", []))
    return {"index_ms_per_epoch": idx / 1e3 / max(len(lines), 1), "passes_ms_per_epoch": passes / 1e3 / max(len(lines), 1),
            "index_share_of_index_plus_passes": idx / (idx + passes) if idx + passes else None}


def set_arm(arm):
    os.environ.pop("NIMFM_DETERMINISTIC", None)
    if arm == "det":
        os.environ["NIMFM_DETERMINISTIC"] = "1"


def ab(name, epoch_call, get_P, reset):
    times, Ps, shares = {"red": [], "det": []}, {}, []
    for rep in range(3):                  # rep 0 warms both arms (allocations, index buffers, CUB scratch)
        for arm in ("red", "det"):
            set_arm(arm)
            reset()
            t0 = time.perf_counter()
            epoch_call()
            dt = time.perf_counter() - t0
            lines = trace_lines()
            if rep < 2:
                Ps[(arm, rep)] = get_P()
            if rep == 0:
                continue
            times[arm].append(dt)
            if arm == "det":
                shares.append(index_share(lines))
    set_arm("red")

    def compare(a, b):
        outside = ~np.isclose(b, a, rtol=1e-8, atol=1e-13)
        return {"within_adagrad_bar": not bool(outside.any()), "elements_outside_bar": int(outside.sum()),
                "elements": int(a.size), "max_abs_diff_over_max_abs": float(np.max(np.abs(b - a)) / np.max(np.abs(a))),
                "bit_identical": bool(np.array_equal(a, b))}

    out = {"config": name, "s_per_epoch": {k: min(v) for k, v in times.items()},
           "rows_per_s": {k: None for k in times}, "det_over_red": min(times["det"]) / min(times["red"]),
           "index": shares[-1],
           "P_after_one_epoch": {"det_vs_red": compare(Ps[("red", 0)], Ps[("det", 0)]),
                                 "red_vs_red": compare(Ps[("red", 0)], Ps[("red", 1)]),
                                 "det_vs_det": compare(Ps[("det", 0)], Ps[("det", 1)])}}
    return out


def c4():
    data, idx, ptr, y = bench.gen_criteo_rows(N4, 11)
    d = bench.D_FEATURES
    ds = nf.newCSRDataset(data, idx, ptr, N4, d)
    ds.set_targets(y)
    ds.handle()
    del data, idx
    rng = np.random.default_rng(4)
    P0 = rng.standard_normal((2, 32, d)) * 0.01
    fm = nf.newFactorizationMachine(nf.classification, degree=3, nComponents=32, fitLower="explicit", warmStart=True)
    fm.P, fm.w, fm.intercept, fm.isInitialized = P0.copy(), np.zeros(d), 0.0, True
    h = fm._to_device(d)
    cfg = _lib.AdagradCfg(nf.Logistic().kind, 1.0, 0.1, 1e-6, 1e-3, 1e-3, 1e-10, MB)
    perm = np.random.default_rng(5).permutation(N4).astype(np.int64)
    w0 = np.zeros(d)

    def reset():
        _lib.check(lib.nimfm_fm_set_params(ctx, h, _lib.ptr(P0), _lib.ptr(w0), 0.0, None))
        _lib.check(lib.nimfm_fm_adagrad_init(ctx, h, 1e-10, 1))

    def epoch():
        it, viol, ls = C.c_int64(1), C.c_double(), C.c_double()
        _lib.check(lib.nimfm_fm_adagrad_epoch(ctx, h, ds.handle(), C.byref(cfg), C.byref(it), _lib.ptr(perm), N4,
                                              C.byref(viol), C.byref(ls)))

    def get_P():
        fm._from_device(h)
        return fm.P.copy()

    try:
        out = ab("C4 AdaGrad: degree 3 explicit, k 32, d 1M, 39 nnz/row, shuffled", epoch, get_P, reset)
        out["rows_per_s"] = {k: N4 / v for k, v in out["s_per_epoch"].items()}
        return out
    finally:
        lib.nimfm_fm_free(ctx, h)
        ds.free()


def c5():
    data, idx, ptr, fields, y = bench.gen_ffm_rows(N5, 12, d=D5)
    ds = nf.newCSRFieldDataset(data, idx, ptr, fields, N5, D5, bench.N_FIELDS)
    ds.set_targets(y)
    ds.handle()
    del data, idx, fields
    P0 = np.random.default_rng(6).standard_normal((bench.N_FIELDS, D5, 8)) * 0.01
    m = nf.newFieldAwareFactorizationMachine(nf.classification, nComponents=8, warmStart=True)
    m.P, m.w, m.intercept, m.isInitialized = P0.copy(), np.zeros(D5), 0.0, True
    h = m._to_device(ds)
    cfg = _lib.AdagradCfg(nf.Logistic().kind, 1.0, 0.1, 1e-6, 1e-3, 1e-3, 1e-10, MB)
    perm = np.random.default_rng(7).permutation(N5).astype(np.int64)
    w0 = np.zeros(D5)

    def reset():
        _lib.check(lib.nimfm_ffm_set_params(ctx, h, _lib.ptr(P0), _lib.ptr(w0), 0.0))
        _lib.check(lib.nimfm_ffm_adagrad_init(ctx, h, 1e-10, 1))

    def epoch():
        it, viol, ls = C.c_int64(1), C.c_double(), C.c_double()
        _lib.check(lib.nimfm_ffm_adagrad_epoch(ctx, h, ds.handle(), C.byref(cfg), C.byref(it), _lib.ptr(perm), N5,
                                               C.byref(viol), C.byref(ls)))

    def get_P():
        m._from_device(h)
        return m.P.copy()

    try:
        out = ab("C5 FFM AdaGrad: 39 fields, k 8, d 100k, shuffled", epoch, get_P, reset)
        out["rows_per_s"] = {k: N5 / v for k, v in out["s_per_epoch"].items()}
        return out
    finally:
        lib.nimfm_ffm_free(ctx, h)
        ds.free()


try:
    results = [c4(), c5()]
finally:
    os.dup2(saved_err, 2)
for r in results:
    print(json.dumps(r), flush=True)
