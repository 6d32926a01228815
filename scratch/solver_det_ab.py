"""MBPSGD and synchronous-minibatch SGD under NIMFM_DETERMINISTIC=1 against the default RED route, one shuffled epoch
each.  Under the switch every shuffled minibatch is a row list, so it builds its own column index (nimfm_mb_index_build)
and runs the stash / FFM forward and the column kernels over its view:
  - C3 MBPSGD: bench.gen_criteo_rows (39 nnz/row, 1 M hashed features), FM degree 2 rank 16, logistic, L1 at gamma 0,
    minibatch 25 641 (the reference default, d·n div nnz) and 1 Mi rows;
  - C4 minibatch SGD: the first rows of the same dataset, HOFM degree 3 explicit rank 32, logistic, eta0 1e-5,
    minibatch 4 096 and 65 536;
  - C5 FFM minibatch SGD: bench.gen_ffm_rows (39 fields, one nonzero each), rank 8, logistic, minibatch 65 536,
    d = 100 000.
The RED arm runs what a user gets without the switch: at C3's default minibatch and C4's 4 096 rows that is the lazy
(touched-features-only) epoch, which the switch turns off.  Each arm starts from the same parameters; an epoch is one
blocking library call timed with the host clock, arms alternating, best of 2 after a warm epoch.  NIMFM_TRACE=1 (both
arms) gives the deterministic epochs' "det index" (gather, sort, segment table and the one device-to-host copy of four
counts) and "det passes" CUDA-event spans.  P after one epoch of each arm is compared (rtol 1e-8, atol 1e-13), and
two deterministic epochs must be bit-identical.
usage: python scratch/solver_det_ab.py [c3_rows] [c4_rows] [c5_rows]   -> JSON lines on stdout"""
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
os.environ["NIMFM_TRACE"] = "1"          # read once per context
import bench  # noqa: E402
import nimfm_b200 as nf  # noqa: E402
from nimfm_b200 import _lib  # noqa: E402

N3 = int(sys.argv[1]) if len(sys.argv) > 1 else 10_000_000
N4 = int(sys.argv[2]) if len(sys.argv) > 2 else 2_000_000
N5 = int(sys.argv[3]) if len(sys.argv) > 3 else 2_000_000
D5 = 100_000
lib, ctx = _lib.load(), _lib.ctx()
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                      text=True).stdout.strip().splitlines()[0]
print(json.dumps({"card": card, "c3_rows": N3, "c4_rows": N4, "c5_rows": N5}), flush=True)

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
    return [ln for ln in text.splitlines() if "det index" in ln]


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


def ab(name, rows, epoch_call, get_P, reset, red_form):
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
        return {"within_1e-8": not bool(outside.any()), "elements_outside": int(outside.sum()),
                "max_abs_diff_over_max_abs": float(np.max(np.abs(b - a)) / np.max(np.abs(a))),
                "bit_identical": bool(np.array_equal(a, b))}

    best = {k: min(v) for k, v in times.items()}
    return {"config": name, "red_arm": red_form, "s_per_epoch": best, "rows_per_s": {k: rows / v for k, v in best.items()},
            "det_over_red": best["det"] / best["red"], "index": shares[-1],
            "P_after_one_epoch": {"det_vs_red": compare(Ps[("red", 0)], Ps[("det", 0)]),
                                  "det_vs_det": compare(Ps[("det", 0)], Ps[("det", 1)])}}


def lazy_rule(B, nnz_per_row, dd):
    """the RED arm's form: the lazy epochs' default rule (fm_api.cu) on one rank"""
    return "lazy" if B * nnz_per_row <= 2.0 * dd else "dense"


def criteo(n):
    data, idx, ptr, y = bench.gen_criteo_rows(n, 11)
    ds = nf.newCSRDataset(data, idx, ptr, n, bench.D_FEATURES)
    ds.set_targets(y)
    ds.handle()
    return ds, len(data)


def c3(ds, nnz):
    d = bench.D_FEATURES
    P0 = np.random.default_rng(2).standard_normal((1, bench.K3, d)) * 0.01
    w0 = np.zeros(d)
    fm = nf.newFactorizationMachine(nf.classification, degree=2, nComponents=bench.K3, warmStart=True)
    fm.P, fm.w, fm.intercept, fm.isInitialized = P0.copy(), w0.copy(), 0.0, True
    h = fm._to_device(d)
    out = []
    try:
        z = nnz / N3
        for mb in (max(d * N3 // nnz, 1), 1 << 20):
            inner = (N3 - 1) // mb + 1
            cfg = _lib.MbpsgdCfg(nf.Logistic().kind, 1.0, 0.1, 1e-6, 1e-3, 1e-4, 0.0, _lib.REG_L1, _lib.SCHED["optimal"],
                                 1.0, mb, inner)
            perm = np.random.default_rng(3).permutation(N3)
            sample = perm[np.arange(mb * inner) % N3].astype(np.int64)   # the host's sample list, one wrap

            def reset():
                _lib.check(lib.nimfm_fm_set_params(ctx, h, _lib.ptr(P0), _lib.ptr(w0), 0.0, None))

            def epoch():
                it, ii, rl = C.c_int64(1), C.c_int64(0), C.c_double()
                _lib.check(lib.nimfm_fm_mbpsgd_epoch(ctx, h, ds.handle(), C.byref(cfg), mb, C.byref(it), C.byref(ii),
                                                     _lib.ptr(sample), C.byref(rl)))

            def get_P():
                fm._from_device(h)
                return fm.P.copy()

            r = ab(f"C3 MBPSGD: degree 2, k 16, d 1M, 39 nnz/row, shuffled, minibatch {mb} x {inner}", mb * inner, epoch,
                   get_P, reset, lazy_rule(mb, z, d))
            out.append(r)
    finally:
        lib.nimfm_fm_free(ctx, h)
    return out


def c4(ds, nnz, n):
    d = bench.D_FEATURES
    z = nnz / N3
    P0 = np.random.default_rng(4).standard_normal((2, 32, d)) * 0.01
    w0 = np.zeros(d)
    fm = nf.newFactorizationMachine(nf.classification, degree=3, nComponents=32, fitLower="explicit", warmStart=True)
    fm.P, fm.w, fm.intercept, fm.isInitialized = P0.copy(), w0.copy(), 0.0, True
    h = fm._to_device(d)
    # eta0 1e-5: a minibatch moves P by B·eta·(mean gradient), and at eta0 = 0.01 a 4 096-row minibatch diverges
    cfg = _lib.SgdCfg(nf.Logistic().kind, 1.0, 1e-5, 1e-6, 1e-3, 1e-3, _lib.SCHED["optimal"], 1.0)
    perm = np.random.default_rng(5).permutation(n).astype(np.int64)
    out = []
    try:
        for B in (4096, 65536):
            def reset():
                _lib.check(lib.nimfm_fm_set_params(ctx, h, _lib.ptr(P0), _lib.ptr(w0), 0.0, None))

            def epoch():
                it, viol, ls = C.c_int64(1), C.c_double(), C.c_double()
                _lib.check(lib.nimfm_fm_sgd_minibatch_epoch(ctx, h, ds.handle(), C.byref(cfg), B, 0, C.byref(it),
                                                            _lib.ptr(perm), n, C.byref(viol), C.byref(ls)))

            def get_P():
                fm._from_device(h)
                return fm.P.copy()

            out.append(ab(f"C4 minibatch SGD: degree 3 explicit, k 32, d 1M, 39 nnz/row, shuffled, minibatch {B}, "
                          f"{n} rows", n, epoch, get_P, reset, lazy_rule(B, z, d)))
    finally:
        lib.nimfm_fm_free(ctx, h)
    return out


def c5():
    data, idx, ptr, fields, y = bench.gen_ffm_rows(N5, 12, d=D5)
    ds = nf.newCSRFieldDataset(data, idx, ptr, fields, N5, D5, bench.N_FIELDS)
    ds.set_targets(y)
    ds.handle()
    del data, idx, fields
    P0 = np.random.default_rng(6).standard_normal((bench.N_FIELDS, D5, 8)) * 0.01
    w0 = np.zeros(D5)
    m = nf.newFieldAwareFactorizationMachine(nf.classification, nComponents=8, warmStart=True)
    m.P, m.w, m.intercept, m.isInitialized = P0.copy(), w0.copy(), 0.0, True
    h = m._to_device(ds)
    cfg = _lib.SgdCfg(nf.Logistic().kind, 1.0, 0.01, 1e-6, 1e-3, 1e-3, _lib.SCHED["optimal"], 1.0)
    perm = np.random.default_rng(7).permutation(N5).astype(np.int64)
    B = 65536

    def reset():
        _lib.check(lib.nimfm_ffm_set_params(ctx, h, _lib.ptr(P0), _lib.ptr(w0), 0.0))

    def epoch():
        it, viol, ls = C.c_int64(1), C.c_double(), C.c_double()
        _lib.check(lib.nimfm_ffm_sgd_minibatch_epoch(ctx, h, ds.handle(), C.byref(cfg), B, 0, C.byref(it),
                                                     _lib.ptr(perm), N5, C.byref(viol), C.byref(ls)))

    def get_P():
        m._from_device(h)
        return m.P.copy()

    try:
        return [ab(f"C5 FFM minibatch SGD: 39 fields, k 8, d 100k, shuffled, minibatch {B}, {N5} rows", N5, epoch, get_P,
                   reset, "dense")]
    finally:
        lib.nimfm_ffm_free(ctx, h)
        ds.free()


results = []
try:
    ds, nnz = criteo(N3)
    try:
        results += c3(ds, nnz)
        results += c4(ds, nnz, N4)            # the first N4 rows of the C3 dataset
    finally:
        ds.free()
    results += c5()
finally:
    os.dup2(saved_err, 2)
for r in results:
    print(json.dumps(r), flush=True)
