"""FFM (nonzero, field) unit kernel (ffm_units.cuh) against the staged and pair-block kernels: forward, predict+grad
and one AdaGrad epoch at 2 M rows of the C5 row shape (39 fields, one nonzero each; bench.gen_ffm_rows with
d = 100 000 so that k = 64 fits) and one multi-hot long-row shape.  Arms alternate within each config and their
outputs are compared.  Kernel times are CUDA events around 3 launches (nimfm_ffm_time_loss_grad); the AdaGrad epoch
is host wall time of one blocking library call.  FP64-add payload: the gradient REDs a row emits (one k-vector per
(nonzero, field) unit with a partner; twice that for AdaGrad's g_sum and g_norm).
usage: python scratch/ffm_shapes_ab.py [rows]   -> JSON lines on stdout"""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
import nimfm_b200 as nf  # noqa: E402
from nimfm_b200 import _lib  # noqa: E402

lib, ctx = _lib.load(), _lib.ctx()
N = int(sys.argv[1]) if len(sys.argv) > 1 else 2_000_000
D = 100_000
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                      text=True).stdout.strip().splitlines()[0]
print(json.dumps({"card": card, "rows_c5": N, "d": D}), flush=True)


def c5(n):
    data, idx, ptr, fields, y = bench.gen_ffm_rows(n, 6000, d=D)
    return data, idx, ptr, fields, y, 39


def multihot(n, seed=7):
    """rows of 150..250 nonzeros over 39 fields, fields repeating within a row, distinct ids"""
    rng = np.random.default_rng(seed)
    z = rng.integers(150, 251, n)
    ptr = np.concatenate([[0], np.cumsum(z)]).astype(np.int64)
    nnz = int(ptr[-1])
    idx = (rng.integers(0, D // 256, nnz) * 256 + (np.arange(nnz) - np.repeat(ptr[:-1], z)) % 256).astype(np.int64)
    fields = rng.integers(0, 39, nnz).astype(np.int64)
    data = np.where(rng.random(nnz) < 0.66, 1.0, rng.random(nnz))
    y = np.sign(rng.standard_normal(n))
    return data, idx, ptr, fields, y, 39


def payload_units(ptr, fields):
    """(nonzero, field) units with at least one partner, summed over the rows"""
    tot = 0
    for r in range(len(ptr) - 1):
        f = fields[ptr[r]:ptr[r + 1]]
        _, cnt = np.unique(f, return_counts=True)
        tot += len(f) * len(cnt) - int(np.sum(cnt == 1))
    return tot


def run(label, gen, k, arms, n):
    data, idx, ptr, fields, y, nF = gen(n)
    ds = nf.newCSRFieldDataset(data, idx, ptr, fields, n, D, nF)
    ds.set_targets(y)
    ds.handle()
    units = payload_units(ptr[:20001], fields) * n / min(n, 20000)   # sampled: rows are i.i.d.
    pay_grad = units * k * 8 / n
    rng = np.random.default_rng(3)
    P = rng.standard_normal((nF, D, k)) * (0.3 / np.sqrt(39 * k))
    w0 = rng.standard_normal(D) * 0.01
    m = nf.newFieldAwareFactorizationMachine(nf.classification, nComponents=k, warmStart=True)
    m.P, m.w, m.intercept, m.isInitialized = P, w0, 0.0, True
    h = m._to_device(ds)
    res = {a: {"fwd_ms": [], "grad_ms": []} for a in arms}
    outs = {}
    try:
        for rep in range(3):
            for arm in arms:
                os.environ["NIMFM_FFM_KERNEL"] = arm
                for key, g in (("fwd_ms", 0), ("grad_ms", 1)):
                    ms = C.c_float()
                    _lib.check(lib.nimfm_ffm_time_loss_grad(ctx, h, ds.handle(), 2, n, n, 1, g, C.byref(ms)))   # warm
                    _lib.check(lib.nimfm_ffm_time_loss_grad(ctx, h, ds.handle(), 2, n, n, 3, g, C.byref(ms)))
                    res[arm][key].append(ms.value)
                if rep == 0:
                    yo = np.zeros(n)
                    _lib.check(lib.nimfm_ffm_decision_function(ctx, h, ds.handle(), _lib.ptr(yo)))
                    ls = C.c_double()
                    _lib.check(lib.nimfm_ffm_loss_grad(ctx, h, ds.handle(), 2, 1.0, 0, n, None, n, 1, 0, C.byref(ls)))
                    gP = np.zeros_like(P)
                    _lib.check(lib.nimfm_ffm_get_grads(ctx, h, _lib.ptr(gP), None, None))
                    outs[arm] = (yo, ls.value, gP)
    finally:
        lib.nimfm_ffm_free(ctx, h)
    ada = {}
    for arm in arms:
        os.environ["NIMFM_FFM_KERNEL"] = arm
        ma = nf.newFieldAwareFactorizationMachine(nf.classification, nComponents=k, warmStart=True)
        ma.P, ma.w, ma.intercept, ma.isInitialized = P.copy(), np.zeros(D), 0.0, True
        opt = nf.newAdaGrad(maxIter=2, eta0=1e-3, loss=nf.Logistic(), verbose=0, tol=0.0, shuffle=False,
                            miniBatchSize=1 << 19)
        opt.fit(ds, y, ma)
        ada[arm] = (min(opt.epoch_seconds), opt.history, ma.P)
    os.environ.pop("NIMFM_FFM_KERNEL", None)
    ref = arms[0]
    for arm in arms:
        fwd, grad = min(res[arm]["fwd_ms"]), min(res[arm]["grad_ms"])
        out = {"shape": label, "k": k, "rows": n, "kernel": arm or "default",
               "fwd_Mrows_s": round(n / fwd / 1e3, 3), "grad_Mrows_s": round(n / grad / 1e3, 3),
               "adagrad_Msamples_s": round(n / ada[arm][0] / 1e6, 3),
               "fp64_add_payload_B_per_row": round(pay_grad, 1),
               "grad_red_TB_s": round(pay_grad * n / (grad * 1e-3) / 1e12, 3),
               "adagrad_red_TB_s": round(2 * pay_grad * n / ada[arm][0] / 1e12, 3),
               "fwd_ms_all": [round(v, 3) for v in res[arm]["fwd_ms"]],
               "grad_ms_all": [round(v, 3) for v in res[arm]["grad_ms"]]}
        if arm != ref:
            y0, l0, g0 = outs[ref]
            y1, l1, g1 = outs[arm]
            out["dec_max_rel"] = float(np.max(np.abs(y1 - y0) / np.maximum(np.abs(y0), 1e-12)))
            out["loss_rel"] = abs(l1 - l0) / abs(l0)
            out["gP_err_vs_max"] = float(np.max(np.abs(g1 - g0)) / np.max(np.abs(g0)))
            out["adagrad_P_err_vs_max"] = float(np.max(np.abs(ada[arm][2] - ada[ref][2])) / np.max(np.abs(ada[ref][2])))
            out["adagrad_loss_rel"] = abs(ada[arm][1][-1][1] - ada[ref][1][-1][1]) / abs(ada[ref][1][-1][1])
        print(json.dumps(out), flush=True)


run("c5", c5, 10, ["units", "block"], N)
run("c5", c5, 16, ["units", ""], N)
run("c5", c5, 20, ["units"], N)
run("c5", c5, 64, ["units"], N)
run("multihot_150_250", multihot, 10, ["units"], max(N // 10, 1000))
