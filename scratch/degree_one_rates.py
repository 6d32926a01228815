"""Rates of the degree-1 (linear) FM routes on the C3 row shape (Criteo-shaped CSR, 39 nonzeros per row, d = 1 M),
next to a degree-2 k = 1 model on the same data, as fractions of the algorithmic-byte roofline (SURVEY 8d with
k*o = 0): B_fwd = z (8 + 4 + 8 l) + 16 per row, B_grad = B_fwd + 8 + 8 l z (l = 1: one w value per nonzero).
Times are CUDA events on the library's stream (nimfm_time_loss_grad, nimfm_timer_*) after a warm-up call.
Usage: python scratch/degree_one_rates.py [n_rows]   (one JSON line per measurement; the card name and power limit
first, read with nvidia-smi --query-gpu)"""
import ctypes as C
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

import bench
import nimfm_b200 as nf
from nimfm_b200 import _lib

HBM_BPS = 6.5297e12   # B200 HBM copy bandwidth measured with a torch copy (SURVEY: 6529.7 GB/s), bytes/s


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 10_000_000
    print(json.dumps({"gpu": gpu_info(), "rows": n}), flush=True)
    data, idx, ptr, y = bench.gen_criteo_rows(n, 2000)
    d = bench.D_FEATURES
    z = 39
    ds = nf.newCSRDataset(data, idx, ptr, n, d)
    ds.set_targets(y)
    ds.handle()
    lib, ctx = _lib.load(), _lib.ctx()
    b_fwd = z * (8 + 4 + 8) + 16
    b_grad = b_fwd + 8 + 8 * z
    rng = np.random.default_rng(1)
    for degree in (1, 2):
        nO = 0 if degree == 1 else 1
        fm = nf.newFactorizationMachine(nf.classification, degree=degree, nComponents=1, warmStart=True)
        fm.P = rng.standard_normal((nO, 1, d)) * 0.01
        fm.w, fm.intercept, fm.isInitialized = rng.standard_normal(d) * 0.01, 0.0, True
        h = fm._to_device(d)
        try:
            for grad, B, what in ((0, b_fwd, "decisionFunction"), (1, b_grad, "predict+grad")):
                ms = C.c_float()
                _lib.check(lib.nimfm_fm_time_loss_grad(ctx, h, ds.handle(), 2, n, n, 1, grad, C.byref(ms)))   # warm-up
                _lib.check(lib.nimfm_fm_time_loss_grad(ctx, h, ds.handle(), 2, n, n, 5, grad, C.byref(ms)))
                rate = n / (ms.value * 1e-3)
                print(json.dumps({"degree": degree, "k": 1, "what": what, "ms": round(ms.value, 4),
                                  "rows_per_s": rate, "algorithmic_bytes_per_row": B,
                                  "fraction_of_hbm_roofline": rate * B / HBM_BPS}), flush=True)
        finally:
            lib.nimfm_fm_free(ctx, h)

        def timed(fit):
            fit()   # warm-up
            _lib.check(lib.nimfm_timer_start(ctx))
            fit()
            ms = C.c_float()
            _lib.check(lib.nimfm_timer_stop(ctx, C.byref(ms)))
            return ms.value

        def model():
            m = nf.newFactorizationMachine(nf.classification, degree=degree, nComponents=1, warmStart=True)
            m.P, m.w, m.intercept, m.isInitialized = fm.P.copy(), fm.w.copy(), 0.0, True
            return m

        mb = 25_641   # the reference's default MBPSGD minibatch on this shape (d n / nnz)
        ms = timed(lambda: nf.newMBPSGD(maxIter=1, loss=nf.Logistic(), reg=nf.newL1(), gamma=0.0, miniBatchSize=mb,
                                        verbose=0, tol=0.0, shuffle=False).fit(ds, y, model()))
        print(json.dumps({"degree": degree, "k": 1, "what": f"MBPSGD epoch (minibatch {mb})", "ms": round(ms, 2),
                          "rows_per_s": n / (ms * 1e-3),
                          "fraction_of_hbm_roofline": n / (ms * 1e-3) * b_grad / HBM_BPS}), flush=True)
        ms = timed(lambda: nf.newAdaGrad(maxIter=1, loss=nf.Logistic(), miniBatchSize=mb, verbose=0, tol=0.0,
                                         shuffle=False).fit(ds, y, model()))
        print(json.dumps({"degree": degree, "k": 1, "what": f"minibatch AdaGrad epoch (minibatch {mb})",
                          "ms": round(ms, 2), "rows_per_s": n / (ms * 1e-3),
                          "fraction_of_hbm_roofline": n / (ms * 1e-3) * b_grad / HBM_BPS}), flush=True)
        m_seq = 200_000
        sub = nf.newCSRDataset(data[:m_seq * z], idx[:m_seq * z], ptr[:m_seq + 1], m_seq, d)
        ms = timed(lambda: nf.newSGD(maxIter=1, loss=nf.Logistic(), verbose=0, tol=0.0, shuffle=False)
                   .fit(sub, y[:m_seq], model()))
        print(json.dumps({"degree": degree, "k": 1, "what": f"sequential SGD epoch ({m_seq} rows)", "ms": round(ms, 2),
                          "samples_per_s": m_seq / (ms * 1e-3)}), flush=True)


if __name__ == "__main__":
    main()
