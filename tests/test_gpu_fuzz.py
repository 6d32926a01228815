"""Seeded random sweep of the FM row kernels against the oracle: shapes that select every dispatch route
(the streaming instances for k in {8,16,32} at degree 2/3, the generic runtime-k kernel otherwise, hot
columns present or not, dummy features, ragged and empty rows, row lists with repeats), through
decisionFunction, predict+grad, a short MBPSGD fit and a short synchronous-minibatch AdaGrad fit."""
import ctypes as C

import numpy as np
import pytest

import nimfm_b200 as nf
from nimfm_b200 import _lib
from oracle import bruteforce as bf
from oracle.oracle import CSR
from helpers import max_rel

pytestmark = pytest.mark.gpu

LOSSES = {"squared": nf.Squared, "logistic": nf.Logistic, "squared_hinge": nf.SquaredHinge, "huber": nf.Huber}


def random_case(seed):
    rng = np.random.default_rng(seed)
    degree = int(rng.choice([2, 2, 3, 3, 4, 5, 6]))
    k = int(rng.choice([1, 3, 5, 8, 8, 16, 16, 32, 32, 40]))
    fit_lower = str(rng.choice(["explicit", "none", "augment"]))
    fit_linear, fit_intercept = bool(rng.integers(0, 2)), bool(rng.integers(0, 2))
    n, d = int(rng.integers(30, 400)), int(rng.integers(4, 120))
    max_nnz = int(rng.integers(1, min(d, 45) + 1))
    n_dense = int(rng.integers(0, min(3, d)))           # always-present columns -> the hot-column table engages
    data, indices, indptr = [], [], [0]
    for i in range(n):
        z = 0 if rng.random() < 0.05 else int(rng.integers(1, max_nnz + 1))
        cols = set(range(n_dense)) if z > 0 else set()
        if d - n_dense > 0 and z > len(cols):
            extra = rng.choice(np.arange(n_dense, d), size=min(z - len(cols), d - n_dense), replace=False)
            cols |= set(int(c) for c in extra)
        cols = np.sort(np.array(sorted(cols), dtype=np.int64))
        indices.extend(cols.tolist())
        data.extend((rng.standard_normal(len(cols)) * 0.8).tolist())
        indptr.append(len(indices))
    csr = CSR(data, indices, indptr, n, d)
    nO, nA = bf.n_orders(degree, fit_lower), bf.n_augments(degree, fit_lower, fit_linear)
    P = rng.standard_normal((nO, k, d + nA)) * 0.15
    w = rng.standard_normal(d) * 0.1 if fit_linear else np.zeros(d)
    b = float(rng.standard_normal() * 0.1) if fit_intercept else 0.0
    loss = str(rng.choice(list(LOSSES)))
    y = rng.standard_normal(n) if loss in ("squared", "huber") else np.sign(rng.standard_normal(n))
    return dict(degree=degree, k=k, fit_lower=fit_lower, fit_linear=fit_linear, fit_intercept=fit_intercept,
                csr=csr, P=P, w=w, b=b, loss=loss, y=y, rng=rng)


def make_fm(c):
    task = nf.regression if c["loss"] in ("squared", "huber") else nf.classification
    fm = nf.newFactorizationMachine(task, degree=c["degree"], nComponents=c["k"], fitLower=c["fit_lower"],
                                    fitLinear=c["fit_linear"], fitIntercept=c["fit_intercept"], warmStart=True)
    fm.P, fm.w, fm.intercept, fm.isInitialized = c["P"].copy(), c["w"].copy(), c["b"], True
    return fm


@pytest.mark.parametrize("seed", range(40))
def test_random_predict_and_grad(oracle, seed):
    c = random_case(1000 + seed)
    csr, fm = c["csr"], make_fm(c)
    ds = nf.newCSRDataset(csr.data, csr.indices, csr.indptr, csr.n, csr.d)
    ref = oracle.fm_decision_function(csr, c["P"], c["w"], c["b"], c["degree"])
    got = fm.decisionFunction(ds)                       # host-streamed route (no device twin yet)
    assert max_rel(got, ref) <= 1e-10
    ds.handle()
    assert max_rel(fm.decisionFunction(ds), ref) <= 1e-10
    # predict+grad over a row list with repeats, coef = dloss / mb
    rows = c["rng"].integers(0, csr.n, size=csr.n + 7)
    sub = oracle.csr_take_rows(csr, rows)
    g = oracle.fm_loss_grad(sub, c["y"][rows], c["P"], c["w"], c["b"], c["degree"], c["loss"],
                            fit_linear=c["fit_linear"], fit_intercept=c["fit_intercept"], mini_batch_size=len(rows))
    lib, ctx = _lib.load(), _lib.ctx()
    ds.set_targets(c["y"])
    h = fm._to_device(csr.d)
    try:
        ls = C.c_double()
        idx = _lib.i64(rows)
        lo = LOSSES[c["loss"]]()
        _lib.check(lib.nimfm_fm_loss_grad(ctx, h, ds.handle(), lo.kind, lo.threshold, 0, len(rows), _lib.ptr(idx),
                                          len(rows), 1, 0, C.byref(ls)))
        gP, gw, gb = np.zeros_like(c["P"]), np.zeros(csr.d), C.c_double()
        _lib.check(lib.nimfm_fm_get_grads(ctx, h, _lib.ptr(gP), _lib.ptr(gw), C.byref(gb)))
    finally:
        lib.nimfm_fm_free(ctx, h)
    assert abs(ls.value - g["loss"]) <= 1e-10 * max(1.0, abs(g["loss"]))
    # (rows with one nonzero have an exactly-cancelling ANOVA derivative: both sides are ~1e-21 of rounding noise
    # there, hence the absolute floor)
    scale = max(float(np.max(np.abs(g["gP"]))), 1e-12)
    np.testing.assert_allclose(gP, g["gP"], rtol=1e-9, atol=max(1e-9 * scale, 1e-15))
    if c["fit_linear"]:
        assert max_rel(gw, g["gw"]) <= 1e-9
    if c["fit_intercept"]:
        assert abs(gb.value - g["gb"]) <= 1e-10 * max(1.0, abs(g["gb"]))


@pytest.mark.parametrize("seed", range(16))
def test_random_solver_epochs(oracle, seed):
    c = random_case(5000 + seed)
    csr = c["csr"]
    ds = nf.newCSRDataset(csr.data, csr.indices, csr.indptr, csr.n, csr.d)
    lo = LOSSES[c["loss"]]()
    mb = int(c["rng"].integers(3, 40))
    kw = dict(eta0=0.05, alpha0=1e-6, alpha=1e-3, beta=1e-3)
    common = (c["degree"], c["loss"], c["fit_linear"], c["fit_intercept"])
    # MBPSGD (L1 prox); warmStart=true keeps MBPSGD.it at its constructor value 0
    r = oracle.mbpsgd_fit(csr, c["y"], c["P"], c["w"], c["b"], *common, max_iter=2, gamma=1e-3, reg="l1",
                          mini_batch_size=mb, it=0, **kw)
    fm = make_fm(c)
    opt = nf.newMBPSGD(maxIter=2, loss=lo, reg=nf.newL1(), gamma=1e-3, miniBatchSize=mb, verbose=0, tol=0.0,
                       shuffle=False, **kw)
    opt.fit(ds, c["y"], fm)
    np.testing.assert_allclose(opt.history, r["epoch_loss"], rtol=1e-8)
    np.testing.assert_allclose(fm.P, r["P"], rtol=1e-8, atol=1e-13)
    np.testing.assert_allclose(fm.w, r["w"], rtol=1e-8, atol=1e-13)
    # AdaGrad, synchronous minibatch
    r = oracle.adagrad_fit(csr, c["y"], c["P"], c["w"], c["b"], *common, max_iter=2, mini_batch_size=mb, **kw)
    fm = make_fm(c)
    opt = nf.newAdaGrad(maxIter=2, loss=lo, miniBatchSize=mb, verbose=0, tol=0.0, shuffle=False, **kw)
    opt.fit(ds, c["y"], fm)
    np.testing.assert_allclose([h[1] for h in opt.history], r["loss"], rtol=1e-8)
    np.testing.assert_allclose(fm.P, r["P"], rtol=1e-8, atol=1e-13)
    np.testing.assert_allclose(fm.w, r["w"], rtol=1e-8, atol=1e-13)
    assert abs(fm.intercept - r["intercept"]) <= 1e-9 * max(1.0, abs(r["intercept"]))
