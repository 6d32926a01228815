"""Degree-1 factorization machines (the linear model b + <w, x>: nOrders = 0, no P) on the device, held to the CPU
oracle at the suite's bars on every FM entry point: decisionFunction (resident CSR, CSC, host-fed, windowed stream
file), predict+grad (four losses, row lists, wrapping ranges), MBPSGD, AdaGrad (sequential and minibatch, warm
start), SGD (every schedule, resetScaling), minibatch SGD, PSGD, CD / PCD, the CLI, the deterministic route and
two ranks.  Sizes reach past one persistent wave of the linear row kernel (fm_linear.cu)."""
import ctypes as C
import json
import os
import sys

import numpy as np
import pytest

import nimfm_b200 as nf
from nimfm_b200 import _lib
from oracle.oracle import CSR
from helpers import make_dense, max_rel
from test_gpu_deterministic import long_column_csr
from test_gpu_fm import csr_ds, dev_loss_grad, ragged_csr
from test_gpu_loaders import write_svm

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEC_TOL = 1e-10
OBJ_TOL = 1e-8
K = 4   # nComponents plays no part at degree 1 (P is empty)
LOSSES = {"squared": nf.Squared, "logistic": nf.Logistic, "squared_hinge": nf.SquaredHinge, "huber": nf.Huber}


def linear_fm(w, b, fit_linear=True, fit_intercept=True, task=nf.regression):
    fm = nf.newFactorizationMachine(task, degree=1, nComponents=K, fitLinear=fit_linear, fitIntercept=fit_intercept,
                                    warmStart=True)
    fm.P, fm.w, fm.intercept, fm.isInitialized = np.zeros((0, K, len(w))), np.asarray(w, float).copy(), b, True
    return fm


def no_p(d):
    return np.zeros((0, K, d))


def big_ragged(n=40_000, d=3_000, max_nnz=40, seed=3):
    """rows of 0..max_nnz nonzeros (every 7th row empty): the 32-lane form, about ten persistent waves"""
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, max_nnz + 1, size=n)
    lens[::7] = 0
    indptr = np.concatenate([[0], np.cumsum(lens)])
    indices = np.concatenate([np.sort(rng.choice(d, size=z, replace=False)) for z in lens]).astype(np.int64)
    data = rng.standard_normal(int(indptr[-1]))
    return CSR(data, indices, indptr, n, d)


def short_rows(n=90_000, d=500, z=6, seed=4):
    """six nonzeros per row (the 8-lane form, four rows per warp), column 0 in every row: a hot column"""
    csr = long_column_csr(n, d, seed, z)
    return csr


@pytest.fixture
def plain(monkeypatch):
    for v in ("NIMFM_DETERMINISTIC", "NIMFM_ROW_KERNEL", "NIMFM_MBPSGD_LAZY", "NIMFM_SGD_MB_LAZY", "NIMFM_ADAGRAD_SEQ"):
        monkeypatch.delenv(v, raising=False)


# ---------------------------------------------------------------- decisionFunction
@pytest.mark.parametrize("make", [big_ragged, short_rows], ids=["ragged_32_lanes", "short_rows_8_lanes"])
def test_decision_function_every_input_form(oracle, plain, make):
    csr = make()
    n, d = csr.n, csr.d
    rng = np.random.default_rng(1)
    w = rng.standard_normal(d)
    ref = oracle.fm_decision_function(csr, no_p(d), w, 0.3, 1)
    np.testing.assert_allclose(ref, np.asarray(csr_dense_dot(csr, w)) + 0.3, rtol=1e-9, atol=1e-12)
    fm = linear_fm(w, 0.3)
    ds = csr_ds(csr)
    got_host = fm.decisionFunction(ds)                     # no device twin: host-fed chunks (pageable memory)
    assert ds._handle is None
    ds.handle()
    got_dev = fm.decisionFunction(ds)                      # resident CSR
    csc = oracle.csr_to_csc(csr)
    got_csc = fm.decisionFunction(nf.newCSCDataset(csc.data, csc.indices, csc.indptr, n, d))
    for got in (got_host, got_dev, got_csc):
        assert max_rel(got, ref) <= DEC_TOL
    lib, ctx = _lib.load(), _lib.ctx()
    h = fm._to_device(d)
    try:
        out = np.zeros(n)
        _lib.check(lib.nimfm_fm_decision_function_host(ctx, h, n, d, _lib.ptr(csr.data), _lib.ptr(csr.indices),
                                                       _lib.ptr(csr.indptr), 4099, _lib.ptr(out)))
        assert np.array_equal(out, got_host)
        # page-locked host arrays (the registered-memory form of the host-fed path)
        import torch
        pins = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in (csr.data, csr.indices, csr.indptr)]
        ptrs = [C.c_void_p(t.data_ptr()) for t in pins]
        out2 = np.zeros(n)
        _lib.check(lib.nimfm_fm_decision_function_host(ctx, h, n, d, ptrs[0], ptrs[1], ptrs[2], 0, _lib.ptr(out2)))
        assert max_rel(out2, ref) <= DEC_TOL
    finally:
        lib.nimfm_fm_free(ctx, h)


def csr_dense_dot(csr, w):
    out = np.zeros(csr.n)
    rows = np.repeat(np.arange(csr.n), np.diff(csr.indptr))
    np.add.at(out, rows, csr.data * w[csr.indices])
    return out


def test_decision_function_windowed_stream_file(oracle, plain, tmp_path):
    csr = ragged_csr(600, 50, 5, 20)
    y = np.sign(np.random.default_rng(2).standard_normal(csr.n))
    txt, fx, fy = (str(tmp_path / f) for f in ("a.svm", "a.bin", "a.lab"))
    write_svm(txt, csr, y)
    nf.convertSVMLightFile(txt, fx, fy)
    win = nf.newStreamCSRDataset(fx, cacheSize=2.0 / 1024.0, resident=False)
    assert win.windowed
    whole = nf.newStreamCSRDataset(fx, resident=True)
    ref_csr = CSR(whole.data, whole.indices, whole.indptr, whole.nSamples, whole.nFeatures)
    w = np.random.default_rng(3).standard_normal(whole.nFeatures)
    ref = oracle.fm_decision_function(ref_csr, no_p(whole.nFeatures), w, -0.2, 1)
    assert max_rel(linear_fm(w, -0.2).decisionFunction(win), ref) <= DEC_TOL


# ---------------------------------------------------------------- predict + grad
@pytest.mark.parametrize("loss_name", list(LOSSES))
def test_loss_grad_matches_oracle(oracle, plain, loss_name):
    csr = big_ragged(seed=11)
    n, d = csr.n, csr.d
    rng = np.random.default_rng(5)
    y = np.sign(rng.standard_normal(n)) if loss_name in ("logistic", "squared_hinge") else rng.standard_normal(n)
    w = rng.standard_normal(d) * 0.1
    fm = linear_fm(w, 0.2)
    ls, gP, gw, gb = dev_loss_grad(fm, csr_ds(csr), y, LOSSES[loss_name]())
    ref = oracle.fm_loss_grad(csr, y, no_p(d), w, 0.2, 1, loss_name)
    assert gP.shape == (0, K, d)
    assert abs(ls - ref["loss"]) <= 1e-10 * abs(ref["loss"])
    assert max_rel(gw, ref["gw"]) <= 1e-8 and abs(gb - ref["gb"]) <= 1e-10 * max(abs(ref["gb"]), 1.0)


def test_loss_grad_row_list_and_wrap(oracle, plain):
    csr = short_rows(seed=6)
    n, d = csr.n, csr.d
    rng = np.random.default_rng(7)
    y = rng.standard_normal(n)
    w = rng.standard_normal(d) * 0.1
    fm = linear_fm(w, 0.0)
    rows = rng.choice(n, size=30_000, replace=False)
    _, _, gw, gb = dev_loss_grad(fm, csr_ds(csr), y, nf.Squared(), rows=rows, mb=17)
    ref = oracle.fm_loss_grad(oracle.csr_take_rows(csr, rows), y[rows], no_p(d), w, 0.0, 1, "squared",
                              mini_batch_size=17)
    assert max_rel(gw, ref["gw"]) <= 1e-8 and abs(gb - ref["gb"]) <= 1e-9 * abs(ref["gb"])
    wrap = (n - 5_000 + np.arange(20_000)) % n
    _, _, gw2, gb2 = dev_loss_grad(fm, csr_ds(csr), y, nf.Squared(), row_begin=n - 5_000, n_rows=20_000, mb=20_000)
    ref2 = oracle.fm_loss_grad(oracle.csr_take_rows(csr, wrap), y[wrap], no_p(d), w, 0.0, 1, "squared",
                               mini_batch_size=20_000)
    assert max_rel(gw2, ref2["gw"]) <= 1e-8 and abs(gb2 - ref2["gb"]) <= 1e-9 * abs(ref2["gb"])


@pytest.mark.parametrize("fit_linear,fit_intercept", [(False, True), (True, False), (False, False)])
def test_fit_linear_and_fit_intercept_off(oracle, plain, fit_linear, fit_intercept):
    csr = ragged_csr(5_000, 60, 8, 12)
    y = np.random.default_rng(8).standard_normal(csr.n)
    w = np.random.default_rng(9).standard_normal(60) if fit_linear else np.zeros(60)
    fm = linear_fm(w, 0.4, fit_linear, fit_intercept)
    ref = oracle.fm_decision_function(csr, no_p(60), w, 0.4, 1)
    assert max_rel(fm.decisionFunction(csr_ds(csr)), ref) <= DEC_TOL
    _, _, gw, _ = dev_loss_grad(fm, csr_ds(csr), y, nf.Squared())
    rg = oracle.fm_loss_grad(csr, y, no_p(60), w, 0.4, 1, "squared", fit_linear=fit_linear, fit_intercept=fit_intercept)
    assert max_rel(gw, rg["gw"]) <= 1e-8
    if not fit_linear:
        assert not np.any(gw)
    kw = dict(eta0=0.1, alpha0=1e-6, alpha=1e-3, beta=1e-4, gamma=1e-3)
    r = oracle.mbpsgd_fit(csr, y, no_p(60), w, 0.4, 1, "squared", fit_linear, fit_intercept, max_iter=2, reg="l1",
                          mini_batch_size=300, it=0, **kw)
    opt = nf.newMBPSGD(maxIter=2, reg=nf.newL1(), miniBatchSize=300, verbose=0, tol=0.0, shuffle=False, **kw)
    opt.fit(csr_ds(csr), y, fm)
    np.testing.assert_allclose(opt.history, r["epoch_loss"], rtol=OBJ_TOL)
    assert max_rel(fm.w, r["w"]) <= 1e-8 and abs(fm.intercept - r["intercept"]) <= 1e-9


# ---------------------------------------------------------------- MBPSGD
@pytest.mark.parametrize("reg", ["l1", "l21"])
@pytest.mark.parametrize("shuffle,mb", [(False, 7_000), (True, 5_000), (False, 50_000)],
                         ids=["cyclic", "shuffled", "minibatch_over_n"])
def test_mbpsgd_matches_oracle(oracle, plain, reg, shuffle, mb):
    csr = short_rows(n=30_000, seed=12)
    n, d = csr.n, csr.d
    rng = np.random.default_rng(13)
    y = np.sign(rng.standard_normal(n))
    w = rng.standard_normal(d) * 0.1
    kw = dict(eta0=0.3, alpha0=1e-3, alpha=5e-2, beta=8e-2, gamma=1e-2)
    fm = linear_fm(w, 0.1, task=nf.classification)
    opt = nf.newMBPSGD(maxIter=3, loss=nf.Logistic(), reg=nf.newL1() if reg == "l1" else nf.newL21(), miniBatchSize=mb,
                       verbose=0, tol=0.0, shuffle=shuffle, **kw)
    opt.fit(csr_ds(csr), y, fm)
    perms = None
    if shuffle:
        r, idx, perms = np.random.default_rng(fm.randomState), np.arange(n), []
        for _ in range(12):
            r.shuffle(idx)
            perms.append(idx.copy())
        perms = np.array(perms)
    ref = oracle.mbpsgd_fit(csr, y, no_p(d), w, 0.1, 1, "logistic", max_iter=3, reg=reg, mini_batch_size=mb, it=0,
                            perms=perms, **kw)
    np.testing.assert_allclose(opt.history, ref["epoch_loss"], rtol=OBJ_TOL)
    assert max_rel(fm.w, ref["w"]) <= 1e-8 and abs(fm.intercept - ref["intercept"]) <= 1e-9
    assert np.array_equal(fm.w == 0.0, ref["w"] == 0.0) and fm.P.shape == (0, K, d)


def test_squaredl12_default_still_raises(plain):
    csr = ragged_csr(50, 10, 1, 5)
    fm = linear_fm(np.zeros(10), 0.0)
    with pytest.raises(ValueError, match="SquaredL12 supports only degree=2"):
        nf.newMBPSGD(maxIter=1, verbose=0).fit(csr_ds(csr), np.zeros(50), fm)
    with pytest.raises(ValueError, match="SquaredL12 supports only degree=2"):
        nf.newPSGD(maxIter=1, verbose=0).fit(csr_ds(csr), np.zeros(50), fm)
    csc = CSR(*_csc_arrays(csr), 50, 10)
    with pytest.raises(ValueError, match="SquaredL12 supports only degree=2"):
        nf.newPCD(maxIter=1, verbose=0).fit(nf.newCSCDataset(csc.data, csc.indices, csc.indptr, 50, 10), np.zeros(50), fm)


def _csc_arrays(csr):
    from oracle import oracle as orc
    c = orc.csr_to_csc(csr)
    return c.data, c.indices, c.indptr


def test_augment_with_fit_linear_is_refused(plain):
    fm = nf.newFactorizationMachine(nf.regression, degree=1, nComponents=2, fitLower=nf.augment, fitLinear=True)
    fm.P, fm.w, fm.isInitialized = np.zeros((0, 2, 6)), np.zeros(6), True
    with pytest.raises(ValueError, match="nAugments = -1"):
        fm.decisionFunction(csr_ds(ragged_csr(20, 6, 1, 3)))
    lib, h = _lib.load(), C.c_void_p()
    with pytest.raises(ValueError, match="nAugments = -1"):
        _lib.check(lib.nimfm_fm_create(_lib.ctx(), 1, 2, 0, -1, 6, 1, 1, C.byref(h)))
    with pytest.raises(ValueError, match="nOrders = 0"):
        _lib.check(lib.nimfm_fm_create(_lib.ctx(), 1, 2, 1, 0, 6, 1, 1, C.byref(h)))


# ---------------------------------------------------------------- AdaGrad
@pytest.mark.parametrize("mb", [1, 9_000])
def test_adagrad_matches_oracle_and_warm_starts(oracle, plain, mb):
    n, d = (3_000, 400) if mb == 1 else (40_000, 2_000)
    csr = ragged_csr(n, d, 14, 30) if mb == 1 else big_ragged(n, d, 30, seed=14)
    y = np.random.default_rng(15).standard_normal(n)
    w = np.zeros(d)
    kw = dict(eta0=0.1, alpha0=1e-6, alpha=1e-3, beta=1e-3)
    ref = oracle.adagrad_fit(csr, y, no_p(d), w, 0.0, 1, "squared", True, True, max_iter=2, mini_batch_size=mb, **kw)
    fm = linear_fm(w, 0.0)
    opt = nf.newAdaGrad(maxIter=2, verbose=0, tol=0.0, shuffle=False, miniBatchSize=mb, **kw)
    opt.fit(csr_ds(csr), y, fm)
    np.testing.assert_allclose([h[1] for h in opt.history], ref["loss"], rtol=OBJ_TOL)
    np.testing.assert_allclose([h[0] for h in opt.history], ref["viol"], rtol=1e-8)
    assert max_rel(fm.w, ref["w"]) <= 1e-8 and abs(fm.intercept - ref["intercept"]) <= 1e-9
    assert opt.g_sum["P"].shape == (0, d, K) and opt.it == ref["it"]
    assert max_rel(opt.g_sum["w"], ref["state"]["gsw"]) <= 1e-8
    # warm start: a second fit continues from g_sum / g_norm (the (0, d, k) P-state included)
    ref2 = oracle.adagrad_fit(csr, y, no_p(d), ref["w"], ref["intercept"], 1, "squared", True, True, max_iter=1,
                              mini_batch_size=mb, it=ref["it"], state=ref["state"], **kw)
    opt2 = nf.newAdaGrad(maxIter=1, verbose=0, tol=0.0, shuffle=False, miniBatchSize=mb, **kw)
    opt2.it, opt2.g_sum, opt2.g_norm = opt.it, opt.g_sum, opt.g_norm
    fm.warmStart = True
    opt2.fit(csr_ds(csr), y, fm)
    np.testing.assert_allclose([h[1] for h in opt2.history], ref2["loss"], rtol=OBJ_TOL)
    assert max_rel(fm.w, ref2["w"]) <= 1e-8 and abs(fm.intercept - ref2["intercept"]) <= 1e-9


# ---------------------------------------------------------------- SGD / minibatch SGD / PSGD
@pytest.mark.parametrize("sched,eta0,alpha,alpha0", [("optimal", 0.01, 1e-3, 1e-3), ("constant", 0.02, 20.0, 1e-3),
                                                      ("invscaling", 0.05, 1e-3, 1e-3), ("pegasos", 0.01, 1.0, 1.0)])
def test_sgd_sequential_every_schedule(oracle, plain, sched, eta0, alpha, alpha0):
    """resetScaling fires: constant with eta0 * alpha = 0.4 takes scaling_w below 1e-9 after ~41 samples, and
    pegasos (eta = 1 / (alpha * it)) zeroes it at the first sample"""
    n, d = 2_500, 300
    csr = ragged_csr(n, d, 16, 25)
    y = np.random.default_rng(17).standard_normal(n)
    w = np.random.default_rng(18).standard_normal(d) * 0.1
    kw = dict(eta0=eta0, alpha0=alpha0, alpha=alpha, beta=1.0, power=0.5 if sched == "invscaling" else 1.0)
    ref = oracle.sgd_fit(csr, y, no_p(d), w, 0.1, 1, "squared", max_iter=2, scheduling=sched, **kw)
    fm = linear_fm(w, 0.1)
    opt = nf.newSGD(maxIter=2, verbose=0, tol=0.0, shuffle=False, scheduling=getattr(nf, sched), **kw)
    opt.it = 1
    opt.fit(csr_ds(csr), y, fm)
    np.testing.assert_allclose([h[1] for h in opt.history], ref["loss"], rtol=OBJ_TOL)
    assert max_rel(fm.w, ref["w"]) <= 1e-8 and abs(fm.intercept - ref["intercept"]) <= 1e-8 * max(abs(ref["intercept"]), 1)


def test_sgd_minibatch_max_threads(oracle, plain):
    csr = short_rows(n=20_000, seed=19)
    n, d = csr.n, csr.d
    y = np.sign(np.random.default_rng(20).standard_normal(n))
    w = np.random.default_rng(21).standard_normal(d) * 0.1
    kw = dict(eta0=0.03, alpha0=1e-3, alpha=2e-2, beta=3e-2)
    perms = np.array([np.random.default_rng(40 + e).permutation(n) for e in range(2)])
    fm = linear_fm(w, 0.1, task=nf.classification)
    opt = nf.newSGD(maxIter=2, loss=nf.Logistic(), verbose=0, tol=0.0, **kw)
    opt.fit(csr_ds(csr), y, fm, maxThreads=700, perms=perms)
    ref = oracle.sgd_minibatch_fit(csr, y, no_p(d), w, 0.1, 1, "logistic", B=700, max_iter=2, perms=perms, it=1, **kw)
    np.testing.assert_allclose([h[1] for h in opt.history], ref["loss"], rtol=OBJ_TOL)
    assert max_rel(fm.w, ref["w"]) <= 1e-8 and abs(fm.intercept - ref["intercept"]) <= 1e-8


@pytest.mark.parametrize("reg", ["l1", "l21"])
def test_psgd_matches_oracle(oracle, plain, reg):
    n, d = 2_000, 200
    csr = ragged_csr(n, d, 22, 20)
    y = np.random.default_rng(23).standard_normal(n)
    w = np.random.default_rng(24).standard_normal(d) * 0.2
    kw = dict(eta0=0.05, alpha0=1e-6, alpha=1e-3, beta=1e-3, gamma=3e-2)
    ref = oracle.psgd_fit(csr, y, no_p(d), w, 0.1, 1, "squared", max_iter=2, reg=reg, **kw)
    fm = linear_fm(w, 0.1)
    opt = nf.newPSGD(maxIter=2, reg=nf.newL1() if reg == "l1" else nf.newL21(), verbose=0, tol=0.0, shuffle=False, **kw)
    opt.it = 1
    opt.fit(csr_ds(csr), y, fm)
    np.testing.assert_allclose(opt.history, ref["epoch_loss"], rtol=OBJ_TOL)
    assert max_rel(fm.w, ref["w"]) <= 1e-8 and abs(fm.intercept - ref["intercept"]) <= 1e-9


# ---------------------------------------------------------------- CD / PCD
@pytest.mark.parametrize("fit_linear,fit_intercept", [(True, True), (False, True), (True, False)])
def test_cd_matches_oracle(oracle, plain, fit_linear, fit_intercept):
    n, d = 3_000, 80
    X = make_dense(n, d, 25, density=0.2, positive=False)
    y = np.random.default_rng(26).standard_normal(n)
    csc = oracle.csr_to_csc(CSR.from_dense(X))
    w = np.random.default_rng(27).standard_normal(d) * 0.1 if fit_linear else np.zeros(d)
    kw = dict(alpha0=1e-6, alpha=1e-3, beta=1e-3)
    ref = oracle.cd_fit(csc, y, no_p(d), w, 0.0, 1, "squared", fit_linear, fit_intercept, max_iter=3, **kw)
    fm = linear_fm(w, 0.0, fit_linear, fit_intercept)
    opt = nf.newCD(maxIter=3, verbose=0, tol=0.0, **kw)
    opt.fit(nf.newCSCDataset(csc.data, csc.indices, csc.indptr, n, d), y, fm)
    np.testing.assert_allclose([h[1] for h in opt.history], ref["loss"], rtol=OBJ_TOL)
    assert max_rel(fm.w, ref["w"]) <= 1e-8 and abs(fm.intercept - ref["intercept"]) <= 1e-9


def test_pcd_l1_matches_oracle(oracle, plain):
    n, d = 2_000, 60
    X = make_dense(n, d, 28, density=0.3, positive=False)
    y = np.random.default_rng(29).standard_normal(n)
    csc = oracle.csr_to_csc(CSR.from_dense(X))
    w = np.random.default_rng(30).standard_normal(d) * 0.1
    kw = dict(alpha0=1e-6, alpha=1e-3, beta=1e-3, gamma=2e-2)
    ref = oracle.pcd_fit(csc, y, no_p(d), w, 0.0, 1, "squared", max_iter=3, reg="l1", **kw)
    fm = linear_fm(w, 0.0)
    opt = nf.newPCD(maxIter=3, verbose=0, tol=0.0, reg=nf.newL1(), **kw)
    opt.fit(nf.newCSCDataset(csc.data, csc.indices, csc.indptr, n, d), y, fm)
    np.testing.assert_allclose([h[1] for h in opt.history], ref["loss"], rtol=OBJ_TOL)
    assert max_rel(fm.w, ref["w"]) <= 1e-8 and abs(fm.intercept - ref["intercept"]) <= 1e-9


# ---------------------------------------------------------------- CLI
def test_cli_train_test_degree_one(oracle, plain, tmp_path, capsys):
    from nimfm_b200.__main__ import main
    X = make_dense(120, 12, 31, density=0.5, positive=False)
    csr = CSR.from_dense(X)
    y = X @ np.random.default_rng(32).standard_normal(12)
    tr = str(tmp_path / "tr.svm")
    write_svm(tr, csr, y)
    model, p1, p2 = (str(tmp_path / f) for f in ("m.txt", "p1.txt", "p2.txt"))
    main(["train", "--task", "r", "--train", tr, "--test", tr, "--degree", "1", "--solver", "cd", "--maxIter", "5",
          "--dump", model, "--predict", p1, "--nFeatures", "12", "--verbose", "0"])
    rmse = float(capsys.readouterr().out.split("Test RMSE: ")[1].split()[0])
    assert "P[" not in open(model).read()
    main(["test", "--task", "r", "--test", tr, "--load", model, "--predict", p2, "--nFeatures", "12", "--verbose", "0"])
    assert abs(float(capsys.readouterr().out.split("Test RMSE: ")[1].split()[0]) - rmse) < 1e-12
    assert np.array_equal(np.loadtxt(p1), np.loadtxt(p2))
    fm = nf.FactorizationMachine.load(model, False)
    ref = oracle.cd_fit(oracle.csr_to_csc(csr), y, no_p(12), np.zeros(12), 0.0, 1, "squared", max_iter=5, alpha0=1e-7,
                        alpha=1e-5, beta=1e-3, tol=1e-5)
    assert max_rel(fm.w, ref["w"]) <= 1e-8
    for solver in ("sgd", "adagrad"):
        main(["train", "--task", "c", "--train", tr, "--test", tr, "--degree", "1", "--solver", solver, "--loss",
              "logistic", "--maxIter", "2", "--verbose", "0"])
        assert "Test" in capsys.readouterr().out


# ---------------------------------------------------------------- NIMFM_DETERMINISTIC=1
@pytest.fixture
def deterministic(monkeypatch, plain):
    monkeypatch.setenv("NIMFM_DETERMINISTIC", "1")


def _det_data(n=6_000, d=4_000, z=8, seed=33):
    """column 0 in every row: a column of n entries, cut into many 512-entry segments (the combine kernels run)"""
    csr = long_column_csr(n, d, seed, z)
    y = np.sign(np.random.default_rng(seed + 1).standard_normal(n))
    w = np.random.default_rng(seed + 2).standard_normal(d) * 0.1
    return csr, y, w


def test_det_predict_grad_matches_oracle_and_repeats(oracle, deterministic):
    csr, y, w = _det_data()
    fm = linear_fm(w, 0.1, task=nf.classification)
    ds = csr_ds(csr)
    got = dev_loss_grad(fm, ds, y, nf.Logistic(), mb=csr.n)
    ref = oracle.fm_loss_grad(csr, y, no_p(csr.d), w, 0.1, 1, "logistic", mini_batch_size=csr.n)
    assert max_rel(got[2], ref["gw"]) <= 1e-8 and abs(got[3] - ref["gb"]) <= 1e-10 * abs(ref["gb"])
    again = dev_loss_grad(fm, ds, y, nf.Logistic(), mb=csr.n)
    assert got[0] == again[0] and got[3] == again[3] and np.array_equal(got[2], again[2])
    sub = dev_loss_grad(fm, ds, y, nf.Logistic(), row_begin=1_003, n_rows=2_500, mb=2_500)
    rows = np.arange(1_003, 3_503)
    rs = oracle.fm_loss_grad(oracle.csr_take_rows(csr, rows), y[rows], no_p(csr.d), w, 0.1, 1, "logistic",
                             mini_batch_size=2_500)
    assert max_rel(sub[2], rs["gw"]) <= 1e-8


def test_det_minibatch_adagrad_matches_oracle_and_repeats(oracle, deterministic):
    csr, y, _ = _det_data(seed=34)
    d = csr.d
    kw = dict(eta0=0.1, alpha0=1e-6, alpha=1e-3, beta=1e-3)
    perms = np.array([np.random.default_rng(50 + e).permutation(csr.n) for e in range(2)])

    def fit():
        fm = linear_fm(np.zeros(d), 0.0, task=nf.classification)
        opt = nf.newAdaGrad(maxIter=2, loss=nf.Logistic(), verbose=0, tol=0.0, miniBatchSize=1_500, **kw)
        opt.fit(csr_ds(csr), y, fm, perms=perms)
        return fm.w.copy(), fm.intercept, list(opt.history)

    w1, b1, h1 = fit()
    ref = oracle.adagrad_fit(csr, y, no_p(d), np.zeros(d), 0.0, 1, "logistic", max_iter=2, mini_batch_size=1_500,
                             perms=perms, **kw)
    np.testing.assert_allclose([h[1] for h in h1], ref["loss"], rtol=OBJ_TOL)
    assert max_rel(w1, ref["w"]) <= 1e-8 and abs(b1 - ref["intercept"]) <= 1e-9
    w2, b2, h2 = fit()
    assert np.array_equal(w1, w2) and b1 == b2 and h1 == h2


def test_det_shuffled_mbpsgd_and_minibatch_sgd_repeat(oracle, deterministic):
    csr, y, w = _det_data(seed=35)
    n, d = csr.n, csr.d
    kw = dict(eta0=0.3, alpha0=1e-3, alpha=5e-2, beta=8e-2, gamma=1e-3)

    def mbpsgd():
        fm = linear_fm(w, 0.1, task=nf.classification)
        opt = nf.newMBPSGD(maxIter=2, loss=nf.Logistic(), reg=nf.newL1(), miniBatchSize=1_700, verbose=0, tol=0.0,
                           shuffle=True, **kw)
        opt.fit(csr_ds(csr), y, fm)
        return fm, opt

    fm, opt = mbpsgd()
    r, idx, perms = np.random.default_rng(fm.randomState), np.arange(n), []
    for _ in range(12):
        r.shuffle(idx)
        perms.append(idx.copy())
    ref = oracle.mbpsgd_fit(csr, y, no_p(d), w, 0.1, 1, "logistic", max_iter=2, reg="l1", mini_batch_size=1_700, it=0,
                            perms=np.array(perms), **kw)
    np.testing.assert_allclose(opt.history, ref["epoch_loss"], rtol=OBJ_TOL)
    assert max_rel(fm.w, ref["w"]) <= 1e-8
    fm2, opt2 = mbpsgd()
    assert np.array_equal(fm.w, fm2.w) and fm.intercept == fm2.intercept and opt.history == opt2.history

    skw = dict(eta0=0.03, alpha0=1e-3, alpha=2e-2, beta=3e-2)
    sperms = np.array([np.random.default_rng(60 + e).permutation(n) for e in range(2)])

    def sgd():
        f = linear_fm(w, 0.1, task=nf.classification)
        o = nf.newSGD(maxIter=2, loss=nf.Logistic(), verbose=0, tol=0.0, **skw)
        o.fit(csr_ds(csr), y, f, maxThreads=700, perms=sperms)
        return f, o

    f1, o1 = sgd()
    rs = oracle.sgd_minibatch_fit(csr, y, no_p(d), w, 0.1, 1, "logistic", B=700, max_iter=2, perms=sperms, it=1, **skw)
    np.testing.assert_allclose([h[1] for h in o1.history], rs["loss"], rtol=OBJ_TOL)
    assert max_rel(f1.w, rs["w"]) <= 1e-8
    f2, o2 = sgd()
    assert np.array_equal(f1.w, f2.w) and f1.intercept == f2.intercept and o1.history == o2.history


# ---------------------------------------------------------------- two ranks
def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from nimfm_b200 import distributed as nd
    from oracle import oracle as orc
    from sharded_parity import _orders
    nd.init_comm(rank, world)
    n, d, mb = 97, 10, 7
    X = make_dense(n, d, 5, density=0.5, positive=False)
    y = np.sign(np.random.default_rng(0).standard_normal(n))
    w = np.random.default_rng(1).standard_normal(d) * 0.1
    csr = CSR.from_dense(X)
    spans, shares, _ = _orders(n, mb, world, nd.shard_rows, nd.local_batch)
    b, e = spans[rank]
    sh = orc.csr_take_rows(csr, np.arange(b, e))
    ds = nf.newCSRDataset(sh.data, sh.indices, sh.indptr, sh.n, d)
    errs = {"decision": max_rel(linear_fm(w, 0.05).decisionFunction(ds),
                                orc.fm_decision_function(csr, no_p(d), w, 0.05, 1)[b:e])}
    inner, epochs = -(-n // mb), 3
    order = np.concatenate([sb + (g * l + np.arange(l)) % (se - sb) for g in range(inner * epochs)
                            for (sb, se), l in zip(spans, shares)])
    kw = dict(eta0=0.1, alpha0=1e-6, alpha=1e-3, beta=1e-4, gamma=1e-3)
    for reg_name, reg in (("l1", nf.newL1()), ("l21", nf.newL21())):
        ref = orc.mbpsgd_fit(orc.csr_take_rows(csr, order), y[order], no_p(d), w, 0.05, 1, "logistic", max_iter=epochs,
                             reg=reg_name, mini_batch_size=mb, max_iter_inner=inner, it=0, **kw)
        fm = linear_fm(w, 0.05, task=nf.classification)
        opt = nf.newMBPSGD(maxIter=epochs, loss=nf.Logistic(), reg=reg, miniBatchSize=mb, verbose=0, tol=0.0,
                           shuffle=False, **kw)
        opt.fit(ds, y[b:e], fm)
        errs[f"mbpsgd_{reg_name}"] = max(max_rel(opt.history, ref["epoch_loss"]), max_rel(fm.w, ref["w"]),
                                         abs(fm.intercept - ref["intercept"]))
    json.dump(errs, open(os.path.join(out_dir, f"res{rank}.json"), "w"))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_parity_at_degree_one(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import socket
    import torch.multiprocessing as mp
    from oracle import oracle as orc
    orc.build()
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        errs = json.load(open(tmp_path / f"res{r}.json"))
        assert errs["decision"] <= DEC_TOL and errs["mbpsgd_l1"] <= 1e-8 and errs["mbpsgd_l21"] <= 1e-8, errs
