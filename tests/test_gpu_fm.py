"""Parity of the CUDA row kernels (K1 decisionFunction, K2 predict+grad, MBPSGD, AdaGrad) against the
CPU oracle, through the C ABI (nimfm_b200 is a thin ctypes mirror of include/nimfm_cuda.h).

Tolerances (BASELINE.json north_star): decision values <= 1e-10 relative; objective after a fixed
number of epochs <= 1e-8 relative; index / nnz bookkeeping bit-exact.
"""
import ctypes as C

import numpy as np
import pytest

import nimfm_b200 as nf
from nimfm_b200 import _lib
from oracle import bruteforce as bf
from oracle.oracle import CSR
from helpers import make_dense, make_fm_params, max_rel

pytestmark = pytest.mark.gpu

DEC_TOL = 1e-10   # decision values, relative
OBJ_TOL = 1e-8    # objective after N epochs, relative


def csr_ds(csr):
    return nf.newCSRDataset(csr.data, csr.indices, csr.indptr, csr.n, csr.d)


def make_fm(degree, k, fit_lower, fit_linear, fit_intercept, P, w, b, task=nf.regression):
    fm = nf.newFactorizationMachine(task, degree=degree, nComponents=k, fitLower=fit_lower,
                                    fitLinear=fit_linear, fitIntercept=fit_intercept, warmStart=True)
    fm.P, fm.w, fm.intercept, fm.isInitialized = P.copy(), w.copy(), b, True
    return fm


def ragged_csr(n, d, seed, max_nnz):
    """rows with 0..max_nnz nonzeros (empty rows included), sorted unique indices"""
    rng = np.random.default_rng(seed)
    data, indices, indptr = [], [], [0]
    for i in range(n):
        z = int(rng.integers(0, max_nnz + 1)) if i % 7 else 0
        cols = np.sort(rng.choice(d, size=min(z, d), replace=False))
        indices.extend(cols.tolist())
        data.extend(rng.standard_normal(len(cols)).tolist())
        indptr.append(len(indices))
    return CSR(data, indices, indptr, n, d)


# ---------------------------------------------------------------- K1
@pytest.mark.parametrize("degree", [2, 3, 4, 5, 6])
@pytest.mark.parametrize("fit_lower", ["explicit", "none", "augment"])
@pytest.mark.parametrize("k", [4, 10, 30])
def test_decision_function_matches_oracle(oracle, degree, fit_lower, k):
    # shapes of tests/test_kernels.nim:7-11 (n=20, d=10) and the k=30 of BASELINE configs 1-2
    n, d = 20, 10
    X = make_dense(n, d, 42 + degree, density=0.7)
    csr = CSR.from_dense(X)
    P, w, nA = make_fm_params(d, degree, k, fit_lower, True, seed=degree * 7 + k)
    fm = make_fm(degree, k, fit_lower, True, True, P, w, 0.25)
    expect = oracle.fm_decision_function(csr, P, w, 0.25, degree)
    got = fm.decisionFunction(csr_ds(csr))
    assert max_rel(got, expect) <= DEC_TOL
    # ColDataset path (kernels.nim:4-11,22-43)
    csc = oracle.csr_to_csc(csr)
    got_c = fm.decisionFunction(nf.newCSCDataset(csc.data, csc.indices, csc.indptr, n, d))
    expect_c = oracle.fm_decision_function(csc, P, w, 0.25, degree, is_csc=True)
    assert max_rel(got_c, expect_c) <= DEC_TOL


def test_decision_function_vs_bruteforce():
    """straight against the subset-enumeration definition (tests/kernels_slow.nim), tol 1e-6 there"""
    n, d, k, degree = 8, 7, 5, 3
    X = make_dense(n, d, 3, density=0.8)
    P, w, nA = make_fm_params(d, degree, k, "augment", True, seed=1)
    fm = make_fm(degree, k, "augment", True, True, P, w, -0.5)
    got = fm.decisionFunction(csr_ds(CSR.from_dense(X)))
    np.testing.assert_allclose(got, bf.fm_decision_function(X, P, w, -0.5, degree), rtol=1e-9, atol=1e-12)


@pytest.mark.parametrize("k,degree,fit_lower", [(33, 3, "explicit"), (70, 2, "explicit"), (64, 4, "none"),
                                                (16, 3, "explicit"), (8, 2, "explicit"), (32, 3, "explicit")])
def test_decision_function_ragged_and_wide(oracle, k, degree, fit_lower):
    """empty rows, ragged rows, rows longer than the staging capacity, k > 32 (component chunks)"""
    n, d = 300, 400
    csr = ragged_csr(n, d, 5, max_nnz=350 if k <= 16 else 120)
    P, w, nA = make_fm_params(d, degree, k, fit_lower, True, seed=k, scale=0.05)
    fm = make_fm(degree, k, fit_lower, True, True, P, w, 0.1)
    expect = oracle.fm_decision_function(csr, P, w, 0.1, degree)
    got = fm.decisionFunction(csr_ds(csr))
    assert max_rel(got, expect) <= DEC_TOL


def test_decision_function_host_streaming(oracle):
    """nimfm_fm_decision_function_host: the host CSR is streamed in chunks (ragged rows, empty rows, a
    chunk size that does not divide n); identical to the resident-dataset call and to the oracle"""
    n, d, k, degree = 700, 40, 8, 3
    csr = ragged_csr(n, d, 77, 15)
    P, w, _ = make_fm_params(d, degree, k, "augment", True, seed=3)
    fm = make_fm(degree, k, "augment", True, True, P, w, 0.2)
    fm.lams = np.random.default_rng(1).random(k) + 0.5
    ref = oracle.fm_decision_function(csr, P, w, 0.2, degree, lams=fm.lams)
    ds = csr_ds(csr)
    assert ds._handle is None
    got_host = fm.decisionFunction(ds)                       # no device twin -> streaming path
    assert ds._handle is None
    ds.handle()
    got_dev = fm.decisionFunction(ds)                        # resident path
    assert max_rel(got_host, ref) <= DEC_TOL and max_rel(got_dev, ref) <= DEC_TOL
    lib, ctx = _lib.load(), _lib.ctx()
    h = fm._to_device(d)
    try:
        out = np.zeros(n)
        _lib.check(lib.nimfm_fm_decision_function_host(ctx, h, n, d, _lib.ptr(csr.data), _lib.ptr(csr.indices),
                                                       _lib.ptr(csr.indptr), 97, _lib.ptr(out)))
        assert np.array_equal(out, got_host)                 # chunking does not change a single bit
        _lib.check(lib.nimfm_fm_decision_function_host(ctx, h, 0, d, None, None, _lib.ptr(csr.indptr), 0, _lib.ptr(out)))
        bad = csr.indices.copy()
        bad[5] = d
        with pytest.raises(ValueError, match="out of range"):
            _lib.check(lib.nimfm_fm_decision_function_host(ctx, h, n, d, _lib.ptr(csr.data), _lib.ptr(bad),
                                                           _lib.ptr(csr.indptr), 0, _lib.ptr(out)))
    finally:
        lib.nimfm_fm_free(ctx, h)


@pytest.mark.parametrize("host_threads", ["0", "1", "3", "8"])
@pytest.mark.parametrize("chunk", [0, 97, 256])
def test_loss_grad_host_streaming(oracle, monkeypatch, host_threads, chunk):
    """nimfm_fm_loss_grad_host / nimfm_fm_decision_function_host (the end-to-end calls bench.py times): host
    CSR in the reference dtypes -> chunks -> row kernel.  Both index-narrowing routes -- on the device
    (NIMFM_HOST_THREADS=0) and by the host staging team into pinned int32 slots (host_stage.h) -- against the
    oracle's updateGradient (minibatch_psgd.nim:67-88) and bit-identical to each other in the predictions."""
    monkeypatch.setenv("NIMFM_HOST_THREADS", host_threads)
    monkeypatch.setenv("NIMFM_HOST_STAGE_MIN_NNZ", "0")
    n, d, k, degree = 1500, 60, 8, 3
    csr = ragged_csr(n, d, 5, 17)
    rng = np.random.default_rng(8)
    y = np.where(rng.random(n) < 0.5, -1.0, 1.0)
    P, w, _ = make_fm_params(d, degree, k, "explicit", True, seed=4)
    fm = make_fm(degree, k, "explicit", True, True, P, w, -0.1, task=nf.classification)
    ref = oracle.fm_loss_grad(csr, y, P, w, -0.1, degree, "logistic", mini_batch_size=n)
    lib, ctx = _lib.load(), _lib.ctx()
    h = fm._to_device(d)
    try:
        ls = C.c_double()
        _lib.check(lib.nimfm_fm_loss_grad_host(ctx, h, n, d, _lib.ptr(csr.data), _lib.ptr(csr.indices), _lib.ptr(csr.indptr),
                                               _lib.ptr(y), 2, 1.0, n, chunk, 1, 0, C.byref(ls)))
        gP, gw, gb = np.zeros_like(P), np.zeros(d), C.c_double()
        _lib.check(lib.nimfm_fm_get_grads(ctx, h, _lib.ptr(gP), _lib.ptr(gw), C.byref(gb)))
        assert abs(ls.value - ref["loss"]) <= DEC_TOL * abs(ref["loss"])
        assert max_rel(gP, ref["gP"]) <= 1e-9 and max_rel(gw, ref["gw"]) <= 1e-9
        assert abs(gb.value - ref["gb"]) <= 1e-9 * max(abs(ref["gb"]), 1e-3)
        out = np.zeros(n)
        _lib.check(lib.nimfm_fm_decision_function_host(ctx, h, n, d, _lib.ptr(csr.data), _lib.ptr(csr.indices),
                                                       _lib.ptr(csr.indptr), chunk, _lib.ptr(out)))
        assert np.array_equal(out, fm.decisionFunction(csr_ds(csr)))
        # a column id outside [0,d) and a negative one, in different chunks; a decreasing indptr
        for pos, val in ((len(csr.indices) - 2, d), (3, -1)):
            bad = csr.indices.copy()
            bad[pos] = val
            with pytest.raises(ValueError, match="out of range"):
                _lib.check(lib.nimfm_fm_loss_grad_host(ctx, h, n, d, _lib.ptr(csr.data), _lib.ptr(bad), _lib.ptr(csr.indptr),
                                                       _lib.ptr(y), 2, 1.0, n, chunk, 1, 0, C.byref(ls)))
        ptr = csr.indptr.copy()
        ptr[700] = ptr[699] - 1 if ptr[699] > 0 else ptr[701] + 1
        with pytest.raises(ValueError, match="monotone"):
            _lib.check(lib.nimfm_fm_loss_grad_host(ctx, h, n, d, _lib.ptr(csr.data), _lib.ptr(csr.indices), _lib.ptr(ptr),
                                                   _lib.ptr(y), 2, 1.0, n, chunk, 1, 0, C.byref(ls)))
        # and the library is still usable afterwards
        _lib.check(lib.nimfm_fm_loss_grad_host(ctx, h, n, d, _lib.ptr(csr.data), _lib.ptr(csr.indices), _lib.ptr(csr.indptr),
                                               _lib.ptr(y), 2, 1.0, n, chunk, 1, 0, C.byref(ls)))
        assert abs(ls.value - ref["loss"]) <= DEC_TOL * abs(ref["loss"])
    finally:
        lib.nimfm_fm_free(ctx, h)


@pytest.mark.parametrize("memory", ["pageable", "registered"])
@pytest.mark.parametrize("chunk", [61, 1000])
def test_loss_grad_host_packed_values(oracle, monkeypatch, memory, chunk):
    """the lossless packed transport of the values (NIMFM_HOST_PACK=1: bit mask '== 1.0' + the other doubles + block
    offsets, expanded on the device) through the whole host-fed call, on pageable arrays and on page-locked ones,
    against the oracle, and bit-identical in the predictions to the resident kernel.  Values: exact ones,
    1 +/- 1 ulp, -0.0, denormals."""
    monkeypatch.setenv("NIMFM_HOST_THREADS", "3")
    monkeypatch.setenv("NIMFM_HOST_STAGE_MIN_NNZ", "0")
    monkeypatch.setenv("NIMFM_HOST_PACK", "1")
    n, d, k, degree = 4000, 80, 8, 3
    csr = ragged_csr(n, d, 23, 12)
    rng = np.random.default_rng(9)
    pick = rng.random(len(csr.data))
    csr.data[pick < 0.6] = 1.0
    csr.data[(pick >= 0.6) & (pick < 0.63)] = np.nextafter(1.0, 2.0)
    csr.data[(pick >= 0.63) & (pick < 0.66)] = np.nextafter(1.0, 0.0)
    csr.data[(pick >= 0.66) & (pick < 0.68)] = -0.0
    csr.data[(pick >= 0.68) & (pick < 0.70)] = 5e-324
    y = np.where(rng.random(n) < 0.5, -1.0, 1.0)
    P, w, _ = make_fm_params(d, degree, k, "explicit", True, seed=6)
    fm = make_fm(degree, k, "explicit", True, True, P, w, 0.2, task=nf.classification)
    ref = oracle.fm_loss_grad(csr, y, P, w, 0.2, degree, "logistic", mini_batch_size=n)
    lib, ctx = _lib.load(), _lib.ctx()
    arrays = (csr.data, csr.indices, csr.indptr, y)
    if memory == "registered":
        for a in arrays:
            _lib.check(lib.nimfm_host_register(ctx, _lib.ptr(a), a.nbytes))
    h = fm._to_device(d)
    try:
        for _ in range(2):
            ls = C.c_double()
            _lib.check(lib.nimfm_fm_loss_grad_host(ctx, h, n, d, _lib.ptr(csr.data), _lib.ptr(csr.indices), _lib.ptr(csr.indptr),
                                                   _lib.ptr(y), 2, 1.0, n, chunk, 1, 0, C.byref(ls)))
            gP, gw, gb = np.zeros_like(P), np.zeros(d), C.c_double()
            _lib.check(lib.nimfm_fm_get_grads(ctx, h, _lib.ptr(gP), _lib.ptr(gw), C.byref(gb)))
            assert abs(ls.value - ref["loss"]) <= DEC_TOL * abs(ref["loss"])
            assert max_rel(gP, ref["gP"]) <= 1e-9 and max_rel(gw, ref["gw"]) <= 1e-9
        out = np.zeros(n)
        _lib.check(lib.nimfm_fm_decision_function_host(ctx, h, n, d, _lib.ptr(csr.data), _lib.ptr(csr.indices),
                                                       _lib.ptr(csr.indptr), chunk, _lib.ptr(out)))
        assert np.array_equal(out, fm.decisionFunction(csr_ds(csr)))
    finally:
        lib.nimfm_fm_free(ctx, h)
        if memory == "registered":
            for a in arrays:
                lib.nimfm_host_unregister(ctx, _lib.ptr(a))


def test_decision_function_errors():
    X = make_dense(5, 6, 1)
    csr = CSR.from_dense(X)
    P, w, _ = make_fm_params(7, 2, 3, "explicit", True, seed=0)   # wrong nFeatures
    fm = make_fm(2, 3, "explicit", True, True, P, w, 0.0)
    with pytest.raises(ValueError):
        fm.decisionFunction(csr_ds(csr))
    fm2 = nf.newFactorizationMachine(nf.regression)
    with pytest.raises(nf.NotFittedError):
        fm2.decisionFunction(csr_ds(csr))


# ---------------------------------------------------------------- K2
def dev_loss_grad(fm, ds, y, loss, rows=None, row_begin=0, n_rows=None, mb=None):
    lib, ctx = _lib.load(), _lib.ctx()
    ds.set_targets(y)
    h = fm._to_device(ds.nFeatures)
    try:
        n_rows = ds.nSamples if n_rows is None else n_rows
        idx = None if rows is None else _lib.i64(rows)
        if idx is not None:
            n_rows = len(idx)
        mb = n_rows if mb is None else mb
        ls = C.c_double()
        _lib.check(lib.nimfm_fm_loss_grad(ctx, h, ds.handle(), loss.kind, loss.threshold, row_begin, n_rows,
                                          _lib.ptr(idx), mb, 1, 0, C.byref(ls)))
        gP = np.zeros_like(fm.P)
        gw = np.zeros(ds.nFeatures)
        gb = C.c_double()
        _lib.check(lib.nimfm_fm_get_grads(ctx, h, _lib.ptr(gP), _lib.ptr(gw), C.byref(gb)))
    finally:
        lib.nimfm_fm_free(ctx, h)
    return ls.value, gP, gw, gb.value


@pytest.mark.parametrize("degree,fit_lower", [(2, "explicit"), (3, "explicit"), (3, "augment"), (3, "none"),
                                              (4, "explicit"), (5, "augment")])
@pytest.mark.parametrize("loss_name", ["squared", "logistic", "squared_hinge"])
def test_loss_grad_matches_oracle(oracle, degree, fit_lower, loss_name):
    n, d, k = 80, 8, 4                      # tests/test_sgd.nim:10-13
    X = make_dense(n, d, 9, density=0.6, positive=False)
    rng = np.random.default_rng(degree)
    y = np.sign(rng.standard_normal(n)) if loss_name != "squared" else rng.standard_normal(n)
    csr = CSR.from_dense(X)
    P, w, nA = make_fm_params(d, degree, k, fit_lower, True, seed=degree + 3, scale=0.3)
    fm = make_fm(degree, k, fit_lower, True, True, P, w, 0.2)
    loss = {"squared": nf.Squared(), "logistic": nf.Logistic(), "squared_hinge": nf.SquaredHinge()}[loss_name]
    ls, gP, gw, gb = dev_loss_grad(fm, csr_ds(csr), y, loss)
    ref = oracle.fm_loss_grad(csr, y, P, w, 0.2, degree, loss_name)
    assert abs(ls - ref["loss"]) <= 1e-10 * max(1.0, abs(ref["loss"]))
    assert max_rel(gP, ref["gP"]) <= 1e-9
    assert max_rel(gw, ref["gw"]) <= 1e-9
    assert abs(gb - ref["gb"]) <= 1e-10 * max(1.0, abs(ref["gb"]))


def test_loss_grad_row_list_and_wrap(oracle):
    """explicit row ids (shuffled minibatch) and the cyclic cursor (rowBegin + q) mod n"""
    n, d, k, degree = 50, 12, 16, 3
    X = make_dense(n, d, 2, density=0.5, positive=False)
    y = np.random.default_rng(1).standard_normal(n)
    csr = CSR.from_dense(X)
    P, w, _ = make_fm_params(d, degree, k, "explicit", True, seed=4, scale=0.2)
    fm = make_fm(degree, k, "explicit", True, True, P, w, 0.0)
    rows = np.random.default_rng(0).permutation(n)[:17]
    ls, gP, gw, gb = dev_loss_grad(fm, csr_ds(csr), y, nf.Squared(), rows=rows, mb=17)
    sub = oracle.csr_take_rows(csr, rows)
    ref = oracle.fm_loss_grad(sub, y[rows], P, w, 0.0, degree, "squared", mini_batch_size=17)
    assert max_rel(gP, ref["gP"]) <= 1e-9 and abs(ls - ref["loss"]) <= 1e-10 * abs(ref["loss"])
    # wrap: rows 45..49,0..4
    ls2, gP2, _, _ = dev_loss_grad(fm, csr_ds(csr), y, nf.Squared(), row_begin=45, n_rows=10, mb=10)
    wrap = np.r_[45:50, 0:5]
    ref2 = oracle.fm_loss_grad(oracle.csr_take_rows(csr, wrap), y[wrap], P, w, 0.0, degree, "squared",
                               mini_batch_size=10)
    assert max_rel(gP2, ref2["gP"]) <= 1e-9 and abs(ls2 - ref2["loss"]) <= 1e-10 * abs(ref2["loss"])


def test_grad_linearity_large():
    """size-independent property at a larger shape: the gradient is linear in the batch, so the
    gradient of rows [0,n) equals the sum over two halves (mb fixed)."""
    n, d, k, degree = 20000, 5000, 32, 3
    rng = np.random.default_rng(8)
    z = 39
    indices = np.sort(rng.integers(0, d // z, size=(n, z)) + (np.arange(z) * (d // z))[None, :], axis=1)
    data = rng.random((n, z))
    ds = nf.newCSRDataset(data.ravel(), indices.ravel(), np.arange(n + 1) * z, n, d)
    y = np.sign(rng.standard_normal(n))
    P = rng.standard_normal((2, k, d)) * 0.05
    w = rng.standard_normal(d) * 0.05
    fm = make_fm(degree, k, "explicit", True, True, P, w, 0.0, task=nf.classification)
    ls, gP, gw, gb = dev_loss_grad(fm, ds, y, nf.Logistic(), mb=n)
    lsa, gPa, gwa, gba = dev_loss_grad(fm, ds, y, nf.Logistic(), row_begin=0, n_rows=n // 2, mb=n)
    lsb, gPb, gwb, gbb = dev_loss_grad(fm, ds, y, nf.Logistic(), row_begin=n // 2, n_rows=n - n // 2, mb=n)
    assert abs(ls - (lsa + lsb)) <= 1e-10 * abs(ls)
    assert max_rel(gPa + gPb, gP) <= 1e-9
    assert max_rel(gwa + gwb, gw) <= 1e-9
    assert abs(gb - (gba + gbb)) <= 1e-10 * max(abs(gb), 1e-3)


# ---------------------------------------------------------------- MBPSGD
def objective(oracle, csr, y, P, w, b, degree, loss_name, alpha0, alpha, beta):
    yp = oracle.fm_decision_function(csr, P, w, b, degree)
    return float(np.mean(oracle.loss_vec(loss_name, y, yp))) + oracle.regularization(P, w, b, alpha0, alpha, beta)


def make_reg(reg):
    return {"identity": nf.newL1, "l1": nf.newL1, "l21": nf.newL21, "squaredl12": nf.newSquaredL12,
            "squaredl12_rows": lambda: nf.newSquaredL12(transpose=False)}[reg]()


@pytest.mark.parametrize("degree,fit_lower,reg", [(2, "explicit", "identity"), (3, "explicit", "identity"),
                                                  (3, "augment", "l1"), (4, "none", "identity"),
                                                  (2, "explicit", "squaredl12"), (2, "augment", "squaredl12"),
                                                  (2, "explicit", "squaredl12_rows"), (3, "explicit", "l21"),
                                                  (2, "none", "l21")])
@pytest.mark.parametrize("fit_linear,fit_intercept", [(True, True), (False, True), (True, False)])
def test_mbpsgd_objective_matches_oracle(oracle, degree, fit_lower, reg, fit_linear, fit_intercept):
    """identity prox == any regulariser at gamma=0 (the default SquaredL12 only exists for degree 2,
    squaredl12.nim:103-106, so the degree-3/4 identity cases go through L1 with gamma=0)"""
    n, d, k = 80, 8, 4
    X = make_dense(n, d, 13, density=0.6, positive=False)
    y = np.sign(np.random.default_rng(2).standard_normal(n))
    csr = CSR.from_dense(X)
    P, w, nA = make_fm_params(d, degree, k, fit_lower, fit_linear, seed=11, scale=0.1)
    gamma = {"identity": 0.0, "l1": 1e-3, "l21": 5e-2, "squaredl12": 2e-1, "squaredl12_rows": 2e-1}[reg]
    kw = dict(eta0=0.1, alpha0=1e-6, alpha=1e-3, beta=1e-4, gamma=gamma)
    # the model is injected with warmStart=true, so MBPSGD.it keeps its constructor value 0
    # (minibatch_psgd.nim:62,151-152); the oracle is started from the same counter
    ref = oracle.mbpsgd_fit(csr, y, P, w, 0.0, degree, "logistic", fit_linear, fit_intercept, max_iter=5,
                            reg=reg, mini_batch_size=7, it=0, **kw)
    fm = make_fm(degree, k, fit_lower, fit_linear, fit_intercept, P, w, 0.0, task=nf.classification)
    opt = nf.newMBPSGD(maxIter=5, loss=nf.Logistic(), reg=make_reg(reg),
                       miniBatchSize=7, verbose=0, tol=0.0, shuffle=False, **kw)
    opt.fit(csr_ds(csr), y, fm)
    np.testing.assert_allclose(opt.history, ref["epoch_loss"], rtol=OBJ_TOL)
    if gamma > 0:   # the prox really acted: same sparsity pattern as the oracle, and some zeros
        assert np.array_equal(fm.P == 0.0, ref["P"] == 0.0)
        assert np.count_nonzero(ref["P"] == 0.0) > 0
    o_ref = objective(oracle, csr, y, ref["P"], ref["w"], ref["intercept"], degree, "logistic", 1e-6, 1e-3, 1e-4)
    o_dev = objective(oracle, csr, y, fm.P, fm.w, fm.intercept, degree, "logistic", 1e-6, 1e-3, 1e-4)
    assert abs(o_dev - o_ref) <= OBJ_TOL * abs(o_ref)
    assert max_rel(fm.P, ref["P"]) <= 1e-8
    assert max_rel(fm.w, ref["w"]) <= 1e-8
    assert opt.it == ref["it"]


@pytest.mark.parametrize("degree,fit_lower", [(2, "explicit"), (3, "explicit"), (3, "augment"), (2, "none")])
@pytest.mark.parametrize("k", [8, 32])
@pytest.mark.parametrize("fit_linear,fit_intercept,shuffle", [(True, True, False), (False, True, True), (True, False, True)])
def test_mbpsgd_lazy_epoch_matches_oracle(oracle, monkeypatch, degree, fit_lower, k, fit_linear, fit_intercept, shuffle):
    """the lazy epoch (touched features only; pending L2 shrink folded into x by the row kernel, K3b) gives
    the reference's iterates (minibatch_psgd.nim:91-124): sparse ragged rows so that most features sit out
    most minibatches, strong L2 so that the skipped shrink steps are visible; the "optimal" schedule gives
    every step its own eta, hence its own shrink factor"""
    n, d = 240, 150
    csr = ragged_csr(n, d, 23, 6)
    y = np.sign(np.random.default_rng(6).standard_normal(n))
    P, w, _ = make_fm_params(d, degree, k, fit_lower, fit_linear, seed=12, scale=0.1)
    if not fit_linear:   # a frozen, nonzero w still enters every prediction and must not be shrunk (params.nim:90-98)
        w = np.random.default_rng(77).standard_normal(d) * 0.1
    kw = dict(eta0=0.3, alpha0=1e-3, alpha=5e-2, beta=8e-2, gamma=0.0)
    perms = None
    if shuffle:   # the permutations the host mirror will draw (initial shuffle + one per wrap-around)
        fm0 = make_fm(degree, k, fit_lower, fit_linear, fit_intercept, P, w, 0.1, task=nf.classification)
        rng = np.random.default_rng(fm0.randomState)
        idx = np.arange(n)
        perms = []
        for _ in range(9):
            rng.shuffle(idx)
            perms.append(idx.copy())
        perms = np.array(perms)
    ref = oracle.mbpsgd_fit(csr, y, P, w, 0.1, degree, "logistic", fit_linear, fit_intercept, max_iter=4,
                            reg="identity", mini_batch_size=9, it=0, perms=perms, **kw)
    got = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("NIMFM_MBPSGD_LAZY", mode)
        fm = make_fm(degree, k, fit_lower, fit_linear, fit_intercept, P, w, 0.1, task=nf.classification)
        opt = nf.newMBPSGD(maxIter=4, loss=nf.Logistic(), reg=nf.L1(), miniBatchSize=9, verbose=0, tol=0.0,
                           shuffle=shuffle, **kw)
        before = _lib.launch_count()
        opt.fit(csr_ds(csr), y, fm)
        got[mode] = (fm, opt, _lib.launch_count() - before)
        np.testing.assert_allclose(opt.history, ref["epoch_loss"], rtol=OBJ_TOL)
        assert max_rel(fm.P, ref["P"]) <= 1e-9 and max_rel(fm.w, ref["w"]) <= 1e-9
        assert abs(fm.intercept - ref["intercept"]) <= 1e-9 * max(abs(ref["intercept"]), 1e-3)
        assert opt.it == ref["it"]
    # the lazy epoch really ran: 2 launches per minibatch instead of 4
    assert got["1"][2] < got["0"][2]
    assert max_rel(got["1"][0].P, got["0"][0].P) <= 1e-11


def test_mbpsgd_default_regulariser_is_degree2_only():
    """newMBPSGD's default reg is SquaredL12 (minibatch_psgd.nim:26-27) whose initSGD raises for any
    other degree (squaredl12.nim:103-106), whatever gamma is"""
    csr = CSR.from_dense(make_dense(10, 5, 1))
    P, w, _ = make_fm_params(5, 3, 2, "explicit", True, seed=1)
    fm = make_fm(3, 2, "explicit", True, True, P, w, 0.0)
    with pytest.raises(ValueError, match="SquaredL12 supports only degree=2"):
        nf.newMBPSGD(maxIter=1, gamma=0.0, verbose=0).fit(csr_ds(csr), np.zeros(10), fm)


@pytest.mark.parametrize("reg,gamma", [("squaredl12", 0.5), ("squaredl12_rows", 0.5), ("l21", 0.05)])
def test_mbpsgd_prox_wide_model(oracle, reg, gamma):
    """wider shapes for the prox kernels: 300 features (several blocks of the column sweep), k=40
    (two elements per lane in the row-wise kernels), ragged rows"""
    n, d, k = 120, 300, 40
    csr = ragged_csr(n, d, 31, 12)
    y = np.random.default_rng(5).standard_normal(n)
    P, w, _ = make_fm_params(d, 2, k, "explicit", True, seed=7, scale=0.05)
    kw = dict(eta0=0.2, alpha0=1e-6, alpha=1e-3, beta=1e-3, gamma=gamma)
    ref = oracle.mbpsgd_fit(csr, y, P, w, 0.0, 2, "squared", max_iter=3, reg=reg, mini_batch_size=16, it=0, **kw)
    fm = make_fm(2, k, "explicit", True, True, P, w, 0.0)
    opt = nf.newMBPSGD(maxIter=3, reg=make_reg(reg), miniBatchSize=16, verbose=0, tol=0.0, shuffle=False, **kw)
    opt.fit(csr_ds(csr), y, fm)
    np.testing.assert_allclose(opt.history, ref["epoch_loss"], rtol=OBJ_TOL)
    assert np.array_equal(fm.P == 0.0, ref["P"] == 0.0) and np.count_nonzero(ref["P"] == 0.0) > 0
    assert max_rel(fm.P, ref["P"]) <= 1e-8 and max_rel(fm.w, ref["w"]) <= 1e-8


def test_mbpsgd_default_minibatch_and_shuffle_contract(oracle):
    """default miniBatchSize = d*n div nnz (minibatch_psgd.nim:157-165); with shuffle the host supplies
    the sample order: replay it through the oracle's `perms` and compare."""
    n, d, k, degree = 60, 10, 3, 2
    X = make_dense(n, d, 17, density=0.3)
    y = np.random.default_rng(3).standard_normal(n)
    csr = CSR.from_dense(X)
    P, w, _ = make_fm_params(d, degree, k, "explicit", True, seed=2)
    fm = make_fm(degree, k, "explicit", True, True, P, w, 0.0)
    opt = nf.newMBPSGD(maxIter=3, gamma=0.0, verbose=0, tol=0.0, shuffle=True)
    ds = csr_ds(csr)
    mb, inner = opt.resolve_sizes(ds)
    assert mb == max((d * n) // len(csr.data), 1) and inner == (n - 1) // mb + 1
    # reproduce the permutations the host will draw
    rng = np.random.default_rng(fm.randomState)
    idx = np.arange(n)
    perms = []
    rng.shuffle(idx)
    perms.append(idx.copy())
    for _ in range(8):
        rng.shuffle(idx)
        perms.append(idx.copy())
    opt.fit(ds, y, fm)
    ref = oracle.mbpsgd_fit(csr, y, P, w, 0.0, degree, "squared", max_iter=3, gamma=0.0, perms=np.array(perms), it=0)
    np.testing.assert_allclose(opt.history, ref["epoch_loss"], rtol=OBJ_TOL)
    assert max_rel(fm.P, ref["P"]) <= 1e-8


# ---------------------------------------------------------------- AdaGrad
@pytest.mark.parametrize("degree,fit_lower", [(2, "explicit"), (3, "explicit"), (3, "augment"), (4, "none")])
@pytest.mark.parametrize("mb", [1, 8])
def test_adagrad_matches_oracle(oracle, degree, fit_lower, mb):
    """mb=1: the reference's sequential semantics (adagrad.nim:164-181); mb=8: synchronous minibatch"""
    n, d, k = 80, 8, 4                      # tests/test_adagrad.nim:10-13
    X = make_dense(n, d, 19, density=0.6, positive=False)
    y = np.random.default_rng(4).standard_normal(n)
    csr = CSR.from_dense(X)
    P, w, nA = make_fm_params(d, degree, k, fit_lower, True, seed=5, scale=0.1)
    w = np.zeros(d)
    ref = oracle.adagrad_fit(csr, y, P, w, 0.0, degree, "squared", True, True, max_iter=3, mini_batch_size=mb)
    fm = make_fm(degree, k, fit_lower, True, True, P, w, 0.0)
    opt = nf.newAdaGrad(maxIter=3, verbose=0, tol=0.0, shuffle=False, miniBatchSize=mb)
    opt.fit(csr_ds(csr), y, fm)
    np.testing.assert_allclose([h[1] for h in opt.history], ref["loss"], rtol=OBJ_TOL)
    np.testing.assert_allclose([h[0] for h in opt.history], ref["viol"], rtol=1e-8)
    # (degree 4 / fitLower=none collapses to |P| ~ 1e-20 where relative error is meaningless: atol)
    np.testing.assert_allclose(fm.P, ref["P"], rtol=1e-8, atol=1e-13)
    np.testing.assert_allclose(fm.w, ref["w"], rtol=1e-8, atol=1e-13)
    assert abs(fm.intercept - ref["intercept"]) <= 1e-9
    assert opt.it == ref["it"]
    np.testing.assert_allclose(opt.g_sum["P"], ref["state"]["gsP"], rtol=1e-8, atol=1e-14)
    np.testing.assert_allclose(opt.g_norm["P"], ref["state"]["gnP"], rtol=1e-8, atol=1e-14)


@pytest.mark.parametrize("route", ["pipe", "staged", "0"])
@pytest.mark.parametrize("shuffle", [False, True])
def test_adagrad_sequential_routes_agree(oracle, monkeypatch, route, shuffle):
    """miniBatchSize=1 has three device routes (adagrad_seq.cuh pipelined / staged kernels, the minibatch pipeline
    with one-row batches): each must give the reference's per-sample result (adagrad.nim:164-181), shuffled or not"""
    monkeypatch.setenv("NIMFM_ADAGRAD_SEQ", route)
    n, d, k, degree = 150, 40, 8, 3
    X = make_dense(n, d, 23, density=0.3, positive=False)
    y = np.sign(np.random.default_rng(6).standard_normal(n))
    csr = CSR.from_dense(X)
    P, w, _ = make_fm_params(d, degree, k, "explicit", True, seed=8, scale=0.1)
    fm = make_fm(degree, k, "explicit", True, True, P, w, 0.0)
    opt = nf.newAdaGrad(maxIter=3, loss=nf.Logistic(), verbose=0, tol=0.0, shuffle=shuffle, miniBatchSize=1)
    perms = [np.random.default_rng(30 + e).permutation(n).astype(np.int64) for e in range(3)] if shuffle else []
    opt.fit(csr_ds(csr), y, fm, perms=perms if shuffle else None)
    ref = oracle.adagrad_fit(csr, y, P, w, 0.0, degree, "logistic", True, True, max_iter=3, mini_batch_size=1,
                             perms=np.array(perms) if shuffle else None)
    np.testing.assert_allclose([h[1] for h in opt.history], ref["loss"], rtol=OBJ_TOL)
    np.testing.assert_allclose(fm.P, ref["P"], rtol=1e-8, atol=1e-13)
    np.testing.assert_allclose(fm.w, ref["w"], rtol=1e-8, atol=1e-13)
    assert abs(fm.intercept - ref["intercept"]) <= 1e-9


def test_adagrad_max_threads_maps_to_synchronous_minibatch(oracle):
    """fit(..., maxThreads=T) (the reference's Hogwild entry point) runs the deterministic synchronous
    minibatch of T samples"""
    n, d, k, degree = 96, 9, 4, 2
    X = make_dense(n, d, 3, density=0.5, positive=False)
    y = np.random.default_rng(2).standard_normal(n)
    csr = CSR.from_dense(X)
    P, w, _ = make_fm_params(d, degree, k, "explicit", True, seed=4)
    ref = oracle.adagrad_fit(csr, y, P, w, 0.0, degree, "squared", max_iter=2, mini_batch_size=8)
    fm = make_fm(degree, k, "explicit", True, True, P, w, 0.0)
    opt = nf.newAdaGrad(maxIter=2, verbose=0, tol=0.0, shuffle=False)
    opt.fit(csr_ds(csr), y, fm, maxThreads=8)
    assert max_rel(fm.P, ref["P"]) <= 1e-8 and max_rel(fm.w, ref["w"]) <= 1e-8


def test_adagrad_warm_start_equals_cold(oracle):
    """tests/test_adagrad.nim:58-90: 2 x (warm-started) epochs == one run of the total length"""
    n, d, k, degree = 40, 8, 4, 3
    X = make_dense(n, d, 23, density=0.6)
    y = np.random.default_rng(5).standard_normal(n)
    csr = CSR.from_dense(X)
    P, w, _ = make_fm_params(d, degree, k, "explicit", True, seed=6)
    fm_cold = make_fm(degree, k, "explicit", True, True, P, w * 0, 0.0)
    nf.newAdaGrad(maxIter=4, verbose=0, tol=0.0, shuffle=False).fit(csr_ds(csr), y, fm_cold)
    fm_warm = make_fm(degree, k, "explicit", True, True, P, w * 0, 0.0)
    opt = nf.newAdaGrad(maxIter=2, verbose=0, tol=0.0, shuffle=False)
    opt.fit(csr_ds(csr), y, fm_warm)
    fm_warm.warmStart = True
    it_mid = opt.it
    opt.fit(csr_ds(csr), y, fm_warm)
    assert opt.it == 2 * (it_mid - 1) + 1
    np.testing.assert_allclose(fm_warm.P, fm_cold.P, rtol=1e-8, atol=1e-8)
    np.testing.assert_allclose(fm_warm.w, fm_cold.w, rtol=1e-8, atol=1e-8)


# ---------------------------------------------------------------- bookkeeping (bit-exact)
def test_dataset_bookkeeping_bit_exact(oracle):
    X = make_dense(37, 19, 29, density=0.35)
    csr = CSR.from_dense(X)
    ds = csr_ds(csr)
    data, indices, indptr, _ = ds.download()
    assert np.array_equal(data, csr.data) and np.array_equal(indices, csr.indices) and np.array_equal(indptr, csr.indptr)
    assert ds.info()["nnz"] == len(csr.data) == np.count_nonzero(X)
    csc_ref = oracle.csr_to_csc(csr)
    csc = ds.toCSCDataset()                       # sparse.nim:510-527 on the library side
    assert np.array_equal(csc.indptr, csc_ref.indptr)
    assert np.array_equal(csc.indices, csc_ref.indices)
    assert np.array_equal(csc.data, csc_ref.data)
    back = csc.toCSRDataset()
    assert np.array_equal(back.indptr, csr.indptr) and np.array_equal(back.indices, csr.indices)
    assert np.array_equal(back.data, csr.data)
    # row shard == X[slice] (sparse.nim:263-290)
    lib, ctx = _lib.load(), _lib.ctx()
    h = C.c_void_p()
    _lib.check(lib.nimfm_csr_upload(ctx, csr.n, csr.d, _lib.ptr(csr.data), _lib.ptr(csr.indices),
                                    _lib.ptr(csr.indptr), None, 0, 10, 25, C.byref(h)))
    shard = nf.CSRDataset.__new__(nf.CSRDataset)
    shard._handle, shard._n, shard._d = h, 15, csr.d
    sd, si, sp, _ = nf.dataset.BaseDataset.download(shard)
    ref = oracle.csr_take_rows(csr, np.arange(10, 25))
    assert np.array_equal(sp, ref.indptr) and np.array_equal(si, ref.indices) and np.array_equal(sd, ref.data)
    shard.free()
    with pytest.raises(ValueError):               # out-of-range column index is rejected at upload
        bad = nf.newCSRDataset([1.0], [99], [0, 1], 1, 5)
        bad.handle()
