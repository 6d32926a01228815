"""Parity of the FFM kernels (K10/K11) and of the sequential SGD kernels (K6) against the CPU oracle,
through the C ABI.  Shapes follow tests/test_sgd_ffm.nim:10-14 (n=80, d=20, 5 fields, k=4) and
tests/test_sgd.nim:10-13 (n=80, d=8, k=4)."""
import ctypes as C

import numpy as np
import pytest

import nimfm_b200 as nf
from nimfm_b200 import _lib
from oracle import bruteforce as bf
from oracle.oracle import CSR
from helpers import make_dense, make_fm_params, make_field_csr, max_rel

pytestmark = pytest.mark.gpu

DEC_TOL, OBJ_TOL = 1e-10, 1e-8


def field_ds(csr):
    return nf.newCSRFieldDataset(csr.data, csr.indices, csr.indptr, csr.fields, csr.n, csr.d, csr.n_fields)


def make_ffm(P, w, b, fit_linear=True, fit_intercept=True, task=nf.regression):
    m = nf.newFieldAwareFactorizationMachine(task, nComponents=P.shape[2], fitLinear=fit_linear,
                                             fitIntercept=fit_intercept, warmStart=True)
    m.P, m.w, m.intercept, m.isInitialized = P.copy(), w.copy(), b, True
    return m


def one_per_field_csr(n, n_fields, per_field, seed):
    """libffm / C5 shape: exactly one feature per field, field f owns ids [f*per_field, (f+1)*per_field)"""
    rng = np.random.default_rng(seed)
    idx = rng.integers(0, per_field, size=(n, n_fields)) + (np.arange(n_fields) * per_field)[None, :]
    data = np.where(rng.random((n, n_fields)) < 0.5, 1.0, rng.random((n, n_fields)))
    csr = CSR(data.ravel(), idx.ravel(), np.arange(n + 1) * n_fields, n, n_fields * per_field,
              fields=np.tile(np.arange(n_fields), n), n_fields=n_fields)
    return csr


@pytest.mark.parametrize("k", [4, 8, 5])
def test_ffm_decision_function(oracle, k):
    n, d, nF = 80, 20, 5
    X, csr, field_of = make_field_csr(n, d, nF, 7)
    rng = np.random.default_rng(k)
    P = rng.standard_normal((nF, d, k)) * 0.3
    w = rng.standard_normal(d) * 0.1
    m = make_ffm(P, w, -0.2)
    got = m.decisionFunction(field_ds(csr))
    assert max_rel(got, oracle.ffm_decision_function(csr, P, w, -0.2)) <= DEC_TOL
    # and straight against the definition (tests/model/ffm_slow.nim:38-56)
    np.testing.assert_allclose(got[:10], bf.ffm_decision_function(X[:10], field_of, P, w, -0.2), rtol=1e-9, atol=1e-12)


def test_ffm_decision_function_one_feature_per_field(oracle):
    n, nF, per, k = 500, 39, 50, 8            # C5 row shape: 39 fields, rank 8
    csr = one_per_field_csr(n, nF, per, 3)
    rng = np.random.default_rng(0)
    P = rng.standard_normal((nF, nF * per, k)) * 0.1
    w = rng.standard_normal(nF * per) * 0.1
    m = make_ffm(P, w, 0.3)
    got = m.decisionFunction(field_ds(csr))
    assert max_rel(got, oracle.ffm_decision_function(csr, P, w, 0.3)) <= DEC_TOL


def test_ffm_errors():
    X, csr, _ = make_field_csr(10, 20, 5, 1)
    P = np.zeros((4, 20, 3))                 # wrong nFields
    m = make_ffm(P, np.zeros(20), 0.0)
    with pytest.raises(ValueError):
        m.decisionFunction(field_ds(csr))


def ffm_dev_loss_grad(m, ds, y, loss, mb=None):
    lib, ctx = _lib.load(), _lib.ctx()
    ds.set_targets(y)
    h = m._to_device(ds)
    try:
        n = ds.nSamples
        ls = C.c_double()
        _lib.check(lib.nimfm_ffm_loss_grad(ctx, h, ds.handle(), loss.kind, loss.threshold, 0, n, None,
                                           n if mb is None else mb, 1, 0, C.byref(ls)))
        gP, gw, gb = np.zeros_like(m.P), np.zeros(ds.nFeatures), C.c_double()
        _lib.check(lib.nimfm_ffm_get_grads(ctx, h, _lib.ptr(gP), _lib.ptr(gw), C.byref(gb)))
    finally:
        lib.nimfm_ffm_free(ctx, h)
    return ls.value, gP, gw, gb.value


@pytest.mark.parametrize("shape", ["dense_fields", "one_per_field"])
@pytest.mark.parametrize("loss_name", ["squared", "logistic"])
def test_ffm_loss_grad(oracle, shape, loss_name):
    if shape == "dense_fields":
        X, csr, _ = make_field_csr(80, 20, 5, 11)
        k = 4
    else:
        csr = one_per_field_csr(200, 13, 20, 5)
        k = 8
    rng = np.random.default_rng(2)
    P = rng.standard_normal((csr.n_fields, csr.d, k)) * 0.2
    w = rng.standard_normal(csr.d) * 0.1
    y = rng.standard_normal(csr.n) if loss_name == "squared" else np.sign(rng.standard_normal(csr.n))
    m = make_ffm(P, w, 0.1)
    loss = nf.Squared() if loss_name == "squared" else nf.Logistic()
    ls, gP, gw, gb = ffm_dev_loss_grad(m, field_ds(csr), y, loss)
    ref = oracle.ffm_loss_grad(csr, y, P, w, 0.1, loss_name)
    assert abs(ls - ref["loss"]) <= 1e-10 * max(1.0, abs(ref["loss"]))
    assert max_rel(gP, ref["gP"]) <= 1e-9
    assert max_rel(gw, ref["gw"]) <= 1e-9
    assert abs(gb - ref["gb"]) <= 1e-10 * max(1.0, abs(ref["gb"]))


@pytest.mark.parametrize("mb", [1, 8])
def test_ffm_adagrad(oracle, mb):
    """tests/test_adagrad_ffm.nim: naive comparison with shuffle=false (mb=1 == reference semantics)"""
    X, csr, _ = make_field_csr(80, 20, 5, 13)
    k = 4
    rng = np.random.default_rng(3)
    P = rng.standard_normal((5, 20, k)) * 0.1
    w = np.zeros(20)
    y = rng.standard_normal(80)
    ref = oracle.ffm_adagrad_fit(csr, y, P, w, 0.0, "squared", max_iter=3, mini_batch_size=mb)
    m = make_ffm(P, w, 0.0)
    opt = nf.newAdaGrad(maxIter=3, verbose=0, tol=0.0, shuffle=False, miniBatchSize=mb)
    opt.fit(field_ds(csr), y, m)
    np.testing.assert_allclose([h[1] for h in opt.history], ref["loss"], rtol=OBJ_TOL)
    np.testing.assert_allclose([h[0] for h in opt.history], ref["viol"], rtol=1e-8)
    np.testing.assert_allclose(m.P, ref["P"], rtol=1e-8, atol=1e-13)
    np.testing.assert_allclose(m.w, ref["w"], rtol=1e-8, atol=1e-13)
    assert abs(m.intercept - ref["intercept"]) <= 1e-9
    assert opt.it == ref["it"]


def test_ffm_sgd(oracle):
    """tests/test_sgd_ffm.nim:87-115"""
    X, csr, _ = make_field_csr(80, 20, 5, 17)
    k = 4
    rng = np.random.default_rng(4)
    P = rng.standard_normal((5, 20, k)) * 0.1
    w = rng.standard_normal(20) * 0.1
    y = rng.standard_normal(80)
    ref = oracle.ffm_sgd_fit(csr, y, P, w, 0.0, "squared", max_iter=4)
    m = make_ffm(P, w, 0.0)
    opt = nf.newSGD(maxIter=4, verbose=0, tol=0.0, shuffle=False)
    opt.fit(field_ds(csr), y, m)
    np.testing.assert_allclose([h[1] for h in opt.history], ref["loss"], rtol=OBJ_TOL)
    np.testing.assert_allclose([h[0] for h in opt.history], ref["viol"], rtol=1e-8)
    np.testing.assert_allclose(m.P, ref["P"], rtol=1e-8, atol=1e-13)
    np.testing.assert_allclose(m.w, ref["w"], rtol=1e-8, atol=1e-13)
    assert abs(m.intercept - ref["intercept"]) <= 1e-9


@pytest.mark.parametrize("degree,fit_lower", [(2, "explicit"), (3, "explicit"), (3, "augment"), (4, "none"), (4, "explicit")])
@pytest.mark.parametrize("sched", ["optimal", "constant", "invscaling"])
def test_fm_sgd(oracle, degree, fit_lower, sched):
    """tests/test_sgd.nim:92-126: SGD with lazy scaling and the step-size schedules of sgd.nim:60-69
    (pegasos is left out: eta*reg == 1 at it == 1 zeroes scaling_P, and the reference itself goes NaN)"""
    n, d, k = 80, 8, 4
    X = make_dense(n, d, 21, density=0.5, positive=False)
    y = np.random.default_rng(5).standard_normal(n)
    csr = CSR.from_dense(X)
    P, w, nA = make_fm_params(d, degree, k, fit_lower, True, seed=7, scale=0.1)
    kw = dict(eta0=0.01, alpha0=1e-6, alpha=1e-3, beta=1e-3, power=0.75 if sched == "invscaling" else 1.0)
    ref = oracle.sgd_fit(csr, y, P, w, 0.0, degree, "squared", max_iter=4, scheduling=sched, **kw)
    fm = nf.newFactorizationMachine(nf.regression, degree=degree, nComponents=k, fitLower=fit_lower, warmStart=True)
    fm.P, fm.w, fm.intercept, fm.isInitialized = P.copy(), w.copy(), 0.0, True
    opt = nf.newSGD(maxIter=4, verbose=0, tol=0.0, shuffle=False, scheduling=sched, **kw)
    opt.fit(nf.newCSRDataset(csr.data, csr.indices, csr.indptr, n, d), y, fm)
    np.testing.assert_allclose([h[1] for h in opt.history], ref["loss"], rtol=OBJ_TOL)
    np.testing.assert_allclose([h[0] for h in opt.history], ref["viol"], rtol=1e-8)
    np.testing.assert_allclose(fm.P, ref["P"], rtol=1e-8, atol=1e-13)
    np.testing.assert_allclose(fm.w, ref["w"], rtol=1e-8, atol=1e-13)
    assert abs(fm.intercept - ref["intercept"]) <= 1e-9
    assert opt.it == ref["it"]


def test_fm_sgd_reset_scaling_and_perms(oracle):
    """strong L2 + large eta drive scaling_P below 1e-9 so resetScaling (sgd.nim:116-131) fires; the
    host-supplied permutation replaces Nim's shuffle"""
    n, d, k, degree = 60, 6, 3, 2
    X = make_dense(n, d, 23, density=0.7, positive=False)
    y = np.random.default_rng(6).standard_normal(n)
    csr = CSR.from_dense(X)
    P, w, _ = make_fm_params(d, degree, k, "explicit", True, seed=8, scale=0.1)
    kw = dict(eta0=0.5, alpha0=1e-6, alpha=0.6, beta=0.6, scheduling="constant")
    perms = np.array([np.random.default_rng(s).permutation(n) for s in range(3)])
    ref = oracle.sgd_fit(csr, y, P, w, 0.0, degree, "squared", max_iter=3, perms=perms, **kw)
    fm = nf.newFactorizationMachine(nf.regression, degree=degree, nComponents=k, warmStart=True)
    fm.P, fm.w, fm.intercept, fm.isInitialized = P.copy(), w.copy(), 0.0, True
    opt = nf.newSGD(maxIter=3, verbose=0, tol=0.0, **kw)
    opt.fit(nf.newCSRDataset(csr.data, csr.indices, csr.indptr, n, d), y, fm, perms=perms)
    np.testing.assert_allclose([h[1] for h in opt.history], ref["loss"], rtol=OBJ_TOL)
    np.testing.assert_allclose(fm.P, ref["P"], rtol=1e-8, atol=1e-13)
    np.testing.assert_allclose(fm.w, ref["w"], rtol=1e-8, atol=1e-13)


# ---------------------------------------------------------------- kernel-variant coverage
def ragged_field_csr(n, d, n_fields, seed, max_nnz):
    """rows with 0..max_nnz nonzeros (every 6th row empty, one row of length 1), random fields"""
    rng = np.random.default_rng(seed)
    data, indices, fields, indptr = [], [], [], [0]
    for i in range(n):
        z = 0 if i % 6 == 0 else (1 if i == 1 else int(rng.integers(2, max_nnz + 1)))
        cols = np.sort(rng.choice(d, size=min(z, d), replace=False))
        indices.extend(cols.tolist())
        data.extend((rng.standard_normal(len(cols)) * 0.7).tolist())
        fields.extend(rng.integers(0, n_fields, len(cols)).tolist())
        indptr.append(len(indices))
    return CSR(data, indices, indptr, n, d, fields=np.array(fields, np.int64), n_fields=n_fields)


@pytest.mark.parametrize("k", [4, 8, 16, 32])
@pytest.mark.parametrize("max_nnz", [9, 64, 90])
@pytest.mark.parametrize("variant", ["default", "block"])
def test_ffm_kernel_variants_ragged(oracle, monkeypatch, k, max_nnz, variant):
    """every compiled rank instance x the kernel forms (pair-block with the shared pair table for rows <= 64
    nonzeros, warp-per-row pair cursor beyond, staged block-per-row fallback) on ragged rows with empty rows and
    repeated fields: forward + gradient equal the oracle"""
    if variant == "block" and max_nnz * 6 * k * 8 > 200_000:
        pytest.skip("staged block kernel: slices do not fit shared memory")
    if variant != "default":
        monkeypatch.setenv("NIMFM_FFM_KERNEL", variant)
    n, d, nF = 60, 120, 6
    csr = ragged_field_csr(n, d, nF, 100 + max_nnz, max_nnz)
    rng = np.random.default_rng(k)
    P = rng.standard_normal((nF, d, k)) * 0.2
    w = rng.standard_normal(d) * 0.1
    y = rng.standard_normal(n)
    m = make_ffm(P, w, 0.05)
    got = m.decisionFunction(field_ds(csr))
    assert max_rel(got, oracle.ffm_decision_function(csr, P, w, 0.05)) <= DEC_TOL
    ls, gP, gw, gb = ffm_dev_loss_grad(m, field_ds(csr), y, nf.Squared())
    ref = oracle.ffm_loss_grad(csr, y, P, w, 0.05, "squared")
    assert abs(ls - ref["loss"]) <= 1e-10 * max(1.0, abs(ref["loss"]))
    assert max_rel(gP, ref["gP"]) <= 1e-9 and max_rel(gw, ref["gw"]) <= 1e-9


@pytest.mark.parametrize("mb", [1, 16, 200])
@pytest.mark.parametrize("variant", ["default", "block", "warp"])
def test_ffm_adagrad_one_feature_per_field(oracle, monkeypatch, mb, variant):
    """C5 row shape (one feature per field): the AdaGrad route runs on the pair kernels, which square
    per-pair contributions -- equal to the oracle's per-sample squares; the staged kernel must agree.  "warp": rows
    of 70 fields, past the pair table's 64 nonzeros, take the warp-per-row pair kernel"""
    if variant == "block":
        monkeypatch.setenv("NIMFM_FFM_KERNEL", variant)
    nF, per = (70, 3) if variant == "warp" else (13, 20)
    csr = one_per_field_csr(200, nF, per, 15)
    k = 8
    rng = np.random.default_rng(4)
    P = rng.standard_normal((nF, csr.d, k)) * 0.1
    w = np.zeros(csr.d)
    y = np.sign(rng.standard_normal(200))
    ref = oracle.ffm_adagrad_fit(csr, y, P, w, 0.0, "logistic", max_iter=3, mini_batch_size=mb)
    m = make_ffm(P, w, 0.0, task=nf.classification)
    opt = nf.newAdaGrad(maxIter=3, loss=nf.Logistic(), verbose=0, tol=0.0, shuffle=False, miniBatchSize=mb)
    opt.fit(field_ds(csr), y, m)
    np.testing.assert_allclose([h[1] for h in opt.history], ref["loss"], rtol=OBJ_TOL)
    np.testing.assert_allclose([h[0] for h in opt.history], ref["viol"], rtol=1e-8)
    np.testing.assert_allclose(m.P, ref["P"], rtol=1e-8, atol=1e-13)
    assert abs(m.intercept - ref["intercept"]) <= 1e-9


def unique_fields_ragged_csr(n, n_fields, per_field, seed):
    """rows holding a random SUBSET of the fields (each at most once; some rows empty, some with every field)"""
    rng = np.random.default_rng(seed)
    data, indices, fields, indptr = [], [], [], [0]
    for i in range(n):
        z = 0 if i % 7 == 0 else (n_fields if i % 5 == 0 else int(rng.integers(1, n_fields + 1)))
        fs = np.sort(rng.choice(n_fields, size=z, replace=False))
        indices.extend((fs * per_field + rng.integers(0, per_field, z)).tolist())
        data.extend(np.where(rng.random(z) < 0.5, 1.0, rng.standard_normal(z)).tolist())
        fields.extend(fs.tolist())
        indptr.append(len(indices))
    return CSR(data, indices, indptr, n, n_fields * per_field, fields=np.array(fields, np.int64), n_fields=n_fields)


@pytest.mark.parametrize("k", [4, 8, 16, 32])
@pytest.mark.parametrize("bulk", ["0", "1"])
def test_ffm_bulk_reduction_route(oracle, monkeypatch, k, bulk):
    """gradient blocks assembled in shared memory and added by TMA bulk reductions (NIMFM_FFM_BULK=1; the default of
    the AdaGrad mode) against the RED route (=0) and the oracle: full rows, rows with absent fields (the zero-filled
    block), empty rows; predict+grad and three AdaGrad epochs"""
    monkeypatch.setenv("NIMFM_FFM_BULK", bulk)
    nF = 13
    for csr in (one_per_field_csr(150, nF, 20, 21), unique_fields_ragged_csr(150, nF, 20, 22)):
        rng = np.random.default_rng(k)
        P = rng.standard_normal((nF, csr.d, k)) * 0.15
        w = rng.standard_normal(csr.d) * 0.1
        y = np.sign(rng.standard_normal(csr.n))
        m = make_ffm(P, w, 0.05, task=nf.classification)
        ls, gP, gw, gb = ffm_dev_loss_grad(m, field_ds(csr), y, nf.Logistic())
        ref = oracle.ffm_loss_grad(csr, y, P, w, 0.05, "logistic")
        assert abs(ls - ref["loss"]) <= 1e-10 * max(1.0, abs(ref["loss"]))
        assert max_rel(gP, ref["gP"]) <= 1e-9 and max_rel(gw, ref["gw"]) <= 1e-9
        refa = oracle.ffm_adagrad_fit(csr, y, P, np.zeros(csr.d), 0.0, "logistic", max_iter=3, mini_batch_size=32)
        ma = make_ffm(P, np.zeros(csr.d), 0.0, task=nf.classification)
        opt = nf.newAdaGrad(maxIter=3, loss=nf.Logistic(), verbose=0, tol=0.0, shuffle=False, miniBatchSize=32)
        opt.fit(field_ds(csr), y, ma)
        np.testing.assert_allclose([h[1] for h in opt.history], refa["loss"], rtol=OBJ_TOL)
        np.testing.assert_allclose(ma.P, refa["P"], rtol=1e-8, atol=1e-13)


def test_ffm_adagrad_repeated_fields_falls_back(oracle):
    """rows with two nonzeros of one field: per-sample squares need the field-bucketed kernel (the pair
    kernel would square each pair's share separately); the dispatcher must notice"""
    csr = ragged_field_csr(60, 40, 3, 7, 10)
    rng = np.random.default_rng(5)
    P = rng.standard_normal((3, 40, 4)) * 0.1
    y = rng.standard_normal(60)
    ref = oracle.ffm_adagrad_fit(csr, y, P, np.zeros(40), 0.0, "squared", max_iter=2, mini_batch_size=8)
    m = make_ffm(P, np.zeros(40), 0.0)
    opt = nf.newAdaGrad(maxIter=2, verbose=0, tol=0.0, shuffle=False, miniBatchSize=8)
    opt.fit(field_ds(csr), y, m)
    np.testing.assert_allclose(m.P, ref["P"], rtol=1e-8, atol=1e-13)
    np.testing.assert_allclose([h[1] for h in opt.history], ref["loss"], rtol=OBJ_TOL)


# ---------------------------------------------------------------- PSGD (optimizer/psgd.nim, SURVEY 8f.2)
def make_sgd_reg(reg):
    return {"l1": nf.newL1, "l21": nf.newL21, "squaredl12": nf.newSquaredL12,
            "squaredl12_rows": lambda: nf.newSquaredL12(transpose=False)}[reg]()


@pytest.mark.parametrize("degree,fit_lower,reg", [(2, "explicit", "l1"), (3, "explicit", "l1"), (4, "augment", "l1"),
                                                  (2, "none", "l21"), (3, "augment", "l21"), (3, "explicit", "l21"),
                                                  (2, "explicit", "squaredl12"), (2, "augment", "squaredl12"),
                                                  (2, "none", "squaredl12_rows")])
@pytest.mark.parametrize("fit_linear,fit_intercept", [(True, True), (False, False)])
@pytest.mark.parametrize("kernel", ["pipe", "staged"])
def test_psgd_matches_oracle(oracle, monkeypatch, degree, fit_lower, reg, fit_linear, fit_intercept, kernel):
    """tests/test_psgd_{l1,l21,squaredl12}.nim shapes (n=80, d=8, k=4): the device's PSGD against the
    literal restatement of psgd.nim (lazy L1 / L21 protocols, dense SquaredL12), shuffle=false; both forms of the
    lazy kernel (psgd.cu: pipelined, staged)"""
    if kernel == "staged" and reg.startswith("squaredl12"):
        pytest.skip("the dense SquaredL12 route has one form")
    monkeypatch.setenv("NIMFM_PSGD_KERNEL", kernel)
    from oracle.oracle import CSR as _CSR
    from helpers import make_dense, make_fm_params
    n, d, k = 80, 8, 4
    X = make_dense(n, d, 61 + degree, density=0.6, positive=False)
    y = np.random.default_rng(degree).standard_normal(n)
    csr = _CSR.from_dense(X)
    P, w, nA = make_fm_params(d, degree, k, fit_lower, fit_linear, seed=23, scale=0.2)
    kw = dict(eta0=0.05, alpha0=1e-6, alpha=1e-3, beta=1e-3, gamma=1.0 if reg == "l21" else 3e-2)
    ref = oracle.psgd_fit(csr, y, P, w, 0.1, degree, "squared", fit_linear, fit_intercept, max_iter=3, reg=reg, **kw)
    fm = nf.newFactorizationMachine(nf.regression, degree=degree, nComponents=k, fitLower=fit_lower,
                                    fitLinear=fit_linear, fitIntercept=fit_intercept, warmStart=True)
    fm.P, fm.w, fm.intercept, fm.isInitialized = P.copy(), w.copy(), 0.1, True
    opt = nf.newPSGD(maxIter=3, reg=make_sgd_reg(reg), verbose=0, tol=0.0, shuffle=False, **kw)
    opt.it = 1
    ds = nf.newCSRDataset(csr.data, csr.indices, csr.indptr, n, d)
    opt.fit(ds, y, fm)
    np.testing.assert_allclose(opt.history, ref["epoch_loss"], rtol=OBJ_TOL)
    np.testing.assert_allclose(fm.P, ref["P"], rtol=1e-8, atol=1e-13)
    np.testing.assert_allclose(fm.w, ref["w"], rtol=1e-8, atol=1e-13)
    assert abs(fm.intercept - ref["intercept"]) <= 1e-9
    assert np.array_equal(fm.P == 0.0, ref["P"] == 0.0) and opt.it == ref["it"]
    if reg in ("l1", "l21"):
        assert np.count_nonzero(ref["P"] == 0.0) > 0                  # the prox really acted


def test_psgd_permutation_logistic_and_rules(oracle):
    """host-supplied permutations, logistic loss, invscaling schedule; the default regulariser
    (SquaredL12) exists for degree 2 only"""
    from oracle.oracle import CSR as _CSR
    from helpers import make_dense, make_fm_params
    n, d, k, degree = 60, 7, 3, 2
    X = make_dense(n, d, 5, density=0.5, positive=False)
    y = np.sign(np.random.default_rng(1).standard_normal(n))
    csr = _CSR.from_dense(X)
    P, w, _ = make_fm_params(d, degree, k, "explicit", True, seed=3, scale=0.2)
    perms = np.array([np.random.default_rng(s).permutation(n) for s in range(2)])
    kw = dict(eta0=0.1, alpha0=1e-6, alpha=1e-3, beta=1e-3, gamma=1e-2)
    ref = oracle.psgd_fit(csr, y, P, w, 0.0, degree, "logistic", max_iter=2, reg="l1", scheduling="invscaling",
                          power=0.5, perms=perms, **kw)
    fm = nf.newFactorizationMachine(nf.classification, degree=degree, nComponents=k, warmStart=True)
    fm.P, fm.w, fm.intercept, fm.isInitialized = P.copy(), w.copy(), 0.0, True
    opt = nf.newPSGD(maxIter=2, loss=nf.Logistic(), reg=nf.newL1(), scheduling=nf.invscaling, power=0.5, verbose=0,
                     tol=0.0, **kw)
    opt.it = 1
    opt.fit(nf.newCSRDataset(csr.data, csr.indices, csr.indptr, n, d), y, fm, perms=perms)
    np.testing.assert_allclose(opt.history, ref["epoch_loss"], rtol=OBJ_TOL)
    np.testing.assert_allclose(fm.P, ref["P"], rtol=1e-8, atol=1e-13)
    fm3 = nf.newFactorizationMachine(nf.regression, degree=3, nComponents=2)
    with pytest.raises(ValueError, match="SquaredL12 supports only degree=2"):
        nf.newPSGD(maxIter=1, verbose=0).fit(nf.newCSRDataset(csr.data, csr.indices, csr.indptr, n, d), y, fm3)


# ---------------------------------------------------------------- synchronous-minibatch SGD (Hogwild's device analogue)
@pytest.mark.parametrize("B", [1, 5, 64])
@pytest.mark.parametrize("degree,fit_lower,k", [(2, "explicit", 8), (3, "explicit", 4), (3, "augment", 16), (2, "none", 30)])
@pytest.mark.parametrize("fit_linear,fit_intercept", [(True, True), (False, True), (True, False)])
@pytest.mark.parametrize("lazy", ["0", "1"])
def test_fm_sgd_minibatch(oracle, monkeypatch, B, degree, fit_lower, k, fit_linear, fit_intercept, lazy):
    """nimfm_fm_sgd_minibatch_epoch against oracle.sgd_minibatch_fit (which, at B = 1, test_oracle.py holds to
    the line-by-line restatement of SGD.fit): ragged rows so that most features sit out most minibatches,
    strong L2 so that their shrink is visible, a shuffled sample order, a partial last minibatch.  lazy: the
    dense step over all parameters vs the touched-features-only form (streaming row kernel shapes only; the
    others fall back to the dense step by themselves)."""
    monkeypatch.setenv("NIMFM_SGD_MB_LAZY", lazy)
    n, d = 203, 60
    rng = np.random.default_rng(31)
    X = make_dense(n, d, 8, density=0.12, positive=False)
    X[5] = 0.0
    csr = CSR.from_dense(X)
    y = np.sign(rng.standard_normal(n))
    P, w, _ = make_fm_params(d, degree, k, fit_lower, fit_linear, seed=9, scale=0.1)
    if not fit_linear:   # a frozen, nonzero w still enters every prediction and is never scaled (sgd.nim:229-236)
        w = np.random.default_rng(78).standard_normal(d) * 0.1
    kw = dict(eta0=0.03, alpha0=1e-3, alpha=2e-2, beta=3e-2)
    perms = np.array([np.random.default_rng(70 + e).permutation(n) for e in range(3)])
    ref = oracle.sgd_minibatch_fit(csr, y, P, w, 0.1, degree, "logistic", B=B, max_iter=3, perms=perms, it=1,
                                   fit_linear=fit_linear, fit_intercept=fit_intercept, **kw)
    fm = nf.newFactorizationMachine(nf.classification, degree=degree, nComponents=k, fitLower=fit_lower,
                                    fitLinear=fit_linear, fitIntercept=fit_intercept, warmStart=True)
    fm.P, fm.w, fm.intercept, fm.isInitialized = P.copy(), w.copy(), 0.1, True
    opt = nf.newSGD(maxIter=3, loss=nf.Logistic(), verbose=0, tol=0.0, miniBatchSize=B if B > 1 else 1, **kw)
    ds = nf.newCSRDataset(csr.data, csr.indices, csr.indptr, n, d)
    opt.fit(ds, y, fm, perms=perms)        # B == 1: the sequential kernel, i.e. the reference's own loop
    np.testing.assert_allclose([h[1] for h in opt.history], ref["loss"], rtol=OBJ_TOL)
    np.testing.assert_allclose([h[0] for h in opt.history], ref["viol"], rtol=1e-8)
    assert max_rel(fm.P, ref["P"]) <= 1e-9 and max_rel(fm.w, ref["w"]) <= 1e-9
    assert abs(fm.intercept - ref["intercept"]) <= 1e-10 and opt.it == ref["it"]


def test_fm_sgd_minibatch_of_one_and_max_threads(oracle):
    """the minibatch entry point with miniBatchSize = 1 reproduces the sequential solver; fit(..., maxThreads=T)
    (the reference's Hogwild entry point, sgd_multi.nim:40) runs the synchronous minibatch of T samples"""
    n, d, k = 90, 25, 8
    X = make_dense(n, d, 3, density=0.3, positive=False)
    csr = CSR.from_dense(X)
    y = np.random.default_rng(2).standard_normal(n)
    P, w, _ = make_fm_params(d, 2, k, "explicit", True, seed=1, scale=0.1)
    kw = dict(eta0=0.02, alpha0=1e-4, alpha=1e-2, beta=1e-2)
    seq = oracle.sgd_fit(csr, y, P, w, 0.0, 2, "squared", max_iter=2, it=1, **kw)
    lib, ctx = _lib.load(), _lib.ctx()
    fm = nf.newFactorizationMachine(nf.regression, degree=2, nComponents=k, warmStart=True)
    fm.P, fm.w, fm.intercept, fm.isInitialized = P.copy(), w.copy(), 0.0, True
    ds = nf.newCSRDataset(csr.data, csr.indices, csr.indptr, n, d)
    ds.set_targets(y)
    h = fm._to_device(d)
    try:
        cfg = _lib.SgdCfg(0, 1.0, kw["eta0"], kw["alpha0"], kw["alpha"], kw["beta"], _lib.SCHED[nf.optimal], 1.0)
        it = C.c_int64(1)
        for ep in range(2):
            viol, ls = C.c_double(), C.c_double()
            _lib.check(lib.nimfm_fm_sgd_minibatch_epoch(ctx, h, ds.handle(), C.byref(cfg), 1, 0, C.byref(it), None, n,
                                                        C.byref(viol), C.byref(ls)))
            assert abs(viol.value - seq["viol"][ep]) <= 1e-8 * seq["viol"][ep]
            assert abs(ls.value / n - seq["loss"][ep]) <= OBJ_TOL * abs(seq["loss"][ep])
        fm._from_device(h)
        assert it.value == seq["it"] and max_rel(fm.P, seq["P"]) <= 1e-9 and max_rel(fm.w, seq["w"]) <= 1e-9
        with pytest.raises(ValueError, match="miniBatchSize"):
            _lib.check(lib.nimfm_fm_sgd_minibatch_epoch(ctx, h, ds.handle(), C.byref(cfg), 0, 0, C.byref(it), None, n, None, None))
    finally:
        lib.nimfm_fm_free(ctx, h)
    ref = oracle.sgd_minibatch_fit(csr, y, P, w, 0.0, 2, "squared", B=7, max_iter=2, it=1, **kw)
    fm2 = nf.newFactorizationMachine(nf.regression, degree=2, nComponents=k, warmStart=True)
    fm2.P, fm2.w, fm2.intercept, fm2.isInitialized = P.copy(), w.copy(), 0.0, True
    opt = nf.newSGD(maxIter=2, verbose=0, tol=0.0, shuffle=False, **kw)
    opt.fit(ds, y, fm2, maxThreads=7)
    assert max_rel(fm2.P, ref["P"]) <= 1e-9 and opt.it == ref["it"]
    np.testing.assert_allclose([h_[0] for h_ in opt.history], ref["viol"], rtol=1e-8)


@pytest.mark.parametrize("B", [1, 6, 50])
def test_ffm_sgd_minibatch(oracle, B):
    X, csr, _ = make_field_csr(83, 24, 4, 19, density=0.3)
    k = 4
    rng = np.random.default_rng(6)
    P, w = rng.standard_normal((4, 24, k)) * 0.1, rng.standard_normal(24) * 0.1
    y = np.sign(rng.standard_normal(83))
    kw = dict(eta0=0.03, alpha0=1e-3, alpha=2e-2, beta=3e-2)
    perms = np.array([np.random.default_rng(11 + e).permutation(83) for e in range(3)])
    ref = oracle.sgd_minibatch_fit(csr, y, P, w, -0.1, loss_kind="logistic", B=B, max_iter=3, perms=perms, it=1,
                                   ffm=True, **kw)
    m = make_ffm(P, w, -0.1, task=nf.classification)
    opt = nf.newSGD(maxIter=3, loss=nf.Logistic(), verbose=0, tol=0.0, **kw)
    opt.fit(field_ds(csr), y, m, maxThreads=B, perms=perms)
    if B == 1:   # maxThreads = 1 is the sequential solver, i.e. the reference itself
        seq = oracle.ffm_sgd_fit(csr, y, P, w, -0.1, "logistic", max_iter=3, perms=perms, it=1, **kw)
        np.testing.assert_allclose(m.P, seq["P"], rtol=1e-8, atol=1e-13)
    np.testing.assert_allclose([h[1] for h in opt.history], ref["loss"], rtol=OBJ_TOL)
    np.testing.assert_allclose([h[0] for h in opt.history], ref["viol"], rtol=1e-8)
    assert max_rel(m.P, ref["P"]) <= 1e-9 and max_rel(m.w, ref["w"]) <= 1e-9
    assert abs(m.intercept - ref["intercept"]) <= 1e-10 and opt.it == ref["it"]
