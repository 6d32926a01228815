"""The deterministic (atomic-free) predict+grad route, NIMFM_DETERMINISTIC=1 (csrc/fm_cols.cu): stash-forward row
kernel + column kernel over the CSC twin.  Held to the oracle like the RED route (minibatch_psgd.nim:67-88 sums in
sample order; the column kernel sums in ascending row order inside fixed segments), and to ITSELF bit for bit:
two runs, and runs over different launch geometries, must agree exactly -- which the RED route cannot promise."""
import ctypes as C

import numpy as np
import pytest

import nimfm_b200 as nf
from nimfm_b200 import _lib
from oracle.oracle import CSR
from helpers import make_fm_params, max_rel, sums_agree
from test_gpu_fm import dev_loss_grad, make_fm, ragged_csr, csr_ds

pytestmark = pytest.mark.gpu


@pytest.fixture
def deterministic(monkeypatch):
    monkeypatch.setenv("NIMFM_DETERMINISTIC", "1")


def long_column_csr(n, d, seed, z):
    """z nonzeros per row: column 0 present in every row (a column longer than one 512-entry segment), the rest
    random; sorted unique indices"""
    rng = np.random.default_rng(seed)
    idx = np.empty((n, z), dtype=np.int64)
    idx[:, 0] = 0
    for i in range(n):
        idx[i, 1:] = np.sort(rng.choice(np.arange(1, d), size=z - 1, replace=False))
    data = rng.standard_normal((n, z))
    return CSR(data.ravel(), idx.ravel(), np.arange(n + 1) * z, n, d)


@pytest.mark.parametrize("degree,fit_lower,k", [(2, "explicit", 8), (2, "explicit", 16), (3, "explicit", 32),
                                               (3, "none", 16), (3, "augment", 8), (2, "augment", 32)])
@pytest.mark.parametrize("loss_name", ["squared", "logistic"])
def test_deterministic_grad_matches_oracle(oracle, deterministic, degree, fit_lower, k, loss_name):
    n, d = 1500, 40
    csr = long_column_csr(n, d, 3 + degree, 7)
    rng = np.random.default_rng(k)
    y = np.sign(rng.standard_normal(n)) if loss_name != "squared" else rng.standard_normal(n)
    P, w, nA = make_fm_params(d, degree, k, fit_lower, True, seed=degree + k, scale=0.2)
    fm = make_fm(degree, k, fit_lower, True, True, P, w, 0.1)
    loss = {"squared": nf.Squared(), "logistic": nf.Logistic()}[loss_name]
    ls, gP, gw, gb = dev_loss_grad(fm, csr_ds(csr), y, loss)
    ref = oracle.fm_loss_grad(csr, y, P, w, 0.1, degree, loss_name)
    assert abs(ls - ref["loss"]) <= 1e-10 * max(1.0, abs(ref["loss"]))
    assert max_rel(gP, ref["gP"]) <= 1e-9 and max_rel(gw, ref["gw"]) <= 1e-9
    assert abs(gb - ref["gb"]) <= 1e-10 * max(1.0, abs(ref["gb"]))
    # bit for bit: a second run, and a sub-range + its complement add up to ... themselves, run twice
    ls2, gP2, gw2, gb2 = dev_loss_grad(fm, csr_ds(csr), y, loss)
    assert ls2 == ls and np.array_equal(gP2, gP) and np.array_equal(gw2, gw) and gb2 == gb


def test_deterministic_row_range_and_ragged(oracle, deterministic):
    """a row sub-range (the column segments are clipped by binary search), empty rows, ragged lengths"""
    n, d, k, degree = 900, 60, 16, 3
    csr = ragged_csr(n, d, 11, 20)
    y = np.random.default_rng(2).standard_normal(n)
    P, w, _ = make_fm_params(d, degree, k, "explicit", True, seed=5, scale=0.2)
    fm = make_fm(degree, k, "explicit", True, True, P, w, 0.0)
    r0, cnt = 137, 555
    ls, gP, gw, gb = dev_loss_grad(fm, csr_ds(csr), y, nf.Squared(), row_begin=r0, n_rows=cnt, mb=cnt)
    rows = np.arange(r0, r0 + cnt)
    ref = oracle.fm_loss_grad(oracle.csr_take_rows(csr, rows), y[rows], P, w, 0.0, degree, "squared", mini_batch_size=cnt)
    assert abs(ls - ref["loss"]) <= 1e-10 * abs(ref["loss"])
    assert max_rel(gP, ref["gP"]) <= 1e-9 and max_rel(gw, ref["gw"]) <= 1e-9
    # unsupported shapes fail loudly instead of silently taking the RED route
    with pytest.raises(Exception, match="contiguous"):
        dev_loss_grad(fm, csr_ds(csr), y, nf.Squared(), rows=np.array([3, 1, 2]), mb=3)
    with pytest.raises(Exception, match="wrap"):
        dev_loss_grad(fm, csr_ds(csr), y, nf.Squared(), row_begin=n - 5, n_rows=10, mb=10)


def test_deterministic_vs_red_route_and_mbpsgd(oracle, monkeypatch):
    """the two routes agree to rounding; an MBPSGD fit under the deterministic route matches the oracle and
    repeats itself bit for bit"""
    n, d, k, degree = 4000, 300, 32, 3
    rng = np.random.default_rng(8)
    z = 13
    idx = np.sort(rng.integers(0, d // z, size=(n, z)) + (np.arange(z) * (d // z))[None, :], axis=1)
    csr = CSR(rng.random((n, z)).ravel(), idx.ravel(), np.arange(n + 1) * z, n, d)
    y = np.sign(rng.standard_normal(n))
    P, w, _ = make_fm_params(d, degree, k, "explicit", True, seed=1, scale=0.05)
    fm = make_fm(degree, k, "explicit", True, True, P, w, 0.0, task=nf.classification)
    monkeypatch.delenv("NIMFM_DETERMINISTIC", raising=False)
    ls_r, gP_r, gw_r, gb_r = dev_loss_grad(fm, csr_ds(csr), y, nf.Logistic())
    monkeypatch.setenv("NIMFM_DETERMINISTIC", "1")
    ls_d, gP_d, gw_d, gb_d = dev_loss_grad(fm, csr_ds(csr), y, nf.Logistic())
    # the RED route adds in arrival order, so its gP elements whose terms nearly cancel move from run to run by up to
    # ~1e-11 of themselves (9.5e-12 over 40 runs on a B200 at 1000 W, as far from the oracle as from this route)
    # while every element stays within ~1e-15 of the largest one: see helpers.sums_agree
    assert sums_agree(gP_d, gP_r, norm_tol=1e-14, elem_tol=5e-11)
    assert max_rel(gw_d, gw_r) <= 1e-11 and abs(ls_d - ls_r) <= 1e-12 * abs(ls_r)

    def fit():
        f = make_fm(degree, k, "explicit", True, True, P, w, 0.0, task=nf.classification)
        opt = nf.newMBPSGD(maxIter=3, gamma=1e-4, reg=nf.newL1(), loss=nf.Logistic(), miniBatchSize=500, verbose=0,
                           tol=0.0, shuffle=False)
        opt.fit(csr_ds(csr), y, f)
        return opt.history, f
    h1, f1 = fit()
    h2, f2 = fit()
    assert h1 == h2 and np.array_equal(f1.P, f2.P) and np.array_equal(f1.w, f2.w) and f1.intercept == f2.intercept
    ref = oracle.mbpsgd_fit(csr, y, P, w, 0.0, degree, "logistic", max_iter=3, gamma=1e-4, reg="l1", mini_batch_size=500,
                            it=0)
    np.testing.assert_allclose(h1, ref["epoch_loss"], rtol=1e-8)
    assert max_rel(f1.P, ref["P"]) <= 1e-8 and max_rel(f1.w, ref["w"]) <= 1e-8


# ---------------------------------------------------------------- FFM: column route (csrc/ffm_cols.cuh)
def one_per_field_csr(n, n_fields, per_field, seed, keep=0.85):
    """libffm-shaped rows: at most one feature per field, field f owns ids [f*per_field, (f+1)*per_field); feature 0
    of field 0 is present in (almost) every row so that its column is longer than one 512-entry segment"""
    rng = np.random.default_rng(seed)
    data, idx, fld, ptr = [], [], [], [0]
    for i in range(n):
        for f in range(n_fields):
            if f == 0 or rng.random() < keep:
                j = 0 if (f == 0 and rng.random() < 0.9) else int(rng.integers(0, per_field))
                idx.append(f * per_field + j)
                fld.append(f)
                data.append(float(rng.standard_normal()))
        ptr.append(len(idx))
    csr = CSR(data, idx, ptr, n, n_fields * per_field)
    csr.fields = np.asarray(fld, dtype=np.int64)
    csr.n_fields = n_fields
    return csr


def ffm_dev_grad(csr, y, P, w, b, loss, row_begin=0, n_rows=None, rows=None):
    lib, ctx = _lib.load(), _lib.ctx()
    nF, d, k = P.shape
    ds = nf.newCSRFieldDataset(csr.data, csr.indices, csr.indptr, csr.fields, csr.n, d, nF)
    ds.set_targets(y)
    m = nf.newFieldAwareFactorizationMachine(nf.regression, nComponents=k, warmStart=True)
    m.P, m.w, m.intercept, m.isInitialized = P.copy(), w.copy(), b, True
    h = m._to_device(ds)
    try:
        n_rows = csr.n if n_rows is None else n_rows
        ids = None if rows is None else _lib.i64(rows)
        if ids is not None:
            n_rows = len(ids)
        ls = C.c_double()
        _lib.check(lib.nimfm_ffm_loss_grad(ctx, h, ds.handle(), loss.kind, loss.threshold, row_begin, n_rows, _lib.ptr(ids),
                                           n_rows, 1, 0, C.byref(ls)))
        gP, gw, gb = np.zeros_like(P), np.zeros(d), C.c_double()
        _lib.check(lib.nimfm_ffm_get_grads(ctx, h, _lib.ptr(gP), _lib.ptr(gw), C.byref(gb)))
    finally:
        lib.nimfm_ffm_free(ctx, h)
        ds.free()
    return ls.value, gP, gw, gb.value


@pytest.mark.parametrize("k", [4, 8, 16])
@pytest.mark.parametrize("route", ["deterministic"])
def test_ffm_column_route_matches_oracle(oracle, monkeypatch, k, route):
    monkeypatch.setenv("NIMFM_DETERMINISTIC", "1")
    n, nF, per = 1300, 7, 9
    csr = one_per_field_csr(n, nF, per, 5 + k)
    d = nF * per
    rng = np.random.default_rng(k)
    y = np.sign(rng.standard_normal(n))
    P = rng.standard_normal((nF, d, k)) * 0.2
    w = rng.standard_normal(d) * 0.1
    ls, gP, gw, gb = ffm_dev_grad(csr, y, P, w, 0.05, nf.Logistic())
    ref = oracle.ffm_loss_grad(csr, y, P, w, 0.05, "logistic")
    assert abs(ls - ref["loss"]) <= 1e-10 * abs(ref["loss"])
    assert max_rel(gP, ref["gP"]) <= 1e-9 and max_rel(gw, ref["gw"]) <= 1e-9
    assert abs(gb - ref["gb"]) <= 1e-10 * max(1.0, abs(ref["gb"]))
    ls2, gP2, gw2, gb2 = ffm_dev_grad(csr, y, P, w, 0.05, nf.Logistic())
    assert ls2 == ls and np.array_equal(gP2, gP) and np.array_equal(gw2, gw) and gb2 == gb     # bit for bit
    # a row sub-range
    r0, cnt = 211, 777
    ls3, gP3, gw3, _ = ffm_dev_grad(csr, y, P, w, 0.05, nf.Logistic(), row_begin=r0, n_rows=cnt)
    rows = np.arange(r0, r0 + cnt)
    sub = oracle.csr_take_rows(csr, rows)
    sub.fields = np.concatenate([csr.fields[csr.indptr[r]:csr.indptr[r + 1]] for r in rows]).astype(np.int64)
    sub.n_fields = nF
    ref3 = oracle.ffm_loss_grad(sub, y[rows], P, w, 0.05, "logistic")
    assert abs(ls3 - ref3["loss"]) <= 1e-10 * abs(ref3["loss"]) and max_rel(gP3, ref3["gP"]) <= 1e-9
    assert max_rel(gw3, ref3["gw"]) <= 1e-9


def test_ffm_deterministic_rejects_repeated_fields(oracle, deterministic):
    from helpers import make_field_csr
    _, fcsr, _ = make_field_csr(60, 12, 4, 9)            # several nonzeros per field in a row
    P = np.random.default_rng(3).standard_normal((4, 12, 4)) * 0.1
    y = np.random.default_rng(4).standard_normal(60)
    with pytest.raises(Exception, match="one nonzero per field"):
        ffm_dev_grad(fcsr, y, P, np.zeros(12), 0.0, nf.Squared())
