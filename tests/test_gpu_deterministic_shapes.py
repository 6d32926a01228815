"""The deterministic FM gradient (NIMFM_DETERMINISTIC=1, csrc/fm_cols.cu) at every degree, nComponents and row length.

The route has two forms of each pass.  The tuned pair -- the streaming row kernel in MODE_STASH and
fm_cols_grad_kernel<D, E, KT> -- runs at degree 2 / 3 with k in {8, 16, 32} and rows of at most 512 entries (dummy
features included).  Every other shape, and every shape under NIMFM_ROW_KERNEL=generic, runs the generic pair: the
runtime-k row kernel fm_rows_kernel<D, E, MODE_STASH, 0> (chunked long rows, component chunks) and
fm_cols_grad_generic_kernel<D, E>.  Both pairs write and read the same stash record, and both add every gradient
element in ascending row order, so:
  - the generic pair is held to the oracle on shapes of every kind, past three persistent waves, and to itself bit for
    bit on a repeat;
  - where both pairs run they give the same gP and gw bits;
  - an MBPSGD fit under the switch repeats itself bit for bit at the default model shape (degree 2, k = 30)."""
import numpy as np
import pytest

import nimfm_b200 as nf
from oracle import bruteforce as bf
from oracle.oracle import CSR
from helpers import make_dense, make_fm_params, max_rel
from test_gpu_fm import dev_loss_grad
from test_gpu_routes import (LOSSES, STAGE_CAP, assert_grad_matches, case_data, csr_ds, expected_route, n_rows,
                             n_wave)

gpu = pytest.mark.gpu
SEG = 512                       # entries per column segment of the column kernels (fm_cols.cu)
TUNED_K = (8, 16, 32)


def det_route(degree, fit_lower, k, z_max, n_aug, env=None):
    """(forward, column kernel) the deterministic route takes.  plan_rows (fm_api.cu) gives the stash forward the
    streaming instance when one exists for (degree, explicit, k) and the longest row incl. dummies fits 512 entries,
    else the generic runtime-k kernel; NIMFM_ROW_KERNEL=generic forces the generic one.  The tuned column kernel runs
    exactly where the streaming forward ran."""
    fwd = expected_route(degree, fit_lower, k, z_max, n_aug, env=env)
    assert fwd in ("stream", "generic")
    return fwd, ("tuned" if fwd == "stream" else "generic")


def col_kt(k):
    """the lane-group width of fm_cols_grad_generic_kernel: fewest idle lanes over ceil(k / KT) chunks, ties to the
    wider group (lane_group_kt in common.cuh)"""
    best = 32
    for kt in (16, 8, 4):
        if -(-k // kt) * kt < -(-k // best) * best:
            best = kt
    return best


def stash_stride(degree, fit_lower, k):
    """doubles per row of the stash: coef + k * sum_o (M_o - 1), padded to an even count"""
    n_o = bf.n_orders(degree, fit_lower)
    s = 1 + k * sum(degree - o - 1 for o in range(n_o))
    return s + (s & 1)


# ------------------------------------------------------------------------------------------------ the case table
def _case(name, degree, fit_lower, k, n_dense=3, max_extra=10, d=400, long_row=0, fit_linear=True):
    # the keys test_gpu_routes.case_data reads
    return dict(name=name, degree=degree, fit_lower=fit_lower, k=k, n_dense=n_dense, max_extra=max_extra, d=d,
                long_row=long_row, spread=False, fit_linear=fit_linear)


CASES = []
# every degree x fitLower, k rotating over the generic ranks; 0, 3 or 20 always-present columns (columns of more than
# one 512-entry segment at the multi-wave size); every fourth case without the linear term
for i, (deg, fl) in enumerate([(d_, f_) for d_ in (2, 3, 4, 5, 6) for f_ in ("explicit", "none", "augment")]):
    k = (4, 12, 30, 33, 64)[i % 5]
    CASES.append(_case(f"d{deg}_{fl}_k{k}", deg, fl, k, n_dense=(20, 3, 0)[i % 3],
                       max_extra=12 if deg <= 3 else 8, d=400 if deg <= 3 else 120, fit_linear=i % 4 != 3))
# rows past 512 entries, at generic and at tuned ranks (the long row alone sends the tuned shape to the generic pair)
for deg, fl, k, L in [(2, "explicit", 30, 1100), (3, "explicit", 32, 700), (4, "augment", 12, 600)]:
    CASES.append(_case(f"longrow_d{deg}_{fl}_k{k}", deg, fl, k, n_dense=20, max_extra=12, d=1200, long_row=L))
# the 512 boundary: maxSegNnz + nAug = 512 takes the tuned pair, 513 the generic one; with augment the dummy tips it
for deg, fl, L in [(2, "explicit", 512), (2, "explicit", 513), (3, "augment", 511), (3, "augment", 512)]:
    CASES.append(_case(f"boundary_d{deg}_{fl}_row{L}", deg, fl, 8, n_dense=20, max_extra=12, d=700, long_row=L))
CASE_BY_NAME = {c["name"]: c for c in CASES}
GENERIC_CASES = [c["name"] for c in CASES if not c["name"].startswith("boundary")]


def case_seed(c):
    return 9100 + CASES.index(c)


def z_max_of(csr):
    return int(np.max(np.diff(csr.indptr)))


# ------------------------------------------------------------------------------------------------ CPU guard
@pytest.mark.parametrize("n_sms", [1, 8, 132, 148, 160])
def test_det_route_table_covers_every_cell(n_sms):
    """Restates the selection rule and checks the case table without a GPU: every degree x fitLower, the generic
    ranks, rows past 512, the 512/513 boundary with and without the augment dummy, columns longer than one segment,
    fitLinear=False, and the multi-wave size."""
    # the rule on its own
    assert det_route(3, "explicit", 32, 39, 0) == ("stream", "tuned")
    assert det_route(3, "explicit", 32, 39, 0, env="generic") == ("generic", "generic")
    assert det_route(2, "explicit", 30, 39, 0) == ("generic", "generic")            # the default model's rank
    assert det_route(4, "explicit", 16, 39, 0) == ("generic", "generic")
    assert det_route(2, "explicit", 8, 512, 0) == ("stream", "tuned")
    assert det_route(2, "explicit", 8, 513, 0) == ("generic", "generic")
    assert det_route(3, "augment", 8, 511, 1) == ("stream", "tuned")
    assert det_route(3, "augment", 8, 512, 1) == ("generic", "generic")
    assert [col_kt(k) for k in (4, 8, 12, 16, 30, 32, 33, 64)] == [4, 8, 4, 16, 32, 32, 4, 32]
    assert stash_stride(3, "explicit", 30) * 8 == 736 and stash_stride(3, "explicit", 32) * 8 == 784

    cells = set()
    for c in CASES:
        cells.add(("degree", c["degree"], c["fit_lower"]))
        cells.add(("k", c["k"]))
        if not c["fit_linear"]:
            cells.add(("no-linear",))
    want = {("degree", dg, fl) for dg in (2, 3, 4, 5, 6) for fl in ("explicit", "none", "augment")}
    want |= {("k", k) for k in (4, 12, 30, 33, 64)} | {("no-linear",)}
    assert want <= cells, sorted(want - cells, key=str)
    assert n_rows(n_sms) >= 3 * n_wave(n_sms)
    if n_sms != 1:
        return
    seen = set()
    for c in CASES:     # the data checks, at one SM's size (the rows are shaped the same way at every size)
        g = case_data(c, n_sms, case_seed(c))
        csr, deg, fl, k = g["csr"], c["degree"], c["fit_lower"], c["k"]
        z, nA = z_max_of(csr), g["n_aug"]
        route = det_route(deg, fl, k, z, nA)
        lens = np.diff(csr.indptr)
        assert np.any(lens == 0) and len(np.unique(lens)) > 3, c["name"]          # empty and ragged rows
        if c["name"] in GENERIC_CASES:
            assert route == ("generic", "generic"), c["name"]
        if c["long_row"]:
            assert z == c["long_row"]
            if z + nA > STAGE_CAP and not c["name"].startswith("boundary"):
                seen.add(("past-512",))
        if c["name"].startswith("boundary"):
            seen.add(("boundary", z + nA, nA > 0))
            assert route[0] == ("stream" if z + nA <= STAGE_CAP else "generic")
        col_len = np.bincount(csr.indices, minlength=csr.d)
        if c["n_dense"]:
            assert col_len.max() > SEG, c["name"]                                   # a multi-segment column
            seen.add(("long-column",))
    assert ("past-512",) in seen
    assert {("boundary", 512, False), ("boundary", 513, False), ("boundary", 512, True), ("boundary", 513, True)} <= seen
    assert ("long-column",) in seen


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture
def deterministic(monkeypatch):
    monkeypatch.delenv("NIMFM_ROW_KERNEL", raising=False)
    monkeypatch.setenv("NIMFM_DETERMINISTIC", "1")


def make_model(c, g):
    task = nf.regression if g["loss"] in ("squared", "huber") else nf.classification
    fm = nf.newFactorizationMachine(task, degree=c["degree"], nComponents=c["k"], fitLower=c["fit_lower"],
                                    fitLinear=c["fit_linear"], fitIntercept=True, warmStart=True)
    fm.P, fm.w, fm.intercept, fm.isInitialized = g["P"].copy(), g["w"].copy(), g["b"], True
    return fm


@gpu
@pytest.mark.parametrize("name", [c["name"] for c in CASES])
def test_det_route_matches_oracle(oracle, deterministic, sms, name):
    """oracle parity past three waves, the same bits on a repeat, and a row sub-range against the oracle on its rows"""
    c = CASE_BY_NAME[name]
    g = case_data(c, sms, case_seed(c))
    csr, y, P, w, b, deg = g["csr"], g["y"], g["P"], g["w"], g["b"], c["degree"]
    n = csr.n
    assert n >= 3 * n_wave(sms)
    if name in GENERIC_CASES:
        assert det_route(deg, c["fit_lower"], c["k"], z_max_of(csr), g["n_aug"]) == ("generic", "generic")
    lo = LOSSES[g["loss"]]()
    fm = make_model(c, g)
    ds = csr_ds(csr)
    ref = oracle.fm_loss_grad(csr, y, P, w, b, deg, g["loss"], fit_linear=c["fit_linear"], mini_batch_size=n)
    got = dev_loss_grad(fm, ds, y, lo, row_begin=0, n_rows=n, mb=n)
    assert_grad_matches(got, ref)
    again = dev_loss_grad(fm, ds, y, lo, row_begin=0, n_rows=n, mb=n)
    assert got[0] == again[0] and got[3] == again[3]
    assert np.array_equal(got[1], again[1]) and np.array_equal(got[2], again[2])
    # a row sub-range that starts and ends inside column segments (the column kernels clip by binary search)
    r0, cnt = n // 5 + 3, n // 2 + 11
    rows = np.arange(r0, r0 + cnt)
    ref_sub = oracle.fm_loss_grad(oracle.csr_take_rows(csr, rows), y[rows], P, w, b, deg, g["loss"],
                                  fit_linear=c["fit_linear"], mini_batch_size=cnt)
    assert_grad_matches(dev_loss_grad(fm, ds, y, lo, row_begin=r0, n_rows=cnt, mb=cnt), ref_sub)


@gpu
@pytest.mark.parametrize("degree", [4, 5, 6])
@pytest.mark.parametrize("fit_lower", ["explicit", "none", "augment"])
def test_det_high_degree_vs_bruteforce(deterministic, degree, fit_lower):
    """degrees 4-6 straight against the subset-enumeration gradient (fm_slow.nim): guards against the oracle and the
    generic kernels sharing a DP mistake"""
    n, d, k = 9, 9, 3
    X = make_dense(n, d, 70 + degree, density=0.8, positive=False)
    X[0] = 0.0                                                       # an empty row
    P, w, _ = make_fm_params(d, degree, k, fit_lower, True, seed=degree + 40, scale=0.4)
    y = np.random.default_rng(degree).standard_normal(n)
    fm = nf.newFactorizationMachine(nf.regression, degree=degree, nComponents=k, fitLower=fit_lower, warmStart=True)
    fm.P, fm.w, fm.intercept, fm.isInitialized = P.copy(), w.copy(), -0.3, True
    csr = CSR.from_dense(X)
    ls, gP, gw, gb = dev_loss_grad(fm, csr_ds(csr), y, nf.Squared(), mb=n)
    yhat = bf.fm_decision_function(X, P, w, -0.3, degree)
    dl = np.array([bf.dloss_val("squared", y[i], yhat[i]) for i in range(n)]) / n
    ref_gP = np.zeros_like(P)
    for i in range(n):
        bf.fm_grad(X, i, P, degree, dl[i], ref_gP)
    assert max_rel(gP, ref_gP) <= 1e-9
    assert max_rel(gw, X.T @ dl) <= 1e-9
    assert abs(gb - dl.sum()) <= 1e-10 * max(1.0, abs(dl.sum()))
    assert abs(ls - sum(bf.loss_val("squared", y[i], yhat[i]) for i in range(n))) <= 1e-10 * max(1.0, abs(ls))


@gpu
@pytest.mark.parametrize("k", TUNED_K)
@pytest.mark.parametrize("degree,fit_lower", [(2, "explicit"), (3, "explicit"), (3, "none"), (3, "augment")])
def test_tuned_and_generic_give_the_same_bits(monkeypatch, sms, degree, fit_lower, k):
    """on the shapes both pairs run, NIMFM_ROW_KERNEL=generic gives gP and gw array_equal to the tuned pair; the loss
    and gb are summed through per-warp partials whose count follows the grid, so they agree to rounding"""
    c = _case(f"bits_d{degree}_{fit_lower}_k{k}", degree, fit_lower, k, n_dense=20, max_extra=12)
    g = case_data(c, sms, 9300 + 10 * degree + k + len(fit_lower))
    csr, y = g["csr"], g["y"]
    assert det_route(degree, fit_lower, k, z_max_of(csr), g["n_aug"]) == ("stream", "tuned")
    lo = LOSSES[g["loss"]]()
    fm = make_model(c, g)
    ds = csr_ds(csr)
    n = csr.n
    monkeypatch.setenv("NIMFM_DETERMINISTIC", "1")
    out = {}
    for env in (None, "generic"):
        if env:
            monkeypatch.setenv("NIMFM_ROW_KERNEL", env)
        else:
            monkeypatch.delenv("NIMFM_ROW_KERNEL", raising=False)
        out[env] = dev_loss_grad(fm, ds, y, lo, row_begin=0, n_rows=n, mb=n)
    (l0, gP0, gw0, gb0), (l1, gP1, gw1, gb1) = out[None], out["generic"]
    assert np.array_equal(gP0, gP1), float(np.max(np.abs(gP0 - gP1)))
    assert np.array_equal(gw0, gw1), float(np.max(np.abs(gw0 - gw1)))
    assert abs(l0 - l1) <= 1e-12 * abs(l0)
    assert abs(gb0 - gb1) <= 1e-12 * max(1.0, abs(gb0))


def c4_like_csr(n, d, seed, z=13):
    rng = np.random.default_rng(seed)
    idx = np.sort(rng.integers(0, d // z, size=(n, z)) + (np.arange(z) * (d // z))[None, :], axis=1)
    idx[:, 0] = 0                                                   # a column in every row: several segments
    return CSR(rng.random((n, z)).ravel(), idx.ravel(), np.arange(n + 1) * z, n, d)


@gpu
@pytest.mark.parametrize("shape", ["default", "d4_augment_k12"])
def test_det_mbpsgd_fit(oracle, deterministic, shape):
    """an MBPSGD fit under the switch: the default model (degree 2, k = 30) and degree 4, k = 12, augment; two fits
    are the same bits, and both match the oracle"""
    n, d, mb = 4000, 300, 500
    csr = c4_like_csr(n, d, 8)
    y = np.sign(np.random.default_rng(9).standard_normal(n))

    def model():
        if shape == "default":
            return nf.newFactorizationMachine(nf.classification, warmStart=True)
        return nf.newFactorizationMachine(nf.classification, degree=4, nComponents=12, fitLower=nf.augment,
                                          warmStart=True)
    m0 = model()
    degree, k, fl = m0.degree, m0.nComponents, m0.fitLower
    if shape == "default":
        assert (degree, k) == (2, 30)
    P, w, _ = make_fm_params(d, degree, k, fl, True, seed=3, scale=0.05)

    def fit():
        f = model()
        f.P, f.w, f.intercept, f.isInitialized = P.copy(), w.copy(), 0.0, True
        opt = nf.newMBPSGD(maxIter=3, gamma=1e-4, reg=nf.newL1(), loss=nf.Logistic(), miniBatchSize=mb, verbose=0,
                           tol=0.0, shuffle=False)
        opt.fit(csr_ds(csr), y, f)
        return opt.history, f
    h1, f1 = fit()
    h2, f2 = fit()
    assert h1 == h2 and np.array_equal(f1.P, f2.P) and np.array_equal(f1.w, f2.w) and f1.intercept == f2.intercept
    ref = oracle.mbpsgd_fit(csr, y, P, w, 0.0, degree, "logistic", max_iter=3, gamma=1e-4, reg="l1", mini_batch_size=mb,
                            it=0)
    np.testing.assert_allclose(h1, ref["epoch_loss"], rtol=1e-8)
    assert max_rel(f1.P, ref["P"]) <= 1e-8 and max_rel(f1.w, ref["w"]) <= 1e-8
    assert abs(f1.intercept - ref["intercept"]) <= 1e-8 * max(1.0, abs(ref["intercept"]))


@gpu
def test_det_refusals_at_a_generic_rank(deterministic):
    """a row list and a wrapping range stay errors at a rank only the generic pair runs"""
    n, d, k = 900, 60, 30
    csr = c4_like_csr(n, d, 4)
    y = np.random.default_rng(2).standard_normal(n)
    P, w, _ = make_fm_params(d, 2, k, "explicit", True, seed=5, scale=0.2)
    fm = nf.newFactorizationMachine(nf.regression, degree=2, nComponents=k, warmStart=True)
    fm.P, fm.w, fm.intercept, fm.isInitialized = P.copy(), w.copy(), 0.0, True
    with pytest.raises(Exception, match="contiguous"):
        dev_loss_grad(fm, csr_ds(csr), y, nf.Squared(), rows=np.array([3, 1, 2]), mb=3)
    with pytest.raises(Exception, match="wrap"):
        dev_loss_grad(fm, csr_ds(csr), y, nf.Squared(), row_begin=n - 5, n_rows=10, mb=10)
