"""Degree-1 factorization machines (the linear model b + <w, x>, nOrders = 0, no P) on the CPU: the oracle against
the brute-force definitions, the model mirror's shape rules and its dump / load format.  The device routes are held
to the same oracle in tests/test_gpu_degree_one.py."""
import numpy as np
import pytest

import nimfm_b200 as nf
from oracle import bruteforce as bf
from oracle.oracle import CSR
from helpers import make_dense, make_fm_params


def _params(d, fit_linear=True, seed=5):
    P, w, nA = make_fm_params(d, 1, 3, "explicit", fit_linear, seed=seed, scale=0.3)
    assert P.shape == (0, 3, d) and nA == 0
    return P, w


def test_oracle_decision_and_gradient_at_degree_one(oracle):
    n, d = 12, 6
    X = make_dense(n, d, 3, density=0.6, positive=False)
    y = np.random.default_rng(4).standard_normal(n)
    P, w = _params(d)
    csr = CSR.from_dense(X)
    got = oracle.fm_decision_function(csr, P, w, 0.3, 1)
    ref = bf.fm_decision_function(X, P, w, 0.3, 1)
    np.testing.assert_allclose(got, ref, rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(got, X @ w + 0.3, rtol=1e-12, atol=1e-14)
    np.testing.assert_allclose(oracle.fm_decision_function(oracle.csr_to_csc(csr), P, w, 0.3, 1, is_csc=True), ref,
                               rtol=1e-12, atol=1e-14)
    res = oracle.fm_loss_grad(csr, y, P, w, 0.3, 1, "squared")
    dL = ref - y
    np.testing.assert_allclose(res["gw"], X.T @ dL / n, rtol=1e-10, atol=1e-13)
    assert abs(res["gb"] - dL.sum() / n) < 1e-12
    assert res["gP"].shape == (0, 3, d)
    gP = np.zeros_like(P)
    for i in range(n):
        bf.fm_grad(X, i, P, 1, dL[i], gP)   # no orders: nothing to add
    assert gP.size == 0


@pytest.mark.parametrize("fit_linear,fit_intercept", [(True, True), (False, True), (True, False)])
def test_oracle_cd_vs_slow_at_degree_one(oracle, fit_linear, fit_intercept):
    n, d = 14, 5
    X = make_dense(n, d, 21, density=0.8)
    y = np.random.default_rng(2).standard_normal(n)
    P, w = _params(d, fit_linear)
    csc = oracle.csr_to_csc(CSR.from_dense(X))
    fast = oracle.cd_fit(csc, y, P, w, 0.0, 1, "squared", fit_linear, fit_intercept, max_iter=3, alpha0=1e-6,
                         alpha=1e-3, beta=1e-3)
    Ps, ws, bs = bf.cd_slow_fit(X, y, P, w, 0.0, 1, fit_linear, fit_intercept, "squared", 3, 1e-6, 1e-3, 1e-3)
    np.testing.assert_allclose(fast["w"], ws, rtol=1e-6, atol=1e-9)
    assert abs(fast["intercept"] - bs) < 1e-7
    assert fast["P"].shape == (0, 3, d)


def test_oracle_sgd_and_adagrad_vs_slow_at_degree_one(oracle):
    n, d = 10, 5
    X = make_dense(n, d, 31, density=0.7)
    y = np.random.default_rng(3).standard_normal(n)
    P, _ = _params(d)
    w = np.zeros(d)
    csr = CSR.from_dense(X)
    fast = oracle.sgd_fit(csr, y, P, w, 0.0, 1, "squared", True, True, max_iter=2)
    Ps, ws, bs = bf.sgd_slow_fit(X, y, P, w, 0.0, 1, True, True, "squared", 2, 0.01, 1e-6, 1e-3, 1e-3)
    np.testing.assert_allclose(fast["w"], ws, rtol=1e-6, atol=1e-9)
    assert abs(fast["intercept"] - bs) < 1e-7
    fast = oracle.adagrad_fit(csr, y, P, w, 0.0, 1, "squared", True, True, max_iter=2)
    Ps, ws, bs = bf.adagrad_slow_fit(X, y, P, w, 0.0, 1, True, True, "squared", 2, 0.1, 1e-6, 1e-3, 1e-3, 1e-10)
    np.testing.assert_allclose(fast["w"], ws, rtol=1e-6, atol=1e-9)
    assert abs(fast["intercept"] - bs) < 1e-7
    assert fast["state"]["gsP"].shape == (0, d, 3)


@pytest.mark.parametrize("reg,gamma", [("identity", 0.0), ("l1", 0.05)])
@pytest.mark.parametrize("mb", [-1, 5])
def test_oracle_mbpsgd_vs_naive_definition_at_degree_one(oracle, reg, gamma, mb):
    n, d = 37, 6
    X = make_dense(n, d, 35, density=0.5, positive=False)
    y = np.sign(np.random.default_rng(9).standard_normal(n))
    P, w = _params(d)
    kw = dict(eta0=0.2, alpha0=1e-3, alpha=1e-2, beta=2e-2)
    got = oracle.mbpsgd_fit(CSR.from_dense(X), y, P, w, 0.1, 1, "logistic", True, True, max_iter=3, gamma=gamma,
                            reg=reg, mini_batch_size=mb, **kw)
    sP, sw, sb, sl = bf.mbpsgd_slow_fit(X, y, P, w, 0.1, 1, True, True, "logistic", 3, kw["eta0"], kw["alpha0"],
                                        kw["alpha"], kw["beta"], gamma=gamma, reg=reg, mini_batch_size=mb)
    np.testing.assert_allclose(got["w"], sw, rtol=1e-9, atol=1e-13)
    assert abs(got["intercept"] - sb) <= 1e-12
    np.testing.assert_allclose(got["epoch_loss"], sl, rtol=1e-10)


def test_mirror_shapes_at_degree_one():
    for fit_lower in (nf.explicit, nf.augment, nf.none):
        fm = nf.newFactorizationMachine(nf.regression, degree=1, nComponents=4, fitLower=fit_lower, fitLinear=False)
        assert fm.nOrders == 0 and fm.nAugments == 0
    fm = nf.newFactorizationMachine(nf.regression, degree=1, nComponents=4)
    assert fm.nOrders == 0 and fm.nAugments == 0
    ds = nf.newCSRDataset(np.ones(3), np.array([0, 1, 2]), np.array([0, 1, 2, 3]), 3, 5)
    fm.init(ds)
    assert fm.P.shape == (0, 4, 5) and fm.w.shape == (5,)


def test_augment_with_fit_linear_is_refused_at_degree_one():
    fm = nf.newFactorizationMachine(nf.regression, degree=1, nComponents=2, fitLower=nf.augment, fitLinear=True)
    assert fm.nAugments == -1   # the reference's formula, degree - 2
    ds = nf.newCSRDataset(np.ones(3), np.array([0, 1, 2]), np.array([0, 1, 2, 3]), 3, 5)
    with pytest.raises(ValueError, match="nAugments = -1"):
        fm.init(ds)


def test_dump_load_round_trip_at_degree_one(tmp_path):
    fm = nf.newFactorizationMachine(nf.classification, degree=1, nComponents=3, fitIntercept=True)
    fm.P = np.zeros((0, 3, 7))
    fm.w = np.random.default_rng(0).standard_normal(7)
    fm.intercept, fm.isInitialized = -0.25, True
    path = tmp_path / "linear.model"
    fm.dump(str(path))
    text = path.read_text()
    assert "P[" not in text and "degree: 1\n" in text and "nFeatures: 7\n" in text
    back = nf.FactorizationMachine.load(str(path))
    assert back.degree == 1 and back.nOrders == 0 and back.P.shape == (0, 3, 7)
    np.testing.assert_array_equal(back.w, fm.w)
    assert back.intercept == fm.intercept
