"""The pipelined sequential solvers against the oracle at the row shapes their machinery engages on.

sgd_fm_pipe_kernel (sgd.cu), adagrad_fm_pipe_kernel (adagrad_seq.cuh) and psgd_lazy_pipe_kernel (psgd.cu) are the
default routes of SGD.fit, AdaGrad(miniBatchSize=1).fit and PSGD(L1 / L21).fit on an FM.  Each one prefetches
sample q+3's row id, q+2's row pointer / target and q+1's indices / values through a 4-slot ring (two lanes per
thread of the prefetching warp: nonzeros u and u + 32), computes the step sizes one sample ahead into a two-slot
table (SGD, PSGD), walks the [z][SB8] row slice (SB8 = nOrders * k) with ElemWalk at up to 12 elements per thread,
and, for PSGD-L21 at k <= 32, runs the prox eight vectors per warp.  None of that engages at the reference's test
shapes (k <= 4, d <= 8).  The case table below spans the kernels' domain -- SB8 from 1 to the pipe maxima, rows
that need one and both prefetch lanes, 1 to 12 elements per thread, degrees 2 to 6 -- and holds every case, and
every other form of the same solver at the same inputs, to the float64 restatement of the reference."""
import ctypes as C

import numpy as np
import pytest

import nimfm_b200 as nf
from nimfm_b200 import _lib
from oracle import bruteforce as bf
from oracle.oracle import CSR

gpu = pytest.mark.gpu

OBJ_TOL = 1e-8
FORM_TOL = 1e-12         # pipe vs another form of the same solver: both reduce y-hat in float64, in different orders

# ------------------------------------------------------------------------------------------------ the dispatch rules
# There is no launch record in the ABI, so the tests restate the predicates that pick the kernel.  The shared-memory
# budgets are evaluated for the B200's opt-in limit per block (cudaDevAttrMaxSharedMemoryPerBlockOptin); a case that
# leaves the pipe on another GPU is a reason to move it, not to drop the route assertion.
SMEM_OPTIN = 232_448
MAX_DEGREE = 6           # NIMFM_MAX_DEGREE (common.cuh): sA holds MAX_DEGREE + 1 doubles per (order, component)
PIPE_THREADS = 512       # SGDP_THREADS, ADAPIPE_THREADS, PSGD_PIPE_THREADS
PIPE_R = 12              # SGDP_R, PSGD_PIPE_R: row slice elements per thread
SEQ_THREADS = 256        # SGD_THREADS, ADASEQ_THREADS, PSGD_THREADS
PIPE_ROW = 64            # nonzeros (dummies included) the prefetching warp loads per row: two per lane

ENV = {"sgd": "NIMFM_SGD_KERNEL", "adagrad": "NIMFM_ADAGRAD_SEQ", "psgd": "NIMFM_PSGD_KERNEL"}
FORMS = {"sgd": ("staged", "unstaged"), "adagrad": ("staged", "0"), "psgd": ("staged",)}
FORM_ROUTE = {("sgd", "staged"): "staged", ("sgd", "unstaged"): "unstaged", ("adagrad", "staged"): "staged",
              ("adagrad", "0"): "minibatch", ("psgd", "staged"): "staged"}


def sgd_route(sb8, zmax, env=None):
    """nimfm_fm_sgd_epoch (sgd.cu:726-740); env: NIMFM_SGD_KERNEL"""
    pipe = (zmax * sb8 + sb8 * (MAX_DEGREE + 1) + 4 * zmax) * 8 + 2 * zmax * 4 + sb8 + 16
    staged = (zmax * sb8 + 3 * zmax) * 8 + zmax * 8
    if (env is None and sb8 <= PIPE_THREADS - 64 and zmax <= PIPE_ROW and zmax * sb8 <= PIPE_R * PIPE_THREADS
            and pipe <= SMEM_OPTIN - 4096):
        return "pipe"
    if sb8 <= SEQ_THREADS and staged <= SMEM_OPTIN - 2048 and env != "unstaged":
        return "staged"
    return "unstaged"


def adagrad_route(sb8, zmax, n_rows, env=None):
    """nimfm_fm_adagrad_epoch, miniBatchSize = 1 on one rank (fm_api.cu:996-1022); env: NIMFM_ADAGRAD_SEQ"""
    staged = (3 * zmax * sb8 + 2 * zmax) * 8 + zmax * 8
    if n_rows > 0 and sb8 <= SEQ_THREADS and staged + 2048 <= SMEM_OPTIN and not (env or " ").startswith("0"):
        pipe = (3 * zmax * sb8 + sb8 * (MAX_DEGREE + 1) + 3 * zmax) * 8 + 2 * zmax * 4 + sb8 + 16
        if zmax <= PIPE_ROW and pipe + 4096 <= SMEM_OPTIN and not (env or " ").startswith("s"):
            return "pipe"
        return "staged"
    return "minibatch"


def psgd_route(sb8, zmax, env=None):
    """nimfm_fm_psgd_epoch, L1 / L21 (psgd.cu:762-789); env: NIMFM_PSGD_KERNEL"""
    staged = (zmax * sb8 + 4 * zmax) * 8 + zmax * 8
    if sb8 > SEQ_THREADS or staged > SMEM_OPTIN - 2048:
        return "unsupported"
    pipe = (zmax * sb8 + sb8 * (MAX_DEGREE + 1) + 5 * zmax) * 8 + 2 * zmax * 4 + sb8 + 16
    if (zmax <= PIPE_ROW and zmax * sb8 <= PIPE_R * PIPE_THREADS and pipe + 4096 <= SMEM_OPTIN
            and not (env or " ").startswith("s")):
        return "pipe"
    return "staged"


def route(solver, sb8, zmax, n_rows, env=None):
    if solver == "sgd":
        return sgd_route(sb8, zmax, env)
    if solver == "adagrad":
        return adagrad_route(sb8, zmax, n_rows, env)
    return psgd_route(sb8, zmax, env)


# ------------------------------------------------------------------------------------------------ the case table
N_ROWS, N_FEAT, EPOCHS = 150, 160, 3
LOSSES = {"squared": nf.Squared, "logistic": nf.Logistic, "squared_hinge": nf.SquaredHinge,
          "huber": lambda: nf.Huber(0.5)}


def _case(name, solver, degree, fit_lower, k, zrow, lo, loss, fit_linear=True, fit_intercept=True,
          sched="optimal", reg=None, gamma=0.0):
    """zrow: the longest row's real nonzeros (one row has exactly this many); the others lo..zrow, every 9th empty"""
    nO, nA = bf.n_orders(degree, fit_lower), bf.n_augments(degree, fit_lower, fit_linear)
    return dict(name=name, solver=solver, degree=degree, fit_lower=fit_lower, k=k, zrow=zrow, lo=lo, loss=loss,
                fit_linear=fit_linear, fit_intercept=fit_intercept, sched=sched, reg=reg, gamma=gamma,
                sb8=nO * k, n_aug=nA, zmax=max(zrow + nA, 1))


CASES = [
    # SGD: SB8 up to 448 (SGDP_THREADS - 64), z * SB8 up to 12 * 512
    _case("sgd_sb1", "sgd", 2, "explicit", 1, 64, 33, "squared"),
    _case("sgd_sb3", "sgd", 2, "explicit", 3, 20, 2, "logistic", sched="constant"),
    _case("sgd_sb37", "sgd", 2, "explicit", 37, 50, 10, "squared_hinge", sched="invscaling"),
    _case("sgd_c4", "sgd", 3, "explicit", 32, 39, 30, "huber"),
    _case("sgd_sb96_row64", "sgd", 3, "explicit", 48, 64, 40, "squared", sched="invscaling", fit_intercept=False),
    _case("sgd_sb256", "sgd", 2, "explicit", 256, 24, 8, "logistic", sched="constant"),
    _case("sgd_sb448", "sgd", 5, "explicit", 112, 13, 4, "squared"),
    _case("sgd_d3_augment", "sgd", 3, "augment", 16, 63, 33, "huber", sched="invscaling"),
    _case("sgd_d4_none", "sgd", 4, "none", 24, 40, 20, "squared_hinge", fit_linear=False),
    _case("sgd_d6_explicit", "sgd", 6, "explicit", 8, 30, 6, "logistic", sched="constant"),
    # AdaGrad (miniBatchSize = 1): SB8 up to 256; three zmax * SB8 slices staged, so SB8 = 256 leaves room for 34
    _case("adagrad_sb1", "adagrad", 2, "explicit", 1, 64, 33, "logistic"),
    _case("adagrad_sb3", "adagrad", 2, "explicit", 3, 25, 3, "squared"),
    _case("adagrad_sb37", "adagrad", 2, "explicit", 37, 45, 12, "huber"),
    _case("adagrad_c4", "adagrad", 3, "explicit", 32, 39, 30, "squared_hinge"),
    _case("adagrad_sb96_row64", "adagrad", 3, "explicit", 48, 64, 40, "squared"),
    _case("adagrad_sb256_row34", "adagrad", 2, "explicit", 256, 34, 10, "logistic", fit_intercept=False),
    _case("adagrad_d3_augment", "adagrad", 3, "augment", 16, 63, 33, "squared"),
    _case("adagrad_d4_none", "adagrad", 4, "none", 24, 40, 20, "huber", fit_linear=False),
    _case("adagrad_d5_explicit", "adagrad", 5, "explicit", 8, 30, 8, "squared_hinge"),
    _case("adagrad_d6_explicit", "adagrad", 6, "explicit", 6, 20, 4, "squared"),
    # PSGD-L21: k <= 32 takes the eight-vectors-per-warp prox, k > 32 the generic one
    _case("psgd_l21_k1", "psgd", 2, "explicit", 1, 64, 33, "squared", reg="l21", gamma=0.02),
    _case("psgd_l21_k7", "psgd", 3, "explicit", 7, 30, 5, "logistic", reg="l21", gamma=0.25, sched="invscaling"),
    _case("psgd_l21_k8", "psgd", 4, "none", 8, 50, 20, "huber", reg="l21", gamma=0.05),
    _case("psgd_l21_k31", "psgd", 2, "explicit", 31, 45, 15, "squared_hinge", reg="l21", gamma=0.1,
          fit_linear=False),
    _case("psgd_l21_k32_c4", "psgd", 3, "explicit", 32, 39, 30, "squared", reg="l21", gamma=0.1),
    _case("psgd_l21_k33", "psgd", 3, "augment", 33, 63, 33, "logistic", reg="l21", gamma=0.1, sched="constant"),
    _case("psgd_l21_k64", "psgd", 2, "explicit", 64, 40, 12, "squared", reg="l21", gamma=0.15),
    # PSGD-L1
    _case("psgd_l1_sb3", "psgd", 2, "explicit", 3, 20, 2, "squared_hinge", reg="l1", gamma=0.02),
    _case("psgd_l1_sb37", "psgd", 2, "explicit", 37, 50, 10, "huber", reg="l1", gamma=0.02, sched="invscaling"),
    _case("psgd_l1_sb96_row64", "psgd", 3, "explicit", 48, 64, 40, "squared", reg="l1", gamma=0.02),
    _case("psgd_l1_sb256", "psgd", 2, "explicit", 256, 24, 8, "logistic", reg="l1", gamma=0.02,
          fit_intercept=False),
    _case("psgd_l1_d5_explicit", "psgd", 5, "explicit", 10, 33, 20, "squared", reg="l1", gamma=0.02),
    _case("psgd_l1_d6_explicit", "psgd", 6, "explicit", 4, 40, 10, "huber", reg="l1", gamma=0.02),
]
CASE_BY_NAME = {c["name"]: c for c in CASES}


def elems_per_thread(c):
    return -(-c["zmax"] * c["sb8"] // PIPE_THREADS)


def rows_csr(lengths, d, rng):
    """one row per entry of lengths, sorted unique columns"""
    data, indices, indptr = [], [], [0]
    for z in lengths:
        indices.extend(np.sort(rng.choice(d, size=z, replace=False)).tolist())
        data.extend((rng.standard_normal(z) * 0.3).tolist())
        indptr.append(len(indices))
    return CSR(np.array(data, dtype=np.float64), np.array(indices, dtype=np.int64), indptr, len(lengths), d)


def shaped_csr(n, d, zrow, lo, seed):
    """rows of lo..zrow nonzeros, every 9th row empty, row n // 3 exactly zrow long"""
    rng = np.random.default_rng(seed)
    lengths = [0 if i % 9 == 4 else (zrow if i == n // 3 else int(rng.integers(lo, zrow + 1))) for i in range(n)]
    return rows_csr(lengths, d, rng)


def case_data(c, csr=None):
    """case c's dataset (or csr) with a seeded model and targets"""
    seed = 9100 + list(CASE_BY_NAME).index(c["name"])
    if csr is None:
        csr = shaped_csr(N_ROWS, N_FEAT, c["zrow"], c["lo"], seed)
    rng = np.random.default_rng(seed + 1)
    nO, k, n, d = bf.n_orders(c["degree"], c["fit_lower"]), c["k"], csr.n, csr.d
    P = rng.standard_normal((nO, k, d + c["n_aug"])) * 0.15
    w = rng.standard_normal(d) * 0.1 if c["fit_linear"] else np.zeros(d)
    y = rng.standard_normal(n) if c["loss"] in ("squared", "huber") else np.sign(rng.standard_normal(n))
    return dict(csr=csr, P=P, w=w, b=0.1 if c["fit_intercept"] else 0.0, y=y)


def solver_kw(c):
    if c["solver"] == "adagrad":
        return dict(eta0=0.05, alpha0=1e-6, alpha=1e-3, beta=1e-3)
    kw = dict(eta0=0.1 if c["sched"] == "invscaling" else 0.02, alpha0=1e-6, alpha=1e-3, beta=1e-3,
              scheduling=c["sched"], power=0.75 if c["sched"] == "invscaling" else 1.0)
    if c["solver"] == "psgd":
        kw["gamma"] = c["gamma"]
    return kw


# ------------------------------------------------------------------------------------------------ running one fit
def make_fm(c, P, w, b):
    task = nf.regression if c["loss"] in ("squared", "huber") else nf.classification
    fm = nf.newFactorizationMachine(task, degree=c["degree"], nComponents=c["k"], fitLower=c["fit_lower"],
                                    fitLinear=c["fit_linear"], fitIntercept=c["fit_intercept"], warmStart=True)
    fm.P, fm.w, fm.intercept, fm.isInitialized = P.copy(), w.copy(), b, True
    return fm


def new_opt(c, max_iter, shuffle=False):
    kw, lo = solver_kw(c), LOSSES[c["loss"]]()
    if c["solver"] == "sgd":
        return nf.newSGD(maxIter=max_iter, loss=lo, verbose=0, tol=0.0, shuffle=shuffle, **kw)
    if c["solver"] == "adagrad":
        return nf.newAdaGrad(maxIter=max_iter, loss=lo, verbose=0, tol=0.0, shuffle=shuffle, miniBatchSize=1, **kw)
    reg = {"l1": nf.newL1, "l21": nf.newL21}[c["reg"]]()
    return nf.newPSGD(maxIter=max_iter, loss=lo, reg=reg, verbose=0, tol=0.0, shuffle=shuffle, **kw)


def history(c, opt):
    """(epoch losses, epoch violations or None)"""
    if c["solver"] == "psgd":
        return np.array(opt.history), None
    h = np.array(opt.history)
    return h[:, 1], h[:, 0]


def device_fit(c, g, monkeypatch, env=None, perms=None):
    for var in ENV.values():
        monkeypatch.delenv(var, raising=False)
    if env is not None:
        monkeypatch.setenv(ENV[c["solver"]], env)
    csr = g["csr"]
    fm = make_fm(c, g["P"], g["w"], g["b"])
    opt = new_opt(c, EPOCHS, shuffle=perms is not None)
    opt.fit(nf.newCSRDataset(csr.data, csr.indices, csr.indptr, csr.n, csr.d), g["y"], fm, perms=perms)
    loss, viol = history(c, opt)
    out = dict(P=fm.P, w=fm.w, intercept=fm.intercept, loss=loss, viol=viol, it=opt.it)
    if c["solver"] == "adagrad":
        out.update(gsP=opt.g_sum["P"], gnP=opt.g_norm["P"])
    return out


def oracle_fit(oracle, c, csr, y, P, w, b, max_iter=EPOCHS, perms=None, it=1):
    kw = solver_kw(c)
    common = dict(fit_linear=c["fit_linear"], fit_intercept=c["fit_intercept"], max_iter=max_iter, perms=perms, it=it,
                  thr=LOSSES[c["loss"]]().threshold)
    if c["solver"] == "sgd":
        r = oracle.sgd_fit(csr, y, P, w, b, c["degree"], c["loss"], **common, **kw)
    elif c["solver"] == "adagrad":
        r = oracle.adagrad_fit(csr, y, P, w, b, c["degree"], c["loss"], mini_batch_size=1, **common, **kw)
        # the solver layout [nOrders, d + nAug, k] of g_sum / g_norm, as AdaGrad.g_sum["P"] holds them
        r.update(gsP=r["state"]["gsP"], gnP=r["state"]["gnP"])
    else:
        r = oracle.psgd_fit(csr, y, P, w, b, c["degree"], c["loss"], reg=c["reg"], **common, **kw)
        r["loss"] = r["epoch_loss"]
    return r


def assert_matches_oracle(c, got, ref):
    assert np.all(np.isfinite(ref["P"])) and np.all(np.isfinite(ref["loss"]))
    np.testing.assert_allclose(got["loss"], ref["loss"], rtol=OBJ_TOL)
    if got["viol"] is not None:
        np.testing.assert_allclose(got["viol"], ref["viol"], rtol=OBJ_TOL)
    np.testing.assert_allclose(got["P"], ref["P"], rtol=1e-8, atol=1e-13)
    np.testing.assert_allclose(got["w"], ref["w"], rtol=1e-8, atol=1e-13)
    assert abs(got["intercept"] - ref["intercept"]) <= 1e-9
    assert got["it"] == ref["it"]
    if c["solver"] == "adagrad":
        np.testing.assert_allclose(got["gsP"], ref["gsP"], rtol=1e-8, atol=1e-14)
        np.testing.assert_allclose(got["gnP"], ref["gnP"], rtol=1e-8, atol=1e-14)
    if c["solver"] == "psgd":
        assert np.array_equal(got["P"] == 0.0, ref["P"] == 0.0)


def assert_forms_agree(a, b):
    """two device forms of one solver: agreement far tighter than the oracle bar"""
    for key in ("P", "w", "loss", "gsP", "gnP"):
        if key in a:
            x, y = np.asarray(a[key]), np.asarray(b[key])
            top = max(float(np.max(np.abs(y))), 1e-300)
            assert float(np.max(np.abs(x - y))) <= FORM_TOL * top, key
    assert abs(a["intercept"] - b["intercept"]) <= FORM_TOL * max(1.0, abs(b["intercept"]))
    assert a["it"] == b["it"]


_PIPE_RESULTS = {}


def pipe_result(c, g, monkeypatch):
    if c["name"] not in _PIPE_RESULTS:
        _PIPE_RESULTS[c["name"]] = device_fit(c, g, monkeypatch)
    return _PIPE_RESULTS[c["name"]]


# ------------------------------------------------------------------------------------------------ 1. the case table
@gpu
@pytest.mark.parametrize("name", [c["name"] for c in CASES])
def test_pipe_matches_oracle(oracle, monkeypatch, name):
    c = CASE_BY_NAME[name]
    g = case_data(c)
    csr = g["csr"]
    assert int(np.max(np.diff(csr.indptr))) + c["n_aug"] == c["zmax"]
    assert route(c["solver"], c["sb8"], c["zmax"], csr.n) == "pipe"
    ref = oracle_fit(oracle, c, csr, g["y"], g["P"], g["w"], g["b"])
    if c["solver"] == "psgd":
        assert 0 < np.count_nonzero(ref["P"] == 0.0) < ref["P"].size          # the prox zeroed some, not all
    assert_matches_oracle(c, pipe_result(c, g, monkeypatch), ref)


# ------------------------------------------------------------------------------------------------ 2. the other forms
@gpu
@pytest.mark.parametrize("name,form", [(c["name"], f) for c in CASES for f in FORMS[c["solver"]]])
def test_other_form_matches_oracle_and_pipe(oracle, monkeypatch, name, form):
    c = CASE_BY_NAME[name]
    expected = FORM_ROUTE[(c["solver"], form)]
    if route(c["solver"], c["sb8"], c["zmax"], N_ROWS, env=form) != expected:
        pytest.skip(f"the {expected} form does not take SB8 = {c['sb8']}, zmax = {c['zmax']}")
    g = case_data(c)
    pipe = pipe_result(c, g, monkeypatch)
    got = device_fit(c, g, monkeypatch, env=form)
    assert_matches_oracle(c, got, oracle_fit(oracle, c, g["csr"], g["y"], g["P"], g["w"], g["b"]))
    assert_forms_agree(pipe, got)


# ------------------------------------------------------------------------------------------------ 3. sample-order edges
# Wide shapes of the table (SB8 = 16..64, rows of 33..64 nonzeros, both prefetch lanes), the SGD / PSGD ones on the
# invscaling schedule, where a step size taken from the wrong slot of the one-ahead table changes the update.
EDGE_CASES = ["sgd_c4", "sgd_d3_augment", "adagrad_c4", "adagrad_d3_augment", "psgd_l21_k32_c4", "psgd_l21_k33"]


def edge_case(name):
    c = dict(CASE_BY_NAME[name])
    if c["solver"] != "adagrad":
        c["sched"] = "invscaling"
    return c


# real nonzeros per row: one row; empty rows first and last; a dataset of empty rows only, where the kernels' zmax
# falls back to max(nAug, 1)
TINY = {"n1": lambda c: [c["zrow"]], "n2": lambda c: [0, c["zrow"]], "n3": lambda c: [0, c["zrow"], 0],
        "n4": lambda c: [0, c["zrow"], c["lo"], 0], "all_empty": lambda c: [0, 0, 0]}


@gpu
@pytest.mark.parametrize("layout", list(TINY))
@pytest.mark.parametrize("name", EDGE_CASES)
def test_tiny_epochs(oracle, monkeypatch, name, layout):
    """epochs of fewer samples than the prefetch ring is deep: the prologue loads samples 0..2 and the loop's
    look-ahead must stop at nRows; three shuffled epochs, the permutations handed to both sides"""
    c = edge_case(name)
    lengths = TINY[layout](c)
    g = case_data(c, rows_csr(lengths, N_FEAT, np.random.default_rng(len(lengths))))
    csr, n = g["csr"], len(lengths)
    zmax = max(max(lengths) + c["n_aug"], 1)
    assert route(c["solver"], c["sb8"], zmax, n) == "pipe"
    perms = np.array([np.random.default_rng(100 + e).permutation(n) for e in range(EPOCHS)])
    ref = oracle_fit(oracle, c, csr, g["y"], g["P"], g["w"], g["b"], perms=perms)
    assert_matches_oracle(c, device_fit(c, g, monkeypatch, perms=perms), ref)


def abi_epoch(c, g, rows):
    """one epoch over a host row list through the C ABI (begin / epoch / end), as SGD.fit, AdaGrad.fit and
    PSGD.fit drive it but with nRows = len(rows) != n; returns the fields assert_matches_oracle reads"""
    lib, ctx = _lib.load(), _lib.ctx()
    csr, kw, lo = g["csr"], solver_kw(c), LOSSES[c["loss"]]()
    fm = make_fm(c, g["P"], g["w"], g["b"])
    ds = nf.newCSRDataset(csr.data, csr.indices, csr.indptr, csr.n, csr.d)
    ds.set_targets(g["y"])
    h = fm._to_device(csr.d)
    idx = _lib.i64(rows)
    it, viol, ls = C.c_int64(1), C.c_double(), C.c_double()
    out = {}
    try:
        if c["solver"] == "sgd":
            cfg = _lib.SgdCfg(lo.kind, lo.threshold, kw["eta0"], kw["alpha0"], kw["alpha"], kw["beta"],
                              _lib.SCHED[kw["scheduling"]], kw["power"])
            _lib.check(lib.nimfm_fm_sgd_begin(ctx, h))
            _lib.check(lib.nimfm_fm_sgd_epoch(ctx, h, ds.handle(), C.byref(cfg), C.byref(it), _lib.ptr(idx), len(idx),
                                              C.byref(viol), C.byref(ls)))
            _lib.check(lib.nimfm_fm_sgd_end(ctx, h))
        elif c["solver"] == "adagrad":
            cfg = _lib.AdagradCfg(lo.kind, lo.threshold, kw["eta0"], kw["alpha0"], kw["alpha"], kw["beta"], 1e-10, 1)
            _lib.check(lib.nimfm_fm_adagrad_init(ctx, h, 1e-10, 1))
            _lib.check(lib.nimfm_fm_adagrad_epoch(ctx, h, ds.handle(), C.byref(cfg), C.byref(it), _lib.ptr(idx),
                                                  len(idx), C.byref(viol), C.byref(ls)))
            state = (len(g["P"]), g["P"].shape[2], c["k"])                 # the solver layout [nOrders, d + nAug, k]
            gs, gn = np.zeros(state), np.zeros(state)
            gsw, gnw, gsb, gnb = np.zeros(csr.d), np.zeros(csr.d), C.c_double(), C.c_double()
            _lib.check(lib.nimfm_fm_adagrad_get_state(ctx, h, _lib.ptr(gs), _lib.ptr(gn), _lib.ptr(gsw), _lib.ptr(gnw),
                                                      C.byref(gsb), C.byref(gnb)))
            _lib.check(lib.nimfm_fm_adagrad_finalize(ctx, h, C.byref(cfg), it.value))
            out.update(gsP=gs, gnP=gn)
        else:
            cfg = _lib.PsgdCfg(lo.kind, lo.threshold, kw["eta0"], kw["alpha0"], kw["alpha"], kw["beta"], kw["gamma"],
                               {"l1": _lib.REG_L1, "l21": _lib.REG_L21}[c["reg"]], _lib.SCHED[kw["scheduling"]],
                               kw["power"])
            _lib.check(lib.nimfm_fm_psgd_begin(ctx, h))
            _lib.check(lib.nimfm_fm_psgd_epoch(ctx, h, ds.handle(), C.byref(cfg), C.byref(it), _lib.ptr(idx), len(idx),
                                               C.byref(ls)))
            _lib.check(lib.nimfm_fm_psgd_end(ctx, h, C.byref(cfg)))
        fm._from_device(h)
    finally:
        lib.nimfm_fm_free(ctx, h)
    out.update(P=fm.P, w=fm.w, intercept=fm.intercept, loss=[ls.value / len(idx)], it=it.value,
               viol=None if c["solver"] == "psgd" else [viol.value])
    return out


@gpu
@pytest.mark.parametrize("name", EDGE_CASES)
def test_row_list_with_repeats(oracle, name):
    """a sequential pass over a row list is a pass over the gathered rows in order: a list longer than the dataset,
    with repeats and runs of one row (the longest one among them), against the oracle on csr_take_rows"""
    c = edge_case(name)
    g = case_data(c, shaped_csr(40, N_FEAT, c["zrow"], c["lo"], seed=len(name)))
    csr = g["csr"]
    rng = np.random.default_rng(5)
    rows = rng.integers(0, csr.n, size=2 * csr.n + 5)
    rows[5:8] = rows[5]                                              # consecutive duplicates
    rows[20:22] = csr.n // 3                                         # the zrow-long row twice in a row
    rows[-1] = 4                                                     # an empty row last
    assert route(c["solver"], c["sb8"], c["zmax"], len(rows)) == "pipe"
    sub = oracle.csr_take_rows(csr, rows)
    ref = oracle_fit(oracle, c, sub, g["y"][rows], g["P"], g["w"], g["b"], max_iter=1)
    assert_matches_oracle(c, abi_epoch(c, g, rows), ref)


@gpu
@pytest.mark.parametrize("name", ["sgd_c4", "psgd_l1_sb96_row64", "psgd_l21_k32_c4"])
def test_warm_start_continues_the_step_size(oracle, monkeypatch, name):
    """SGD and PSGD keep `it` across warm-started fits (optimizers.py: SGD.init runs only without warmStart, PSGD
    resets it only without it), so the second fit's first sample takes eta(it) from where the first fit stopped:
    2 epochs, then 1 more, against the oracle run the same way.  PSGD starts from a preset it.  Where the lazy
    caches fold in exactly (SGD's scalings, L1's threshold) the split run also equals a 3-epoch run; L21's catch-up
    at the end of a fit is not algebraically the same as catching up later (l21.nim:86), so there the oracle is
    split the same way the device run is."""
    c = edge_case(name)
    g = case_data(c)
    csr = g["csr"]
    it0 = 1 if c["solver"] == "sgd" else 41
    for var in ENV.values():
        monkeypatch.delenv(var, raising=False)
    fm = make_fm(c, g["P"], g["w"], g["b"])
    ds = nf.newCSRDataset(csr.data, csr.indices, csr.indptr, csr.n, csr.d)
    opt = new_opt(c, 2)
    if c["solver"] == "psgd":
        opt.it = it0
    fits = []
    for max_iter in (2, 1):
        opt.maxIter = max_iter
        opt.fit(ds, g["y"], fm)
        loss, viol = history(c, opt)
        fits.append(dict(P=fm.P, w=fm.w, intercept=fm.intercept, loss=loss, viol=viol, it=opt.it))
    r2 = oracle_fit(oracle, c, csr, g["y"], g["P"], g["w"], g["b"], max_iter=2, it=it0)
    assert_matches_oracle(c, fits[0], r2)
    ref = oracle_fit(oracle, c, csr, g["y"], r2["P"], r2["w"], r2["intercept"], max_iter=1, it=r2["it"])
    got = fits[1]
    assert_matches_oracle(c, got, ref)
    assert got["it"] == it0 + EPOCHS * csr.n
    if c["reg"] != "l21":
        r3 = oracle_fit(oracle, c, csr, g["y"], g["P"], g["w"], g["b"], max_iter=3, it=it0)
        np.testing.assert_allclose(got["P"], r3["P"], rtol=1e-8, atol=1e-13)
        np.testing.assert_allclose(got["loss"], r3["loss"][-1:], rtol=OBJ_TOL)


@gpu
def test_reset_scaling_in_a_wide_pipe(oracle, monkeypatch):
    """test_fm_sgd_reset_scaling_and_perms's recipe (eta0 = 0.5, alpha = beta = 0.6, constant schedule) at the C4
    width: degree 3, k = 32, rows of 39..64 nonzeros.  With a constant step the scalings after q samples since the
    last reset are (1 - eta0 * beta)^q = 0.7^q (sgd.nim:116-131), below 1e-9 from q = 59 on, so resetScaling fires
    for P and for w at samples 59, 118, 177 and 236 of the three 90-sample epochs: inside every epoch.  That shrink
    takes P to ~1e-40 by the end, so P is also held to the oracle relative to its largest element."""
    c = dict(CASE_BY_NAME["sgd_c4"], zrow=64, lo=39, loss="squared", sched="constant")
    c["zmax"] = c["zrow"]
    n, d = 90, N_FEAT
    g = case_data(c, shaped_csr(n, d, c["zrow"], c["lo"], seed=77))
    kw = dict(eta0=0.5, alpha0=1e-6, alpha=0.6, beta=0.6, scheduling="constant")
    q = int(np.argmax((1 - kw["eta0"] * kw["beta"]) ** np.arange(1, n + 1) < 1e-9)) + 1
    assert q == 59 and all(np.any((np.arange(1, EPOCHS * n + 1) % q == 0)[e * n:(e + 1) * n]) for e in range(EPOCHS))
    assert route("sgd", c["sb8"], c["zmax"], n) == "pipe"
    perms = np.array([np.random.default_rng(200 + e).permutation(n) for e in range(EPOCHS)])
    ref = oracle.sgd_fit(g["csr"], g["y"], g["P"], g["w"], g["b"], c["degree"], "squared", max_iter=EPOCHS,
                         perms=perms, **kw)
    for var in ENV.values():
        monkeypatch.delenv(var, raising=False)
    fm = make_fm(c, g["P"], g["w"], g["b"])
    opt = nf.newSGD(maxIter=EPOCHS, verbose=0, tol=0.0, **kw)
    opt.fit(nf.newCSRDataset(g["csr"].data, g["csr"].indices, g["csr"].indptr, n, d), g["y"], fm, perms=perms)
    got = dict(P=fm.P, w=fm.w, intercept=fm.intercept, loss=[h[1] for h in opt.history],
               viol=[h[0] for h in opt.history], it=opt.it)
    assert_matches_oracle(c, got, ref)
    top = float(np.max(np.abs(ref["P"])))
    assert 0.0 < top < 1e-20
    np.testing.assert_allclose(got["P"] / top, ref["P"] / top, rtol=1e-8, atol=1e-13)


# ------------------------------------------------------------------------------------------------ CPU guard
def test_case_table_covers_every_cell():
    """Checks the case table without a GPU: every value each axis of the pipe kernels' domain asks for has a case
    for every solver it applies to, and every case lands on the pipe by the restated predicates."""
    cells = set()
    for c in CASES:
        s = c["solver"]
        assert route(s, c["sb8"], c["zmax"], N_ROWS) == "pipe", c["name"]
        cells.add((s, "sb8", c["sb8"] if c["sb8"] in (1, 3, 64, 256, 448) else
                   ("odd-not-dividing-512" if c["sb8"] % 2 and 512 % c["sb8"] else
                    ("96-row64" if c["sb8"] == 96 and c["zmax"] == 64 else c["sb8"]))))
        cells.add((s, "row", "one-lane" if c["zmax"] <= 32 else ("64" if c["zmax"] == 64 else "two-lanes")))
        if c["zmax"] == 64:
            cells.add((s, "row", "two-lanes"))
        cells.add((s, "ept", elems_per_thread(c)))
        cells.add((s, "degree", c["degree"], c["fit_lower"]))
        cells.add((s, "fit", c["fit_linear"], c["fit_intercept"]))
        cells.add((s, "loss", c["loss"]))
        if s != "adagrad":
            cells.add((s, "sched", c["sched"]))
        if s == "psgd":
            cells.add((s, "reg", c["reg"]))
            if c["reg"] == "l21":
                cells.add((s, "l21-k", c["k"]))
        # the data: the longest row is exactly zmax - nAug, every 9th row empty, the rest at least lo
        lens = np.diff(case_data(c)["csr"].indptr)
        assert lens.max() == c["zrow"] and np.all(lens[4::9] == 0) and np.count_nonzero(lens == c["zrow"]) >= 1
        assert np.all((lens == 0) | (lens >= c["lo"])), c["name"]
    want = set()
    for s in ("sgd", "adagrad", "psgd"):
        sb8s = [1, 3, "odd-not-dividing-512", 64, "96-row64", 256] + ([448] if s == "sgd" else [])
        want |= {(s, "sb8", v) for v in sb8s}
        want |= {(s, "row", v) for v in ("one-lane", "two-lanes", "64")}
        want |= {(s, "ept", v) for v in (1, 2, 5, 12)}
        want |= {(s, "degree", dg, fl) for dg, fl in [(2, "explicit"), (3, "explicit"), (3, "augment"), (4, "none"),
                                                       (5, "explicit"), (6, "explicit")]}
        want |= {(s, "fit", fl, fi) for fl, fi in [(True, True), (False, True), (True, False)]}
        want |= {(s, "loss", v) for v in LOSSES}
    want |= {("sgd", "sched", v) for v in ("optimal", "constant", "invscaling")}
    want |= {("psgd", "reg", v) for v in ("l1", "l21")}
    want |= {("psgd", "l21-k", k) for k in (1, 7, 8, 31, 32, 33, 64)}
    assert want <= cells, sorted(want - cells, key=str)
    # the AdaGrad pipe's three staged slices: SB8 = 256 fits 34 nonzeros, not 35
    assert adagrad_route(256, 34, 1) == "pipe" and adagrad_route(256, 35, 1) == "staged"
    # the SGD pipe's widest slice: 448 = SGDP_THREADS - 64 and no more, and the staged form stops at 256
    assert sgd_route(448, 13) == "pipe" and sgd_route(449, 13) != "pipe" and sgd_route(448, 13, "staged") == "unstaged"
    assert all(route(s, 96, 64, 1) == "pipe" for s in ("sgd", "adagrad", "psgd"))      # zmax * SB8 = 6144 exactly
    assert sgd_route(97, 64) != "pipe" and psgd_route(97, 64) != "pipe"
