"""Every FM row-kernel route against the oracle past its first persistent wave.

plan_rows (nimfm_b200/csrc/fm_api.cu) picks one of two row kernels per call -- the streaming instances
fm_rows_stream_kernel<D,E,M,KT> or the generic runtime-k kernel -- and caps the grid at occupancy x SMs, so past
one wave every warp grid-strides over several row tiles.  The cases below are built to reach each route naturally (or through the A/B switch), at
n = 3 * n_wave + 7 rows so that every warp takes at least three tiles and the last tile is partial.  This is
where a lost or double-counted tile, a hot-column accumulator flushed at the wrong time, or a chunk boundary off
by one would show, and the oracle restates every one of these operations in float64.

Also here: the sequential-solver fallbacks (SGD / AdaGrad miniBatchSize=1 / PSGD on long rows and wide slices)
and the CD column-kernel block sizes (cd.cu:420)."""
import numpy as np
import pytest

import nimfm_b200 as nf
from oracle import bruteforce as bf
from oracle.oracle import CSR
from helpers import make_dense, make_fm_params, max_rel
from test_gpu_fm import dev_loss_grad

gpu = pytest.mark.gpu

LOSSES = {"squared": nf.Squared, "logistic": nf.Logistic, "squared_hinge": nf.SquaredHinge, "huber": nf.Huber}
LOSS_ORDER = list(LOSSES)
WARPS_PER_SM, ROWS_PER_WARP = 64, 4      # resident warps per SM; rows per warp-tile at KT = 8 (4 groups of 8 lanes)
HOT_SLOTS = 16                            # hot-column table size (dataset.cu:15-46)
STAGE_CAP = 512                           # longest row (maxSegNnz + nAug) the streaming kernel takes


def n_wave(sms):
    """Upper bound on the rows one persistent wave of any row-kernel instance covers."""
    return sms * WARPS_PER_SM * ROWS_PER_WARP


def n_rows(sms):
    """Multi-wave size: every warp takes at least three tiles, and the last tile is partial."""
    return 3 * n_wave(sms) + 7


def expected_route(degree, fit_lower, k, z_max, n_aug, env=None):
    """The row kernel plan_rows (fm_api.cu) selects, the same for every mode (predict, grad, AdaGrad and the stash
    forward of the deterministic route): the streaming instance when one exists for (degree, explicit, k) and the
    longest row incl. dummies fits 512 entries; else the generic kernel.  There is no route query in the ABI, so the
    tests name the route each case is built for and this function is the one place that restates the rule.
    env: NIMFM_ROW_KERNEL (None | "generic")."""
    tuned = degree in (2, 3) and k in (8, 16, 32)
    if env != "generic" and tuned and max(z_max + n_aug, 1) <= STAGE_CAP:
        return "stream"
    return "generic"


# ------------------------------------------------------------------------------------------------ the case table
def _case(name, degree, fit_lower, k, route, modes, n_dense=3, max_extra=10, d=400, long_row=0, spread=False,
          fit_linear=True, forced=()):
    return dict(name=name, degree=degree, fit_lower=fit_lower, k=k, route=route, modes=tuple(modes), n_dense=n_dense,
                max_extra=max_extra, d=d, long_row=long_row, spread=spread, fit_linear=fit_linear, forced=tuple(forced))


PG = ("predict", "grad")
CASES = []
# streaming: degree 2, 3-none, 3-explicit, 3-augment x k in {8, 16, 32}; AdaGrad and the deterministic route rotate
for i, (deg, fl) in enumerate([(2, "explicit"), (3, "none"), (3, "explicit"), (3, "augment")]):
    for j, k in enumerate((8, 16, 32)):
        extra = ("adagrad",) if (i + j) % 2 == 0 else ("det",)
        CASES.append(_case(f"stream_d{deg}_{fl}_k{k}", deg, fl, k, "stream", PG + extra,
                           n_dense=(20, 3, 0)[(i + j) % 3], max_extra=(12, 24, 40)[j], spread=(i + j) % 3 == 1,
                           fit_linear=(i + j) % 4 != 3, forced=("generic",)))
# generic, reached naturally: k not in {8,16,32}; degree 4-6; a single row past 512 entries
for deg, fl, k in [(3, "explicit", 12), (2, "explicit", 33), (2, "explicit", 64)]:
    CASES.append(_case(f"generic_d{deg}_{fl}_k{k}", deg, fl, k, "generic", PG + ("adagrad",), n_dense=20, max_extra=12))
for i, (deg, fl) in enumerate([(d_, f_) for d_ in (4, 5, 6) for f_ in ("explicit", "none", "augment")]):
    CASES.append(_case(f"generic_d{deg}_{fl}", deg, fl, (4, 8, 16)[i % 3], "generic", PG + ("adagrad",),
                       n_dense=(20, 3, 0)[i % 3], max_extra=8, d=120, fit_linear=i % 2 == 0))
for deg, fl, k, L in [(2, "explicit", 8, 1100), (2, "explicit", 32, 700), (3, "explicit", 32, 600),
                      (3, "augment", 8, 1100)]:
    CASES.append(_case(f"longrow_d{deg}_{fl}_k{k}", deg, fl, k, "generic", PG + ("adagrad",), n_dense=20,
                       max_extra=12, d=1200, long_row=L))
# the 512 boundary: maxSegNnz + nAug = 512 streams, 513 does not -- with augment the dummy feature tips it over
for deg, fl, L, route in [(2, "explicit", 512, "stream"), (2, "explicit", 513, "generic"),
                          (3, "augment", 511, "stream"), (3, "augment", 512, "generic")]:
    CASES.append(_case(f"boundary_d{deg}_{fl}_row{L}", deg, fl, 8, route, PG, n_dense=20, max_extra=12, d=700,
                       long_row=L))
CASE_BY_NAME = {c["name"]: c for c in CASES}


def case_data(c, sms, seed):
    """A seeded dataset + model for case c at the multi-wave size: empty and ragged rows, c["n_dense"]
    always-present columns, stored exact zeros, values over 1e-3..1e3 when c["spread"], one row of c["long_row"]
    entries in the middle, non-unit lams."""
    rng = np.random.default_rng(seed)
    n, d, nd, m = n_rows(sms), c["d"], c["n_dense"], c["max_extra"]
    width = (d - nd) // m
    fill = rng.random(n)                                            # ragged: each row its own fill rate
    extra = rng.random((n, m)) < fill[:, None]
    empty = rng.random(n) < 0.05
    extra[empty] = False
    cols = np.concatenate([np.broadcast_to(np.arange(nd), (n, nd)),
                           nd + np.arange(m) * width + rng.integers(0, width, size=(n, m))], axis=1)
    mask = np.concatenate([np.broadcast_to(~empty[:, None], (n, nd)), extra], axis=1)
    lens = mask.sum(axis=1)
    indices = cols[mask]                                            # row-major: ascending within a row
    if c["long_row"]:
        r, L = n // 2, c["long_row"]
        lo, hi = int(lens[:r].sum()), int(lens[:r + 1].sum())
        indices = np.concatenate([indices[:lo], np.sort(rng.choice(d, size=L, replace=False)), indices[hi:]])
        lens[r] = L
    nnz = len(indices)
    if c["spread"]:
        data = np.where(rng.random(nnz) < 0.5, -1.0, 1.0) * 10.0 ** rng.uniform(-3, 3, nnz)
    else:
        data = rng.standard_normal(nnz) * 0.8
    data[rng.random(nnz) < 0.02] = 0.0                              # stored exact zeros
    csr = CSR(data, indices, np.concatenate([[0], np.cumsum(lens)]), n, d)
    deg, fl, k = c["degree"], c["fit_lower"], c["k"]
    nO, nA = bf.n_orders(deg, fl), bf.n_augments(deg, fl, c["fit_linear"])
    scale = 0.05 if c["spread"] else 0.15
    P = rng.standard_normal((nO, k, d + nA)) * scale
    w = rng.standard_normal(d) * 0.1 if c["fit_linear"] else np.zeros(d)
    loss = LOSS_ORDER[seed % len(LOSS_ORDER)]
    y = rng.standard_normal(n) if loss in ("squared", "huber") else np.sign(rng.standard_normal(n))
    return dict(csr=csr, P=P, w=w, b=0.1, lams=rng.random(k) + 0.5, y=y, loss=loss, n_aug=nA, rng=rng)


def find_hot_candidates(csr, max_sample=16384):
    """Columns that qualify as hot under dataset.cu:15-46 (before the table keeps the 16 most frequent)."""
    stride = max(1, csr.n // max_sample)
    rows = np.arange(0, csr.n, stride)
    cnt = np.zeros(csr.d, np.int64)
    for r in rows:
        cnt[csr.indices[csr.indptr[r]:csr.indptr[r + 1]]] += 1
    return int(np.count_nonzero((cnt * 16 >= len(rows)) & (cnt >= 2)))


def case_seed(c):
    return 7000 + CASES.index(c)


# ------------------------------------------------------------------------------------------------ helpers
@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def make_fm(c, g):
    task = nf.regression if g["loss"] in ("squared", "huber") else nf.classification
    fm = nf.newFactorizationMachine(task, degree=c["degree"], nComponents=c["k"], fitLower=c["fit_lower"],
                                    fitLinear=c["fit_linear"], fitIntercept=True, warmStart=True)
    fm.P, fm.w, fm.intercept, fm.isInitialized = g["P"].copy(), g["w"].copy(), g["b"], True
    fm.lams = g["lams"].copy()       # predict applies them; the gradient does not (minibatch_psgd.nim:67-88)
    return fm


def csr_ds(csr):
    ds = nf.newCSRDataset(csr.data, csr.indices, csr.indptr, csr.n, csr.d)
    ds.handle()
    return ds


def assert_grad_matches(got, ref):
    ls, gP, gw, gb = got
    assert abs(ls - ref["loss"]) <= 1e-10 * max(1.0, abs(ref["loss"]))
    # (rows with one nonzero have an exactly-cancelling ANOVA derivative: rounding noise on both sides, hence atol)
    scale = max(float(np.max(np.abs(ref["gP"]))), 1e-12)
    np.testing.assert_allclose(gP, ref["gP"], rtol=1e-9, atol=max(1e-9 * scale, 1e-15))
    assert max_rel(gw, ref["gw"]) <= 1e-9
    assert abs(gb - ref["gb"]) <= 1e-10 * max(1.0, abs(ref["gb"]))


# ------------------------------------------------------------------------------------------------ the route matrix
@gpu
@pytest.mark.parametrize("name", [c["name"] for c in CASES])
def test_row_route_matches_oracle(oracle, monkeypatch, sms, name):
    c = CASE_BY_NAME[name]
    g = case_data(c, sms, case_seed(c))
    csr, y, P, w, b, deg = g["csr"], g["y"], g["P"], g["w"], g["b"], c["degree"]
    n = csr.n
    assert n >= 3 * n_wave(sms)
    z_max = int(np.max(np.diff(csr.indptr)))
    assert expected_route(deg, c["fit_lower"], c["k"], z_max, g["n_aug"]) == c["route"]
    lo = LOSSES[g["loss"]]()
    fm = make_fm(c, g)
    ds = csr_ds(csr)
    ds.set_targets(y)
    monkeypatch.delenv("NIMFM_ROW_KERNEL", raising=False)
    monkeypatch.delenv("NIMFM_DETERMINISTIC", raising=False)

    ref_pred = oracle.fm_decision_function(csr, P, w, b, deg, lams=g["lams"])
    preds = {None: fm.decisionFunction(ds)}
    assert max_rel(preds[None], ref_pred) <= 1e-10

    # predict+grad over a row list with repeats, and over a cursor that wraps past n
    rows = g["rng"].integers(0, n, size=n + 7)
    start = n // 3
    wrap = (start + np.arange(n - 5)) % n
    refs = [oracle.fm_loss_grad(oracle.csr_take_rows(csr, r), y[r], P, w, b, deg, g["loss"],
                                fit_linear=c["fit_linear"], mini_batch_size=len(r)) for r in (rows, wrap)]

    def grads():
        assert_grad_matches(dev_loss_grad(fm, ds, y, lo, rows=rows, mb=len(rows)), refs[0])
        assert_grad_matches(dev_loss_grad(fm, ds, y, lo, row_begin=start, n_rows=len(wrap), mb=len(wrap)), refs[1])

    grads()
    for env in c["forced"]:
        monkeypatch.setenv("NIMFM_ROW_KERNEL", env)
        preds[env] = fm.decisionFunction(ds)
        assert max_rel(preds[env], ref_pred) <= 1e-10
        grads()
    monkeypatch.delenv("NIMFM_ROW_KERNEL", raising=False)
    # stream and generic share their arithmetic and summation structure (fm_rows_stream.cuh, header): the decision
    # values are the same bits whichever kernel computes them
    for env in c["forced"]:
        assert np.array_equal(preds[env], preds[None]), (env, float(np.max(np.abs(preds[env] - preds[None]))))

    if "det" in c["modes"]:
        monkeypatch.setenv("NIMFM_DETERMINISTIC", "1")
        ref = oracle.fm_loss_grad(csr, y, P, w, b, deg, g["loss"], fit_linear=c["fit_linear"], mini_batch_size=n)
        got = dev_loss_grad(fm, ds, y, lo, row_begin=0, n_rows=n, mb=n)
        assert_grad_matches(got, ref)
        again = dev_loss_grad(fm, ds, y, lo, row_begin=0, n_rows=n, mb=n)
        assert got[0] == again[0] and got[3] == again[3]
        assert np.array_equal(got[1], again[1]) and np.array_equal(got[2], again[2])
        monkeypatch.delenv("NIMFM_DETERMINISTIC")

    if "adagrad" in c["modes"]:
        # two minibatches per epoch: one of two waves, one of the rest (partial last tile)
        mb = 2 * n_wave(sms) + 3
        kw = dict(eta0=0.05, alpha0=1e-6, alpha=1e-3, beta=1e-3)
        r = oracle.adagrad_fit(csr, y, P, w, b, deg, g["loss"], c["fit_linear"], True, max_iter=2,
                               mini_batch_size=mb, **kw)
        fm2 = make_fm(c, g)
        opt = nf.newAdaGrad(maxIter=2, loss=lo, miniBatchSize=mb, verbose=0, tol=0.0, shuffle=False, **kw)
        opt.fit(ds, y, fm2)
        np.testing.assert_allclose([h[1] for h in opt.history], r["loss"], rtol=1e-8)
        np.testing.assert_allclose(fm2.P, r["P"], rtol=1e-8, atol=1e-13)
        np.testing.assert_allclose(fm2.w, r["w"], rtol=1e-8, atol=1e-13)
        assert abs(fm2.intercept - r["intercept"]) <= 1e-9 * max(1.0, abs(r["intercept"]))
        np.testing.assert_allclose(opt.g_sum["P"], r["state"]["gsP"], rtol=1e-8, atol=1e-14)
        np.testing.assert_allclose(opt.g_norm["P"], r["state"]["gnP"], rtol=1e-8, atol=1e-14)


@gpu
@pytest.mark.parametrize("degree", [4, 5, 6])
@pytest.mark.parametrize("fit_lower", ["explicit", "none", "augment"])
def test_high_degree_vs_bruteforce(degree, fit_lower):
    """degrees the tuned kernels do not cover, straight against the subset-enumeration definition
    (kernels_slow.nim): guards against the oracle and the generic kernel sharing a DP mistake"""
    n, d, k = 9, 9, 3
    X = make_dense(n, d, 50 + degree, density=0.8, positive=False)
    X[0] = 0.0                                                       # an empty row
    P, w, _ = make_fm_params(d, degree, k, fit_lower, True, seed=degree, scale=0.4)
    fm = nf.newFactorizationMachine(nf.regression, degree=degree, nComponents=k, fitLower=fit_lower, warmStart=True)
    fm.P, fm.w, fm.intercept, fm.isInitialized = P.copy(), w.copy(), -0.3, True
    csr = CSR.from_dense(X)
    got = fm.decisionFunction(csr_ds(csr))
    assert max_rel(got, bf.fm_decision_function(X, P, w, -0.3, degree)) <= 1e-9


# ------------------------------------------------------------------------------------------------ CPU guard
@pytest.mark.parametrize("n_sms", [1, 8, 132, 148, 160])
def test_route_table_covers_every_cell(n_sms):
    """Checks the case table without a GPU: every route x mode cell has a case, the multi-wave size is at least
    three waves, long rows cross 512 once nAug is counted, and the 20-column cases overflow the hot table."""
    cells = set()
    for c in CASES:
        for mode in c["modes"]:
            cells.add((c["route"], mode))
        for env in c["forced"]:
            for mode in PG:
                cells.add((f"forced-{env}", mode))
        if c["long_row"]:
            cells.add(("long-row", c["degree"], c["k"]))
        if c["name"].startswith("boundary"):
            cells.add(("boundary", c["route"], c["fit_lower"]))
        if c["route"] == "stream":
            cells.add(("stream-shape", c["degree"], c["fit_lower"], c["k"]))
        if c["degree"] >= 4:
            cells.add(("high-degree", c["degree"], c["fit_lower"]))
        if c["k"] not in (8, 16, 32):
            cells.add(("generic-k", c["k"]))
    want = {("stream", m) for m in ("predict", "grad", "adagrad", "det")}
    want |= {("generic", m) for m in ("predict", "grad", "adagrad")}
    want |= {("forced-generic", m) for m in PG}
    want |= {("long-row", dg, k) for dg in (2, 3) for k in (8, 32)}
    want |= {("boundary", r, fl) for r in ("stream", "generic") for fl in ("explicit", "augment")}
    want |= {("stream-shape", 2, "explicit", k) for k in (8, 16, 32)}
    want |= {("stream-shape", 3, fl, k) for fl in ("none", "explicit", "augment") for k in (8, 16, 32)}
    want |= {("high-degree", dg, fl) for dg in (4, 5, 6) for fl in ("explicit", "none", "augment")}
    want |= {("generic-k", k) for k in (12, 33, 64)}
    assert want <= cells, sorted(want - cells, key=str)

    assert n_rows(n_sms) >= 3 * n_wave(n_sms) and n_rows(n_sms) % ROWS_PER_WARP != 0
    if n_sms != 1:
        return
    for c in CASES:     # the data checks: at one SM's size, which shapes rows the same way as the full size
        g = case_data(c, n_sms, case_seed(c))
        csr = g["csr"]
        z_max = int(np.max(np.diff(csr.indptr)))
        deg, fl, k = c["degree"], c["fit_lower"], c["k"]
        assert expected_route(deg, fl, k, z_max, g["n_aug"]) == c["route"], c["name"]
        if c["long_row"]:
            assert z_max == c["long_row"]
            if not c["name"].startswith("boundary"):
                assert z_max + g["n_aug"] > STAGE_CAP
        if c["name"].startswith("boundary"):
            assert z_max + g["n_aug"] == (STAGE_CAP if c["route"] == "stream" else STAGE_CAP + 1)
        if c["n_dense"] == 20:
            assert find_hot_candidates(csr) > HOT_SLOTS, c["name"]
        lens = np.diff(csr.indptr)
        assert np.any(lens == 0) and len(np.unique(lens)) > 3          # empty and ragged rows
        assert np.any(csr.data == 0.0)                                  # stored exact zeros
        if c["spread"]:
            a = np.abs(csr.data[csr.data != 0.0])
            assert a.min() < 1e-2 and a.max() > 1e2
    # the losses rotate by seed: every loss appears on some case of every route
    for route in ("stream", "generic"):
        assert {LOSS_ORDER[case_seed(c) % 4] for c in CASES if c["route"] == route} == set(LOSS_ORDER)


# ------------------------------------------------------------------------------------------------ sequential solvers
def long_row_csr(n, d, lo, hi, seed):
    """rows of lo..hi nonzeros (sorted unique columns), every 9th row empty"""
    rng = np.random.default_rng(seed)
    data, indices, indptr = [], [], [0]
    for i in range(n):
        z = 0 if i % 9 == 4 else int(rng.integers(lo, hi + 1))
        indices.extend(np.sort(rng.choice(d, size=z, replace=False)).tolist())
        data.extend((rng.standard_normal(z) * 0.3).tolist())
        indptr.append(len(indices))
    return CSR(data, indices, indptr, n, d)


# (name, solver, degree, fit_lower, k, row lengths, NIMFM_SGD_KERNEL).  The pipelined kernels take rows of at most 64
# nonzeros (sgd.cu:731, fm_api.cu:1017, psgd.cu:781); longer rows go to the staged kernels, and an SGD slice of more
# than 256 doubles that does not fit the pipeline (zmax * SB8 > 6144) to the unstaged sgd_epoch_kernel.
SEQ_CASES = [
    ("sgd_staged_long_rows", "sgd", 3, "explicit", 8, (65, 300), None),
    ("sgd_unstaged_wide_slice", "sgd", 4, "explicit", 100, (21, 30), None),
    ("sgd_forced_staged", "sgd", 3, "explicit", 32, (39, 39), "staged"),
    ("sgd_forced_unstaged", "sgd", 3, "explicit", 32, (39, 39), "unstaged"),
    ("adagrad_seq_long_rows", "adagrad", 3, "augment", 16, (65, 200), None),
    ("psgd_l1_long_rows", "psgd_l1", 2, "explicit", 8, (65, 200), None),
    ("psgd_l21_long_rows", "psgd_l21", 3, "explicit", 8, (65, 200), None),
]


@gpu
@pytest.mark.parametrize("case", SEQ_CASES, ids=[c[0] for c in SEQ_CASES])
def test_sequential_fallbacks_match_oracle(oracle, monkeypatch, case):
    name, solver, degree, fit_lower, k, (lo, hi), env = case
    monkeypatch.delenv("NIMFM_ADAGRAD_SEQ", raising=False)
    monkeypatch.delenv("NIMFM_PSGD_KERNEL", raising=False)
    if env:
        monkeypatch.setenv("NIMFM_SGD_KERNEL", env)
    else:
        monkeypatch.delenv("NIMFM_SGD_KERNEL", raising=False)
    n, d = 300, 400
    csr = long_row_csr(n, d, lo, hi, seed=len(name))
    z_max = int(np.max(np.diff(csr.indptr)))
    if lo > 64:
        assert z_max > 64                                             # past the pipelined kernels
    if k == 100:
        assert (degree - 1) * k > 256 and z_max * (degree - 1) * k > 6144
    y = np.random.default_rng(3).standard_normal(n)
    P, w, _ = make_fm_params(d, degree, k, fit_lower, True, seed=k + degree, scale=0.03)
    fm = nf.newFactorizationMachine(nf.regression, degree=degree, nComponents=k, fitLower=fit_lower, warmStart=True)
    fm.P, fm.w, fm.intercept, fm.isInitialized = P.copy(), w.copy(), 0.1, True
    ds = nf.newCSRDataset(csr.data, csr.indices, csr.indptr, n, d)
    kw = dict(eta0=0.01, alpha0=1e-6, alpha=1e-3, beta=1e-3)
    if solver == "sgd":
        ref = oracle.sgd_fit(csr, y, P, w, 0.1, degree, "squared", max_iter=2, **kw)
        opt = nf.newSGD(maxIter=2, verbose=0, tol=0.0, shuffle=False, **kw)
        hist = lambda: [h[1] for h in opt.history]
        ref_hist = ref["loss"]
    elif solver == "adagrad":
        ref = oracle.adagrad_fit(csr, y, P, w, 0.1, degree, "squared", max_iter=2, mini_batch_size=1, **kw)
        opt = nf.newAdaGrad(maxIter=2, verbose=0, tol=0.0, shuffle=False, miniBatchSize=1, **kw)
        hist = lambda: [h[1] for h in opt.history]
        ref_hist = ref["loss"]
    else:
        reg = solver.split("_")[1]
        kw["gamma"] = 1e-2 if reg == "l21" else 3e-3                  # zeroes some coordinates, not all
        ref = oracle.psgd_fit(csr, y, P, w, 0.1, degree, "squared", max_iter=2, reg=reg, **kw)
        opt = nf.newPSGD(maxIter=2, reg={"l1": nf.newL1, "l21": nf.newL21}[reg](), verbose=0, tol=0.0, shuffle=False,
                         **kw)
        opt.it = 1
        hist = lambda: opt.history
        ref_hist = ref["epoch_loss"]
        assert 0 < np.count_nonzero(ref["P"] == 0.0) < ref["P"].size     # the prox really acted
    opt.fit(ds, y, fm)
    assert np.all(np.isfinite(ref["P"]))
    np.testing.assert_allclose(hist(), ref_hist, rtol=1e-8)
    np.testing.assert_allclose(fm.P, ref["P"], rtol=1e-8, atol=1e-13)
    np.testing.assert_allclose(fm.w, ref["w"], rtol=1e-8, atol=1e-13)
    assert abs(fm.intercept - ref["intercept"]) <= 1e-9
    assert opt.it == ref["it"]
    if solver.startswith("psgd"):
        assert np.array_equal(fm.P == 0.0, ref["P"] == 0.0)


# ------------------------------------------------------------------------------------------------ CD block sizes
CD_LENGTH_BOUNDS = (48, 256, 2048)   # longest column of a batch: warp per column / 128 / 256 / 1024 threads (cd.cu:420)


def cd_columns_csr(seed, n=5000):
    """Columns of every length class of the CD column kernel, in ascending order of length so that each class
    forms batches of its own: under 48 rows, 49-256, 257-2048, and two past 2048 (one in every row)."""
    rng = np.random.default_rng(seed)
    lengths = np.concatenate([rng.integers(5, 48, 16), rng.integers(49, 257, 6), rng.integers(257, 2049, 4),
                              [3000, n]])
    X = np.zeros((n, len(lengths)))
    for j, L in enumerate(np.sort(lengths)):
        X[rng.choice(n, size=L, replace=False), j] = rng.standard_normal(L) * 0.5
    rows = [np.nonzero(X[i])[0] for i in range(n)]
    indptr = np.concatenate([[0], np.cumsum([len(r) for r in rows])])
    idx = np.concatenate(rows)
    csr = CSR(X[np.repeat(np.arange(n), np.diff(indptr)), idx], idx, indptr, n, X.shape[1])
    return csr, np.sort(lengths)


@gpu
@pytest.mark.parametrize("solver,degree,fit_lower", [("cd", 2, "explicit"), ("cd", 3, "augment"), ("pcd", 3, "explicit")])
def test_cd_block_sizes_match_oracle(oracle, monkeypatch, solver, degree, fit_lower):
    """every block shape of the CD column kernel, with and without the captured epoch graph (NIMFM_CD_GRAPH=0)"""
    csr, lengths = cd_columns_csr(11 + degree)
    for bound in CD_LENGTH_BOUNDS:
        assert np.any(lengths <= bound) and np.any(lengths > bound)
    csc = oracle.csr_to_csc(csr)
    n, d, k = csr.n, csr.d, 4
    y = np.random.default_rng(degree).standard_normal(n)
    P, w, _ = make_fm_params(d, degree, k, fit_lower, True, seed=9, scale=0.1)
    kw = dict(alpha0=1e-6, alpha=1e-3, beta=1e-3)
    if solver == "cd":
        ref = oracle.cd_fit(csc, y, P, w, 0.0, degree, "squared", True, True, max_iter=3, **kw)
    else:
        kw["gamma"] = 2e-2
        ref = oracle.pcd_fit(csc, y, P, w, 0.0, degree, "squared", True, True, max_iter=3, reg="l1", **kw)
        assert np.count_nonzero(ref["P"] == 0.0) > 0
    got = {}
    for graph in (None, "0"):
        if graph:
            monkeypatch.setenv("NIMFM_CD_GRAPH", graph)
        else:
            monkeypatch.delenv("NIMFM_CD_GRAPH", raising=False)
        fm = nf.newFactorizationMachine(nf.regression, degree=degree, nComponents=k, fitLower=fit_lower, warmStart=True)
        fm.P, fm.w, fm.intercept, fm.isInitialized = P.copy(), w.copy(), 0.0, True
        ds = nf.newCSCDataset(csc.data, csc.indices, csc.indptr, n, d)
        opt = (nf.newCD(maxIter=3, verbose=0, tol=0.0, **kw) if solver == "cd"
               else nf.newPCD(maxIter=3, verbose=0, tol=0.0, reg=nf.newL1(), **kw))
        opt.fit(ds, y, fm)
        h = np.array(opt.history)
        np.testing.assert_allclose(h[:, 0], ref["viol"], rtol=1e-8)
        np.testing.assert_allclose(h[:, 1], ref["loss"], rtol=1e-8)
        if solver == "cd":
            assert abs((h[-1, 1] + h[-1, 2]) - (ref["loss"][-1] + ref["reg"][-1])) <= 1e-8 * abs(ref["loss"][-1] + ref["reg"][-1])
        else:
            assert np.array_equal(fm.P == 0.0, ref["P"] == 0.0)
        np.testing.assert_allclose(fm.P, ref["P"], rtol=1e-8, atol=1e-12)
        np.testing.assert_allclose(fm.w, ref["w"], rtol=1e-8, atol=1e-12)
        assert abs(fm.intercept - ref["intercept"]) <= 1e-8 * max(1.0, abs(ref["intercept"]))
        got[graph] = (h, fm.P, fm.w, fm.intercept)
    # the graph replays the same launches: the same bits
    (h1, P1, w1, b1), (h2, P2, w2, b2) = got[None], got["0"]
    assert np.array_equal(h1, h2) and np.array_equal(P1, P2) and np.array_equal(w1, w2) and b1 == b2
