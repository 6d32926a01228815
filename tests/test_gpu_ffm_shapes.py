"""FFM at the shapes the staged block-per-row kernel cannot hold in shared memory, against the oracle.

ffm_plan_mode (nimfm_b200/csrc/ffm.cu) takes a pair kernel when k is 4/8/16/32, the longest row has at most 1024
nonzeros, d * nFields < 2^31 and (AdaGrad) no row repeats a field; otherwise the staged ffm_rows_kernel, which
copies the row's z x nFields x k slices into shared memory; and where those do not fit, the (nonzero, field) kernel
ffm_units_kernel (ffm_units.cuh), whose shared memory does not grow with nFields x k and which takes rows past
2048 nonzeros through a global scratch area.  Each case below is built to land on the unit kernel and is run
through every FFM entry point -- decisionFunction, predict+grad over a contiguous range and over a row list with
repeats, AdaGrad at miniBatchSize 1 and > 1, minibatch SGD -- at n >= 3 waves of the persistent grid, so every
block handles several rows.  NIMFM_FFM_KERNEL=units forces the unit kernel onto shapes the other kernels serve."""
import ctypes as C

import numpy as np
import pytest

import nimfm_b200 as nf
from nimfm_b200 import _lib
from oracle.oracle import CSR
from helpers import max_rel, sums_agree
from test_gpu_ffm_sgd import field_ds, make_ffm, one_per_field_csr, ragged_field_csr

gpu = pytest.mark.gpu

DEC_TOL, GRAD_TOL, FIT_TOL = 1e-10, 1e-9, 1e-8
SMEM_OPTIN = 232448               # opt-in shared memory per block on the B200 (227 KB)
PAIR_KS = (4, 8, 16, 32)          # ranks with pair-kernel instances
PAIR_MAXZ = 1024                  # longest row the pair kernels take
UNITS_SMEM_CAP = 2048             # longest row the unit kernel buckets in shared memory
UNIT_BLOCKS_PER_SM = 8            # upper bound on resident 256-thread blocks of the unit kernel


def staged_smem_bytes(max_z, n_fields, k):
    """ffm_smem_bytes (ffm.cu): the staged kernel's slices, records, order and two field tables."""
    ch = max(max_z, 1)
    b = ((ch * n_fields * k * 8 + 15) & ~15) + ch * 16 + ch * 4 + (n_fields + 1) * 8
    return (b + 15) & ~15


def expected_route(k, n_fields, d, max_z, mode, field_dups, env=None):
    """The FFM kernel ffm_plan_mode selects ("pair" | "staged" | "units" | "units_long"; the last is the unit kernel
    with rows past its shared-memory cap).  There is no route query in the ABI, so this is the one place that
    restates the rule.  env: NIMFM_FFM_KERNEL (None | "units")."""
    long = "units_long" if max(max_z, 1) > UNITS_SMEM_CAP else "units"
    if env == "units":
        return long
    pair = k in PAIR_KS and max(max_z, 1) <= PAIR_MAXZ and d * n_fields < 2 ** 31 - 1
    if pair and not (mode == "adagrad" and field_dups):
        return "pair"
    return "staged" if staged_smem_bytes(max_z, n_fields, k) <= SMEM_OPTIN else long


# ------------------------------------------------------------------------------------------------ the case table
def field_rows(n, d, n_fields, lengths, seed, layout):
    """Rows with distinct feature ids; layout "one_per_field" (the C5 shape: every field once, in a shuffled order)
    or "multi" (fields drawn independently, so they repeat within a row).  Row 0 is empty, row 1 holds one nonzero,
    row 2 puts all its nonzeros in one field; about 5 % of the values are stored zeros."""
    rng = np.random.default_rng(seed)
    data, indices, fields, indptr = [], [], [], [0]
    for i in range(n):
        z = n_fields if layout == "one_per_field" else int(lengths[i])
        z = 0 if i == 0 else (1 if i == 1 else z)
        ids = np.sort(rng.choice(d, size=z, replace=False))
        if i == 2:
            fs = np.full(z, rng.integers(n_fields))
        elif layout == "one_per_field" and z == n_fields:
            fs = rng.permutation(n_fields)
        else:
            fs = rng.integers(0, n_fields, z)
        x = np.where(rng.random(z) < 0.3, 1.0, rng.standard_normal(z))
        x[rng.random(z) < 0.05] = 0.0
        indices.extend(ids.tolist())
        fields.extend(fs.tolist())
        data.extend(x.tolist())
        indptr.append(len(indices))
    return CSR(np.array(data), np.array(indices, np.int64), np.array(indptr, np.int64), n, d,
               fields=np.array(fields, np.int64), n_fields=n_fields)


def _lengths(kind):
    def f(n, rng):
        if kind == "long":   # short ragged rows, rows of about 1 500 nonzeros, and a few past the shared-memory cap
            z = rng.integers(2, 40, n)
            z[rng.choice(np.arange(3, n), 24, replace=False)] = rng.integers(1400, 1600, 24)
            z[[5, 40, n - 1]] = (2300, 2100, 2400)
            return z
        lo, hi = kind
        return rng.integers(lo, hi + 1, n)
    return f


def _case(name, k, n_fields, d, layout, lengths, modes=("predict", "grad", "adagrad"), fit_rows=None):
    """fit_rows: rows the minibatch solvers run on (all when None; the oracle's solvers cost nFields x d x k per row)"""
    return dict(name=name, k=k, n_fields=n_fields, d=d, layout=layout, lengths=lengths, modes=modes, fit_rows=fit_rows)


CASES = [
    _case("c5_k20", 20, 39, 2000, "one_per_field", None),
    _case("c5_k64", 64, 39, 2000, "one_per_field", None),
    _case("multihot_k10", 10, 39, 2000, "multi", _lengths((80, 300))),
    _case("adagrad_dups_k8", 8, 39, 2000, "multi", _lengths((60, 130)), modes=("adagrad",)),
    _case("k1_odd", 1, 151, 1000, "multi", _lengths((100, 200))),
    _case("k3_odd", 3, 39, 1000, "multi", _lengths((150, 260))),
    _case("k33_odd", 33, 13, 500, "multi", _lengths((40, 80))),
    _case("long_k8", 8, 39, 5000, "multi", _lengths("long")),
    _case("fields1e4_k10", 10, 10000, 16, "multi", _lengths((5, 16)), fit_rows=600),
]
CASE_IDS = [c["name"] for c in CASES]


def case_by_name(name):
    return next(c for c in CASES if c["name"] == name)


def case_data(c, n):
    seed = 500 + CASE_IDS.index(c["name"])
    rng = np.random.default_rng(seed)
    lengths = c["lengths"](n, rng) if c["lengths"] else None
    csr = field_rows(n, c["d"], c["n_fields"], lengths, seed, c["layout"])
    max_z = int(np.max(np.diff(csr.indptr)))
    scale = (max(max_z, 1) * np.sqrt(c["k"])) ** -0.5
    P = rng.standard_normal((c["n_fields"], c["d"], c["k"])) * scale
    w = rng.standard_normal(c["d"]) * 0.1
    y = np.sign(rng.standard_normal(n))
    return csr, P, w, y


def has_field_dups(csr):
    for i in range(csr.n):
        f = csr.fields[csr.indptr[i]:csr.indptr[i + 1]]
        if len(np.unique(f)) != len(f):
            return True
    return False


def sub_rows(csr, rows):
    """the rows `rows` (repeats kept) as a CSR of their own"""
    data, indices, fields, indptr = [], [], [], [0]
    for r in rows:
        a, b = csr.indptr[r], csr.indptr[r + 1]
        data.append(csr.data[a:b]); indices.append(csr.indices[a:b]); fields.append(csr.fields[a:b])
        indptr.append(indptr[-1] + b - a)
    cat = lambda xs, dt: np.concatenate(xs).astype(dt) if xs else np.zeros(0, dt)
    return CSR(cat(data, np.float64), cat(indices, np.int64), np.array(indptr, np.int64), len(rows), csr.d,
               fields=cat(fields, np.int64), n_fields=csr.n_fields)


# ------------------------------------------------------------------------------------------------ CPU guard
def test_case_table_routes():
    """Every case lands on the unit kernel in the modes it was built for, and the staged kernel needs more than
    the opt-in shared memory there (so these shapes were refused before the unit kernel existed)."""
    n = 3 * UNIT_BLOCKS_PER_SM * 148 + 7
    seen_long = False
    for c in CASES:
        csr, _, _, _ = case_data(c, n)
        max_z = int(np.max(np.diff(csr.indptr)))
        dups = has_field_dups(csr)
        assert dups   # the all-one-field row repeats a field in every case
        assert staged_smem_bytes(max_z, c["n_fields"], c["k"]) > SMEM_OPTIN, c["name"]
        for mode in c["modes"]:
            route = expected_route(c["k"], c["n_fields"], c["d"], max_z, mode, dups)
            assert route.startswith("units"), (c["name"], mode, route)
            seen_long |= route == "units_long"
        lens = np.diff(csr.indptr)
        assert lens[0] == 0 and lens[1] == 1 and np.any(csr.data == 0.0)
        f2 = csr.fields[csr.indptr[2]:csr.indptr[3]]
        assert len(f2) > 1 and np.all(f2 == f2[0])
        for i in range(csr.n):   # no repeated feature id within a row
            ids = csr.indices[csr.indptr[i]:csr.indptr[i + 1]]
            assert len(np.unique(ids)) == len(ids)
    assert seen_long
    c = case_by_name("long_k8")
    csr, _, _, _ = case_data(c, n)
    lens = np.diff(csr.indptr)
    assert np.sum((lens >= 1400) & (lens < 1600)) >= 20 and np.sum(lens > UNITS_SMEM_CAP) >= 3
    # the C5 row shape at rank 20 needs 243 360 B of slices alone
    assert 39 * 39 * 20 * 8 == 243360 and expected_route(20, 39, 1950, 39, "predict", False) == "units"
    # the forced shapes below keep their kernels by default
    assert expected_route(8, 39, 1950, 39, "grad", False) == "pair"
    assert expected_route(5, 6, 120, 64, "grad", True) == "staged"
    assert expected_route(8, 6, 120, 64, "grad", True, env="units") == "units"


# ------------------------------------------------------------------------------------------------ GPU helpers
@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def n_rows(sms):
    """three waves of the largest possible unit-kernel grid, plus a partial one"""
    return 3 * UNIT_BLOCKS_PER_SM * sms + 7


def dev_loss_grad(m, ds, y, loss, row_begin=0, n=None, rows=None, mb=None):
    lib, ctx = _lib.load(), _lib.ctx()
    ds.set_targets(y)
    h = m._to_device(ds)
    try:
        ls = C.c_double()
        idx = None if rows is None else _lib.i64(rows)
        cnt = len(rows) if rows is not None else n
        _lib.check(lib.nimfm_ffm_loss_grad(ctx, h, ds.handle(), loss.kind, loss.threshold, row_begin, cnt,
                                           _lib.ptr(idx), cnt if mb is None else mb, 1, 0, C.byref(ls)))
        gP, gw, gb = np.zeros_like(m.P), np.zeros(ds.nFeatures), C.c_double()
        _lib.check(lib.nimfm_ffm_get_grads(ctx, h, _lib.ptr(gP), _lib.ptr(gw), C.byref(gb)))
    finally:
        lib.nimfm_ffm_free(ctx, h)
    return ls.value, gP, gw, gb.value


def check_loss_grad(got, ref):
    ls, gP, gw, gb = got
    assert abs(ls - ref["loss"]) <= DEC_TOL * max(1.0, abs(ref["loss"]))
    # rows of hundreds of nonzeros make gradient elements whose terms nearly cancel: those carry the rounding of the
    # RED arrival order, so P's gradient is held as the suite holds such sums (helpers.sums_agree)
    assert sums_agree(gP, ref["gP"])
    assert max_rel(gw, ref["gw"]) <= GRAD_TOL
    assert abs(gb - ref["gb"]) <= DEC_TOL * max(1.0, abs(ref["gb"]))


def check_fit(opt, m, ref):
    np.testing.assert_allclose([h[1] for h in opt.history], ref["loss"], rtol=FIT_TOL)
    np.testing.assert_allclose([h[0] for h in opt.history], ref["viol"], rtol=1e-8)
    # the bars of the suite's own AdaGrad / SGD tests: an element of g_sum whose terms nearly cancel carries the
    # rounding of their arrival order, so tiny elements are held to an absolute 1e-13
    np.testing.assert_allclose(m.P, ref["P"], rtol=FIT_TOL, atol=1e-13)
    np.testing.assert_allclose(m.w, ref["w"], rtol=FIT_TOL, atol=1e-13)
    assert abs(m.intercept - ref["intercept"]) <= FIT_TOL and opt.it == ref["it"]


def run_adagrad(oracle, csr, P, w, y, mb, max_iter=2):
    ref = oracle.ffm_adagrad_fit(csr, y, P, w, 0.05, "logistic", max_iter=max_iter, mini_batch_size=mb)
    m = make_ffm(P, w, 0.05, task=nf.classification)
    opt = nf.newAdaGrad(maxIter=max_iter, loss=nf.Logistic(), verbose=0, tol=0.0, shuffle=False, miniBatchSize=mb)
    opt.fit(field_ds(csr), y, m)
    check_fit(opt, m, ref)


def run_sgd_minibatch(oracle, csr, P, w, y, B, max_iter=2):
    kw = dict(eta0=0.03, alpha0=1e-3, alpha=2e-2, beta=3e-2)
    perms = np.array([np.random.default_rng(90 + e).permutation(csr.n) for e in range(max_iter)])
    ref = oracle.sgd_minibatch_fit(csr, y, P, w, 0.05, loss_kind="logistic", B=B, max_iter=max_iter, perms=perms,
                                   it=1, ffm=True, **kw)
    m = make_ffm(P, w, 0.05, task=nf.classification)
    opt = nf.newSGD(maxIter=max_iter, loss=nf.Logistic(), verbose=0, tol=0.0, **kw)
    opt.fit(field_ds(csr), y, m, maxThreads=B, perms=perms)
    check_fit(opt, m, ref)


# ------------------------------------------------------------------------------------------------ refused before
@gpu
@pytest.mark.parametrize("name", CASE_IDS)
def test_unit_kernel_shapes_match_oracle(oracle, sms, name):
    """every FFM entry point on a shape built for the unit kernel (in the modes the case table names; the others
    run on whichever kernel the planner picks and are held to the same bars)"""
    c = case_by_name(name)
    n = n_rows(sms)
    csr, P, w, y = case_data(c, n)
    assert n >= 3 * UNIT_BLOCKS_PER_SM * sms
    m = make_ffm(P, w, 0.05, task=nf.classification)
    got = m.decisionFunction(field_ds(csr))
    assert max_rel(got, oracle.ffm_decision_function(csr, P, w, 0.05)) <= DEC_TOL
    # a contiguous range that starts past row 0 and ends before n
    b0, cnt = 3, n - 10
    got = dev_loss_grad(m, field_ds(csr), y, nf.Logistic(), row_begin=b0, n=cnt, mb=cnt + 5)
    check_loss_grad(got, oracle.ffm_loss_grad(csr, y, P, w, 0.05, "logistic", row_begin=b0, row_end=b0 + cnt,
                                              mini_batch_size=cnt + 5))
    # a row list with repeats (the long rows included)
    rng = np.random.default_rng(7)
    rows = rng.integers(0, n, n // 2)
    rows[:6] = (0, 1, 2, 5, 5, n - 1)
    got = dev_loss_grad(m, field_ds(csr), y, nf.Logistic(), rows=rows)
    check_loss_grad(got, oracle.ffm_loss_grad(sub_rows(csr, rows), y[rows], P, w, 0.05, "logistic"))
    # minibatches of more than one wave (but fit_rows), the last one partial
    nf_ = c["fit_rows"] or n
    fit = sub_rows(csr, np.arange(nf_)) if nf_ < n else csr
    run_sgd_minibatch(oracle, fit, P, w, y[:nf_], B=nf_ // 3)
    # AdaGrad: miniBatchSize 1 on a prefix that holds every special row (and, for long_k8, two long ones); > 1 on all
    pre = sub_rows(csr, np.arange(48))
    run_adagrad(oracle, pre, P, np.zeros(csr.d), y[:48], mb=1)
    run_adagrad(oracle, fit, P, np.zeros(csr.d), y[:nf_], mb=nf_ // 2 + 1)


# ------------------------------------------------------------------------------------------------ forced
def forced_shapes():
    out = []
    for k in PAIR_KS:
        out.append((f"ragged_k{k}", k))
        out.append((f"one_per_field_k{k}", k))
    return out


@gpu
@pytest.mark.parametrize("shape,k", forced_shapes())
def test_forced_unit_kernel_matches_oracle_and_default(oracle, monkeypatch, shape, k):
    """NIMFM_FFM_KERNEL=units on shapes the pair / staged kernels serve: the oracle's bars, and the same sums as
    the default route"""
    if shape.startswith("ragged"):
        csr = ragged_field_csr(60, 120, 6, 100 + k, 64)
    else:
        csr = one_per_field_csr(200, 13, 20, 15 + k)
    rng = np.random.default_rng(k)
    P = rng.standard_normal((csr.n_fields, csr.d, k)) * 0.2
    w = rng.standard_normal(csr.d) * 0.1
    y = np.sign(rng.standard_normal(csr.n))
    m = make_ffm(P, w, 0.05, task=nf.classification)
    n = csr.n
    rows = np.random.default_rng(3).integers(0, n, 2 * n)
    dflt = (m.decisionFunction(field_ds(csr)), dev_loss_grad(m, field_ds(csr), y, nf.Logistic(), n=n),
            dev_loss_grad(m, field_ds(csr), y, nf.Logistic(), rows=rows))
    monkeypatch.setenv("NIMFM_FFM_KERNEL", "units")
    got = m.decisionFunction(field_ds(csr))
    assert max_rel(got, oracle.ffm_decision_function(csr, P, w, 0.05)) <= DEC_TOL
    assert sums_agree(got, dflt[0])
    for g, d_, ref in ((dev_loss_grad(m, field_ds(csr), y, nf.Logistic(), n=n), dflt[1],
                        oracle.ffm_loss_grad(csr, y, P, w, 0.05, "logistic")),
                       (dev_loss_grad(m, field_ds(csr), y, nf.Logistic(), rows=rows), dflt[2],
                        oracle.ffm_loss_grad(sub_rows(csr, rows), y[rows], P, w, 0.05, "logistic"))):
        check_loss_grad(g, ref)
        assert sums_agree(g[1], d_[1]) and sums_agree(g[2], d_[2])
        assert abs(g[0] - d_[0]) <= 1e-12 * max(1.0, abs(d_[0]))
    run_adagrad(oracle, csr, P, np.zeros(csr.d), y, mb=16)
    run_adagrad(oracle, sub_rows(csr, np.arange(30)), P, np.zeros(csr.d), y[:30], mb=1)
    run_sgd_minibatch(oracle, csr, P, w, y, B=7)


# ------------------------------------------------------------------------------------------------ windows
@gpu
def test_windowed_field_stream_at_rank_20(tmp_path):
    """decisionFunction over a windowed STREAMCSRFIELD file of the C5 row shape at k = 20 (the unit kernel, one
    fresh dataset per window) equals the resident result"""
    csr = one_per_field_csr(600, 39, 30, 41)
    y = np.sign(np.random.default_rng(1).standard_normal(csr.n))
    ds0 = field_ds(csr)
    txt, fx, fy = (str(tmp_path / f) for f in ("a.ffm", "a.bin", "a.lab"))
    nf.dumpFFMFile(txt, ds0, y)
    nf.convertFFMFile(txt, fx, fy)
    whole = nf.newStreamCSRFieldDataset(fx, resident=True)
    win = nf.newStreamCSRFieldDataset(fx, cacheSize=64 / 1024.0, resident=False)
    assert win.windowed and len(list(win.windows())) > 1
    rng = np.random.default_rng(2)
    P = rng.standard_normal((39, whole.nFeatures, 20)) * 0.05
    w = rng.standard_normal(whole.nFeatures) * 0.1
    got = make_ffm(P, w, 0.05).decisionFunction(win)
    res = make_ffm(P, w, 0.05).decisionFunction(whole)
    assert np.array_equal(got, res)
    ref = CSR(whole.data, whole.indices, whole.indptr, whole.nSamples, whole.nFeatures, fields=whole.fields,
              n_fields=39)
    from oracle import oracle as orc
    assert max_rel(got, orc.ffm_decision_function(ref, P, w, 0.05)) <= DEC_TOL
