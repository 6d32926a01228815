"""AdaGrad keeps g_sum / g_norm across warm-started fits of a field-aware FM, as it does for an FM (adagrad.nim:47-62:
init keeps the state when warmStart is set and the shapes match).

AdaGrad.fit reads the state back through nimfm_ffm_adagrad_get_state before the last finalize and hands it to the
next warm fit through nimfm_ffm_adagrad_set_state, g_sum.P / g_norm.P in ffm.P's layout [nFields, nFeatures, k].  So:
  - one fit of two epochs equals a fit of one epoch followed by a warm fit of one more on the same optimizer, on every
    FFM AdaGrad route (ffm_plan_mode, ffm.cu): the bulk-reduction pair kernel (k = 8, one nonzero per field), the pair
    kernel with NIMFM_FFM_BULK=0, the staged kernel (k = 10, or rows that repeat a field), the unit kernel
    (NIMFM_FFM_KERNEL=units) and, under NIMFM_DETERMINISTIC=1, the tuned and the generic column kernels.  Bit for bit
    where the route adds every element once or in a fixed order, at the suite's AdaGrad bar on the RED routes;
  - the warm fit matches the oracle started from the first fit's finalized parameters, `it` and state;
  - a warm fit over a windowed StreamCSRFieldDataset gives what the resident dataset gives;
  - a warm fit without a state, or with a state of another shape, is refused with the reference's messages, and the
    state calls refuse to run before nimfm_ffm_adagrad_init."""
import ctypes as C
import os

import numpy as np
import pytest

import nimfm_b200 as nf
from nimfm_b200 import _lib
from oracle.oracle import CSR

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

KW = dict(eta0=0.05, alpha0=1e-6, alpha=1e-3, beta=1e-3)
N_ROWS = 300
MB = 32                       # 9 full minibatches and a partial tenth
NIMFM_ERR_INVALID, NIMFM_ERR_STATE = -1, -5
ENV_VARS = ("NIMFM_DETERMINISTIC", "NIMFM_FFM_BULK", "NIMFM_FFM_KERNEL", "NIMFM_FFM_COLS")


# ------------------------------------------------------------------------------------------------ data
def one_per_field_rows(n, n_fields, per_field, seed):
    """every row holds each field once; field f owns the ids [f * per_field, (f + 1) * per_field)"""
    rng = np.random.default_rng(seed)
    idx = rng.integers(0, per_field, size=(n, n_fields)) + (np.arange(n_fields) * per_field)[None, :]
    data = np.where(rng.random((n, n_fields)) < 0.5, 1.0, rng.standard_normal((n, n_fields)))
    return CSR(data.ravel(), idx.ravel(), np.arange(n + 1) * n_fields, n, n_fields * per_field,
               fields=np.tile(np.arange(n_fields), n), n_fields=n_fields)


def repeated_field_rows(n, n_fields, d, seed, max_nnz=20):
    """rows of 0 .. max_nnz distinct ids whose fields are drawn with replacement, so most rows repeat a field"""
    rng = np.random.default_rng(seed)
    data, indices, fields, indptr = [], [], [], [0]
    for i in range(n):
        z = 0 if i % 11 == 0 else int(rng.integers(2, max_nnz + 1))
        indices.extend(np.sort(rng.choice(d, size=z, replace=False)).tolist())
        data.extend(rng.standard_normal(z).tolist())
        fields.extend(rng.integers(0, n_fields, z).tolist())
        indptr.append(len(indices))
    return CSR(np.array(data), np.array(indices, np.int64), np.array(indptr, np.int64), n, d,
               fields=np.array(fields, np.int64), n_fields=n_fields)


def field_ds(csr):
    return nf.newCSRFieldDataset(csr.data, csr.indices, csr.indptr, csr.fields, csr.n, csr.d, csr.n_fields)


def problem(csr, k, seed):
    rng = np.random.default_rng(seed)
    P = rng.standard_normal((csr.n_fields, csr.d, k)) * 0.1
    w = rng.standard_normal(csr.d) * 0.1
    y = np.sign(rng.standard_normal(csr.n))
    return P, w, y


def make_ffm(P, w, b):
    m = nf.newFieldAwareFactorizationMachine(nf.classification, nComponents=P.shape[2], warmStart=True)
    m.P, m.w, m.intercept, m.isInitialized = P.copy(), w.copy(), b, True
    return m


def make_opt(max_iter, mb):
    return nf.newAdaGrad(maxIter=max_iter, loss=nf.Logistic(), miniBatchSize=mb, verbose=0, tol=0.0, **KW)


def perms_for(n, seed, epochs=2):
    rng = np.random.default_rng(seed)
    return np.stack([rng.permutation(n) for _ in range(epochs)]).astype(np.int64)


# route -> (rows, k, environment); ffm_plan_mode picks the kernel from these (no route query crosses the ABI)
ROUTES = {
    "bulk": ("one_per_field", 8, {}),
    "pair": ("one_per_field", 8, {"NIMFM_FFM_BULK": "0"}),
    "staged_k10": ("one_per_field", 10, {}),
    "staged_dups": ("repeated_fields", 8, {}),
    "units": ("one_per_field", 8, {"NIMFM_FFM_KERNEL": "units"}),
    "det_tuned": ("one_per_field", 8, {"NIMFM_DETERMINISTIC": "1"}),
    "det_generic": ("one_per_field", 8, {"NIMFM_DETERMINISTIC": "1", "NIMFM_FFM_COLS": "generic"}),
}


def route_data(route):
    rows, k, _ = ROUTES[route]
    seed = 700 + list(ROUTES).index(route)
    csr = one_per_field_rows(N_ROWS, 13, 20, seed) if rows == "one_per_field" else \
        repeated_field_rows(N_ROWS, 6, 240, seed)
    return (csr,) + problem(csr, k, seed)


def bit_exact(route, mb):
    """Deterministic minibatches add in sample order; a one-row minibatch of a row with one nonzero per field adds
    every gradient element once.  Everything else adds with REDs in arrival order."""
    rows, _, env = ROUTES[route]
    return (mb > 1 and env.get("NIMFM_DETERMINISTIC") == "1") or (mb == 1 and rows == "one_per_field")


# ------------------------------------------------------------------------------------------------ comparison
def snapshot(opt, m):
    return dict(P=m.P.copy(), w=m.w.copy(), intercept=m.intercept, it=opt.it, hist=list(opt.history),
                gsP=opt.g_sum["P"].copy(), gnP=opt.g_norm["P"].copy(), gsw=opt.g_sum["w"].copy(),
                gnw=opt.g_norm["w"].copy(), gsb=opt.g_sum["intercept"], gnb=opt.g_norm["intercept"])


ARRAYS = ("P", "w", "gsP", "gnP", "gsw", "gnw")
SCALARS = ("intercept", "gsb", "gnb")


def assert_same(got, ref, exact):
    """exact: array_equal.  Otherwise the suite's AdaGrad bars: arrays at rtol 1e-8 / atol 1e-13 (an element whose
    terms nearly cancel carries the rounding of their arrival order), scalars at 1e-9 of max(1, |ref|)."""
    assert got["it"] == ref["it"]
    for key in ARRAYS:
        if exact:
            assert np.array_equal(got[key], ref[key]), (key, float(np.max(np.abs(got[key] - ref[key]))))
        else:
            np.testing.assert_allclose(got[key], ref[key], rtol=1e-8, atol=1e-13, err_msg=key)
    for key in SCALARS:
        if exact:
            assert got[key] == ref[key], key
        else:
            assert abs(got[key] - ref[key]) <= 1e-9 * max(1.0, abs(ref[key])), key


# ------------------------------------------------------------------------------------------------ CPU
def test_route_table():
    """the route datasets have the shapes their kernels need: one nonzero per field where the pair, unit and column
    kernels run, a repeated field in some row for the staged route, a partial last minibatch"""
    assert N_ROWS % MB > 0 and N_ROWS // MB >= 3
    for route, (rows, k, env) in ROUTES.items():
        csr = route_data(route)[0]
        dups = any(len(np.unique(f)) != len(f) for f in np.split(csr.fields, csr.indptr[1:-1]))
        assert dups == (rows == "repeated_fields"), route
        if k not in (4, 8, 16, 32):
            assert route.startswith("staged")
        for i in range(csr.n):
            ids = csr.indices[csr.indptr[i]:csr.indptr[i + 1]]
            assert len(np.unique(ids)) == len(ids)


def test_nim_layer_carries_the_ffm_state():
    """nim/fit_ffm.nim sets the state on a warm start and reads it back before the last finalize, like
    nim/fit_adagrad.nim does for an FM"""
    src = open(os.path.join(ROOT, "nim", "fit_ffm.nim")).read()
    body = src[src.index("proc runAdaGradFFM"):src.index("proc fit*[L](self: AdaGrad[L]")]
    init = body.index("nimfm_ffm_adagrad_init(")
    warm = body.index("if self.it != 1:")
    setter = body.index("nimfm_ffm_adagrad_set_state(")
    getter = body.index("nimfm_ffm_adagrad_get_state(")
    last_finalize = body.rindex("nimfm_ffm_adagrad_finalize(")
    assert init < warm < setter < body.index("for epoch in") < getter < last_finalize
    assert "newParams([ffm.P.shape[0], ffm.P.shape[1], ffm.P.shape[2]]" in body


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture
def route_env(monkeypatch, request):
    for v in ENV_VARS + ("NIMFM_ADAGRAD_SEQ", "NIMFM_ROW_KERNEL"):
        monkeypatch.delenv(v, raising=False)
    for v, val in ROUTES[request.param][2].items():
        monkeypatch.setenv(v, val)
    return request.param


@gpu
@pytest.mark.parametrize("mb", [1, MB])
@pytest.mark.parametrize("route_env", list(ROUTES), indirect=True)
def test_resume_equals_continue(route_env, mb):
    """A: fit(maxIter=2).  B: fit(maxIter=1), then a warm fit(maxIter=1) on the same optimizer.  Same orders; B's second
    fit must carry on from A's state: P, w, intercept, it, g_sum, g_norm and the last epoch's loss agree"""
    csr, P, w, y = route_data(route_env)
    perms = perms_for(csr.n, 11)
    ma, oa = make_ffm(P, w, 0.05), make_opt(2, mb)
    oa.fit(field_ds(csr), y, ma, perms=perms)
    mb_, ob = make_ffm(P, w, 0.05), make_opt(1, mb)
    ob.fit(field_ds(csr), y, mb_, perms=perms[:1])
    ob.fit(field_ds(csr), y, mb_, perms=perms[1:])
    a, b = snapshot(oa, ma), snapshot(ob, mb_)
    exact = bit_exact(route_env, mb)
    assert_same(b, a, exact)
    if exact:
        assert b["hist"][-1][1] == a["hist"][-1][1]
    else:
        np.testing.assert_allclose(b["hist"][-1][1], a["hist"][-1][1], rtol=1e-8)


@gpu
@pytest.mark.parametrize("mb", [1, MB])
@pytest.mark.parametrize("route_env", ["bulk", "staged_k10", "det_tuned"], indirect=True)
def test_warm_fit_matches_oracle(oracle, route_env, mb):
    """the first fit's state equals the oracle's; the warm fit equals oracle.ffm_adagrad_fit started from the first
    fit's finalized P, w, intercept, `it` and state: P, w, intercept, g_sum, g_norm and the (viol, loss) history"""
    csr, P, w, y = route_data(route_env)
    perms = perms_for(csr.n, 12)
    m, opt = make_ffm(P, w, 0.05), make_opt(1, mb)
    opt.fit(field_ds(csr), y, m, perms=perms[:1])
    first = snapshot(opt, m)
    r1 = oracle.ffm_adagrad_fit(csr, y, P, w, 0.05, "logistic", max_iter=1, mini_batch_size=mb, perms=perms[:1], **KW)
    ref1 = dict(r1, **{k_: r1["state"][k_] for k_ in r1["state"]})
    assert_same(first, ref1, exact=False)
    st1 = dict(gsP=first["gsP"], gnP=first["gnP"], gsw=first["gsw"], gnw=first["gnw"], gsb=first["gsb"],
               gnb=first["gnb"])
    opt.fit(field_ds(csr), y, m, perms=perms[1:])
    got = snapshot(opt, m)
    r2 = oracle.ffm_adagrad_fit(csr, y, first["P"], first["w"], first["intercept"], "logistic", max_iter=1,
                                mini_batch_size=mb, perms=perms[1:], it=first["it"], state=st1, **KW)
    ref2 = dict(r2, **{k_: r2["state"][k_] for k_ in r2["state"]})
    assert_same(got, ref2, exact=False)
    np.testing.assert_allclose([h[0] for h in got["hist"]], r2["viol"], rtol=1e-8, atol=1e-13)
    np.testing.assert_allclose([h[1] for h in got["hist"]], r2["loss"], rtol=1e-8, atol=1e-13)
    # a restart from g_sum = 0 would land far from the warm reference
    cold = oracle.ffm_adagrad_fit(csr, y, first["P"], first["w"], first["intercept"], "logistic", max_iter=1,
                                  mini_batch_size=mb, perms=perms[1:], it=first["it"], **KW)
    assert not np.allclose(cold["P"], r2["P"], rtol=1e-6, atol=1e-10)


@gpu
@pytest.mark.parametrize("mb", [1, 16])
def test_windowed_warm_fit_equals_resident(tmp_path, monkeypatch, mb):
    """a fit and a warm fit over a StreamCSRFieldDataset walked in windows equal the same two fits over the resident
    dataset (windows hold whole minibatches; neither dataset is shuffled)"""
    for v in ENV_VARS:
        monkeypatch.delenv(v, raising=False)
    csr = one_per_field_rows(N_ROWS, 13, 20, 41)
    y = np.sign(np.random.default_rng(1).standard_normal(csr.n))
    txt, fx, fy = (str(tmp_path / f) for f in ("a.ffm", "a.bin", "a.lab"))
    nf.dumpFFMFile(txt, field_ds(csr), y)
    nf.convertFFMFile(txt, fx, fy)
    whole = nf.newStreamCSRFieldDataset(fx, resident=True)
    win = nf.newStreamCSRFieldDataset(fx, cacheSize=16 / 1024.0, resident=False)
    try:
        assert win.windowed and len(list(win.windows(multiple=mb))) > 2
        P, w, _ = problem(CSR(whole.data, whole.indices, whole.indptr, whole.nSamples, whole.nFeatures,
                              fields=whole.fields, n_fields=whole.nFields), 8, 42)
        out = []
        for ds in (win, whole):
            m = make_ffm(P, w, 0.05)
            opt = nf.newAdaGrad(maxIter=1, loss=nf.Logistic(), miniBatchSize=mb, verbose=0, tol=0.0, shuffle=False,
                                **KW)
            opt.fit(ds, y, m)
            opt.fit(ds, y, m)
            out.append(snapshot(opt, m))
        assert_same(out[0], out[1], exact=False)
        np.testing.assert_allclose(out[0]["hist"], out[1]["hist"], rtol=1e-10, atol=0)
    finally:
        win.close()


@gpu
def test_warm_start_without_a_state_is_refused(monkeypatch):
    for v in ENV_VARS:
        monkeypatch.delenv(v, raising=False)
    csr = one_per_field_rows(40, 5, 4, 3)
    P, w, y = problem(csr, 4, 3)
    opt = make_opt(1, 8)
    opt.it = 41
    with pytest.raises(ValueError, match=r"^warmStart=true but the optimizer has no g_sum / g_norm state\.$"):
        opt.fit(field_ds(csr), y, make_ffm(P, w, 0.0))
    # a model without warmStart starts over and needs no state
    m = make_ffm(P, w, 0.0)
    m.warmStart = False
    opt.fit(field_ds(csr), y, m)
    assert opt.it == 1 + csr.n and opt.g_sum["P"].shape == P.shape


@gpu
def test_state_of_another_shape_is_refused(monkeypatch):
    """an FM optimizer's state handed to an FFM fit, and an FFM state of another nFields"""
    for v in ENV_VARS:
        monkeypatch.delenv(v, raising=False)
    shape_msg = r"^warmStart=true but P\.shape != g_sum\.P\.shape\.$"
    csr = one_per_field_rows(40, 5, 4, 5)
    P, w, y = problem(csr, 4, 5)
    # FM state: [nOrders, d, k] = [1, 20, 4] against the FFM's [5, 20, 4]
    opt = make_opt(1, 8)
    fm = nf.newFactorizationMachine(nf.classification, degree=2, nComponents=4, warmStart=True)
    fm.P, fm.w, fm.intercept, fm.isInitialized = P[:1].transpose(0, 2, 1).copy(), w.copy(), 0.0, True
    opt.fit(nf.newCSRDataset(csr.data, csr.indices, csr.indptr, csr.n, csr.d), y, fm)
    assert opt.it != 1 and opt.g_sum["P"].shape == (1, csr.d, 4)
    with pytest.raises(ValueError, match=shape_msg):
        opt.fit(field_ds(csr), y, make_ffm(P, w, 0.0))
    # FFM state of 5 fields against a model and dataset of 4
    opt = make_opt(1, 8)
    opt.fit(field_ds(csr), y, make_ffm(P, w, 0.0))
    assert opt.g_sum["P"].shape == (5, csr.d, 4)
    csr4 = one_per_field_rows(40, 4, 5, 6)
    P4, w4, y4 = problem(csr4, 4, 6)
    with pytest.raises(ValueError, match=shape_msg):
        opt.fit(field_ds(csr4), y4, make_ffm(P4, w4, 0.0))


@gpu
def test_state_calls_need_init():
    """get_state / set_state before nimfm_ffm_adagrad_init return NIMFM_ERR_STATE; set_state refuses NULL arrays;
    after init, set_state then get_state round-trips the reference layout bit for bit"""
    lib, ctx = _lib.load(), _lib.ctx()
    csr = one_per_field_rows(20, 3, 5, 7)
    P, w, _ = problem(csr, 4, 7)
    ds = field_ds(csr)
    h = make_ffm(P, w, 0.0)._to_device(ds)
    try:
        rng = np.random.default_rng(8)
        gsP, gsw = rng.standard_normal(P.shape), rng.standard_normal(csr.d)
        gnP, gnw = rng.random(P.shape) + 1e-3, rng.random(csr.d) + 1e-3
        ptrs = [_lib.ptr(a) for a in (gsP, gnP, gsw, gnw)]
        gsb, gnb = C.c_double(), C.c_double()
        assert lib.nimfm_ffm_adagrad_set_state(ctx, h, *ptrs, 0.25, 0.5) == NIMFM_ERR_STATE
        assert lib.nimfm_ffm_adagrad_get_state(ctx, h, *ptrs, C.byref(gsb), C.byref(gnb)) == NIMFM_ERR_STATE
        assert "nimfm_ffm_adagrad_init" in lib.nimfm_last_error(ctx).decode()
        _lib.check(lib.nimfm_ffm_adagrad_init(ctx, h, 1e-10, 1))
        assert lib.nimfm_ffm_adagrad_set_state(ctx, h, ptrs[0], None, ptrs[2], ptrs[3], 0.25, 0.5) == NIMFM_ERR_INVALID
        _lib.check(lib.nimfm_ffm_adagrad_set_state(ctx, h, *ptrs, 0.25, 0.5))
        back = [np.zeros(P.shape), np.zeros(P.shape), np.zeros(csr.d), np.zeros(csr.d)]
        _lib.check(lib.nimfm_ffm_adagrad_get_state(ctx, h, *[_lib.ptr(a) for a in back], C.byref(gsb), C.byref(gnb)))
        for a, b in zip(back, (gsP, gnP, gsw, gnw)):
            assert np.array_equal(a, b)
        assert (gsb.value, gnb.value) == (0.25, 0.5)
    finally:
        lib.nimfm_ffm_free(ctx, h)
        ds.free()
