"""Deterministic synchronous-minibatch AdaGrad (NIMFM_DETERMINISTIC=1, miniBatchSize > 1) for FM and FFM.

Under the switch every minibatch builds its own column index on the device (nimfm_mb_index_build, dataset_ops.cu):
the minibatch's rows gathered into a CSR view, its stable column-major twin (entries of a column in sample order, a
row listed twice giving two positions) and the 512-entry segment table.  The stash forward (FM) or the FFM forward
runs over the view, and the AdaGrad forms of the column kernels add every gradient element and its square in sample
order, long columns by segments added in segment order.  So:
  - FM at the tuned and the generic column kernels, with dummy columns, a row past 512 nonzeros, without the linear
    term and without the intercept, and FFM at the tuned kernel, the generic one, component chunks and 80 fields, are
    held to the oracle's AdaGrad with shuffled and identity sample orders, and repeat themselves bit for bit;
  - the generic kernels forced give the tuned kernels' bits, and an identity order gives the bits of no order;
  - an FFM dataset that repeats a field in a row stays an error;
  - miniBatchSize = 1 keeps its per-sample route under the switch (a one-row minibatch adds each element once)."""
import ctypes as C

import numpy as np
import pytest

import nimfm_b200 as nf
from nimfm_b200 import _lib
from oracle.oracle import CSR
from test_gpu_routes import LOSSES, case_data, csr_ds, n_rows
from test_gpu_ffm_deterministic_shapes import det_rows
from test_gpu_ffm_sgd import field_ds, make_ffm

gpu = pytest.mark.gpu
SEG = 512                     # entries per column segment (fm_cols.cu, dataset_ops.cu)
B200_SMS = 148
KW = dict(eta0=0.05, alpha0=1e-6, alpha=1e-3, beta=1e-3)
EPOCHS = 2


# ------------------------------------------------------------------------------------------------ the case tables
def _fm(name, degree, fit_lower, k, n_dense=20, max_extra=12, d=400, long_row=0, fit_linear=True, fit_intercept=True,
        tuned=False):
    # the keys test_gpu_routes.case_data reads, and whether the tuned column kernel runs
    return dict(name=name, degree=degree, fit_lower=fit_lower, k=k, n_dense=n_dense, max_extra=max_extra, d=d,
                long_row=long_row, spread=False, fit_linear=fit_linear, fit_intercept=fit_intercept, tuned=tuned)


FM_CASES = [
    _fm("d3_explicit_k32", 3, "explicit", 32, tuned=True),                 # C4's shape: the tuned pair
    _fm("d2_k8_nolinear", 2, "explicit", 8, fit_linear=False, tuned=True),
    _fm("d3_none_k16", 3, "none", 16, tuned=True),
    _fm("d2_k30_default", 2, "explicit", 30),                             # the default model: the generic pair
    _fm("d4_augment_k12_nointercept", 4, "augment", 12, d=120, max_extra=8, fit_intercept=False),
    _fm("longrow_d2_k8", 2, "explicit", 8, d=1200, long_row=700),          # a row past 512: the generic pair
]
FM_IDS = [c["name"] for c in FM_CASES]
FM_BY_NAME = {c["name"]: c for c in FM_CASES}


def fm_batch(n):
    """three full minibatches and a partial fourth"""
    return n // 3 - 1001


def _ffm(name, k, n_fields, d, z_range, n=3000):
    return dict(name=name, k=k, n_fields=n_fields, d=d, z_range=z_range, n=n)


C5 = (35, 39)
FFM_CASES = [
    _ffm("c5_k4_tuned", 4, 39, 3000, C5),
    _ffm("c5_k8_tuned", 8, 39, 3000, C5),
    _ffm("c5_k16_tuned", 16, 39, 3000, C5),                 # the tuned AdaGrad kernel's two-entry form
    _ffm("c5_k10_generic", 10, 39, 3000, C5),
    _ffm("c5_k64_chunks", 64, 39, 1500, C5, n=2400),
    _ffm("fields80_k8", 8, 80, 3000, (80, 80), n=2400),
]
FFM_IDS = [c["name"] for c in FFM_CASES]
FFM_BY_NAME = {c["name"]: c for c in FFM_CASES}
FFM_BATCH = 700


def fm_data(c, sms):
    return case_data(c, sms, 9100 + FM_IDS.index(c["name"]))


def ffm_data(c):
    seed = 9300 + FFM_IDS.index(c["name"])
    csr = det_rows(c["n"], c["d"], c["n_fields"], c["z_range"], seed, hot=0.85)
    rng = np.random.default_rng(seed)
    P = rng.standard_normal((c["n_fields"], c["d"], c["k"])) * (c["z_range"][1] * np.sqrt(c["k"])) ** -0.5
    w = rng.standard_normal(c["d"]) * 0.1
    y = np.sign(rng.standard_normal(c["n"]))
    return csr, P, w, y


def perms_for(n, seed, shuffled):
    rng = np.random.default_rng(seed)
    return np.stack([rng.permutation(n) if shuffled else np.arange(n) for _ in range(EPOCHS)]).astype(np.int64)


def max_column_in_a_batch(csr, perm, B):
    """the longest column inside one minibatch of the order perm"""
    best = 0
    for s in range(0, csr.n, B):
        rows = perm[s:s + B]
        idx = np.concatenate([csr.indices[csr.indptr[r]:csr.indptr[r + 1]] for r in rows])
        best = max(best, int(np.bincount(idx, minlength=csr.d).max()))
    return best


# ------------------------------------------------------------------------------------------------ CPU guard
def test_case_tables():
    """without a GPU: every FM case runs past three persistent waves at the B200's SM count in three full minibatches
    and a partial one, with a column longer than one segment inside a minibatch of a shuffled order; the cases cover
    the tuned and the generic kernels, dummy columns, a row past 512, no linear term and no intercept.  Every FFM case
    has one nonzero per field, a column longer than one segment in a minibatch and a partial last minibatch."""
    n = n_rows(B200_SMS)
    B = fm_batch(n)
    assert n > 3 * B and n % B > 0 and n // B == 3
    assert {c["tuned"] for c in FM_CASES} == {True, False}
    assert any(c["fit_lower"] == "augment" for c in FM_CASES) and any(c["long_row"] > SEG for c in FM_CASES)
    assert any(not c["fit_linear"] for c in FM_CASES) and any(not c["fit_intercept"] for c in FM_CASES)
    assert nf.newFactorizationMachine(nf.regression).nComponents == 30
    c = FM_CASES[0]
    g = fm_data(c, B200_SMS)
    assert max_column_in_a_batch(g["csr"], perms_for(n, 1, True)[0], B) > SEG
    for c in FFM_CASES:
        csr, _, _, _ = ffm_data(c)
        assert c["n"] % FFM_BATCH > 0 and c["n"] // FFM_BATCH >= 3
        for i in range(csr.n):
            f = csr.fields[csr.indptr[i]:csr.indptr[i + 1]]
            assert len(np.unique(f)) == len(f)
        assert max_column_in_a_batch(csr, perms_for(csr.n, 2, True)[0], FFM_BATCH) > SEG, c["name"]
    assert {c["k"] for c in FFM_CASES} >= {8, 10, 64} and max(c["n_fields"] for c in FFM_CASES) > 64


# ------------------------------------------------------------------------------------------------ GPU helpers
@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture
def deterministic(monkeypatch):
    for v in ("NIMFM_ROW_KERNEL", "NIMFM_FFM_COLS", "NIMFM_ADAGRAD_SEQ"):
        monkeypatch.delenv(v, raising=False)
    monkeypatch.setenv("NIMFM_DETERMINISTIC", "1")


def make_fm(c, g):
    task = nf.regression if g["loss"] in ("squared", "huber") else nf.classification
    fm = nf.newFactorizationMachine(task, degree=c["degree"], nComponents=c["k"], fitLower=c["fit_lower"],
                                    fitLinear=c["fit_linear"], fitIntercept=c["fit_intercept"], warmStart=True)
    fm.P, fm.w, fm.isInitialized = g["P"].copy(), g["w"].copy(), True
    fm.intercept = g["b"] if c["fit_intercept"] else 0.0
    return fm


def fm_fit(c, g, B, perms):
    """EPOCHS AdaGrad epochs through the ABI, as AdaGrad.fit runs them; perms None passes no sample order.  Returns
    P, w, intercept, the (viol, loss) history, it and the four g_sum / g_norm arrays."""
    lib, ctx = _lib.load(), _lib.ctx()
    fm = make_fm(c, g)
    ds = csr_ds(g["csr"])
    n = g["csr"].n
    loss = LOSSES[g["loss"]]()
    fm.init(ds)
    ds.set_targets(fm.checkTarget(g["y"]))
    h = fm._to_device(ds.nFeatures)
    try:
        cfg = _lib.AdagradCfg(loss.kind, loss.threshold, KW["eta0"], KW["alpha0"], KW["alpha"], KW["beta"], 1e-10, B)
        _lib.check(lib.nimfm_fm_adagrad_init(ctx, h, 1e-10, 1))
        it, hist = C.c_int64(1), []
        for ep in range(EPOCHS):
            order = None if perms is None else _lib.i64(perms[ep])
            viol, ls = C.c_double(), C.c_double()
            _lib.check(lib.nimfm_fm_adagrad_epoch(ctx, h, ds.handle(), C.byref(cfg), C.byref(it),
                                                  None if order is None else _lib.ptr(order), n, C.byref(viol),
                                                  C.byref(ls)))
            hist.append((viol.value, ls.value / n))
        dd = g["csr"].d + g["n_aug"]
        nO = g["P"].shape[0]
        st = [np.zeros((nO, dd, c["k"])), np.zeros((nO, dd, c["k"])), np.zeros(g["csr"].d), np.zeros(g["csr"].d)]
        gsb, gnb = C.c_double(), C.c_double()
        _lib.check(lib.nimfm_fm_adagrad_get_state(ctx, h, *[_lib.ptr(a) for a in st], C.byref(gsb), C.byref(gnb)))
        _lib.check(lib.nimfm_fm_adagrad_finalize(ctx, h, C.byref(cfg), it.value))
        fm._from_device(h)
    finally:
        lib.nimfm_fm_free(ctx, h)
        ds.free()
    return dict(P=fm.P.copy(), w=fm.w.copy(), intercept=fm.intercept, hist=hist, it=it.value, state=st,
                gsb=gsb.value, gnb=gnb.value)


def same_fit(a, b):
    return (np.array_equal(a["P"], b["P"]) and np.array_equal(a["w"], b["w"]) and a["intercept"] == b["intercept"]
            and a["hist"] == b["hist"] and a.get("it") == b.get("it")
            and all(np.array_equal(x, y) for x, y in zip(a.get("state", []), b.get("state", [])))
            and a.get("gsb") == b.get("gsb") and a.get("gnb") == b.get("gnb"))


def check_fit(got, ref, fit_intercept=True, state=True):
    """the suite's AdaGrad bars: P, w and the g_sum / g_norm state at rtol 1e-8 / atol 1e-13"""
    np.testing.assert_allclose([h[1] for h in got["hist"]], ref["loss"], rtol=1e-8)
    np.testing.assert_allclose([h[0] for h in got["hist"]], ref["viol"], rtol=1e-8, atol=1e-13)
    np.testing.assert_allclose(got["P"], ref["P"], rtol=1e-8, atol=1e-13)
    np.testing.assert_allclose(got["w"], ref["w"], rtol=1e-8, atol=1e-13)
    assert abs(got["intercept"] - ref["intercept"]) <= 1e-9 * max(1.0, abs(ref["intercept"]))
    if not fit_intercept:
        assert got["intercept"] == 0.0
    assert got["it"] == ref["it"]
    if state:
        st = ref["state"]
        for a, key in zip(got["state"], ("gsP", "gnP", "gsw", "gnw")):
            np.testing.assert_allclose(a, st[key], rtol=1e-8, atol=1e-13, err_msg=key)


# ------------------------------------------------------------------------------------------------ FM
@gpu
@pytest.mark.parametrize("shuffled", [True, False], ids=["shuffled", "identity"])
@pytest.mark.parametrize("name", FM_IDS)
def test_fm_adagrad_matches_oracle_and_repeats(oracle, deterministic, sms, name, shuffled):
    """two epochs of four minibatches (the last partial) against the oracle given the same orders, then the same fit
    again: array_equal P, w, intercept, history and g_sum / g_norm"""
    c = FM_BY_NAME[name]
    g = fm_data(c, sms)
    csr = g["csr"]
    B = fm_batch(csr.n)
    perms = perms_for(csr.n, FM_IDS.index(name), shuffled)
    got = fm_fit(c, g, B, perms)
    ref = oracle.adagrad_fit(csr, g["y"], g["P"], g["w"], g["b"] if c["fit_intercept"] else 0.0, c["degree"],
                             g["loss"], c["fit_linear"], c["fit_intercept"], max_iter=EPOCHS, mini_batch_size=B,
                             perms=perms, **KW)
    check_fit(got, ref, c["fit_intercept"])
    if not c["fit_linear"]:
        assert not np.any(got["w"]) and not np.any(got["state"][2])
    assert same_fit(got, fm_fit(c, g, B, perms))


@gpu
@pytest.mark.parametrize("name", [c["name"] for c in FM_CASES if c["tuned"]])
def test_fm_generic_forms_give_the_tuned_bits(monkeypatch, deterministic, sms, name):
    """NIMFM_ROW_KERNEL=generic (the generic stash forward and the generic AdaGrad column kernel) gives the bits of the
    tuned pair"""
    c = FM_BY_NAME[name]
    g = fm_data(c, sms)
    B = fm_batch(g["csr"].n)
    perms = perms_for(g["csr"].n, 77, True)
    tuned = fm_fit(c, g, B, perms)
    monkeypatch.setenv("NIMFM_ROW_KERNEL", "generic")
    generic = fm_fit(c, g, B, perms)
    assert same_fit(tuned, generic), float(np.max(np.abs(tuned["P"] - generic["P"])))


@gpu
@pytest.mark.parametrize("name", ["d3_explicit_k32", "d2_k30_default"])
def test_fm_identity_order_is_no_order(deterministic, sms, name):
    """perm = arange(n) and perm = NULL both run through the minibatch index: the same bits"""
    c = FM_BY_NAME[name]
    g = fm_data(c, sms)
    B = fm_batch(g["csr"].n)
    assert same_fit(fm_fit(c, g, B, perms_for(g["csr"].n, 0, False)), fm_fit(c, g, B, None))


# ------------------------------------------------------------------------------------------------ FFM
def ffm_fit(c, data, perms, B=FFM_BATCH):
    csr, P, w, y = data
    m = make_ffm(P, w, 0.05, task=nf.classification)
    opt = nf.newAdaGrad(maxIter=EPOCHS, loss=nf.Logistic(), miniBatchSize=B, verbose=0, tol=0.0, **KW)
    opt.fit(field_ds(csr), y, m, perms=perms)
    return dict(P=m.P.copy(), w=m.w.copy(), intercept=m.intercept, hist=list(opt.history), it=opt.it)


@gpu
@pytest.mark.parametrize("name", FFM_IDS)
def test_ffm_adagrad_matches_oracle_and_repeats(oracle, deterministic, name):
    """a shuffled two-epoch fit against the oracle, then bit for bit on a repeat"""
    c = FFM_BY_NAME[name]
    data = ffm_data(c)
    csr, P, w, y = data
    perms = perms_for(csr.n, 40 + FFM_IDS.index(name), True)
    got = ffm_fit(c, data, perms)
    ref = oracle.ffm_adagrad_fit(csr, y, P, w, 0.05, "logistic", max_iter=EPOCHS, mini_batch_size=FFM_BATCH,
                                 perms=perms, **KW)
    check_fit(got, ref, state=False)
    assert same_fit(got, ffm_fit(c, data, perms))


@gpu
@pytest.mark.parametrize("name", ["c5_k4_tuned", "c5_k8_tuned", "c5_k16_tuned"])
def test_ffm_generic_gives_the_tuned_bits(monkeypatch, deterministic, name):
    """at every tuned rank NIMFM_FFM_COLS=generic gives the tuned column kernel's bits"""
    c = FFM_BY_NAME[name]
    data = ffm_data(c)
    perms = perms_for(data[0].n, 5, True)
    tuned = ffm_fit(c, data, perms)
    monkeypatch.setenv("NIMFM_FFM_COLS", "generic")
    assert same_fit(tuned, ffm_fit(c, data, perms))


@gpu
def test_single_row_minibatches_keep_their_route(oracle, deterministic):
    """miniBatchSize = 1 under the switch keeps the per-sample routes (a one-row minibatch adds each element once):
    an FFM dataset that repeats a field in a row still fits, and matches the oracle"""
    c = FFM_BY_NAME["c5_k10_generic"]
    csr, P, w, y = ffm_data(c)
    n = 300
    keep = csr.indptr[n]
    dup = CSR(csr.data[:keep], csr.indices[:keep], csr.indptr[:n + 1], n, csr.d, fields=csr.fields[:keep].copy(),
              n_fields=csr.n_fields)
    a = dup.indptr[5]
    dup.fields[a + 1] = dup.fields[a]                              # row 5 holds two nonzeros of one field
    perms = perms_for(n, 3, True)
    got = ffm_fit(c, (dup, P, w, y[:n]), perms, B=1)
    ref = oracle.ffm_adagrad_fit(dup, y[:n], P, w, 0.05, "logistic", max_iter=EPOCHS, mini_batch_size=1, perms=perms,
                                 **KW)
    check_fit(got, ref, state=False)


@gpu
def test_ffm_repeated_field_is_refused(deterministic):
    c = FFM_BY_NAME["c5_k10_generic"]
    csr, P, w, y = ffm_data(c)
    dup = CSR(csr.data, csr.indices, csr.indptr, csr.n, csr.d, fields=csr.fields.copy(), n_fields=csr.n_fields)
    a = dup.indptr[5]
    dup.fields[a + 1] = dup.fields[a]                              # row 5 holds two nonzeros of one field
    with pytest.raises(Exception, match="one nonzero per field"):
        ffm_fit(c, (dup, P, w, y), perms_for(csr.n, 0, True))
