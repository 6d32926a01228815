"""Deterministic MBPSGD and synchronous-minibatch SGD (NIMFM_DETERMINISTIC=1) for FM and FFM, with their default
sample orders: shuffled minibatches and cursors that wrap past the last row.

A minibatch that is a contiguous row range inside the dataset keeps the dataset's column twin.  A row list (a shuffled
order) or a cursor that wraps gets its own column index (nimfm_mb_index_build, dataset_ops.cu): the rows gathered into
a view, in sample order, a row that occurs twice giving two positions.  The stash forward (FM) or the FFM forward and
the column kernels run over that view.  So:
  - FM MBPSGD through newMBPSGD(shuffle=True), at the tuned pair, the default model (the generic pair) and degree 4
    augment, with identity and L1, is held to the oracle given the host's permutations, and repeats bit for bit;
  - FM MBPSGD with shuffle=False and a wrapping cursor, miniBatchSize > n included, likewise;
  - the generic forms forced give the tuned pair's bits over the index;
  - FM and FFM minibatch SGD (fit(..., maxThreads)) are held to oracle.sgd_minibatch_fit and repeat; the FM lazy form
    steps aside under the switch, so the default and NIMFM_SGD_MB_LAZY=0 give the same bits;
  - an FFM dataset that repeats a field in a row stays an error."""
import numpy as np
import pytest

import nimfm_b200 as nf
from oracle.oracle import CSR
from helpers import make_fm_params, max_rel
from test_gpu_deterministic import long_column_csr
from test_gpu_ffm_deterministic_shapes import det_rows
from test_gpu_ffm_sgd import field_ds, make_ffm
from test_gpu_fm import csr_ds, make_fm

gpu = pytest.mark.gpu
SEG = 512                                   # entries per column segment (fm_cols.cu, dataset_ops.cu)
N, D, Z = 2000, 5000, 8                     # FM rows: column 0 in every row, 7 more at random
MBPSGD_KW = dict(eta0=0.3, alpha0=1e-3, alpha=5e-2, beta=8e-2)
SGD_KW = dict(eta0=0.03, alpha0=1e-3, alpha=2e-2, beta=3e-2)
EPOCHS = 3

# (name, degree, fitLower, k): the tuned pair, the default model (the generic pair), degree 4 with dummy features
SHAPES = [("d3_explicit_k32", 3, "explicit", 32), ("d2_explicit_k30", 2, "explicit", 30), ("d4_augment_k8", 4, "augment", 8)]
SHAPE = {s[0]: s for s in SHAPES}
REGS = {"identity": 0.0, "l1": 1e-3}        # gamma: L1 at gamma = 0 is the identity (as test_gpu_fm.make_reg)
WRAP_MB = 600                               # unshuffled: 2000 % 600 > 0, so the cursor wraps in the last minibatch
OVER_N, OVER_MB = 300, 700                  # miniBatchSize > n: every row occurs two or three times in a minibatch
SGD_B = 700
LAZY_B = 512                                # d3 k32: 512 x 8 touched features <= 2 d, so the lazy form is the default
FFM_N, FFM_D, FFM_FIELDS, FFM_B = 3000, 3000, 39, 700


def default_mb(n, d, nnz):
    """MBPSGD's default miniBatchSize (minibatch_psgd.nim:157-165, MBPSGD.resolve_sizes)"""
    return max((d * n) // nnz, 1)


def fm_rows(n=N, seed=7):
    csr = long_column_csr(n, D, seed, Z)
    y = np.sign(np.random.default_rng(seed + 1).standard_normal(n))
    return csr, y


def host_perms(fm, n, count=12):
    """the permutations the host mirror draws: the initial shuffle, then one per wrap (MBPSGD.fit)"""
    rng = np.random.default_rng(fm.randomState)
    idx, perms = np.arange(n), []
    for _ in range(count):
        rng.shuffle(idx)
        perms.append(idx.copy())
    return np.array(perms)


def longest_batch_column(csr, order, B):
    """the longest column inside one minibatch of B consecutive positions of order (wrapping)"""
    best = 0
    for s in range(0, len(order), B):
        rows = order[np.arange(s, s + B) % len(order)]
        idx = np.concatenate([csr.indices[csr.indptr[r]:csr.indptr[r + 1]] for r in rows])
        best = max(best, int(np.bincount(idx, minlength=csr.d).max()))
    return best


# ------------------------------------------------------------------------------------------------ CPU guard
def test_case_tables():
    """without a GPU: the default minibatch does not divide n (the sample list wraps and reshuffles inside an epoch)
    and holds a column longer than one segment; the unshuffled cursor wraps; one case has miniBatchSize > n; the
    lazy-form shape meets the lazy rule of nimfm_fm_sgd_mb_lazy_epoch; every FFM row holds one nonzero per field"""
    csr, _ = fm_rows()
    mb = default_mb(N, D, len(csr.data))
    assert N % mb > 0 and mb > SEG and -(-N // mb) * mb > N
    assert longest_batch_column(csr, np.arange(N), mb) > SEG
    assert N % WRAP_MB > 0 and OVER_MB > OVER_N
    assert LAZY_B * Z <= 2 * D and N // LAZY_B >= 2 and longest_batch_column(csr, np.arange(N), SGD_B) > SEG
    default_model = nf.newFactorizationMachine(nf.regression)
    assert default_model.nComponents == 30 and default_model.degree == 2
    f = det_rows(300, FFM_D, FFM_FIELDS, (35, 39), 1, hot=0.85)
    for i in range(f.n):
        fl = f.fields[f.indptr[i]:f.indptr[i + 1]]
        assert len(np.unique(fl)) == len(fl)


# ------------------------------------------------------------------------------------------------ GPU helpers
@pytest.fixture
def deterministic(monkeypatch):
    for v in ("NIMFM_ROW_KERNEL", "NIMFM_FFM_COLS", "NIMFM_MBPSGD_LAZY", "NIMFM_SGD_MB_LAZY"):
        monkeypatch.delenv(v, raising=False)
    monkeypatch.setenv("NIMFM_DETERMINISTIC", "1")


def fm_params(shape, seed):
    _, degree, fit_lower, k = shape
    P, w, _ = make_fm_params(D, degree, k, fit_lower, True, seed=seed, scale=0.1)
    return P, w


def same_fit(a, b):
    return (np.array_equal(a["P"], b["P"]) and np.array_equal(a["w"], b["w"]) and a["intercept"] == b["intercept"]
            and a["hist"] == b["hist"] and a["it"] == b["it"])


def mbpsgd_fit(shape, csr, y, P, w, reg, shuffle, mb=-1):
    _, degree, fit_lower, k = shape
    fm = make_fm(degree, k, fit_lower, True, True, P, w, 0.1, task=nf.classification)
    opt = nf.newMBPSGD(maxIter=EPOCHS, loss=nf.Logistic(), reg=nf.newL1(), gamma=REGS[reg], miniBatchSize=mb,
                       verbose=0, tol=0.0, shuffle=shuffle, **MBPSGD_KW)
    opt.fit(csr_ds(csr), y, fm)
    return dict(P=fm.P.copy(), w=fm.w.copy(), intercept=fm.intercept, hist=list(opt.history), it=opt.it, fm=fm)


def check_mbpsgd(got, ref):
    np.testing.assert_allclose(got["hist"], ref["epoch_loss"], rtol=1e-8)
    assert max_rel(got["P"], ref["P"]) <= 1e-8 and max_rel(got["w"], ref["w"]) <= 1e-8
    assert abs(got["intercept"] - ref["intercept"]) <= 1e-8 * max(abs(ref["intercept"]), 1e-3)
    assert got["it"] == ref["it"]


# ------------------------------------------------------------------------------------------------ FM MBPSGD
@gpu
@pytest.mark.parametrize("reg", list(REGS))
@pytest.mark.parametrize("name", list(SHAPE))
def test_mbpsgd_shuffled_matches_oracle_and_repeats(oracle, deterministic, name, reg):
    """newMBPSGD(shuffle=True) with the default minibatch (625 rows over 2 000: the sample list wraps and reshuffles
    inside every epoch; column 0 holds 625 entries of a minibatch) against the oracle given the host's
    permutations, then the same fit again: array_equal P, w, intercept and history"""
    shape = SHAPE[name]
    csr, y = fm_rows()
    P, w = fm_params(shape, 3)
    got = mbpsgd_fit(shape, csr, y, P, w, reg, True)
    ref = oracle.mbpsgd_fit(csr, y, P, w, 0.1, shape[1], "logistic", max_iter=EPOCHS, gamma=REGS[reg], reg=reg,
                            it=0, perms=host_perms(got["fm"], N), **MBPSGD_KW)
    check_mbpsgd(got, ref)
    assert same_fit(got, mbpsgd_fit(shape, csr, y, P, w, reg, True))


@gpu
@pytest.mark.parametrize("n,mb", [(N, WRAP_MB), (OVER_N, OVER_MB)], ids=["wrapping_cursor", "minibatch_over_n"])
def test_mbpsgd_wrapping_cursor_matches_oracle_and_repeats(oracle, deterministic, n, mb):
    """shuffle=False: the cursor wraps past the last row in the last minibatch of the first epoch, and with
    miniBatchSize > n a minibatch passes every row two or three times"""
    shape = SHAPE["d3_explicit_k32"]
    csr, y = fm_rows(n)
    P, w = fm_params(shape, 4)
    got = mbpsgd_fit(shape, csr, y, P, w, "l1", False, mb)
    ref = oracle.mbpsgd_fit(csr, y, P, w, 0.1, shape[1], "logistic", max_iter=EPOCHS, gamma=REGS["l1"], reg="l1",
                            mini_batch_size=mb, it=0, **MBPSGD_KW)
    check_mbpsgd(got, ref)
    assert same_fit(got, mbpsgd_fit(shape, csr, y, P, w, "l1", False, mb))


@gpu
def test_mbpsgd_generic_forms_give_the_tuned_bits(monkeypatch, deterministic):
    """NIMFM_ROW_KERNEL=generic (the generic stash forward and column kernel) over the index: the tuned pair's bits"""
    shape = SHAPE["d3_explicit_k32"]
    csr, y = fm_rows()
    P, w = fm_params(shape, 5)
    tuned = mbpsgd_fit(shape, csr, y, P, w, "identity", True)
    monkeypatch.setenv("NIMFM_ROW_KERNEL", "generic")
    generic = mbpsgd_fit(shape, csr, y, P, w, "identity", True)
    assert same_fit(tuned, generic), float(np.max(np.abs(tuned["P"] - generic["P"])))


# ------------------------------------------------------------------------------------------------ minibatch SGD
def sgd_perms(n, seed):
    return np.array([np.random.default_rng(seed + e).permutation(n) for e in range(EPOCHS)])


def fm_sgd_fit(shape, csr, y, P, w, B, perms):
    _, degree, fit_lower, k = shape
    fm = make_fm(degree, k, fit_lower, True, True, P, w, 0.1, task=nf.classification)
    opt = nf.newSGD(maxIter=EPOCHS, loss=nf.Logistic(), verbose=0, tol=0.0, **SGD_KW)
    opt.fit(csr_ds(csr), y, fm, maxThreads=B, perms=perms)
    return dict(P=fm.P.copy(), w=fm.w.copy(), intercept=fm.intercept, hist=list(opt.history), it=opt.it)


def check_sgd(got, ref):
    np.testing.assert_allclose([h[1] for h in got["hist"]], ref["loss"], rtol=1e-8)
    np.testing.assert_allclose([h[0] for h in got["hist"]], ref["viol"], rtol=1e-8)
    assert max_rel(got["P"], ref["P"]) <= 1e-8 and max_rel(got["w"], ref["w"]) <= 1e-8
    assert abs(got["intercept"] - ref["intercept"]) <= 1e-8 * max(abs(ref["intercept"]), 1e-3)
    assert got["it"] == ref["it"]


@gpu
@pytest.mark.parametrize("name", ["d3_explicit_k32", "d2_explicit_k30"])
def test_fm_sgd_minibatch_matches_oracle_and_repeats(oracle, deterministic, name):
    """fit(..., maxThreads=700, perms): shuffled minibatches of 700 rows (column 0: 700 entries), the last partial"""
    shape = SHAPE[name]
    csr, y = fm_rows()
    P, w = fm_params(shape, 6)
    perms = sgd_perms(N, 20)
    got = fm_sgd_fit(shape, csr, y, P, w, SGD_B, perms)
    ref = oracle.sgd_minibatch_fit(csr, y, P, w, 0.1, shape[1], "logistic", B=SGD_B, max_iter=EPOCHS, perms=perms,
                                   it=1, **SGD_KW)
    check_sgd(got, ref)
    assert same_fit(got, fm_sgd_fit(shape, csr, y, P, w, SGD_B, perms))


@gpu
def test_fm_sgd_minibatch_lazy_form_steps_aside(oracle, monkeypatch, deterministic):
    """on a shape whose default is the lazy (touched-features-only) form, the switch turns it off: the default and
    NIMFM_SGD_MB_LAZY=0 give the same bits, and NIMFM_SGD_MB_LAZY=1 does not bring the RED route back"""
    shape = SHAPE["d3_explicit_k32"]
    csr, y = fm_rows()
    P, w = fm_params(shape, 8)
    perms = sgd_perms(N, 30)
    default = fm_sgd_fit(shape, csr, y, P, w, LAZY_B, perms)
    ref = oracle.sgd_minibatch_fit(csr, y, P, w, 0.1, shape[1], "logistic", B=LAZY_B, max_iter=EPOCHS, perms=perms,
                                   it=1, **SGD_KW)
    check_sgd(default, ref)
    for mode in ("0", "1"):
        monkeypatch.setenv("NIMFM_SGD_MB_LAZY", mode)
        assert same_fit(default, fm_sgd_fit(shape, csr, y, P, w, LAZY_B, perms)), mode


def ffm_data(k, seed):
    csr = det_rows(FFM_N, FFM_D, FFM_FIELDS, (35, 39), seed, hot=0.85)
    rng = np.random.default_rng(seed)
    P = rng.standard_normal((FFM_FIELDS, FFM_D, k)) * (39 * k) ** -0.5
    w = rng.standard_normal(FFM_D) * 0.1
    y = np.sign(rng.standard_normal(FFM_N))
    return csr, P, w, y


def ffm_sgd_fit(csr, P, w, y, perms, B=FFM_B):
    m = make_ffm(P, w, 0.05, task=nf.classification)
    opt = nf.newSGD(maxIter=EPOCHS, loss=nf.Logistic(), verbose=0, tol=0.0, **SGD_KW)
    opt.fit(field_ds(csr), y, m, maxThreads=B, perms=perms)
    return dict(P=m.P.copy(), w=m.w.copy(), intercept=m.intercept, hist=list(opt.history), it=opt.it)


@gpu
@pytest.mark.parametrize("k", [8, 10], ids=["k8_tuned", "k10_generic"])
def test_ffm_sgd_minibatch_matches_oracle_and_repeats(oracle, deterministic, k):
    """shuffled minibatches of 700 rows with 35-39 fields each, column 0 in ~85 % of the rows"""
    csr, P, w, y = ffm_data(k, 50 + k)
    perms = sgd_perms(FFM_N, 60 + k)
    got = ffm_sgd_fit(csr, P, w, y, perms)
    ref = oracle.sgd_minibatch_fit(csr, y, P, w, 0.05, loss_kind="logistic", B=FFM_B, max_iter=EPOCHS, perms=perms,
                                   it=1, ffm=True, **SGD_KW)
    check_sgd(got, ref)
    assert same_fit(got, ffm_sgd_fit(csr, P, w, y, perms))


@gpu
def test_ffm_sgd_minibatch_generic_gives_the_tuned_bits(monkeypatch, deterministic):
    csr, P, w, y = ffm_data(8, 70)
    perms = sgd_perms(FFM_N, 71)
    tuned = ffm_sgd_fit(csr, P, w, y, perms)
    monkeypatch.setenv("NIMFM_FFM_COLS", "generic")
    assert same_fit(tuned, ffm_sgd_fit(csr, P, w, y, perms))


@gpu
def test_ffm_sgd_minibatch_repeated_field_is_refused(deterministic):
    csr, P, w, y = ffm_data(8, 80)
    dup = CSR(csr.data, csr.indices, csr.indptr, csr.n, csr.d, fields=csr.fields.copy(), n_fields=csr.n_fields)
    a = dup.indptr[5]
    dup.fields[a + 1] = dup.fields[a]                              # row 5 holds two nonzeros of one field
    with pytest.raises(Exception, match="one nonzero per field"):
        ffm_sgd_fit(dup, P, w, y, sgd_perms(FFM_N, 81))


# ------------------------------------------------------------------------------------------------ defaults
@gpu
def test_default_arguments_run_and_repeat(deterministic):
    """newMBPSGD() and newSGD().fit(..., maxThreads=-1) with their defaults (shuffled; MBPSGD's SquaredL12 on the
    default degree-2 model) run under the switch and repeat bit for bit, for FM and (SGD) FFM"""
    csr, y = fm_rows()
    yr = np.random.default_rng(9).standard_normal(N)
    P, w = fm_params(SHAPE["d2_explicit_k30"], 10)

    def fm_default(solver):
        fm = make_fm(2, 30, "explicit", True, True, P, w, 0.0)
        if solver == "mbpsgd":
            opt = nf.newMBPSGD(maxIter=2, verbose=0)
            opt.fit(csr_ds(csr), yr, fm)
        else:
            opt = nf.newSGD(maxIter=2, verbose=0)
            opt.fit(csr_ds(csr), yr, fm, maxThreads=-1)
        return dict(P=fm.P.copy(), w=fm.w.copy(), intercept=fm.intercept, hist=list(opt.history), it=opt.it)

    for solver in ("mbpsgd", "sgd"):
        a = fm_default(solver)
        assert np.all(np.isfinite(a["P"])) and same_fit(a, fm_default(solver)), solver
    fcsr, fP, fw, fy = ffm_data(10, 90)

    def ffm_default():
        m = make_ffm(fP, fw, 0.0, task=nf.classification)
        opt = nf.newSGD(maxIter=2, loss=nf.Logistic(), verbose=0)
        opt.fit(field_ds(fcsr), fy, m, maxThreads=-1)
        return dict(P=m.P.copy(), w=m.w.copy(), intercept=m.intercept, hist=list(opt.history), it=opt.it)

    assert same_fit(ffm_default(), ffm_default())
