"""The deterministic FFM gradient (NIMFM_DETERMINISTIC=1, csrc/ffm_cols.cuh) at every nComponents and field count.

Pass 1 is the FFM forward ffm_plan_mode picks (pair, staged or unit kernel); pass 2 is a column kernel over the CSC
twin of the dataset.  The tuned ffm_cols_grad_kernel<KT, E> runs where k is 4, 8 or 16, nFields <= 64, rows hold at
most 64 nonzeros and d * nFields < 2^31; every other shape, and every shape under NIMFM_FFM_COLS=generic, takes
ffm_cols_grad_generic_kernel<KT, E> (a warp per (column segment, block of 32 fields, chunk of KT components)).  Both
add every gradient element in ascending row order inside fixed 512-entry segments, so:
  - the generic kernel is held to the oracle at the shapes the tuned one refuses, past three waves of its grid, and
    to itself bit for bit on a repeat;
  - where both run they give the same bits;
  - a minibatch SGD solver under the switch repeats itself bit for bit at the default model's rank.
A row list and a dataset with a repeated field in a row stay errors."""
import ctypes as C

import numpy as np
import pytest

import nimfm_b200 as nf
from nimfm_b200 import _lib
from oracle.oracle import CSR
from helpers import max_rel
from test_gpu_ffm_sgd import field_ds, make_ffm
from test_gpu_ffm_shapes import dev_loss_grad, has_field_dups

gpu = pytest.mark.gpu

SEG = 512                         # entries per column segment (the CSC twin's task list, fm_cols.cu)
TUNED_KS = (4, 8, 16)             # ranks with a tuned column-kernel instance
TUNED_MAX_FIELDS = 64
TUNED_MAX_Z = 64                  # longest row the tuned kernel takes
GENERIC_BLOCKS_PER_SM = 4         # FFM_COLS_GENERIC_BLOCKS_PER_SM (ffm.cu): grid cap of the generic kernel
WARPS_PER_BLOCK = 4               # 128-thread blocks
B200_SMS = 148


def generic_kt(k):
    """ffm_cols_generic_kt (ffm_cols.cuh): the narrowest width in {4, 8, 16} that holds k, else chunks of 32"""
    return 4 if k <= 4 else 8 if k <= 8 else 16 if k <= 16 else 32


def cols_route(k, n_fields, d, max_z, contiguous, field_dups, env=None):
    """the column kernel ffm_launch_grad_cols runs under NIMFM_DETERMINISTIC=1 ("tuned" | "generic"), or the phrase
    of its refusal.  env: NIMFM_FFM_COLS (None | "generic")."""
    if not contiguous:
        return "contiguous"
    if field_dups:
        return "one nonzero per field"
    tuned = (k in TUNED_KS and max(max_z, 1) <= TUNED_MAX_Z and n_fields <= TUNED_MAX_FIELDS
             and d * n_fields < 2 ** 31 - 1)
    return "tuned" if tuned and env != "generic" else "generic"


def warp_tasks(csr, k):
    """warp tasks of the generic kernel: column segments x blocks of 32 fields x component chunks"""
    col_len = np.bincount(csr.indices, minlength=csr.d)
    segs = int(np.sum(-(-col_len // SEG)))
    return segs * -(-csr.n_fields // 32) * -(-k // generic_kt(k))


def resident_warps(sms):
    """an upper bound on the generic kernel's resident warps: its grid is capped at this many"""
    return GENERIC_BLOCKS_PER_SM * WARPS_PER_BLOCK * sms


# ------------------------------------------------------------------------------------------------ the case table
def det_rows(n, d, n_fields, z_range, seed, hot=0.6):
    """Rows that repeat no field and no feature: z fields drawn without replacement (z uniform in z_range, at most
    nFields), one feature from 1 .. d-1 each.  Row 0 is empty, row 1 holds one nonzero; in about `hot` of the rows
    feature 0 takes field 0, so its column is longer than one 512-entry segment; about 5 % of the values are stored
    zeros."""
    rng = np.random.default_rng(seed)
    lo, hi = z_range
    data, indices, fields, indptr = [], [], [], [0]
    for i in range(n):
        z = 0 if i == 0 else 1 if i == 1 else min(int(rng.integers(lo, hi + 1)), n_fields)
        fs = rng.choice(n_fields, size=z, replace=False)
        ids = rng.choice(np.arange(1, d), size=z, replace=False)
        if z and rng.random() < hot:
            at = np.flatnonzero(fs == 0)
            p = int(at[0]) if len(at) else 0
            fs[p], ids[p] = 0, 0
        order = np.argsort(ids)
        x = np.where(rng.random(z) < 0.3, 1.0, rng.standard_normal(z))
        x[rng.random(z) < 0.05] = 0.0
        indices.extend(ids[order].tolist())
        fields.extend(fs[order].tolist())
        data.extend(x[order].tolist())
        indptr.append(len(indices))
    return CSR(np.array(data), np.array(indices, np.int64), np.array(indptr, np.int64), n, d,
               fields=np.array(fields, np.int64), n_fields=n_fields)


def _case(name, k, n_fields, d, z_range, n=1500, fit_linear=True):
    return dict(name=name, k=k, n_fields=n_fields, d=d, z_range=z_range, n=n, fit_linear=fit_linear)


C5 = (35, 39)                     # the C5 row shape: 39 fields, a few missing in most rows
CASES = [
    _case("c5_k10", 10, 39, 6000, C5),                      # the default model's rank
    _case("c5_k20", 20, 39, 6000, C5),
    _case("k1_odd", 1, 39, 6000, (30, 39)),
    _case("k3_odd", 3, 50, 5000, (20, 50)),
    _case("k5_odd_nolinear", 5, 39, 6000, (30, 39), fit_linear=False),
    _case("k33_two_chunks", 33, 39, 3000, C5),
    _case("k64_two_chunks", 64, 39, 3000, C5),
    _case("fields80_k8", 8, 80, 3000, (80, 80), n=1200),    # more than 64 fields, rows of more than 64 nonzeros
    _case("fields1000_k6", 6, 1000, 400, (5, 40)),
]
CASE_IDS = [c["name"] for c in CASES]
CASE_BY_NAME = {c["name"]: c for c in CASES}


def case_data(c):
    seed = 700 + CASE_IDS.index(c["name"])
    csr = det_rows(c["n"], c["d"], c["n_fields"], c["z_range"], seed)
    rng = np.random.default_rng(seed)
    max_z = int(np.max(np.diff(csr.indptr)))
    P = rng.standard_normal((c["n_fields"], c["d"], c["k"])) * (max(max_z, 1) * np.sqrt(c["k"])) ** -0.5
    w = rng.standard_normal(c["d"]) * 0.1
    y = np.sign(rng.standard_normal(c["n"]))
    return csr, P, w, y


def sub_range(n):
    """a row range that starts and ends inside the long column's segments"""
    return n // 5 + 3, n // 2 + 11


# ------------------------------------------------------------------------------------------------ CPU guard
def test_case_table_routes():
    """Restates the selection rule and checks the case table against it: every case reaches the generic kernel, past
    three waves of its grid at the B200's SM count, with an empty row, stored zeros and a column longer than one
    segment (also inside the sub-range)."""
    assert cols_route(8, 39, 6000, 39, True, False) == "tuned"
    assert cols_route(8, 39, 6000, 39, True, False, env="generic") == "generic"
    assert cols_route(10, 39, 6000, 39, True, False) == "generic"                 # the default model
    assert cols_route(16, 65, 100, 39, True, False) == "generic"
    assert cols_route(4, 39, 100, 65, True, False) == "generic"
    assert cols_route(4, 39, 2 ** 26, 39, True, False) == "generic"               # 32-bit j * nFields offsets
    assert cols_route(10, 39, 6000, 39, False, False) == "contiguous"
    assert cols_route(10, 39, 6000, 39, True, True) == "one nonzero per field"
    assert [generic_kt(k) for k in (1, 3, 4, 5, 8, 10, 16, 20, 33, 64)] == [4, 4, 4, 8, 8, 16, 16, 32, 32, 32]
    assert nf.newFieldAwareFactorizationMachine(nf.classification).nComponents == 10
    ks = set()
    for c in CASES:
        csr, _, _, _ = case_data(c)
        k, lens = c["k"], np.diff(csr.indptr)
        ks.add(k)
        assert not has_field_dups(csr), c["name"]
        for i in range(csr.n):
            ids = csr.indices[csr.indptr[i]:csr.indptr[i + 1]]
            assert len(np.unique(ids)) == len(ids)
        assert cols_route(k, c["n_fields"], c["d"], int(lens.max()), True, False) == "generic", c["name"]
        assert lens[0] == 0 and np.any(csr.data == 0.0), c["name"]
        assert warp_tasks(csr, k) >= 3 * resident_warps(B200_SMS), (c["name"], warp_tasks(csr, k))
        assert np.bincount(csr.indices, minlength=csr.d).max() > SEG, c["name"]
        r0, cnt = sub_range(csr.n)
        hot_rows = np.flatnonzero([0 in csr.indices[csr.indptr[i]:csr.indptr[i + 1]] for i in range(csr.n)])
        inside = hot_rows[(hot_rows >= r0) & (hot_rows < r0 + cnt)]
        assert hot_rows[0] < r0 and hot_rows[-1] >= r0 + cnt and len(inside) > SEG // 2, c["name"]
        if c["name"].startswith("fields80"):
            assert lens.max() == 80 > TUNED_MAX_Z
    assert {1, 3, 5} <= ks and {33, 64} <= ks and {10, 20} <= ks
    assert any(not c["fit_linear"] for c in CASES)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture
def deterministic(monkeypatch):
    monkeypatch.delenv("NIMFM_FFM_COLS", raising=False)
    monkeypatch.setenv("NIMFM_DETERMINISTIC", "1")


def check_grad(got, ref):
    """the bars of test_ffm_column_route_matches_oracle"""
    ls, gP, gw, gb = got
    assert abs(ls - ref["loss"]) <= 1e-10 * abs(ref["loss"])
    assert max_rel(gP, ref["gP"]) <= 1e-9 and max_rel(gw, ref["gw"]) <= 1e-9
    assert abs(gb - ref["gb"]) <= 1e-10 * max(1.0, abs(ref["gb"]))


def same_bits(a, b):
    return a[0] == b[0] and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2]) and a[3] == b[3]


@gpu
@pytest.mark.parametrize("name", CASE_IDS)
def test_refused_shapes_match_oracle(oracle, deterministic, sms, name):
    """the full range against the oracle, the same bits on a repeat, and a sub-range against the oracle on its rows"""
    c = CASE_BY_NAME[name]
    csr, P, w, y = case_data(c)
    n, k = csr.n, c["k"]
    assert warp_tasks(csr, k) >= 3 * resident_warps(sms)
    m = make_ffm(P, w, 0.05, fit_linear=c["fit_linear"], task=nf.classification)
    ds = field_ds(csr)
    got = dev_loss_grad(m, ds, y, nf.Logistic(), n=n)
    check_grad(got, oracle.ffm_loss_grad(csr, y, P, w, 0.05, "logistic", fit_linear=c["fit_linear"]))
    if not c["fit_linear"]:
        assert not np.any(got[2])
    assert same_bits(got, dev_loss_grad(m, ds, y, nf.Logistic(), n=n))
    r0, cnt = sub_range(n)
    got = dev_loss_grad(m, ds, y, nf.Logistic(), row_begin=r0, n=cnt)
    check_grad(got, oracle.ffm_loss_grad(csr, y, P, w, 0.05, "logistic", row_begin=r0, row_end=r0 + cnt,
                                         fit_linear=c["fit_linear"]))


@gpu
@pytest.mark.parametrize("k", TUNED_KS)
@pytest.mark.parametrize("n_fields,z_range", [(13, (8, 13)), (39, C5)])
def test_generic_gives_the_tuned_bits(monkeypatch, k, n_fields, z_range):
    """on the tuned kernel's shapes NIMFM_FFM_COLS=generic gives loss, gP, gw and gb array_equal to the default route
    (the forward pass is the same; the column kernels add the same products in the same order).  39 fields hold the
    tuned kernel's second pass over fields 32.. to the generic kernel's second field block."""
    csr = det_rows(1300, 600, n_fields, z_range, 40 + k + n_fields)
    assert cols_route(k, n_fields, 600, int(np.max(np.diff(csr.indptr))), True, False) == "tuned"
    rng = np.random.default_rng(k)
    P = rng.standard_normal((n_fields, 600, k)) * 0.2
    w = rng.standard_normal(600) * 0.1
    y = np.sign(rng.standard_normal(csr.n))
    m = make_ffm(P, w, 0.05, task=nf.classification)
    ds = field_ds(csr)
    monkeypatch.setenv("NIMFM_DETERMINISTIC", "1")
    out = {}
    for env in (None, "generic"):
        if env:
            monkeypatch.setenv("NIMFM_FFM_COLS", env)
        else:
            monkeypatch.delenv("NIMFM_FFM_COLS", raising=False)
        out[env] = [dev_loss_grad(m, ds, y, nf.Logistic(), n=csr.n),
                    dev_loss_grad(m, ds, y, nf.Logistic(), row_begin=301, n=777)]
    for a, b in zip(out[None], out["generic"]):
        assert same_bits(a, b), float(np.max(np.abs(a[1] - b[1])))


def mb_sgd_epochs(csr, y, P, w, b, B, epochs, kw):
    """nimfm_ffm_sgd_minibatch_epoch through the ABI with perm = NULL: the minibatches are contiguous row ranges"""
    lib, ctx = _lib.load(), _lib.ctx()
    ds = field_ds(csr)
    ds.set_targets(y)
    m = make_ffm(P, w, b, task=nf.classification)
    h = m._to_device(ds)
    try:
        cfg = _lib.SgdCfg(nf.Logistic().kind, 1.0, kw["eta0"], kw["alpha0"], kw["alpha"], kw["beta"],
                          _lib.SCHED["optimal"], 1.0)
        it, hist = C.c_int64(1), []
        for _ in range(epochs):
            viol, ls = C.c_double(), C.c_double()
            _lib.check(lib.nimfm_ffm_sgd_minibatch_epoch(ctx, h, ds.handle(), C.byref(cfg), B, B, C.byref(it), None,
                                                         csr.n, C.byref(viol), C.byref(ls)))
            hist.append((viol.value, ls.value / csr.n))
        Pd, wd, bd = np.zeros_like(P), np.zeros(csr.d), C.c_double()
        _lib.check(lib.nimfm_ffm_get_params(ctx, h, _lib.ptr(Pd), _lib.ptr(wd), C.byref(bd)))
    finally:
        lib.nimfm_ffm_free(ctx, h)
        ds.free()
    return hist, Pd, wd, bd.value, it.value


@gpu
def test_minibatch_sgd_under_the_switch(oracle, deterministic):
    """two epochs of minibatch SGD at the C5 row shape and k = 10 (the generic kernel): two runs give the same bits,
    and both match the oracle with identity sample orders"""
    c = CASE_BY_NAME["c5_k10"]
    csr, P, w, y = case_data(c)
    n, B, epochs = csr.n, 400, 2
    kw = dict(eta0=0.03, alpha0=1e-3, alpha=2e-2, beta=3e-2)
    r1 = mb_sgd_epochs(csr, y, P, w, 0.05, B, epochs, kw)
    r2 = mb_sgd_epochs(csr, y, P, w, 0.05, B, epochs, kw)
    assert r1[0] == r2[0] and np.array_equal(r1[1], r2[1]) and np.array_equal(r1[2], r2[2]) and r1[3] == r2[3]
    perms = np.tile(np.arange(n), (epochs, 1))
    ref = oracle.sgd_minibatch_fit(csr, y, P, w, 0.05, loss_kind="logistic", B=B, max_iter=epochs, perms=perms, it=1,
                                   ffm=True, **kw)
    hist, Pd, wd, bd, it = r1
    np.testing.assert_allclose([h[1] for h in hist], ref["loss"], rtol=1e-8)
    np.testing.assert_allclose([h[0] for h in hist], ref["viol"], rtol=1e-8)
    np.testing.assert_allclose(Pd, ref["P"], rtol=1e-8, atol=1e-13)
    np.testing.assert_allclose(wd, ref["w"], rtol=1e-8, atol=1e-13)
    assert abs(bd - ref["intercept"]) <= 1e-8 and it == ref["it"]


@gpu
def test_refusals_at_the_default_rank(deterministic):
    """at k = 10 (only the generic kernel runs there) a row list and a dataset that repeats a field stay errors"""
    c = CASE_BY_NAME["c5_k10"]
    csr, P, w, y = case_data(c)
    m = make_ffm(P, w, 0.0)
    with pytest.raises(Exception, match="contiguous"):
        dev_loss_grad(m, field_ds(csr), y, nf.Squared(), rows=np.array([3, 1, 2]))
    dup = CSR(csr.data, csr.indices, csr.indptr, csr.n, csr.d, fields=csr.fields.copy(), n_fields=csr.n_fields)
    a = dup.indptr[5]
    dup.fields[a + 1] = dup.fields[a]                              # row 5 holds two nonzeros of one field
    assert has_field_dups(dup)
    with pytest.raises(Exception, match="one nonzero per field"):
        dev_loss_grad(m, field_ds(dup), y, nf.Squared(), n=csr.n)
