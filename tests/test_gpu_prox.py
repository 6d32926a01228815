"""The proximal operators of MBPSGD and PSGD (nimfm_b200/csrc/prox_kernels.cuh) against oracle.prox_matrix, at
the shapes where the kernels change how they split the work.

An MBPSGD minibatch whose gradient is exactly zero is exactly one prox call.  The dataset is one row of stored 0.0
values (the upload keeps them), so every P and w gradient term carries a factor x = 0, and the squared loss of
y = 0 against a prediction of 0 has dL = 0 as well.  With beta = alpha = 0, the constant schedule and eta0 = 1 the
step (P - 1*0) * 1/(1+0) leaves P bit-identical, and lam = gamma*eta/(1+eta*beta) is gamma bit for bit.  One PSGD
sample under the same settings is one prox call with lam = gamma*etaS = gamma.

Kernel shapes covered:
  - SquaredL12(transpose=true): sql12_pass / update / apply.  R = max(1, 256/SB8) features per block, R*SB8
    threads, a grid capped at numSMs*8 blocks past which a thread walks several features, SB8 <= 1024.
  - L21 and SquaredL12(transpose=false): prox_rows_kernel.  One warp per (feature, order) vector, k <= 128, so 1
    to 4 elements per lane, numSMs*16 blocks of 8 warps past which a warp takes several vectors.
  - L1: fused into mbpsgd_step_kernel.

Both SquaredL12 kernels find the threshold with Michelot's iteration.  A pass counts the elements above the current
threshold and recomputes it from them.  In floating point an element that sits exactly at the threshold of the
others makes that iteration cycle: the pass that includes it rounds the threshold up to it, so it drops out, and the
pass without it rounds the threshold one ulp below it, so it comes back.  TIES holds such columns.  The CPU tests
below restate the device's operation order and show that each of them cycles under a stop-when-the-count-repeats
rule and terminates under the stop-when-the-count-does-not-decrease rule the kernels use.  The GPU tests then require
the device to give the restated rule's bits on them.
"""
from fractions import Fraction

import numpy as np
import pytest

import nimfm_b200 as nf
from nimfm_b200 import _lib
from oracle.oracle import CSR

gpu = pytest.mark.gpu
EPS = np.finfo(np.float64).eps

# Columns at lam = 1 in which one element equals, after rounding, the threshold of the others.  They were found by a
# seeded search over 2 to 5 magnitudes in [0.5, 2] with random signs; every one cycles in both summation orders
# below.
TIE_LAM = 1.0
TIES = [
    [0.9624079957639571, 1.2811139403761498, 1.1249060490337428],
    [1.1377894620623865, 0.906409173378932, -0.8176794541765274],
    [-1.9696880026970587, 1.5437612605290878, -1.8897151486256607],
    [-0.6765758981243482, 0.592006980009303, -0.6285589781068958, 0.7668895538013163],
]


# ------------------------------------------------------------------------------------------ the restated iteration
def _fma(a, b, c):
    """a*b + c with one rounding: the device contracts 1 + (2*lam)*cnt into a DFMA"""
    return float(Fraction(a) * Fraction(b) + Fraction(c))


def seq_sum(v):
    s = 0.0
    for x in v:
        s += x
    return s


def column_sum(R):
    """the column kernel's order when every nonzero lies in the first grid*R features: each block adds its R
    features in order, then the block partials are added in order (seq_sum when the nonzeros share a block)"""
    return lambda v: seq_sum([seq_sum(v[i:i + R]) for i in range(0, len(v), R)])


def butterfly_sum(v):
    """warp_sum (common.cuh) over lanes 0..len(v)-1, the other lanes 0: the row kernel's order for a vector
    whose nonzeros are in lanes 0..31"""
    lanes = list(v) + [0.0] * (32 - len(v))
    off = 16
    while off:
        lanes = [lanes[i] + lanes[i ^ off] for i in range(32)]
        off >>= 1
    return lanes[0]


def michelot(vals, lam, total, rule, n_zeros=0, cap=4096):
    """Michelot's iteration in the device's operation order on |vals| plus n_zeros stored zeros.
    rule "repeat": stop when a pass counts as many elements as the one before and apply that pass's threshold.
    rule "no_decrease": stop when a pass counts no fewer elements than the one before and apply the threshold
    that pass took as input.  Returns (threshold, passes), or (None, passes) once the state repeats, which
    proves the iteration never stops."""
    a = [abs(x) for x in vals]
    tau, prev = -1.0, (-1.0 if rule == "repeat" else float("inf"))
    seen = set()
    for it in range(cap):
        act = [x if x > tau else 0.0 for x in a]
        cnt = float(sum(x > tau for x in a) + (n_zeros if tau < 0.0 else 0))
        if rule == "no_decrease" and cnt >= prev:
            return tau, it + 1
        new = 2 * lam * (total(act) / _fma(2.0 * lam, cnt, 1.0))
        if rule == "repeat" and cnt == prev:
            return new, it + 1
        tau, prev = new, cnt
        if (tau, prev) in seen:
            return None, it + 1
        seen.add((tau, prev))
    return None, cap


def soft(p, tau):
    p = np.asarray(p, dtype=np.float64)
    return np.sign(p) * np.maximum(np.abs(p) - tau, 0.0)


def greedy_chain(lam, n_max=64):
    """Magnitudes such that each Michelot pass drops exactly one of them: grown from the top, each new element
    is just below both the threshold of the set with it and the smallest element so far."""
    A = [1.0]
    while len(A) < n_max:
        m, S, n = min(A), sum(A), len(A)
        x = min(m * (1 + 2 * lam * (n + 1)) / (2 * lam) - S, 2 * lam * S / (1 + 2 * lam * n), m) * (1 - 1e-9)
        if not (0 < x < m):
            break
        A.append(x)
    return A


# ------------------------------------------------------------------------------------------ CPU: the tie fixtures
@pytest.mark.parametrize("order", ["column", "row"])
@pytest.mark.parametrize("pad", [0, 1, 29])
@pytest.mark.parametrize("lit", range(len(TIES)))
def test_tie_fixture_cycles_under_the_repeat_rule_only(oracle, lit, pad, order):
    """Each literal of TIES, padded with stored zeros, cycles under the repeat rule in the kernel's summation
    order, terminates under the no-decrease rule, and the oracle (randomised selection) terminates on it too
    and agrees with the no-decrease rule's result."""
    col, total = TIES[lit], (seq_sum if order == "column" else butterfly_sum)
    assert michelot(col, TIE_LAM, total, "repeat", n_zeros=pad)[0] is None
    tau, passes = michelot(col, TIE_LAM, total, "no_decrease", n_zeros=pad)
    assert tau is not None and passes <= len(col) + 2
    full = np.array(col + [0.0] * pad)
    ref = oracle.prox_matrix(full[:, None], TIE_LAM, "squaredl12").ravel()
    assert np.max(np.abs(soft(full, tau) - ref)) <= 8 * EPS * np.max(np.abs(full))
    # the tied element really sits at the threshold: it keeps at most a few ulps
    tied = np.argmin(np.abs(np.abs(col) - tau))
    assert abs(abs(col[tied]) - tau) <= 4 * EPS * abs(col[tied])


@pytest.mark.parametrize("lam", [1e-2, 1.0, 100.0])
def test_greedy_chain_outlasts_the_host_checks(oracle, lam):
    """The chain column drops one element per pass, so the column kernel's iteration runs past several of the
    host's convergence checks (one every 4 passes)."""
    chain = greedy_chain(lam)
    tau, passes = michelot(chain, lam, seq_sum, "no_decrease", n_zeros=5)
    assert passes >= len(chain) + 1   # the zeros drop out in the first pass, then (almost) one element per pass
    if lam >= 1.0:
        assert passes >= 13
    # without a tie both rules stop after the same pass with the same bits
    assert michelot(chain, lam, seq_sum, "repeat", n_zeros=5) == (tau, passes)
    ref = oracle.prox_matrix(np.array(chain + [0.0] * 5)[:, None], lam, "squaredl12").ravel()
    assert np.count_nonzero(ref) == 1


# ------------------------------------------------------------------------------------------ GPU harness
@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def zero_row(d):
    """one row of stored 0.0 values, over the first, last and a few middle features"""
    cols = np.unique(np.linspace(0, d - 1, min(d, 6)).astype(np.int64))
    return CSR(np.zeros(len(cols)), cols, [0, len(cols)], 1, d)


def reg_obj(reg):
    return {"l1": nf.newL1, "l21": nf.newL21, "squaredl12": nf.newSquaredL12,
            "squaredl12_rows": lambda: nf.newSquaredL12(transpose=False)}[reg]()


def make_fm(P, degree, fit_lower):
    nO, k, d = P.shape
    fm = nf.newFactorizationMachine(nf.regression, degree=degree, nComponents=k, fitLower=fit_lower,
                                    fitLinear=True, fitIntercept=False, warmStart=True)
    fm.P, fm.w, fm.intercept, fm.isInitialized = P.copy(), np.zeros(d), 0.0, True
    return fm


def device_prox(P, gamma, reg, degree=2, fit_lower="explicit", solver="mbpsgd"):
    """reg.prox(P, gamma) on the device through one zero-gradient MBPSGD minibatch (or PSGD sample)"""
    d = P.shape[2]
    csr = zero_row(d)
    ds = nf.newCSRDataset(csr.data, csr.indices, csr.indptr, 1, d)
    fm = make_fm(P, degree, fit_lower)
    kw = dict(maxIter=1, eta0=1.0, alpha0=0.0, alpha=0.0, beta=0.0, gamma=gamma, reg=reg_obj(reg),
              scheduling=nf.constant, verbose=0, tol=0.0, shuffle=False)
    opt = nf.newMBPSGD(miniBatchSize=1, **kw) if solver == "mbpsgd" else nf.newPSGD(**kw)
    opt.fit(ds, np.zeros(1), fm)
    return np.asarray(fm.P, dtype=np.float64)


def sorted_threshold(V, lam):
    """per row of V: the closed-form SquaredL12 threshold tau (bruteforce.prox_squaredl12_sorted) and the
    number of elements above it"""
    a = -np.sort(-np.abs(V), axis=1)
    c = np.cumsum(a, axis=1)
    m = np.arange(1, a.shape[1] + 1)
    ok = a > 2 * lam * c / (1.0 + 2.0 * lam * m)
    theta = np.where(ok.any(axis=1), a.shape[1] - np.argmax(ok[:, ::-1], axis=1), 0)
    S = np.where(theta > 0, c[np.arange(len(V)), np.maximum(theta - 1, 0)], 0.0)
    return 2 * lam * S / (1.0 + 2.0 * lam * theta), theta


def assert_sql12(got, ref, V, lam, what):
    """V: input vectors as rows.  The device and the oracle add the same active elements in different orders;
    each sum of n positive terms is within n*eps/2 of the exact one, so the thresholds agree to
    n_active*eps*tau, and an element to 8*eps*max|p| beyond that.  The zero pattern must match except for
    elements within that tolerance of the threshold."""
    tau, theta = sorted_threshold(V, lam)
    tol = EPS * (8 * np.max(np.abs(V), axis=1) + theta * tau)
    err = np.abs(got - ref)
    bad = np.argwhere(err > tol[:, None])
    assert bad.size == 0, f"{what}: {len(bad)} elements off, first {tuple(bad[0])}: got {got[tuple(bad[0])]!r} " \
                          f"oracle {ref[tuple(bad[0])]!r} tol {tol[bad[0][0]]:.3e}"
    near = np.abs(np.abs(V) - tau[:, None]) <= tol[:, None]
    mism = ((got == 0.0) != (ref == 0.0)) & ~near
    assert not mism.any(), f"{what}: zero pattern differs at {tuple(np.argwhere(mism)[0])}"


# ------------------------------------------------------------------------------------------ column contents
KINDS = ["gauss", "single", "zeros", "equal", "negzero", "spread", "chain", "tie"]


def fill_columns(P2, lam, rng, offset):
    """P2: [k, dd] (one order, model layout), filled in place; vector s gets KINDS[(s + offset) % len].
    Returns {s: tie literal index} for the tie vectors (tie elements at features 0..n-1, zeros elsewhere)."""
    k, dd = P2.shape
    ties = {}
    chain = greedy_chain(lam)
    for s in range(k):
        kind = KINDS[(s + offset) % len(KINDS)]
        if kind == "tie" and (lam != TIE_LAM or dd < 4):
            kind = "gauss"
        if kind == "chain" and dd < len(chain):
            kind = "spread"
        v = np.zeros(dd)
        if kind == "gauss":
            v = rng.standard_normal(dd) * 10.0 ** rng.uniform(-3, 3)
        elif kind == "single":
            v[rng.integers(dd)] = rng.choice([-1.0, 1.0]) * rng.uniform(0.1, 10.0)
        elif kind == "equal":
            v = np.where(rng.random(dd) < 0.5, -0.75, 0.75)
        elif kind == "negzero":
            v = rng.standard_normal(dd)
            v[rng.random(dd) < 0.4] = -0.0
        elif kind == "spread":
            v = np.where(rng.random(dd) < 0.5, -1.0, 1.0) * 10.0 ** rng.uniform(-8, 3, dd)
        elif kind == "chain":
            v[rng.choice(dd, size=len(chain), replace=False)] = np.array(chain) * rng.choice([-1.0, 1.0], len(chain))
        elif kind == "tie":
            lit = (s + offset) // len(KINDS) % len(TIES)
            v[:len(TIES[lit])] = TIES[lit]
            ties[s] = lit
        P2[s] = v
    return ties


def check_tie_bits(got_vec, lit, n_zeros, total):
    """the device's bits on a tie vector are those of the restated no-decrease rule"""
    col = TIES[lit]
    tau, _ = michelot(col, TIE_LAM, total, "no_decrease", n_zeros=n_zeros)
    want = soft(col, tau)
    assert np.array_equal(got_vec[:len(col)], want), f"tie {lit}: got {got_vec[:len(col)]!r} want {want!r}"
    assert not np.any(got_vec[len(col):])


# ------------------------------------------------------------------------------------------ column-wise SquaredL12
def column_shapes(k, sms):
    R = max(1, 256 // k)
    G = sms * 8
    dds = {1, R - 1, R, R + 1, 5 * R + 3, 2 * G * R + 1}
    if k >= 1000:
        dds = {1, 2, 7, 600, 2 * G + 1}   # R = 1: past the grid cap at 2*numSMs*8+1 features
    return sorted(x for x in dds if x >= 1)


COLUMN_K = [1, 3, 16, 30, 100, 256, 257, 1000, 1024]


@gpu
@pytest.mark.parametrize("lam_kind", ["tie", "wide"])
@pytest.mark.parametrize("k", COLUMN_K)
def test_squaredl12_columns_match_oracle(oracle, sms, k, lam_kind):
    """every (order, component) vector over all features, at every block size and past the grid cap, with
    lam = 1 (tie and chain columns, few active elements) and lam = 0.25/dd (most elements active)"""
    for i, dd in enumerate(column_shapes(k, sms)):
        rng = np.random.default_rng(1000 * k + i + (7 if lam_kind == "wide" else 0))
        lam = TIE_LAM if lam_kind == "tie" else 0.25 / dd
        P = np.zeros((1, k, dd))
        ties = fill_columns(P[0], lam, rng, offset=i + k)
        got = device_prox(P, lam, "squaredl12")
        ref = oracle.prox_matrix(P[0].T, lam, "squaredl12").T
        assert_sql12(got[0], ref, P[0], lam, f"k={k} dd={dd}")
        for s, lit in ties.items():
            check_tie_bits(got[0, s], lit, dd - len(TIES[lit]), column_sum(max(1, 256 // k)))


@gpu
@pytest.mark.parametrize("lam", [1e-12, 1e6])
@pytest.mark.parametrize("k,dd", [(3, 90), (30, 9), (257, 5000)])
def test_squaredl12_columns_extreme_lambda(oracle, k, dd, lam):
    """lam tiny (the threshold is ~2*lam*sum|p|, nearly every element survives) and huge (only each column's
    largest element survives, as |p|/(1+2*lam))"""
    rng = np.random.default_rng(k + dd)
    P = np.zeros((1, k, dd))
    fill_columns(P[0], lam, rng, offset=k)
    got = device_prox(P, lam, "squaredl12")
    ref = oracle.prox_matrix(P[0].T, lam, "squaredl12").T
    assert_sql12(got[0], ref, P[0], lam, f"k={k} dd={dd} lam={lam}")


@gpu
def test_squaredl12_columns_converge_apart(oracle):
    """one call where the columns need from 2 to 14 passes: chains of every length at lam = 1 next to tie
    columns that stop after 4 passes and constant columns that stop after 2"""
    lam, dd = TIE_LAM, 700
    chain = greedy_chain(lam)
    cols = []
    for L in range(1, len(chain) + 1):
        v = np.zeros(dd)
        v[np.arange(L) * 37] = chain[:L]
        cols.append(v)
    for lit in range(len(TIES)):
        v = np.zeros(dd)
        v[:len(TIES[lit])] = TIES[lit]
        cols.append(v)
    cols.append(np.full(dd, -0.5))
    P = np.array(cols)[None]
    got = device_prox(P, lam, "squaredl12")
    ref = oracle.prox_matrix(P[0].T, lam, "squaredl12").T
    assert_sql12(got[0], ref, P[0], lam, "mixed passes")
    for lit in range(len(TIES)):
        check_tie_bits(got[0, len(chain) + lit], lit, dd - len(TIES[lit]), column_sum(256 // len(cols)))


@gpu
def test_squaredl12_refuses_more_than_1024_columns():
    P = np.random.default_rng(0).standard_normal((1, 1025, 4))
    with pytest.raises(_lib.NimfmCudaError, match="nOrders\\*nComponents=1025 > 1024"):
        device_prox(P, 0.5, "squaredl12")


@gpu
@pytest.mark.parametrize("k,dd", [(1, 3), (30, 700), (1024, 40)])
def test_zero_gamma_leaves_P_bit_identical(k, dd):
    """the harness itself: with gamma = 0 no prox runs, and the zero-gradient step changes no bit of P"""
    P = np.random.default_rng(k).standard_normal((1, k, dd)) * 3.0
    got = device_prox(P, 0.0, "squaredl12")
    assert np.array_equal(got.view(np.int64), P.view(np.int64))


# ------------------------------------------------------------------------------------------ row-wise
ROW_K = [1, 7, 31, 32, 33, 64, 65, 100, 128]


def row_vectors(nO, k, dd, rng):
    """[nO, k, dd]: Gaussian vectors of random scale, with zero vectors and single-element vectors mixed in"""
    P = rng.standard_normal((nO, k, dd)) * 10.0 ** rng.uniform(-2, 1, (nO, 1, dd))
    P[:, :, rng.random(dd) < 0.05] = 0.0
    one = rng.random(dd) < 0.05
    P[:, 1:, one] = 0.0
    return P


@gpu
@pytest.mark.parametrize("k", ROW_K)
def test_l21_rows_match_oracle(oracle, sms, k):
    """L21 at degrees 2 to 6 (1 to 5 orders of vectors), more vectors than one grid of warps covers"""
    warps = sms * 16 * 8
    for degree in range(2, 7):
        nO = degree - 1
        dd = (2 * warps + 5) // nO + 1 if degree in (2, 6) else 50 + degree
        rng = np.random.default_rng(100 * k + degree)
        P = row_vectors(nO, k, dd, rng)
        # about half the vectors vanish; the factor keeps lam off every vector's norm
        lam = float(np.median(np.sqrt(np.sum(P ** 2, axis=1)))) * (1.0 + 1.23e-6)
        got = device_prox(P, lam, "l21", degree=degree)
        for o in range(nO):
            ref = oracle.prox_matrix(P[o].T, lam, "l21").T
            V = P[o].T
            tol = EPS * (8 + k) * np.max(np.abs(V), axis=1)
            assert np.all(np.abs(got[o] - ref).T <= tol[:, None]), f"degree={degree} order={o}"
            assert np.array_equal(got[o] == 0.0, ref == 0.0), f"degree={degree} order={o}: zero pattern"


@gpu
@pytest.mark.parametrize("k", [1, 4, 16, 33, 64, 128])
def test_l21_at_its_boundary(oracle, k):
    """||v|| == lam exactly (single elements and, where k is a power of 4, k equal elements of a power of two)
    must become 0; ||v|| one ulp above lam must not; zero vectors stay zero"""
    lam = 0.5
    up = np.nextafter(0.5, 1.0)
    vecs = []
    for i in sorted({0, k // 2, k - 1}):
        for val in (0.5, -0.5, up, -up, np.nextafter(0.5, 0.0)):
            v = np.zeros(k)
            v[i] = val
            vecs.append(v)
    if k in (4, 16, 64):
        vecs.append(np.full(k, 0.5 / np.sqrt(k)))   # exact: 0.25, 0.125, 0.0625
    vecs.append(np.zeros(k))
    V = np.array(vecs)
    got = device_prox(V.T[None].copy(), lam, "l21")[0].T
    ref = oracle.prox_matrix(V, lam, "l21")
    norms = np.sqrt(np.sum(V ** 2, axis=1))
    assert np.all((ref == 0.0).all(axis=1) == (norms <= lam))
    assert np.array_equal(got, ref)


@gpu
def test_row_prox_refuses_more_than_128_components():
    P = np.random.default_rng(0).standard_normal((1, 129, 4))
    for reg in ("l21", "squaredl12_rows"):
        with pytest.raises(_lib.NimfmCudaError, match="row-wise prox supports nComponents <= 128"):
            device_prox(P, 0.5, reg)


@gpu
@pytest.mark.parametrize("k", ROW_K)
def test_squaredl12_rows_match_oracle(oracle, sms, k):
    """SquaredL12(transpose=false): one vector per feature, lam = 1 with tie vectors in lanes 0..n-1, and a
    wider lam; past one grid of warps"""
    warps = sms * 16 * 8
    dd = 2 * warps + 3
    for lam in (TIE_LAM, 0.05):
        rng = np.random.default_rng(k + int(lam * 100))
        P = row_vectors(1, k, dd, rng)
        ties = {}
        if lam == TIE_LAM:
            for j in range(0, dd, 997):
                lit = (j // 997) % len(TIES)
                if k >= len(TIES[lit]):
                    P[0, :, j] = 0.0
                    P[0, :len(TIES[lit]), j] = TIES[lit]
                    ties[j] = lit
        got = device_prox(P, lam, "squaredl12_rows")
        ref = oracle.prox_matrix(P[0].T, lam, "squaredl12_rows")
        assert_sql12(got[0].T, ref, P[0].T, lam, f"k={k} lam={lam}")
        for j, lit in ties.items():
            check_tie_bits(got[0, :, j], lit, k - len(TIES[lit]), butterfly_sum)


# ------------------------------------------------------------------------------------------ L1 (fused in the step)
@gpu
def test_l1_at_its_boundary(oracle):
    lam = 0.375
    edge = [lam, np.nextafter(lam, 1.0), np.nextafter(lam, 0.0)]
    vals = np.array(edge + [-x for x in edge] + [0.0, -0.0, 1e-300, 2.0, -7.5])
    rng = np.random.default_rng(3)
    P = np.concatenate([vals, rng.standard_normal(37 * 9 - len(vals))]).reshape(1, 9, 37)
    got = device_prox(P, lam, "l1")
    ref = oracle.prox_matrix(P[0].T, lam, "l1").T
    assert np.array_equal(got[0], ref)
    assert np.all(got[0].ravel()[[0, 3]] == 0.0) and np.all(got[0].ravel()[[1, 4]] != 0.0)


# ------------------------------------------------------------------------------------------ PSGD call site
@gpu
@pytest.mark.parametrize("reg", ["squaredl12", "squaredl12_rows"])
def test_psgd_prox_matches_oracle(oracle, reg):
    """PSGD's SquaredL12 route proxes after every sample with lam = gamma*etaS; one zero-gradient sample is one
    prox call at lam = gamma"""
    k, dd = 40, 2000
    rng = np.random.default_rng(11)
    P = row_vectors(1, k, dd, rng)
    if reg == "squaredl12":
        P[0, 5] = 0.0
        P[0, 5, :3] = TIES[0]
    else:
        P[0, :, 9] = 0.0
        P[0, :4, 9] = TIES[3]
    got = device_prox(P, TIE_LAM, reg, solver="psgd")
    if reg == "squaredl12":
        ref = oracle.prox_matrix(P[0].T, TIE_LAM, reg).T
        assert_sql12(got[0], ref, P[0], TIE_LAM, "psgd columns")
        check_tie_bits(got[0, 5], 0, dd - 3, column_sum(256 // k))
    else:
        ref = oracle.prox_matrix(P[0].T, TIE_LAM, reg)
        assert_sql12(got[0].T, ref, P[0].T, TIE_LAM, "psgd rows")
        check_tie_bits(got[0, :, 9], 3, k - 4, butterfly_sum)
