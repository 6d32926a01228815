"""Host-side mirror of nimfm's solver objects: constructor signatures, fit() control flow (epoch
loop, verbose printing, callback, tol stopping, NaN check) stay here exactly where the reference has
them; every epoch body is ONE call into libnimfm_cuda.so.

  CD      optimizer/cd.nim:12-13, 110-194
  SGD     optimizer/sgd.nim:23-52, 261-328        (FFM: optimizer/sgd_ffm.nim:49-106)
  AdaGrad optimizer/adagrad.nim:20-44, 137-203    (FFM: optimizer/adagrad_ffm.nim:11-66)
  MBPSGD  optimizer/minibatch_psgd.nim:25-64, 127-211

Shuffling uses a NumPy generator seeded from fm.randomState (Nim's RNG stream is not reproduced;
SURVEY Appendix B): pass shuffle=False, or perms=..., for reproducible parity runs.
"""
import ctypes as C
import math
import sys
import time

import numpy as np

from . import _lib
from . import distributed as _dist
from .dataset import CSCDataset, CSRDataset, CSRFieldDataset
from .loss import Squared
from .model import FactorizationMachine, FieldAwareFactorizationMachine

constant, optimal, invscaling, pegasos = "constant", "optimal", "invscaling", "pegasos"


# ---------------------------------------------------------------- optimizer/utils.nim:26-59
def echoHeader(maxIter, viol=True, loss=True, regul=True):
    s = "Epoch".ljust(len(str(maxIter)))
    if viol:
        s += "   " + "Violation".ljust(10)
    if loss:
        s += "   " + "Loss".ljust(10)
    if regul:
        s += "   Regularization"
    sys.stdout.write(s + "\n")
    sys.stdout.flush()


def echoInfo(it, maxIter, viol, loss, regul):
    s = str(it).ljust(max(5, len(str(maxIter))))
    for v in (viol, loss, regul):
        if v >= 0:
            s += "   " + f"{v:<10.4e}"
    sys.stdout.write(s + "\n")
    sys.stdout.flush()


def regularization(P, w, intercept, alpha0, alpha, beta):
    """utils.nim:56-59 (host-side, for verbose output and objective checks)"""
    return (0.5 * alpha0 * intercept ** 2 + 0.5 * alpha * float(np.sum(np.square(w)))
            + 0.5 * beta * float(np.sum(np.square(P))))


class _Base:                                  # optimizer_base.nim:1-14
    def _rng(self, fm):
        return np.random.default_rng(fm.randomState)

    def _stopping(self, fm, lossVal, viol, epoch):   # sgd.nim:72-89 stoppingCriterion
        if math.isnan(lossVal):
            print("Loss is NaN. Use smaller learning rate.")
            return False
        if self.verbose > 0:
            reg = regularization(fm.P, fm.w, fm.intercept, self.alpha0, self.alpha, self.beta)
            echoInfo(epoch + 1, self.maxIter, viol, lossVal, reg)
        if viol < self.tol:
            if self.verbose > 0:
                print(f"Converged at epoch {epoch}.")
            self._converged = True
            return False
        return True


# ================================================================ CD
class CD(_Base):
    def __init__(self, maxIter=100, alpha0=1e-6, alpha=1e-3, beta=1e-3, loss=None, verbose=1, tol=1e-3):
        self.maxIter, self.alpha0, self.alpha, self.beta = maxIter, alpha0, alpha, beta
        self.loss = loss if loss is not None else Squared()
        self.verbose, self.tol = verbose, tol

    def fit(self, X, y, fm, callback=None):
        """cd.nim:110-194.  X must be a CSCDataset (ColDataset)."""
        if not isinstance(X, CSCDataset):
            raise TypeError("CD.fit needs a CSCDataset")
        fm.init(X)
        y = fm.checkTarget(y)
        lib, ctx = _lib.load(), _lib.ctx()
        X.set_targets(y)
        h = fm._to_device(X.nFeatures)
        cfg = _lib.CdCfg(self.loss.kind, self.loss.threshold, self.alpha0, self.alpha, self.beta)
        self.history = []
        self.epoch_seconds = []     # host wall time of each epoch's single library call (blocking)
        try:
            _lib.check(lib.nimfm_fm_cd_begin(ctx, h, X.handle(), C.byref(cfg)))
            if self.verbose > 0:
                echoHeader(self.maxIter)
            converged = False
            for it in range(self.maxIter):
                viol, lossMean, reg = C.c_double(), C.c_double(), C.c_double()
                t0 = time.perf_counter()
                _lib.check(lib.nimfm_fm_cd_epoch(ctx, h, X.handle(), C.byref(cfg), C.byref(viol),
                                                 C.byref(lossMean), C.byref(reg)))
                self.epoch_seconds.append(time.perf_counter() - t0)
                self.history.append((viol.value, lossMean.value, reg.value))
                if callback is not None:
                    fm._from_device(h)
                    callback(self, fm)
                if self.verbose > 0:
                    echoInfo(it + 1, self.maxIter, viol.value, lossMean.value, reg.value)
                if viol.value < self.tol:
                    if self.verbose > 0:
                        print(f"Converged at iteration {it + 1}.")
                    converged = True
                    break
            if not converged and self.verbose > 0:
                print("Objective did not converge. Increase maxIter.")
            _lib.check(lib.nimfm_fm_cd_end(ctx, h))
            fm._from_device(h)
        finally:
            lib.nimfm_fm_free(ctx, h)


def newCD(maxIter=100, alpha0=1e-6, alpha=1e-3, beta=1e-3, loss=None, verbose=1, tol=1e-3):
    return CD(maxIter, alpha0, alpha, beta, loss, verbose, tol)


class PCD(_Base):
    """Proximal coordinate descent (optimizer/pcd.nim:10-200): CD's sweeps with the sparsity
    regulariser's per-coordinate prox.  reg: L1 or SquaredL12 (default, degree 2 only)."""

    def __init__(self, maxIter=100, alpha0=1e-6, alpha=1e-3, beta=1e-4, gamma=1e-4, loss=None, reg=None,
                 verbose=1, tol=1e-3):
        self.maxIter, self.alpha0, self.alpha, self.beta, self.gamma = maxIter, alpha0, alpha, beta, gamma
        self.loss = loss if loss is not None else Squared()
        self.reg = reg if reg is not None else SquaredL12()
        self.verbose, self.tol = verbose, tol

    def fit(self, X, y, sfm, callback=None):
        """pcd.nim:108-200.  X must be a CSCDataset (ColDataset)."""
        if not isinstance(X, CSCDataset):
            raise TypeError("PCD.fit needs a CSCDataset")
        if isinstance(self.reg, L21):
            raise TypeError("L21 has no coordinate-wise prox (it is a PBCD regulariser, l21.nim:24-29)")
        sfm.init(X)
        y = sfm.checkTarget(y)
        lib, ctx = _lib.load(), _lib.ctx()
        X.set_targets(y)
        n = X.nSamples
        h = sfm._to_device(X.nFeatures)
        cdcfg = _lib.CdCfg(self.loss.kind, self.loss.threshold, self.alpha0, self.alpha, self.beta)
        cfg = _lib.PcdCfg(self.loss.kind, self.loss.threshold, self.alpha0, self.alpha, self.beta, self.gamma,
                          self.reg.kind)
        self.history = []
        self.epoch_seconds = []
        try:
            self.reg.initCD(sfm.degree, X.nFeatures + sfm.nAugments, sfm.nComponents)   # :151
            _lib.check(lib.nimfm_fm_cd_begin(ctx, h, X.handle(), C.byref(cdcfg)))
            if self.verbose > 0:
                echoHeader(self.maxIter)
            converged = False
            for it in range(self.maxIter):
                viol, lossMean, reg = C.c_double(), C.c_double(), C.c_double()
                t0 = time.perf_counter()
                _lib.check(lib.nimfm_fm_pcd_epoch(ctx, h, X.handle(), C.byref(cfg), C.byref(viol),
                                                  C.byref(lossMean), C.byref(reg)))
                self.epoch_seconds.append(time.perf_counter() - t0)
                regVal = reg.value
                if self.verbose > 0 or callback is not None:
                    sfm._from_device(h)
                if self.verbose > 0:            # :178-185: gamma (n-scaled) * reg.eval(P[order].T), all over n
                    for order in range(sfm.nOrders):
                        regVal += self.gamma * self.reg.eval(np.asarray(sfm.P[order]).T, sfm.degree - order)
                self.history.append((viol.value, lossMean.value, regVal))
                if self.verbose > 0:
                    echoInfo(it + 1, self.maxIter, viol.value, lossMean.value, regVal)
                if callback is not None:
                    callback(self, sfm)
                if viol.value < self.tol:
                    if self.verbose > 0:
                        print(f"Converged at iteration {it + 1}.")
                    converged = True
                    break
            if not converged and self.verbose > 0:
                print("Objective did not converge. Increase maxIter.")
            _lib.check(lib.nimfm_fm_cd_end(ctx, h))
            sfm._from_device(h)
        finally:
            lib.nimfm_fm_free(ctx, h)


def newPCD(maxIter=100, alpha0=1e-6, alpha=1e-3, beta=1e-4, gamma=1e-4, loss=None, reg=None, verbose=1, tol=1e-3):
    return PCD(maxIter, alpha0, alpha, beta, gamma, loss, reg, verbose, tol)


def _windowed_epoch(epoch, ctx, h, X, cfg, it, viol, lossSum, multiple):
    """One SGD / AdaGrad epoch over a StreamCSRDataset kept on disk: the per-sample (or per-minibatch) loop
    runs over one resident window of rows after another, in file order, with the iteration counter and the
    optimizer state carried across windows; viol and the loss sum add up (sgd.nim:298-307)."""
    v, ls = C.c_double(), C.c_double()
    viol.value, lossSum.value = 0.0, 0.0
    for a, b, win in X.windows(multiple=multiple):
        _lib.check(epoch(ctx, h, win.handle(), C.byref(cfg), C.byref(it), None, b - a, C.byref(v), C.byref(ls)))
        viol.value += v.value
        lossSum.value += ls.value


# ================================================================ SGD
class SGD(_Base):
    def __init__(self, maxIter=100, eta0=0.01, alpha0=1e-6, alpha=1e-3, beta=1e-3, loss=None,
                 scheduling=optimal, power=1.0, verbose=1, tol=1e-3, shuffle=True, nCalls=-1, miniBatchSize=1):
        """newSGD (sgd.nim:23-52).  miniBatchSize is this implementation's extra knob: 1 is the reference's
        strictly sequential semantics; >1 is the synchronous-minibatch variant (the deterministic analogue of
        the Hogwild fit(..., maxThreads), DESIGN.md)."""
        self.maxIter, self.eta0, self.alpha0, self.alpha, self.beta = maxIter, eta0, alpha0, alpha, beta
        self.loss = loss if loss is not None else Squared()
        self.scheduling, self.power = scheduling, power
        self.verbose, self.tol, self.shuffle, self.nCalls = verbose, tol, shuffle, nCalls
        self.miniBatchSize = int(miniBatchSize)
        self.it = 1

    def init(self):                            # sgd.nim:55-57
        self.it = 1
        if self.verbose > 0:
            echoHeader(self.maxIter)

    def fit(self, X, y, fm, maxThreads=None, callback=None, perms=None):
        """sgd.nim:261-328 / sgd_ffm.nim:49-106.  fit(..., maxThreads) is the reference's Hogwild variant
        (sgd_multi.nim:40-120, sgd_ffm_multi.nim:31-103: T lock-free threads, every sample sees parameters up
        to ~T updates stale, results nondeterministic); its deterministic device analogue is the synchronous
        minibatch of T samples (nimfm_*_sgd_minibatch_epoch).  maxThreads < 0 means "as many as the machine
        runs at once" there (2 x cores, sgd_multi.nim:13-18) and here (4096 resident rows).  Without
        maxThreads (and miniBatchSize = 1) the device keeps the exact sequential semantics."""
        is_ffm = isinstance(fm, FieldAwareFactorizationMachine)
        fm.init(X)
        y = fm.checkTarget(y)
        lib, ctx = _lib.load(), _lib.ctx()
        X.set_targets(y)
        n = X.nSamples
        h = fm._to_device(X) if is_ffm else fm._to_device(X.nFeatures)
        begin, epoch, end, free = ((lib.nimfm_ffm_sgd_begin, lib.nimfm_ffm_sgd_epoch, lib.nimfm_ffm_sgd_end,
                                    lib.nimfm_ffm_free) if is_ffm else
                                   (lib.nimfm_fm_sgd_begin, lib.nimfm_fm_sgd_epoch, lib.nimfm_fm_sgd_end,
                                    lib.nimfm_fm_free))
        cfg = _lib.SgdCfg(self.loss.kind, self.loss.threshold, self.eta0, self.alpha0, self.alpha, self.beta,
                          _lib.SCHED[self.scheduling], self.power)
        mbs = self.miniBatchSize
        world = 1
        if self.nCalls > 0 and callback is not None:
            raise NotImplementedError("nCalls > 0 (a callback inside the sample loop, sgd.nim:300-305) is not "
                                      "supported: one library call runs a whole epoch; use nCalls <= 0")
        if maxThreads is not None and mbs == 1:
            mbs = 4096 if maxThreads < 0 else max(1, int(maxThreads))
        if mbs == 1 and _dist.world() > 1:
            raise ValueError("per-sample SGD is sequential and does not shard across ranks (replicas only); "
                             "pass miniBatchSize > 1 or fit(..., maxThreads) for the synchronous-minibatch form")
        if mbs > 1:
            if X.windowed:
                raise ValueError("minibatch SGD needs a resident dataset")
            mb_epoch = lib.nimfm_ffm_sgd_minibatch_epoch if is_ffm else lib.nimfm_fm_sgd_minibatch_epoch
            # data parallel (distributed.init_comm): X is this rank's shard, mbs the GLOBAL minibatch; the shares
            # (and the shards) may be uneven -- the library agrees the schedule across ranks
            world = _dist.world()
            local = _dist.local_batch(mbs, _dist.rank(), world)
            if local < 1:
                raise ValueError("miniBatchSize is smaller than the number of ranks")
            begin = end = lambda *_: 0          # parameters stay canonical: no scaling caches to set up / fold in
            epoch = lambda c_, h_, x_, cfg_, it_, idx_, n_, v_, l_: mb_epoch(c_, h_, x_, cfg_, mbs, local, it_, idx_, n_,
                                                                            v_, l_)
        if not fm.warmStart:
            self.init()
        n_glob = _dist.global_shape(X)[0] if world > 1 else n
        rng = self._rng(fm)
        indices = np.arange(n, dtype=np.int64)
        self._converged = False
        self.history = []
        self.epoch_seconds = []     # host wall time of each epoch's single library call (blocking)
        try:
            _lib.check(begin(ctx, h))
            for ep in range(self.maxIter):
                if perms is not None:
                    indices = _lib.i64(perms[ep])
                elif self.shuffle and not X.windowed:      # sgd.nim:297: only a fully cached dataset is shuffled
                    rng.shuffle(indices)
                it = C.c_int64(self.it)
                viol, lossSum = C.c_double(), C.c_double()
                t0 = time.perf_counter()
                if X.windowed:
                    _windowed_epoch(epoch, ctx, h, X, cfg, it, viol, lossSum, 1)
                else:
                    _lib.check(epoch(ctx, h, X.handle(), C.byref(cfg), C.byref(it), _lib.ptr(indices), n,
                                     C.byref(viol), C.byref(lossSum)))
                self.epoch_seconds.append(time.perf_counter() - t0)
                self.it = it.value
                runningLoss = lossSum.value / n_glob           # minibatch form: the loss sum is all-reduced
                self.history.append((viol.value, runningLoss))
                if callback is not None:
                    # finalize + transpose back before the user sees the model (sgd.nim:310-316)
                    _lib.check(end(ctx, h))
                    fm._from_device(h)
                    callback(self, fm)
                elif self.verbose > 0:
                    fm._from_device(h)      # un-finalized, as the reference's verbose line sees it
                if not self._stopping(fm, runningLoss, viol.value, ep):
                    break
            if not self._converged and self.verbose > 0:
                print("Objective did not converge. Increase maxIter.")
            _lib.check(end(ctx, h))
            fm._from_device(h)
        finally:
            free(ctx, h)


def newSGD(maxIter=100, eta0=0.01, alpha0=1e-6, alpha=1e-3, beta=1e-3, loss=None, scheduling=optimal,
           power=1.0, verbose=1, tol=1e-3, shuffle=True, nCalls=-1, miniBatchSize=1):
    return SGD(maxIter, eta0, alpha0, alpha, beta, loss, scheduling, power, verbose, tol, shuffle, nCalls,
               miniBatchSize)


# ================================================================ AdaGrad
class AdaGrad(_Base):
    def __init__(self, maxIter=100, eta0=0.1, alpha0=1e-6, alpha=1e-3, beta=1e-3, loss=None, eps=1e-10,
                 verbose=1, tol=1e-3, shuffle=True, nCalls=-1, miniBatchSize=1):
        """newAdaGrad (adagrad.nim:20-44).  miniBatchSize is this implementation's extra knob: 1 is
        the reference's strictly sequential semantics; >1 is the synchronous-minibatch variant that
        shards over GPUs (DESIGN.md)."""
        self.maxIter, self.eta0, self.alpha0, self.alpha, self.beta = maxIter, eta0, alpha0, alpha, beta
        self.loss = loss if loss is not None else Squared()
        self.eps, self.verbose, self.tol, self.shuffle, self.nCalls = eps, verbose, tol, shuffle, nCalls
        self.miniBatchSize = int(miniBatchSize)
        self.it = 1
        self.g_sum = None
        self.g_norm = None

    def fit(self, X, y, fm, maxThreads=None, callback=None, perms=None):
        """adagrad.nim:137-203 / adagrad_ffm.nim:11-66; fit(..., maxThreads=T) (adagrad_multi.nim:39) runs the
        synchronous minibatch of T samples, see below."""
        is_ffm = isinstance(fm, FieldAwareFactorizationMachine)
        fm.init(X)
        y = fm.checkTarget(y)
        lib, ctx = _lib.load(), _lib.ctx()
        X.set_targets(y)
        n = X.nSamples
        h = fm._to_device(X) if is_ffm else fm._to_device(X.nFeatures)
        init, epoch, fin, free, get_state, set_state = (
            (lib.nimfm_ffm_adagrad_init, lib.nimfm_ffm_adagrad_epoch, lib.nimfm_ffm_adagrad_finalize, lib.nimfm_ffm_free,
             lib.nimfm_ffm_adagrad_get_state, lib.nimfm_ffm_adagrad_set_state) if is_ffm else
            (lib.nimfm_fm_adagrad_init, lib.nimfm_fm_adagrad_epoch, lib.nimfm_fm_adagrad_finalize, lib.nimfm_fm_free,
             lib.nimfm_fm_adagrad_get_state, lib.nimfm_fm_adagrad_set_state))
        # g_sum.P / g_norm.P: the FM solver layout [nOrders, d+nAug, k], the FFM reference layout of ffm.P [nFields, d, k]
        state_shape = ((X.nFields, X.nFeatures, fm.nComponents) if is_ffm else
                       (fm.nOrders, X.nFeatures + fm.nAugments, fm.nComponents))
        # data parallel (distributed.init_comm): X is this rank's shard and miniBatchSize the GLOBAL
        # synchronous minibatch; the library all-reduces the per-minibatch deltas
        world = _dist.world()
        mbs = self.miniBatchSize
        if self.nCalls > 0 and callback is not None:
            raise NotImplementedError("nCalls > 0 (a callback inside the sample loop, adagrad.nim:170-181) is not "
                                      "supported: one library call runs a whole epoch; use nCalls <= 0")
        if maxThreads is not None and mbs == 1:
            # fit(..., maxThreads) is the reference's Hogwild variant (adagrad_multi.nim:39-115: T lock-free
            # threads, every sample sees parameters up to ~T updates stale, results nondeterministic).  Its
            # deterministic device analogue is the synchronous minibatch of T samples; maxThreads < 0 means
            # "as many as the machine runs at once" there (2 x cores, sgd_multi.nim:13-18) and here (4096
            # resident rows).
            mbs = 4096 if maxThreads < 0 else max(1, int(maxThreads))
        local = _dist.local_batch(mbs, _dist.rank(), world)
        if local < 1:
            raise ValueError("miniBatchSize is smaller than the number of ranks")
        if mbs == 1 and world > 1:
            raise ValueError("per-sample AdaGrad is sequential and does not shard across ranks (replicas only); "
                             "pass miniBatchSize > 1 or fit(..., maxThreads) for the synchronous-minibatch form")
        n_glob = _dist.global_shape(X)[0] if world > 1 else n
        cfg = _lib.AdagradCfg(self.loss.kind, self.loss.threshold, self.eta0, self.alpha0, self.alpha,
                              self.beta, self.eps, local)
        if not fm.warmStart:                   # AdaGrad.init, adagrad.nim:47-62
            self.it = 1
        rng = self._rng(fm)
        indices = np.arange(n, dtype=np.int64)
        self._converged = False
        self.history = []
        self.epoch_seconds = []     # host wall time of each epoch's single library call (blocking)
        try:
            _lib.check(init(ctx, h, self.eps, 1))
            if self.it != 1:
                if self.g_sum is None:
                    raise ValueError("warmStart=true but the optimizer has no g_sum / g_norm state.")
                if self.g_sum["P"].shape != state_shape:
                    raise ValueError("warmStart=true but P.shape != g_sum.P.shape.")   # adagrad.nim:57-59
                _lib.check(set_state(
                    ctx, h, _lib.ptr(_lib.f64(self.g_sum["P"])), _lib.ptr(_lib.f64(self.g_norm["P"])),
                    _lib.ptr(_lib.f64(self.g_sum["w"])), _lib.ptr(_lib.f64(self.g_norm["w"])),
                    float(self.g_sum["intercept"]), float(self.g_norm["intercept"])))
            if self.verbose > 0:
                echoHeader(self.maxIter)
            for ep in range(self.maxIter):
                if perms is not None:
                    indices = _lib.i64(perms[ep])
                elif self.shuffle and not X.windowed:      # adagrad.nim:168: only a fully cached dataset is shuffled
                    rng.shuffle(indices)
                it = C.c_int64(self.it)
                viol, lossSum = C.c_double(), C.c_double()
                t0 = time.perf_counter()
                if X.windowed:
                    _windowed_epoch(epoch, ctx, h, X, cfg, it, viol, lossSum, local)
                else:
                    _lib.check(epoch(ctx, h, X.handle(), C.byref(cfg), C.byref(it), _lib.ptr(indices), n,
                                     C.byref(viol), C.byref(lossSum)))
                self.epoch_seconds.append(time.perf_counter() - t0)
                self.it = it.value
                runningLoss = lossSum.value / n_glob           # the loss sum is all-reduced over the shards
                self.history.append((viol.value, runningLoss))
                if callback is not None:
                    _lib.check(fin(ctx, h, C.byref(cfg), self.it))
                    fm._from_device(h)
                    callback(self, fm)
                elif self.verbose > 0:
                    fm._from_device(h)
                if not self._stopping(fm, runningLoss, viol.value, ep):
                    break
            if not self._converged and self.verbose > 0:
                print("Objective did not converge. Increase maxIter.")
            gsP, gnP = np.zeros(state_shape), np.zeros(state_shape)
            gsw, gnw = np.zeros(X.nFeatures), np.zeros(X.nFeatures)
            gsb, gnb = C.c_double(), C.c_double()
            _lib.check(get_state(ctx, h, _lib.ptr(gsP), _lib.ptr(gnP), _lib.ptr(gsw), _lib.ptr(gnw), C.byref(gsb),
                                 C.byref(gnb)))
            self.g_sum = dict(P=gsP, w=gsw, intercept=gsb.value)
            self.g_norm = dict(P=gnP, w=gnw, intercept=gnb.value)
            _lib.check(fin(ctx, h, C.byref(cfg), self.it))     # finalize, adagrad.nim:65-84
            fm._from_device(h)
        finally:
            free(ctx, h)


def newAdaGrad(maxIter=100, eta0=0.1, alpha0=1e-6, alpha=1e-3, beta=1e-3, loss=None, eps=1e-10, verbose=1,
               tol=1e-3, shuffle=True, nCalls=-1, miniBatchSize=1):
    return AdaGrad(maxIter, eta0, alpha0, alpha, beta, loss, eps, verbose, tol, shuffle, nCalls, miniBatchSize)


# ================================================================ PSGD
class PSGD(_Base):
    """Proximal SGD (optimizer/psgd.nim:10-215).  Strictly sequential per sample like SGD; reg: L1 / L21
    (the reference's lazy protocols, reproduced on the device) or SquaredL12 (default; dense step + full
    prox every sample, as in the reference)."""

    def __init__(self, maxIter=100, eta0=0.01, alpha0=1e-6, alpha=1e-3, beta=1e-4, gamma=1e-4, loss=None,
                 reg=None, scheduling=optimal, power=1.0, verbose=1, tol=1e-3, shuffle=True, nCalls=-1):
        self.maxIter, self.eta0, self.alpha0, self.alpha, self.beta, self.gamma = maxIter, eta0, alpha0, alpha, beta, gamma
        self.loss = loss if loss is not None else Squared()
        self.reg = reg if reg is not None else SquaredL12()
        self.scheduling, self.power, self.verbose, self.tol = scheduling, power, verbose, tol
        self.shuffle, self.nCalls = shuffle, nCalls
        self.it = 1

    def fit(self, X, y, sfm, callback=None, perms=None):
        """psgd.nim:76-215 (nCalls > 0, a callback inside the sample loop, is not supported: one library
        call runs a whole epoch)"""
        if not isinstance(X, CSRDataset):
            raise TypeError("PSGD.fit needs a CSRDataset")
        sfm.init(X)
        y = sfm.checkTarget(y)
        lib, ctx = _lib.load(), _lib.ctx()
        X.set_targets(y)
        n = X.nSamples
        h = sfm._to_device(X.nFeatures)
        if not sfm.warmStart:
            self.it = 1                        # :104-105
        cfg = _lib.PsgdCfg(self.loss.kind, self.loss.threshold, self.eta0, self.alpha0, self.alpha, self.beta,
                           self.gamma, self.reg.kind, _lib.SCHED[self.scheduling], self.power)
        rng = self._rng(sfm)
        indices = np.arange(n, dtype=np.int64)
        self.history = []
        self.epoch_seconds = []
        converged = False
        runningLossOld = 0.0                   # :103
        try:
            self.reg.initSGD(sfm.degree, X.nFeatures + sfm.nAugments, sfm.nComponents)   # :111
            _lib.check(lib.nimfm_fm_psgd_begin(ctx, h))
            if self.verbose > 0:
                echoHeader(self.maxIter, viol=False)
            for ep in range(self.maxIter):
                if perms is not None:
                    indices = _lib.i64(perms[ep])
                elif self.shuffle:
                    rng.shuffle(indices)
                itc, ls = C.c_int64(self.it), C.c_double()
                t0 = time.perf_counter()
                _lib.check(lib.nimfm_fm_psgd_epoch(ctx, h, X.handle(), C.byref(cfg), C.byref(itc),
                                                   _lib.ptr(indices), n, C.byref(ls)))
                self.epoch_seconds.append(time.perf_counter() - t0)
                self.it = itc.value
                runningLoss = ls.value / n
                self.history.append(runningLoss)
                if callback is not None and self.nCalls <= 0:      # :181-183 (finalize, then callback)
                    _lib.check(lib.nimfm_fm_psgd_end(ctx, h, C.byref(cfg)))
                    sfm._from_device(h)
                    callback(self, sfm)
                if math.isnan(runningLoss):
                    print("Loss is NaN. Use smaller learning rate.")
                    break
                if abs(runningLoss - runningLossOld) < self.tol:   # :189-192
                    if self.verbose > 0:
                        print("Converged at epoch ", ep, ".")
                    converged = True
                    break
                if self.verbose > 0:                                # :194-198 (stale P, as the reference prints it)
                    sfm._from_device(h)
                    regVal = regularization(sfm.P, sfm.w, sfm.intercept, self.alpha0, self.alpha, self.beta)
                    for order in range(sfm.nOrders):
                        regVal += self.gamma * self.reg.eval(np.asarray(sfm.P[order]).T, sfm.degree - order)
                    echoInfo(ep + 1, self.maxIter, -1, runningLoss, regVal)
                runningLossOld = runningLoss
            if not converged and self.verbose > 0:
                print("Objective did not converge. Increase maxIter.")
            _lib.check(lib.nimfm_fm_psgd_end(ctx, h, C.byref(cfg)))   # finalize, :204
            sfm._from_device(h)
        finally:
            lib.nimfm_fm_free(ctx, h)


def newPSGD(maxIter=100, eta0=0.01, alpha0=1e-6, alpha=1e-3, beta=1e-4, gamma=1e-4, loss=None, reg=None,
            scheduling=optimal, power=1.0, verbose=1, tol=1e-3, shuffle=True, nCalls=-1):
    return PSGD(maxIter, eta0, alpha0, alpha, beta, gamma, loss, reg, scheduling, power, verbose, tol, shuffle, nCalls)


# ================================================================ MBPSGD
class L1:                                      # regularizer/l1.nim
    kind = _lib.REG_L1

    def eval(self, P, degree=2):               # P: one order, solver layout [nFeatures, nComponents]
        return float(np.sum(np.abs(P)))

    def initSGD(self, degree, nFeatures, nComponents):
        pass

    initCD = initSGD                           # l1.nim:44


class SquaredL12:                              # regularizer/squaredl12.nim
    def __init__(self, transpose=True):        # newSquaredL12(transpose=true), :84-87
        self.transpose = bool(transpose)

    @property
    def kind(self):
        return _lib.REG_SQUAREDL12 if self.transpose else _lib.REG_SQUAREDL12_ROWS

    def eval(self, P, degree=2):               # :72-81
        if degree > 2:
            raise ValueError("SquaredL12 supports only degree=2.")
        return float(np.sum(np.sum(np.abs(P), axis=0 if self.transpose else 1) ** 2))

    def initSGD(self, degree, nFeatures, nComponents):   # :103-106
        if degree != 2:
            raise ValueError("SquaredL12 supports only degree=2.")

    initCD = initSGD                           # :90-93


class L21:                                     # regularizer/l21.nim
    kind = _lib.REG_L21

    def eval(self, P, degree=2):               # :17-21
        return float(np.sum(np.sqrt(np.sum(np.asarray(P) ** 2, axis=1))))

    def initSGD(self, degree, nFeatures, nComponents):
        pass


def newL1():
    return L1()


def newSquaredL12(transpose=True):
    return SquaredL12(transpose)


def newL21():
    return L21()


class MBPSGD(_Base):
    def __init__(self, maxIter=100, eta0=0.1, alpha0=1e-6, alpha=1e-3, beta=1e-4, gamma=1e-4, loss=None,
                 reg=None, miniBatchSize=-1, maxIterInner=-1, scheduling=optimal, power=1.0, verbose=1,
                 tol=1e-6, shuffle=True, nCalls=-1):
        self.maxIter, self.eta0, self.alpha0, self.alpha, self.beta, self.gamma = maxIter, eta0, alpha0, alpha, beta, gamma
        self.loss = loss if loss is not None else Squared()
        self.reg = reg if reg is not None else SquaredL12()
        self.miniBatchSize, self.maxIterInner = miniBatchSize, maxIterInner
        self.scheduling, self.power, self.verbose, self.tol, self.shuffle = scheduling, power, verbose, tol, shuffle
        self.it = 0                            # minibatch_psgd.nim:62

    def resolve_sizes(self, X):
        """minibatch_psgd.nim:157-165, on the GLOBAL shape: with a communicator X is this rank's shard and the
        rule sees the sum of the shards, so every rank resolves the same sizes whatever its own share is"""
        n, nnz = _dist.global_shape(X)
        mb = self.miniBatchSize
        if mb <= 0:
            mb = max((X.nFeatures * n) // nnz, 1)
        inner = self.maxIterInner
        if inner <= 0:
            inner = max((n - 1) // mb + 1, 1)
        return mb, inner

    def fit(self, X, y, sfm, callback=None):
        """minibatch_psgd.nim:127-211"""
        sfm.init(X)
        y = sfm.checkTarget(y)
        lib, ctx = _lib.load(), _lib.ctx()
        X.set_targets(y)
        n = X.nSamples
        h = sfm._to_device(X.nFeatures)
        if not sfm.warmStart:
            self.it = 1                        # :151-152
        mb, inner = self.resolve_sizes(X)
        # data parallel (distributed.init_comm): X is this rank's shard, mb the GLOBAL minibatch; every
        # rank feeds its share of each minibatch and the library all-reduces grad P / w / b / loss
        local = _dist.local_batch(mb, _dist.rank(), _dist.world())
        if _dist.world() > 1 and local < 1:
            raise ValueError("miniBatchSize is smaller than the number of ranks")
        # self.reg.initSGD(degree, nFeatures+nAugments, nComponents) (:172): SquaredL12 -- the default --
        # raises for degree != 2 whatever gamma is (squaredl12.nim:103-106)
        self.reg.initSGD(sfm.degree, X.nFeatures + sfm.nAugments, sfm.nComponents)
        cfg = _lib.MbpsgdCfg(self.loss.kind, self.loss.threshold, self.eta0, self.alpha0, self.alpha, self.beta,
                             self.gamma, self.reg.kind, _lib.SCHED[self.scheduling], self.power, mb, inner)
        rng = self._rng(sfm)
        indices = np.arange(n, dtype=np.int64)
        if X.windowed:
            if _dist.world() > 1:
                raise ValueError("a windowed StreamCSRDataset is not sharded across ranks")
            self_shuffle, self.shuffle = self.shuffle, False    # :110-111,169: nCached < nSamples never shuffles
        if self.shuffle:
            rng.shuffle(indices)               # :169-170
        if self.verbose > 0:
            print("Minibatch size: ", mb)
            print("Number of inner iteration: ", inner)
            echoHeader(self.maxIter, viol=False)
        ii = 0
        oldLoss = float("inf")
        converged = False
        self.history = []
        self.epoch_seconds = []     # host wall time of each epoch's single library call (blocking)
        try:
            for ep in range(self.maxIter):
                sample = None
                if self.shuffle:
                    # the cursor + reshuffle-at-wrap logic of epoch() (:102-111), evaluated on the host
                    total = local * inner
                    sample = np.empty(total, dtype=np.int64)
                    filled = 0
                    while filled < total:
                        take = min(total - filled, n - ii)
                        sample[filled:filled + take] = indices[ii:ii + take]
                        filled += take
                        ii += take
                        if ii >= n:
                            ii = 0
                            rng.shuffle(indices)
                itc, iic, rl = C.c_int64(self.it), C.c_int64(ii), C.c_double()
                t0 = time.perf_counter()
                if X.windowed:
                    rl.value, ii = self._windowed_epoch(lib, ctx, h, X, cfg, mb, inner, itc, ii)
                    iic.value = ii
                else:
                    _lib.check(lib.nimfm_fm_mbpsgd_epoch(ctx, h, X.handle(), C.byref(cfg), local, C.byref(itc),
                                                         C.byref(iic), _lib.ptr(sample), C.byref(rl)))
                self.epoch_seconds.append(time.perf_counter() - t0)
                self.it = itc.value
                if not self.shuffle:
                    ii = iic.value
                runningLoss = rl.value
                self.history.append(runningLoss)
                if callback is not None or self.verbose > 0:
                    sfm._from_device(h)        # pgd.finalize, pgd.nim:45-51
                    if callback is not None:
                        callback(self, sfm)
                if math.isnan(runningLoss):
                    print("Loss is NaN. Use smaller learning rate.")
                    break
                if self.verbose > 0:
                    regVal = regularization(sfm.P, sfm.w, sfm.intercept, self.alpha0, self.alpha, self.beta)
                    for order in range(sfm.nOrders):                      # :195-196
                        regVal += self.gamma * self.reg.eval(np.asarray(sfm.P[order]).T, sfm.degree - order)
                    echoInfo(ep + 1, self.maxIter, -1, runningLoss, regVal)
                if abs(oldLoss - runningLoss) < self.tol:
                    if self.verbose > 0:
                        print("Converged at epoch ", ep + 1, ".")
                    converged = True
                    break
                oldLoss = runningLoss
            if not converged and self.verbose > 0:
                print("Objective did not converge. Increase maxIter.")
            sfm._from_device(h)
        finally:
            lib.nimfm_fm_free(ctx, h)
            if X.windowed:
                self.shuffle = self_shuffle

    @staticmethod
    def _windowed_epoch(lib, ctx, h, X, cfg, mb, inner, itc, ii):
        """epoch() (minibatch_psgd.nim:91-124) over a StreamCSRDataset kept on disk: the `inner` minibatches
        are taken from resident windows of whole minibatches starting at the row cursor ii, wrapping to the
        top of the file like the reference's cursor; returns (runningLoss, new cursor)."""
        n = X.nSamples
        total, left = 0.0, inner
        while left > 0:
            # as many whole minibatches as one cache window holds (at least one), without wrapping twice
            b = X.window_end(ii)
            k = max((b - ii) // mb, 1)
            k = min(k, left, max((n - ii + mb - 1) // mb, 1))
            rows = k * mb
            parts = [X.load_rows(ii, min(n, ii + rows))]
            rest = rows - (min(n, ii + rows) - ii)
            while rest > 0:                     # the cursor wrapped (n < mb wraps more than once)
                take = min(rest, n)
                parts.append(X.load_rows(0, take))
                rest -= take
            win = parts[0]
            if len(parts) > 1:
                arr = (C.c_void_p * len(parts))(*[p_.handle() for p_ in parts])
                hv = C.c_void_p()
                _lib.check(lib.nimfm_dataset_vstack(ctx, arr, len(parts), C.byref(hv)))
                from .dataset import _DeviceCSRDataset
                win = _DeviceCSRDataset(hv)
                win.set_targets(np.concatenate([X._y[ii:min(n, ii + rows)]] +
                                               [X._y[:p_.nSamples] for p_ in parts[1:]]))
            try:
                sub = _lib.MbpsgdCfg.from_buffer_copy(cfg)
                sub.maxIterInner = k
                cur, rl = C.c_int64(0), C.c_double()
                _lib.check(lib.nimfm_fm_mbpsgd_epoch(ctx, h, win.handle(), C.byref(sub), mb, C.byref(itc),
                                                     C.byref(cur), None, C.byref(rl)))
                total += rl.value * mb * k
            finally:
                for p_ in parts:
                    p_.free()
                if win is not parts[0]:
                    win.free()
            ii = (ii + rows) % n
            left -= k
        return total / (mb * inner), ii


def newMBPSGD(maxIter=100, eta0=0.1, alpha0=1e-6, alpha=1e-3, beta=1e-4, gamma=1e-4, loss=None, reg=None,
              miniBatchSize=-1, maxIterInner=-1, scheduling=optimal, power=1.0, verbose=1, tol=1e-6,
              shuffle=True, nCalls=-1):
    return MBPSGD(maxIter, eta0, alpha0, alpha, beta, gamma, loss, reg, miniBatchSize, maxIterInner,
                  scheduling, power, verbose, tol, shuffle, nCalls)
