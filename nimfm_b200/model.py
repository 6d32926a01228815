"""Host-side mirror of nimfm's model objects (model/factorization_machine.nim:11-139,
model/field_aware_factorization_machine.nim:6-92, model/fm_base.nim:18-47).

Public fields keep the reference's names and layouts (fm.P is [nOrders, nComponents,
nFeatures+nAugments], ffm.P is [nFields, nFeatures, nComponents]; tests and users read/write them
directly, e.g. tests/test_cd.nim:33-34).  All arithmetic runs in libnimfm_cuda.so.
"""
import ctypes as C

import numpy as np

from . import _lib
from .dataset import BaseDataset, CSCDataset

regression, classification = "r", "c"       # fm_base.nim:5-8 TaskKind
explicit, augment, none = "explicit", "augment", "none"   # factorization_machine.nim:5-9


class NotFittedError(Exception):             # fm_base.nim:10
    pass


class _FMBase:
    """fm_base.nim:13-47"""

    def checkInitialized(self):
        if not self.isInitialized:
            raise NotFittedError("Factorization machines is not fitted.")

    def predict(self, X):
        return np.sign(self.decisionFunction(X)).astype(np.int64)

    def predictProba(self, X):
        return 1.0 / (1.0 + np.exp(-self.decisionFunction(X)))     # utils.nim:33 expit

    def checkTarget(self, y):
        y = np.asarray(y, dtype=np.float64)
        return np.sign(y) if self.task == classification else y.copy()

    def score(self, X, y):
        yPred = self.decisionFunction(X)
        y = np.asarray(y, dtype=np.float64)
        if self.task == regression:
            return float(np.sqrt(np.mean((y - yPred) ** 2)))       # metrics.nim rmse
        return float(np.mean(np.sign(y) == np.sign(yPred)))        # metrics.nim accuracy


class FactorizationMachine(_FMBase):
    def __init__(self, task, degree=2, nComponents=30, fitLower=explicit, fitIntercept=True,
                 fitLinear=True, warmStart=False, randomState=1, scale=0.01):
        if degree < 1:
            raise ValueError("degree < 1.")
        if nComponents < 1:
            raise ValueError("nComponents < 1.")
        self.task, self.degree, self.nComponents, self.fitLower = task, int(degree), int(nComponents), fitLower
        self.fitIntercept, self.fitLinear, self.warmStart = bool(fitIntercept), bool(fitLinear), bool(warmStart)
        self.randomState, self.scale = randomState, float(scale)
        self.isInitialized = False
        self.lams = np.ones(self.nComponents)
        self.P, self.w, self.intercept = None, None, 0.0

    @property
    def nAugments(self):                       # factorization_machine.nim:81-86
        if self.fitLower == augment:
            return self.degree - 2 if self.fitLinear else self.degree - 1
        return 0

    @property
    def nOrders(self):                         # factorization_machine.nim:89-97
        if self.degree == 1:
            return 0
        return self.degree - 1 if self.fitLower == explicit else 1

    def _check_augments(self):
        # degree 1 with fitLower=augment and fitLinear=true: the reference's formula gives degree - 2 = -1 dummy
        # features, and what it does with them is not pinned down -- refused rather than guessed
        if self.nAugments < 0:
            raise ValueError(f"nAugments = {self.nAugments} < 0: fitLower=augment with fitLinear=true adds degree - 2 "
                             f"dummy features, which is negative at degree {self.degree}.")

    def init(self, X, force=False):            # factorization_machine.nim:125-139
        self._check_augments()
        if force or not (self.warmStart and self.isInitialized):
            rng = np.random.default_rng(self.randomState)   # Nim's RNG stream is unpinned (SURVEY App. B)
            d = X.nFeatures
            self.w = np.zeros(d)
            self.P = rng.standard_normal((self.nOrders, self.nComponents, d + self.nAugments)) * self.scale
            self.intercept = 0.0
        self.isInitialized = True

    # ---- device twin
    def _to_device(self, nFeatures):
        self._check_augments()
        P = _lib.f64(self.P)
        if P.ndim != 3 or P.shape[0] != self.nOrders or P.shape[1] != self.nComponents:
            raise ValueError("fm.P has the wrong shape")
        if nFeatures + self.nAugments != P.shape[2]:
            raise ValueError("Invalid nFeatures.")         # factorization_machine.nim:114-115
        lib = _lib.load()
        h = C.c_void_p()
        _lib.check(lib.nimfm_fm_create(_lib.ctx(), self.degree, self.nComponents, self.nOrders,
                                       self.nAugments, nFeatures, int(self.fitLinear),
                                       int(self.fitIntercept), C.byref(h)))
        w = _lib.f64(self.w)
        lams = _lib.f64(self.lams)
        _lib.check(lib.nimfm_fm_set_params(_lib.ctx(), h, _lib.ptr(P), _lib.ptr(w), float(self.intercept),
                                           _lib.ptr(lams)))
        return h

    def _from_device(self, h):
        P = np.zeros_like(_lib.f64(self.P))
        w = np.zeros_like(_lib.f64(self.w))
        b = C.c_double()
        _lib.check(_lib.load().nimfm_fm_get_params(_lib.ctx(), h, _lib.ptr(P), _lib.ptr(w), C.byref(b)))
        self.P, self.w, self.intercept = P, w, b.value

    def decisionFunction(self, X):             # factorization_machine.nim:100-122
        self.checkInitialized()
        if not isinstance(X, BaseDataset):
            raise TypeError("X must be a CSRDataset or CSCDataset")
        h = self._to_device(X.nFeatures)
        try:
            out = np.zeros(X.nSamples)
            lib = _lib.load()
            if X.windowed:
                # a stream file kept on disk: one resident window of rows after another
                for a, b, win in X.windows():
                    _lib.check(lib.nimfm_fm_decision_function(_lib.ctx(), h, win.handle(), _lib.ptr(out[a:b])))
            elif X._handle is None and not isinstance(X, CSCDataset):
                # no device twin yet: stream the host CSR through the row kernel (copy of chunk c+1
                # overlaps the kernel of chunk c) instead of uploading a dataset first
                _lib.check(lib.nimfm_fm_decision_function_host(
                    _lib.ctx(), h, X.nSamples, X.nFeatures, _lib.ptr(X.data), _lib.ptr(X.indices),
                    _lib.ptr(X.indptr), 0, _lib.ptr(out)))
            else:
                _lib.check(lib.nimfm_fm_decision_function(_lib.ctx(), h, X.handle(), _lib.ptr(out)))
        finally:
            _lib.load().nimfm_fm_free(_lib.ctx(), h)
        return out


    def dump(self, fname):                     # factorization_machine.nim:142-165 (same text layout)
        self.checkInitialized()
        P = _lib.f64(self.P)
        with open(fname, "w") as f:
            f.write(f"task: {self.task}\n")
            f.write(f"nFeatures: {P.shape[2] - self.nAugments}\n")
            f.write(f"degree: {self.degree}\n")
            f.write(f"nComponents: {self.nComponents}\n")
            f.write(f"fitLower: {self.fitLower}\n")
            f.write(f"fitIntercept: {_nim_bool(self.fitIntercept)}\n")
            f.write(f"fitLinear: {_nim_bool(self.fitLinear)}\n")
            f.write(f"randomState: {int(self.randomState)}\n")
            f.write(f"scale: {_nim_float(self.scale)}\n")
            f.write("lams:\n")
            f.write(_join(self.lams) + "\n")
            for order in range(P.shape[0]):
                f.write(f"P[{order}]:\n")
                for s in range(self.nComponents):
                    f.write(_join(P[order, s]) + "\n")
            f.write("w:\n")
            f.write(_join(self.w) + "\n")
            f.write(f"intercept: {_nim_float(self.intercept)}\n")

    @classmethod
    def load(cls, fname, warmStart=False):     # factorization_machine.nim:168-220
        with open(fname) as f:
            val = lambda: f.readline().rstrip("\n").split(" ")[1]
            task = val()
            nFeatures, degree, nComponents = int(val()), int(val()), int(val())
            fitLower = val()
            fitIntercept, fitLinear = _parse_bool(val()), _parse_bool(val())
            randomState, scale = int(val()), float(val())
            fm = cls(task, degree, nComponents, fitLower, fitIntercept, fitLinear, warmStart, randomState, scale)
            f.readline()                                               # "lams:"
            fm.lams = _parse_row(f.readline(), nComponents)
            dd = nFeatures + fm.nAugments
            fm.P = np.zeros((fm.nOrders, nComponents, dd))
            for order in range(fm.nOrders):
                f.readline()                                           # "P[order]:"
                for s in range(nComponents):
                    fm.P[order, s] = _parse_row(f.readline(), dd)
            f.readline()                                               # "w:"
            fm.w = _parse_row(f.readline(), nFeatures)
            fm.intercept = float(f.readline().rstrip("\n").split(" ")[1])
        fm.isInitialized = True
        return fm


def _nim_bool(b):
    return "true" if b else "false"


def _parse_bool(s):                            # strutils.parseBool
    t = s.strip().lower()
    if t in ("y", "yes", "true", "1", "on"):
        return True
    if t in ("n", "no", "false", "0", "off"):
        return False
    raise ValueError(f"cannot interpret as a bool: {s}")


def _nim_float(x):
    """Shortest round-trip decimal, as Nim's `$` (float64)."""
    return repr(float(x))


def _join(v):
    return " ".join(_nim_float(x) for x in np.asarray(v, dtype=np.float64).ravel())


def _parse_row(line, count):
    vals = np.array(line.split(), dtype=np.float64)
    if len(vals) < count:
        raise ValueError(f"expected {count} values, found {len(vals)}")
    return vals[:count].copy()


def newFactorizationMachine(task, degree=2, nComponents=30, fitLower=explicit, fitIntercept=True,
                            fitLinear=True, warmStart=False, randomState=1, scale=0.01):
    """factorization_machine.nim:43-78"""
    return FactorizationMachine(task, degree, nComponents, fitLower, fitIntercept, fitLinear, warmStart,
                                randomState, scale)


class FieldAwareFactorizationMachine(_FMBase):
    def __init__(self, task, nComponents=10, fitIntercept=True, fitLinear=True, warmStart=False,
                 randomState=1, scale=0.01):
        if nComponents < 1:
            raise ValueError("nComponents < 1.")
        self.task, self.nComponents = task, int(nComponents)
        self.fitIntercept, self.fitLinear, self.warmStart = bool(fitIntercept), bool(fitLinear), bool(warmStart)
        self.randomState, self.scale = randomState, float(scale)
        self.isInitialized = False
        self.P, self.w, self.intercept = None, None, 0.0

    nAugments = 0                              # field_aware_factorization_machine.nim:49

    def init(self, X, force=False):            # :79-92
        if force or not (self.warmStart and self.isInitialized):
            rng = np.random.default_rng(self.randomState)
            self.w = np.zeros(X.nFeatures)
            self.P = rng.standard_normal((X.nFields, X.nFeatures, self.nComponents)) * self.scale
            self.intercept = 0.0
        self.isInitialized = True

    def _to_device(self, X):
        P = _lib.f64(self.P)
        if P.ndim != 3 or X.nFeatures != P.shape[1]:
            raise ValueError("Invalid nFeatures.")     # :60-61
        if X.nFields != P.shape[0]:
            raise ValueError("Invalid nFields.")       # :62-64
        lib = _lib.load()
        h = C.c_void_p()
        _lib.check(lib.nimfm_ffm_create(_lib.ctx(), self.nComponents, P.shape[0], P.shape[1],
                                        int(self.fitLinear), int(self.fitIntercept), C.byref(h)))
        _lib.check(lib.nimfm_ffm_set_params(_lib.ctx(), h, _lib.ptr(P), _lib.ptr(_lib.f64(self.w)),
                                            float(self.intercept)))
        return h

    def _from_device(self, h):
        P = np.zeros_like(_lib.f64(self.P))
        w = np.zeros_like(_lib.f64(self.w))
        b = C.c_double()
        _lib.check(_lib.load().nimfm_ffm_get_params(_lib.ctx(), h, _lib.ptr(P), _lib.ptr(w), C.byref(b)))
        self.P, self.w, self.intercept = P, w, b.value

    def decisionFunction(self, X):             # :52-76
        self.checkInitialized()
        h = self._to_device(X)
        try:
            out = np.zeros(X.nSamples)
            if X.windowed:      # a field stream file kept on disk: one resident window of rows after another
                for a, b, win in X.windows():
                    _lib.check(_lib.load().nimfm_ffm_decision_function(_lib.ctx(), h, win.handle(), _lib.ptr(out[a:b])))
            else:
                _lib.check(_lib.load().nimfm_ffm_decision_function(_lib.ctx(), h, X.handle(), _lib.ptr(out)))
        finally:
            _lib.load().nimfm_ffm_free(_lib.ctx(), h)
        return out


    def dump(self, fname):                     # field_aware_factorization_machine.nim:95-115
        self.checkInitialized()
        P = _lib.f64(self.P)
        with open(fname, "w") as f:
            f.write(f"task: {self.task}\n")
            f.write(f"nFields: {P.shape[0]}\n")
            f.write(f"nFeatures: {P.shape[1]}\n")
            f.write(f"nComponents: {self.nComponents}\n")
            f.write(f"fitIntercept: {_nim_bool(self.fitIntercept)}\n")
            f.write(f"fitLinear: {_nim_bool(self.fitLinear)}\n")
            f.write(f"randomState: {int(self.randomState)}\n")
            f.write(f"scale: {_nim_float(self.scale)}\n")
            for field in range(P.shape[0]):
                f.write(f"P[{field}]:\n")
                for j in range(P.shape[1]):
                    f.write(_join(P[field, j]) + "\n")
            f.write("w:\n")
            f.write(_join(self.w) + "\n")
            f.write(f"intercept: {_nim_float(self.intercept)}\n")

    @classmethod
    def load(cls, fname, warmStart=False):     # field_aware_factorization_machine.nim:118-158
        with open(fname) as f:
            val = lambda: f.readline().rstrip("\n").split(" ")[1]
            task = val()
            nFields, nFeatures, nComponents = int(val()), int(val()), int(val())
            fitIntercept, fitLinear = _parse_bool(val()), _parse_bool(val())
            randomState, scale = int(val()), float(val())
            ffm = cls(task, nComponents, fitIntercept, fitLinear, warmStart, randomState, scale)
            ffm.P = np.zeros((nFields, nFeatures, nComponents))
            for field in range(nFields):
                f.readline()
                for j in range(nFeatures):
                    ffm.P[field, j] = _parse_row(f.readline(), nComponents)
            f.readline()
            ffm.w = _parse_row(f.readline(), nFeatures)
            ffm.intercept = float(f.readline().rstrip("\n").split(" ")[1])
        ffm.isInitialized = True
        return ffm


def newFieldAwareFactorizationMachine(task, nComponents=10, fitIntercept=True, fitLinear=True,
                                      warmStart=False, randomState=1, scale=0.01):
    """field_aware_factorization_machine.nim:24-46"""
    return FieldAwareFactorizationMachine(task, nComponents, fitIntercept, fitLinear, warmStart,
                                          randomState, scale)
