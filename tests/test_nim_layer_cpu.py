"""The Nim host layer (nim/*.nim) cannot be compiled here (no Nim toolchain), so it is held to what CAN be checked:
every `fit` / `decisionFunction` it exports has, character for character after whitespace normalisation, the
signature of the reference proc it replaces (tests/golden/nim_signatures.json, extracted from the reference by
tests/golden/make_nim_signatures.py: cd.nim:110-112, minibatch_psgd.nim:127-129, adagrad.nim:137-139, sgd.nim:261-263,
the *_multi / *_ffm twins, factorization_machine.nim:100, field_aware_factorization_machine.nim:52-53); every
reference signature in scope is covered; and every library symbol the layer calls is declared by the binding file
and by include/nimfm_cuda.h."""
import glob
import importlib.util
import json
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NIM = os.path.join(ROOT, "nim")


def _extractor():
    spec = importlib.util.spec_from_file_location("make_nim_signatures",
                                                  os.path.join(ROOT, "tests", "golden", "make_nim_signatures.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_fit_signatures_equal_the_reference():
    mod = _extractor()
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "nim_signatures.json")))
    want = [s for sigs in golden.values() for s in sigs]
    assert len(want) == 12 and len(set(want)) == 12
    ours = []
    for f in sorted(glob.glob(os.path.join(NIM, "*.nim"))):
        ours += mod.signatures(open(f).read())
    assert sorted(ours) == sorted(want), set(ours) ^ set(want)


def test_layer_calls_only_bound_symbols():
    bound = set(re.findall(r"^proc (nimfm_\w+)\*", open(os.path.join(NIM, "nimfm_cuda.nim")).read(), flags=re.M))
    header = set(re.findall(r"\b(nimfm_\w+)\s*\(", open(os.path.join(ROOT, "include", "nimfm_cuda.h")).read()))
    used = set()
    for f in glob.glob(os.path.join(NIM, "*.nim")):
        if not f.endswith("nimfm_cuda.nim"):
            used |= set(re.findall(r"\b(nimfm_\w+)\(", open(f).read()))
    assert used and used <= bound, used - bound
    assert used <= header, used - header


def test_layer_keeps_the_reference_control_flow():
    """the pieces of fit() that stay on the host are all there: header / info lines, callback, tol test, NaN check,
    warm start, shuffling -- one grep per reference line the replacement must keep"""
    cd = open(os.path.join(NIM, "fit_cd.nim")).read()
    for needle in ("fm.init(X)", "fm.checkTarget(y)", "echoHeader(self.maxIter)", "callback(self, fm)",
                   "if viol < self.tol:", 'echo("Converged at iteration ", it+1, ".")',
                   'echo("Objective did not converge. Increase maxIter.")'):
        assert needle in cd, needle
    mb = open(os.path.join(NIM, "fit_mbpsgd.nim")).read()
    for needle in ("miniBatchSize = (nFeatures * nSamples) div X.nnz", "maxIterInner = (nSamples-1) div miniBatchSize + 1",
                   "self.reg.initSGD(degree, nFeatures+nAugments, nComponents)", "runningLoss.classify == fcNan",
                   "if abs(oldLossVal - runningLoss) < self.tol:", "if not sfm.warmstart:", "shuffle(indices)"):
        assert needle in mb, needle
    for name in ("fit_sgd.nim", "fit_adagrad.nim", "fit_ffm.nim"):
        s = open(os.path.join(NIM, name)).read()
        for needle in ("if X.nCached == X.nSamples and self.shuffle: shuffle(indices)", "stoppingCriterion(",
                       "lossSum / float(nSamples)", "callback(self, "):
            assert needle in s, (name, needle)
