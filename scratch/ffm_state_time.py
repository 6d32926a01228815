"""Host time of nimfm_ffm_adagrad_get_state / _set_state at the C5 size (39 fields, 10^6 features, k = 8: g_sum.P and
g_norm.P are 2.5 GB each), the copies AdaGrad.fit makes at the end of an FFM fit and at the start of a warm one.
get_state writes into fresh np.zeros arrays, as fit does.  Prints the card and its power limit with the numbers."""
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from nimfm_b200 import _lib  # noqa: E402


def main():
    nF, d, k = 39, 1_000_000, 8
    lib, ctx = _lib.load(), _lib.ctx()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()[0]
    h = C.c_void_p()
    _lib.check(lib.nimfm_ffm_create(ctx, k, nF, d, 1, 1, C.byref(h)))
    try:
        _lib.check(lib.nimfm_ffm_adagrad_init(ctx, h, 1e-10, 1))
        gets, sets = [], []
        for _ in range(3):
            st = [np.zeros((nF, d, k)), np.zeros((nF, d, k)), np.zeros(d), np.zeros(d)]
            gsb, gnb = C.c_double(), C.c_double()
            t0 = time.perf_counter()
            _lib.check(lib.nimfm_ffm_adagrad_get_state(ctx, h, *[_lib.ptr(a) for a in st], C.byref(gsb),
                                                       C.byref(gnb)))
            gets.append(time.perf_counter() - t0)
            assert st[1].flat[12345] == 1e-10
            t0 = time.perf_counter()
            _lib.check(lib.nimfm_ffm_adagrad_set_state(ctx, h, *[_lib.ptr(a) for a in st], gsb.value, gnb.value))
            sets.append(time.perf_counter() - t0)
            del st
    finally:
        lib.nimfm_ffm_free(ctx, h)
    out = dict(card=card, nFields=nF, nFeatures=d, k=k, bytes_per_array=nF * d * k * 8, get_state_s=gets,
               set_state_s=sets)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
