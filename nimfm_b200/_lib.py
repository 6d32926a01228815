"""ctypes binding of libnimfm_cuda.so -- the same symbols nimfm's Nim modules would bind with
{.importc, dynlib.} (see nim/nimfm_cuda.nim and INTEGRATION.md).

There is no CPU fallback: if the shared library is missing or no CUDA device is present every
entry point raises (NimfmCudaError), it never silently computes on the host.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libnimfm_cuda.so")

c_i32, c_i64, c_dbl = C.c_int32, C.c_int64, C.c_double
PD, PI64, VP = C.POINTER(C.c_double), C.POINTER(C.c_int64), C.c_void_p

LOSS_SQUARED, LOSS_SQUARED_HINGE, LOSS_LOGISTIC, LOSS_HUBER = 0, 1, 2, 3
SCHED = {"constant": 0, "optimal": 1, "invscaling": 2, "pegasos": 3}
REG_IDENTITY, REG_L1, REG_SQUAREDL12, REG_SQUAREDL12_ROWS, REG_L21 = 0, 1, 2, 3, 4
DS_CSR, DS_CSC, DS_CSR_FIELD = 0, 1, 2


class NimfmCudaError(RuntimeError):
    pass


class MbpsgdCfg(C.Structure):
    _fields_ = [("loss", c_i32), ("huberThreshold", c_dbl), ("eta0", c_dbl), ("alpha0", c_dbl),
                ("alpha", c_dbl), ("beta", c_dbl), ("gamma", c_dbl), ("reg", c_i32),
                ("scheduling", c_i32), ("power", c_dbl), ("miniBatchSize", c_i64),
                ("maxIterInner", c_i64)]


class AdagradCfg(C.Structure):
    _fields_ = [("loss", c_i32), ("huberThreshold", c_dbl), ("eta0", c_dbl), ("alpha0", c_dbl),
                ("alpha", c_dbl), ("beta", c_dbl), ("eps", c_dbl), ("miniBatchSize", c_i64)]


class SgdCfg(C.Structure):
    _fields_ = [("loss", c_i32), ("huberThreshold", c_dbl), ("eta0", c_dbl), ("alpha0", c_dbl),
                ("alpha", c_dbl), ("beta", c_dbl), ("scheduling", c_i32), ("power", c_dbl)]


class CdCfg(C.Structure):
    _fields_ = [("loss", c_i32), ("huberThreshold", c_dbl), ("alpha0", c_dbl), ("alpha", c_dbl),
                ("beta", c_dbl)]


class PsgdCfg(C.Structure):
    _fields_ = [("loss", c_i32), ("huberThreshold", c_dbl), ("eta0", c_dbl), ("alpha0", c_dbl),
                ("alpha", c_dbl), ("beta", c_dbl), ("gamma", c_dbl), ("reg", c_i32),
                ("scheduling", c_i32), ("power", c_dbl)]


class PcdCfg(C.Structure):
    _fields_ = [("loss", c_i32), ("huberThreshold", c_dbl), ("alpha0", c_dbl), ("alpha", c_dbl),
                ("beta", c_dbl), ("gamma", c_dbl), ("reg", c_i32)]


# every symbol include/nimfm_cuda.h declares: name -> (restype, argtypes)
PVP = C.POINTER(C.c_void_p)
SYMBOLS = {
    "nimfm_ctx_create": (c_i32, [c_i32, PVP]),
    "nimfm_ctx_destroy": (c_i32, [VP]),
    "nimfm_last_error": (C.c_char_p, [VP]),
    "nimfm_version": (c_i32, []),
    "nimfm_launch_count": (c_i64, [VP]),
    "nimfm_stream_stats": (c_i32, [VP, VP, VP, VP]),
    "nimfm_mem_info": (c_i32, [VP, VP, VP]),
    "nimfm_host_register": (c_i32, [VP, VP, c_i64]),
    "nimfm_host_unregister": (c_i32, [VP, VP]),
    "nimfm_stream_open": (c_i32, [VP, C.c_char_p, C.c_char_p, PVP]),
    "nimfm_stream_info": (c_i32, [VP, VP, VP, VP, VP, VP, VP]),
    "nimfm_stream_window_end": (c_i64, [VP, c_i64, c_i64]),
    "nimfm_stream_load_window": (c_i32, [VP, VP, c_i64, c_i64, PVP]),
    "nimfm_stream_close": (c_i32, [VP]),
    "nimfm_comm_unique_id": (c_i32, [VP]),
    "nimfm_comm_init": (c_i32, [VP, c_i32, c_i32, VP]),
    "nimfm_comm_size": (c_i32, [VP]),
    "nimfm_comm_allgather_i64": (c_i32, [VP, VP, c_i32, VP]),
    "nimfm_csr_upload": (c_i32, [VP, c_i64, c_i64, VP, VP, VP, VP, c_i64, c_i64, c_i64, PVP]),
    "nimfm_csc_upload": (c_i32, [VP, c_i64, c_i64, VP, VP, VP, PVP]),
    "nimfm_dataset_transpose": (c_i32, [VP, VP, PVP]),
    "nimfm_dataset_take_rows": (c_i32, [VP, VP, VP, c_i64, PVP]),
    "nimfm_dataset_slice_rows": (c_i32, [VP, VP, c_i64, c_i64, PVP]),
    "nimfm_dataset_vstack": (c_i32, [VP, PVP, c_i32, PVP]),
    "nimfm_dataset_set_targets": (c_i32, [VP, VP, VP]),
    "nimfm_dataset_info": (c_i32, [VP, PI64, PI64, PI64, C.POINTER(c_i32), PI64, PI64]),
    "nimfm_dataset_download": (c_i32, [VP, VP, VP, VP, VP, VP]),
    "nimfm_dataset_free": (c_i32, [VP, VP]),
    "nimfm_load_svmlight": (c_i32, [VP, C.c_char_p, c_i64, c_i32, PVP]),
    "nimfm_load_ffm": (c_i32, [VP, C.c_char_p, c_i64, c_i64, PVP]),
    "nimfm_load_user_item_rating": (c_i32, [VP, C.c_char_p, c_i32, PVP]),
    "nimfm_load_stream": (c_i32, [VP, C.c_char_p, C.c_char_p, PVP]),
    "nimfm_dataset_get_targets": (c_i32, [VP, VP, VP]),
    "nimfm_fm_create": (c_i32, [VP, c_i32, c_i32, c_i32, c_i32, c_i64, c_i32, c_i32, PVP]),
    "nimfm_fm_set_params": (c_i32, [VP, VP, VP, VP, c_dbl, VP]),
    "nimfm_fm_get_params": (c_i32, [VP, VP, VP, VP, PD]),
    "nimfm_fm_free": (c_i32, [VP, VP]),
    "nimfm_fm_decision_function": (c_i32, [VP, VP, VP, VP]),
    "nimfm_fm_loss_grad": (c_i32, [VP, VP, VP, c_i32, c_dbl, c_i64, c_i64, VP, c_i64, c_i32, c_i32, PD]),
    "nimfm_fm_loss_grad_host": (c_i32, [VP, VP, c_i64, c_i64, VP, VP, VP, VP, c_i32, c_dbl, c_i64, c_i64, c_i32,
                                        c_i32, PD]),
    "nimfm_fm_decision_function_host": (c_i32, [VP, VP, c_i64, c_i64, VP, VP, VP, c_i64, VP]),
    "nimfm_fm_get_grads": (c_i32, [VP, VP, VP, VP, PD]),
    "nimfm_fm_mbpsgd_epoch": (c_i32, [VP, VP, VP, C.POINTER(MbpsgdCfg), c_i64, PI64, PI64, VP, PD]),
    "nimfm_fm_adagrad_init": (c_i32, [VP, VP, c_dbl, c_i32]),
    "nimfm_fm_adagrad_epoch": (c_i32, [VP, VP, VP, C.POINTER(AdagradCfg), PI64, VP, c_i64, PD, PD]),
    "nimfm_fm_adagrad_finalize": (c_i32, [VP, VP, C.POINTER(AdagradCfg), c_i64]),
    "nimfm_fm_adagrad_get_state": (c_i32, [VP, VP, VP, VP, VP, VP, PD, PD]),
    "nimfm_fm_adagrad_set_state": (c_i32, [VP, VP, VP, VP, VP, VP, c_dbl, c_dbl]),
    "nimfm_fm_sgd_begin": (c_i32, [VP, VP]),
    "nimfm_fm_sgd_epoch": (c_i32, [VP, VP, VP, C.POINTER(SgdCfg), PI64, VP, c_i64, PD, PD]),
    "nimfm_fm_sgd_end": (c_i32, [VP, VP]),
    "nimfm_fm_psgd_begin": (c_i32, [VP, VP]),
    "nimfm_fm_psgd_epoch": (c_i32, [VP, VP, VP, C.POINTER(PsgdCfg), PI64, VP, c_i64, PD]),
    "nimfm_fm_psgd_end": (c_i32, [VP, VP, C.POINTER(PsgdCfg)]),
    "nimfm_fm_cd_begin": (c_i32, [VP, VP, VP, C.POINTER(CdCfg)]),
    "nimfm_fm_cd_epoch": (c_i32, [VP, VP, VP, C.POINTER(CdCfg), PD, PD, PD]),
    "nimfm_fm_pcd_epoch": (c_i32, [VP, VP, VP, C.POINTER(PcdCfg), PD, PD, PD]),
    "nimfm_fm_cd_get_ypred": (c_i32, [VP, VP, VP]),
    "nimfm_fm_cd_end": (c_i32, [VP, VP]),
    "nimfm_ffm_create": (c_i32, [VP, c_i32, c_i64, c_i64, c_i32, c_i32, PVP]),
    "nimfm_ffm_set_params": (c_i32, [VP, VP, VP, VP, c_dbl]),
    "nimfm_ffm_get_params": (c_i32, [VP, VP, VP, VP, PD]),
    "nimfm_ffm_free": (c_i32, [VP, VP]),
    "nimfm_ffm_decision_function": (c_i32, [VP, VP, VP, VP]),
    "nimfm_ffm_loss_grad": (c_i32, [VP, VP, VP, c_i32, c_dbl, c_i64, c_i64, VP, c_i64, c_i32, c_i32, PD]),
    "nimfm_ffm_get_grads": (c_i32, [VP, VP, VP, VP, PD]),
    "nimfm_ffm_adagrad_init": (c_i32, [VP, VP, c_dbl, c_i32]),
    "nimfm_ffm_adagrad_epoch": (c_i32, [VP, VP, VP, C.POINTER(AdagradCfg), PI64, VP, c_i64, PD, PD]),
    "nimfm_ffm_adagrad_finalize": (c_i32, [VP, VP, C.POINTER(AdagradCfg), c_i64]),
    "nimfm_ffm_adagrad_get_state": (c_i32, [VP, VP, VP, VP, VP, VP, PD, PD]),
    "nimfm_ffm_adagrad_set_state": (c_i32, [VP, VP, VP, VP, VP, VP, c_dbl, c_dbl]),
    "nimfm_ffm_sgd_begin": (c_i32, [VP, VP]),
    "nimfm_ffm_sgd_epoch": (c_i32, [VP, VP, VP, C.POINTER(SgdCfg), PI64, VP, c_i64, PD, PD]),
    "nimfm_fm_sgd_minibatch_epoch": (c_i32, [VP, VP, VP, C.POINTER(SgdCfg), c_i64, c_i64, PI64, VP, c_i64, PD, PD]),
    "nimfm_ffm_sgd_minibatch_epoch": (c_i32, [VP, VP, VP, C.POINTER(SgdCfg), c_i64, c_i64, PI64, VP, c_i64, PD, PD]),
    "nimfm_ffm_sgd_end": (c_i32, [VP, VP]),
    "nimfm_fm_time_loss_grad": (c_i32, [VP, VP, VP, c_i32, c_i64, c_i64, c_i32, c_i32, C.POINTER(C.c_float)]),
    "nimfm_ffm_time_loss_grad": (c_i32, [VP, VP, VP, c_i32, c_i64, c_i64, c_i32, c_i32, C.POINTER(C.c_float)]),
    "nimfm_timer_start": (c_i32, [VP]),
    "nimfm_timer_stop": (c_i32, [VP, C.POINTER(C.c_float)]),
    "nimfm_fm_grad_device_ptr": (c_i32, [VP, PVP, PI64]),
}

_lib = None
_ctx = None


def load():
    """dlopen the in-tree library and declare every prototype.  Raises if it is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise NimfmCudaError(
                f"{SO_PATH} is not built (run `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C nimfm_b200/csrc`); nimfm_b200 has no CPU fallback")
        lib = C.CDLL(SO_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def ctx(device=None):
    """The process-wide device context (one process per GPU)."""
    global _ctx
    if _ctx is None:
        lib = load()
        if device is None:
            device = int(os.environ.get("LOCAL_RANK", "0"))
        h = C.c_void_p()
        rc = lib.nimfm_ctx_create(device, C.byref(h))
        if rc != 0:
            raise NimfmCudaError(f"nimfm_ctx_create failed ({rc}): "
                                 f"{lib.nimfm_last_error(None).decode()}")
        _ctx = h
    return _ctx


def destroy_ctx():
    global _ctx
    if _ctx is not None:
        load().nimfm_ctx_destroy(_ctx)
        _ctx = None


def check(rc):
    if rc != 0:
        msg = load().nimfm_last_error(_ctx).decode() if _ctx is not None else "?"
        exc = ValueError if rc == -1 else NimfmCudaError
        raise exc(f"libnimfm_cuda error {rc}: {msg}")


def launch_count():
    return int(load().nimfm_launch_count(ctx()))


def ptr(a):
    """void* of a C-contiguous numpy array (None -> NULL)."""
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)
