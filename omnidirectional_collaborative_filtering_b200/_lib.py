"""ctypes binding of `csrc/libocf_b200.so` (C ABI: `include/ocf.h`).

The library is the product; there is no CPU fallback. `lib()` raises `OcfError` when the
shared object is missing (run `python -c "import __graft_entry__ as g; g.build()"` or
`make -C omnidirectional_collaborative_filtering_b200/csrc`), and every compute call raises
when no CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(HERE, "csrc", "libocf_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(HERE), "include", "ocf.h")


class OcfError(RuntimeError):
    pass


class ModelConfig(C.Structure):
    _fields_ = [
        ("n_cols", C.c_int32), ("n_cols_total", C.c_int32), ("n_layers", C.c_int32),
        ("widths", C.c_int32 * 8), ("aux", C.c_int32), ("activation", C.c_int32),
        ("loss", C.c_int32), ("l2", C.c_float), ("dropout_p", C.c_float),
        ("aux_var_value", C.c_float), ("rating_range", C.c_float), ("max_rows", C.c_int32),
        ("max_entries", C.c_int64), ("sharded", C.c_int32),
    ]


class RngSlice(C.Structure):
    _fields_ = [("n_draw_rows", C.c_int32), ("row0", C.c_int32), ("draws_before", C.c_int64), ("draws_total", C.c_int64)]


class StepArgs(C.Structure):
    _fields_ = [("dropout_seed", C.c_uint64), ("step", C.c_uint32), ("row0", C.c_int32),
                ("rows_total", C.c_int32), ("phase", C.c_int32)]


ACTIVATIONS = {"linear": 0, None: 0, "sigmoid": 1, "tanh": 2, "relu": 3, "elu": 4, "selu": 5, "softplus": 6}
AUX_TYPES = {None: 0, "causal": 1, "dropout": 2, "zeros": 3, "both": 4}
LOSSES = {"mean_squared_error": 0, "mse": 0, "mean_absolute_error": 1, "mae": 1}
OPTIMIZERS = {"sgd": 0, "adagrad": 1, "rmsprop": 2, "adam": 3}
N_METRICS = 8
BUF_Z, BUF_DH, BUF_ROWSTATS, BUF_STATS_DH = 0, 1, 2, 3
PAR_COLUMNS, PAR_ROWS = 1, 2

_P = C.c_void_p
_SIGNATURES = {
    "ocf_last_error": (C.c_char_p, []),
    "ocf_version": (C.c_int, []),
    "ocf_device_count": (C.c_int, []),
    "ocf_kernel_launches": (C.c_int64, []),
    "ocf_host_alloc": (C.c_int, [C.c_int64, C.POINTER(_P)]),
    "ocf_host_free": (C.c_int, [_P]),
    "ocf_store_create": (C.c_int, [C.c_int64, C.c_int64, _P, _P, _P, C.POINTER(_P)]),
    "ocf_store_destroy": (C.c_int, [_P]),
    "ocf_store_info": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "ocf_pair_create": (C.c_int, [_P, _P, C.POINTER(_P)]),
    "ocf_pair_destroy": (C.c_int, [_P]),
    "ocf_batch_create": (C.c_int, [C.c_int32, C.c_int64, C.POINTER(_P)]),
    "ocf_batch_destroy": (C.c_int, [_P]),
    "ocf_batch_fill_split": (C.c_int, [_P, _P, _P, C.c_int32, _P, C.c_int64, C.c_int, C.c_float, _P]),
    "ocf_batch_fill_split_uniform": (C.c_int, [_P, _P, _P, C.c_int32, _P, C.c_int64, _P, _P, _P, C.c_int, C.c_float, _P]),
    "ocf_batch_fill_fixed": (C.c_int, [_P, _P, _P, C.c_int32, C.c_float, _P]),
    "ocf_batch_regather": (C.c_int, [_P, _P]),
    "ocf_rng_create": (C.c_int, [C.POINTER(_P)]),
    "ocf_rng_destroy": (C.c_int, [_P]),
    "ocf_rng_set_state": (C.c_int, [_P, _P, C.c_int32]),
    "ocf_rng_get_state": (C.c_int, [_P, _P, C.POINTER(C.c_int32)]),
    "ocf_rng_skip": (C.c_int, [_P, C.c_int64]),
    "ocf_rng_prefetch": (C.c_int, [_P, C.c_int64]),
    "ocf_rng_configure": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int64]),
    "ocf_rng_info": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "ocf_mt_jump_poly": (C.c_int, [C.c_int64, _P]),
    "ocf_mt_jump_apply_host": (C.c_int, [_P, _P, _P]),
    "ocf_rng_last_timing": (C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "ocf_store_set_orig_pos": (C.c_int, [_P, _P]),
    "ocf_batch_fill_split_rng": (C.c_int, [_P, _P, _P, C.c_int32, _P, C.c_double, C.c_double, _P, C.c_int, C.c_float,
                                           C.POINTER(RngSlice), _P]),
    "ocf_comm_unique_id": (C.c_int, [_P]),
    "ocf_comm_create": (C.c_int, [_P, C.c_int32, C.c_int32, C.POINTER(_P)]),
    "ocf_comm_destroy": (C.c_int, [_P]),
    "ocf_comm_info": (C.c_int, [_P, C.POINTER(C.c_int32)]),
    "ocf_model_set_comm": (C.c_int, [_P, _P, C.c_int]),
    "ocf_batch_read_flags": (C.c_int, [_P, _P, C.c_int64, _P]),
    "ocf_profile_enable": (C.c_int, [C.c_int]),
    "ocf_profile_reset": (C.c_int, []),
    "ocf_profile_read": (C.c_int, [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "ocf_batch_info": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "ocf_batch_densify": (C.c_int, [_P, C.c_int, _P, _P]),
    "ocf_model_create": (C.c_int, [C.POINTER(ModelConfig), C.POINTER(_P)]),
    "ocf_model_destroy": (C.c_int, [_P]),
    "ocf_model_reserve": (C.c_int, [_P, C.c_int32, C.c_int64]),
    "ocf_model_num_weights": (C.c_int, [_P]),
    "ocf_model_weight_shape": (C.c_int, [_P, C.c_int, C.POINTER(C.c_int64)]),
    "ocf_model_set_weight": (C.c_int, [_P, C.c_int, _P, C.c_int64]),
    "ocf_model_get_weight": (C.c_int, [_P, C.c_int, _P, C.c_int64]),
    "ocf_model_set_optimizer": (C.c_int, [_P, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float]),
    "ocf_model_set_loss": (C.c_int, [_P, C.c_int, C.c_float]),
    "ocf_model_set_aux": (C.c_int, [_P, C.c_int]),
    "ocf_model_set_trainable": (C.c_int, [_P, C.c_int, C.c_int]),
    "ocf_model_reset_optimizer": (C.c_int, [_P]),
    "ocf_train_step": (C.c_int, [_P, _P, C.POINTER(StepArgs), _P, _P]),
    "ocf_eval_step": (C.c_int, [_P, _P, C.POINTER(StepArgs), _P, _P]),
    "ocf_predict": (C.c_int, [_P, _P, _P, _P]),
    "ocf_score": (C.c_int, [_P, _P, _P, C.c_int, _P]),
    "ocf_score_topk": (C.c_int, [_P, _P, C.c_int32, C.c_int, _P, _P, _P]),
    "ocf_rank_targets": (C.c_int, [_P, _P, C.c_int, C.c_float, _P, _P, _P, _P, _P]),
    "ocf_gemm_tc": (C.c_int, [_P, C.c_int, _P, C.c_int, C.c_int32, C.c_int32, C.c_int32, C.c_int, C.c_int, _P]),
    "ocf_gemm_tc_profile": (C.c_int, [C.c_int, C.c_int, C.c_int32, C.c_int32, C.c_int32, C.c_int, C.c_int, C.c_int,
                                      C.POINTER(C.c_float), C.POINTER(C.c_int64)]),
    "ocf_model_read_metrics": (C.c_int, [_P, C.c_int64, C.c_int32, _P, _P]),
    "ocf_model_wait_metrics": (C.c_int, [_P, C.c_int64, _P]),
    "ocf_model_steps_logged": (C.c_int64, [_P]),
    "ocf_model_buffer": (C.c_int, [_P, C.c_int, C.POINTER(_P), C.POINTER(C.c_int64)]),
    "ocf_model_weight_device": (C.c_int, [_P, C.c_int, C.POINTER(_P), C.POINTER(C.c_int64)]),
    "ocf_vocab_load_json": (C.c_int, [C.c_char_p, C.POINTER(_P)]),
    "ocf_vocab_size": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "ocf_vocab_destroy": (C.c_int, [_P]),
    "ocf_ratings_load_json": (C.c_int, [C.c_char_p, _P, C.c_int, C.POINTER(_P)]),
    "ocf_ratings_info": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "ocf_ratings_keys": (C.c_int, [_P, _P, _P]),
    "ocf_ratings_csr": (C.c_int, [_P, C.c_int, _P, _P, _P, _P]),
    "ocf_ratings_destroy": (C.c_int, [_P]),
    "ocf_csv_load": (C.c_int, [C.c_char_p, C.c_int, C.POINTER(_P)]),
    "ocf_csv_rows": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "ocf_csv_destroy": (C.c_int, [_P]),
    "ocf_split_write": (C.c_int, [_P, _P, C.c_int64, C.POINTER(C.c_double), C.c_char_p, C.c_int, C.c_int, C.c_int,
                                  C.c_int, C.c_int]),
    "ocf_split_build": (C.c_int, [_P, _P, C.c_int64, C.POINTER(C.c_double), C.c_int, C.c_int, C.POINTER(_P)]),
    "ocf_split_info": (C.c_int, [_P, C.POINTER(C.c_int64)]),
    "ocf_split_keys": (C.c_int, [_P, C.c_int, _P, _P]),
    "ocf_split_csr": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, _P, _P]),
    "ocf_split_columns_json": (C.c_int, [_P, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "ocf_split_destroy": (C.c_int, [_P]),
}

_lib = None


def header_symbols():
    """Every function name `include/ocf.h` declares."""
    with open(HEADER_PATH) as f:
        text = f.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ocf_[a-z0-9_]+)\s*\(", text)))


def lib():
    """The loaded library; raises OcfError if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise OcfError("libocf_b200.so is not built (%s); there is no CPU fallback" % SO_PATH)
        handle = C.CDLL(SO_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(status):
    if status != 0:
        msg = lib().ocf_last_error()
        raise OcfError("ocf error %d: %s" % (status, msg.decode() if msg else "?"))


def require_gpu():
    if lib().ocf_device_count() < 1:
        raise OcfError("no CUDA device: the hot path is CUDA-only (sm_100a), there is no CPU fallback")


class PinnedArray(object):
    """A float32 NumPy array over page-locked host memory (freed with the object)."""

    def __init__(self, shape):
        self.shape = tuple(int(x) for x in shape)
        n = 1
        for x in self.shape:
            n *= x
        self._ptr = C.c_void_p()
        check(lib().ocf_host_alloc(4 * n, C.byref(self._ptr)))
        import numpy as np
        buf = (C.c_float * max(n, 1)).from_address(self._ptr.value)
        self.array = np.frombuffer(buf, dtype=np.float32, count=n).reshape(self.shape)

    def __del__(self):
        try:
            if self._ptr is not None and self._ptr.value:
                lib().ocf_host_free(self._ptr)
                self._ptr = None
        except Exception:
            pass


def ptr(array):
    """Host pointer of a C-contiguous NumPy array (None -> NULL)."""
    if array is None:
        return None
    assert array.flags.c_contiguous
    return C.c_void_p(array.ctypes.data)
