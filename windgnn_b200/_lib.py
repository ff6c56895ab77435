"""ctypes binding of the C-ABI library (``include/windgnn_b200.h``).

The library is CUDA-only: if it is missing this module raises at import of the first
symbol — there is no fallback path.
"""

from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_int, c_int64, c_size_t, c_uint64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
# WINDGNN_B200_LIB: an experiment build of the same library (windgnn_b200/build.py, WG_LIB_SUFFIX)
LIB_PATH = os.environ.get("WINDGNN_B200_LIB") or os.path.join(HERE, "lib", "libwindgnn_b200.so")

WG_OK = 0
WG_ERR_BAD_ARG = -1
WG_ERR_UNSUPPORTED = -2
WG_ERR_WORKSPACE = -3
WG_ERR_CUDA = -4
ABI_VERSION = 4
FLAG_TENSOR_CORES = 1


class WindGNNError(RuntimeError):
    """Raised when a C-ABI call returns a non-zero status."""

    def __init__(self, code: int, message: str):
        super().__init__(f"windgnn_b200 error {code}: {message}")
        self.code = code


_P = c_void_p
_DIMS = [c_int, c_int, c_int, c_int, c_int, c_int]  # T, S, F_in, F_hid, F_out, H

_SIGNATURES = {
    "wg_abi_version": (c_int, []),
    "wg_last_error": (c_char_p, []),
    "wg_gcn_gru_workspace_bytes": (c_size_t, [c_int64, *_DIMS, c_int64, c_int]),
    "wg_gcn_gru_forward_f32": (c_int, [_P] * 11 + [c_int64, *_DIMS, c_int64, c_int, _P, c_size_t, c_int, _P]),
    "wg_gcn_gru_csr_workspace_bytes": (c_size_t, [c_int64, *_DIMS, c_int64, c_int]),
    "wg_gcn_gru_forward_csr_f32": (c_int, [_P] * 13 + [c_int64, *_DIMS, c_int64, c_int, _P, c_size_t, c_int, _P]),
    # N, Ttot, then the dims with T = L
    "wg_gcn_gru_forecast_workspace_bytes": (c_size_t, [c_int64, c_int64, *_DIMS, c_int64, c_int]),
    "wg_gcn_gru_forecast_f32": (c_int, [_P] * 12 + [c_int64, c_int64, *_DIMS, c_int64, c_int, _P, c_size_t, c_int,
                                                    _P]),
    "wg_gcn_gru_forecast_csr_workspace_bytes": (c_size_t, [c_int64, c_int64, *_DIMS, c_int64, c_int]),
    "wg_gcn_gru_forecast_csr_f32": (c_int, [_P] * 14 + [c_int64, c_int64, *_DIMS, c_int64, c_int, _P, c_size_t,
                                                        c_int, _P]),
    "wg_gcn_gru_host_workspace_bytes": (c_size_t, [c_int64, *_DIMS, c_int64, c_int]),
    "wg_gcn_gru_forward_host_f32": (c_int, [_P] * 11 + [c_int64, *_DIMS, c_int64, c_int, _P, c_size_t, c_int]),
    "wg_gcn_gru_predict_host_f32": (c_int, [_P] * 11 + [c_int64, *_DIMS, c_int64, c_int, c_double, c_double, _P,
                                            c_size_t, c_int]),
    "wg_gcn_layer_f32": (c_int, [_P] * 5 + [c_int64, c_int, c_int, c_int, c_int, _P]),
    "wg_stage_pack_f32": (c_int, [_P] * 4 + [*_DIMS, c_int64, c_int, _P, c_size_t, c_int, _P]),
    "wg_stage_gcn_f32": (c_int, [_P] * 6 + [c_int64, *_DIMS, c_int64, c_int, _P, c_size_t, c_int, _P]),
    "wg_stage_inproj_f32": (c_int, [c_int64, *_DIMS, c_int64, c_int, _P, c_size_t, c_int, _P]),
    "wg_stage_recur_f32": (c_int, [_P, c_int64, *_DIMS, c_int64, c_int, _P, c_size_t, c_int, _P]),
    "wg_build_graph_workspace_bytes": (c_size_t, [c_int, c_int]),
    "wg_build_graph_f64": (c_int, [_P, _P, _P, c_int, c_int, _P, c_size_t, c_int, _P]),
    "wg_build_graph_csr_workspace_bytes": (c_size_t, [c_int, c_int]),
    "wg_build_graph_csr_f64": (c_int, [_P, c_int, c_int, _P, _P, _P, _P, c_int64, _P, c_size_t, c_int, _P]),
    "wg_synthetic_coordinates_f64": (c_int, [_P, c_int, c_uint64, c_int, _P]),
    "wg_pivot_table_f32": (c_int, [_P, _P, _P, _P, c_int64, c_int, c_int, c_int64, c_int, _P]),
    "wg_num_windows": (c_int64, [c_int64, c_int, c_int]),
    "wg_make_windows_f32": (c_int, [_P, _P, _P, _P, c_int64, c_int, c_int, c_int, c_int, c_int, c_int64, c_int, _P]),
    "wg_denorm_last_step_f32": (c_int, [_P, _P, c_int64, c_int, c_int, c_double, c_double, c_int, _P]),
    "wg_measure_ffma_tflops": (c_double, [c_int, c_int]),
    "wg_gcn_gru_param_count": (c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    "wg_gcn_gru_train_workspace_bytes": (c_size_t, [c_int64, *_DIMS]),
    "wg_gcn_gru_forward_train_f32": (c_int, [_P] * 11 + [c_int64, *_DIMS, _P, c_size_t, c_int, _P]),
    "wg_gcn_gru_backward_f32": (c_int, [_P] * 11 + [c_int64, *_DIMS, _P, c_size_t, c_int, _P]),
    # N, Ttot, L, S, F_in, F_hid, F_out, H
    "wg_gcn_gru_train_windows_workspace_bytes": (c_size_t, [c_int64, c_int64, *_DIMS]),
    "wg_gcn_gru_forward_train_windows_f32": (c_int, [_P] * 12 + [c_int64, c_int64, *_DIMS, _P, c_size_t, c_int, _P]),
    "wg_gcn_gru_backward_windows_f32": (c_int, [_P] * 12 + [c_int64, c_int64, *_DIMS, _P, c_size_t, c_int, _P]),
    "wg_mse_window_labels_workspace_bytes": (c_size_t, [c_int64]),
    "wg_mse_window_labels_f32": (c_int, [_P, _P, _P, c_int64, c_int, c_int64, c_int, c_int, c_int, c_int, _P, _P, _P,
                                         c_size_t, c_int, _P]),
    "wg_mse_workspace_bytes": (c_size_t, []),
    "wg_mse_loss_grad_f32": (c_int, [_P, _P, c_int64, _P, _P, _P, c_size_t, c_int, _P]),
    "wg_adam_step_f32": (c_int, [_P, _P, _P, _P, c_int64, c_double, c_double, c_double, c_double, c_int64,
                                 c_double, c_int, _P]),
}

_lib = None


def load() -> ctypes.CDLL:
    """Load (once) and type the shared library.  Fails loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m windgnn_b200.build` "
            "(windgnn_b200 has no CPU or PyTorch fallback)"
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export it
        fn.restype = restype
        fn.argtypes = argtypes
    got = lib.wg_abi_version()
    if got != ABI_VERSION:
        raise ImportError(f"libwindgnn_b200.so has ABI {got}, the Python side expects {ABI_VERSION}")
    _lib = lib
    return lib


def last_error() -> str:
    return (load().wg_last_error() or b"").decode("utf-8", "replace")


def check(status: int) -> None:
    if status != WG_OK:
        raise WindGNNError(status, last_error())


def exported_names():
    return sorted(_SIGNATURES)
