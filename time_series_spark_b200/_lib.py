"""ctypes binding of libprophet_b200.so (C ABI in include/prophet_b200.h).

There is no CPU fallback: importing this module never builds or emulates anything, and
``load()`` raises if the CUDA library is missing; ``Context()`` raises if no B200 is visible.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_VARIANT = os.environ.get("PB200_VARIANT", "")          # dev only: load an A/B build (see build.py)
LIB_PATH = os.path.join(_HERE, f"libprophet_b200{'_' + _VARIANT if _VARIANT else ''}.so")

ABI_VERSION = 1
Y_I32, Y_F32, Y_F64 = 0, 1, 2
GROWTH_LINEAR, GROWTH_LOGISTIC = 0, 1
SEAS_AUTO = -1

# per-series status codes (include/prophet_b200.h)
ST_ABSX, ST_ABSF, ST_RELF, ST_ABSGRAD, ST_RELGRAD, ST_MAXIT, ST_CONST_LINEAR = 10, 20, 21, 30, 31, 40, 50
ST_NEWTON = 60
ALG_LBFGS_NEWTON, ALG_LBFGS, ALG_NEWTON = 0, 1, 2
ST_LSFAIL, ST_INIT_ERROR, ST_TOO_FEW, ST_CAP_LE_FLOOR, ST_BAD_INPUT = -1, -2, -3, -4, -5


class Options(C.Structure):
    """struct pb200_options."""
    _fields_ = [
        ("abi_version", C.c_int32), ("growth", C.c_int32), ("multiplicative", C.c_int32),
        ("n_changepoints", C.c_int32), ("changepoint_range", C.c_double),
        ("changepoint_prior_scale", C.c_double), ("seasonality_prior_scale", C.c_double),
        ("yearly", C.c_int32), ("weekly", C.c_int32), ("daily", C.c_int32),
        ("max_iter", C.c_int32), ("history_size", C.c_int32),
        ("init_alpha", C.c_double), ("tol_obj", C.c_double), ("tol_rel_obj", C.c_double),
        ("tol_grad", C.c_double), ("tol_rel_grad", C.c_double), ("tol_param", C.c_double),
        ("interval_width", C.c_double), ("uncertainty_samples", C.c_int32), ("algorithm", C.c_int32),
    ]


class Layout(C.Structure):
    """struct pb200_layout."""
    _fields_ = [("smax", C.c_int32), ("kmax", C.c_int32), ("pstride", C.c_int32),
                ("meta_i32_stride", C.c_int32), ("meta_i64_stride", C.c_int32), ("meta_f64_stride", C.c_int32)]


EXPORTS = [
    "pb200_default_options", "pb200_get_layout", "pb200_create", "pb200_destroy", "pb200_last_error",
    "pb200_stream", "pb200_launch_count", "pb200_last_fit_variant_counts", "pb200_tab_chunk", "pb200_fit_device", "pb200_fit_host", "pb200_predict_device",
    "pb200_predict_host", "pb200_make_future_device", "pb200_synchronize", "pb200_objective_host",
    "pb200_fit_trace_host", "pb200_forecast_csv_lengths_device", "pb200_forecast_csv_rows_device", "pb200_forecast_csv_row_host",
    "pb200_input_csv_count_device", "pb200_input_csv_index_device", "pb200_input_csv_parse_device", "pb200_input_csv_row_host",
]
INPUT_CSV_TILE = 4096       # PB200_INPUT_CSV_TILE

_lib = None


def load() -> C.CDLL:
    """dlopen the in-tree library and declare prototypes.  Raises if it was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m time_series_spark_b200.build` "
            "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    vp, i64, i32, dbl, u64 = C.c_void_p, C.c_int64, C.c_int32, C.c_double, C.c_uint64
    OP = C.POINTER(Options)
    lib.pb200_default_options.argtypes = [OP]
    lib.pb200_default_options.restype = None
    lib.pb200_get_layout.argtypes = [OP, C.POINTER(Layout)]
    lib.pb200_get_layout.restype = C.c_int
    lib.pb200_create.argtypes = [C.c_int]
    lib.pb200_create.restype = vp
    lib.pb200_destroy.argtypes = [vp]
    lib.pb200_destroy.restype = None
    lib.pb200_last_error.argtypes = []
    lib.pb200_last_error.restype = C.c_char_p
    lib.pb200_stream.argtypes = [vp]
    lib.pb200_stream.restype = vp
    lib.pb200_launch_count.argtypes = [vp]
    lib.pb200_launch_count.restype = i64
    lib.pb200_tab_chunk.argtypes = [i32, i32]
    lib.pb200_tab_chunk.restype = i32
    lib.pb200_last_fit_variant_counts.argtypes = [vp, vp]
    lib.pb200_last_fit_variant_counts.restype = C.c_int
    fit_args = [vp, OP, vp, vp, i32, vp, i64, dbl, dbl, vp, vp, vp, vp, vp, vp]
    lib.pb200_fit_device.argtypes = fit_args
    lib.pb200_fit_device.restype = C.c_int
    lib.pb200_fit_host.argtypes = fit_args
    lib.pb200_fit_host.restype = C.c_int
    pred_args = [vp, OP, vp, vp, vp, vp, vp, i64, vp, i32, vp, vp, u64, vp, vp, vp, vp]
    lib.pb200_predict_device.argtypes = pred_args
    lib.pb200_predict_device.restype = C.c_int
    lib.pb200_predict_host.argtypes = pred_args
    lib.pb200_predict_host.restype = C.c_int
    lib.pb200_make_future_device.argtypes = [vp, vp, i64, i32, i64, vp]
    lib.pb200_make_future_device.restype = C.c_int
    lib.pb200_objective_host.argtypes = [vp, OP, vp, vp, i32, vp, i64, dbl, dbl, vp, vp, vp, vp]
    lib.pb200_objective_host.restype = C.c_int
    lib.pb200_fit_trace_host.argtypes = [vp, OP, vp, vp, i32, vp, i64, dbl, dbl, vp, vp, vp, vp, vp, vp, i32]
    lib.pb200_fit_trace_host.restype = C.c_int
    lib.pb200_forecast_csv_lengths_device.argtypes = [vp, vp, vp, vp, i64, i32, vp]
    lib.pb200_forecast_csv_lengths_device.restype = C.c_int
    lib.pb200_forecast_csv_rows_device.argtypes = [vp, vp, vp, vp, vp, i64, C.c_char_p, i32, vp, vp]
    lib.pb200_forecast_csv_rows_device.restype = C.c_int
    lib.pb200_forecast_csv_row_host.argtypes = [i32, i32, i64, i32, C.c_char_p, i32, C.c_char_p]
    lib.pb200_forecast_csv_row_host.restype = i32
    lib.pb200_input_csv_count_device.argtypes = [vp, vp, i64, vp]
    lib.pb200_input_csv_count_device.restype = C.c_int
    lib.pb200_input_csv_index_device.argtypes = [vp, vp, i64, vp, vp]
    lib.pb200_input_csv_index_device.restype = C.c_int
    lib.pb200_input_csv_parse_device.argtypes = [vp, vp, vp, i64, vp, vp, i32, vp, vp, vp, vp, vp, vp]
    lib.pb200_input_csv_parse_device.restype = C.c_int
    lib.pb200_input_csv_row_host.argtypes = [C.c_char_p, i64, vp, vp, vp, vp]
    lib.pb200_input_csv_row_host.restype = i32
    lib.pb200_synchronize.argtypes = [vp]
    lib.pb200_synchronize.restype = C.c_int
    _lib = lib
    return lib


def default_options() -> Options:
    o = Options()
    load().pb200_default_options(C.byref(o))
    return o


def get_layout(opts: Options) -> Layout:
    lay = Layout()
    rc = load().pb200_get_layout(C.byref(opts), C.byref(lay))
    if rc != 0:
        raise ValueError(f"pb200_get_layout failed ({rc}): {last_error()}")
    return lay


def last_error() -> str:
    return (load().pb200_last_error() or b"").decode()


class Pb200Error(RuntimeError):
    pass


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise Pb200Error(f"{what} failed ({rc}): {last_error()}")


class Context:
    """pb200_ctx handle: one per process per GPU."""

    def __init__(self, device: int = 0):
        self._lib = load()
        self._h = self._lib.pb200_create(int(device))
        if not self._h:
            raise Pb200Error("pb200_create failed: " + last_error())
        self.device = int(device)

    @property
    def handle(self):
        return self._h

    @property
    def stream(self) -> int:
        return int(self._lib.pb200_stream(self._h) or 0)

    @property
    def launch_count(self) -> int:
        return int(self._lib.pb200_launch_count(self._h))

    def last_fit_variant_counts(self):
        """(4, 8) int32: series of the last fit per kernel variant (planes, rotation, week table, day table)
        x seasonality mask."""
        import numpy as np
        out = np.zeros(32, np.int32)
        check(self._lib.pb200_last_fit_variant_counts(self._h, out.ctypes.data), "pb200_last_fit_variant_counts")
        return out.reshape(4, 8)

    def synchronize(self) -> None:
        check(self._lib.pb200_synchronize(self._h), "pb200_synchronize")

    def close(self) -> None:
        if self._h:
            self._lib.pb200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
