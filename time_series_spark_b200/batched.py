"""Batched fit / predict: the host side of the GPU call that replaces the reference's
per-group pandas UDFs (model_time_series_udf, src/jobs/prophet_modeler.py:41-85;
forecast_time_series_udf, src/jobs/prophet_scorer.py:35-102).

All arithmetic happens in libprophet_b200.so; this module only moves buffers.
torch is used for device memory / streams when the caller wants inputs resident in HBM;
the *_host entry points take numpy arrays and stage through the library's own buffers.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional

import numpy as np

from . import _lib as L


def make_options(growth: str = "logistic", seasonality_mode: str = "multiplicative",
                 yearly_seasonality="auto", weekly_seasonality="auto", daily_seasonality="auto",
                 n_changepoints: int = 25, changepoint_range: float = 0.8,
                 changepoint_prior_scale: float = 0.05, seasonality_prior_scale: float = 10.0,
                 interval_width: float = 0.8, uncertainty_samples: int = 1000,
                 max_iter: int = 10000, algorithm: str = "LBFGS+Newton") -> L.Options:
    """Prophet.__init__ arguments -> pb200_options.  Defaults = the reference's hard-coded
    ``Prophet(growth='logistic', seasonality_mode='multiplicative')`` (prophet_modeler.py:65)."""
    o = L.default_options()
    if growth not in ("linear", "logistic"):
        raise ValueError('Parameter "growth" should be "linear" or "logistic".')
    if seasonality_mode not in ("additive", "multiplicative"):
        raise ValueError('seasonality_mode must be "additive" or "multiplicative"')
    o.growth = L.GROWTH_LOGISTIC if growth == "logistic" else L.GROWTH_LINEAR
    o.multiplicative = 1 if seasonality_mode == "multiplicative" else 0

    def sw(v, default_order):
        if isinstance(v, str) and v == "auto":
            return L.SEAS_AUTO
        if v is True:
            return 1
        if v is False:
            return 0
        if int(v) == 0:
            return 0
        if int(v) == default_order:
            return 1
        raise ValueError(f"only the default Fourier order {default_order} is compiled in (got {v})")

    o.yearly, o.weekly, o.daily = sw(yearly_seasonality, 10), sw(weekly_seasonality, 3), sw(daily_seasonality, 4)
    o.n_changepoints = int(n_changepoints)
    o.changepoint_range = float(changepoint_range)
    o.changepoint_prior_scale = float(changepoint_prior_scale)
    o.seasonality_prior_scale = float(seasonality_prior_scale)
    o.interval_width = float(interval_width)
    o.uncertainty_samples = int(uncertainty_samples)
    o.max_iter = int(max_iter)
    o.algorithm = {"LBFGS+Newton": L.ALG_LBFGS_NEWTON, "LBFGS": L.ALG_LBFGS, "Newton": L.ALG_NEWTON}[algorithm]
    return o


@dataclass
class FittedBatch:
    """Fitted-model arrays of one shard (numpy on host, or torch tensors on device)."""
    params: object       # [N, pstride] f64: k, m, sigma_obs, delta[smax], beta[kmax]
    tchange: object      # [N, smax]    f64
    meta_i32: object     # [N, 8]  T, S, n_cp_real, seasonality mask, status, iters, n_evals, i1
    meta_i64: object     # [N, 2]  start_ns, t_scale_ns
    meta_f64: object     # [N, 4]  y_scale, floor, cap, neg_log_posterior
    smax: int
    kmax: int

    @property
    def n(self) -> int:
        return int(self.params.shape[0])

    @property
    def status(self):
        return self.meta_i32[:, 4]

    def to_host(self) -> "FittedBatch":
        if isinstance(self.params, np.ndarray):
            return self
        return FittedBatch(*(x.cpu().numpy() for x in (self.params, self.tchange, self.meta_i32,
                                                       self.meta_i64, self.meta_f64)),
                           smax=self.smax, kmax=self.kmax)


def _y_dtype(y) -> int:
    dt = str(y.dtype).replace("torch.", "")
    if dt == "int32":
        return L.Y_I32
    if dt == "float32":
        return L.Y_F32
    if dt == "float64":
        return L.Y_F64
    raise TypeError(f"y must be int32, float32 or float64 (got {y.dtype})")


def _np_ptr(a: np.ndarray) -> int:
    return a.ctypes.data


def fit_batch_host(ctx: L.Context, opts: L.Options, ds_ns: np.ndarray, y: np.ndarray, offsets: np.ndarray,
                   floor: float, cap_multiplier: float, cap: Optional[np.ndarray] = None) -> FittedBatch:
    """pb200_fit_host: numpy (ideally pinned) buffers in, numpy out; copies inside the call."""
    ds_ns = np.ascontiguousarray(ds_ns, dtype=np.int64)
    y = np.ascontiguousarray(y)
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    n = offsets.size - 1
    lay = L.get_layout(opts)
    params = np.empty((n, lay.pstride), np.float64)
    tchange = np.empty((n, lay.smax), np.float64)
    mi32 = np.empty((n, 8), np.int32)
    mi64 = np.empty((n, 2), np.int64)
    mf64 = np.empty((n, 4), np.float64)
    capp = None
    if cap is not None:
        cap = np.ascontiguousarray(cap, dtype=np.float64)
        capp = _np_ptr(cap)
    if n > 0:
        rc = L.load().pb200_fit_host(ctx.handle, C.byref(opts), _np_ptr(ds_ns), _np_ptr(y), _y_dtype(y),
                                     _np_ptr(offsets), n, float(floor), float(cap_multiplier), capp,
                                     _np_ptr(params), _np_ptr(tchange), _np_ptr(mi32), _np_ptr(mi64), _np_ptr(mf64))
        L.check(rc, "pb200_fit_host")
    return FittedBatch(params, tchange, mi32, mi64, mf64, lay.smax, lay.kmax)


def fit_batch_trace_host(ctx: L.Context, opts: L.Options, ds_ns: np.ndarray, y: np.ndarray, offsets: np.ndarray,
                         floor: float, cap_multiplier: float, trace_cap: int = 256):
    """pb200_fit_trace_host (parity-test hook): the fit plus, per series, one row
    ``(iteration, f_k, alpha_k, n_evals)`` per accepted L-BFGS iteration (``[n, trace_cap, 4]``)."""
    ds_ns = np.ascontiguousarray(ds_ns, dtype=np.int64)
    y = np.ascontiguousarray(y)
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    n = offsets.size - 1
    lay = L.get_layout(opts)
    params = np.empty((n, lay.pstride), np.float64)
    tchange = np.empty((n, lay.smax), np.float64)
    mi32 = np.empty((n, 8), np.int32)
    mi64 = np.empty((n, 2), np.int64)
    mf64 = np.empty((n, 4), np.float64)
    trace = np.zeros((n, trace_cap, 4), np.float64)
    if n > 0:
        rc = L.load().pb200_fit_trace_host(ctx.handle, C.byref(opts), _np_ptr(ds_ns), _np_ptr(y), _y_dtype(y),
                                           _np_ptr(offsets), n, float(floor), float(cap_multiplier),
                                           _np_ptr(params), _np_ptr(tchange), _np_ptr(mi32), _np_ptr(mi64), _np_ptr(mf64),
                                           _np_ptr(trace), int(trace_cap))
        L.check(rc, "pb200_fit_trace_host")
    return FittedBatch(params, tchange, mi32, mi64, mf64, lay.smax, lay.kmax), trace


def fit_batch_device(ctx: L.Context, opts: L.Options, ds_ns, y, offsets_host: np.ndarray,
                     floor: float, cap_multiplier: float, cap=None, out: Optional[FittedBatch] = None,
                     sync: bool = True) -> FittedBatch:
    """pb200_fit_device: ``ds_ns`` / ``y`` / ``cap`` are torch CUDA tensors already in HBM."""
    import torch
    offsets_host = np.ascontiguousarray(offsets_host, dtype=np.int64)
    n = offsets_host.size - 1
    lay = L.get_layout(opts)
    dev = ds_ns.device
    if out is None:
        out = FittedBatch(torch.empty((n, lay.pstride), dtype=torch.float64, device=dev),
                          torch.empty((n, lay.smax), dtype=torch.float64, device=dev),
                          torch.empty((n, 8), dtype=torch.int32, device=dev),
                          torch.empty((n, 2), dtype=torch.int64, device=dev),
                          torch.empty((n, 4), dtype=torch.float64, device=dev), lay.smax, lay.kmax)
    if n > 0:
        # inputs were produced on torch's current stream; the library has its own stream
        torch.cuda.current_stream(dev).synchronize()
        rc = L.load().pb200_fit_device(ctx.handle, C.byref(opts), ds_ns.data_ptr(), y.data_ptr(), _y_dtype(y),
                                       _np_ptr(offsets_host), n, float(floor), float(cap_multiplier),
                                       cap.data_ptr() if cap is not None else None,
                                       out.params.data_ptr(), out.tchange.data_ptr(), out.meta_i32.data_ptr(),
                                       out.meta_i64.data_ptr(), out.meta_f64.data_ptr())
        L.check(rc, "pb200_fit_device")
        if sync:
            ctx.synchronize()
    return out


@dataclass
class ForecastBatch:
    future_ds: object    # [N, H] int64 ns
    yhat: object         # [N, H] f64
    yhat_lower: object   # [N, H] f64 or None
    yhat_upper: object
    yhat_int: object     # [N, H] int32 (truncated, floor-clamped)


def make_future(last_ds_ns: np.ndarray, periods: int, freq_ns: int) -> np.ndarray:
    """Prophet.make_future_dataframe(include_history=False) for a fixed-width frequency
    (prophet_scorer.py:64-66): last + (1..periods) * freq."""
    last = np.asarray(last_ds_ns, dtype=np.int64)
    return last[:, None] + np.int64(freq_ns) * np.arange(1, periods + 1, dtype=np.int64)[None, :]


def make_future_device(ctx: L.Context, last_ds_ns, periods: int, freq_ns: int):
    """pb200_make_future_device: the same grid built on the GPU from a CUDA int64 tensor of last history timestamps
    (for callers that keep the scorer's inputs resident)."""
    import torch
    n = int(last_ds_ns.shape[0])
    out = torch.empty((n, periods), dtype=torch.int64, device=last_ds_ns.device)
    if n and periods:
        torch.cuda.current_stream(last_ds_ns.device).synchronize()
        rc = L.load().pb200_make_future_device(ctx.handle, last_ds_ns.data_ptr(), n, int(periods), int(freq_ns), out.data_ptr())
        L.check(rc, "pb200_make_future_device")
        ctx.synchronize()
    return out


def forecast_csv_device(ctx: L.Context, series_id, dim_id, ds_ns, quantity, created: bytes):
    """The CSV text of forecast rows, formatted on the GPU (pb200_forecast_csv_{lengths,rows}_device): int32 / int32 /
    int64 ns / int32 CUDA tensors of equal length in, one uint8 CUDA tensor out (no header line).  Row format and the
    supported timestamp range: include/prophet_b200.h."""
    import torch
    n = int(series_id.shape[0])
    dev = series_id.device
    if n == 0:
        return torch.empty(0, dtype=torch.uint8, device=dev)
    for t, dt in ((series_id, torch.int32), (dim_id, torch.int32), (ds_ns, torch.int64), (quantity, torch.int32)):
        if t.dtype != dt or not t.is_contiguous() or int(t.shape[0]) != n or t.device != dev:
            raise ValueError("forecast_csv_device wants contiguous int32 / int32 / int64 / int32 tensors of one length on one device")
    lib = L.load()
    lens = torch.empty(n, dtype=torch.int64, device=dev)
    torch.cuda.current_stream(dev).synchronize()
    L.check(lib.pb200_forecast_csv_lengths_device(ctx.handle, series_id.data_ptr(), dim_id.data_ptr(), quantity.data_ptr(), n,
                                                  len(created), lens.data_ptr()), "pb200_forecast_csv_lengths_device")
    ctx.synchronize()
    ends = torch.cumsum(lens, 0)                      # the scan is plumbing (torch); the two passes over the rows are the kernels
    total = int(ends[-1].item())
    offs = ends - lens
    out = torch.empty(total, dtype=torch.uint8, device=dev)
    torch.cuda.current_stream(dev).synchronize()
    L.check(lib.pb200_forecast_csv_rows_device(ctx.handle, series_id.data_ptr(), dim_id.data_ptr(), ds_ns.data_ptr(),
                                               quantity.data_ptr(), n, created, len(created), offs.data_ptr(), out.data_ptr()),
            "pb200_forecast_csv_rows_device")
    ctx.synchronize()
    return out


def forecast_csv_row_host(series_id: int, dim_id: int, ds_ns: int, quantity: int, created: bytes) -> bytes:
    """One row through the same formatter on the host (pb200_forecast_csv_row_host; tests)."""
    import ctypes
    buf = ctypes.create_string_buffer(160)
    n = L.load().pb200_forecast_csv_row_host(int(series_id), int(dim_id), int(ds_ns), int(quantity), created, len(created), buf)
    if n < 0:
        raise ValueError("pb200_forecast_csv_row_host refused the row")
    return buf.raw[:n]


def parse_input_csv_device(ctx: L.Context, text, n_bytes: int, file_start, file_sid):
    """The modeler's input CSV parsed on the GPU (pb200_input_csv_{count,index,parse}_device): ``text`` a uint8 CUDA
    tensor holding the concatenated files in its first ``n_bytes`` (every file ending in '\\n', numel a multiple of 16),
    ``file_start`` / ``file_sid`` int64 / int32 CUDA tensors with each file's first byte and series_id.  Returns
    (series_id, dim_id, ds_ns, quantity, quantity_valid, row_end, n_refused, first_refused): six CUDA tensors of one
    entry per row (row_end: the offset one past the row's '\\n') and two ints (first_refused is -1 when no row was
    refused).  Grammar: include/prophet_b200.h."""
    import torch
    dev = text.device
    if text.dtype != torch.uint8 or not text.is_contiguous() or text.numel() % 16 or text.numel() < n_bytes:
        raise ValueError("parse_input_csv_device wants a contiguous uint8 tensor padded to a multiple of 16 bytes")
    lib = L.load()
    tiles = -(-n_bytes // L.INPUT_CSV_TILE)
    counts = torch.empty(tiles, dtype=torch.int64, device=dev)
    torch.cuda.current_stream(dev).synchronize()
    L.check(lib.pb200_input_csv_count_device(ctx.handle, text.data_ptr(), n_bytes, counts.data_ptr()),
            "pb200_input_csv_count_device")
    ctx.synchronize()
    ends = torch.cumsum(counts, 0)                    # the scan is plumbing (torch); the passes over the bytes are the kernels
    n_rows = int(ends[-1].item()) if tiles else 0
    row_end = torch.empty(n_rows, dtype=torch.int64, device=dev)
    offs = ends - counts
    torch.cuda.current_stream(dev).synchronize()
    L.check(lib.pb200_input_csv_index_device(ctx.handle, text.data_ptr(), n_bytes, offs.data_ptr(), row_end.data_ptr()),
            "pb200_input_csv_index_device")
    del counts, ends, offs
    sid = torch.empty(n_rows, dtype=torch.int32, device=dev)
    did = torch.empty(n_rows, dtype=torch.int32, device=dev)
    ds = torch.empty(n_rows, dtype=torch.int64, device=dev)
    qty = torch.empty(n_rows, dtype=torch.int32, device=dev)
    valid = torch.empty(n_rows, dtype=torch.uint8, device=dev)
    refused = torch.empty(2, dtype=torch.int64, device=dev)
    torch.cuda.current_stream(dev).synchronize()
    L.check(lib.pb200_input_csv_parse_device(ctx.handle, text.data_ptr(), row_end.data_ptr(), n_rows, file_start.data_ptr(),
                                             file_sid.data_ptr(), int(file_start.numel()), sid.data_ptr(), did.data_ptr(),
                                             ds.data_ptr(), qty.data_ptr(), valid.data_ptr(), refused.data_ptr()),
            "pb200_input_csv_parse_device")
    ctx.synchronize()
    n_bad, first = (int(v) for v in refused.cpu().tolist())
    return sid, did, ds, qty, valid, row_end, n_bad, first


def input_csv_row_host(line: bytes):
    """One input line, its line end included, through the same row parser on the host (pb200_input_csv_row_host;
    tests): (dim_id, ds_ns, quantity or None), or None when the parser refuses the line."""
    import ctypes
    dim, ds, q, qv = ctypes.c_int32(), ctypes.c_int64(), ctypes.c_int32(), ctypes.c_int32()
    rc = L.load().pb200_input_csv_row_host(line, len(line), ctypes.addressof(dim), ctypes.addressof(ds),
                                           ctypes.addressof(q), ctypes.addressof(qv))
    if rc < 0:
        raise ValueError("pb200_input_csv_row_host: bad argument")
    return (dim.value, ds.value, q.value if qv.value else None) if rc == 1 else None


def predict_batch_host(ctx: L.Context, opts: L.Options, fitted: FittedBatch, future_ds: np.ndarray,
                       floor: np.ndarray, cap: np.ndarray, seed: int = 0, intervals: bool = True) -> ForecastBatch:
    """pb200_predict_host.  ``floor`` / ``cap`` per model as the scorer reads them back from
    the float32 model-table columns (prophet_scorer.py:46-47,67-68)."""
    fitted = fitted.to_host()
    n = fitted.n
    future_ds = np.ascontiguousarray(future_ds, dtype=np.int64).reshape(n, -1)
    h = future_ds.shape[1]
    floor = np.ascontiguousarray(np.broadcast_to(np.asarray(floor, dtype=np.float64), (n,)))
    cap = np.ascontiguousarray(np.broadcast_to(np.asarray(cap, dtype=np.float64), (n,)))
    yhat = np.empty((n, h), np.float64)
    yint = np.empty((n, h), np.int32)
    do_mc = intervals and opts.uncertainty_samples > 0
    lo = np.empty((n, h), np.float64) if do_mc else None
    hi = np.empty((n, h), np.float64) if do_mc else None
    if n > 0 and h > 0:
        rc = L.load().pb200_predict_host(
            ctx.handle, C.byref(opts), _np_ptr(np.ascontiguousarray(fitted.params)),
            _np_ptr(np.ascontiguousarray(fitted.tchange)), _np_ptr(np.ascontiguousarray(fitted.meta_i32)),
            _np_ptr(np.ascontiguousarray(fitted.meta_i64)), _np_ptr(np.ascontiguousarray(fitted.meta_f64)),
            n, _np_ptr(future_ds), h, _np_ptr(floor), _np_ptr(cap), int(seed) & (2**64 - 1),
            _np_ptr(yhat), _np_ptr(lo) if do_mc else None, _np_ptr(hi) if do_mc else None, _np_ptr(yint))
        L.check(rc, "pb200_predict_host")
    return ForecastBatch(future_ds, yhat, lo, hi, yint)


def predict_batch_device(ctx: L.Context, opts: L.Options, fitted: FittedBatch, future_ds, floor, cap,
                         seed: int = 0, intervals: bool = True, sync: bool = True,
                         out: Optional["ForecastBatch"] = None) -> ForecastBatch:
    """pb200_predict_device with torch CUDA tensors (``out`` reuses a previous result's buffers)."""
    import torch
    n = fitted.n
    h = int(future_ds.shape[1])
    dev = future_ds.device
    do_mc = intervals and opts.uncertainty_samples > 0
    if out is not None:
        yhat, yint, lo, hi = out.yhat, out.yhat_int, out.yhat_lower, out.yhat_upper
    else:
        yhat = torch.empty((n, h), dtype=torch.float64, device=dev)
        yint = torch.empty((n, h), dtype=torch.int32, device=dev)
        lo = torch.empty((n, h), dtype=torch.float64, device=dev) if do_mc else None
        hi = torch.empty((n, h), dtype=torch.float64, device=dev) if do_mc else None
    if n > 0 and h > 0:
        if out is None:
            torch.cuda.current_stream(dev).synchronize()
        rc = L.load().pb200_predict_device(
            ctx.handle, C.byref(opts), fitted.params.data_ptr(), fitted.tchange.data_ptr(),
            fitted.meta_i32.data_ptr(), fitted.meta_i64.data_ptr(), fitted.meta_f64.data_ptr(), n,
            future_ds.data_ptr(), h, floor.data_ptr(), cap.data_ptr(), int(seed) & (2**64 - 1),
            yhat.data_ptr(), lo.data_ptr() if do_mc else None, hi.data_ptr() if do_mc else None, yint.data_ptr())
        L.check(rc, "pb200_predict_device")
        if sync:
            ctx.synchronize()
    return ForecastBatch(future_ds, yhat, lo, hi, yint)


def objective_host(ctx: L.Context, opts: L.Options, ds_ns: np.ndarray, y: np.ndarray, offsets: np.ndarray,
                   floor: float, cap_multiplier: float, theta: np.ndarray):
    """pb200_objective_host (parity-test hook): objective and gradient at ``theta`` rows
    (Stan unconstrained order k, m, delta[S], log sigma, beta[K], zero-padded to pstride)."""
    ds_ns = np.ascontiguousarray(ds_ns, dtype=np.int64)
    y = np.ascontiguousarray(y)
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    n = offsets.size - 1
    lay = L.get_layout(opts)
    th = np.zeros((n, lay.pstride), np.float64)
    th[:, :theta.shape[1]] = theta
    f = np.empty(n, np.float64)
    g = np.empty((n, lay.pstride), np.float64)
    mi32 = np.empty((n, 8), np.int32)
    rc = L.load().pb200_objective_host(ctx.handle, C.byref(opts), _np_ptr(ds_ns), _np_ptr(y), _y_dtype(y),
                                       _np_ptr(offsets), n, float(floor), float(cap_multiplier), _np_ptr(th),
                                       _np_ptr(f), _np_ptr(g), _np_ptr(mi32))
    L.check(rc, "pb200_objective_host")
    return f, g, mi32
