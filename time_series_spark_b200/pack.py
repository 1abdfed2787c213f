"""Arrow -> ragged (pinned) buffers: the host side of the grouped-map boundary.

Replaces Spark's shuffle + Arrow hand-off of ``groupby('series_id','dim_id').apply``
(reference src/jobs/prophet_modeler.py:139-141): rows are sorted by (series_id, dim_id, ds)
-- the sort fbprophet's setup_dataframe does per group -- and cut into CSR offsets.
Null ``y`` rows are dropped from the fit buffers (fbprophet: ``df[df['y'].notnull()]``) but
still count for ``history_dates.max()`` (the anchor of make_future_dataframe).
"""
from __future__ import annotations

import bisect
from dataclasses import dataclass

import numpy as np
import pyarrow as pa
import pyarrow.compute as pc


@dataclass
class PackedGroups:
    series_id: np.ndarray    # [N] int32
    dim_id: np.ndarray       # [N] int32
    offsets: np.ndarray      # [N+1] int64 into ds / y
    ds: np.ndarray           # [R] int64 ns, ascending within a group
    y: np.ndarray            # [R] int32 (or float64 when the input was not integral)
    last_ds: np.ndarray      # [N] int64: max ds of the group INCLUDING null-y rows
    n_rows_in: np.ndarray    # [N] rows of the group before dropping nulls

    @property
    def n(self) -> int:
        return self.offsets.size - 1

    def take(self, lo: int, hi: int) -> "PackedGroups":
        """Groups [lo, hi) (a rank's shard; see dist.shard_bounds)."""
        a, b = int(self.offsets[lo]), int(self.offsets[hi])
        return PackedGroups(self.series_id[lo:hi], self.dim_id[lo:hi], self.offsets[lo:hi + 1] - a,
                            self.ds[a:b], self.y[a:b], self.last_ds[lo:hi], self.n_rows_in[lo:hi])

    @property
    def on_device(self) -> bool:
        return not isinstance(self.ds, np.ndarray)


def _pinned_like(a: np.ndarray) -> np.ndarray:
    """Copy into page-locked memory when a CUDA runtime is usable (faster H2D), else return as is."""
    try:
        import torch
        if torch.cuda.is_available():
            t = torch.empty(a.shape, dtype=torch.from_numpy(a[:0]).dtype, pin_memory=True)
            out = t.numpy()
            out[...] = a
            return _Keep(out, t)
    except Exception:
        pass
    return a


def _group_keys(table: pa.Table, keys):
    """The two int group-key columns as int64 numpy arrays.  A null key is refused: Spark would make null its own
    group, and the reference's fixed schema never produces one (series_id comes from the directory name, an empty
    dim_id field is a malformed row) -- silently merging it into another group would be worse than failing."""
    out = []
    for k in keys[:2]:
        col = table[k]
        if col.null_count:
            raise ValueError(f"group key column {k!r} holds {col.null_count} null value(s); every row needs both "
                             f"{keys[0]!r} and {keys[1]!r}")
        out.append(np.asarray(col.combine_chunks().to_numpy(zero_copy_only=False)).astype(np.int64))
    return out


class _Keep(np.ndarray):
    """ndarray view that keeps the owning pinned torch tensor alive."""
    def __new__(cls, arr, owner):
        obj = np.asarray(arr).view(cls)
        obj._owner = owner
        return obj

    def __array_finalize__(self, obj):
        self._owner = getattr(obj, "_owner", None)


def pack_groups(table: pa.Table, keys=("series_id", "dim_id"), ds_col="ds", y_col="y", pin: bool = True) -> PackedGroups:
    if table.num_rows == 0:
        z = np.zeros(0, np.int32)
        return PackedGroups(z, z, np.zeros(1, np.int64), np.zeros(0, np.int64), z, np.zeros(0, np.int64), np.zeros(0, np.int64))
    ds_arr = table[ds_col]
    if pa.types.is_timestamp(ds_arr.type):
        ds_arr = pc.cast(ds_arr, pa.timestamp("ns"))
        if ds_arr.null_count:
            raise ValueError("Found NaN in column ds.")       # fbprophet setup_dataframe
        ds_np = pc.cast(ds_arr, pa.int64()).to_numpy() if isinstance(ds_arr, pa.Array) else \
            pc.cast(ds_arr, pa.int64()).combine_chunks().to_numpy()
    else:
        ds_np = ds_arr.to_numpy() if isinstance(ds_arr, pa.Array) else ds_arr.combine_chunks().to_numpy()
        ds_np = np.asarray(ds_np, dtype=np.int64)
    k0, k1 = _group_keys(table, keys)
    ycol = table[y_col].combine_chunks()
    y_null = np.asarray(ycol.is_null().to_numpy(zero_copy_only=False)) if ycol.null_count else None
    if pa.types.is_integer(ycol.type):
        y_np = np.asarray(ycol.fill_null(0).to_numpy(zero_copy_only=False)).astype(np.int32)
    else:
        y_np = np.asarray(ycol.to_numpy(zero_copy_only=False)).astype(np.float64)
        nanmask = np.isnan(y_np)
        if nanmask.any():
            y_null = nanmask if y_null is None else (y_null | nanmask)
    order = np.lexsort((ds_np, k1, k0))            # stable: by series_id, dim_id, ds
    k0, k1, ds_np, y_np = k0[order], k1[order], ds_np[order], y_np[order]
    if y_null is not None:
        y_null = y_null[order]
    new_grp = np.empty(k0.size, dtype=bool)
    new_grp[0] = True
    np.logical_or(k0[1:] != k0[:-1], k1[1:] != k1[:-1], out=new_grp[1:])
    starts = np.flatnonzero(new_grp)
    ends = np.append(starts[1:], k0.size)
    last_ds = ds_np[ends - 1]
    n_rows_in = (ends - starts).astype(np.int64)
    sid, did = k0[starts].astype(np.int32), k1[starts].astype(np.int32)
    if y_null is not None and y_null.any():
        keep = ~y_null
        grp_id = np.cumsum(new_grp) - 1
        counts = np.bincount(grp_id[keep], minlength=starts.size).astype(np.int64)
        ds_np, y_np = ds_np[keep], y_np[keep]
    else:
        counts = n_rows_in
    offsets = np.zeros(starts.size + 1, np.int64)
    np.cumsum(counts, out=offsets[1:])
    ds_np, y_np = np.ascontiguousarray(ds_np), np.ascontiguousarray(y_np)
    if pin:
        ds_np, y_np = _pinned_like(ds_np), _pinned_like(y_np)
    return PackedGroups(sid, did, offsets, ds_np, y_np, last_ds.astype(np.int64), n_rows_in)


_SLOT_BYTES = 32 << 20
_slots = {}            # device index -> (two pinned byte tensors, two CUDA events): the H2D staging ring


def ring_upload(out, fill) -> None:
    """Fills the contiguous device tensor ``out`` through a small ring of pinned slots: ``fill(dst, lo, hi)`` writes
    bytes [lo, hi) of ``out``'s contents into the pinned uint8 numpy array ``dst``, and each slot is DMA'd to the
    device while the next one fills.  The copies are queued on the current stream."""
    import torch
    dev = out.device
    ring = _slots.get(dev.index)
    if ring is None:
        ring = ([torch.empty(_SLOT_BYTES, dtype=torch.uint8, pin_memory=True) for _ in range(2)],
                [torch.cuda.Event() for _ in range(2)])
        _slots[dev.index] = ring
    bufs, evs = ring
    dst = out.view(torch.uint8)
    n = dst.numel()
    slot = bufs[0].numel()
    cur = 0
    for lo in range(0, n, slot):
        hi = min(n, lo + slot)
        evs[cur].synchronize()              # the slot about to be refilled has left for the device
        fill(bufs[cur].numpy()[:hi - lo], lo, hi)
        dst[lo:hi].copy_(bufs[cur][:hi - lo], non_blocking=True)
        evs[cur].record()
        cur ^= 1


def _device_column(col, arrow_type, dev):
    """A null-free primitive Arrow column (ChunkedArray) -> one contiguous device tensor.  The chunks are memcpy'd
    back to back into the pinned ring (ring_upload): the only host pass over the column is that memcpy (no
    combine_chunks, no pageable cudaMemcpy of a 64-bit key built in numpy -- the two things that made the pack 42 % of
    the modeler job's wall time in profiles/r2u_e2e_stage_breakdown.log)."""
    import torch
    tdtype = {pa.int64(): torch.int64, pa.int32(): torch.int32, pa.float64(): torch.float64}[arrow_type]
    out = torch.empty(len(col), dtype=tdtype, device=dev)
    pieces, starts = [], [0]
    for ch in col.chunks if isinstance(col, pa.ChunkedArray) else [col]:
        if len(ch) == 0:
            continue
        if pa.types.is_timestamp(ch.type):
            ch = ch.view(pa.int64())
        elif ch.type != arrow_type:
            ch = pc.cast(ch, arrow_type, safe=False)
        pieces.append(ch.to_numpy(zero_copy_only=True).view(np.uint8))
        starts.append(starts[-1] + pieces[-1].size)

    def fill(dst, lo, hi):
        k, o = bisect.bisect_right(starts, lo) - 1, 0
        while o < dst.size:
            a = lo + o - starts[k]
            m = min(dst.size - o, pieces[k].size - a)
            dst[o:o + m] = pieces[k][a:a + m]
            o += m
            k += 1

    ring_upload(out, fill)
    return out


def pack_groups_cuda(table: pa.Table, device=None, keys=("series_id", "dim_id"), ds_col="ds", y_col="y"):
    """GPU version of :func:`pack_groups` (SURVEY 8f-2): the columns go to HBM as they are (32-bit ids and y, 64-bit
    ds) and :func:`pack_device_columns` groups and sorts them there.  ``ds`` / ``y`` stay resident in HBM for
    ``pb200_fit_device``.  Returns a PackedGroups whose ``ds`` / ``y`` are CUDA tensors; ids, offsets and last_ds are
    host numpy arrays.  Null ``y`` rows are dropped exactly as on the host path."""
    import torch
    if table.num_rows == 0:
        return pack_groups(table, keys, ds_col, y_col, pin=False)
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    ds_arr = table[ds_col]
    mult = 1
    if pa.types.is_timestamp(ds_arr.type):
        if ds_arr.null_count:
            raise ValueError("Found NaN in column ds.")
        mult = {"s": 10**9, "ms": 10**6, "us": 10**3, "ns": 1}[ds_arr.type.unit]
    for k in keys[:2]:
        if table[k].null_count:
            raise ValueError(f"group key column {k!r} holds {table[k].null_count} null value(s); every row needs both "
                             f"{keys[0]!r} and {keys[1]!r}")
    ycol = table[y_col]
    integral = pa.types.is_integer(ycol.type)
    y_null = None
    if ycol.null_count:
        y_null = np.asarray(ycol.combine_chunks().is_null().to_numpy(zero_copy_only=False))
        ycol = pc.fill_null(ycol, 0)
    ds_t = _device_column(ds_arr, pa.int64(), dev)
    if mult != 1:
        ds_t *= mult                                       # timestamp[s|ms|us] -> ns, on the device
    k0 = _device_column(table[keys[0]], pa.int32(), dev)
    k1 = _device_column(table[keys[1]], pa.int32(), dev)
    y_t = _device_column(ycol, pa.int32() if integral else pa.float64(), dev)
    return pack_device_columns(k0, k1, ds_t, y_t, y_null)


def pack_device_columns(k0, k1, ds_t, y_t, y_null=None) -> PackedGroups:
    """The device half of :func:`pack_groups_cuda`: int32 series_id / dim_id, int64 ns ds and int32 or float64 y, CUDA
    tensors of one length on one device, in input row order; ``y_null`` marks null y rows (None, a host bool array or
    a CUDA bool tensor).  The sort key is formed on the device and the (series_id, dim_id, ds) sort of the whole frame
    runs on the B200 as two stable radix sorts (``torch.sort`` -- plumbing, not a hand-written kernel; skipped when the
    frame already is in that order, as a hive-partitioned input written per series is).  Float y NaNs count as
    nulls.  The input tensors may be consumed."""
    import torch
    dev = ds_t.device
    if ds_t.numel() == 0:
        z = np.zeros(0, np.int32)
        y_dtype = np.int32 if y_t.dtype == torch.int32 else np.float64
        return PackedGroups(z, z, np.zeros(1, np.int64), np.zeros(0, np.int64), np.zeros(0, y_dtype), np.zeros(0, np.int64),
                            np.zeros(0, np.int64))
    if y_null is not None and not isinstance(y_null, torch.Tensor):
        y_null = torch.from_numpy(np.asarray(y_null, dtype=bool)).to(dev)
    if y_t.is_floating_point():
        nan = torch.isnan(y_t)
        y_null = nan if y_null is None else (y_null | nan)
    # one signed 64-bit sort key: series_id in the high word, dim_id biased by 2^31 in the low word, so that the
    # signed order of the key is the (series_id, dim_id) order of the host path's lexsort for negative ids too
    key = (k0.to(torch.int64) << 32) | (k1.to(torch.int64) + (1 << 31))
    del k0, k1
    in_order = bool(((key[1:] > key[:-1]) | ((key[1:] == key[:-1]) & (ds_t[1:] >= ds_t[:-1]))).all())
    order = None
    if not in_order:
        i1 = torch.argsort(ds_t, stable=True)
        i2 = torch.argsort(key[i1], stable=True)
        order = i1[i2]
        key, ds_t, y_t = key[order], ds_t[order], y_t[order]
    new_grp = torch.ones(key.numel(), dtype=torch.bool, device=dev)
    new_grp[1:] = key[1:] != key[:-1]
    starts = torch.nonzero(new_grp).flatten()
    ends = torch.cat((starts[1:], torch.tensor([key.numel()], device=dev)))
    last_ds = ds_t[ends - 1].cpu().numpy()
    n_rows_in = (ends - starts).cpu().numpy().astype(np.int64)
    gkeys = key[starts].cpu().numpy()
    sid, did = (gkeys >> 32).astype(np.int32), ((gkeys & 0xFFFFFFFF) - (1 << 31)).astype(np.int32)
    if y_null is not None and bool(y_null.any()):
        keep = ~y_null
        if order is not None:
            keep = keep[order]
        grp_id = torch.cumsum(new_grp.to(torch.int64), 0) - 1
        counts = torch.bincount(grp_id[keep], minlength=starts.numel()).cpu().numpy().astype(np.int64)
        ds_t, y_t = ds_t[keep].contiguous(), y_t[keep].contiguous()
    else:
        counts = n_rows_in
    offsets = np.zeros(sid.size + 1, np.int64)
    np.cumsum(counts, out=offsets[1:])
    return PackedGroups(sid, did, offsets, ds_t.contiguous(), y_t.contiguous(), last_ds.astype(np.int64), n_rows_in)
