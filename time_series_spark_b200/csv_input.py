"""The modeler's input CSV read on the GPU (``io.reader``: auto | gpu | arrow).

The files of the hive-partitioned input (``series_id=<int>/``, header-less ``dim_id,timestamp,quantity``) are read by
a thread pool straight into the pinned staging ring of :mod:`pack` and copied into one device byte buffer; the kernels
of csrc/csv_reader.cuh split it into rows and parse them, so ``ds`` and ``y`` land in HBM where the pack and the fit
want them.  The row parser accepts a strict grammar (include/prophet_b200.h); pyarrow accepts much more (padded,
quoted or hexadecimal fields, null tokens, lenient dates, blank lines, a BOM).  Whatever the parser refuses, and inputs
it is not written for, make :func:`read_device` return the reason instead of columns, and the caller reads the input
with pyarrow as before, so the result is always Arrow's.
"""
from __future__ import annotations

import bisect
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pyarrow.dataset as pads

from . import batched
from .frame import DeviceColumns
from .pack import ring_upload

# extensions Arrow decompresses on the fly: the device parser reads raw bytes only
_COMPRESSED = (".gz", ".bz2", ".lz4", ".zst", ".zstd", ".br", ".snappy", ".xz", ".lzo", ".z", ".zip")
# the read (text, row ends, five columns: ~2 B of HBM per input byte) and the pack's sort after it must fit this share
# of the free device memory
_DEVICE_BYTES_PER_INPUT_BYTE = 4
_FREE_FRACTION = 0.5
_READ_PIECE = 1 << 20           # bytes per read job of the thread pool


def input_files(dset: pads.Dataset):
    """[(path, size, series_id)] of the dataset's files in its order (the row order of ``dset.to_table()``), or the
    reason the device reader does not take them."""
    files = []
    for f in dset.get_fragments():
        sid = pads.get_partition_keys(f.partition_expression).get("series_id")
        if sid is None:
            return f"{f.path} has no series_id partition key"
        if not -2**31 <= int(sid) < 2**31:
            return f"{f.path}: series_id {sid} is outside int32"
        if f.path.lower().endswith(_COMPRESSED):
            return f"{f.path} is compressed"
        size = os.path.getsize(f.path)
        if size == 0:
            return f"{f.path} is empty"
        files.append((f.path, size, int(sid)))
    if not files:
        return "no input files"
    return files


def _read_exact(path: str, offset: int, dst) -> None:
    with open(path, "rb", buffering=0) as fh:
        fh.seek(offset)
        view = memoryview(dst)
        while len(view):
            n = fh.readinto(view)
            if not n:
                raise OSError(f"{path} became shorter while it was read")
            view = view[n:]


def _ends_in_newline(path: str) -> bool:
    with open(path, "rb", buffering=0) as fh:
        fh.seek(-1, os.SEEK_END)
        return fh.read(1) == b"\n"


def read_device(dset: pads.Dataset, get_context, threads: int):
    """(DeviceColumns, None) for the dataset's rows in ``dset.to_table()`` order, on the device of the pb200 context
    ``get_context()`` returns (called only when CUDA is usable), or (None, reason) when the device reader does not take
    this input."""
    try:
        import torch
        if not torch.cuda.is_available():
            return None, "no CUDA device"
    except Exception:
        return None, "no CUDA device"
    files = input_files(dset)
    if isinstance(files, str):
        return None, files
    paths = [p for p, _, _ in files]
    ctx = get_context()
    with ThreadPoolExecutor(max_workers=max(1, threads)) as pool:
        newline = list(pool.map(_ends_in_newline, paths))
        # file k occupies [starts[k], starts[k] + size) of the buffer, followed by a '\n' when it does not end in one
        sizes = np.array([s for _, s, _ in files], np.int64)
        spans = sizes + np.logical_not(newline)
        starts = np.concatenate(([0], np.cumsum(spans)))
        total = int(starts[-1])
        torch.cuda.set_device(ctx.device)
        dev = torch.device("cuda", ctx.device)
        free = torch.cuda.mem_get_info(dev)[0]
        if _DEVICE_BYTES_PER_INPUT_BYTE * total > _FREE_FRACTION * free:
            return None, f"{total} bytes of input do not fit {_FREE_FRACTION:.0%} of the free device memory"
        text = torch.empty(-(-total // 16) * 16, dtype=torch.uint8, device=dev)
        text[total:].zero_()
        start_list = starts.tolist()

        def fill(dst, lo, hi):
            jobs = []
            k = bisect.bisect_right(start_list, lo) - 1
            while k < len(files) and start_list[k] < hi:
                a, e = max(lo, start_list[k]), min(hi, start_list[k] + int(sizes[k]))
                for p in range(a, e, _READ_PIECE):
                    q = min(e, p + _READ_PIECE)
                    jobs.append(pool.submit(_read_exact, paths[k], p - start_list[k], dst[p - lo:q - lo]))
                pad = start_list[k] + int(sizes[k])
                if not newline[k] and lo <= pad < hi:
                    dst[pad - lo] = 10
                k += 1
            for j in jobs:
                j.result()

        ring_upload(text[:total], fill)
    file_start = torch.from_numpy(starts[:-1].copy()).to(dev)
    file_sid = torch.tensor([s for _, _, s in files], dtype=torch.int32).to(dev)
    sid, did, ds, qty, valid, row_end, n_bad, first = batched.parse_input_csv_device(ctx, text, total, file_start, file_sid)
    if n_bad:
        s = int(row_end[first - 1]) if first else 0
        e = int(row_end[first])
        k = bisect.bisect_right(start_list, s) - 1
        line = bytes(text[s:min(e, s + 80)].cpu().numpy())
        return None, (f"{n_bad} row(s) outside the strict grammar, the first at byte {s - start_list[k]} of {paths[k]}: "
                      f"{line!r}")
    return DeviceColumns(sid, did, ds, qty, valid), None
