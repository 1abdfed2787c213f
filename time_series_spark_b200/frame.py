"""Minimal DataFrame stand-in over a pyarrow.Table.

The reference drives its per-series operators through a handful of Spark DataFrame calls
(``groupby(...).apply(udf)`` src/jobs/prophet_modeler.py:139-141, src/jobs/prophet_scorer.py:159-161;
``count``/``columns``/``filter``/``select(...).distinct()``/``collect`` in tests/unit/*.py).
There is no Spark (no JVM) on the B200 path, so this class offers exactly that subset on an
Arrow table; ``groupby(keys).apply(op)`` hands ALL groups to the batched operator at once
instead of one pandas frame per Python worker.

A frame read by the GPU input reader holds its columns in HBM (``device_columns``) and builds the Arrow table only when
a caller asks for it; ``groupby(...).apply(op)`` hands those columns to an operator that takes them directly.
"""
from __future__ import annotations

import re
from dataclasses import dataclass
from typing import List, Sequence

import pyarrow as pa
import pyarrow.compute as pc


@dataclass
class DeviceColumns:
    """The modeler's input frame as CUDA tensors of one length, in row order: int32 series_id / dim_id, int64 ns ds,
    int32 y and its uint8 valid mask (0 = null y)."""
    series_id: object
    dim_id: object
    ds: object
    y: object
    y_valid: object

    def __len__(self) -> int:
        return int(self.ds.shape[0])

    def to_arrow(self) -> pa.Table:
        """(series_id int32, dim_id int32, ds timestamp[ns], y int32 with nulls): the Arrow reader's table."""
        valid = self.y_valid.cpu().numpy().astype(bool)
        return pa.table({
            "series_id": pa.array(self.series_id.cpu().numpy(), pa.int32()),
            "dim_id": pa.array(self.dim_id.cpu().numpy(), pa.int32()),
            "ds": pa.array(self.ds.cpu().numpy(), pa.int64()).cast(pa.timestamp("ns")),
            "y": pa.array(self.y.cpu().numpy(), pa.int32(), mask=None if valid.all() else ~valid),
        })


class Frame:
    def __init__(self, table: pa.Table = None, device_columns: DeviceColumns = None):
        if (table is None) == (device_columns is None):
            raise ValueError("a Frame holds either an Arrow table or device columns")
        self._table = table
        self.device_columns = device_columns

    @property
    def table(self) -> pa.Table:
        if self._table is None:
            self._table = self.device_columns.to_arrow()
        return self._table

    # -- Spark-like surface ------------------------------------------------------------
    @property
    def columns(self) -> List[str]:
        return list(self.table.column_names)

    def count(self) -> int:
        return self.table.num_rows if self._table is not None else len(self.device_columns)

    def select(self, *cols: str) -> "Frame":
        return Frame(self.table.select(list(cols)))

    def distinct(self) -> "Frame":
        if self.table.num_rows == 0:
            return self
        return Frame(self.table.group_by(self.table.column_names).aggregate([]))

    def filter(self, expr: str) -> "Frame":
        """Conjunctions of ``col = <int>`` (all the reference's tests use)."""
        mask = None
        for clause in re.split(r"\s+and\s+", expr.strip(), flags=re.IGNORECASE):
            m = re.fullmatch(r"\s*(\w+)\s*=\s*(-?\d+)\s*", clause)
            if not m:
                raise ValueError(f"unsupported filter clause: {clause!r}")
            c = pc.equal(self.table[m.group(1)], int(m.group(2)))
            mask = c if mask is None else pc.and_(mask, c)
        return Frame(self.table.filter(mask))

    def withColumnRenamed(self, old: str, new: str) -> "Frame":
        return Frame(self.table.rename_columns([new if c == old else c for c in self.table.column_names]))

    def collect(self) -> list:
        cols = [self.table[c].to_pylist() for c in self.table.column_names]
        return [tuple(r) for r in zip(*cols)]

    def groupby(self, *keys: str) -> "GroupedFrame":
        return GroupedFrame(self, list(keys))

    def toPandas(self):
        return self.table.to_pandas()

    def __repr__(self):
        if self._table is None:
            return f"Frame(device columns, rows={len(self.device_columns)})"
        return f"Frame({self.table.schema}, rows={self.table.num_rows})"


class GroupedFrame:
    def __init__(self, frame: Frame, keys: Sequence[str]):
        self.frame, self.keys = frame, list(keys)

    def apply(self, op) -> Frame:
        """``op`` is a batched grouped-map operator (see jobs.prophet_modeler.model_time_series).  A frame that holds
        device columns hands them to an operator with ``apply_device_columns(columns, keys)``."""
        cols = self.frame.device_columns
        if cols is not None and hasattr(op, "apply_device_columns"):
            return Frame(op.apply_device_columns(cols, self.keys))
        if not hasattr(op, "apply_batched"):
            raise TypeError("groupby().apply() needs a batched operator with .apply_batched(table, keys)")
        return Frame(op.apply_batched(self.frame.table, self.keys))
