"""B200 drop-in for the reference's src/jobs/prophet_modeler.py.

Same names and contracts -- ``MODEL_INPUT_SCHEMA``, ``model_time_series(config)``,
``ProphetModeler(config).read_input_dataframe / persist_models``, ``ProphetModeler.model`` --
same YAML keys (``io.input``, ``io.models``, ``model.floor``, ``model.cap_multiplier``), same
header-less hive-partitioned CSV input and the same 5-column models table
``(series_id, dim_id, floor float32, cap float32, model binary)``.  What changes is the
engine: ``groupby('series_id','dim_id').apply(model_time_series(config))`` is ONE batched GPU
call over all groups (libprophet_b200.so) instead of one fbprophet/Stan fit per Spark task.
There is no Spark and no CPU fallback; ``spark`` arguments are accepted and ignored.

Optional keys beyond the reference (defaults reproduce prophet_modeler.py:65 exactly):
``model.growth``, ``model.seasonality_mode``, ``model.yearly_seasonality``,
``model.weekly_seasonality``, ``model.daily_seasonality``, ``model.n_changepoints``,
``model.changepoint_range``, ``model.changepoint_prior_scale``, ``model.seasonality_prior_scale``.
"""
from __future__ import annotations

import glob
import logging
import os
import time

import numpy as np
import pyarrow as pa
import pyarrow.csv as pacsv
import pyarrow.dataset as pads
import pyarrow.parquet as pq

from .. import _lib as L
from .. import batched, model_record
from .. import dist as pdist
from .. import csv_input
from ..frame import DeviceColumns, Frame
from ..pack import pack_device_columns, pack_groups_cuda

# reference prophet_modeler.py:12-17 (Spark StructType -> Arrow)
MODEL_INPUT_SCHEMA = pa.schema([
    pa.field("series_id", pa.int32(), True),
    pa.field("dim_id", pa.int32(), True),
    pa.field("start_time", pa.timestamp("ns"), True),
    pa.field("quantity", pa.int32(), True),
])

# reference prophet_modeler.py:32-38
MODEL_OUTPUT_SCHEMA = pa.schema([
    pa.field("series_id", pa.int32(), True),
    pa.field("dim_id", pa.int32(), True),
    pa.field("floor", pa.float32(), True),
    pa.field("cap", pa.float32(), True),
    pa.field("model", pa.binary(), True),
])

# Whether io.reader = auto takes the GPU reader.  It does so only once a measurement on the B200
# (tools/bench_reader.py) shows it faster than Arrow on the 16 000-series config-#3 tree; that run has not been made yet.
AUTO_READS_ON_GPU = False

_contexts = {}


def get_context(device=None) -> L.Context:
    """One pb200 context per (process, device); LOCAL_RANK picks the device under torchrun."""
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    if device not in _contexts:
        _contexts[device] = L.Context(device)
    return _contexts[device]


def options_from_config(config) -> L.Options:
    m = dict(config.get("model", {}) or {})
    return batched.make_options(
        growth=m.get("growth", "logistic"),
        seasonality_mode=m.get("seasonality_mode", "multiplicative"),
        yearly_seasonality=m.get("yearly_seasonality", "auto"),
        weekly_seasonality=m.get("weekly_seasonality", "auto"),
        daily_seasonality=m.get("daily_seasonality", "auto"),
        n_changepoints=m.get("n_changepoints", 25),
        changepoint_range=m.get("changepoint_range", 0.8),
        changepoint_prior_scale=m.get("changepoint_prior_scale", 0.05),
        seasonality_prior_scale=m.get("seasonality_prior_scale", 10.0),
    )


class _ModelTimeSeriesOp:
    """Batched GROUPED_MAP operator: all (series_id, dim_id) groups in one GPU launch."""

    def __init__(self, config):
        self.config = config

    def apply_batched(self, table: pa.Table, keys) -> pa.Table:
        execution_time = time.time()
        ctx = self._start(keys)
        # upload, then group + sort on the GPU (two radix sorts), ds / y stay in HBM for the fit
        return self._fit_packed(pack_groups_cuda(table, device=f"cuda:{ctx.device}"), execution_time)

    def apply_device_columns(self, cols: DeviceColumns, keys) -> pa.Table:
        """The same for a frame the GPU input reader left in HBM: no copy back to the host and up again."""
        execution_time = time.time()
        self._start(keys)
        return self._fit_packed(pack_device_columns(cols.series_id, cols.dim_id, cols.ds, cols.y, cols.y_valid == 0),
                                execution_time)

    @staticmethod
    def _start(keys) -> L.Context:
        if list(keys) != ["series_id", "dim_id"]:
            raise ValueError("model_time_series groups by ('series_id', 'dim_id')")
        ctx = get_context()
        import torch
        torch.cuda.set_device(ctx.device)
        return ctx

    def _fit_packed(self, pk, execution_time: float) -> pa.Table:
        import torch
        floor = self.config["model"]["floor"]
        cap_multiplier = self.config["model"]["cap_multiplier"]
        ctx = get_context()
        torch.cuda.synchronize()
        t_pack = time.time()
        rank, ws, _ = pdist.world()
        if ws > 1 and not getattr(self, "rank_local_input", False):
            # the table holds EVERY group (the caller did not read rank-locally): this rank fits its contiguous,
            # row-balanced shard of them
            lo, hi = pdist.shard_bounds(pk.offsets, ws)[rank]
            pk = pk.take(lo, hi)
        if pk.n == 0:
            return MODEL_OUTPUT_SCHEMA.empty_table()
        opts = options_from_config(self.config)
        print(f"Modeling {pk.n} series with {int(pk.offsets[-1])} modeling rows")
        # fbprophet raises ValueError (task failure, not RuntimeError) for < 2 rows:
        # keep that observable behaviour (prophet_modeler.py:81 only catches RuntimeError)
        def _who(mask):
            i = int(np.flatnonzero(mask)[0])
            return (f" (first offender: series_id {int(pk.series_id[i])}, dim_id {int(pk.dim_id[i])}; "
                    f"{int(np.count_nonzero(mask))} group(s) in all)")

        short = np.diff(pk.offsets) < 2
        if np.any(short):
            raise ValueError("Dataframe has less than 2 non-NaN rows." + _who(short))
        fitted = batched.fit_batch_device(ctx, opts, pk.ds.contiguous(), pk.y.contiguous(), pk.offsets,
                                          float(floor), float(cap_multiplier)).to_host()
        t_fit = time.time()
        status = fitted.meta_i32[:, 4]
        if np.any(status == L.ST_CAP_LE_FLOOR):
            raise ValueError("cap must be greater than floor (which defaults to 0)." + _who(status == L.ST_CAP_LE_FLOOR))
        if np.any(status == L.ST_BAD_INPUT):
            raise ValueError("Found non-finite y or a zero time span in a series." + _who(status == L.ST_BAD_INPUT))
        ok = status >= 0
        for i in np.flatnonzero(~ok):
            # reference: RuntimeError -> print + empty frame (prophet_modeler.py:81-85)
            print(f"Runtime error (solver status {int(status[i])}) for series_id: {int(pk.series_id[i])}, "
                  f"dim_id: {int(pk.dim_id[i])}")
        blobs = model_record.encode(fitted, pk.last_ds, opts)
        cap64 = fitted.meta_f64[:, 2]
        out = pa.table({
            "series_id": pa.array(pk.series_id, pa.int32()),
            "dim_id": pa.array(pk.dim_id, pa.int32()),
            "floor": pa.array(np.full(pk.n, floor, dtype=np.float32), pa.float32()),
            "cap": pa.array(cap64.astype(np.float32), pa.float32()),   # FloatType column, prophet_modeler.py:36
            "model": blobs,
        })
        if not ok.all():
            out = out.filter(pa.array(ok))
        # wall time per stage of the last call (tools/e2e_scaling.py reports them): upload + group + sort, GPU fit + D2H, encode
        self.last_timings = {"pack_s": t_pack - execution_time, "fit_s": t_fit - t_pack, "encode_s": time.time() - t_fit}
        print(f"Output df {out.num_rows} models trained in {time.time() - execution_time}")
        return out

    def __call__(self, pdf):
        """Per-group form of the UDF (one pandas frame in, one-row frame out), for callers that
        still iterate groups themselves."""
        tbl = pa.Table.from_pandas(pdf[["series_id", "dim_id", "ds", "y"]], preserve_index=False)
        return self.apply_batched(tbl, ["series_id", "dim_id"]).to_pandas()


def rank_local_files(dset, rank: int, world_size: int):
    """Files of the hive-partitioned input this rank reads: the ``series_id=`` directories in ascending id order,
    cut into ``world_size`` contiguous ranges of (nearly) equal bytes.  Returns None when there are fewer
    directories than ranks (the caller then reads everything and shards the packed groups instead)."""
    by_sid = {}
    for f in dset.get_fragments():
        sid = pads.get_partition_keys(f.partition_expression).get("series_id")
        if sid is None:
            return None
        try:
            size = os.path.getsize(f.path)
        except OSError:
            size = 1
        ent = by_sid.setdefault(int(sid), [0, []])
        ent[0] += max(size, 1)
        ent[1].append(f.path)
    sids = sorted(by_sid)
    if len(sids) < world_size:
        return None
    sizes = np.array([by_sid[s][0] for s in sids], dtype=np.int64)
    offs = np.concatenate(([0], np.cumsum(sizes)))
    lo, hi = pdist.shard_bounds(offs, world_size)[rank]
    return [p for s in sids[lo:hi] for p in sorted(by_sid[s][1])]


def input_csv_format() -> pads.CsvFileFormat:
    """How the Arrow reader parses one input file: header-less ``dim_id,start_time,quantity`` at the types of
    MODEL_INPUT_SCHEMA."""
    names = [f.name for f in MODEL_INPUT_SCHEMA if f.name != "series_id"]
    return pads.CsvFileFormat(
        read_options=pacsv.ReadOptions(column_names=names),
        convert_options=pacsv.ConvertOptions(
            column_types={f.name: f.type for f in MODEL_INPUT_SCHEMA if f.name != "series_id"},
            timestamp_parsers=["%Y-%m-%d %H:%M:%S", pacsv.ISO8601]))


def model_time_series(config):
    """Model time series per dimensions (series_id, dim_id)  -- reference prophet_modeler.py:22-87."""
    return _ModelTimeSeriesOp(config)


class ProphetModeler:
    """Create models to forecast quantities (reference prophet_modeler.py:90-143)."""

    def __init__(self, config, logger=None):
        self.logger = logger or logging.getLogger(self.__class__.__name__)
        self.config = config

    def read_input_dataframe(self, spark=None) -> Frame:
        """Header-less CSV ``dim_id,timestamp,quantity`` under hive dirs ``series_id=<int>/``
        (reference :102-116; fixture tests/fixtures/model-input).  Returns columns
        series_id, dim_id, ds, y.

        ``io.reader`` picks the parser: ``arrow`` (pyarrow on the host), ``gpu`` (csrc/csv_reader.cuh; raises
        ValueError for an input it does not take) or ``auto`` (the default: the GPU reader when AUTO_READS_ON_GPU and
        CUDA is usable, else -- and for any input the GPU reader does not take -- Arrow).  Both give the same table."""
        reader = (self.config["io"].get("reader") or "auto")
        if reader not in ("auto", "gpu", "arrow"):
            raise ValueError("io.reader must be 'auto', 'gpu' or 'arrow'")
        threads = pdist.size_host_pools()   # pyarrow threads = this rank's share of the lease, not os.cpu_count()
        path = self.config["io"]["input"]
        part = pads.partitioning(pa.schema([("series_id", pa.int32())]), flavor="hive")
        fmt = input_csv_format()
        dset = pads.dataset(path, format=fmt, partitioning=part, exclude_invalid_files=False,
                            ignore_prefixes=[".", "_"])
        # Rank-local ingestion (SURVEY 8e): a group never spans two ``series_id=`` directories, so under torchrun each
        # rank parses, uploads and sorts only its own contiguous, byte-balanced range of directories -- the
        # counterpart of Spark tasks reading their own input splits.  With fewer directories than ranks every
        # rank reads everything and the groups are range-sharded after the pack instead.
        rank, ws, _ = pdist.world()
        self.rank_local_input = False
        if ws > 1:
            mine = rank_local_files(dset, rank, ws)
            if mine is not None:
                self.rank_local_input = True
                if not mine:
                    empty = pa.schema([("series_id", pa.int32()), ("dim_id", pa.int32()), ("ds", pa.timestamp("ns")),
                                       ("y", pa.int32())]).empty_table()
                    return Frame(empty)
                dset = pads.dataset(mine, format=fmt, partitioning=part, partition_base_dir=path,
                                    exclude_invalid_files=False)
        if reader == "gpu" or (reader == "auto" and AUTO_READS_ON_GPU):
            cols, why = csv_input.read_device(dset, get_context, threads)
            if cols is not None:
                return Frame(device_columns=cols)
            if reader == "gpu":
                raise ValueError("io.reader = 'gpu' cannot read this input: " + why)
            print(f"Reading the input with Arrow: {why}")
        tbl = dset.to_table(columns=["series_id", "dim_id", "start_time", "quantity"])
        tbl = tbl.rename_columns(["series_id", "dim_id", "ds", "y"])
        return Frame(tbl)

    def persist_models(self, model_df: Frame):
        """Parquet, mode='overwrite' (reference :118-125); one part file per writer."""
        out = self.config["io"]["models"]
        rank = pdist.world()[0]
        pdist.prepare_output_dir(out)
        pq.write_table(model_df.table, os.path.join(out, f"part-{rank:05d}.parquet"))

    @staticmethod
    def model(spark_session, config):
        """Create the trained time series models (reference :127-143)."""
        pdist.init_process_group()          # no-op unless launched by torchrun with WORLD_SIZE > 1
        scorer = ProphetModeler(config)
        input_df = scorer.read_input_dataframe(spark_session)
        op = model_time_series(scorer.config)
        op.rank_local_input = getattr(scorer, "rank_local_input", False)
        model_df = input_df.groupby("series_id", "dim_id").apply(op)
        scorer.persist_models(model_df)
