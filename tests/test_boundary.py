"""CPU tests of the drop-in boundary: the reference's plumbing contract (SURVEY.md section 4,
ported from the reference's tests/unit/prophet_modeler_test.py and prophet_scorer_test.py
minus Spark), the packer, the model-record wire format, and the C-ABI exports."""
import ctypes
import os
import re
from datetime import datetime

import numpy as np
import pyarrow as pa
import pytest

from time_series_spark_b200 import _lib as L
from time_series_spark_b200 import batched, model_record
from time_series_spark_b200.frame import Frame
from time_series_spark_b200.jobs.prophet_modeler import MODEL_INPUT_SCHEMA, ProphetModeler
from time_series_spark_b200.jobs.prophet_scorer import ProphetScorer, extract_date, frequency_to_future
from time_series_spark_b200.pack import pack_groups

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- reference tests/unit/prophet_modeler_test.py:52-56 -------------------------------------
def test_read_dataframe(model_input_dir):
    modeler = ProphetModeler({"io": {"input": model_input_dir, "models": "unused"},
                              "model": {"floor": 0, "cap_multiplier": 1.1}})
    spark_input_df = modeler.read_input_dataframe(None)
    assert spark_input_df.columns == ["series_id", "dim_id", "ds", "y"]
    assert spark_input_df.select("series_id").distinct().count() == 1
    assert spark_input_df.select("dim_id").distinct().count() == 2
    assert spark_input_df.count() == 816
    assert [f.name for f in MODEL_INPUT_SCHEMA] == ["series_id", "dim_id", "start_time", "quantity"]
    t = spark_input_df.table
    assert t["series_id"].type == pa.int32() and t["y"].type == pa.int32() and pa.types.is_timestamp(t["ds"].type)
    assert spark_input_df.filter("series_id = 751 and dim_id = 91").count() == 410


# ---- reference tests/unit/prophet_scorer_test.py:55-80 --------------------------------------
def test_convert_forecasts():
    tbl = pa.table({"series_id": pa.array([101], pa.int32()), "dim_id": pa.array([66], pa.int32()),
                    "ds": pa.array([datetime.strptime("2015-07-05 10:15:00", "%Y-%m-%d %H:%M:%S")], pa.timestamp("ns")),
                    "yhat": pa.array([873242], pa.int32())})
    output_df = ProphetScorer.convert_forecasts(Frame(tbl))
    timestamp_regex = re.compile(r"^([0-9]{4})-(1[0-2]|0[1-9])-(3[01]|0[1-9]|[12][0-9])T"
                                 r"(2[0-3]|[01][0-9]):([0-5][0-9]):([0-5][0-9])(\+00:00)$")
    row = output_df.collect()[0]
    assert timestamp_regex.match(row[0])
    assert row[1] == 101
    assert row[2] == 66
    assert row[3] == "2015-07-05"
    assert row[4] == datetime(2015, 7, 5, 10, 15)
    assert row[5] == 873242
    assert output_df.columns == ["created_timestamp", "series_id", "dim_id", "forecast_date",
                                 "forecast_timestamp", "forecast_quantity"]
    assert extract_date(datetime(2015, 7, 5, 10, 15)) == "2015-07-05"


def test_write_forecasts_roundtrip(tmp_path):
    import pyarrow.csv as pacsv
    import pyarrow.dataset as pads
    tbl = pa.table({"series_id": pa.array([1, 1], pa.int32()), "dim_id": pa.array([2, 2], pa.int32()),
                    "ds": pa.array([0, 900 * 10**9], pa.int64()).cast(pa.timestamp("ns")),
                    "yhat": pa.array([5, 6], pa.int32())})
    scorer = ProphetScorer({"io": {"models": "unused", "forecasts": str(tmp_path / "forecasts")},
                            "forecast": {"periods": 2, "frequency": "15min"}})
    scorer.write_forecasts(scorer.convert_forecasts(Frame(tbl)))
    scorer.write_forecasts(scorer.convert_forecasts(Frame(tbl)))      # mode='overwrite'
    back = pads.dataset(str(tmp_path / "forecasts"), format="csv").to_table()
    assert back.column_names == ["created_timestamp", "series_id", "dim_id", "forecast_date",
                                 "forecast_timestamp", "forecast_quantity"]
    assert back.num_rows == 2 and back["forecast_quantity"].to_pylist() == [5, 6]
    assert back["forecast_date"].to_pylist()[0].strftime("%Y-%m-%d") == "1970-01-01" \
        if not isinstance(back["forecast_date"][0].as_py(), str) else back["forecast_date"][0].as_py() == "1970-01-01"


def test_pack_groups_sorts_groups_and_drops_null_y():
    ns = 10**9
    tbl = pa.table({
        "series_id": pa.array([2, 1, 1, 1, 2, 1], pa.int32()),
        "dim_id": pa.array([7, 5, 5, 5, 7, 9], pa.int32()),
        "ds": pa.array([30 * ns, 20 * ns, 10 * ns, 40 * ns, 10 * ns, 5 * ns], pa.int64()).cast(pa.timestamp("ns")),
        "y": pa.array([3, 2, 1, None, 4, 9], pa.int32()),
    })
    pk = pack_groups(tbl, pin=False)
    assert pk.n == 3
    assert pk.series_id.tolist() == [1, 1, 2] and pk.dim_id.tolist() == [5, 9, 7]
    assert pk.offsets.tolist() == [0, 2, 3, 5]
    assert pk.ds.tolist() == [10 * ns, 20 * ns, 5 * ns, 10 * ns, 30 * ns]
    assert pk.y.tolist() == [1, 2, 9, 4, 3] and pk.y.dtype == np.int32
    assert pk.last_ds.tolist() == [40 * ns, 5 * ns, 30 * ns]      # null-y row still anchors the future frame
    assert pk.n_rows_in.tolist() == [3, 1, 2]
    empty = pack_groups(tbl.slice(0, 0), pin=False)
    assert empty.n == 0 and empty.offsets.tolist() == [0]


def test_frame_subset():
    f = Frame(pa.table({"a": [1, 1, 2], "b": [3, 3, 4]}))
    assert f.count() == 3 and f.columns == ["a", "b"]
    assert f.select("a").distinct().count() == 2
    assert f.filter("a = 1 and b = 3").count() == 2
    assert f.withColumnRenamed("a", "c").columns == ["c", "b"]
    with pytest.raises(ValueError):
        f.filter("a > 1")
    with pytest.raises(TypeError):
        f.groupby("a").apply(lambda t: t)


def test_model_record_roundtrip():
    opts = batched.make_options()
    lay = L.get_layout(opts)
    n = 5
    rng = np.random.RandomState(0)
    fb = batched.FittedBatch(rng.randn(n, lay.pstride), rng.randn(n, lay.smax),
                             rng.randint(0, 100, (n, 8)).astype(np.int32), rng.randint(0, 10**15, (n, 2)).astype(np.int64),
                             rng.randn(n, 4), lay.smax, lay.kmax)
    last = rng.randint(0, 10**15, n).astype(np.int64)
    col = model_record.encode(fb, last, opts)
    assert len(col) == n and pa.types.is_binary(col.type)
    tbl = pa.table({"model": col})
    fb2, last2, info = model_record.decode(tbl["model"])
    for a, b in ((fb.params, fb2.params), (fb.tchange, fb2.tchange), (fb.meta_i32, fb2.meta_i32),
                 (fb.meta_i64, fb2.meta_i64), (fb.meta_f64, fb2.meta_f64), (last, last2)):
        assert np.array_equal(a, b)
    assert info == {"logistic": True, "multiplicative": True, "yearly": -1, "weekly": -1, "daily": -1,
                    "n_changepoints": 25}
    with pytest.raises(ValueError):
        model_record.decode(pa.array([b"not a record, e.g. a pickle"], pa.binary()))


def test_frequency_to_future_matches_pandas():
    import pandas as pd
    last = np.array([pd.Timestamp("2002-12-28 21:45:00").value, pd.Timestamp("2021-03-15 23:45:00").value])
    for freq in ("15min", "H", "D", "W", "MS"):
        fut = frequency_to_future(last, 5, freq)
        for i, l in enumerate(last):
            f = pd.offsets.Week() if freq == "W" else ("h" if freq == "H" else freq)   # 'W': prophet_scorer.py:59-62
            ld = pd.Timestamp(int(l))
            dates = pd.date_range(start=ld, periods=6, freq=f)
            dates = dates[dates > ld][:5]
            assert np.array_equal(fut[i], dates.values.astype("datetime64[ns]").astype(np.int64)), freq


def test_make_options_defaults_are_the_reference_constructor():
    o = batched.make_options()
    assert (o.growth, o.multiplicative, o.n_changepoints) == (L.GROWTH_LOGISTIC, 1, 25)   # prophet_modeler.py:65
    assert (o.yearly, o.weekly, o.daily) == (L.SEAS_AUTO,) * 3
    assert (o.max_iter, o.history_size, o.init_alpha, o.tol_rel_grad) == (10000, 5, 1e-3, 1e7)
    with pytest.raises(ValueError):
        batched.make_options(yearly_seasonality=7)
    with pytest.raises(ValueError):
        batched.make_options(growth="flat")


def test_c_abi_exports_every_declared_symbol():
    """The shared library loads without a GPU and exports everything include/prophet_b200.h declares."""
    hdr = open(os.path.join(ROOT, "include", "prophet_b200.h")).read()
    declared = sorted(set(re.findall(r"PB200_API[^;(]*?\b(pb200_\w+)\s*\(", hdr)))
    assert declared == sorted(L.EXPORTS)
    lib = ctypes.CDLL(L.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    o = L.default_options()
    lay = L.get_layout(o)
    assert (lay.smax, lay.kmax, lay.pstride) == (25, 34, 62)
    assert ctypes.sizeof(L.Options) == 128


def test_no_cpu_fallback_without_a_gpu():
    """On a box without CUDA the product path fails loudly instead of computing on the host."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(L.Pb200Error):
        L.Context(0)


def test_tab_chunk_gives_conflict_free_bins():
    """Host arithmetic behind the seasonal-table fit-kernel variants (csrc/fit_kernel.cuh tab_chunk /
    point_pass_tab): lane l owns points [l*chunk, (l+1)*chunk) and in loop step m updates the residual bins
    (l*chunk + 2m) % P and (l*chunk + 2m + 1) % P without atomics -- valid only if those 64 bins are pairwise
    distinct in every step.  Checked exhaustively for the table periods the variants accept."""
    lib = L.load()
    slack = 12                                              # TAB_CHUNK_SLACK: what the planes workspace allows for
    lanes = np.arange(32)
    for P in range(64, 169):
        for T in list(range(2 * P + 1, 2 * P + 70)) + [1440, 1400, 2016, 4321, 10080, 43200]:
            c = lib.pb200_tab_chunk(T, P)
            c0 = -(-T // 32)
            if c < 0:
                continue                                    # no chunk within the slack: prep_kernel keeps the rotation variant
            assert c0 <= c <= c0 + slack
            assert -(-T // c) <= 32                         # still at most 32 active lanes
            for m in (0, 1, c // 2):                        # bins are a rigid shift of step 0's: three steps suffice
                bins = np.concatenate([(lanes * c + 2 * m) % P, (lanes * c + 2 * m + 1) % P])
                assert np.unique(bins).size == 64, (P, T, c, m)
    # the bench workload and the hourly case get a chunk, and it is the documented one
    assert lib.pb200_tab_chunk(1440, 96) == 45
    assert lib.pb200_tab_chunk(1400, 96) == 45              # 44 would collide
    assert lib.pb200_tab_chunk(1440, 168) > 0
    assert lib.pb200_tab_chunk(1440, 65) == -1 or lib.pb200_tab_chunk(1440, 65) >= 45


def test_written_forecast_timestamps_look_like_sparks(tmp_path):
    """Spark's CSV writer prints timestamps as yyyy-MM-dd'T'HH:mm:ss.SSSXXX (reference prophet_scorer.py:147-150
    relies on that default): 2019-01-01T00:00:05.000Z, not nine fractional digits."""
    import re as _re
    tbl = pa.table({"series_id": pa.array([1, 1], pa.int32()), "dim_id": pa.array([2, 2], pa.int32()),
                    "ds": pa.array([1546300805 * 10**9, 1546301705 * 10**9], pa.int64()).cast(pa.timestamp("ns")),
                    "yhat": pa.array([5, 6], pa.int32())})
    scorer = ProphetScorer({"io": {"models": "unused", "forecasts": str(tmp_path / "fc")},
                            "forecast": {"periods": 2, "frequency": "15min"}})
    scorer.write_forecasts(scorer.convert_forecasts(Frame(tbl)))
    lines = open(tmp_path / "fc" / "part-00000.csv").read().strip().split("\n")
    assert lines[0].replace('"', "") == "created_timestamp,series_id,dim_id,forecast_date,forecast_timestamp,forecast_quantity"
    f = lines[1].replace('"', "").split(",")
    assert f[4] == "2019-01-01T00:00:05.000Z" and f[3] == "2019-01-01" and f[5] == "5"
    assert _re.fullmatch(r"\d{4}-\d\d-\d\dT\d\d:\d\d:\d\d\.\d{3}Z", lines[2].replace('"', "").split(",")[4])


def test_big_forecast_frame_is_written_as_parallel_part_files(tmp_path, monkeypatch):
    """A frame above _ROWS_PER_PART rows goes out as several part files written concurrently, timestamps formatted
    through their dictionary: the concatenated rows must be exactly what the single-file path writes."""
    import pyarrow.compute as pc
    from time_series_spark_b200.jobs import prophet_scorer as ps
    rng = np.random.RandomState(1)
    n_models, H = 37, 53
    grid = 1546300805 * 10**9 + 900 * 10**9 * np.arange(H, dtype=np.int64)
    tbl = pa.table({"series_id": pa.array(np.repeat(np.arange(n_models, dtype=np.int32) // 5, H)),
                    "dim_id": pa.array(np.repeat(np.arange(n_models, dtype=np.int32) % 5, H)),
                    "ds": pa.array(np.tile(grid, n_models)).cast(pa.timestamp("ns")),
                    "yhat": pa.array(rng.randint(0, 10**6, n_models * H).astype(np.int32))})
    # the Arrow writer's split: under the default writer (auto) a big frame goes to the GPU formatter where CUDA is present
    cfg = lambda d: {"io": {"models": "unused", "forecasts": str(tmp_path / d)},
                     "forecast": {"periods": H, "frequency": "15min", "writer": "arrow"}}
    frame = ProphetScorer.convert_forecasts(Frame(tbl))
    ProphetScorer(cfg("one")).write_forecasts(frame)
    monkeypatch.setattr(ps, "_ROWS_PER_PART", 300)
    ProphetScorer(cfg("many")).write_forecasts(frame)
    one = open(tmp_path / "one" / "part-00000.csv").read().strip().split("\n")
    parts = sorted(os.listdir(tmp_path / "many"))
    assert len(parts) == -(-n_models * H // 300) and parts[0] == "part-00000-0000.csv"
    many = []
    for i, fn in enumerate(parts):
        lines = open(tmp_path / "many" / fn).read().strip().split("\n")
        assert lines[0] == one[0]                                   # every part file carries the header, as Spark's do
        many += lines[1:]
    assert many == one[1:] and len(many) == n_models * H
    # the dictionary route == pc.strftime: few distinct values, all distinct values, chunked input, empty input
    for arr in (tbl["ds"], pa.chunked_array([tbl["ds"].chunk(0).slice(0, 100), tbl["ds"].chunk(0).slice(100, 0), tbl["ds"].chunk(0).slice(100)]),
                pa.array(np.sort(rng.randint(0, 2**40, 500)).astype(np.int64) * 1000).cast(pa.timestamp("ns")),
                pa.array([], pa.timestamp("ns"))):
        for fmt in ("%Y-%m-%d", "%Y-%m-%dT%H:%M:%SZ"):
            src = pc.cast(arr, pa.timestamp("ms"), safe=False) if "T" in fmt else arr
            got, want = ps._strftime_via_dictionary(src, fmt), pc.strftime(src, format=fmt)
            assert got.to_pylist() == want.to_pylist() and got.type == pa.string()


def test_gpu_writer_eligibility_rules(tmp_path):
    """Which frames write_forecasts hands to the GPU row formatter (forecast.writer = auto) -- decided on the host."""
    from time_series_spark_b200.jobs import prophet_scorer as ps
    H = 8
    mk = lambda ds0: pa.table({"series_id": pa.array(np.zeros(H, np.int32)), "dim_id": pa.array(np.arange(H, dtype=np.int32)),
                               "ds": pa.array(ds0 + 900 * 10**9 * np.arange(H, dtype=np.int64)).cast(pa.timestamp("ns")),
                               "yhat": pa.array(np.arange(H, dtype=np.int32))})
    f = ProphetScorer.convert_forecasts(Frame(mk(1_650_000_000 * 10**9)))
    assert f.forecast_source[1].num_rows == H
    assert ps._gpu_writer_refusal(f, big_only=True) == "small frame"
    why = ps._gpu_writer_refusal(f, big_only=False)
    try:
        import torch
        cuda = torch.cuda.is_available()
    except Exception:
        cuda = False
    assert why == (None if cuda else "no CUDA device")
    assert "convert_forecasts" in ps._gpu_writer_refusal(Frame(f.table), big_only=False)                  # provenance unknown
    old = ProphetScorer.convert_forecasts(Frame(mk(-5 * 86400 * 10**9)))
    assert ps._gpu_writer_refusal(old, big_only=False) == "timestamps before 1970"
    iv = mk(0).append_column("yhat_lower", pa.array(np.zeros(H))).append_column("yhat_upper", pa.array(np.ones(H)))
    assert "standard six" in ps._gpu_writer_refusal(ProphetScorer.convert_forecasts(Frame(iv)), big_only=False)
    with pytest.raises(ValueError):
        ProphetScorer({"io": {"forecasts": str(tmp_path / "x")}, "forecast": {"writer": "fpga"}}).write_forecasts(f)
    if not cuda:                                        # forcing the GPU route without a device fails loudly, no silent fallback
        with pytest.raises(ValueError):
            ProphetScorer({"io": {"forecasts": str(tmp_path / "y")}, "forecast": {"writer": "gpu"}}).write_forecasts(f)
    # the one-row host formatter (the code the kernel runs) against a hand-written row
    from time_series_spark_b200 import batched
    assert batched.forecast_csv_row_host(12, -3, 1_546_300_805_123_456_789, 42, b"2019-01-01T00:00:00+00:00") == \
        b'"2019-01-01T00:00:00+00:00",12,-3,"2019-01-01","2019-01-01T00:00:05.123Z",42\n'


def test_rank_local_files_cover_the_input_once(tmp_path):
    """SURVEY 8e "rank r reads only its row range": the series_id= directories are cut into contiguous,
    byte-balanced ranges, one per rank; together they are the whole input, pairwise disjoint."""
    import pyarrow.dataset as pads
    from time_series_spark_b200.jobs.prophet_modeler import rank_local_files
    root = tmp_path / "in"
    sizes = {}
    for sid in (3, 11, 7, 20, 5, 1):
        d = root / f"series_id={sid}"
        d.mkdir(parents=True)
        rows = 10 * (sid % 4 + 1)
        (d / "a.csv").write_text("".join(f"{sid},2020-01-01 00:{i % 60:02d}:00,{i}\n" for i in range(rows)))
        sizes[sid] = (d / "a.csv").stat().st_size
    part = pads.partitioning(pa.schema([("series_id", pa.int32())]), flavor="hive")
    dset = pads.dataset(str(root), format="csv", partitioning=part)
    for ws in (2, 3, 6):
        got = [rank_local_files(dset, r, ws) for r in range(ws)]
        flat = [p for g in got for p in g]
        assert sorted(flat) == sorted(f.path for f in dset.get_fragments()) and len(set(flat)) == len(flat)
        # contiguous in series_id order
        ids = [[int(p.split("series_id=")[1].split("/")[0]) for p in g] for g in got]
        assert sum(ids, []) == sorted(sizes)
    assert rank_local_files(dset, 0, 7) is None        # fewer directories than ranks: caller shards the groups instead


def test_null_group_key_is_refused():
    from time_series_spark_b200.pack import pack_groups
    tbl = pa.table({"series_id": pa.array([1, 1], pa.int32()), "dim_id": pa.array([2, None], pa.int32()),
                    "ds": pa.array([0, 1], pa.int64()).cast(pa.timestamp("ns")), "y": pa.array([1, 2], pa.int32())})
    with pytest.raises(ValueError, match="null"):
        pack_groups(tbl, pin=False)


def test_fbprophet_pickle_importer_says_why_it_cannot_run_here():
    """The reference's models are pickled Prophet objects; importing them needs fbprophet itself (absent here)."""
    from time_series_spark_b200 import model_record
    try:
        import fbprophet  # noqa: F401
        pytest.skip("fbprophet is importable: the importer can actually run")
    except ImportError:
        pass
    try:
        import prophet  # noqa: F401
        pytest.skip("prophet is importable")
    except ImportError:
        pass
    with pytest.raises(ImportError, match="fbprophet"):
        model_record.from_fbprophet_pickle([b"not a pickle"])
