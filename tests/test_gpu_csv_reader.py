"""The modeler's GPU input reader on a B200: the table it gives equals the Arrow reader's, table for table, the pack from
its device columns equals the host pack, inputs it does not take fall back to Arrow (or are refused under
io.reader = gpu), and the modeler job writes the same models either way.  io.reader = auto must give Arrow's table
whichever reader it takes."""
import gzip
import os

import numpy as np
import pyarrow.dataset as pads
import pytest

from time_series_spark_b200 import csv_input, pack
from time_series_spark_b200.jobs import prophet_modeler as pm

pytestmark = pytest.mark.gpu


def _cfg(path, reader, models="unused"):
    return {"io": {"input": str(path), "models": str(models), "reader": reader}, "model": {"floor": 0, "cap_multiplier": 1.1}}


def _read(path, reader):
    """The frame, or the exception the read raised."""
    try:
        return pm.ProphetModeler(_cfg(path, reader)).read_input_dataframe()
    except Exception as exc:              # noqa: BLE001 -- compared by type below
        return exc


def _gpu_equals_arrow(path):
    want = _read(path, "arrow").table
    got = _read(path, "gpu")
    assert got.device_columns is not None and got.count() == want.num_rows
    assert got.table.schema == want.schema and got.table.equals(want)
    auto = _read(path, "auto")
    assert (auto.device_columns is not None) == pm.AUTO_READS_ON_GPU and auto.table.equals(want)
    return got, want


def _write(path, text: bytes):
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "wb") as f:
        f.write(text)


def _synthetic_tree(root, rng, rows_per_file=(1, 57, 300)):
    """series_id directories that sort differently as text and as numbers, several files per directory, files with and
    without a trailing line end, CRLF files, null quantities, 'T' separators and fractions."""
    k = 0
    for sid in (-12, -3, 0, 2, 7, 10, 100, 2147483647):
        for j, n in enumerate(rows_per_file):
            lines = []
            for i in range(n):
                sec = int(rng.randint(-2208988800, 7258118399))
                ts = str(np.datetime64(sec, "s")).replace("T", "T" if (i + k) % 5 == 0 else " ")
                if (i + k) % 7 == 0:
                    ts += "." + str(int(rng.randint(0, 10**6))).zfill(6)
                q = "" if (i + k) % 11 == 0 else str(int(rng.randint(-2**31, 2**31, dtype=np.int64)))
                lines.append(f"{int(rng.randint(-50, 50))},{ts},{q}")
            end = "\r\n" if k % 3 == 1 else "\n"
            text = end.join(lines) + ("" if k % 4 == 2 else end)
            _write(os.path.join(root, f"series_id={sid}", f"part-{j}.csv"), text.encode())
            k += 1
    return root


def test_fixture_tree(model_input_dir):
    got, want = _gpu_equals_arrow(model_input_dir)
    assert want.num_rows > 0
    # the frame surface builds the table on first use
    assert got.columns == ["series_id", "dim_id", "ds", "y"]
    assert got.filter("series_id = 751 and dim_id = 91").count() == _read(model_input_dir, "arrow").filter(
        "series_id = 751 and dim_id = 91").count()
    assert got.collect()[:5] == _read(model_input_dir, "arrow").collect()[:5]
    assert got.toPandas().equals(want.to_pandas())


def test_synthetic_tree(tmp_path):
    root = _synthetic_tree(str(tmp_path / "in"), np.random.RandomState(1))
    got, want = _gpu_equals_arrow(root)
    assert want["y"].null_count > 0
    sids = want["series_id"].to_numpy()
    assert list(dict.fromkeys(sids.tolist())) == [-12, -3, 0, 10, 100, 2, 2147483647, 7]     # Arrow's (path) order


def test_file_bigger_than_a_ring_slot(tmp_path, monkeypatch):
    monkeypatch.setattr(pack, "_SLOT_BYTES", 4096)
    monkeypatch.setattr(pack, "_slots", {})
    monkeypatch.setattr(csv_input, "_READ_PIECE", 1000)
    root = _synthetic_tree(str(tmp_path / "in"), np.random.RandomState(2), rows_per_file=(3000, 1, 700))
    assert max(os.path.getsize(os.path.join(d, f)) for d, _, fs in os.walk(root) for f in fs) > 20 * 4096
    _gpu_equals_arrow(root)


@pytest.mark.parametrize("tree", ["fixture", "synthetic"])
def test_pack_from_device_columns(tree, tmp_path, model_input_dir):
    root = model_input_dir if tree == "fixture" else _synthetic_tree(str(tmp_path / "in"), np.random.RandomState(3))
    frame = _read(root, "gpu")
    c = frame.device_columns
    g = pack.pack_device_columns(c.series_id, c.dim_id, c.ds, c.y, c.y_valid == 0)
    h = pack.pack_groups(_read(root, "arrow").table, pin=False)
    assert g.on_device and not h.on_device
    assert np.array_equal(h.series_id, g.series_id) and np.array_equal(h.dim_id, g.dim_id)
    assert np.array_equal(h.offsets, g.offsets) and np.array_equal(h.last_ds, g.last_ds)
    assert np.array_equal(h.n_rows_in, g.n_rows_in)
    assert np.array_equal(h.ds, g.ds.cpu().numpy()) and np.array_equal(h.y, g.y.cpu().numpy())


@pytest.mark.parametrize("case", ["quirk_row", "arrow_error_row", "gzip_file", "empty_file", "no_partition_key"])
def test_fallback(case, tmp_path, monkeypatch):
    """An input the GPU reader does not take: auto gives Arrow's table or raises Arrow's exception; gpu raises ValueError."""
    monkeypatch.setattr(pm, "AUTO_READS_ON_GPU", True)
    root = str(tmp_path / "in")
    good = b"5,2001-01-05 11:15:00,3\n6,2001-01-05 11:30:00,4\n"
    _write(os.path.join(root, "series_id=1", "a.csv"), good)
    if case == "quirk_row":
        _write(os.path.join(root, "series_id=2", "a.csv"), good + b"7, 2001-01-05 11:45:00,NA\n")
    elif case == "arrow_error_row":
        _write(os.path.join(root, "series_id=2", "a.csv"), good + b"+7,2001-01-05 11:45:00,5\n")
    elif case == "gzip_file":
        _write(os.path.join(root, "series_id=2", "b.csv.gz"), gzip.compress(good))
    elif case == "empty_file":
        _write(os.path.join(root, "series_id=2", "b.csv"), b"")
    else:
        _write(os.path.join(root, "loose.csv"), good)
    want = _read(root, "arrow")
    got = _read(root, "auto")
    if isinstance(want, Exception):
        assert type(got) is type(want), (got, want)
    else:
        assert got.device_columns is None and got.table.equals(want.table)
    with pytest.raises(ValueError, match="io.reader = 'gpu' cannot read this input"):
        pm.ProphetModeler(_cfg(root, "gpu")).read_input_dataframe()


@pytest.mark.parametrize("tree", ["fixture", "config3"])
def test_modeler_job_writes_the_same_models(tree, tmp_path, model_input_dir):
    if tree == "fixture":
        root = model_input_dir
    else:
        import subprocess
        import sys
        pytest.importorskip("yaml")
        repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        subprocess.run([sys.executable, os.path.join(repo, "tools", "e2e_scaling.py"), "make", str(tmp_path / "e2e"), "400", "300"],
                       check=True, capture_output=True)
        root = str(tmp_path / "e2e" / "input")
    out = {}
    for reader in ("gpu", "auto", "arrow"):
        pm.ProphetModeler.model(None, _cfg(root, reader, tmp_path / f"models_{reader}"))
        out[reader] = pads.dataset(str(tmp_path / f"models_{reader}"), format="parquet").to_table()
    assert out["gpu"].num_rows > 0 and out["gpu"].equals(out["arrow"]) and out["auto"].equals(out["arrow"])
