"""The modeler's GPU input reader, without a GPU: the row parser of csrc/csv_reader.cuh (run on the host through
pb200_input_csv_row_host) against pyarrow's parse with the modeler's own options, and the io.reader selection rules."""
import io
import os
import subprocess
import sys

import numpy as np
import pyarrow as pa
import pyarrow.csv as pacsv
import pytest

from time_series_spark_b200 import batched
from time_series_spark_b200.jobs import prophet_modeler as pm

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _arrow_rows(data: bytes):
    """[(dim_id, ds_ns, quantity or None)] as the modeler's Arrow reader parses one file, or None if it raises."""
    fmt = pm.input_csv_format()
    try:
        t = pacsv.read_csv(io.BytesIO(data), read_options=fmt.default_fragment_scan_options.read_options,
                           parse_options=fmt.parse_options,
                           convert_options=fmt.default_fragment_scan_options.convert_options)
    except (pa.ArrowInvalid, ValueError):
        return None
    return list(zip(t["dim_id"].to_pylist(), t["start_time"].cast(pa.int64()).to_pylist(), t["quantity"].to_pylist()))


def _standard_lines(rng, n):
    """Lines inside the parser's grammar: extreme int32 values, 1900..2199, leap days, 0-9 fraction digits, ' ' or 'T',
    LF or CRLF, empty quantities."""
    edge = [0, -1, 1, 2**31 - 1, -2**31, 10, -10, 999999999, 1000000000, -1000000000]
    lo, hi = -2208988800, 7258118399                      # 1900-01-01 .. 2199-12-31 23:59:59 in seconds
    fixed = [-2208988800, 7258118399, 951782400, 951868799, 4107456000, -2082844800 + 59 * 86400, 0, 68169600]
    lines = []
    for i in range(n):
        dim = edge[i % len(edge)] if i % 3 == 0 else int(rng.randint(-2**31, 2**31, dtype=np.int64))
        sec = fixed[i % len(fixed)] if i % 5 == 0 else int(rng.randint(lo, hi + 1))
        ts = str(np.datetime64(sec, "s")).replace("T", "T" if i % 4 == 0 else " ")
        nf = i % 10
        if nf:
            ts += "." + "".join(str(d) for d in rng.randint(0, 10, nf))
        q = "" if i % 7 == 0 else str(edge[i % len(edge)] if i % 2 else int(rng.randint(-2**31, 2**31, dtype=np.int64)))
        end = "\r\n" if i % 6 == 0 else "\n"
        lines.append(f"{dim},{ts},{q}{end}".encode())
    return lines


# outside the grammar: pyarrow reinterprets, tolerates or rejects each of these; the parser must refuse all of them
QUIRKS = [
    b" 5,2001-01-05 11:15:00,3\n", b"5, 2001-01-05 11:15:00,3\n", b"5,2001-01-05 11:15:00, 3\n", b"5,2001-01-05 11:15:00,3 \n",
    b"0x10,2001-01-05 11:15:00,3\n", b"5,2001-01-05 11:15:00,0x10\n",
    b"5,2001-01-05 11:15:00,NA\n", b"5,2001-01-05 11:15:00,null\n", b"5,2001-01-05 11:15:00,N/A\n",
    b"5,2001-01-05 11:15:00,nan\n", b"5,2001-01-05 11:15:00,NaN\n", b"5,2001-01-05 11:15:00,NULL\n",
    b"5,2001-01-05 11:15:00,#N/A\n", b"5,2001-01-05 11:15:00,-nan\n", b"5,2001-01-05 11:15:00,None\n",
    b'"5",2001-01-05 11:15:00,3\n', b'5,"2001-01-05 11:15:00",3\n', b'5,2001-01-05 11:15:00,"3"\n', b'5,2001-01-05 11:15:00,""\n',
    b"\xef\xbb\xbf5,2001-01-05 11:15:00,3\n", b"\n", b"\r\n", b"5,2001-01-05 11:15:00,3\r", b"5,2001-01-05 11:15:00,3\r\r\n",
    b"5,2001-1-5 11:15:00,3\n", b"5,2001-01-5 11:15:00,3\n", b"5,2001-02-29 00:00:00,3\n", b"5,1900-02-29 00:00:00,3\n",
    b"5,2100-02-29 00:00:00,3\n", b"5,2001-04-31 00:00:00,3\n", b"5,2001-01-05 23:59:60,3\n", b"5,2001-01-05  11:15:00,3\n",
    b"5,2001-01-05,3\n", b"5,2001-01-05 11,3\n", b"5,2001-01-05 11:15,3\n", b"5,11:15,3\n", b"5,2001-01-05T11:15,3\n",
    b"+5,2001-01-05 11:15:00,3\n", b"5,2001-01-05 11:15:00,+3\n", b"5.0,2001-01-05 11:15:00,3\n", b"5,2001-01-05 11:15:00,3.0\n",
    b"5,2001-01-05 24:00:00,3\n", b"5,2001-01-05 11:60:00,3\n", b"5,2001-01-05T11:15:00Z,3\n",
    b"5,2001-01-05T11:15:00+01:00,3\n", b"5,2001-01-05 11:15:00.,3\n", b"5,2001-01-05 11:15:00.1234567891,3\n",
    b"5,1899-12-31 23:59:59,3\n", b"5,2200-01-01 00:00:00,3\n", b"5,0001-01-01 00:00:00,3\n", b"5,2001-13-01 00:00:00,3\n",
    b"5,2001-00-10 00:00:00,3\n", b"5,2001-01-00 00:00:00,3\n", b"2147483648,2001-01-05 11:15:00,3\n",
    b"-2147483649,2001-01-05 11:15:00,3\n", b"5,2001-01-05 11:15:00,2147483648\n", b"00000000005,2001-01-05 11:15:00,3\n",
    b",2001-01-05 11:15:00,3\n", b"-,2001-01-05 11:15:00,3\n", b"5,,3\n", b"5,2001-01-05 11:15:00\n",
    b"5,2001-01-05 11:15:00,3,\n", b"5,2001-01-05 11:15:00,3,4\n", b"5;2001-01-05 11:15:00;3\n", b"5,2001/01/05 11:15:00,3\n",
    b"5,2001-01-05 11:15:00,-\n", b"5,2001-01-05 11:15:00,3", b"", b"5,2001-01-05\t11:15:00,3\n",
]


def test_row_parser_refuses_or_matches_pyarrow():
    """Several thousand lines: every accepted line gives exactly pyarrow's (dim_id, ns, quantity / null); every line
    inside the grammar is accepted; every quirk is refused."""
    rng = np.random.RandomState(20261017)
    std = _standard_lines(rng, 4000)
    inside = [b"007,2001-01-05 11:15:00,-0\n", b"-0,2000-02-29 23:59:59.999999999,0010\r\n",
              b"5,1904-02-29T00:00:00.000000001,\n", b"5,2196-02-29 12:00:00,\r\n"]
    # random byte-level damage to standard lines: whatever the parser makes of them must still be pyarrow's answer
    damaged = []
    for i in range(1500):
        b = bytearray(std[i])
        j = int(rng.randint(0, len(b)))
        op = i % 3
        if op == 0:
            b[j] = int(rng.choice(list(b" +-.:,Tx0123456789\r\"")))
        elif op == 1:
            del b[j]
        else:
            b.insert(j, int(rng.choice(list(b" 0-:"))))
        damaged.append(bytes(b))
    accepted = 0
    for line in std + inside + QUIRKS + damaged:
        got = batched.input_csv_row_host(line)
        if got is None:
            continue
        accepted += 1
        assert _arrow_rows(line) == [got], line
    for line in std + inside:
        assert batched.input_csv_row_host(line) is not None, line
    for line in QUIRKS:
        assert batched.input_csv_row_host(line) is None, line
    assert accepted >= len(std) + len(inside)


def _check_tree_accepted(root):
    n = 0
    for d, _, files in os.walk(root):
        for fn in files:
            data = open(os.path.join(d, fn), "rb").read()
            lines = data.splitlines(keepends=True)
            if lines and not lines[-1].endswith(b"\n"):
                lines[-1] += b"\n"                    # the reader appends the missing line end
            got = [batched.input_csv_row_host(l) for l in lines]
            assert None not in got, (fn, lines[got.index(None)])
            assert got == _arrow_rows(data)
            n += len(got)
    return n


def test_generated_and_fixture_inputs_take_the_fast_path(tmp_path, model_input_dir):
    """Every line of the reference's fixture and of tools/e2e_scaling.py's config-#3 trees is inside the grammar."""
    assert _check_tree_accepted(model_input_dir) > 0
    pytest.importorskip("yaml")
    subprocess.run([sys.executable, os.path.join(ROOT, "tools", "e2e_scaling.py"), "make", str(tmp_path / "e2e"), "300", "50"],
                   check=True, capture_output=True)
    assert _check_tree_accepted(tmp_path / "e2e" / "input") == 300 * 50


def _cfg(path, reader):
    return {"io": {"input": path, "models": "unused", "reader": reader}, "model": {"floor": 0, "cap_multiplier": 1.1}}


def test_reader_selection(model_input_dir, monkeypatch):
    """io.reader accepts auto | gpu | arrow; without CUDA, auto reads through Arrow and gpu says why it cannot."""
    import torch
    for bad in ("GPU", "pyarrow", 1):
        with pytest.raises(ValueError):
            pm.ProphetModeler(_cfg(model_input_dir, bad)).read_input_dataframe()
    monkeypatch.setattr(pm, "AUTO_READS_ON_GPU", True)
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    want = pm.ProphetModeler(_cfg(model_input_dir, "arrow")).read_input_dataframe()
    got = pm.ProphetModeler(_cfg(model_input_dir, "auto")).read_input_dataframe()
    assert got.device_columns is None and got.table.equals(want.table) and got.table.schema == want.table.schema
    cfg = _cfg(model_input_dir, None)
    del cfg["io"]["reader"]
    assert pm.ProphetModeler(cfg).read_input_dataframe().table.equals(want.table)
    with pytest.raises(ValueError, match="no CUDA device"):
        pm.ProphetModeler(_cfg(model_input_dir, "gpu")).read_input_dataframe()
