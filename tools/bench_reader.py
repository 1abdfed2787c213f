"""The modeler's input read + pack on config-#3 trees, Arrow reader vs GPU reader, in one process.
    python tools/bench_reader.py [--series 16000,50000] [--T 1440] [--reps 3] [--work DIR]
Builds each tree with tools/e2e_scaling.py make (under --work, default a temporary directory), warms both readers up
once, then times read_input_dataframe + pack `--reps` times per reader, alternating them.  The page cache cannot be
dropped without changing host settings, so these are WARM reads (the files were just written or read).  Prints one
JSON line per (tree, reader) with the device name and power limit read in the same run."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402  (imported before the timed work)

from e2e_scaling import make  # noqa: E402
from time_series_spark_b200.jobs.prophet_modeler import ProphetModeler, get_context  # noqa: E402
from time_series_spark_b200.pack import pack_device_columns, pack_groups_cuda  # noqa: E402


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power = r.stdout.strip() or "unknown"
    except Exception:
        power = "unknown"
    return name, power


def read_and_pack(cfg):
    job = ProphetModeler(cfg)
    t0 = time.perf_counter()
    frame = job.read_input_dataframe()
    t1 = time.perf_counter()
    c = frame.device_columns
    if c is not None:
        pk = pack_device_columns(c.series_id, c.dim_id, c.ds, c.y, c.y_valid == 0)
    else:
        pk = pack_groups_cuda(frame.table, device=f"cuda:{get_context().device}")
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    return t1 - t0, t2 - t0, frame.count(), pk


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--series", default="16000,50000")
    ap.add_argument("--T", type=int, default=1440)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--work", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_reader.py needs a CUDA device")
    name, power = device_info()
    work = a.work or tempfile.mkdtemp(prefix="bench_reader_")
    try:
        for n in (int(s) for s in a.series.split(",")):
            d = os.path.join(work, f"c3_{n}")
            if not os.path.isdir(os.path.join(d, "input")):
                make(d, n, a.T)
            inp = os.path.join(d, "input")
            nbytes = sum(os.path.getsize(os.path.join(r, f)) for r, _, fs in os.walk(inp) for f in fs)
            cfg = lambda reader: {"io": {"input": inp, "models": "unused", "reader": reader},       # noqa: E731
                                  "model": {"floor": 0, "cap_multiplier": 1.1}}
            times = {"arrow": [], "gpu": []}
            packs = {}
            for rep in range(a.reps + 1):                   # rep 0 warms up both (context, pinned ring, page cache)
                for reader in ("arrow", "gpu"):
                    r, rp, rows, pk = read_and_pack(cfg(reader))
                    packs[reader] = pk
                    if rep:
                        times[reader].append((r, rp))
            h, g = packs["arrow"], packs["gpu"]
            same = (np.array_equal(h.offsets, g.offsets) and np.array_equal(h.series_id, g.series_id)
                    and np.array_equal(h.dim_id, g.dim_id) and bool(torch.equal(h.ds, g.ds)) and bool(torch.equal(h.y, g.y)))
            for reader, ts in times.items():
                read_s = float(np.median([t[0] for t in ts]))
                rp_s = float(np.median([t[1] for t in ts]))
                print(json.dumps({"tree": f"config3 {n} x {a.T}", "reader": reader, "rows": rows, "csv_bytes": nbytes,
                                  "page_cache": "warm", "reps": a.reps, "read_s_median": round(read_s, 4),
                                  "read_plus_pack_s_median": round(rp_s, 4), "read_plus_pack_s_all": [round(t[1], 4) for t in ts],
                                  "rows_per_s": round(rows / rp_s), "csv_GB_per_s": round(nbytes / rp_s / 1e9, 3),
                                  "same_pack_as_arrow": same, "device": name, "power_limit": power}), flush=True)
    finally:
        if a.work is None:
            shutil.rmtree(work, ignore_errors=True)


if __name__ == "__main__":
    main()
