"""Modeler job end to end on a config-#3-shaped hive-partitioned CSV, timed per stage, for 1..N ranks (SURVEY 8e:
"rank r reads only its row range").  Usage:
    python tools/e2e_scaling.py make <dir> <n_series> [T]                 # write the input once
    python -m torch.distributed.run --nproc-per-node N ... tools/e2e_scaling.py run <dir> [auto|gpu|arrow]
`run` reads the input with the given io.reader (default: the config's) and prints one JSON line on rank 0: wall time
of read / fit (pack + GPU fit + encode) / write, max over ranks, and what each rank read."""
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np


def make(d, n, T=1440):
    import pyarrow as pa
    import pyarrow.compute as pc
    import pyarrow.csv as pacsv
    import yaml
    from time_series_spark_b200 import synth
    inp = os.path.join(d, "input")
    t0 = time.time()
    per = 100                                   # series per series_id directory (config #3: series_id = i // 100)
    for lo in range(0, n, 2000):
        b = synth.config3(n=n, T=T, lo=lo, hi=min(n, lo + 2000))
        ts = pc.strftime(pa.array(b.ds, pa.int64()).cast(pa.timestamp("ns")).cast(pa.timestamp("s")), format="%Y-%m-%d %H:%M:%S")
        dim = np.repeat(b.dim_id, np.diff(b.offsets))
        for sid in np.unique(b.series_id):
            sel = np.flatnonzero(b.series_id == sid)
            a, e = int(b.offsets[sel[0]]), int(b.offsets[sel[-1] + 1])
            p = os.path.join(inp, f"series_id={sid}")
            os.makedirs(p, exist_ok=True)
            tbl = pa.table({"dim_id": pa.array(dim[a:e], pa.int32()), "ts": ts.slice(a, e - a), "q": pa.array(b.y[a:e], pa.int32())})
            pacsv.write_csv(tbl, os.path.join(p, "part-0.csv"), write_options=pacsv.WriteOptions(include_header=False, quoting_style="none"))
    yaml.safe_dump({"io": {"input": inp, "models": os.path.join(d, "models")},
                    "model": {"floor": 0, "cap_multiplier": 1.1}}, open(os.path.join(d, "modeler.yaml"), "w"))
    print(f"wrote {n} series x {T} points under {inp} in {time.time() - t0:.1f} s")


def run(d, reader=None):
    import torch
    import yaml
    from time_series_spark_b200 import dist as pdist
    from time_series_spark_b200.jobs.prophet_modeler import ProphetModeler, model_time_series
    cfg = yaml.safe_load(open(os.path.join(d, "modeler.yaml")))
    if reader:
        cfg["io"]["reader"] = reader
    pdist.init_process_group()
    rank, ws, local = pdist.world()
    torch.cuda.set_device(local)
    job = ProphetModeler(cfg)
    stages = {}
    for rep in range(2):                        # rep 0 warms up (CUDA context, page cache, pinned pools)
        pdist.barrier()
        t0 = time.perf_counter()
        df = job.read_input_dataframe()
        t1 = time.perf_counter()
        op = model_time_series(cfg)
        op.rank_local_input = getattr(job, "rank_local_input", False)
        models = df.groupby("series_id", "dim_id").apply(op)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        job.persist_models(models)
        pdist.barrier()
        t3 = time.perf_counter()
        stages = {"read_s": t1 - t0, "fit_s": t2 - t1, "write_s": t3 - t2, "total_s": t3 - t0,
                  "rows_read": df.count(), "models": models.count()}
        stages.update({"op_" + k: v for k, v in getattr(op, "last_timings", {}).items()})
    keys = ("read_s", "fit_s", "write_s", "total_s", "op_pack_s", "op_fit_s", "op_encode_s")
    vals = torch.tensor([stages.get(k, 0.0) for k in keys], dtype=torch.float64, device="cuda")
    cnt = torch.tensor([stages["rows_read"], stages["models"]], dtype=torch.int64, device="cuda")
    if ws > 1:
        import torch.distributed as dist
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
        allc = [torch.zeros_like(cnt) for _ in range(ws)]
        dist.all_gather(allc, cnt)
    else:
        allc = [cnt]
    if rank == 0:
        r, f, w, t, opk, ofi, oen = [float(x) for x in vals.tolist()]
        print(json.dumps({"ranks": ws, "reader": cfg["io"].get("reader", "auto"), "rank_local_input": bool(getattr(job, "rank_local_input", False)),
                          "read_s": r, "fit_s": f, "write_s": w, "total_s": t,
                          "fit_stage": {"pack_upload_group_sort_s": opk, "gpu_fit_and_d2h_s": ofi, "encode_records_s": oen},
                          "rows_read_by_rank": [int(c[0]) for c in allc], "models_by_rank": [int(c[1]) for c in allc]}))
    if ws > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    if sys.argv[1] == "make":
        make(sys.argv[2], int(sys.argv[3]), int(sys.argv[4]) if len(sys.argv) > 4 else 1440)
    else:
        run(sys.argv[2], sys.argv[3] if len(sys.argv) > 3 else None)
