"""Config-5 measurement (SURVEY 8d): k overlapping SSTs of one segment -> one sorted, deduplicated run
(hg_compact_open = Executor::do_compaction's plan, keep_builtin), and the same through the GPU SST writer (hg_compact_to_sst).
Prints one JSON line.

Usage: bench_compaction.py [k=16] [series=4000] [points=1000] [keep=0.5] [codec=snappy] [procs=16] [out_codec=snappy]
BASELINE config 5 at size: bench_compaction.py 64 15625 1000 0.25 snappy 32   (64 SSTs x 3.9 M rows = 250 M rows in)
`codec` is the inputs' page codec, `out_codec` the one hg_compact_to_sst writes.  Given explicitly, `out_codec` also adds a "writer"
section: compact_to_sst with none / snappy / zstd pages (time, file and column-chunk bytes), the ratio to pyarrow's Zstd level 1 on the
same table, the host path GPU Zstd replaces (hg_compact_open + pyarrow Zstd write), the encode kernels' device time (torch.profiler,
separate run), and the card's name and power limit."""
import io
import json
import os
import sys
import tempfile
import time
from concurrent.futures import ProcessPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

k = int(sys.argv[1]) if len(sys.argv) > 1 else 16
series = int(sys.argv[2]) if len(sys.argv) > 2 else 4000
points = int(sys.argv[3]) if len(sys.argv) > 3 else 1000
keep = float(sys.argv[4]) if len(sys.argv) > 4 else 0.5
codec = sys.argv[5] if len(sys.argv) > 5 else "snappy"
procs = int(sys.argv[6]) if len(sys.argv) > 6 else 16
out_codec = sys.argv[7] if len(sys.argv) > 7 else "snappy"


def _chunk_bytes(data):
    import pyarrow.parquet as pq
    md = pq.ParquetFile(io.BytesIO(data)).metadata
    return sum(md.row_group(g).column(c).total_compressed_size for g in range(md.num_row_groups) for c in range(md.num_columns))


def _writer_section(eng, handle, inputs, merged, path):
    import subprocess
    import numpy as np
    import pyarrow as pa
    from horaedb_b200 import sstgen
    from horaedb_b200.config import WriteConfig
    res = {}
    for c in ("none", "snappy", "zstd"):
        t = []
        for it in range(3):
            t0 = time.perf_counter()
            eng.compact_to_sst(handle, inputs, path, compression=c)
            t.append(((time.perf_counter() - t0) * 1e3, eng.stats()["gpu_ms"]))
        t = np.median(np.array(t[1:]), axis=0)
        data = open(path, "rb").read()
        res[c] = {"wall_ms": float(t[0]), "gpu_ms": float(t[1]), "file_bytes": len(data), "chunk_bytes": _chunk_bytes(data)}
    # the path GPU Zstd replaces: the merged run exported to the host, pyarrow writes the file (Zstd level 1, as storage.py does)
    schema = sstgen.metric_storage_schema()
    host = []
    for it in range(3):
        t0 = time.perf_counter()
        tbl = eng.compact(handle, inputs).read_all()
        data = sstgen.write_sst_with_seq(schema, tbl.combine_chunks().to_batches()[0], WriteConfig(compression="zstd"))
        with open(path + ".host", "wb") as f:
            f.write(data)
        host.append((time.perf_counter() - t0) * 1e3)
    ref = _chunk_bytes(data)
    res["host_compact_open_plus_pyarrow_zstd_ms"] = float(np.median(host[1:]))
    res["pyarrow_zstd_level1_chunk_bytes"] = ref
    res["zstd_chunk_ratio_to_pyarrow"] = res["zstd"]["chunk_bytes"] / ref
    res["zstd_speedup_vs_host_path"] = res["host_compact_open_plus_pyarrow_zstd_ms"] / res["zstd"]["wall_ms"]
    # device time of the page encoders, one profiled run per codec
    import torch
    from torch.profiler import ProfilerActivity, profile
    kern = {}
    for c, name in (("snappy", "snappy_encode_kernel"), ("zstd", "zstd_encode_kernel")):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            eng.compact_to_sst(handle, inputs, path, compression=c)
            torch.cuda.synchronize()
        kern[name + "_ms"] = sum(e.device_time_total for e in prof.key_averages() if name in e.key) / 1e3
    res["encode_kernels"] = kern
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    res["gpu"] = q.stdout.strip() or torch.cuda.get_device_name(0)
    return res


def _one(f):
    from horaedb_b200 import sstgen
    return sstgen.synth_overlapping_ssts(1, series, points, 1000, keep, compression=codec, base_seq=1000 + f)[0]


if __name__ == "__main__":
    t0 = time.perf_counter()
    with ProcessPoolExecutor(max_workers=procs) as ex:
        ssts = list(ex.map(_one, range(k)))
    gen_s = time.perf_counter() - t0

    import numpy as np
    from horaedb_b200 import sstgen
    from horaedb_b200._ffi import HG_FLAG_PAIRWISE_MERGE, Engine, SchemaHandle, SstInput

    schema = sstgen.metric_storage_schema()
    handle = SchemaHandle(schema.arrow_schema, 2)
    eng = Engine(device=0)
    inputs = []
    for i, (data, n, seq) in enumerate(ssts):
        eng.load_sst(handle, SstInput(id=seq, data=data, num_rows=n))
        inputs.append(SstInput(id=seq, num_rows=n, time_start=0, time_end=1, max_sequence=seq))
    rows_in = sum(n for _, n, _ in ssts)
    peak = 6578.0
    try:
        peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
    except Exception:
        pass

    def run(reps=4):
        res = []
        out = None
        for it in range(reps):
            t = time.perf_counter()
            out = eng.compact(handle, inputs).read_all()
            wall = time.perf_counter() - t
            st = eng.stats()
            res.append((st["merge_ms"], st["kernel_ms"], st["gpu_ms"], wall * 1e3))
        return np.median(np.array(res[1:]), axis=0), out, eng.stats()

    m, out, st = run()
    sid, ts = out["series_id"].to_numpy(), out["ts"].to_numpy()
    key = sid.astype(np.uint64) * np.uint64(1 << 32) + (ts - sstgen.T0_MS).astype(np.uint64)
    assert np.all(key[1:] > key[:-1]), "output must be sorted and duplicate-free"
    eng.set_flags(HG_FLAG_PAIRWISE_MERGE)
    mp, outp, _ = run(3)
    assert outp.num_rows == out.num_rows
    eng.set_flags(0)
    # end to end on the GPU: merge + dedup + Parquet encode (Snappy) + file written
    path = os.path.join(tempfile.mkdtemp(), "out.sst")
    wt = []
    for it in range(3):
        t = time.perf_counter()
        meta = eng.compact_to_sst(handle, inputs, path, compression=out_codec)
        wt.append(((time.perf_counter() - t) * 1e3, eng.stats()["gpu_ms"]))
    wt = np.median(np.array(wt[1:]), axis=0)
    alg = rows_in * 64
    writer = _writer_section(eng, handle, inputs, out, path) if len(sys.argv) > 7 else None
    print(json.dumps({"workload": f"merge-compaction: {k} overlapping SSTs, {rows_in} rows in, {out.num_rows} rows out, codec {codec}"
                      + (f", written as {out_codec}" if out_codec != "snappy" else ""),
                      "rows_in": rows_in, "rows_out": out.num_rows, "merge_ms": float(m[0]), "decode_ms": float(m[1]), "call_gpu_ms": float(m[2]),
                      "wall_ms": float(m[3]), "merge_rows_per_s": rows_in / (m[0] / 1e3), "call_rows_per_s": rows_in / (m[3] / 1e3),
                      "roofline_merge": {"alg_bytes": alg, "bytes_model": "64 B per input row (SURVEY 8d: read 4 columns incl. __seq__ + write them once)",
                                         "achieved_GBps": alg / (m[0] / 1e3) / 1e9, "peak_GBps": peak, "frac": alg / (m[0] / 1e3) / 1e9 / peak},
                      "pairwise_passes": {"merge_ms": float(mp[0]), "frac": alg / (mp[0] / 1e3) / 1e9 / peak,
                                          "note": "HG_FLAG_PAIRWISE_MERGE: log2(k) merge-path passes over 32-byte records (round 1)"},
                      "compact_to_sst": {"wall_ms": float(wt[0]), "gpu_ms": float(wt[1]), "file_bytes": int(meta.size), "rows": int(meta.num_rows),
                                         "rows_in_per_s": rows_in / (wt[0] / 1e3)},
                      "kernel_launches": st["kernel_launches"], "generate_s": gen_s, **({"writer": writer} if writer else {})}))
    eng.close()
