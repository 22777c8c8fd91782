#!/usr/bin/env python
"""bench.py — the hot path's headline measurement (BASELINE.json metric: scanned rows/s and decoded GB/s vs HBM peak).

Workload (BASELINE.json configs[1], SURVEY §8d "Config 2"): per GPU 100k series x 1k points = 100 M rows in 16 SSTs
(PK-disjoint series ranges, one segment), predicate `tag = 3 AND ts in [t0+250d, t0+750d)`, `sum(value), count(*)` per
series.  A step = one full scan+decode+filter+dedup+aggregate pass over all of the rank's SSTs.

  value  : rows/s with the SST bytes already resident in HBM (CUDA events on the engine's stream).
  e2e    : the same metric through the C ABI with HOST (pinned) SST buffers: H2D of the file bytes, footer/page-table
           parse, kernels and D2H of the result are all inside the timed region.
  roofline.achieved : algorithmic bytes (SURVEY §8d: 28 B per decoded row for this query) / dominant-kernel time.
  cpu_baseline : the CPU oracle (C restatement of the reference path) on a bounded sample, all host threads.

`--impl reference` times that CPU restatement alone (the reference itself is Rust and cannot be built here).
`--dump-outputs DIR` writes the result of the last timed step (series_id, count, sum, min, max of every group) as float64
DIR/<column>.npy; the inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ProcessPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SERIES_PER_FILE = 6250
POINTS = 1000
DELTA_MS = 1000
FILES_PER_GPU = 16
ALG_BYTES_PER_ROW = 28  # series_id 8 + ts 8 + value 8 + tag 4 (SURVEY §8d)


def _gen_file(args):
    lo, seq, codec = args
    from horaedb_b200 import sstgen
    data, n = sstgen.synth_sst(lo, lo + SERIES_PER_FILE, POINTS, DELTA_MS, seq=seq, compression=codec)
    return seq, data, n


def gen_ssts(rank, codec, nfiles, workers):
    base = rank * FILES_PER_GPU * SERIES_PER_FILE
    jobs = [(base + f * SERIES_PER_FILE, 1_000_000 + rank * 1000 + f, codec) for f in range(nfiles)]
    import multiprocessing
    cuda_live = "torch" in sys.modules and sys.modules["torch"].cuda.is_initialized()
    ctx = multiprocessing.get_context("spawn" if cuda_live else "fork")   # never fork a process that already owns a CUDA context
    with ProcessPoolExecutor(max_workers=workers, mp_context=ctx) as ex:
        return list(ex.map(_gen_file, jobs))


def bind_to_gpu_numa(device_index):
    """Pin this rank (and therefore the pinned SST buffers it allocates next: first touch) to the NUMA node its GPU hangs off, like
    `numactl --cpunodebind --membind` in a real deployment.  Best effort: returns the node or None."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(device_index)], capture_output=True, text=True,
                             timeout=20).stdout.strip()
        bdf = out.lower()
        if bdf.startswith("00000000:"):
            bdf = bdf[4:]
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


def preds():
    from horaedb_b200 import sstgen
    t0 = sstgen.T0_MS
    return [("tag", "eq", 3), ("ts", "ge", t0 + 250 * DELTA_MS), ("ts", "lt", t0 + 750 * DELTA_MS)]


class ClockSampler:
    """One background `nvidia-smi -lms 50` process sampling SM clocks and throttle reasons during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.proc = None
        self.samples = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                          str(self.device), "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            out = ""
        for line in out.splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) >= 6:
                self.samples.append(parts)

    def summary(self):
        sm = [int(s[0]) for s in self.samples if s[0].isdigit()]
        mx = [int(s[1]) for s in self.samples if s[1].isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": int(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_reference(ssts, threads, steps=1, warmup=0, queries=1):
    """The oracle port timed on the host cores.  `queries` independent copies of the query run concurrently (each one
    thread per SST, like the reference's one partition per file): the CPU analogue of `queries` GPUs scanning their own
    shards.  Returns (rows/s over all queries, rows per query, seconds per step, result of one query)."""
    from horaedb_b200 import sstgen
    from oracle import oracle
    schema = sstgen.metric_storage_schema()
    datas = [d for _, d, _ in ssts]
    rows = sum(n for _, _, n in ssts)
    out = [None] * queries

    def one(i):
        out[i] = oracle.scan_aggregate(datas, schema.arrow_schema, 2, preds(), group_col=0, value_col=2, threads=threads)

    def step():
        if queries == 1:
            one(0)
            return
        ths = [threading.Thread(target=one, args=(i,)) for i in range(queries)]     # ctypes releases the GIL inside the oracle
        for t in ths:
            t.start()
        for t in ths:
            t.join()

    for _ in range(warmup):
        step()
    t = time.perf_counter()
    for _ in range(max(steps, 1)):
        step()
    dt = (time.perf_counter() - t) / max(steps, 1)
    return rows * queries / dt, rows, dt, out[0]


def check_parity(tbl, exp):
    """Bit-exact comparison of a GPU aggregate (pyarrow table: series_id, count, sum, min, max) with the oracle's result."""
    def bits(a):
        return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)
    ok = (tbl.num_rows == len(exp.count)
          and np.array_equal(tbl["series_id"].to_numpy(), exp.gkey)
          and np.array_equal(tbl["count"].to_numpy(), exp.count)
          and np.array_equal(bits(tbl["sum"].to_numpy()), bits(exp.sum))
          and np.array_equal(bits(tbl["min"].to_numpy()), bits(exp.min))
          and np.array_equal(bits(tbl["max"].to_numpy()), bits(exp.max)))
    return bool(ok)


DUMP_LIMIT_BYTES = 64 << 20


def unpack_outputs(block):
    """[6, n] packed aggregate (key, bucket, count, sum / min / max bits; count == 0 pads) -> the result columns a caller of
    scan_aggregate receives for this query (no time buckets), as float64 (series ids and counts stay below 2**53)."""
    live = block[2] > 0
    f64 = lambda r: np.ascontiguousarray(block[r][live]).view(np.float64)
    return {"series_id": block[0][live].astype(np.float64), "count": block[2][live].astype(np.float64),
            "sum": f64(3), "min": f64(4), "max": f64(5)}


def dump_outputs(out_dir, cols):
    """One DIR/<name>.npy per column.  Above DUMP_LIMIT_BYTES in all, a fixed seeded sample of the groups is kept, in result
    order, and `row_index` records which rows it holds."""
    n = len(cols["count"])
    keep = DUMP_LIMIT_BYTES // (8 * (len(cols) + 1)) - 16        # room for row_index and the .npy headers
    if n > keep:
        idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        cols = {"row_index": idx.astype(np.float64), **{k: v[idx] for k, v in cols.items()}}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in cols.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--codec", default="snappy", choices=["none", "snappy"],
                    help="SST page codec of the main line (snappy = the reference's WriteConfig::default, config.rs:120-133)")
    ap.add_argument("--files", type=int, default=FILES_PER_GPU)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-variant", action="store_true", help="skip the secondary codec measurement")
    ap.add_argument("--no-compaction", action="store_true", help="skip the merge-compaction variant (N=1 only, own process)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's result (all GPUs' groups, main codec) as DIR/<column>.npy in float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    # stdout carries exactly ONE JSON line: route everything else (NCCL banners, library chatter) to stderr
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    ncores = os.cpu_count() or 1
    workload = (f"config2: {args.files} SSTs/GPU x {SERIES_PER_FILE} series x {POINTS} pts, tag=3 AND ts in [t0+250d,t0+750d), "
                "sum(value),count per series")

    # ------------------------------------------------------------------------------------------- reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        nsample = args.files
        ssts = gen_ssts(0, args.codec, nsample, min(ncores, nsample))  # the SAME files as our arm's main line (same codec)
        nq = max(1, args.gpus)           # our arm scans gpus x files: the CPU arm runs as many independent queries side by side
        rps, rows, dt, _ = cpu_reference(ssts, ncores, steps=max(args.steps, 1), warmup=min(args.warmup, 1), queries=nq)
        used = min(ncores, nsample * nq)  # one decode/filter thread per SST (the reference's one partition per file, read.rs:442-450)
        line = {"impl": "reference", "metric": "scanned rows/s", "value": rps, "unit": "rows/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": workload, "codec": args.codec},
                "cpu_baseline": {"value": rps, "unit": "rows/s", "cores": used, "kind": "port",
                                 "sample": f"{nq} concurrent quer{'y' if nq == 1 else 'ies'} x {nsample} SSTs = {rows * nq} rows per step (C restatement of the "
                                           f"reference path; the Rust reference cannot be built here); {used} threads busy = one per SST like the "
                                           f"reference's one partition per file, merge/dedup/aggregate single-threaded per query like MergeExec; "
                                           f"host has {ncores} cores"},
                "e2e": {"value": rps, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        emit(line)
        return

    # ------------------------------------------------------------------------------------------------- our arm (GPU)
    codecs = [args.codec] + ([] if args.no_variant else [c for c in ("none", "snappy") if c != args.codec])
    gen = {c: gen_ssts(rank, c, args.files, min(ncores, 16)) for c in codecs}     # before CUDA init (fork-safe)

    import torch
    import torch.distributed as dist
    from horaedb_b200 import sstgen
    from horaedb_b200._ffi import DeviceArray, Engine, SchemaHandle, SstInput

    torch.cuda.set_device(local_rank)
    numa_node = bind_to_gpu_numa(local_rank) if world > 1 else None      # several ranks share the host: keep each next to its GPU
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    schema = sstgen.metric_storage_schema()
    handle = SchemaHandle(schema.arrow_schema, 2)
    eng = Engine(device=local_rank)
    stream = torch.cuda.ExternalStream(eng.stream_ptr, device=torch.device("cuda", local_rank))
    P = preds()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if world > 1:
        # the library's own NCCL communicator (csrc/comm.cu); torch.distributed only ships the 128-byte id, like a Rust host's RPC
        uid = [Engine.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        eng.comm_init(uid[0], rank, world)
    comb_state = {"cap": 0, "last": None}

    def combine(dev, settle=False):
        """Cross-GPU combine of the per-GPU partial aggregates: ONE ncclAllGather per step, issued by the library on its combine
        stream behind a pack kernel (hg_agg_combine): the next step's scan overlaps it.  The block width is agreed during
        warm-up (`settle`); timed steps have no size exchange and no host sync."""
        g = int(dev.num_groups)
        if world == 1:
            return g
        from horaedb_b200._ffi import HG_COMBINE_GATHER
        cmb = eng.combine(HG_COMBINE_GATHER, 0 if settle else comb_state["cap"])
        comb_state["cap"] = int(cmb.capacity)
        comb_state["last"] = cmb
        return cmb

    def gathered_block(cmb):
        eng.comm_sync()
        cap = int(cmb.capacity)
        return torch.as_tensor(DeviceArray(cmb.d_blocks, world * 6 * cap, "<i8"), device=f"cuda:{local_rank}").view(world, 6, cap)

    # ---- the CPU oracle's answer for THIS rank's files (same data under every codec): the timed GPU results are compared
    #      with it bit for bit below; rank 0's run doubles as the cpu_baseline measurement
    cpu_rps, cpu_rows, cpu_dt, expected = cpu_reference(gen[args.codec], ncores)

    def packed_matches(block, exp):
        """block: [6, cap] int64 host array (key, bucket, count, sum bits, min bits, max bits) vs the oracle result."""
        g = len(exp.count)
        if block.shape[1] < g or (block[2, g:] != 0).any():
            return False
        f = lambda a: np.ascontiguousarray(a, dtype=np.float64).view(np.int64)
        return bool(np.array_equal(block[0, :g], exp.gkey.astype(np.int64)) and np.array_equal(block[2, :g], exp.count.astype(np.int64))
                    and np.array_equal(block[3, :g], f(exp.sum)) and np.array_equal(block[4, :g], f(exp.min)) and np.array_equal(block[5, :g], f(exp.max)))

    def block_checksum(block):
        return int(block.astype(np.uint64).sum(dtype=np.uint64)) & 0x7FFFFFFFFFFFFFFF

    def measure(codec, steps, warmup, e2e_steps):
        ssts = gen[codec]
        rows = sum(n for _, _, n in ssts)
        file_bytes = sum(len(d) for _, d, _ in ssts)
        inputs_host = []
        pinned = []
        for sid, data, n in ssts:                      # pinned host copies of the SST bytes (the e2e source)
            t = torch.empty(len(data), dtype=torch.uint8, pin_memory=True)
            t.numpy()[:] = np.frombuffer(data, dtype=np.uint8)
            pinned.append(t)
            inputs_host.append(SstInput(id=sid, ptr=t.data_ptr(), size=len(data), num_rows=n))
        resident = [SstInput(id=sid, num_rows=n) for sid, _, n in ssts]
        # ---- e2e: host buffers in, host result out, every step (SSTs are evicted between steps)
        d2h = 0
        h2d = 0

        for sid, _, _ in ssts:                       # nothing of these files may be resident: every e2e call moves its bytes itself
            try:
                eng.unload_sst(sid)
            except Exception:
                pass

        def e2e_step():                              # (SSTs given as host buffers are transient: gone from HBM when the call returns)
            return eng.scan_aggregate(handle, inputs_host, P, group_col=0, ts_col=-1, window_ms=0, value_col=2)

        # two untimed calls: the first sizes the engine's arena and pinned staging, the second runs on the consolidated arena
        for _ in range(2):
            tbl = e2e_step()
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        for it in range(e2e_steps):          # each call returns the host result: H2D, kernels and D2H are inside it
            tbl = e2e_step()
        torch.cuda.synchronize()
        e2e_dt = (time.perf_counter() - t0) / max(e2e_steps, 1)
        d2h = eng.stats()["bytes_d2h"]
        h2d = eng.stats()["bytes_h2d"]
        if world > 1:
            tt = torch.tensor([e2e_dt], device="cuda", dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            e2e_dt = float(tt.item())
        groups_local = tbl.num_rows
        parity_e2e = check_parity(tbl, expected)
        # ---- HBM-resident steps: make the SSTs resident once (untimed), then every step is one scan call
        for inp in inputs_host:
            eng.load_sst(handle, inp)
        for _ in range(max(warmup, 1)):
            dev = eng.scan_aggregate_device(handle, resident, P, group_col=0, ts_col=-1, window_ms=0, value_col=2)
            combine(dev, settle=True)
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
            time.sleep(0.15)
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        kernel_ms, call_ms, decomp_ms, launches = [], [], [], 0
        prep = eng.prepare_aggregate(handle, resident, P, group_col=0, ts_col=-1, window_ms=0, value_col=2)   # arguments marshalled once
        prep.run()
        ev0.record(stream)
        for _ in range(steps):
            dev = prep.run()
            sst_ = eng.stats_struct()
            kernel_ms.append(sst_.kernel_ms)
            call_ms.append(sst_.gpu_ms)
            decomp_ms.append(sst_.decomp_ms)
            launches += sst_.kernel_launches
            last = combine(dev)
        if world > 1:
            eng.comm_sync()               # the last step's all-gather is part of the timed region
        ev1.record(stream)
        barrier()
        ms = ev0.elapsed_time(ev1)
        # the last timed step's device result, packed before any later call replaces the engine's last aggregate
        g_local = int(dev.num_groups)
        cap = max(g_local, 1)
        blk = torch.empty(6, cap, device="cuda", dtype=torch.int64)     # pack_agg writes all `cap` columns
        with torch.cuda.stream(stream):
            eng.export_packed(blk.data_ptr(), cap)
        stream.synchronize()
        own = blk.cpu().numpy()
        if world > 1:
            last = gathered_block(last)
        if rank == 0:
            # the K timed steps last only ~K ms; keep the same load running ~0.4 s so the clock sampler sees it
            t_end = time.perf_counter() + 0.4
            while time.perf_counter() < t_end:
                eng.scan_aggregate_device(handle, resident, P, group_col=0, ts_col=-1, window_ms=0, value_col=2)
            sampler.stop()
        if world > 1:
            tt = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = float(tt.item())
        st = eng.stats()
        # ---- parity of the TIMED configuration: the last timed step's device result against the oracle
        parity_resident = packed_matches(own, expected)
        parity_combined = None
        outputs = unpack_outputs(own)
        if world > 1:
            # every rank's slot of the gathered block must carry exactly that rank's partial (checked through checksums of
            # the ranks' ORACLE results), and this rank's slot must equal its own oracle result bit for bit
            gathered = last.cpu().numpy()                       # [world, 6, cap]
            outputs = unpack_outputs(np.concatenate(list(gathered), axis=1))   # every rank's groups, rank by rank
            mine = gathered[rank]
            ok = packed_matches(mine, expected)
            exp_blk = np.zeros((6, len(expected.count)), dtype=np.int64)
            f = lambda a: np.ascontiguousarray(a, dtype=np.float64).view(np.int64)
            exp_blk[0], exp_blk[2] = expected.gkey.astype(np.int64), expected.count.astype(np.int64)
            exp_blk[3], exp_blk[4], exp_blk[5] = f(expected.sum), f(expected.min), f(expected.max)
            sums = torch.zeros(world, device="cuda", dtype=torch.int64)
            sums[rank] = block_checksum(exp_blk)
            dist.all_reduce(sums)
            want = sums.cpu().numpy()
            for r in range(world):
                ok = ok and block_checksum(gathered[r]) == int(want[r])
            flag = torch.tensor([1 if ok else 0], device="cuda", dtype=torch.int64)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            parity_combined = bool(flag.item())
        # A/B: the same resident scan with the late-materialisation gate off (every needed column of every row is read)
        ungated_ms = None
        if st["path"] == 1:
            from horaedb_b200._ffi import HG_FLAG_NO_LATE_MATERIALIZATION
            eng.set_flags(HG_FLAG_NO_LATE_MATERIALIZATION)
            ks = []
            for _ in range(6):
                eng.scan_aggregate_device(handle, resident, P, group_col=0, ts_col=-1, window_ms=0, value_col=2)
                ks.append(eng.stats()["kernel_ms"])
            ungated_ms = float(np.mean(ks[2:]))
            eng.set_flags(0)
        total_groups = last if world == 1 else int((last[:, 2, :] > 0).sum().item())
        return {"parity": {"resident": parity_resident, "e2e": parity_e2e, "combined": parity_combined, "groups": g_local},
                "decomp_ms": float(np.mean(decomp_ms)) if decomp_ms else 0.0,
                "ungated_kernel_ms": ungated_ms,"rows": rows, "file_bytes": file_bytes, "ms_total": ms, "ms_per_step": ms / steps, "kernel_ms": float(np.mean(kernel_ms)),
                "call_ms": float(np.mean(call_ms)), "launches": launches, "e2e_s": e2e_dt, "d2h": d2h, "h2d": h2d, "stats": st,
                "groups": total_groups, "groups_local": groups_local,
                "clocks": sampler.summary() if rank == 0 else None, "ssts": ssts, "outputs": outputs}

    res = {c: measure(c, args.steps, args.warmup, args.e2e_steps) for c in codecs}
    main_r = res[args.codec]

    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, main_r["outputs"])
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        rows_all = main_r["rows"] * world
        value = rows_all / (main_r["ms_per_step"] / 1e3)
        st = main_r["stats"]
        survey_bytes = st["rows_decoded"] * ALG_BYTES_PER_ROW      # SURVEY 8(d): every needed column of every decoded row
        gate_bytes = st["rows_decoded"] * 4 + st["rows_materialized"] * 16 + st["rows_filtered"] * 8
        traffic_tbl = {}
        try:  # dram__bytes_read.sum + dram__bytes_write.sum of one launch, from the committed `ncu --set full` captures
            traffic_tbl = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        except Exception:
            pass

        def scan_kernel_block(r):
            """Roofline of the fused scan kernel: late-materialising, so `achieved` counts the bytes THAT algorithm must read."""
            sr = r["stats"]
            ab = (sr["rows_decoded"] * 4 + sr["rows_materialized"] * 16 + sr["rows_filtered"] * 8) if sr["path"] == 1 else sr["rows_decoded"] * ALG_BYTES_PER_ROW
            ach = ab / (r["kernel_ms"] / 1e3) / 1e9
            blk = {"kernel": "fused_scan_kernel" if sr["path"] == 1 else "decode_chunks", "kernel_ms": r["kernel_ms"], "alg_bytes_per_launch": ab,
                   "achieved": ach, "frac": ach / peak, "traffic": traffic_tbl.get("fused_scan_kernel"),
                   "bytes_model": "late materialisation: 4 B x rows_decoded + 16 B x rows_materialized + 8 B x rows_filtered",
                   "rows_materialized": sr["rows_materialized"]}
            if r["ungated_kernel_ms"]:
                sb = sr["rows_decoded"] * ALG_BYTES_PER_ROW
                blk["ungated"] = {"kernel_ms": r["ungated_kernel_ms"], "achieved": sb / (r["ungated_kernel_ms"] / 1e3) / 1e9,
                                  "frac": sb / (r["ungated_kernel_ms"] / 1e3) / 1e9 / peak,
                                  "note": "HG_FLAG_NO_LATE_MATERIALIZATION: all 28 B of every decoded row are read (SURVEY 8d byte model); "
                                          "kernel_ms measured live after the timed region"}
            return blk

        if args.codec == "snappy" and main_r["decomp_ms"] > 0:
            # dominant stage = Snappy page decompression (two launches of snappy_pages_kernel + the row-group gate between them).
            # Algorithmic bytes = UNCOMPRESSED page bytes of the needed columns of every row group that survives statistics
            # pruning (SURVEY 8d: 28 B x rows_decoded) — what a decompress-everything implementation must produce; this
            # engine reaches the same result producing fewer (stored value pages are read in place, row groups without a
            # passing row are only decompressed for the gate column).
            alg_bytes = survey_bytes
            kms = main_r["decomp_ms"]
            achieved = alg_bytes / (kms / 1e3) / 1e9
            roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                        "traffic": traffic_tbl.get("snappy_pages_kernel"), "kernel": "snappy_pages_kernel (gate column, row-group gate, other columns)",
                        "kernel_ms": kms, "alg_bytes_per_launch": alg_bytes, "peak_source": peak_src,
                        "bytes_model": "28 B x rows_decoded = uncompressed page bytes of series_id, ts, value, tag in the row groups that survive "
                                       "statistics pruning, / device time of the decompression stage (CUDA events on the engine stream)",
                        "scan_kernel": scan_kernel_block(main_r)}
        else:
            blk = scan_kernel_block(main_r)
            roofline = {"bound": "hbm", "achieved": blk["achieved"], "peak": peak, "unit": "GB/s", "frac": blk["frac"], "traffic": blk["traffic"],
                        "kernel": blk["kernel"], "kernel_ms": blk["kernel_ms"], "alg_bytes_per_launch": blk["alg_bytes_per_launch"],
                        "peak_source": peak_src, "bytes_model": blk["bytes_model"], "rows_materialized": blk["rows_materialized"],
                        "survey_bytes_per_launch": survey_bytes, "survey_GBps": survey_bytes / (main_r["kernel_ms"] / 1e3) / 1e9,
                        "ungated": blk.get("ungated")}
        nsample = len(main_r["ssts"])
        parity_ok = all(r["parity"]["resident"] and r["parity"]["e2e"] and r["parity"]["combined"] is not False for r in res.values())
        # all host cores: as many independent copies of the query as fit, side by side (one thread per SST each)
        nq_all = max(1, ncores // max(1, min(ncores, nsample)))
        all_rps, _, all_dt, _ = cpu_reference(main_r["ssts"], ncores, queries=nq_all) if nq_all > 1 else (cpu_rps, 0, cpu_dt, None)
        line = {
            "metric": "scanned rows/s", "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": main_r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload, "codec": args.codec,
                       "codec_note": ("main line = WriteConfig::default (Snappy, config.rs:120-133); the UNCOMPRESSED writer variant of SURVEY 8(d) is "
                                      "under `variants`") if args.codec == "snappy"
                       else "main line = the SURVEY 8(d) UNCOMPRESSED writer variant; the reference-default Snappy run is under `variants`",
                       "rows_per_gpu": main_r["rows"], "sst_bytes_per_gpu": main_r["file_bytes"],
                       "l2_policy": "inputs (>=1 GB per step) far exceed the 126 MB L2; no flush needed",
                       "path": "fused" if st["path"] == 1 else "general", "rows_decoded_per_gpu": st["rows_decoded"],
                       "rows_filtered_per_gpu": st["rows_filtered"], "groups": main_r["groups"],
                       "decoded_GBps": rows_all * ALG_BYTES_PER_ROW / (main_r["ms_per_step"] / 1e3) / 1e9,
                       "decoded_GBps_note": "SURVEY 8(d) convention: ALL rows of the files x 28 B / step time.  Statistics pruning, stored-page "
                                            "bypass and late materialisation skip bytes that cannot contribute; the physical figures are "
                                            "roofline.achieved / roofline.traffic",
                       "late_materialisation_bytes": gate_bytes, "numa_node_rank0": numa_node},
            "roofline": roofline,
            "parity": {"checked": True, "ok": parity_ok, "against": "CPU oracle on the same SSTs, bit-exact keys / counts / f64 sum, min, max",
                       **{c: r["parity"] for c, r in res.items()}},
            "cpu_baseline": {"value": cpu_rps, "unit": "rows/s", "cores": min(ncores, nsample), "kind": "port",
                             "sample": f"{nsample} of the same SSTs = {cpu_rows} rows, oracle (C restatement of the reference path): "
                                       f"{min(ncores, nsample)} threads busy = one per SST like the reference's one partition per file "
                                       f"(read.rs:442-450), merge/dedup/aggregate single-threaded like MergeExec; host has {ncores} cores",
                             "all_cores": {"value": all_rps, "unit": "rows/s", "cores": min(ncores, nsample * nq_all),
                                           "sample": f"{nq_all} independent copies of the query side by side, {nsample} SSTs each"}},
            "e2e": {"value": rows_all / main_r["e2e_s"], "unit": "rows/s", "h2d_bytes_per_step": int(main_r["h2d"]) * world,
                    "d2h_bytes_per_step": int(main_r["d2h"]) * world, "ms_per_step": main_r["e2e_s"] * 1e3},
            "gpu_launches": main_r["launches"],
            "clocks": main_r["clocks"],
            "variants": {c: {"rows_per_s": r["rows"] * world / (r["ms_per_step"] / 1e3), "ms_per_step": r["ms_per_step"],
                             "kernel_ms": r["kernel_ms"], "decomp_ms": r["decomp_ms"], "path": "fused" if r["stats"]["path"] == 1 else "general",
                             "e2e_rows_per_s": r["rows"] * world / r["e2e_s"], "sst_bytes_per_gpu": r["file_bytes"],
                             "launches": r["launches"], "scan_kernel": scan_kernel_block(r)} for c, r in res.items() if c != args.codec},
        }
        if world == 1 and not args.no_compaction:
            # BASELINE config 5's shape at a size that keeps the default run short: 16 overlapping Snappy SSTs (32 M rows in) -> one sorted,
            # deduplicated run (hg_compact_open) and the same through the GPU SST writer (hg_compact_to_sst).  Its own process (own engine);
            # config 5 at full size (64 SSTs, 250 M rows): tools/bench_compaction.py 64 15625 1000 0.25 snappy 32 -> profiles/.
            try:
                out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_compaction.py"), "16", "4000", "1000", "0.5", "snappy", "16"],
                                     capture_output=True, text=True, timeout=300)
                cj = json.loads(out.stdout.strip().splitlines()[-1])
                line["variants"]["compaction"] = {
                    "workload": cj["workload"], "rows_in": cj["rows_in"], "rows_out": cj["rows_out"],
                    "merge_rows_per_s": cj["merge_rows_per_s"], "merge_ms": cj["merge_ms"], "decode_ms": cj["decode_ms"], "call_gpu_ms": cj["call_gpu_ms"],
                    "roofline": {"bound": "hbm", "kernel": "kway_merge_kernel (+ build_keys64, splitters, bounds, survivor compaction): S4-S6",
                                 "achieved": cj["roofline_merge"]["achieved_GBps"], "peak": cj["roofline_merge"]["peak_GBps"], "unit": "GB/s",
                                 "frac": cj["roofline_merge"]["frac"], "alg_bytes_per_launch": cj["roofline_merge"]["alg_bytes"],
                                 "bytes_model": cj["roofline_merge"]["bytes_model"]},
                    "pairwise_passes_merge_ms": cj["pairwise_passes"]["merge_ms"], "compact_to_sst": cj["compact_to_sst"]}
            except Exception as ex:      # the main line stands on its own
                line["variants"]["compaction"] = {"error": f"{type(ex).__name__}: {ex}"[:300]}
        emit(line)
    ok_all = all(r["parity"]["resident"] and r["parity"]["e2e"] and r["parity"]["combined"] is not False for r in res.values())
    if world > 1:
        eng.comm_destroy()
        dist.barrier()
        dist.destroy_process_group()
    eng.close()
    if not ok_all:
        sys.stderr.write(f"[bench] rank {rank}: PARITY MISMATCH against the CPU oracle: { {c: r['parity'] for c, r in res.items()} }\n")
        sys.exit(3)


if __name__ == "__main__":
    main()
