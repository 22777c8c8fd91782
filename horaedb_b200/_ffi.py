"""ctypes binding of libhorae_gpu.so (include/horae_gpu.h).  Fails loudly when the CUDA library is missing:
there is no CPU fallback anywhere in this package."""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np
import pyarrow as pa

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libhorae_gpu.so")

HG_TYPES = {pa.uint8(): 0, pa.int8(): 1, pa.uint16(): 2, pa.int16(): 3, pa.uint32(): 4, pa.int32(): 5,
            pa.uint64(): 6, pa.int64(): 7, pa.float32(): 8, pa.float64(): 9, pa.binary(): 10}
HG_OPS = {"eq": 0, "ne": 1, "lt": 2, "le": 3, "gt": 4, "ge": 5, "in": 6}
HG_FLAG_NO_PRUNING = 1
HG_FLAG_NO_FUSED = 2
HG_FLAG_NO_LATE_MATERIALIZATION = 4
HG_FLAG_PAIRWISE_MERGE = 8
HG_AGG_RUNS, HG_AGG_HASH = 0, 1

STATUS = {0: "OK", 1: "INVALID", 2: "UNSUPPORTED", 3: "CUDA", 4: "FORMAT", 5: "OOM", 6: "NOT_FOUND", 7: "INTERNAL"}


class HgError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"HG_ERR_{STATUS.get(code, code)}: {msg}")
        self.code = code


class HgSchemaDesc(C.Structure):
    _fields_ = [("num_columns", C.c_uint32), ("num_primary_keys", C.c_uint32), ("update_mode", C.c_uint32),
                ("_pad", C.c_uint32), ("types", C.POINTER(C.c_uint32)), ("names", C.POINTER(C.c_char_p))]


class HgConfig(C.Structure):
    _fields_ = [("device", C.c_int32), ("batch_size", C.c_uint32), ("hbm_budget_bytes", C.c_uint64),
                ("flags", C.c_uint32), ("_pad", C.c_uint32)]


class HgSstDesc(C.Structure):
    _fields_ = [("id", C.c_uint64), ("data", C.c_void_p), ("size", C.c_uint64), ("path", C.c_char_p),
                ("num_rows", C.c_uint32), ("_pad", C.c_uint32), ("time_start", C.c_int64), ("time_end", C.c_int64),
                ("max_sequence", C.c_uint64)]


class HgPredicate(C.Structure):
    _fields_ = [("column", C.c_uint32), ("op", C.c_uint32), ("i64", C.c_int64), ("u64", C.c_uint64), ("f64", C.c_double),
                ("in_values", C.POINTER(C.c_uint64)), ("in_count", C.c_uint32), ("_pad", C.c_uint32)]


class HgAggSpec(C.Structure):
    _fields_ = [("group_col", C.c_int32), ("ts_col", C.c_int32), ("window_ms", C.c_int64), ("value_col", C.c_int32),
                ("mode", C.c_uint32)]


class HgScanStats(C.Structure):
    _fields_ = [("rows_in_files", C.c_uint64), ("rows_decoded", C.c_uint64), ("rows_filtered", C.c_uint64),
                ("rows_out", C.c_uint64), ("groups_out", C.c_uint64), ("bytes_h2d", C.c_uint64), ("bytes_d2h", C.c_uint64),
                ("kernel_launches", C.c_uint32), ("path", C.c_uint32), ("gpu_ms", C.c_float), ("kernel_ms", C.c_float), ("merge_ms", C.c_float), ("decomp_ms", C.c_float),
                ("rows_materialized", C.c_uint64)]


class HgAggDevice(C.Structure):
    _fields_ = [("num_groups", C.c_uint64), ("d_gkey", C.c_void_p), ("d_bucket", C.c_void_p), ("d_count", C.c_void_p),
                ("d_sum", C.c_void_p), ("d_min", C.c_void_p), ("d_max", C.c_void_p)]


class HgWriteProps(C.Structure):
    _fields_ = [("max_row_group_size", C.c_uint32), ("compression", C.c_uint32), ("enable_sorting_columns", C.c_uint32), ("_pad", C.c_uint32)]


# codec names of the GPU writer -> Parquet codec ids (hg_write_props.compression)
_CODECS = {"none": 0, "uncompressed": 0, "snappy": 1, "zstd": 6}


class HgFileMeta(C.Structure):
    _fields_ = [("size", C.c_uint64), ("num_rows", C.c_uint32), ("_pad", C.c_uint32), ("time_start", C.c_int64), ("time_end", C.c_int64),
                ("max_sequence", C.c_uint64)]


class HgAggCombined(C.Structure):
    _fields_ = [("capacity", C.c_uint64), ("world", C.c_uint32), ("_pad", C.c_uint32), ("d_blocks", C.c_void_p), ("num_groups", C.c_uint64),
                ("reduced_capacity", C.c_uint64), ("d_reduced", C.c_void_p)]


HG_COMBINE_GATHER, HG_COMBINE_REDUCE = 0, 1


class ArrowArrayStream(C.Structure):
    _fields_ = [("get_schema", C.c_void_p), ("get_next", C.c_void_p), ("get_last_error", C.c_void_p),
                ("release", C.c_void_p), ("private_data", C.c_void_p)]


class HgParquetSummary(C.Structure):
    _fields_ = [("num_rows", C.c_uint64), ("num_row_groups", C.c_uint32), ("num_columns", C.c_uint32), ("num_data_pages", C.c_uint64),
                ("sum_page_values", C.c_uint64), ("sum_uncompressed_bytes", C.c_uint64), ("sum_compressed_bytes", C.c_uint64),
                ("codec_mask", C.c_uint32), ("max_pages_per_chunk", C.c_uint32)]


class HgParquetChunk(C.Structure):
    _fields_ = [("num_rows", C.c_uint64), ("num_values", C.c_uint64), ("data_page_offset", C.c_int64), ("total_compressed_size", C.c_int64),
                ("null_count", C.c_int64), ("min", C.c_uint8 * 8), ("max", C.c_uint8 * 8), ("has_min_max", C.c_uint32),
                ("physical_type", C.c_uint32), ("codec", C.c_uint32), ("num_pages", C.c_uint32), ("first_page_payload_offset", C.c_uint64),
                ("first_page_num_values", C.c_uint32), ("first_page_type", C.c_uint32)]


EXPORTS = ["hg_abi_version", "hg_last_error", "hg_engine_create", "hg_engine_destroy", "hg_engine_stream", "hg_engine_set_flags", "hg_sst_load",
           "hg_sst_unload", "hg_sst_resident_bytes", "hg_scan_open", "hg_compact_open", "hg_scan_aggregate",
           "hg_scan_aggregate_device", "hg_agg_export_packed", "hg_last_stats", "hg_parquet_inspect", "hg_parquet_chunk_info", "hg_plan_row_groups",
           "hg_compact_to_sst", "hg_write_batch", "hg_plan_pk_splitters", "hg_comm_unique_id", "hg_comm_init", "hg_comm_destroy", "hg_agg_combine", "hg_comm_sync"]

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(horaedb_b200 has no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        L.hg_abi_version.restype = C.c_uint32
        L.hg_last_error.restype = C.c_char_p
        L.hg_engine_stream.restype = C.c_void_p
        L.hg_engine_stream.argtypes = [C.c_void_p]
        L.hg_engine_set_flags.argtypes = [C.c_void_p, C.c_uint32]
        L.hg_engine_destroy.argtypes = [C.c_void_p]
        L.hg_engine_destroy.restype = None
        L.hg_comm_init.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        L.hg_comm_destroy.argtypes = [C.c_void_p]
        L.hg_comm_sync.argtypes = [C.c_void_p]
        L.hg_agg_combine.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p]
        _lib = L
    return _lib


def _check(rc: int):
    if rc != 0:
        raise HgError(rc, lib().hg_last_error().decode())


@dataclass
class SstInput:
    """`SstFile` + `FileMeta` (sst.rs:51-53, 155-160) as passed across the ABI."""
    id: int
    data: Optional[object] = None   # bytes / numpy uint8 / None when resident
    path: Optional[str] = None
    num_rows: int = 0
    time_start: int = 0
    time_end: int = 0
    max_sequence: int = 0
    ptr: int = 0                    # raw host pointer (e.g. pinned memory) used instead of `data`
    size: int = 0


class DeviceArray:
    """Zero-copy view of an engine-owned device buffer (`__cuda_array_interface__`), e.g. for torch.as_tensor(...)."""

    def __init__(self, ptr: int, n: int, typestr: str):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": typestr, "data": (int(ptr or 0), False), "version": 2}


class SchemaHandle:
    """Keeps the ctypes arrays behind an hg_schema_desc alive."""

    def __init__(self, arrow_schema: pa.Schema, num_primary_keys: int, update_mode: int = 0):
        n = len(arrow_schema)
        self.types = (C.c_uint32 * n)(*[HG_TYPES[f.type] if f.type in HG_TYPES else 0xFFFF for f in arrow_schema])
        self.names = (C.c_char_p * n)(*[f.name.encode() for f in arrow_schema])
        self.desc = HgSchemaDesc(n, num_primary_keys, update_mode, 0, self.types, self.names)
        self.arrow_schema = arrow_schema


def _make_preds(arrow_schema: pa.Schema, preds: Sequence[tuple]):
    arr = (HgPredicate * max(len(preds), 1))()
    keep = []
    for k, (col, op, lit) in enumerate(preds):
        idx = col if isinstance(col, int) else arrow_schema.get_field_index(col)
        t = arrow_schema.field(idx).type
        arr[k].column = idx
        arr[k].op = HG_OPS[op]
        if op == "in":
            bits = []
            for v in lit:
                if pa.types.is_floating(t):
                    bits.append(int(np.array([float(v)], dtype=np.float64).view(np.uint64)[0]))
                else:
                    if isinstance(v, float) and not v.is_integer():
                        raise HgError(1, f"IN literal {v!r} is not integral for column {arrow_schema.field(idx).name}")
                    bits.append(int(v) & 0xFFFFFFFFFFFFFFFF)
            vals = (C.c_uint64 * max(len(bits), 1))(*bits)
            keep.append(vals)
            arr[k].in_values = vals
            arr[k].in_count = len(bits)
        elif pa.types.is_floating(t):
            arr[k].f64 = float(lit)
        else:
            # no silent truncation / wrap-around: a literal the column type cannot hold must be rewritten by the caller
            # (DataFusion would coerce the comparison to a wider type; this ABI compares in the column's own domain)
            if isinstance(lit, float) and not lit.is_integer():
                raise HgError(1, f"predicate literal {lit!r} is not integral for column {arrow_schema.field(idx).name}")
            if not pa.types.is_integer(t):
                raise HgError(2, f"predicates on {t} column {arrow_schema.field(idx).name} are not implemented on the GPU path")
            iv = int(lit)
            bits = t.bit_width
            lo, hi = (-(1 << (bits - 1)), (1 << (bits - 1)) - 1) if pa.types.is_signed_integer(t) else (0, (1 << bits) - 1)
            if not lo <= iv <= hi:
                raise HgError(1, f"predicate literal {iv} does not fit column {arrow_schema.field(idx).name} ({t})")
            if pa.types.is_signed_integer(t):
                arr[k].i64 = iv
            else:
                arr[k].u64 = iv
    arr._keep = keep              # IN lists must outlive the call
    return arr


class Engine:
    """One engine per GPU (per rank).  Thin object wrapper over the C ABI."""

    def __init__(self, device: int = 0, batch_size: int = 8192, hbm_budget_bytes: int = 0, flags: int = 0):
        self._L = lib()
        self._h = C.c_void_p()
        cfg = HgConfig(device, batch_size, hbm_budget_bytes, flags, 0)
        _check(self._L.hg_engine_create(C.byref(cfg), C.byref(self._h)))
        self._keep = []
        self._stats_buf = HgScanStats()

    def close(self):
        if self._h:
            self._L.hg_engine_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def stream_ptr(self) -> int:
        return self._L.hg_engine_stream(self._h)

    def set_flags(self, flags: int) -> None:
        _check(self._L.hg_engine_set_flags(self._h, flags))

    # -- residency
    def _descs(self, ssts: Sequence[SstInput]):
        arr = (HgSstDesc * max(len(ssts), 1))()
        keep = []
        for i, s in enumerate(ssts):
            arr[i].id = s.id
            if s.ptr:
                arr[i].data = s.ptr
                arr[i].size = s.size
            elif s.data is not None:
                buf = np.frombuffer(s.data, dtype=np.uint8) if not isinstance(s.data, np.ndarray) else s.data
                keep.append(buf)
                arr[i].data = buf.ctypes.data
                arr[i].size = buf.nbytes
            else:
                arr[i].data = None
                arr[i].size = 0
            arr[i].path = s.path.encode() if s.path else None
            arr[i].num_rows = s.num_rows
            arr[i].time_start = s.time_start
            arr[i].time_end = s.time_end
            arr[i].max_sequence = s.max_sequence
        return arr, keep

    def load_sst(self, schema: SchemaHandle, sst: SstInput):
        arr, keep = self._descs([sst])
        _check(self._L.hg_sst_load(self._h, C.byref(schema.desc), C.byref(arr[0])))

    def unload_sst(self, id: int):
        _check(self._L.hg_sst_unload(self._h, C.c_uint64(id)))

    def resident_bytes(self) -> int:
        out = C.c_uint64()
        _check(self._L.hg_sst_resident_bytes(self._h, C.byref(out)))
        return out.value

    # -- scan / compaction
    def scan(self, schema: SchemaHandle, ssts: Sequence[SstInput], preds: Sequence[tuple] = (),
             projection: Optional[Sequence[int]] = None, keep_builtin: bool = False) -> pa.RecordBatchReader:
        arr, keep = self._descs(ssts)
        p = _make_preds(schema.arrow_schema, preds)
        proj = (C.c_uint32 * max(len(projection), 1))(*projection) if projection is not None else None
        stream = ArrowArrayStream()
        _check(self._L.hg_scan_open(self._h, C.byref(schema.desc), arr, C.c_size_t(len(ssts)), p, C.c_size_t(len(preds)),
                                    proj, C.c_size_t(len(projection) if projection is not None else 0), int(keep_builtin),
                                    C.byref(stream)))
        return pa.RecordBatchReader._import_from_c(C.addressof(stream))

    def compact(self, schema: SchemaHandle, ssts: Sequence[SstInput]) -> pa.RecordBatchReader:
        arr, keep = self._descs(ssts)
        stream = ArrowArrayStream()
        _check(self._L.hg_compact_open(self._h, C.byref(schema.desc), arr, C.c_size_t(len(ssts)), C.byref(stream)))
        return pa.RecordBatchReader._import_from_c(C.addressof(stream))

    def compact_to_sst(self, schema: SchemaHandle, ssts: Sequence[SstInput], out_path: str, max_row_group_size: int = 8192,
                       compression: str = "snappy", enable_sorting_columns: bool = True, shard_preds: Sequence[tuple] = ()) -> "HgFileMeta":
        """`Executor::do_compaction` on the GPU end to end: merge + dedup + Parquet encode, written to `out_path`.
        `shard_preds` = this GPU's pk0 range in a multi-GPU compaction (see `plan_pk_splitters`)."""
        arr, keep = self._descs(ssts)
        p = _make_preds(schema.arrow_schema, shard_preds)
        props = HgWriteProps(max_row_group_size, _CODECS[compression.lower()], int(enable_sorting_columns), 0)
        meta = HgFileMeta()
        _check(self._L.hg_compact_to_sst(self._h, C.byref(schema.desc), arr, C.c_size_t(len(ssts)), p, C.c_size_t(len(shard_preds)), C.byref(props),
                                         out_path.encode(), C.byref(meta)))
        return meta

    def write_batch(self, schema: SchemaHandle, batch: pa.RecordBatch, sequence: int, out_path: str, max_row_group_size: int = 8192,
                    compression: str = "snappy", enable_sorting_columns: bool = True) -> "HgFileMeta":
        """`ObjectBasedStorage::write_batch` on the GPU (storage.rs:189-225): sort by the primary keys, append the builtin columns,
        encode, write `out_path`.  `batch` holds the USER columns; it travels as an Arrow C struct array."""
        user = len(schema.arrow_schema) - 2
        if batch.num_columns != user:
            raise HgError(1, f"batch has {batch.num_columns} columns, the schema has {user} user columns")
        cols = [batch.column(i).cast(schema.arrow_schema.field(i).type) for i in range(user)]
        st = pa.StructArray.from_arrays(cols, fields=[schema.arrow_schema.field(i) for i in range(user)])

        class _CArray(C.Structure):
            _fields_ = [("length", C.c_int64), ("null_count", C.c_int64), ("offset", C.c_int64), ("n_buffers", C.c_int64), ("n_children", C.c_int64),
                        ("buffers", C.c_void_p), ("children", C.c_void_p), ("dictionary", C.c_void_p), ("release", C.c_void_p), ("private_data", C.c_void_p)]

        carr = _CArray()
        st._export_to_c(C.addressof(carr))
        props = HgWriteProps(max_row_group_size, _CODECS[compression.lower()], int(enable_sorting_columns), 0)
        meta = HgFileMeta()
        try:
            _check(self._L.hg_write_batch(self._h, C.byref(schema.desc), C.byref(carr), C.c_uint64(sequence), C.byref(props), out_path.encode(), C.byref(meta)))
        finally:
            pa.Array._import_from_c(C.addressof(carr), st.type)      # takes the exported array back: its release callback runs on GC
        return meta

    def scan_aggregate(self, schema: SchemaHandle, ssts: Sequence[SstInput], preds: Sequence[tuple] = (), group_col: int = 0,
                       ts_col: int = -1, window_ms: int = 0, value_col: int = -1, mode: int = 0) -> pa.Table:
        arr, keep = self._descs(ssts)
        p = _make_preds(schema.arrow_schema, preds)
        spec = HgAggSpec(group_col, ts_col, window_ms, value_col, mode)
        stream = ArrowArrayStream()
        _check(self._L.hg_scan_aggregate(self._h, C.byref(schema.desc), arr, C.c_size_t(len(ssts)), p, C.c_size_t(len(preds)),
                                         C.byref(spec), C.byref(stream)))
        return pa.RecordBatchReader._import_from_c(C.addressof(stream)).read_all()

    def scan_aggregate_device(self, schema: SchemaHandle, ssts: Sequence[SstInput], preds: Sequence[tuple] = (),
                              group_col: int = 0, ts_col: int = -1, window_ms: int = 0, value_col: int = -1, mode: int = 0) -> HgAggDevice:
        arr, keep = self._descs(ssts)
        p = _make_preds(schema.arrow_schema, preds)
        spec = HgAggSpec(group_col, ts_col, window_ms, value_col, mode)
        out = HgAggDevice()
        _check(self._L.hg_scan_aggregate_device(self._h, C.byref(schema.desc), arr, C.c_size_t(len(ssts)), p,
                                                C.c_size_t(len(preds)), C.byref(spec), C.byref(out)))
        return out

    def prepare_aggregate(self, schema: SchemaHandle, ssts: Sequence[SstInput], preds: Sequence[tuple] = (), group_col: int = 0,
                          ts_col: int = -1, window_ms: int = 0, value_col: int = -1, mode: int = 0) -> "PreparedAggregate":
        """Marshal the arguments of `scan_aggregate_device` once; `run()` is then a single C call (what a compiled host pays)."""
        return PreparedAggregate(self, schema, ssts, preds, group_col, ts_col, window_ms, value_col, mode)

    def stats_struct(self) -> "HgScanStats":
        """hg_last_stats into a reused ctypes struct (no dict): for tight measurement loops."""
        _check(self._L.hg_last_stats(self._h, C.byref(self._stats_buf)))
        return self._stats_buf

    def export_packed(self, d_dst: int, cap: int) -> None:
        """Pack the last device aggregate into a caller-owned [6, cap] int64 device buffer (engine stream)."""
        _check(self._L.hg_agg_export_packed(self._h, C.c_void_p(d_dst), C.c_uint64(cap)))

    # -- multi-GPU combine (comm.cu): the NCCL id travels over the host's own channel (here: torch.distributed)
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = (C.c_uint8 * 128)()
        _check(lib().hg_comm_unique_id(buf))
        return bytes(buf)

    def comm_init(self, uid: bytes, rank: int, world: int) -> None:
        buf = (C.c_uint8 * 128)(*uid)
        _check(self._L.hg_comm_init(self._h, buf, rank, world))

    def comm_destroy(self) -> None:
        _check(self._L.hg_comm_destroy(self._h))

    def combine(self, mode: int = 0, capacity_hint: int = 0) -> "HgAggCombined":
        out = HgAggCombined()
        _check(self._L.hg_agg_combine(self._h, C.c_uint32(mode), C.c_uint64(capacity_hint), C.byref(out)))
        return out

    def comm_sync(self) -> None:
        _check(self._L.hg_comm_sync(self._h))

    def stats(self) -> dict:
        st = HgScanStats()
        _check(self._L.hg_last_stats(self._h, C.byref(st)))
        return {f[0]: getattr(st, f[0]) for f in HgScanStats._fields_ if not f[0].startswith("_")}


class PreparedAggregate:
    """The ctypes argument block of one `hg_scan_aggregate_device` call, built once and reused."""

    def __init__(self, eng: Engine, schema: SchemaHandle, ssts, preds, group_col, ts_col, window_ms, value_col, mode=0):
        self._eng = eng
        self._schema = schema
        self._arr, self._keep = eng._descs(ssts)
        self._p = _make_preds(schema.arrow_schema, preds)
        self._spec = HgAggSpec(group_col, ts_col, window_ms, value_col, mode)
        self.out = HgAggDevice()
        self._fn = eng._L.hg_scan_aggregate_device
        self._args = (eng._h, C.byref(schema.desc), self._arr, C.c_size_t(len(ssts)), self._p, C.c_size_t(len(preds)),
                      C.byref(self._spec), C.byref(self.out))

    def run(self) -> HgAggDevice:
        rc = self._fn(*self._args)
        if rc:
            _check(rc)
        return self.out


def parquet_inspect(data: bytes) -> dict:
    """Host-only (no GPU): the library's reading of an SST's footer and page headers."""
    L = lib()
    buf = np.frombuffer(data, dtype=np.uint8)
    out = HgParquetSummary()
    _check(L.hg_parquet_inspect(C.c_void_p(buf.ctypes.data), C.c_uint64(buf.nbytes), C.byref(out)))
    return {f[0]: getattr(out, f[0]) for f in HgParquetSummary._fields_}


def parquet_chunk_info(data: bytes, row_group: int, column: int) -> dict:
    L = lib()
    buf = np.frombuffer(data, dtype=np.uint8)
    out = HgParquetChunk()
    _check(L.hg_parquet_chunk_info(C.c_void_p(buf.ctypes.data), C.c_uint64(buf.nbytes), C.c_uint32(row_group), C.c_uint32(column), C.byref(out)))
    d = {f[0]: getattr(out, f[0]) for f in HgParquetChunk._fields_}
    d["min"], d["max"] = bytes(out.min), bytes(out.max)
    return d


def plan_pk_splitters(schema: "SchemaHandle", datas: Sequence[bytes], parts: int) -> list:
    """Host-only (no GPU): `parts - 1` pk0 splitters that balance the rows of the inputs (multi-GPU compaction, SURVEY 8e)."""
    L = lib()
    arr = (HgSstDesc * max(len(datas), 1))()
    keep = []
    for i, d in enumerate(datas):
        buf = np.frombuffer(d, dtype=np.uint8)
        keep.append(buf)
        arr[i].id = i
        arr[i].data = buf.ctypes.data
        arr[i].size = buf.nbytes
    out = (C.c_uint64 * max(parts - 1, 1))()
    _check(L.hg_plan_pk_splitters(C.byref(schema.desc), arr, C.c_size_t(len(datas)), C.c_uint32(parts), out))
    t = schema.arrow_schema.field(0).type
    vals = [int(out[i]) for i in range(parts - 1)]
    if pa.types.is_signed_integer(t):
        vals = [v - (1 << 64) if v >= (1 << 63) else v for v in vals]
    return vals


def shard_range_preds(schema: "SchemaHandle", splitters: Sequence[int], rank: int) -> list:
    """The pk0 range of `rank` among len(splitters) + 1 shards, as predicates for `compact_to_sst(shard_preds=...)`."""
    name = schema.arrow_schema.field(0).name
    preds = []
    if rank > 0:
        preds.append((name, "ge", splitters[rank - 1]))
    if rank < len(splitters):
        preds.append((name, "lt", splitters[rank]))
    return preds


def plan_row_groups(schema: "SchemaHandle", data: bytes, preds: Sequence[tuple] = ()) -> list:
    """Host-only (no GPU): the planner's statistics pruning for one SST -> one 0/1 flag per row group."""
    L = lib()
    buf = np.frombuffer(data, dtype=np.uint8)
    p = _make_preds(schema.arrow_schema, preds)
    cap = 1 << 16
    keep = (C.c_uint8 * cap)()
    n = C.c_uint32()
    _check(L.hg_plan_row_groups(C.byref(schema.desc), C.c_void_p(buf.ctypes.data), C.c_uint64(buf.nbytes), p, C.c_size_t(len(preds)),
                                keep, C.c_uint32(cap), C.byref(n)))
    return [int(keep[i]) for i in range(n.value)]
