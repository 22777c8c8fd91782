"""Host-side mirror of `columnar_storage::storage` (storage.rs:58-375) and the compaction executor
(compaction/executor.rs:155-222, compaction/mod.rs:27-36) on top of the C ABI.

Same names, argument meaning and error behaviour as the reference so the parity tests read like its own
(`test_storage_write_and_scan`, storage.rs:391-491).  The manifest is an in-memory catalogue — the reference's
persistent manifest (manifest/mod.rs) is host control plane and out of scope (SURVEY §2 row 9).
"""
from __future__ import annotations

import itertools
import os
from dataclasses import dataclass, field
from typing import Iterator, List, Optional, Sequence

import pyarrow as pa

from . import sstgen
from ._ffi import Engine, SchemaHandle, SstInput
from .config import StorageConfig
from .sst import FileMeta, SstFile, SstPathGenerator, allocate_id
from .types import HoraeError, StorageSchema, TimeRange, ensure, _trunc_div


# ---- logical expressions (the subset of datafusion::Expr the GPU path lowers; anything else is rejected) ---------------
@dataclass
class Expr:
    column: str
    op: str
    literal: object


class _Col:
    def __init__(self, name):
        self.name = name

    def eq(self, lit_): return Expr(self.name, "eq", lit_)
    def not_eq(self, lit_): return Expr(self.name, "ne", lit_)
    def lt(self, lit_): return Expr(self.name, "lt", lit_)
    def lt_eq(self, lit_): return Expr(self.name, "le", lit_)
    def gt(self, lit_): return Expr(self.name, "gt", lit_)
    def gt_eq(self, lit_): return Expr(self.name, "ge", lit_)


def col(name: str) -> _Col:
    return _Col(name)


def lit(v):
    return v


@dataclass
class WriteRequest:  # storage.rs:58-63
    batch: pa.RecordBatch
    time_range: TimeRange
    enable_check: bool = True


@dataclass
class ScanRequest:  # storage.rs:65-70
    range: TimeRange
    predicate: List[Expr] = field(default_factory=list)
    projections: Optional[List[int]] = None


@dataclass
class CompactRequest:  # storage.rs:72-73
    pass


@dataclass
class Task:  # compaction/mod.rs:27-36
    inputs: List[SstFile]
    expireds: List[SstFile] = field(default_factory=list)

    def input_size(self) -> int:
        return sum(f.size() for f in self.inputs)


class Manifest:
    """In-memory stand-in for manifest/mod.rs:67-177 (`find_ssts` = linear overlap filter, mod.rs:165-172)."""

    def __init__(self):
        self.ssts: List[SstFile] = []

    def add_file(self, id: int, meta: FileMeta):
        self.ssts.append(SstFile(id, meta))

    def find_ssts(self, rng: TimeRange) -> List[SstFile]:
        return [f for f in self.ssts if f.meta().time_range.overlaps(rng)]

    def all_ssts(self) -> List[SstFile]:
        return list(self.ssts)

    def update(self, to_adds: List[SstFile], to_deletes: List[int]):
        self.ssts = [f for f in self.ssts if f.id() not in set(to_deletes)] + to_adds


class ObjectBasedStorage:
    """`ObjectBasedStorage` (storage.rs:106-375) with the scan/compaction data path on the GPU engine."""

    def __init__(self, path: str, segment_duration_ms: int, arrow_schema: pa.Schema, num_primary_keys: int,
                 config: Optional[StorageConfig] = None, engine: Optional[Engine] = None):
        self.config = config or StorageConfig()
        self.segment_duration = segment_duration_ms
        self.path = path
        self.schema_ = StorageSchema.try_new(arrow_schema, num_primary_keys, self.config.update_mode)
        self.manifest = Manifest()
        self.sst_path_gen = SstPathGenerator(path)
        self._engine = engine            # created on first use: the write path never touches the GPU
        self.handle = SchemaHandle(self.schema_.arrow_schema, num_primary_keys, self.config.update_mode)
        self.inused_memory = 0
        os.makedirs(os.path.join(path, "data"), exist_ok=True)

    @property
    def engine(self) -> Engine:
        if self._engine is None:
            self._engine = Engine()
        return self._engine

    def schema(self) -> pa.Schema:
        return self.schema_.arrow_schema

    # ---- write (storage.rs:189-225, 307-333): defines the SST; not on the accelerated path
    def write(self, req: WriteRequest) -> None:
        if req.enable_check:
            seg = self.segment_duration
            ensure(_trunc_div(req.time_range.start, seg) == _trunc_div(req.time_range.end - 1, seg),
                   f"time range can't cross segment, value:{req.time_range!r}")
        file_id = allocate_id()
        fpath = self.sst_path_gen.generate(file_id)
        w = self.config.write
        gpu_writer = (hasattr(self.engine, "write_batch") and w.encoding == "PLAIN" and not w.enable_dict and not w.column_options
                      and not any(pa.types.is_binary(f.type) for f in self.schema_.arrow_schema)
                      and str(w.compression).lower() in ("snappy", "zstd", "uncompressed", "none")
                      and all(req.batch.column(i).null_count == 0 for i in range(self.schema_.num_primary_keys)))
        if gpu_writer:
            # write_batch on the GPU (hg_write_batch): PK sort, builtin columns, Parquet encode
            meta = self.engine.write_batch(self.handle, req.batch, file_id, fpath, max_row_group_size=w.max_row_group_size,
                                           compression=str(w.compression), enable_sorting_columns=w.enable_sorting_columns)
            size = meta.size
        else:
            # writer options the GPU encoder does not implement (dictionary / delta encodings, NULL keys): host Parquet writer
            data = sstgen.write_sst(self.schema_, req.batch, file_id, self.config.write)
            with open(fpath, "wb") as f:
                f.write(data)
            size = len(data)
        self.manifest.add_file(file_id, FileMeta(max_sequence=file_id, num_rows=req.batch.num_rows, size=size,
                                                 time_range=req.time_range))

    def _inputs(self, ssts: Sequence[SstFile]) -> List[SstInput]:
        return [SstInput(id=f.id(), path=self.sst_path_gen.generate(f.id()), num_rows=f.meta().num_rows,
                         time_start=f.meta().time_range.start, time_end=f.meta().time_range.end,
                         max_sequence=f.meta().max_sequence) for f in ssts]

    def _lower(self, exprs: Sequence[Expr]):
        preds = []
        for e in exprs:
            if not isinstance(e, Expr):
                raise HoraeError(f"predicate {e!r} cannot be lowered to the GPU path (no CPU fallback)")
            preds.append((e.column, e.op, e.literal))
        return preds

    # ---- scan (storage.rs:335-370)
    def scan(self, req: ScanRequest) -> Iterator[pa.RecordBatch]:
        total_ssts = self.manifest.find_ssts(req.range)          # `range` prunes FILES only (SURVEY §8 quirk 1)
        if not total_ssts:
            return iter(())
        seg = self.segment_duration
        groups = [(k, list(g)) for k, g in itertools.groupby(
            total_ssts, key=lambda f: _trunc_div(f.meta().time_range.start, seg))]   # consecutive files (quirk 4)
        groups.sort(key=lambda kv: kv[0])
        preds = self._lower(req.predicate)
        projection = None if req.projections is None else list(req.projections)

        def gen():
            for _, ssts in groups:
                reader = self.engine.scan(self.handle, self._inputs(ssts), preds, projection, keep_builtin=False)
                for b in reader:
                    yield b
        return gen()

    # ---- compaction (executor.rs:155-222)
    def pre_check(self, task: Task) -> None:  # executor.rs:93-114
        assert task.inputs
        limit = self.config.scheduler.memory_limit
        ensure(self.inused_memory + task.input_size() <= limit,
               f"Compaction memory usage too high, inused:{self.inused_memory}, task_size:{task.input_size()}, limit:{limit}")
        self.inused_memory += task.input_size()

    def do_compaction(self, task: Task) -> SstFile:
        self.pre_check(task)
        try:
            time_range = TimeRange(task.inputs[0].meta().time_range.start, task.inputs[0].meta().time_range.end)
            for f in task.inputs[1:]:
                time_range.merge(f.meta().time_range)
            file_id = allocate_id()
            w = self.config.write
            if (w.encoding == "PLAIN" and not w.enable_dict and not w.column_options and str(w.compression).lower() in ("snappy", "zstd", "uncompressed", "none")
                    and not any(pa.types.is_binary(f.type) for f in self.schema_.arrow_schema)):
                # the whole of do_compaction on the GPU: merge + dedup (keep_builtin = true) AND the Parquet encode (hg_compact_to_sst)
                meta = self.engine.compact_to_sst(self.handle, self._inputs(task.inputs), self.sst_path_gen.generate(file_id),
                                                  max_row_group_size=w.max_row_group_size, compression=str(w.compression),
                                                  enable_sorting_columns=w.enable_sorting_columns)
                num_rows, size = meta.num_rows, meta.size
            else:
                # writer options the GPU encoder does not implement (dictionary / delta encodings ..): the merged stream comes
                # back as Arrow batches (hg_compact_open) and the host writes the file, like the reference's AsyncArrowWriter
                reader = self.engine.compact(self.handle, self._inputs(task.inputs))   # same plan, keep_builtin=true
                tbl = reader.read_all()
                batch = tbl.combine_chunks().to_batches()[0] if tbl.num_rows else pa.RecordBatch.from_arrays(
                    [pa.array([], f.type) for f in self.schema_.arrow_schema], schema=self.schema_.arrow_schema)
                data = sstgen.write_sst_with_seq(self.schema_, batch, self.config.write)
                with open(self.sst_path_gen.generate(file_id), "wb") as f:
                    f.write(data)
                num_rows, size = tbl.num_rows, len(data)
            new = SstFile(file_id, FileMeta(max_sequence=file_id, num_rows=num_rows, size=size, time_range=time_range))
            to_deletes = [f.id() for f in task.expireds] + [f.id() for f in task.inputs]
            self.manifest.update([new], to_deletes)          # manifest first, then delete (executor.rs:205-220)
            for fid in to_deletes:
                try:
                    self.engine.unload_sst(fid)
                except Exception:
                    pass
                try:
                    os.remove(self.sst_path_gen.generate(fid))
                except OSError:
                    pass
            self.inused_memory -= task.input_size()           # on_success (executor.rs:116-121)
            return new
        except Exception:
            self.inused_memory -= task.input_size()           # on_failure (executor.rs:123-137)
            for f in task.inputs + task.expireds:
                f.unmark_compaction()
            raise

    def compact(self, req: CompactRequest = CompactRequest()) -> List[SstFile]:
        """storage.rs:372-374 triggers the scheduler; this mirror compacts every segment that has > 1 SST."""
        seg = self.segment_duration
        by_seg = {}
        for f in self.manifest.all_ssts():
            by_seg.setdefault(_trunc_div(f.meta().time_range.start, seg), []).append(f)
        out = []
        for _, files in sorted(by_seg.items()):
            if len(files) > 1:
                for f in files:
                    f.mark_compaction()
                out.append(self.do_compaction(Task(files)))
        return out
