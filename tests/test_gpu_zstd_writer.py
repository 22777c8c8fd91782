"""GPU SST writer with Zstandard pages (hg_compact_to_sst / hg_write_batch with compression = 6, csrc/sst_writer.cu
zstd_encode_kernel).  Every file is read by three independent Zstandard decoders — pyarrow (libzstd), the CPU oracle
(oracle/zstd_oracle.h) and the engine itself (zstd_core.h) — and must hold the rows the host writer would write.  The files
must also be worth choosing Zstd for: well under the GPU's own Snappy output, and within 1.30x of libzstd level 1."""
import io

import numpy as np
import pyarrow as pa
import pyarrow.parquet as pq
import pytest

from horaedb_b200 import sstgen
from horaedb_b200._ffi import Engine, SchemaHandle, SstInput, parquet_inspect
from horaedb_b200.config import WriteConfig
from oracle import oracle

from helpers import arrays_equal, arrow_schema, record_batch

pytestmark = pytest.mark.gpu
_ids = iter(range(95_000_000, 99_000_000))


def _inputs(datas):
    return [SstInput(id=next(_ids), data=d, time_start=10 * i, time_end=10 * i + 5, max_sequence=100 + i) for i, d in enumerate(datas)]


def _chunk_bytes(data):
    """sum of total_compressed_size over all column chunks (page headers + page bytes)"""
    md = pq.ParquetFile(io.BytesIO(data)).metadata
    return sum(md.row_group(g).column(c).total_compressed_size for g in range(md.num_row_groups) for c in range(md.num_columns))


def _check_file(eng, schema, npk, data, exp, rg, aggregate=False):
    """the file against the expected table: pyarrow (libzstd), the oracle, the engine; statistics, sort order, codec"""
    names = exp.schema.names
    pf = pq.ParquetFile(io.BytesIO(data))
    got = pf.read()
    assert got.schema.names == names
    for name in names:
        assert got[name].type == exp[name].type, name
        assert arrays_equal(got[name], exp[name]), name
    md = pf.metadata
    assert md.num_row_groups == (exp.num_rows + rg - 1) // rg
    for g in range(md.num_row_groups):
        lo, hi = g * rg, min(exp.num_rows, (g + 1) * rg)
        assert md.row_group(g).num_rows == hi - lo
        assert [x.column_index for x in md.row_group(g).sorting_columns] == list(range(npk))
        for c, name in enumerate(names):
            col = md.row_group(g).column(c)
            assert col.compression == "ZSTD", (g, name)
            part = exp[name].combine_chunks().slice(lo, hi - lo)
            st = col.statistics
            assert st.null_count == part.null_count, (g, name)
            if part.null_count < len(part) and not pa.types.is_floating(part.type):
                assert st.min == pa.compute.min(part).as_py() and st.max == pa.compute.max(part).as_py(), (g, name)
    if md.num_row_groups:
        assert parquet_inspect(data)["codec_mask"] & (1 << 6)
    again = pa.Table.from_batches(oracle.scan([data], schema.arrow_schema, npk, (), True, 8192).batches, schema=exp.schema)
    assert all(arrays_equal(again[name], exp[name]) for name in names)
    handle = SchemaHandle(schema.arrow_schema, npk)
    rescan = pa.Table.from_batches(list(eng.scan(handle, [SstInput(id=next(_ids), data=data)], (), None, True)), schema=exp.schema)
    assert all(arrays_equal(rescan[name], exp[name]) for name in names)
    if aggregate:
        preds = [("tag", "eq", 3), ("ts", "ge", sstgen.T0_MS + 100_000)]
        kw = dict(group_col=0, ts_col=-1, window_ms=0, value_col=2)
        a = eng.scan_aggregate(handle, [SstInput(id=next(_ids), data=data)], preds, **kw)
        b = oracle.scan_aggregate([data], schema.arrow_schema, npk, preds, **kw)
        assert a["count"].to_numpy().tolist() == b.count.tolist() and np.array_equal(a["sum"].to_numpy(), b.sum)


@pytest.mark.parametrize("rg", [8192, 1000])
def test_zstd_compaction_round_trips(tmp_path, rg):
    schema = sstgen.metric_storage_schema()
    handle = SchemaHandle(schema.arrow_schema, 2)
    datas = [s[0] for s in sstgen.synth_overlapping_ssts(9, series=60, points=700, delta_ms=1000, keep_frac=0.4, compression="snappy")]
    exp = pa.Table.from_batches(oracle.scan(datas, schema.arrow_schema, 2, (), True, 8192).batches)
    eng = Engine(device=0)
    files = {}
    for codec in ("zstd", "snappy"):
        path = str(tmp_path / f"{codec}.sst")
        meta = eng.compact_to_sst(handle, _inputs(datas), path, max_row_group_size=rg, compression=codec)
        files[codec] = open(path, "rb").read()
        assert meta.size == len(files[codec]) and meta.num_rows == exp.num_rows and meta.max_sequence == 108
    _check_file(eng, schema, 2, files["zstd"], exp, rg, aggregate=True)
    assert _chunk_bytes(files["zstd"]) < _chunk_bytes(files["snappy"])
    # the same compaction again: the same bytes
    path = str(tmp_path / "again.sst")
    eng.compact_to_sst(handle, _inputs(datas), path, max_row_group_size=rg, compression="zstd")
    assert open(path, "rb").read() == files["zstd"]
    eng.close()


@pytest.fixture(scope="module")
def metric_100k():
    """a metric compaction of > 100 k rows (4 overlapping SSTs of 120 series x 1000 points)"""
    schema = sstgen.metric_storage_schema()
    datas = [s[0] for s in sstgen.synth_overlapping_ssts(4, series=120, points=1000, delta_ms=1000, keep_frac=0.5, compression="none")]
    exp = pa.Table.from_batches(oracle.scan(datas, schema.arrow_schema, 2, (), True, 8192).batches)
    assert exp.num_rows >= 100_000
    return schema, datas, exp


def test_zstd_ratio_against_libzstd_level_1(tmp_path, metric_100k):
    """the bar: at most 1.30x the column-chunk bytes of pyarrow's Zstd level 1 on the same table, and below the GPU's own Snappy"""
    schema, datas, exp = metric_100k
    handle = SchemaHandle(schema.arrow_schema, 2)
    eng = Engine(device=0)
    got = {}
    for codec in ("zstd", "snappy"):
        path = str(tmp_path / f"{codec}.sst")
        eng.compact_to_sst(handle, _inputs(datas), path, max_row_group_size=8192, compression=codec)
        got[codec] = open(path, "rb").read()
    _check_file(eng, schema, 2, got["zstd"], exp, 8192, aggregate=True)
    buf = io.BytesIO()
    pq.write_table(exp, buf, row_group_size=8192, compression="zstd", compression_level=1, use_dictionary=False)
    ref = _chunk_bytes(buf.getvalue())
    z, s = _chunk_bytes(got["zstd"]), _chunk_bytes(got["snappy"])
    assert z <= 1.30 * ref, (z, ref, z / ref)
    assert z < s, (z, s)
    eng.close()


def test_zstd_pages_of_several_blocks(tmp_path, metric_100k):
    """row groups of 50 000 rows: an 8-byte column's page is 400 KB, i.e. four 128 KB Zstandard blocks in one frame"""
    schema, datas, exp = metric_100k
    handle = SchemaHandle(schema.arrow_schema, 2)
    eng = Engine(device=0)
    path = str(tmp_path / "big.sst")
    eng.compact_to_sst(handle, _inputs(datas), path, max_row_group_size=50_000, compression="zstd")
    data = open(path, "rb").read()
    md = pq.ParquetFile(io.BytesIO(data)).metadata
    assert md.row_group(0).column(exp.schema.names.index("ts")).total_uncompressed_size > 3 * (128 << 10)
    _check_file(eng, schema, 2, data, exp, 50_000, aggregate=True)
    path_s = str(tmp_path / "big_snappy.sst")
    eng.compact_to_sst(handle, _inputs(datas), path_s, max_row_group_size=50_000, compression="snappy")
    assert _chunk_bytes(data) < _chunk_bytes(open(path_s, "rb").read())
    eng.close()


def test_zstd_all_types_nulls_and_empty(tmp_path):
    """Every primitive type, NULLs (bit-packed definition levels, all-null pages), NaN / -0.0, a one-row tail row group, an empty output."""
    from horaedb_b200.types import StorageSchema
    rng = np.random.default_rng(5)
    user = arrow_schema([("a", "int64"), ("b", "uint32"), ("u8", "uint8"), ("i8", "int8"), ("u16", "uint16"), ("i16", "int16"), ("i32", "int32"),
                         ("u64", "uint64"), ("f32", "float32"), ("f64", "float64")])
    schema = StorageSchema.try_new(user, 2)
    n = 2501

    def maybe(vals, p):
        return [None if rng.random() < p else v for v in vals]

    cols = {"a": (np.arange(n) - 1000).tolist(), "b": rng.integers(0, 7, n).tolist(),
            "u8": maybe(rng.integers(0, 256, n).tolist(), 0.2), "i8": maybe(rng.integers(-128, 128, n).tolist(), 0.0),
            "u16": maybe(rng.integers(0, 65536, n).tolist(), 0.5), "i16": maybe(rng.integers(-32768, 32768, n).tolist(), 0.01),
            "i32": maybe(rng.integers(-2**31, 2**31, n).tolist(), 0.3), "u64": maybe(rng.integers(0, 2**63, n).tolist(), 1.0),
            "f32": maybe(rng.choice([float("nan"), -0.0, 0.0, 1.5, -3.25], n).tolist(), 0.1),
            "f64": maybe(rng.choice([float("nan"), -0.0, 0.0, 2.5, 1e300], n).tolist(), 0.1)}
    b = record_batch(user, cols)
    b = pa.Table.from_batches([b]).sort_by([("a", "ascending"), ("b", "ascending")]).combine_chunks().to_batches()[0]
    data = sstgen.write_sst(schema, b, seq=77, cfg=WriteConfig(max_row_group_size=400))
    handle = SchemaHandle(schema.arrow_schema, 2)
    eng = Engine(device=0)
    exp = pa.Table.from_batches(oracle.scan([data], schema.arrow_schema, 2, (), True, 8192).batches)
    path = str(tmp_path / "t.sst")
    meta = eng.compact_to_sst(handle, [SstInput(id=next(_ids), data=data)], path, max_row_group_size=500, compression="zstd")
    assert meta.num_rows == n
    out = open(path, "rb").read()
    _check_file(eng, schema, 2, out, exp, 500)
    md = pq.ParquetFile(io.BytesIO(out)).metadata
    assert md.row_group(5).num_rows == 1
    f64 = pq.read_table(io.BytesIO(out))["f64"].to_numpy(zero_copy_only=False)
    assert np.array_equal(np.signbit(f64), np.signbit(exp["f64"].to_numpy(zero_copy_only=False)))
    assert "ZSTD" in md.created_by
    # empty output
    empty = sstgen.write_sst(schema, b.slice(0, 0), seq=78)
    path = str(tmp_path / "empty.sst")
    meta = eng.compact_to_sst(handle, [SstInput(id=next(_ids), data=empty)], path, compression="zstd")
    assert meta.num_rows == 0 and pq.read_table(path).num_rows == 0
    eng.close()


def test_zstd_incompressible_and_constant_columns(tmp_path):
    """random 64 / 32-bit values are stored (Raw blocks) at most a few bytes per page above their uncompressed size;
    a constant column shrinks to a few dozen bytes per page"""
    from horaedb_b200.types import StorageSchema
    rng = np.random.default_rng(6)
    user = arrow_schema([("k", "int64"), ("r", "uint64"), ("q", "int32"), ("c", "float64"), ("d", "int32")])
    schema = StorageSchema.try_new(user, 1)
    n = 45_000
    batch = record_batch(user, {"k": np.arange(n).tolist(), "r": rng.integers(0, 2**64 - 1, n, dtype=np.uint64).tolist(),
                                "q": rng.integers(-2**31, 2**31, n).tolist(), "c": [42.5] * n, "d": [7] * n})
    handle = SchemaHandle(schema.arrow_schema, 1)
    eng = Engine(device=0)
    files = {}
    for codec in ("zstd", "none"):
        path = str(tmp_path / f"{codec}.sst")
        eng.write_batch(handle, batch, 9, path, max_row_group_size=20_000, compression=codec)
        files[codec] = open(path, "rb").read()
    exp = pq.read_table(io.BytesIO(files["none"]))
    _check_file(eng, schema, 1, files["zstd"], exp, 20_000)
    mz, mn = pq.ParquetFile(io.BytesIO(files["zstd"])).metadata, pq.ParquetFile(io.BytesIO(files["none"])).metadata
    for g in range(mz.num_row_groups):
        for name in ("r", "q"):
            c = exp.schema.names.index(name)
            z, u = mz.row_group(g).column(c).total_compressed_size, mn.row_group(g).column(c).total_compressed_size
            blocks = (mn.row_group(g).column(c).total_uncompressed_size + (128 << 10) - 1) // (128 << 10)
            assert z <= u + 12 + 3 * blocks, (g, name, z, u)
        for name in ("c", "d"):
            assert mz.row_group(g).column(exp.schema.names.index(name)).total_compressed_size < 100, (g, name)
    eng.close()


@pytest.mark.parametrize("world", [2])
def test_zstd_range_sharded_compaction(tmp_path, world):
    from horaedb_b200._ffi import plan_pk_splitters, shard_range_preds
    schema = sstgen.metric_storage_schema()
    handle = SchemaHandle(schema.arrow_schema, 2)
    datas = [s[0] for s in sstgen.synth_overlapping_ssts(12, series=300, points=400, delta_ms=1000, keep_frac=0.3, compression="snappy")]
    exp = pa.Table.from_batches(oracle.scan(datas, schema.arrow_schema, 2, (), True, 8192).batches)
    eng = Engine(device=0)
    sp = plan_pk_splitters(handle, datas, world)
    parts = []
    for r in range(world):
        path = str(tmp_path / f"shard{r}.sst")
        meta = eng.compact_to_sst(handle, _inputs(datas), path, shard_preds=shard_range_preds(handle, sp, r), compression="zstd")
        data = open(path, "rb").read()
        t = pq.read_table(io.BytesIO(data))
        assert t.num_rows == meta.num_rows
        assert all(pq.ParquetFile(io.BytesIO(data)).metadata.row_group(g).column(0).compression == "ZSTD"
                   for g in range(pq.ParquetFile(io.BytesIO(data)).metadata.num_row_groups))
        parts.append(t)
    got = pa.concat_tables(parts)
    for name in exp.schema.names:
        assert got[name].combine_chunks().equals(exp[name].combine_chunks()), name
    eng.close()


def test_zstd_write_batch_matches_the_host_writer(tmp_path):
    """hg_write_batch with Zstd: the same contents as the host writer (pyarrow, WriteConfig compression = Zstd) for the same batch"""
    from horaedb_b200.types import StorageSchema
    rng = np.random.default_rng(13)
    user = arrow_schema([("a", "int32"), ("b", "uint64"), ("c", "int8"), ("v", "float64"), ("w", "uint16")])
    schema = StorageSchema.try_new(user, 3)
    n = 30_000
    cols = {"a": rng.integers(-50, 50, n).tolist(), "b": rng.integers(0, 2**40, n).tolist(), "c": rng.integers(-128, 128, n).tolist(),
            "v": [None if rng.random() < 0.1 else float(x) for x in rng.random(n)],
            "w": [None if rng.random() < 0.5 else int(x) for x in rng.integers(0, 65536, n)]}
    batch = record_batch(user, cols)
    handle = SchemaHandle(schema.arrow_schema, 3)
    eng = Engine(device=0)
    for rg in (8192, 1000):
        path = str(tmp_path / f"w_{rg}.sst")
        meta = eng.write_batch(handle, batch, 4242, path, max_row_group_size=rg, compression="zstd")
        assert meta.num_rows == n and meta.max_sequence == 4242
        data = open(path, "rb").read()
        host = sstgen.write_sst(schema, batch, 4242, WriteConfig(max_row_group_size=rg, compression="zstd"))
        want = pq.read_table(io.BytesIO(host))
        _check_file(eng, schema, 3, data, want, rg)
    eng.close()
