/*
 * horae_gpu.h — C ABI of libhorae_gpu.so, the B200 (sm_100a) implementation of HoraeDB's columnar hot path.
 *
 * Every entry point replaces one seam of the reference (paths relative to apache/horaedb @ 9cec5636,
 * src/columnar_storage/src/):
 *
 *   hg_scan_open         ParquetReader::build_df_plan(ssts, projection, predicates, keep_builtin=false)
 *                        + execute_stream                      read.rs:429-494, storage.rs:350-369
 *                        i.e. ParquetExec -> FilterExec -> SortPreservingMergeExec -> MergeExec(LastValue)
 *   hg_compact_open      the same plan as built by Executor::do_compaction: no predicate, keep_builtin=true
 *                                                              compaction/executor.rs:164-171
 *   hg_scan_aggregate*   the time-bucket aggregation the metric engine is meant to run on top of the scan
 *                        (absent in the reference: metric_engine/src/metric/mod.rs:37-49 is todo!();
 *                        window arithmetic = Timestamp::truncate_by, types.rs:82-85)
 *   hg_sst_load/unload   residency of immutable SST bytes in HBM, keyed by FileId (sst.rs:48, 193-205)
 *   hg_schema_desc       StorageSchema (types.rs:143-157);   hg_sst_desc = SstFile + FileMeta (sst.rs:51-53,155-160)
 *   hg_predicate         the lowered form of ScanRequest.predicate: Vec<Expr> (storage.rs:65-70) — a conjunction of
 *                        `column <op> literal`; anything else must be rejected by the caller (no CPU fallback)
 *
 * Results travel as Arrow C streams (arrow_c_abi.h): the Rust shim wraps them with
 * arrow::ffi_stream::ArrowArrayStreamReader and hands the batches to DataFusion (see INTEGRATION.md).
 *
 * Conventions: plain C types only; every function returns an hg_status (0 = OK) and records a message readable with
 * hg_last_error() on the calling thread; nothing throws or aborts across the boundary.  The engine handle is
 * thread-safe (calls are serialised per engine); streams may be consumed from any thread.
 */
#ifndef HORAE_GPU_H
#define HORAE_GPU_H

#include <stddef.h>
#include <stdint.h>

#include "arrow_c_abi.h"

#ifdef __cplusplus
extern "C" {
#endif

#define HG_ABI_VERSION 4u

typedef struct hg_engine hg_engine;

typedef enum {
  HG_OK = 0,
  HG_ERR_INVALID = 1,      /* bad argument / schema mismatch                       (ensure!, macros.rs:36-52) */
  HG_ERR_UNSUPPORTED = 2,  /* encoding / codec / type / expression not implemented on the GPU path (never a CPU fallback) */
  HG_ERR_CUDA = 3,
  HG_ERR_FORMAT = 4,       /* malformed Parquet: footer / page headers, or page contents found inconsistent on the device (levels, dictionary
                              indices, compressed streams, rows that contradict their chunk statistics or the file's sort order) */
  HG_ERR_OOM = 5,          /* HBM admission control (the analogue of Executor::pre_check, executor.rs:93-114) */
  HG_ERR_NOT_FOUND = 6,
  HG_ERR_INTERNAL = 7
} hg_status;

/* Arrow primitive types the reference's primary_key_eq / value columns use (read.rs:269-286) */
typedef enum {
  HG_U8 = 0, HG_I8 = 1, HG_U16 = 2, HG_I16 = 3, HG_U32 = 4, HG_I32 = 5, HG_U64 = 6, HG_I64 = 7, HG_F32 = 8, HG_F64 = 9,
  HG_BINARY = 10   /* Arrow Binary / Parquet BYTE_ARRAY: value columns only (what BytesMergeOperator concatenates, operator.rs:47-111) */
} hg_type;

typedef enum { HG_UPDATE_OVERWRITE = 0, HG_UPDATE_APPEND = 1 } hg_update_mode; /* config.rs:166-172 */

typedef enum { HG_OP_EQ = 0, HG_OP_NE = 1, HG_OP_LT = 2, HG_OP_LE = 3, HG_OP_GT = 4, HG_OP_GE = 5, HG_OP_IN = 6 } hg_op;
#define HG_MAX_IN_LIST 64u

/* StorageSchema (types.rs:143-157): columns = pk0..pkN-1, values..., __seq__ (u64), __reserved__ (u64) */
typedef struct {
  uint32_t num_columns;       /* including the two builtin columns */
  uint32_t num_primary_keys;
  uint32_t update_mode;       /* hg_update_mode: OVERWRITE = LastValueOperator (operator.rs:37-44); APPEND = BytesMergeOperator
                                 (operator.rs:47-111: every value column must be HG_BINARY; the run's values are concatenated in
                                 (pk, seq) order, the other columns come from the run's FIRST row) */
  uint32_t _pad;
  const uint32_t* types;      /* hg_type per column */
  const char* const* names;   /* column names (for the exported Arrow schema) */
} hg_schema_desc;

typedef struct {
  int32_t device;             /* CUDA ordinal (one engine per GPU / per rank) */
  uint32_t batch_size;        /* DataFusion batch_size the merge re-batches at; 0 = 8192 */
  uint64_t hbm_budget_bytes;  /* 0 = no admission limit */
  uint32_t flags;             /* HG_FLAG_* */
  uint32_t _pad;
} hg_config;

#define HG_FLAG_NO_PRUNING 1u   /* disable row-group pruning by chunk statistics (for A/B measurements) */
#define HG_FLAG_NO_FUSED 2u     /* force the general (materialising) pipeline even when the fused fast path applies */
#define HG_FLAG_NO_LATE_MATERIALIZATION 4u   /* fused path: load every needed column of every row (no predicate gate) */
#define HG_FLAG_PAIRWISE_MERGE 8u   /* k-way merge by log2(k) pairwise passes over 32-byte records even when the packed-key single pass applies (A/B) */

/* SstFile + FileMeta (sst.rs:51-53, 155-160).  `data` may be NULL when the file is already resident (hg_sst_load). */
typedef struct {
  uint64_t id;
  const uint8_t* data;        /* whole-file bytes in host memory, or NULL */
  uint64_t size;
  const char* path;           /* optional: "{root}/data/{id}.sst" (sst.rs:202-204), read when data == NULL and not resident */
  uint32_t num_rows;
  uint32_t _pad;
  int64_t time_start, time_end;   /* [start, end) */
  uint64_t max_sequence;
} hg_sst_desc;

typedef struct {
  uint32_t column;            /* index into the storage schema */
  uint32_t op;                /* hg_op */
  int64_t i64;                /* literal for signed integer columns */
  uint64_t u64;               /* literal for unsigned integer columns */
  double f64;                 /* literal for float columns */
  const uint64_t* in_values;  /* HG_OP_IN (`col IN (..)`, DataFusion InListExpr): in_count values in the column's widened domain */
  uint32_t in_count, _pad;    /*   (i64 / u64 two's complement, f64 bit patterns); at most HG_MAX_IN_LIST; NULL IN (..) is false */
} hg_predicate;

/* GROUP BY (group column, time bucket) over the post-dedup scan output.
 * mode HG_AGG_RUNS: groups are the maximal runs of equal (group value, bucket) in the stream — exact GROUP BY when the key
 *   is a prefix of the sort order (series_id [, ts bucket]); groups come out in stream (key) order.
 * mode HG_AGG_HASH: true GROUP BY for ANY key (e.g. per-(tag, bucket)): radix-partitioned, every group's rows are added in
 *   stream order, groups come out sorted by (group value, bucket).  Identical to RUNS for sort-prefix keys. */
typedef enum { HG_AGG_RUNS = 0, HG_AGG_HASH = 1 } hg_agg_mode;
typedef struct {
  int32_t group_col;          /* -1: one global group */
  int32_t ts_col;             /* -1: no bucketing */
  int64_t window_ms;          /* bucket = ts / window_ms * window_ms (truncating, types.rs:82-85) */
  int32_t value_col;          /* -1: count(*) only */
  uint32_t mode;              /* hg_agg_mode */
} hg_agg_spec;

typedef struct {
  uint64_t rows_in_files;     /* rows of the selected SSTs */
  uint64_t rows_decoded;      /* after row-group pruning */
  uint64_t rows_filtered;     /* after the predicate */
  uint64_t rows_out;          /* after merge + dedup */
  uint64_t groups_out;
  uint64_t bytes_h2d, bytes_d2h;
  uint32_t kernel_launches;   /* kernels launched by the last call */
  uint32_t path;              /* bit 0: 0 = general pipeline, 1 = fused fast path;  bit 1: the call ran twice (a transient load's
                                 compressed page prefix ended before the last needed row: repeated with whole pages) */
  float gpu_ms;               /* device time of the last call, first kernel to last (CUDA events on the engine stream) */
  float kernel_ms;            /* device time of the call's dominant kernel alone (fused scan / page decode) */
  float merge_ms;             /* device time of S4-S6 (sort records, merge passes, dedup, compaction of survivors) */
  float decomp_ms;            /* device time of the page-decompression stage (Snappy; fused path), when one ran */
  uint64_t rows_materialized; /* fused path: rows whose non-gate columns were read (== rows_decoded without the gate);
                                 general pipeline: rows_decoded */
} hg_scan_stats;

/* Device-resident aggregate (for the NCCL combine and HBM-resident timing); valid until the next call on the engine. */
typedef struct {
  uint64_t num_groups;
  const void* d_gkey;         /* group column values, native width */
  const int64_t* d_bucket;
  const uint64_t* d_count;
  const double* d_sum;
  const double* d_min;
  const double* d_max;
} hg_agg_device;

uint32_t hg_abi_version(void);
const char* hg_last_error(void);

int hg_engine_create(const hg_config* cfg, hg_engine** out);
void hg_engine_destroy(hg_engine* e);
void* hg_engine_stream(hg_engine* e); /* the cudaStream_t every kernel of this engine is launched on */
int hg_engine_set_flags(hg_engine* e, uint32_t flags); /* replaces hg_config.flags for the following calls (A/B measurements) */

int hg_sst_load(hg_engine* e, const hg_schema_desc* schema, const hg_sst_desc* sst);
int hg_sst_unload(hg_engine* e, uint64_t id);
int hg_sst_resident_bytes(hg_engine* e, uint64_t* out);

int hg_scan_open(hg_engine* e, const hg_schema_desc* schema, const hg_sst_desc* ssts, size_t n_ssts,
                 const hg_predicate* preds, size_t n_preds, const uint32_t* projection, size_t n_projection,
                 int keep_builtin, struct ArrowArrayStream* out);

int hg_compact_open(hg_engine* e, const hg_schema_desc* schema, const hg_sst_desc* ssts, size_t n_ssts,
                    struct ArrowArrayStream* out);

/* build_write_props (storage.rs:258-298) / WriteConfig (config.rs:120-133) as far as the GPU writer implements them:
 * PLAIN values, RLE definition levels, dictionary off, bloom filters off, chunk statistics on, one DataPage V1 per chunk. */
typedef struct {
  uint32_t max_row_group_size;      /* 0 = 8192 (WriteConfig::default) */
  uint32_t compression;             /* Parquet codec id the WRITER applies (config.rs:78-94): 0 UNCOMPRESSED, 1 SNAPPY (the default),
                                       6 ZSTD (one frame per page, blocks of <= 128 KB).  Zstd SSTs are read on the general pipeline */
  uint32_t enable_sorting_columns;  /* sorting_columns = primary keys, ascending, nulls first */
  uint32_t _pad;
} hg_write_props;

/* FileMeta (sst.rs:155-160) of the file just written.  num_rows / size are u32 in the reference: larger outputs are refused. */
typedef struct {
  uint64_t size;
  uint32_t num_rows, _pad;
  int64_t time_start, time_end;     /* union of the inputs' ranges (executor.rs:157-163) */
  uint64_t max_sequence;            /* max over the inputs */
} hg_file_meta;

/* Executor::do_compaction end to end on the GPU (compaction/executor.rs:155-222): merge + dedup of the input SSTs (builtin
 * columns kept) AND the Parquet encode of the result, written to `out_path` ("{root}/data/{id}.sst", sst.rs:202-204).
 * The Rust side keeps the manifest update (executor.rs:206-216). */
int hg_compact_to_sst(hg_engine* e, const hg_schema_desc* schema, const hg_sst_desc* ssts, size_t n_ssts, const hg_predicate* shard_preds,
                      size_t n_shard_preds, const hg_write_props* props, const char* out_path, hg_file_meta* out);
/* `shard_preds` (normally none) restricts the compaction to a primary-key range: the multi-GPU split of SURVEY 8(e) — GPU g
 * compacts `pk0 >= splitter[g-1] AND pk0 < splitter[g]` of ALL inputs (only the row groups overlapping its range are read:
 * SSTs are PK-sorted), the outputs concatenated in rank order are the globally sorted, deduplicated run.  A range on pk0
 * never cuts a primary-key run, so LastValue sees every version of a key on one GPU.
 *
 * hg_plan_pk_splitters: host only, deterministic — every rank computes the same `parts - 1` splitters (pk0 values in the
 * column's widened domain: i64 / u64 two's complement) from the row-group statistics of the inputs, balancing rows. */
int hg_plan_pk_splitters(const hg_schema_desc* schema, const hg_sst_desc* ssts, size_t n_ssts, uint32_t parts, uint64_t* splitters);

/* ObjectBasedStorage::write_batch on the GPU (storage.rs:189-225): sort the batch by its primary keys (sort_batch, storage.rs:244-256:
 * ascending; equal keys keep their input order), append __seq__ = `sequence` and an all-null __reserved__ (fill_builtin_columns,
 * types.rs:219-239), encode with the writer above and write `out_path`.  `batch` is an Arrow C struct array holding the USER columns
 * (schema->num_columns - 2 children, primitive types matching schema->types); it stays owned by the caller.
 * NULL primary keys are refused (HG_ERR_UNSUPPORTED), like everywhere else on the GPU path. */
int hg_write_batch(hg_engine* e, const hg_schema_desc* schema, const struct ArrowArray* batch, uint64_t sequence, const hg_write_props* props,
                   const char* out_path, hg_file_meta* out);

int hg_scan_aggregate(hg_engine* e, const hg_schema_desc* schema, const hg_sst_desc* ssts, size_t n_ssts,
                      const hg_predicate* preds, size_t n_preds, const hg_agg_spec* agg,
                      struct ArrowArrayStream* out);

int hg_scan_aggregate_device(hg_engine* e, const hg_schema_desc* schema, const hg_sst_desc* ssts, size_t n_ssts,
                             const hg_predicate* preds, size_t n_preds, const hg_agg_spec* agg,
                             hg_agg_device* out);

/* Packs the last hg_scan_aggregate_device result into a caller-owned device buffer of 6 x cap int64 words
 * (rows: group key, bucket, count, sum bits, min bits, max bits; columns >= num_groups are zero) on the engine's stream:
 * the block one NCCL all-gather combines across GPUs.  HG_ERR_INVALID if cap < num_groups. */
int hg_agg_export_packed(hg_engine* e, void* d_dst, uint64_t cap);

int hg_last_stats(hg_engine* e, hg_scan_stats* out);

/* ---- multi-GPU combine of the per-GPU partial aggregates (SURVEY 8e): one engine per GPU / process, NCCL over NVLink.
 * The aggregation stage and its combine are absent in the reference (metric_engine/src/metric/mod.rs:37-49 is todo!());
 * SSTs shard by file (one partition per SST, read.rs:442-450), so every rank scans its own files and ONE collective
 * combines the partials.  The host ships the NCCL id between ranks over its own channel. */
#define HG_COMM_ID_BYTES 128
typedef enum {
  HG_COMBINE_GATHER = 0,  /* partials are disjoint (keys contain the series id): all-gather of the packed blocks */
  HG_COMBINE_REDUCE = 1   /* keys cross ranks (per-(tag, bucket)): all-gather + per-group combine on every rank: counts summed,
                             min / max taken, f64 sums added in RANK order (deterministic) */
} hg_combine_mode;
typedef struct {
  uint64_t capacity;          /* columns per rank block */
  uint32_t world, _pad;
  const int64_t* d_blocks;    /* device, [world][6][capacity] int64: rows key, bucket, count, sum / min / max bits; count == 0 pads */
  uint64_t num_groups;        /* REDUCE: groups of the combined table */
  uint64_t reduced_capacity;
  const int64_t* d_reduced;   /* REDUCE: device, [6][reduced_capacity], sorted by (key, bucket); identical on every rank */
} hg_agg_combined;
int hg_comm_unique_id(uint8_t* id /* HG_COMM_ID_BYTES */);
int hg_comm_init(hg_engine* e, const uint8_t* id, int rank, int world);
int hg_comm_destroy(hg_engine* e);
/* Collective over all ranks of the communicator: combines the results of their last hg_scan_aggregate_device calls.  The pack
 * kernel runs on the engine stream behind the scan, the collective on the engine's combine stream (the next scan overlaps it);
 * GATHER results are valid after hg_comm_sync.  capacity_hint = 0: the ranks first agree on the block width (one extra small
 * collective + host sync); > 0: every rank passes the same value and promises num_groups <= capacity_hint. */
int hg_agg_combine(hg_engine* e, uint32_t mode, uint64_t capacity_hint, hg_agg_combined* out);
int hg_comm_sync(hg_engine* e);

/* ---- host-only inspection of an SST (no engine, no GPU): what the planner reads from the footer and the page headers.
 * In the reference this is parquet-rs's metadata reader behind ParquetExec (read.rs:66-93, 442-465); the CPU test-suite
 * checks it against pyarrow's reading of the same bytes. */
typedef struct {
  uint64_t num_rows;
  uint32_t num_row_groups, num_columns;
  uint64_t num_data_pages;
  uint64_t sum_page_values;          /* sum of num_values over all data pages */
  uint64_t sum_uncompressed_bytes;   /* sum of uncompressed page payload sizes (page headers excluded) */
  uint64_t sum_compressed_bytes;     /* the same, as stored */
  uint32_t codec_mask;               /* bit c set: some column chunk uses Parquet codec id c (0 uncompressed, 1 Snappy, 6 Zstd) */
  uint32_t max_pages_per_chunk;
} hg_parquet_summary;

typedef struct {
  uint64_t num_rows;                 /* rows of the row group */
  uint64_t num_values;               /* values of the column chunk (nulls included) */
  int64_t data_page_offset, total_compressed_size;
  int64_t null_count;                /* -1: not recorded */
  uint8_t min[8], max[8];            /* PLAIN-encoded statistics (little endian), valid if has_min_max */
  uint32_t has_min_max, physical_type, codec, num_pages;
  uint64_t first_page_payload_offset;
  uint32_t first_page_num_values, first_page_type;   /* 0 = DataPage V1, 3 = DataPage V2 */
} hg_parquet_chunk;

/* The planner's statistics pruning for ONE SST, host only: keep[g] = 1 iff row group g can hold a row matching the
 * conjunction (DataFusion's PruningPredicate as pinned by the plan text at read.rs:613: CASE WHEN null_count = row_count
 * THEN false ELSE <min/max rewrite> END).  Also runs the schema / predicate / file validation every scan call runs.
 * HG_ERR_INVALID if cap < number of row groups. */
int hg_plan_row_groups(const hg_schema_desc* schema, const uint8_t* data, uint64_t size, const hg_predicate* preds, size_t n_preds,
                       uint8_t* keep, uint32_t cap, uint32_t* num_row_groups);

int hg_parquet_inspect(const uint8_t* data, uint64_t size, hg_parquet_summary* out);
int hg_parquet_chunk_info(const uint8_t* data, uint64_t size, uint32_t row_group, uint32_t column, hg_parquet_chunk* out);

#ifdef __cplusplus
}
#endif
#endif /* HORAE_GPU_H */
