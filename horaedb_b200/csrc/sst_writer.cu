// sst_writer.cu — GPU Parquet page encoder + SST assembly: the second half of Executor::do_compaction
// (compaction/executor.rs:173-203: AsyncArrowWriter over the merged stream) and of write_batch (storage.rs:189-225), with
// the writer properties of build_write_props (storage.rs:258-298) and WriteConfig::default (config.rs:120-133):
// row groups of max_row_group_size rows, one DataPage V1 per column chunk, PLAIN values, RLE/bit-packed definition levels
// (every field is nullable), dictionary off, bloom filters off, chunk statistics (min / max / null_count), Snappy,
// Zstandard or uncompressed pages, sorting_columns = primary keys ascending nulls first, Thrift-compact footer.
//
// Device work: page bodies (level prefix + compacted non-null values), chunk statistics, page compression and the final
// gather into one contiguous file image.  Host work: the few KB of Thrift (page headers, footer) and the offsets.
//
// The Snappy compressor is written for what these pages hold — fixed-width numbers: value i is compared with value i-1
// (8-byte columns: how many HIGH bytes agree; 4-byte columns: equal or not) and the page becomes literal runs, 2-byte
// copies of the agreeing high bytes (offset = value width) and 64-byte run-length copies.  Every value computes its own
// emitted size, one prefix sum gives all positions, every value writes its own bytes: no serial parse, any Snappy decoder
// reads the result.  (On the synthetic metric data it lands within a few percent of the reference compressor's ratio.)
//
// The Zstandard compressor (RFC 8878) sees the same values, with one more match source: a per-block hash table finds an
// earlier equal value further back (in a timestamp column: the same timestamp one series earlier), and consecutive values
// that match at the same distance become one long match.  Every sequence uses an explicit offset (never a repeat code), so
// the 128 KB blocks of a page are independent and compress in parallel, one CTA each.  Literals are stored raw; literal
// lengths, match lengths and offsets are entropy coded (RLE / predefined / FSE tables chosen per block by estimated size).
// The code tables are the decoder's (zstd_core.h).  A block that would not shrink is stored as a Raw block.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>
#include <string>
#include <vector>

#include "engine_internal.h"
#include "sst_writer.h"

// zstd_core.h's primitives (the decoder itself is not used here: only its code tables and predefined distributions)
#define SNP_FN __device__ __forceinline__
#define SNP_CONST __constant__ const
#define snp_any(p) __any_sync(0xffffffffu, (p))
#define snp_syncwarp() __syncwarp()
#define snp_ldg8(p) __ldg(p)
#define snp_ldcg8(p) (*(p))
#define snp_set_err(err, code) atomicExch((err), (code))
namespace horae {
namespace zst {
__device__ __forceinline__ uint64_t snp_ldg64u(const uint8_t* p) {
  uint64_t v = 0;
  for (int i = 0; i < 8; i++) v |= uint64_t(__ldg(p + i)) << (8 * i);
  return v;
}
}  // namespace zst
}  // namespace horae
#include "zstd_core.h"

namespace horae {
namespace writer {

namespace {

constexpr int kThreads = 256;

struct PageMetaDev {
  uint32_t uncomp_size, comp_size, null_count, has_minmax;
  uint64_t mn, mx;             // PLAIN bytes of min / max (little endian, low `width` bytes)
};

struct PageJob {
  const void* vals;            // dense column
  const uint8_t* valid;        // one byte per row or nullptr
  uint32_t type, width;        // hg_type, value width in the column array
  uint32_t pwidth;             // physical width in the page (4 or 8)
};

__device__ __forceinline__ uint32_t varint_put(uint8_t* p, uint32_t v) {
  uint32_t n = 0;
  while (v >= 0x80) { p[n++] = uint8_t(v | 0x80); v >>= 7; }
  p[n++] = uint8_t(v);
  return n;
}

// block-wide exclusive scan of one value per thread (256 threads); *total = block sum
__device__ __forceinline__ uint32_t block_scan(uint32_t v, uint32_t* total, uint32_t* s_w /*[9]*/) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  uint32_t inc = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t; }
  if (lane == 31) s_w[w] = inc;
  __syncthreads();
  if (threadIdx.x == 0) { uint32_t run = 0; for (int x = 0; x < kThreads / 32; x++) { uint32_t c = s_w[x]; s_w[x] = run; run += c; } s_w[8] = run; }
  __syncthreads();
  const uint32_t r = s_w[w] + inc - v;
  *total = s_w[8];
  __syncthreads();
  return r;
}

__device__ __forceinline__ uint64_t load_phys(const PageJob& j, uint32_t row) {
  // the value as PLAIN physical bytes: 1/2-byte integers widen to INT32 (sign- or zero-extended by their type)
  switch (j.type) {
    case T_U8: return reinterpret_cast<const uint8_t*>(j.vals)[row];
    case T_I8: return uint32_t(int32_t(reinterpret_cast<const int8_t*>(j.vals)[row]));
    case T_U16: return reinterpret_cast<const uint16_t*>(j.vals)[row];
    case T_I16: return uint32_t(int32_t(reinterpret_cast<const int16_t*>(j.vals)[row]));
    case T_U32: case T_I32: case T_F32: return reinterpret_cast<const uint32_t*>(j.vals)[row];
    default: return reinterpret_cast<const uint64_t*>(j.vals)[row];
  }
}

// order key of a physical value for the chunk statistics (unsigned compare of the key == typed compare of the value)
__device__ __forceinline__ uint64_t stat_key(uint64_t phys, uint32_t type, bool* is_nan) {
  *is_nan = false;
  switch (type) {
    case T_I8: case T_I16: case T_I32: return uint64_t(int64_t(int32_t(uint32_t(phys)))) ^ (1ull << 63);
    case T_I64: return phys ^ (1ull << 63);
    case T_F32: {
      const float f = __uint_as_float(uint32_t(phys));
      *is_nan = f != f;
      const uint32_t b = uint32_t(phys);
      return uint64_t(b ^ ((b >> 31) ? 0xffffffffu : 0x80000000u));
    }
    case T_F64: {
      const double d = __longlong_as_double((long long)phys);
      *is_nan = d != d;
      return phys ^ ((phys >> 63) ? ~0ull : (1ull << 63));
    }
    default: return phys;
  }
}
__device__ __forceinline__ uint64_t stat_unkey(uint64_t key, uint32_t type) {
  switch (type) {
    case T_I8: case T_I16: case T_I32: return uint64_t(uint32_t(key ^ (1ull << 63)));
    case T_I64: return key ^ (1ull << 63);
    case T_F32: { const uint32_t k = uint32_t(key); return uint64_t(k ^ ((k >> 31) ? 0x80000000u : 0xffffffffu)); }
    case T_F64: return key ^ ((key >> 63) ? (1ull << 63) : ~0ull);
    default: return key;
  }
}

// One block per page (row group g, column c): [u32 level bytes][definition levels][PLAIN values of the non-null rows]
__global__ void __launch_bounds__(kThreads) page_body_kernel(const PageJob* __restrict__ jobs, uint32_t ncols, uint32_t R, uint32_t rg_rows,
                                                            uint8_t* __restrict__ body, uint64_t bstride, PageMetaDev* __restrict__ meta) {
  __shared__ uint32_t s_w[9];
  __shared__ uint32_t s_nulls, s_prefix;
  __shared__ unsigned long long s_mn, s_mx;
  __shared__ uint32_t s_seen;
  const uint32_t page = blockIdx.x, g = page / ncols, c = page % ncols;
  const PageJob j = jobs[c];
  const uint32_t row0 = g * rg_rows, rows = (R - row0) < rg_rows ? (R - row0) : rg_rows;
  uint8_t* out = body + uint64_t(page) * bstride;
  const int tid = threadIdx.x;
  if (tid == 0) { s_nulls = 0; s_mn = ~0ull; s_mx = 0; s_seen = 0; }
  __syncthreads();
  // ---- null count
  uint32_t nulls = 0;
  if (j.valid) for (uint32_t i = tid; i < rows; i += kThreads) nulls += j.valid[row0 + i] == 0;
  for (int d = 16; d > 0; d >>= 1) nulls += __shfl_down_sync(0xffffffffu, nulls, d);
  if ((tid & 31) == 0 && nulls) atomicAdd(&s_nulls, nulls);
  __syncthreads();
  const uint32_t nnull = s_nulls;
  // ---- definition levels (bit width 1): one RLE run when uniform, else one bit-packed run of ceil(rows/8) groups
  if (tid == 0) {
    uint32_t n = 0;
    uint8_t* lv = out + 4;
    if (nnull == 0 || nnull == rows) { n = varint_put(lv, rows << 1); lv[n++] = nnull == 0 ? 1 : 0; }
    else { const uint32_t groups = (rows + 7) / 8; n = varint_put(lv, (groups << 1) | 1u); n += groups; }
    out[0] = uint8_t(n); out[1] = uint8_t(n >> 8); out[2] = uint8_t(n >> 16); out[3] = uint8_t(n >> 24);
    s_prefix = 4 + n;
  }
  __syncthreads();
  const uint32_t prefix = s_prefix;
  if (nnull != 0 && nnull != rows) {
    const uint32_t groups = (rows + 7) / 8;
    uint8_t* bits = out + prefix - groups;
    for (uint32_t b = tid; b < groups; b += kThreads) {
      uint32_t v = 0;
#pragma unroll
      for (int k2 = 0; k2 < 8; k2++) { const uint32_t i = b * 8 + k2; if (i < rows && j.valid[row0 + i]) v |= 1u << k2; }
      bits[b] = uint8_t(v);
    }
  }
  // ---- values of the non-null rows, compacted in order; statistics
  uint8_t* vout = out + prefix;
  uint32_t running = 0;
  unsigned long long mn = ~0ull, mx = 0;
  bool seen = false;
  for (uint32_t base = 0; base < rows; base += kThreads) {
    const uint32_t i = base + tid;
    const uint32_t v = (i < rows && (!j.valid || j.valid[row0 + i])) ? 1u : 0u;
    uint32_t total;
    const uint32_t k2 = running + block_scan(v, &total, s_w);
    if (v) {
      const uint64_t x = load_phys(j, row0 + i);
      // (the page body starts 64-byte aligned; the level prefix is usually 8 bytes, so the values are naturally aligned)
      if (j.pwidth == 8) {
        uint8_t* q = vout + size_t(k2) * 8;
        if ((prefix & 7) == 0) *reinterpret_cast<uint64_t*>(q) = x;
        else for (int b = 0; b < 8; b++) q[b] = uint8_t(x >> (8 * b));
      } else {
        uint8_t* q = vout + size_t(k2) * 4;
        if ((prefix & 3) == 0) *reinterpret_cast<uint32_t*>(q) = uint32_t(x);
        else for (int b = 0; b < 4; b++) q[b] = uint8_t(x >> (8 * b));
      }
      bool nan;
      const uint64_t key = stat_key(x, j.type, &nan);
      if (!nan) { mn = key < mn ? key : mn; mx = key > mx ? key : mx; seen = true; }
    }
    running += total;
  }
  if (seen) { atomicMin(&s_mn, mn); atomicMax(&s_mx, mx); atomicOr(&s_seen, 1u); }
  __syncthreads();
  if (tid == 0) {
    PageMetaDev m;
    m.uncomp_size = prefix + (rows - nnull) * j.pwidth;
    m.comp_size = m.uncomp_size;
    m.null_count = nnull;
    m.has_minmax = s_seen;
    m.mn = s_seen ? stat_unkey(s_mn, j.type) : 0;
    m.mx = s_seen ? stat_unkey(s_mx, j.type) : 0;
    meta[page] = m;
  }
}

// ------------------------------------------------------------------------------------------------ Snappy compression
__device__ __forceinline__ uint32_t lit_header_len(uint32_t len) { return len <= 60 ? 1u : (len <= 0x100 ? 2u : (len <= 0x10000 ? 3u : (len <= 0x1000000 ? 4u : 5u))); }
__device__ __forceinline__ uint32_t lit_header_put(uint8_t* p, uint32_t len) {
  const uint32_t n = len - 1;
  if (len <= 60) { p[0] = uint8_t(n << 2); return 1; }
  const uint32_t nb = lit_header_len(len) - 1;
  p[0] = uint8_t((59 + nb) << 2);
  for (uint32_t i = 0; i < nb; i++) p[1 + i] = uint8_t(n >> (8 * i));
  return 1 + nb;
}
// copy of len (4..64) bytes at offset off (< 2048): 2-byte form when len <= 11, else the 3-byte form
__device__ __forceinline__ uint32_t copy_len(uint32_t len) { return len <= 11 ? 2u : 3u; }
__device__ __forceinline__ uint32_t copy_put(uint8_t* p, uint32_t len, uint32_t off) {
  if (len <= 11) { p[0] = uint8_t(1 | ((len - 4) << 2) | ((off >> 8) << 5)); p[1] = uint8_t(off); return 2; }
  p[0] = uint8_t(2 | ((len - 1) << 2)); p[1] = uint8_t(off); p[2] = uint8_t(off >> 8);
  return 3;
}

// class of value i relative to value i-1:  0 = no usable match (literal bytes), 1..4 = k low bytes differ, the 8-k high bytes
// are copied (8-byte values only), 9 = equal (run-length copy)
constexpr uint8_t kClsN = 0, kClsF = 9;

// One block per page.  scratch: per page `sstride` bytes = cls[nv] (u8) + run id / offsets (u32 x 2 per value).
__global__ void __launch_bounds__(kThreads) snappy_encode_kernel(const uint8_t* __restrict__ body, uint64_t bstride, PageMetaDev* __restrict__ meta,
                                                                const PageJob* __restrict__ jobs, uint32_t ncols, uint8_t* __restrict__ comp, uint64_t cstride,
                                                                uint8_t* __restrict__ scratch, uint64_t sstride, uint32_t max_vals) {
  __shared__ uint32_t s_w[9];
  __shared__ uint32_t s_total;
  const uint32_t page = blockIdx.x;
  const PageJob j = jobs[page % ncols];
  const uint32_t w = j.pwidth;
  const uint8_t* in = body + uint64_t(page) * bstride;
  uint8_t* out = comp + uint64_t(page) * cstride;
  const uint32_t ulen = meta[page].uncomp_size;
  const uint32_t prefix = 4 + (uint32_t(in[0]) | (uint32_t(in[1]) << 8) | (uint32_t(in[2]) << 16) | (uint32_t(in[3]) << 24));
  const uint32_t nv = (ulen - prefix) / w;
  uint8_t* cls = scratch + uint64_t(page) * sstride;
  uint32_t* run_of = reinterpret_cast<uint32_t*>(cls + ((max_vals + 15u) & ~15u));   // run index of value i
  uint32_t* run_pos = run_of + max_vals;                                            // first value of run r, then: output offset of run r
  uint32_t* run_out = run_pos + max_vals + 1;
  const int tid = threadIdx.x;
  const uint8_t* v = in + prefix;
  const bool val_aligned = (prefix & (w - 1)) == 0;
  auto val_at = [&](uint32_t i) -> uint64_t {
    if (val_aligned) return w == 8 ? *reinterpret_cast<const uint64_t*>(v + size_t(i) * 8) : uint64_t(*reinterpret_cast<const uint32_t*>(v + size_t(i) * 4));
    uint64_t x = 0;
    for (uint32_t b = 0; b < w; b++) x |= uint64_t(v[size_t(i) * w + b]) << (8 * b);
    return x;
  };
  // ---- classes
  for (uint32_t i = tid; i < nv; i += kThreads) {
    uint8_t c = kClsN;
    if (i > 0) {
      const uint64_t x = val_at(i) ^ val_at(i - 1);
      if (x == 0) c = kClsF;
      else if (w == 8) { const uint32_t k = (71u - uint32_t(__clzll((long long)x))) / 8u; if (k <= 4) c = uint8_t(k); }   // k = differing low bytes
    }
    cls[i] = c;
  }
  __syncthreads();
  // ---- runs: a new run starts where the class changes; partial-match values are runs of their own
  uint32_t running = 0;
  for (uint32_t base = 0; base < nv; base += kThreads) {
    const uint32_t i = base + tid;
    uint32_t st = 0;
    if (i < nv) { const uint8_t c = cls[i]; st = (i == 0 || c != cls[i - 1] || (c >= 1 && c <= 4)) ? 1u : 0u; }
    uint32_t total;
    const uint32_t r = running + block_scan(st, &total, s_w) + st - 1;      // inclusive - 1 = run index
    if (i < nv) { run_of[i] = r; if (st) run_pos[r] = i; }
    running += total;
  }
  const uint32_t nruns = running;
  if (tid == 0) run_pos[nruns] = nv;
  __syncthreads();
  // ---- emitted size of every run; the level prefix joins the first literal run
  uint32_t pre = 0;
  { uint32_t u = ulen; while (u >= 0x80) { pre++; u >>= 7; } pre++; }       // varint(uncompressed length)
  running = 0;
  for (uint32_t base = 0; base < nruns + (nv == 0 ? 1u : 0u); base += kThreads) {
    const uint32_t r = base + tid;
    uint32_t sz = 0;
    if (nv == 0) { if (r == 0) sz = lit_header_len(prefix) + prefix; }
    else if (r < nruns) {
      const uint32_t a = run_pos[r], b = run_pos[r + 1], c = cls[a];
      if (c == kClsN) { const uint32_t len = (b - a) * w + (r == 0 ? prefix : 0); sz = lit_header_len(len) + len; }
      else if (c == kClsF) { const uint32_t bytes = (b - a) * w, full = bytes / 64, rem = bytes % 64; sz = full * 3 + (rem ? copy_len(rem) : 0); }
      else sz = 1 + c + 2;                                                   // literal(c) + copy(8 - c, offset 8)
    }
    uint32_t total;
    const uint32_t o = running + block_scan(sz, &total, s_w);
    if (r < nruns) run_out[r] = o;
    running += total;
  }
  if (tid == 0) s_total = running;
  __syncthreads();
  uint8_t* body_out = out + pre;
  if (tid == 0) {
    varint_put(out, ulen);
    meta[page].comp_size = pre + s_total;
    if (nv == 0) { const uint32_t h = lit_header_put(body_out, prefix); for (uint32_t i = 0; i < prefix; i++) body_out[h + i] = in[i]; }
  }
  if (nv == 0) return;
  // ---- emission: every value writes its own share
  {
    // the first run is a literal run (value 0 has no predecessor): header + level prefix
    const uint32_t len0 = (run_pos[1] - run_pos[0]) * w + prefix;
    const uint32_t h0 = lit_header_len(len0);
    if (tid == 0) lit_header_put(body_out, len0);
    for (uint32_t i = tid; i < prefix; i += kThreads) body_out[h0 + i] = in[i];
  }
  for (uint32_t i = tid; i < nv; i += kThreads) {
    const uint32_t r = run_of[i], a = run_pos[r], b = run_pos[r + 1];
    const uint8_t c = cls[i];
    uint8_t* o = body_out + run_out[r];
    if (c == kClsN) {
      const uint32_t len = (b - a) * w + (r == 0 ? prefix : 0);
      const uint32_t h = lit_header_len(len);
      if (i == a && r != 0) lit_header_put(o, len);
      uint8_t* q = o + h + (r == 0 ? prefix : 0) + (i - a) * w;
      for (uint32_t bb = 0; bb < w; bb++) q[bb] = v[size_t(i) * w + bb];
    } else if (c == kClsF) {
      const uint32_t per = 64 / w, qn = i - a;
      if (qn % per == 0) {
        const uint32_t left = (b - i) * w;
        copy_put(o + (qn / per) * 3, left < 64 ? left : 64, w);
      }
    } else {
      o[0] = uint8_t((uint32_t(c) - 1) << 2);
      for (uint32_t bb = 0; bb < c; bb++) o[1 + bb] = v[size_t(i) * w + bb];
      copy_put(o + 1 + c, 8 - c, 8);
    }
  }
}

// ------------------------------------------------------------------------------------------------ Zstandard compression
constexpr uint32_t kZBlk = zst::kBlockMax;      // bytes of page content per block
constexpr int kZHashLog = 13;                   // per-block table of earlier values: 8192 slots, the most recent index wins
constexpr uint32_t kZFront = 16;                // room in front of block 0 for the frame header
constexpr uint32_t kZPad = 512;                 // slot bytes beyond the block content: block / literal / sequence headers, tables
constexpr uint32_t kZArrays = 10;               // u32 scratch arrays per CTA, one entry per value of the block (+1)

// frame header: magic, descriptor (Single_Segment, no checksum, no dictionary), content size in 1 / 2 (+256) / 4 bytes
__host__ __device__ __forceinline__ uint32_t zframe_header_len(uint32_t ulen) { return 5u + (ulen < 256 ? 1u : (ulen < 65536 + 256 ? 2u : 4u)); }
__host__ __device__ __forceinline__ uint32_t zblocks_of(uint32_t ulen) { return (ulen + kZBlk - 1) / kZBlk; }

__device__ __forceinline__ int hbit(uint32_t v) { return 31 - __clz(int(v)); }      // v > 0
__device__ __forceinline__ uint32_t zcode_ll(uint32_t v) {
  if (v < 16) return v;
  uint32_t lo = 16, hi = zst::kMaxLL - 1;
  while (lo < hi) { const uint32_t m = (lo + hi + 1) >> 1; if (zst::ll_base(m) <= v) lo = m; else hi = m - 1; }
  return lo;
}
__device__ __forceinline__ uint32_t zcode_ml(uint32_t v) {      // v >= 3
  if (v < 35) return v - 3;
  uint32_t lo = 32, hi = zst::kMaxML - 1;
  while (lo < hi) { const uint32_t m = (lo + hi + 1) >> 1; if (zst::ml_base(m) <= v) lo = m; else hi = m - 1; }
  return lo;
}

// FSE encoding table (the inverse of zstd_core.h's fse_build): state table + per-symbol transforms
struct ZFseCT {
  uint16_t state[1 << zst::kLLLog];
  int32_t dnb[64], dfs[64];                     // deltaNbBits, deltaFindState
  uint32_t log;
};
struct ZSmem {
  uint32_t hash[1 << kZHashLog];
  ZFseCT ct[3];                                 // literal lengths, offsets, match lengths (the order of the sequence section)
  uint32_t hist[3][64];
  int16_t norm[3][64];
  uint8_t cell_sym[1 << zst::kLLLog];
  uint32_t w[9];                                // block_scan
  uint32_t raw;                                 // the block is stored uncompressed
};

// normalised counts of `total` events: every used symbol >= 1, the sum is 2^L (L >= highbit(symbols used) + 1)
__device__ void zfse_normalize(const uint32_t* cnt, int nsym, uint32_t total, int L, int16_t* norm) {
  const uint32_t size = 1u << L;
  uint32_t sum = 0;
  int big = 0;
  for (int s = 0; s < nsym; s++) {
    uint32_t n = cnt[s] ? uint32_t((uint64_t(cnt[s]) << L) / total) : 0u;
    if (cnt[s] && n == 0) n = 1;
    norm[s] = int16_t(n);
    sum += n;
    if (cnt[s] > cnt[big]) big = s;
  }
  if (sum <= size) { norm[big] = int16_t(norm[big] + int(size - sum)); return; }
  for (uint32_t excess = sum - size; excess; excess--) {       // the rounded-up rare symbols took too many cells: the largest give back
    int m = 0;
    for (int s = 1; s < nsym; s++) if (norm[s] > norm[m]) m = s;
    norm[m]--;
  }
}
// table description (RFC 8878 4.1.1) of norm[0 .. nsym), nsym - 1 = the last used symbol; returns the bytes written
__device__ uint32_t zfse_write_ncount(uint8_t* out, const int16_t* norm, int nsym, int L) {
  uint64_t acc = 0;
  int nb = 0;
  uint32_t n = 0;
  auto put = [&](uint32_t v, int bits) { acc |= uint64_t(v) << nb; nb += bits; while (nb >= 8) { out[n++] = uint8_t(acc); acc >>= 8; nb -= 8; } };
  put(uint32_t(L - 5), 4);
  int remaining = 1 << L, s = 0;
  while (remaining > 0 && s < nsym) {
    const int p = norm[s++];
    const uint32_t mx = uint32_t(remaining + 1), v = uint32_t(p + 1);
    const int bits = hbit(mx) + 1;
    const uint32_t lower = (1u << (bits - 1)) - 1u, thr = (1u << bits) - 1u - mx;
    if (v < thr) put(v, bits - 1);
    else if (v <= lower) put(v, bits);
    else put(v + thr, bits);
    remaining -= p;
    if (p == 0) {
      int z = 0;
      while (s + z < nsym && norm[s + z] == 0) z++;
      s += z;
      for (; z >= 3; z -= 3) put(3, 2);
      put(uint32_t(z), 2);
    }
  }
  if (nb) out[n++] = uint8_t(acc);
  return n;
}
// encoding table of norm[0 .. nsym) at accuracy L (norm -1 = "less than one" cell, as in the predefined distributions)
__device__ void zfse_build_ct(ZFseCT& ct, const int16_t* norm, int nsym, int L, uint8_t* cell_sym) {
  const uint32_t size = 1u << L, mask = size - 1, step = (size >> 1) + (size >> 3) + 3;
  uint32_t high = size - 1, cumul[65];
  cumul[0] = 0;
  for (int s = 0; s < nsym; s++) {
    if (norm[s] == -1) { cumul[s + 1] = cumul[s] + 1; cell_sym[high--] = uint8_t(s); }
    else cumul[s + 1] = cumul[s] + uint32_t(norm[s]);
  }
  uint32_t pos = 0;
  for (int s = 0; s < nsym; s++)
    for (int i = 0; i < norm[s]; i++) { cell_sym[pos] = uint8_t(s); do { pos = (pos + step) & mask; } while (pos > high); }
  for (uint32_t u = 0; u < size; u++) ct.state[cumul[cell_sym[u]]++] = uint16_t(size + u);
  int total = 0;
  for (int s = 0; s < nsym; s++) {
    const int c = norm[s];
    if (c == 0) { ct.dnb[s] = int32_t(((uint32_t(L) + 1) << 16) - size); ct.dfs[s] = 0; }
    else if (c == -1 || c == 1) { ct.dnb[s] = int32_t((uint32_t(L) << 16) - size); ct.dfs[s] = total - 1; total++; }
    else {
      const uint32_t mbo = uint32_t(L - hbit(uint32_t(c - 1)));
      ct.dnb[s] = int32_t((mbo << 16) - (uint32_t(c) << mbo));
      ct.dfs[s] = total - c;
      total += c;
    }
  }
  ct.log = uint32_t(L);
}

// forward bit writer of the sequence bitstream (read backwards by the decoder); `over` once it would pass `cap`
struct ZBitW {
  uint8_t* p; uint32_t n, cap; uint64_t acc; int nb; bool over;
  __device__ void add(uint32_t v, int bits) {
    acc |= (uint64_t(v) & ((1ull << bits) - 1ull)) << nb;
    nb += bits;
    while (nb >= 8) { if (n < cap) p[n] = uint8_t(acc); else over = true; n++; acc >>= 8; nb -= 8; }
  }
};
__device__ __forceinline__ uint32_t zfse_init(const ZFseCT& ct, uint32_t sym) {
  const uint32_t nbo = uint32_t(ct.dnb[sym] + (1 << 15)) >> 16;
  const uint32_t v = (nbo << 16) - uint32_t(ct.dnb[sym]);
  return ct.state[(v >> nbo) + ct.dfs[sym]];
}
__device__ __forceinline__ void zfse_encode(ZBitW& bw, const ZFseCT& ct, uint32_t& st, uint32_t sym) {
  const uint32_t nbo = (st + uint32_t(ct.dnb[sym])) >> 16;
  bw.add(st, int(nbo));
  st = ct.state[(st >> nbo) + ct.dfs[sym]];
}

// One CTA per (page, 128 KB block).  The block's values (those wholly inside it) are classed like the Snappy path's, plus
// F(d) = equal to the value d positions back (hash table); runs of equal class become sequences; the level prefix and partial
// values at the block's edges are literals.  Output: [frame header (block 0)][block header][literals][sequences] in the
// block's slot of `comp`; zsz[page * nbmax + b] = its bytes (0: no such block).
__global__ void __launch_bounds__(kThreads) zstd_encode_kernel(const uint8_t* __restrict__ body, uint64_t bstride, const PageMetaDev* __restrict__ meta,
                                                              const PageJob* __restrict__ jobs, uint32_t ncols, uint32_t nbmax, uint8_t* __restrict__ comp,
                                                              uint64_t cstride, uint64_t zslot, uint32_t* __restrict__ zsz, uint8_t* __restrict__ scratch,
                                                              uint64_t sstride, uint32_t vcap) {
  __shared__ ZSmem sm;
  const uint32_t page = blockIdx.x / nbmax, b = blockIdx.x % nbmax;
  const uint32_t w = jobs[page % ncols].pwidth;
  const uint8_t* in = body + uint64_t(page) * bstride;
  const uint32_t ulen = meta[page].uncomp_size;
  const int tid = threadIdx.x;
  if (b >= zblocks_of(ulen)) { if (tid == 0) zsz[blockIdx.x] = 0; return; }
  uint8_t* const slot = comp + uint64_t(page) * cstride + uint64_t(b) * zslot;
  uint8_t* const out = slot + kZFront;                        // block header
  const uint32_t prefix = 4 + (uint32_t(in[0]) | (uint32_t(in[1]) << 8) | (uint32_t(in[2]) << 16) | (uint32_t(in[3]) << 24));
  const uint32_t nv = (ulen - prefix) / w;
  const uint32_t bstart = b * kZBlk, bend = min(bstart + kZBlk, ulen), content = bend - bstart;
  const bool last = bend == ulen;
  // values wholly inside the block: [fi, li); head = literal bytes in front of them, tail = behind them
  const uint32_t fi = bstart <= prefix ? 0u : min(nv, (bstart - prefix + w - 1) / w);
  uint32_t li = bend <= prefix ? 0u : min(nv, (bend - prefix) / w);
  if (li < fi) li = fi;
  const uint32_t nvb = li - fi;
  const uint32_t head = nvb ? prefix + fi * w - bstart : content, tail = nvb ? bend - (prefix + li * w) : 0u;
  const uint8_t* v = in + prefix;
  const bool val_aligned = (prefix & (w - 1)) == 0;
  auto val_at = [&](uint32_t i) -> uint64_t {
    if (val_aligned) return w == 8 ? *reinterpret_cast<const uint64_t*>(v + size_t(i) * 8) : uint64_t(*reinterpret_cast<const uint32_t*>(v + size_t(i) * 4));
    uint64_t x = 0;
    for (uint32_t k = 0; k < w; k++) x |= uint64_t(v[size_t(i) * w + k]) << (8 * k);
    return x;
  };
  uint32_t* const cd = reinterpret_cast<uint32_t*>(scratch + uint64_t(blockIdx.x) * sstride);   // candidate distance, then run of value
  uint32_t* const key = cd + vcap;                            // 0 literal, 1..5 P(k): k low bytes + match of 8-k at offset 8, d << 3: F(d)
  uint32_t* const run_pos = key + vcap;                       // [vcap + 1]
  uint32_t* const run_lit = run_pos + vcap + 1;               // literal bytes in front of run r (value literals only)
  uint32_t* const seq_end = run_lit + vcap;                   // literal bytes up to the match of sequence j (head included)
  uint32_t* const seq_run = seq_end + vcap;
  uint32_t* const seq_ll = seq_run + vcap;
  uint32_t* const seq_ml = seq_ll + vcap;
  uint32_t* const seq_of = seq_ml + vcap;                     // offset + 3
  uint32_t* const seq_code = seq_of + vcap;                   // LL code | ML code << 8 | OF code << 16
  for (uint32_t i = tid; i < (1u << kZHashLog); i += kThreads) sm.hash[i] = 0;
  for (uint32_t i = tid; i < 3 * 64; i += kThreads) sm.hist[i / 64][i % 64] = 0;
  __syncthreads();
  // ---- earlier equal values: chunks of 256 look up what the chunks before them inserted (the largest index per slot)
  for (uint32_t base = 0; base < nvb; base += kThreads) {
    const uint32_t q = base + tid;
    uint32_t h = 0;
    uint64_t x = 0;
    if (q < nvb) {
      x = val_at(fi + q);
      h = uint32_t((x * 0x9E3779B97F4A7C15ull) >> (64 - kZHashLog));
      const uint32_t c = sm.hash[h];
      cd[q] = (c && val_at(fi + c - 1) == x) ? q - (c - 1) : 0u;
    }
    __syncthreads();
    if (q < nvb) atomicMax(&sm.hash[h], q + 1);
    __syncthreads();
  }
  // ---- classes
  for (uint32_t q = tid; q < nvb; q += kThreads) {
    uint32_t k2 = 0;
    if (q > 0) {
      const uint64_t x = val_at(fi + q) ^ val_at(fi + q - 1);
      if (x == 0) k2 = 1u << 3;
      else {
        const uint32_t k = (71u - uint32_t(__clzll((long long)x))) / 8u;
        const bool p_ok = w == 8 && k <= 5;
        const uint32_t d = cd[q];
        // a lone far match is a whole sequence with a long offset: a close partial match is cheaper
        if (d && !(p_ok && k <= 2 && cd[q - 1] != d && (q + 1 >= nvb || cd[q + 1] != d))) k2 = d << 3;
        else if (p_ok) k2 = k;
      }
    }
    key[q] = k2;
  }
  __syncthreads();
  // ---- runs: a new run starts where the class changes; P values are runs of their own
  uint32_t running = 0;
  for (uint32_t base = 0; base < nvb; base += kThreads) {
    const uint32_t q = base + tid;
    uint32_t st = 0;
    if (q < nvb) { const uint32_t c = key[q]; st = (q == 0 || c != key[q - 1] || (c >= 1 && c < 8)) ? 1u : 0u; }
    uint32_t total;
    const uint32_t r = running + block_scan(st, &total, sm.w) + st - 1;
    if (q < nvb) { cd[q] = r; if (st) run_pos[r] = q; }
    running += total;
  }
  const uint32_t nruns = running;
  if (tid == 0) run_pos[nruns] = nvb;
  __syncthreads();
  // ---- literal bytes and sequences per run
  uint32_t lrun = 0, srun = 0;
  for (uint32_t base = 0; base < nruns; base += kThreads) {
    const uint32_t r = base + tid;
    uint32_t lit = 0, isseq = 0;
    if (r < nruns) {
      const uint32_t a = run_pos[r], c = key[a];
      lit = c == 0 ? (run_pos[r + 1] - a) * w : (c < 8 ? c : 0u);
      isseq = c != 0;
    }
    uint32_t lt, stot;
    const uint32_t lo = lrun + block_scan(lit, &lt, sm.w);
    const uint32_t so = srun + block_scan(isseq, &stot, sm.w);
    if (r < nruns) {
      run_lit[r] = lo;
      if (isseq) { seq_end[so] = head + lo + lit; seq_run[so] = r; }
    }
    lrun += lt;
    srun += stot;
  }
  const uint32_t nseq = srun, ltot = head + lrun + tail;
  __syncthreads();
  // ---- sequence values and codes
  for (uint32_t j = tid; j < nseq; j += kThreads) {
    const uint32_t r = seq_run[j], a = run_pos[r], c = key[a];
    const uint32_t ll = seq_end[j] - (j ? seq_end[j - 1] : 0u);
    const uint32_t ml = c < 8 ? 8 - c : (run_pos[r + 1] - a) * w;
    const uint32_t ofb = (c < 8 ? 8u : (c >> 3) * w) + 3u;
    const uint32_t llc = zcode_ll(ll), mlc = zcode_ml(ml), ofc = uint32_t(hbit(ofb));
    seq_ll[j] = ll; seq_ml[j] = ml; seq_of[j] = ofb;
    seq_code[j] = llc | (mlc << 8) | (ofc << 16);
    atomicAdd(&sm.hist[0][llc], 1u);
    atomicAdd(&sm.hist[1][ofc], 1u);
    atomicAdd(&sm.hist[2][mlc], 1u);
  }
  // ---- literals, stored raw: head, the literal bytes of the values, tail
  const uint32_t lh = ltot < 32 ? 1u : (ltot < 4096 ? 2u : 3u);
  uint8_t* const lits = out + 3 + lh;
  for (uint32_t x = tid; x < head; x += kThreads) lits[x] = in[bstart + x];
  for (uint32_t x = tid; x < tail; x += kThreads) lits[head + lrun + x] = in[prefix + li * w + x];
  for (uint32_t q = tid; q < nvb; q += kThreads) {
    const uint32_t c = key[q];
    if (c >= 8) continue;
    const uint32_t r = cd[q];
    const uint8_t* src = v + size_t(fi + q) * w;
    uint8_t* dst = lits + head + run_lit[r] + (c == 0 ? (q - run_pos[r]) * w : 0u);
    for (uint32_t k = 0; k < (c == 0 ? w : c); k++) dst[k] = src[k];
  }
  __syncthreads();
  // ---- sequences section: one thread (the FSE states are a serial chain)
  if (tid == 0) {
    if (lh == 1) out[3] = uint8_t(ltot << 3);
    else if (lh == 2) { out[3] = uint8_t(((ltot & 15) << 4) | 4); out[4] = uint8_t(ltot >> 4); }
    else { out[3] = uint8_t(((ltot & 15) << 4) | 12); out[4] = uint8_t(ltot >> 4); out[5] = uint8_t(ltot >> 12); }
    uint32_t pos = 3 + lh + ltot;
    uint8_t* o = out;
    if (nseq < 128) o[pos++] = uint8_t(nseq);
    else if (nseq < 0x7f00) { o[pos++] = uint8_t((nseq >> 8) + 128); o[pos++] = uint8_t(nseq); }
    else { o[pos++] = 255; o[pos++] = uint8_t(nseq - 0x7f00); o[pos++] = uint8_t((nseq - 0x7f00) >> 8); }
    bool ok = pos < content;
    uint32_t mode[3] = {0, 0, 0};
    if (nseq && ok) {
      const uint32_t mpos = pos++;
      for (int t = 0; t < 3; t++) {
        const int nsym = t == 0 ? zst::kMaxLL : (t == 1 ? zst::kMaxOF : zst::kMaxML);
        const int max_log = t == 0 ? zst::kLLLog : (t == 1 ? zst::kOFLog : zst::kMLLog);
        const uint32_t* cnt = sm.hist[t];
        int used = 0, lastsym = 0;
        for (int s = 0; s < nsym; s++) if (cnt[s]) { used++; lastsym = s; }
        if (used == 1) { mode[t] = 1; o[pos++] = uint8_t(lastsym); continue; }
        // predefined distribution: accuracy 6 (5 for offsets), defined up to code 35 / 28 / 52
        const int dlog = t == 1 ? 5 : 6, dsym = t == 0 ? 36 : (t == 1 ? 29 : 53);
        uint64_t cost_pre = ~0ull;
        if (lastsym < dsym) {
          cost_pre = 0;
          for (int s = 0; s <= lastsym; s++) {
            if (!cnt[s]) continue;
            const int d = t == 0 ? zst::ll_default(s) : (t == 1 ? zst::of_default(s) : zst::ml_default(s));
            cost_pre += uint64_t(cnt[s]) * uint32_t(dlog - hbit(uint32_t(d < 1 ? 1 : d)));
          }
        }
        int L = hbit(nseq) + 1;
        L = L < 5 ? 5 : (L > max_log ? max_log : L);
        if ((1 << L) <= used) L = hbit(uint32_t(used)) + 1;
        int16_t* norm = sm.norm[t];
        zfse_normalize(cnt, lastsym + 1, nseq, L, norm);
        const uint32_t hdr = zfse_write_ncount(o + pos, norm, lastsym + 1, L);
        uint64_t cost_cmp = uint64_t(hdr) * 8;
        for (int s = 0; s <= lastsym; s++) if (cnt[s]) cost_cmp += uint64_t(cnt[s]) * uint32_t(L - hbit(uint32_t(norm[s])));
        if (cost_cmp < cost_pre) { mode[t] = 2; pos += hdr; zfse_build_ct(sm.ct[t], norm, lastsym + 1, L, sm.cell_sym); }
        else {
          for (int s = 0; s < dsym; s++) norm[s] = int16_t(t == 0 ? zst::ll_default(s) : (t == 1 ? zst::of_default(s) : zst::ml_default(s)));
          zfse_build_ct(sm.ct[t], norm, dsym, dlog, sm.cell_sym);
        }
      }
      o[mpos] = uint8_t((mode[0] << 6) | (mode[1] << 4) | (mode[2] << 2));
      ok = pos < content;
      if (ok) {
        ZBitW bw{o + pos, 0, content - pos, 0, 0, false};
        uint32_t st[3] = {0, 0, 0};
        const uint32_t c0 = seq_code[nseq - 1];
        const uint32_t sym_last[3] = {c0 & 0xffu, (c0 >> 16) & 0xffu, (c0 >> 8) & 0xffu};
        for (int t = 0; t < 3; t++) if (mode[t] != 1) st[t] = zfse_init(sm.ct[t], sym_last[t]);
        auto extras = [&](uint32_t j, uint32_t code) {
          const uint32_t llc = code & 0xffu, mlc = (code >> 8) & 0xffu, ofc = (code >> 16) & 0xffu;
          bw.add(seq_ll[j] - zst::ll_base(llc), int(zst::ll_bits(llc)));
          bw.add(seq_ml[j] - zst::ml_base(mlc), int(zst::ml_bits(mlc)));
          bw.add(seq_of[j], int(ofc));
        };
        extras(nseq - 1, c0);
        for (uint32_t j = nseq - 1; j-- > 0 && !bw.over;) {
          const uint32_t c = seq_code[j];
          if (mode[1] != 1) zfse_encode(bw, sm.ct[1], st[1], (c >> 16) & 0xffu);
          if (mode[2] != 1) zfse_encode(bw, sm.ct[2], st[2], (c >> 8) & 0xffu);
          if (mode[0] != 1) zfse_encode(bw, sm.ct[0], st[0], c & 0xffu);
          extras(j, c);
        }
        if (mode[2] != 1) bw.add(st[2], int(sm.ct[2].log));
        if (mode[1] != 1) bw.add(st[1], int(sm.ct[1].log));
        if (mode[0] != 1) bw.add(st[0], int(sm.ct[0].log));
        bw.add(1, 1);                                         // end mark
        if (bw.nb) { if (bw.n < bw.cap) bw.p[bw.n] = uint8_t(bw.acc); else bw.over = true; bw.n++; }
        pos += bw.n;
        ok = !bw.over && pos - 3 < content;
      }
    }
    ok = ok && pos - 3 < content;
    const uint32_t bsize = ok ? pos - 3 : content;
    const uint32_t bh = (last ? 1u : 0u) | ((ok ? 2u : 0u) << 1) | (bsize << 3);
    out[0] = uint8_t(bh); out[1] = uint8_t(bh >> 8); out[2] = uint8_t(bh >> 16);
    sm.raw = ok ? 0u : 1u;
    uint32_t n = 3 + bsize;
    if (b == 0) {
      const uint32_t fh = zframe_header_len(ulen);
      uint8_t* f = out - fh;
      f[0] = 0x28; f[1] = 0xb5; f[2] = 0x2f; f[3] = 0xfd;
      if (ulen < 256) { f[4] = 0x20; f[5] = uint8_t(ulen); }
      else if (ulen < 65536 + 256) { f[4] = 0x60; f[5] = uint8_t(ulen - 256); f[6] = uint8_t((ulen - 256) >> 8); }
      else { f[4] = 0xa0; for (int k = 0; k < 4; k++) f[5 + k] = uint8_t(ulen >> (8 * k)); }
      n += fh;
    }
    zsz[blockIdx.x] = n;
  }
  __syncthreads();
  if (sm.raw) for (uint32_t x = tid; x < content; x += kThreads) out[3 + x] = in[bstart + x];
}

struct GatherDesc { uint64_t src_off, dst_off; uint32_t bytes, _pad; };
__global__ void __launch_bounds__(kThreads) gather_pages_kernel(const uint8_t* __restrict__ src, const GatherDesc* __restrict__ d, uint8_t* __restrict__ file) {
  const GatherDesc g = d[blockIdx.x];
  const uint8_t* s = src + g.src_off;
  uint8_t* t = file + g.dst_off;
  // destination-aligned 8-byte stores; the source word comes from two aligned loads + a funnel shift (any relative alignment)
  uint32_t head = uint32_t((8 - (reinterpret_cast<uintptr_t>(t) & 7)) & 7);
  if (head > g.bytes) head = g.bytes;
  if (threadIdx.x < head) t[threadIdx.x] = s[threadIdx.x];
  const uint32_t nwords = (g.bytes - head) >> 3;
  uint64_t* t8 = reinterpret_cast<uint64_t*>(t + head);
  const uint8_t* s0 = s + head;
  for (uint32_t wi = threadIdx.x; wi < nwords; wi += kThreads) {
    const uintptr_t a = reinterpret_cast<uintptr_t>(s0 + (size_t(wi) << 3));
    const uint64_t* q = reinterpret_cast<const uint64_t*>(a & ~uintptr_t(7));
    const uint32_t sh = uint32_t(a & 7) * 8;
    const uint64_t lo = q[0];
    t8[wi] = sh ? ((lo >> sh) | (q[1] << (64 - sh))) : lo;
  }
  for (uint32_t i = head + (nwords << 3) + threadIdx.x; i < g.bytes; i += kThreads) t[i] = s[i];
}

// ------------------------------------------------------------------------------------------------ Thrift compact writer
class TOut {
 public:
  std::vector<uint8_t> b;
  std::vector<int> last;
  void uvar(uint64_t v) { while (v >= 0x80) { b.push_back(uint8_t(v | 0x80)); v >>= 7; } b.push_back(uint8_t(v)); }
  void svar(int64_t v) { uvar((uint64_t(v) << 1) ^ uint64_t(v >> 63)); }
  void begin() { last.push_back(0); }
  void end() { b.push_back(0); last.pop_back(); }
  void field(int id, int type) {
    const int delta = id - last.back();
    if (delta > 0 && delta <= 15) b.push_back(uint8_t((delta << 4) | type));
    else { b.push_back(uint8_t(type)); svar(id); }
    last.back() = id;
  }
  void i32(int id, int64_t v) { field(id, 5); svar(v); }
  void i64(int id, int64_t v) { field(id, 6); svar(v); }
  void boolean(int id, bool v) { field(id, v ? 1 : 2); }
  void binary(int id, const void* p, size_t n) { field(id, 8); uvar(n); const uint8_t* q = static_cast<const uint8_t*>(p); b.insert(b.end(), q, q + n); }
  void str(int id, const std::string& s) { binary(id, s.data(), s.size()); }
  void list(int id, int etype, size_t n) { field(id, 9); if (n < 15) b.push_back(uint8_t((n << 4) | etype)); else { b.push_back(uint8_t(0xf0 | etype)); uvar(n); } }
  void struct_field(int id) { field(id, 12); begin(); }
  void list_str(const std::string& s) { uvar(s.size()); b.insert(b.end(), s.begin(), s.end()); }
};

int phys_of(uint32_t t) { return t == T_U64 || t == T_I64 ? 2 : (t == T_F32 ? 4 : (t == T_F64 ? 5 : 1)); }
int converted_of(uint32_t t) {      // parquet ConvertedType for the integer types that need one (-1: none)
  switch (t) {
    case T_U8: return 11; case T_U16: return 12; case T_U32: return 13; case T_U64: return 14;
    case T_I8: return 15; case T_I16: return 16;
    default: return -1;
  }
}

}  // namespace

int write_sst(hg_engine* e, const hg_schema_desc* schema, const ColIn* cols, uint32_t ncols, uint32_t R, const hg_write_props* props,
              uint8_t** host_out, uint64_t* size_out) {
  cudaStream_t s = e->stream;
  const uint32_t rg_rows = props->max_row_group_size ? props->max_row_group_size : 8192;
  const uint32_t codec = props->compression;
  const bool snappy = codec == 1, zstd = codec == 6;
  if (codec != 0 && !snappy && !zstd) return set_error(HG_ERR_UNSUPPORTED, "write: only UNCOMPRESSED, SNAPPY and ZSTD pages are implemented");
  const uint32_t nrg = (R + rg_rows - 1) / rg_rows;
  const uint64_t npages = uint64_t(nrg) * ncols;
  std::vector<PageJob> jobs(ncols);
  for (uint32_t c = 0; c < ncols; c++) {
    jobs[c] = PageJob{cols[c].vals, cols[c].valid, cols[c].type, cols[c].width, (cols[c].type == T_U64 || cols[c].type == T_I64 || cols[c].type == T_F64) ? 8u : 4u};
  }
  const uint32_t max_vals = std::min<uint32_t>(rg_rows, R ? R : 1);
  const uint64_t bstride = (uint64_t(16) + (max_vals + 7) / 8 + 8 + uint64_t(max_vals) * 8 + 63) & ~uint64_t(63);
  const uint64_t cstride = bstride + 64;
  const uint64_t sstride = ((uint64_t(max_vals) + 15) & ~uint64_t(15)) + (uint64_t(max_vals) * 3 + 4) * 4;
  // Zstandard: one slot per 128 KB block of a page (a page never exceeds bstride bytes); scratch per (page, block)
  const uint32_t nbmax = zblocks_of(uint32_t(std::min<uint64_t>(bstride, 0xffffffffull)));
  const uint32_t vcap = std::min<uint32_t>(max_vals, kZBlk / 4);
  const uint64_t zslot = (kZFront + 3 + std::min<uint64_t>(bstride, kZBlk) + kZPad + 63) & ~uint64_t(63);
  const uint64_t zcstride = nbmax * zslot;
  const uint64_t zsstride = (uint64_t(kZArrays) * vcap * 4 + 4 + 63) & ~uint64_t(63);
  DevBuf d_jobs, d_body, d_comp, d_meta, d_scratch, d_zsz;
  std::vector<PageMetaDev> meta(npages);
  std::vector<uint32_t> zsz(zstd ? npages * nbmax : 0);
  if (npages) {
    CU_TRY(d_jobs.alloc(jobs.size() * sizeof(PageJob), s));
    CU_TRY(d_body.alloc(npages * bstride, s));
    CU_TRY(d_meta.alloc(npages * sizeof(PageMetaDev), s));
    int rc = stage_upload(e, d_jobs.p, jobs.data(), jobs.size() * sizeof(PageJob), nullptr);
    if (rc) return rc;
    page_body_kernel<<<uint32_t(npages), kThreads, 0, s>>>(d_jobs.as<PageJob>(), ncols, R, rg_rows, d_body.as<uint8_t>(), bstride, d_meta.as<PageMetaDev>());
    e->launches++;
    if (snappy) {
      CU_TRY(d_comp.alloc(npages * cstride, s));
      CU_TRY(d_scratch.alloc(npages * sstride, s));
      snappy_encode_kernel<<<uint32_t(npages), kThreads, 0, s>>>(d_body.as<uint8_t>(), bstride, d_meta.as<PageMetaDev>(), d_jobs.as<PageJob>(), ncols,
                                                                d_comp.as<uint8_t>(), cstride, d_scratch.as<uint8_t>(), sstride, max_vals);
      e->launches++;
    } else if (zstd) {
      CU_TRY(d_comp.alloc(npages * zcstride, s));
      CU_TRY(d_scratch.alloc(npages * nbmax * zsstride, s));
      CU_TRY(d_zsz.alloc(npages * nbmax * sizeof(uint32_t), s));
      zstd_encode_kernel<<<uint32_t(npages * nbmax), kThreads, 0, s>>>(d_body.as<uint8_t>(), bstride, d_meta.as<PageMetaDev>(), d_jobs.as<PageJob>(), ncols, nbmax,
                                                                      d_comp.as<uint8_t>(), zcstride, zslot, d_zsz.as<uint32_t>(), d_scratch.as<uint8_t>(), zsstride, vcap);
      e->launches++;
      CU_TRY(cudaMemcpyAsync(zsz.data(), d_zsz.p, zsz.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    }
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpyAsync(meta.data(), d_meta.p, npages * sizeof(PageMetaDev), cudaMemcpyDeviceToHost, s));
    CU_TRY(cudaStreamSynchronize(s));
    if (zstd)
      for (uint64_t p = 0; p < npages; p++) {
        uint64_t c = 0;
        for (uint32_t b = 0; b < nbmax; b++) c += zsz[p * nbmax + b];
        meta[p].comp_size = uint32_t(c);
      }
  }
  // ---- host: page headers, offsets, footer
  std::vector<std::vector<uint8_t>> headers(npages);
  std::vector<GatherDesc> gd;
  gd.reserve(npages);
  std::vector<uint64_t> hdr_off(npages);
  uint64_t pos = 4;
  for (uint64_t p = 0; p < npages; p++) {
    const uint32_t g = uint32_t(p / ncols);
    const uint32_t rows = std::min<uint32_t>(rg_rows, R - g * rg_rows);
    TOut t;
    t.begin();
    t.i32(1, 0);                           // DATA_PAGE
    t.i32(2, meta[p].uncomp_size);
    t.i32(3, meta[p].comp_size);
    t.struct_field(5);                     // DataPageHeader
    t.i32(1, rows);
    t.i32(2, 0);                           // PLAIN
    t.i32(3, 3);                           // definition levels: RLE
    t.i32(4, 3);                           // repetition levels: RLE
    t.end();
    t.end();
    headers[p] = std::move(t.b);
    hdr_off[p] = pos;
    pos += headers[p].size();
    if (zstd) {                            // the frame: its blocks' slots, the frame header in front of block 0
      uint64_t at = pos;
      for (uint32_t b = 0; b < nbmax; b++) {
        const uint32_t n = zsz[p * nbmax + b];
        if (!n) continue;
        gd.push_back(GatherDesc{p * zcstride + b * zslot + kZFront - (b == 0 ? zframe_header_len(meta[p].uncomp_size) : 0u), at, n, 0});
        at += n;
      }
    } else {
      gd.push_back(GatherDesc{p * (snappy ? cstride : bstride), pos, meta[p].comp_size, 0});
    }
    pos += meta[p].comp_size;
  }
  TOut f;
  f.begin();
  f.i32(1, 1);                             // version (WriterVersion::PARQUET_1_0)
  f.list(2, 12, size_t(ncols) + 1);        // schema
  {
    f.begin();
    f.str(4, "arrow_schema");
    f.i32(5, ncols);
    f.end();
    for (uint32_t c = 0; c < ncols; c++) {
      f.begin();
      f.i32(1, phys_of(cols[c].type));
      f.i32(3, 1);                         // OPTIONAL: every field of the reference's schemas is nullable
      std::string tmp;
      f.str(4, schema->names && schema->names[c] ? std::string(schema->names[c]) : "c" + std::to_string(c));
      const int cv = converted_of(cols[c].type);
      if (cv >= 0) f.i32(6, cv);
      f.end();
    }
  }
  f.i64(3, R);
  f.list(4, 12, nrg);
  for (uint32_t g = 0; g < nrg; g++) {
    const uint32_t rows = std::min<uint32_t>(rg_rows, R - g * rg_rows);
    f.begin();
    f.list(1, 12, ncols);
    uint64_t rg_uncomp = 0, rg_comp = 0;
    for (uint32_t c = 0; c < ncols; c++) {
      const uint64_t p = uint64_t(g) * ncols + c;
      const uint64_t hsz = headers[p].size();
      f.begin();                           // ColumnChunk
      f.i64(2, int64_t(hdr_off[p]));       // file_offset
      f.struct_field(3);                   // ColumnMetaData
      f.i32(1, phys_of(cols[c].type));
      f.list(2, 5, 2); f.svar(0); f.svar(3);      // encodings: PLAIN, RLE
      f.list(3, 8, 1); f.list_str(schema->names && schema->names[c] ? std::string(schema->names[c]) : "c" + std::to_string(c));
      f.i32(4, int(codec));
      f.i64(5, rows);
      f.i64(6, int64_t(meta[p].uncomp_size + hsz));
      f.i64(7, int64_t(meta[p].comp_size + hsz));
      f.i64(9, int64_t(hdr_off[p]));       // data_page_offset
      f.struct_field(12);                  // Statistics
      f.i64(3, meta[p].null_count);
      if (meta[p].has_minmax) {
        const uint32_t pw = jobs[c].pwidth;
        f.binary(5, &meta[p].mx, pw);      // max_value
        f.binary(6, &meta[p].mn, pw);      // min_value
      }
      f.end();
      f.end();
      f.end();
      rg_uncomp += meta[p].uncomp_size + hsz;
      rg_comp += meta[p].comp_size + hsz;
    }
    f.i64(2, int64_t(rg_uncomp));
    f.i64(3, rows);
    if (props->enable_sorting_columns) {
      f.list(4, 12, schema->num_primary_keys);
      for (uint32_t c = 0; c < schema->num_primary_keys; c++) { f.begin(); f.i32(1, c); f.boolean(2, false); f.boolean(3, true); f.end(); }
    }
    f.i64(5, int64_t(hdr_off[uint64_t(g) * ncols]));
    f.i64(6, int64_t(rg_comp));
    f.field(7, 4); f.svar(g);              // ordinal (i16)
    f.end();
  }
  f.str(6, "horaedb_b200 GPU SST writer (PLAIN, RLE levels, " + std::string(snappy ? "SNAPPY" : (zstd ? "ZSTD" : "UNCOMPRESSED")) + ")");
  f.list(7, 12, ncols);                    // column_orders: TYPE_ORDER for every column (makes min_value / max_value usable)
  for (uint32_t c = 0; c < ncols; c++) { f.begin(); f.struct_field(1); f.end(); f.end(); }
  f.end();
  const uint64_t footer_off = pos;
  const uint64_t total = footer_off + f.b.size() + 8;
  if (total > 0xffffffffull) return set_error(HG_ERR_UNSUPPORTED, "output SST larger than 4 GiB (FileMeta.size is u32, sst.rs:155-160)");
  // ---- assemble on the device, one copy back
  uint8_t* host = nullptr;
  CU_TRY(cudaMallocHost(&host, total + 16));
  DevBuf d_file, d_gd;
  CU_TRY(d_file.alloc(total + 16, s));
  std::memcpy(host, "PAR1", 4);
  if (npages) {
    CU_TRY(d_gd.alloc(gd.size() * sizeof(GatherDesc), s));
    CU_TRY(cudaMemcpyAsync(d_gd.p, gd.data(), gd.size() * sizeof(GatherDesc), cudaMemcpyHostToDevice, s));
    gather_pages_kernel<<<uint32_t(gd.size()), kThreads, 0, s>>>(snappy || zstd ? d_comp.as<uint8_t>() : d_body.as<uint8_t>(), d_gd.as<GatherDesc>(), d_file.as<uint8_t>());
    e->launches++;
    CU_TRY(cudaMemcpyAsync(host + 4, d_file.as<uint8_t>() + 4, footer_off - 4, cudaMemcpyDeviceToHost, s));
    CU_TRY(cudaStreamSynchronize(s));
    for (uint64_t p = 0; p < npages; p++) std::memcpy(host + hdr_off[p], headers[p].data(), headers[p].size());   // a few dozen bytes each
  }
  std::memcpy(host + footer_off, f.b.data(), f.b.size());
  const uint32_t flen = uint32_t(f.b.size());
  std::memcpy(host + footer_off + f.b.size(), &flen, 4);
  std::memcpy(host + footer_off + f.b.size() + 4, "PAR1", 4);
  *host_out = host;
  *size_out = total;
  e->stats.bytes_d2h += total;
  return HG_OK;
}

}  // namespace writer
}  // namespace horae
