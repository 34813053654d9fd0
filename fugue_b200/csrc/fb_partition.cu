// K1+K2+K3: hash partition of a columnar table on sm_100a.
//
// Replaces the grouping/repartition step of the reference's map path:
//   fugue/execution/native_execution_engine.py:166-168  (safe_groupby_apply)
//   fugue_dask/_utils.py:44-59, 124-130, 146-169        (hash_repartition)
//
// Design (HBM-bound byte movement; no tensor-core work exists on this path):
//   * the row range is cut into contiguous chunks of whole TILE-row tiles (at most
//     2 x #SM of them) plus one tail chunk holding the final partial tile;
//   * pass 1 (fb_hist_kernel)   : per-chunk histogram of partition ids (reads the
//     key column(s) only: 8 B/row for the benchmark schema);
//   * scan  (fb_scan_*_kernel)  : exclusive prefix per partition over chunks, then
//     over partitions -> part_offsets[num+1] and chunk bases;
//   * pass 2, fast path (fb_scatter_tma_kernel; single 8-byte key, 8-byte columns):
//     one persistent CTA per SM = 1 producer warp + 16 consumer warps.  The producer
//     streams (tile, column) units into a ring of 32 KB shared-memory stages with
//     TMA bulk copies (cp.async.bulk + mbarrier complete_tx), running several units
//     ahead of the consumers, across tile and chunk boundaries.  Consumers hash the
//     staged key tile, rank rows stably per partition (ballot match + warp-private
//     counters), build the slot -> source-row map of the partition-ordered tile and
//     then, per column, gather straight from the staged tile and store contiguous
//     runs (one run per partition present in the tile) to global memory.  Running
//     per-partition output cursors live in shared memory for the whole chunk.
//   * pass 2, generic path (fb_scatter_kernel; any widths/keys, partial tiles):
//     register-staged loads, permutation through double-buffered shared memory.
//   Algorithmic traffic 128 B/row (read 64 + write 64) for the 8x8-byte schema;
//   the implementation adds the 8 B/row key re-read of pass 1.
#include <stdlib.h>

#include <mutex>

#include "fb_common.cuh"

namespace {

constexpr int kBlock = 512;             // threads per CTA
constexpr int kItems = 8;               // rows per thread per tile
constexpr int kTile = kBlock * kItems;  // 4096 rows per tile
constexpr int kWarps = kBlock / 32;
constexpr int kCtasPerSm = 2;

struct FbCols {
  const void* src[FB_MAX_COLS];
  void* dst[FB_MAX_COLS];
  int32_t width[FB_MAX_COLS];
  int32_t ncols;
};

struct ChunkGeom {
  int64_t nrows;
  int64_t full_rows;        // rows covered by whole tiles
  int64_t tiles_per_chunk;  // whole tiles per full chunk
  int32_t nchunks_full;     // chunks made of whole tiles
  int32_t nchunks;          // + 1 if there is a partial tail tile
};

inline ChunkGeom make_geom(int dev, int64_t nrows) {
  ChunkGeom g;
  g.nrows = nrows;
  const int64_t ntiles_full = nrows / kTile;
  g.full_rows = ntiles_full * kTile;
  const int64_t max_chunks = (int64_t)fb_sm_count(dev) * kCtasPerSm;
  g.tiles_per_chunk = ntiles_full > 0 ? (ntiles_full + max_chunks - 1) / max_chunks : 1;
  g.nchunks_full = (int32_t)((ntiles_full + g.tiles_per_chunk - 1) / g.tiles_per_chunk);
  g.nchunks = g.nchunks_full + (g.full_rows < nrows ? 1 : 0);
  return g;
}

__host__ __device__ __forceinline__ void chunk_range(const ChunkGeom& g, int c, int64_t& r0, int64_t& r1) {
  if (c < g.nchunks_full) {
    r0 = (int64_t)c * g.tiles_per_chunk * kTile;
    r1 = r0 + g.tiles_per_chunk * kTile;
    if (r1 > g.full_rows) r1 = g.full_rows;
  } else {
    r0 = g.full_rows;
    r1 = g.nrows;
  }
}

template <bool kSingleU64>
__device__ __forceinline__ uint32_t compute_pid(const FbKeys& keys, const FbDiv& dv, int64_t row) {
  uint64_t h;
  if (kSingleU64) {
    h = fb_hash_single_u64(__ldg((const unsigned long long*)keys.ptr[0] + row));
  } else {
    if (keys.digit_shift >= 0)  // one pass of an LSD radix sort on an 8-byte unsigned sort key
      return (uint32_t)(__ldg((const unsigned long long*)keys.ptr[0] + row) >> keys.digit_shift) & (dv.d - 1);
    h = fb_row_hash(keys, row);
  }
  return fb_fastmod(h, dv);
}

// ---------------------------------------------------------------------------
// K1 alone: materialise partition ids (tests, repartition planning)
// ---------------------------------------------------------------------------
template <bool kSingleU64>
__global__ void fb_pid_kernel(FbKeys keys, FbDiv dv, int64_t nrows, uint32_t* __restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < nrows; i += stride) out[i] = compute_pid<kSingleU64>(keys, dv, i);
}

__global__ void fb_row_hash_kernel(FbKeys keys, int64_t nrows, uint64_t* __restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < nrows; i += stride) out[i] = fb_row_hash(keys, i);
}

// ---------------------------------------------------------------------------
// Warp-level "which lanes hold my value": kBits ballots instead of the hardware
// MATCH instruction (MATCH.ANY runs on the ADU pipe at ~70 cycles per warp
// instruction on sm_100 - measured with ncu, profiles/r1_v1_* - and caps the
// whole kernel; ballots issue at full rate).  `m` starts as the mask of lanes
// that take part.
// ---------------------------------------------------------------------------
template <int kBits>
__device__ __forceinline__ unsigned match_lanes(uint32_t v, unsigned m) {
#pragma unroll
  for (int b = 0; b < kBits; ++b) {
    const bool bit = (v >> b) & 1u;
    const unsigned bal = __ballot_sync(0xFFFFFFFFu, bit);
    m &= bit ? bal : ~bal;
  }
  return m;
}

// ---------------------------------------------------------------------------
// pass 1: per-chunk histogram. hist layout: [chunk][num]
// shared: cnt[kWarps][num] warp-private counters (no atomics)
// ---------------------------------------------------------------------------
constexpr int kHistBlock = 1024;  // 2 CTAs/SM -> full occupancy (32 registers/thread)
constexpr int kHistWarps = kHistBlock / 32;
constexpr int kHistRows = kHistBlock * kItems;

template <bool kSingleU64, int kBits>
__global__ void __launch_bounds__(kHistBlock, 2)
fb_hist_kernel(FbKeys keys, FbDiv dv, uint32_t num, ChunkGeom g, int chunk0, uint32_t* __restrict__ hist) {
  extern __shared__ uint32_t s_cnt[];
  for (uint32_t i = threadIdx.x; i < (uint32_t)kHistWarps * num; i += kHistBlock) s_cnt[i] = 0;
  __syncthreads();
  int64_t row0, row1;
  chunk_range(g, chunk0 + (int)blockIdx.x, row0, row1);
  const unsigned lt = fb_lanemask_lt();
  uint32_t* my = s_cnt + (size_t)(threadIdx.x >> 5) * num;
  for (int64_t base = row0; base < row1; base += kHistRows) {
    uint32_t pid[kItems];
    const bool full = base + kHistRows <= row1;
#pragma unroll
    for (int r = 0; r < kItems; ++r) {
      int64_t row = base + (int64_t)r * kHistBlock + threadIdx.x;
      pid[r] = (full || row < row1) ? compute_pid<kSingleU64>(keys, dv, row) : 0xFFFFFFFFu;
    }
#pragma unroll
    for (int r = 0; r < kItems; ++r) {
      const bool ok = pid[r] != 0xFFFFFFFFu;
      unsigned m = match_lanes<kBits>(pid[r], __ballot_sync(0xFFFFFFFFu, ok));
      if (ok && (m & lt) == 0) my[pid[r]] += (uint32_t)__popc(m);
      __syncwarp();
    }
  }
  __syncthreads();
  uint32_t* out = hist + (size_t)(chunk0 + (int)blockIdx.x) * num;
  for (uint32_t b = threadIdx.x; b < num; b += kHistBlock) {
    uint32_t t = 0;
#pragma unroll 8
    for (int w = 0; w < kHistWarps; ++w) t += s_cnt[(size_t)w * num + b];
    out[b] = t;
  }
}

// ---------------------------------------------------------------------------
// pass 1 for num <= 256 (full tiles): histogram AND the complete ranking of every 4096-row tile, so
// that pass 2 never hashes, matches or counts.  One 12800-byte record per tile in scratch:
//   [0, 4096)       uint8  partition id of every row
//   [4096, 12288)   uint16 rank of the row among the rows of the same partition in this tile
//   [12288, 12800)  uint16 rows per partition in this tile (256 entries)
// Pass 2 loads one record per tile with a single TMA bulk copy.
//
// One warp ranks a whole tile, 32 rows per step in row order, against warp-private counters: the
// rank of a row is the counter of its partition plus the lanes of the same partition below it, so
// no prefix over warps and no block barrier is needed, and the counters are the tile's counts when
// the tile ends.  The lanes of the same partition come from kBits ballots turned into two
// 16-entry lookup tables (lane i holds the lanes whose low / high nibble is not i), read back with
// two shuffles: one vote and one LOP3 per bit instead of a per-bit select and merge in every lane.
// The CTA (2 x 1024 threads per SM) owns one chunk; its warps take the chunk's tiles in turn.
// ---------------------------------------------------------------------------
constexpr int kRankBlock = 1024, kRankWarps = kRankBlock / 32;
constexpr uint32_t kMetaRank = kTile, kMetaCnt = 3 * kTile, kMetaBytes = 3 * kTile + 512;

// ballot of (v & bit) != 0; spelled in PTX so that the test stays one predicate-setting instruction
__device__ __forceinline__ unsigned ballot_bit(uint32_t v, uint32_t bit) {
  unsigned r;
  asm("{\n\t.reg .pred p;\n\t.reg .b32 t;\n\tand.b32 t, %1, %2;\n\tsetp.ne.u32 p, t, 0;\n\t"
      "vote.sync.ballot.b32 %0, p, 0xffffffff;\n}"
      : "=r"(r)
      : "r"(v), "r"(bit));
  return r;
}

template <bool kSingleU64, int kBits, bool kPow2>
__global__ void __launch_bounds__(kRankBlock, 2)
fb_rank_kernel(FbKeys keys, FbDiv dv, uint32_t num, ChunkGeom g, uint32_t* __restrict__ hist,
               uint8_t* __restrict__ meta) {
  static_assert(kBits == 4 || kBits == 8, "partition ids of 4 or 8 bits");
  // steps whose keys are loaded together; the 64-bit division by other counts needs the registers
  constexpr int kUnroll = kSingleU64 && !kPow2 ? 2 : 4;
  __shared__ __align__(16) uint16_t s_cnt[kRankWarps][256];
  __shared__ uint32_t s_hist[256];
  for (uint32_t i = threadIdx.x; i < (uint32_t)kRankWarps * 128; i += kRankBlock) ((uint32_t*)s_cnt)[i] = 0;
  if (threadIdx.x < 256) s_hist[threadIdx.x] = 0;
  __syncthreads();
  int64_t row0, row1;
  chunk_range(g, (int)blockIdx.x, row0, row1);  // launched over the full chunks only
  const uint32_t tile0 = (uint32_t)(row0 / kTile), ntiles = (uint32_t)((row1 - row0) / kTile);
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned lt = fb_lanemask_lt();
  uint16_t* __restrict__ my = s_cnt[warp];
  unsigned neg[4];  // lane i, table entry i & 15: bit b of i spread over the word
#pragma unroll
  for (int b = 0; b < 4; ++b) neg[b] = 0u - ((lane >> b) & 1u);
  for (uint32_t t = tile0 + warp; t < tile0 + ntiles; t += kRankWarps) {
    const int64_t t0 = (int64_t)t * kTile;
    uint8_t* __restrict__ rec = meta + (size_t)t * kMetaBytes;
    uint8_t* __restrict__ rp = rec + lane;
    uint16_t* __restrict__ rq = (uint16_t*)(rec + kMetaRank) + lane;
    const uint32_t r0 = (uint32_t)t0 + lane;  // plan_impl limits nrows to 32 bits
#pragma unroll 1
    for (int i = 0; i < kTile / 32; i += kUnroll) {
      uint32_t pid[kUnroll];
#pragma unroll
      for (int u = 0; u < kUnroll; ++u) {
        if (kSingleU64) {  // compute_pid with the divisor's kind known at compile time
          const uint64_t h = fb_hash_single_u64(__ldg((const unsigned long long*)keys.ptr[0] + (r0 + (i + u) * 32)));
          pid[u] = kPow2 ? (uint32_t)h & (dv.d - 1) : fb_fastmod_magic(h, dv);
        } else {
          pid[u] = compute_pid<false>(keys, dv, r0 + (i + u) * 32);
        }
      }
#pragma unroll
      for (int u = 0; u < kUnroll; ++u) {
        const uint32_t p = pid[u];
        // lo / hi: lanes whose low / high nibble differs from table entry lane & 15
        unsigned lo = ballot_bit(p, 1) ^ neg[0], hi = kBits > 4 ? ballot_bit(p, 16) ^ neg[0] : 0;
#pragma unroll
        for (int b = 1; b < 4; ++b) {
          lo |= ballot_bit(p, 1u << b) ^ neg[b];
          if (kBits > 4) hi |= ballot_bit(p, 16u << b) ^ neg[b];
        }
        lo = __shfl_sync(0xFFFFFFFFu, lo, p, 16);
        if (kBits > 4) hi = __shfl_sync(0xFFFFFFFFu, hi, p >> 4, 16);
        const unsigned m = ~(lo | hi);  // lanes with partition p
        const uint32_t old = my[p];
        __syncwarp();
        my[p] = (uint16_t)(old + __popc(m));  // the same value from every lane of the partition
        __syncwarp();
        rp[(i + u) * 32] = (uint8_t)p;
        rq[(i + u) * 32] = (uint16_t)(old + __popc(m & lt));
      }
    }
    // the counters are the tile's counts: lane l moves partitions 8l .. 8l + 7 and clears them
    const uint4 c = ((const uint4*)my)[lane];
    ((uint4*)(rec + kMetaCnt))[lane] = c;
    ((uint4*)my)[lane] = make_uint4(0, 0, 0, 0);
    const uint32_t w[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      atomicAdd(&s_hist[lane * 8 + 2 * j], w[j] & 0xFFFFu);
      atomicAdd(&s_hist[lane * 8 + 2 * j + 1], w[j] >> 16);
    }
    __syncwarp();
  }
  __syncthreads();
  if (threadIdx.x < num) hist[(size_t)blockIdx.x * num + threadIdx.x] = s_hist[threadIdx.x];
}

// ---------------------------------------------------------------------------
// scan A: one CTA per partition id: exclusive prefix over chunks (in place),
// total -> totals[b].  nchunks <= 2 * SM count (<= 1024 handled generally).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
fb_scan_chunks_kernel(uint32_t* __restrict__ hist, uint32_t num, int32_t nchunks,
                      int64_t* __restrict__ totals) {
  __shared__ uint32_t s_warp[8];
  __shared__ uint32_t s_carry;
  const uint32_t b = blockIdx.x;
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (int32_t c0 = 0; c0 < nchunks; c0 += 256) {
    int32_t c = c0 + threadIdx.x;
    uint32_t v = c < nchunks ? hist[(size_t)c * num + b] : 0;
    uint32_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
      if (lane >= (unsigned)o) x += y;
    }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    uint32_t wbase = 0;
    for (unsigned w = 0; w < warp; ++w) wbase += s_warp[w];
    uint32_t carry = s_carry;
    if (c < nchunks) hist[(size_t)c * num + b] = carry + wbase + x - v;
    __syncthreads();
    if (threadIdx.x == 255) s_carry = carry + wbase + x;
    __syncthreads();
  }
  if (threadIdx.x == 0) totals[b] = (int64_t)s_carry;
}

// scan B: single CTA: exclusive prefix over partitions (int64), in place on
// offsets[0..num]; input totals in offsets[0..num-1].
__global__ void __launch_bounds__(1024)
fb_scan_parts_kernel(int64_t* __restrict__ offsets, uint32_t num) {
  __shared__ int64_t s_warp[32];
  __shared__ int64_t s_carry;
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (uint32_t b0 = 0; b0 < num; b0 += 1024) {
    uint32_t b = b0 + threadIdx.x;
    int64_t v = b < num ? offsets[b] : 0;
    int64_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int64_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
      if (lane >= (unsigned)o) x += y;
    }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    int64_t wbase = 0;
    for (unsigned w = 0; w < warp; ++w) wbase += s_warp[w];
    int64_t carry = s_carry;
    if (b < num) offsets[b] = carry + wbase + x - v;
    __syncthreads();
    if (threadIdx.x == 1023) s_carry = carry + wbase + x;
    __syncthreads();
  }
  if (threadIdx.x == 0) offsets[num] = s_carry;
}

// ---------------------------------------------------------------------------
// pass 2: scatter.  Dynamic shared memory, addressed from one extern array so
// that every access compiles to LDS/STS with offsets computed once per tile:
//   [0, 2*T*8)                buf[2][T] uint64   column staging, double buffered
//   then uint32 regions (nbp = padded number of bins; bins = num + 1 sentinel that
//   collects the slots past the end of a partial tile):
//     delta[nbp]              (cursor - bin_start) of the current tile, mod 2^32
//     cursor[nbp]             running output row of every partition for this chunk
//     bin_start[nbp]          exclusive prefix of the tile histogram
//     cnt[kWarps][nbp]        warp-private counters -> exclusive prefix over warps
//     scanw[32]               warp totals of the block scan
//   then pid_sorted[T] uint16 partition id of every slot of the permuted tile
// ---------------------------------------------------------------------------
__host__ __device__ inline uint32_t nb_padded(uint32_t num) { return (num + 1 + 3) & ~3u; }

__host__ __device__ inline size_t scatter_smem_bytes(uint32_t num) {
  size_t nbp = nb_padded(num);
  return 2 * (size_t)kTile * 8 + (3 + (size_t)kWarps) * nbp * 4 + 32 * 4 + (size_t)kTile * 2;
}

constexpr int kMaxPer = (FB_MAX_PARTITIONS + 1 + kBlock - 1) / kBlock;  // bins per thread in the scan

struct TileCtx {  // all pointers are into shared memory
  uint64_t* buf;
  uint32_t* delta;
  uint32_t* cursor;
  uint32_t* bin_start;
  uint32_t* cnt;
  uint32_t* scanw;
  uint16_t* pid_sorted;
  uint32_t nbp;
};

template <typename T, bool kFull>
__device__ __forceinline__ void load_col(const void* __restrict__ src, int64_t warp_row0, int warp_rows,
                                         unsigned lane, T (&v)[kItems]) {
  const T* __restrict__ p = (const T*)src + warp_row0 + lane;
#pragma unroll
  for (int r = 0; r < kItems; ++r)
    if (kFull || r * 32 + (int)lane < warp_rows) v[r] = __ldg(p + r * 32);
}

// Moves every column of width sizeof(T): coalesced load -> permute through shared memory ->
// run-coalesced store.  One barrier per column (double buffered staging).
template <typename T, bool kFull>
__device__ __forceinline__ void move_columns(const FbCols& cols, const TileCtx& cx,
                                             const uint32_t (&pos)[kItems], const uint32_t (&dst)[kItems],
                                             int64_t warp_row0, int warp_rows, int tile_rows,
                                             unsigned lane, int& phase) {
  int c = 0;
  while (c < cols.ncols && cols.width[c] != (int)sizeof(T)) ++c;
  if (c >= cols.ncols) return;
  T v[kItems];
  load_col<T, kFull>(cols.src[c], warp_row0, warp_rows, lane, v);
  while (c < cols.ncols) {
    T* __restrict__ buf = (T*)(cx.buf + (size_t)(phase & 1) * kTile);
#pragma unroll
    for (int r = 0; r < kItems; ++r) buf[pos[r]] = v[r];
    int nxt = c + 1;
    while (nxt < cols.ncols && cols.width[nxt] != (int)sizeof(T)) ++nxt;
    if (nxt < cols.ncols) load_col<T, kFull>(cols.src[nxt], warp_row0, warp_rows, lane, v);  // prefetch
    __syncthreads();
    T* __restrict__ out = (T*)cols.dst[c];
#pragma unroll
    for (int k = 0; k < kItems; ++k) {
      const int j = k * kBlock + (int)threadIdx.x;
      if (kFull || j < tile_rows) out[dst[k]] = buf[j];
    }
    ++phase;
    c = nxt;
  }
}

template <bool kSingleU64, int kBits, bool kFull, bool kAll8>
__device__ __forceinline__ void scatter_tile(const FbKeys& keys, const FbDiv& dv, const uint32_t num,
                                             const FbCols& cols, const TileCtx& cx,
                                             const int64_t tile_row0, const int tile_rows, int& phase) {
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned lt = fb_lanemask_lt();
  const uint32_t nb = num + 1;
  const uint32_t nbp = cx.nbp;
  uint32_t* __restrict__ my_cnt = cx.cnt + warp * nbp;
  const int64_t warp_row0 = tile_row0 + (int64_t)warp * (32 * kItems);
  const int warp_rows = tile_rows - (int)warp * (32 * kItems);  // rows of this warp's stripe that exist

  // -- 1. partition ids of my rows (warp-striped: row = warp_row0 + r*32 + lane)
  uint32_t pid[kItems];
#pragma unroll
  for (int r = 0; r < kItems; ++r) {
    const bool ok = kFull || (r * 32 + (int)lane) < warp_rows;
    pid[r] = ok ? compute_pid<kSingleU64>(keys, dv, warp_row0 + r * 32 + lane) : num;
  }

  // -- 2. stable rank inside (warp, partition): ballot match + warp-private counters
  //       (counters are zero here: cleared before the tile loop and at the end of every tile)
  uint32_t pos[kItems];
#pragma unroll
  for (int r = 0; r < kItems; ++r) {
    const unsigned m = match_lanes<kBits + (kFull ? 0 : 1)>(pid[r], 0xFFFFFFFFu);
    const unsigned before = __popc(m & lt);
    uint32_t old = 0;
    if (before == 0) {
      old = my_cnt[pid[r]];
      my_cnt[pid[r]] = old + __popc(m);
    }
    __syncwarp();
    old = __shfl_sync(0xFFFFFFFFu, old, __ffs(m) - 1);
    pos[r] = old + before;
  }
  __syncthreads();

  // -- 3. per partition: exclusive prefix over warps, then block-wide exclusive scan of the
  //       tile histogram.  Thread t owns bins [t*per, t*per + per).
  {
    const uint32_t per = (nb + kBlock - 1) / kBlock;
    const uint32_t b0 = threadIdx.x * per;
    uint32_t tot[kMaxPer];
    uint32_t sum = 0;
#pragma unroll
    for (int i = 0; i < kMaxPer; ++i) {
      tot[i] = 0;
      if ((uint32_t)i < per && b0 + i < nb) {
        uint32_t run = 0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) {
          const uint32_t t = cx.cnt[w * nbp + b0 + i];
          cx.cnt[w * nbp + b0 + i] = run;
          run += t;
        }
        tot[i] = run;
        sum += run;
      }
    }
    uint32_t x = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
      if (lane >= (unsigned)o) x += y;
    }
    if (lane == 31) cx.scanw[warp] = x;
    __syncthreads();
    uint32_t run = x - sum;
    {
      const uint32_t wt = lane < kWarps ? cx.scanw[lane] : 0;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) {
        const uint32_t v = __shfl_sync(0xFFFFFFFFu, wt, w);
        if ((unsigned)w < warp) run += v;
      }
    }
#pragma unroll
    for (int i = 0; i < kMaxPer; ++i) {
      if ((uint32_t)i < per && b0 + i < nb) {
        const uint32_t cur = cx.cursor[b0 + i];
        cx.bin_start[b0 + i] = run;
        cx.delta[b0 + i] = cur - run;  // slot j of the permuted tile lands at output row delta + j
        cx.cursor[b0 + i] = cur + tot[i];
        run += tot[i];
      }
    }
  }
  __syncthreads();

  // -- 4. final slot of every row inside the permuted tile; publish the slot -> pid map
#pragma unroll
  for (int r = 0; r < kItems; ++r) {
    pos[r] += cx.bin_start[pid[r]] + my_cnt[pid[r]];
    cx.pid_sorted[pos[r]] = (uint16_t)pid[r];
  }
  __syncthreads();
  // output row of the slots this thread writes (same for every column)
  uint32_t dst[kItems];
#pragma unroll
  for (int k = 0; k < kItems; ++k) {
    const int j = k * kBlock + (int)threadIdx.x;
    dst[k] = cx.delta[cx.pid_sorted[j]] + (uint32_t)j;
  }
  // counters are dead from here on: clear them for the next tile (visibility is covered by the
  // barriers of the column loop / the trailing barrier)
  for (uint32_t i = threadIdx.x; i < (uint32_t)kWarps * nbp; i += kBlock) cx.cnt[i] = 0;

  // -- 5. move the columns
  move_columns<uint64_t, kFull>(cols, cx, pos, dst, warp_row0, warp_rows, tile_rows, lane, phase);
  if (!kAll8) {
    move_columns<uint32_t, kFull>(cols, cx, pos, dst, warp_row0, warp_rows, tile_rows, lane, phase);
    move_columns<uint16_t, kFull>(cols, cx, pos, dst, warp_row0, warp_rows, tile_rows, lane, phase);
    move_columns<uint8_t, kFull>(cols, cx, pos, dst, warp_row0, warp_rows, tile_rows, lane, phase);
  }
  __syncthreads();  // staging buffers, delta, pid_sorted are rewritten by the next tile
}

template <bool kSingleU64, int kBits, bool kAll8>
__global__ void __launch_bounds__(kBlock, kCtasPerSm)
fb_scatter_kernel(FbKeys keys, FbDiv dv, uint32_t num, ChunkGeom g, int chunk0,
                  const uint32_t* __restrict__ chunk_base, const int64_t* __restrict__ part_offsets,
                  FbCols cols) {
  extern __shared__ __align__(128) uint64_t smem64[];
  TileCtx cx;
  cx.nbp = nb_padded(num);
  cx.buf = smem64;
  cx.delta = (uint32_t*)(smem64 + 2 * kTile);
  cx.cursor = cx.delta + cx.nbp;
  cx.bin_start = cx.cursor + cx.nbp;
  cx.cnt = cx.bin_start + cx.nbp;
  cx.scanw = cx.cnt + kWarps * cx.nbp;
  cx.pid_sorted = (uint16_t*)(cx.scanw + 32);

  const int chunk = chunk0 + (int)blockIdx.x;
  int64_t chunk_row0, chunk_row1;
  chunk_range(g, chunk, chunk_row0, chunk_row1);

  for (uint32_t b = threadIdx.x; b < cx.nbp; b += kBlock)
    cx.cursor[b] = b < num ? (uint32_t)part_offsets[b] + chunk_base[(size_t)chunk * num + b] : 0u;
  for (uint32_t i = threadIdx.x; i < (uint32_t)kWarps * cx.nbp; i += kBlock) cx.cnt[i] = 0;
  __syncthreads();

  int phase = 0;
  for (int64_t tile_row0 = chunk_row0; tile_row0 < chunk_row1; tile_row0 += kTile) {
    const int64_t left = chunk_row1 - tile_row0;
    if (left >= kTile)
      scatter_tile<kSingleU64, kBits, true, kAll8>(keys, dv, num, cols, cx, tile_row0, kTile, phase);
    else
      scatter_tile<kSingleU64, kBits, false, kAll8>(keys, dv, num, cols, cx, tile_row0, (int)left, phase);
  }
}

// ---------------------------------------------------------------------------
// pass 2, fast path: TMA-pipelined scatter with software write-combining.
//
// Measured on B200 (profiles/r1_notes.md): a partition-ordered tile written as
// 8-byte-aligned runs costs 4.8 ms / 100 M rows because run heads/tails are partial
// 32-byte sectors (L2 fills them from DRAM and writes them back twice); the same
// traffic with sector-aligned runs costs 3.2 ms, with linear stores 2.2 ms.  So every
// partition keeps its last (< G) rows per column in a shared-memory carry buffer and
// only whole G-row groups (G * 8 B = one or more full sectors) are stored; the
// carried rows are prepended to the partition's rows of the next tile.  Partial
// stores happen only at chunk heads/tails (2 per partition per column per chunk).
//
// Shared memory (dynamic, one CTA per SM), T = kTile, E = num * (G - 1):
//   ring[S][T] uint64          S x 32 KB stages filled by cp.async.bulk (TMA)
//   carry[ncols + 1][E] uint64 carried rows per column (+1 spare: new carry is written
//                              to the spare buffer, buffers rotate every column step)
//   slotinfo[T + E] uint32     output slot -> (partition << 16 | source descriptor)
//   carryinfo[E] uint16        new carry entry -> source descriptor
//   per-partition uint32 arrays: wpos, kcnt, binfo, bin_start, wstart, wdelta
//   cnt[kWarps][nbp] uint16, scanw[64] uint32, mbarriers
// Source descriptor: [0, T) row of the staged tile; [T, T + E) old carry entry;
// 0xFFFF nothing (phantom row at a chunk head / unused carry entry).
// ---------------------------------------------------------------------------
constexpr int kSwcMaxCols = 8;             // payload columns per launch (carry buffers in smem)
constexpr uint32_t kSwcMaxNum = 256;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// Relaxed arrive: releasing a ring stage does not have to order this warp's global stores.
// The stage reads are ordered by issue: the arrive is issued after the instructions that
// consume the LDS results.
__device__ __forceinline__ void mbar_arrive_relaxed(uint32_t bar) {
  asm volatile("mbarrier.arrive.relaxed.cta.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "FB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra FB_DONE;\n"
      "bra FB_WAIT;\n"
      "FB_DONE:\n"
      "}\n" ::"r"(bar), "r"(parity)
      : "memory");
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
// 1-D bulk copy global -> shared, completion signalled on an mbarrier (TMA engine; SASS: UBLKCP)
__device__ __forceinline__ void tma_load_1d(uint32_t dst_smem, const void* src, uint32_t bytes, uint32_t bar,
                                            uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
      ::"r"(dst_smem), "l"(src), "r"(bytes), "r"(bar), "l"(policy)
      : "memory");
}

// ---------------------------------------------------------------------------
// pass 2, fast path v5: warp-specialised scatter (producer / rankers / movers).
//
// Measured on v4 (profiles/r1_notes.md): one third of the kernel is the per-tile ranking
// (hash, match, scans), during which no byte moves; the column phase itself runs near the HBM
// peak.  Here the two run concurrently on different warps of the same persistent CTA:
//   warp 24      producer : TMA bulk loads - the rank record of tile t+1 (partition id, rank and
//                           per-partition counts, written by pass 1: nothing is hashed, matched or
//                           counted here and ANY key shape takes this path) and the payload column
//                           tiles of tile t into the ring
//   warps 16-23  rankers  : place tile t+1: advance the write-combining state of every partition,
//                           build the slot list of the tile
//   warps 0-15   movers   : tile t: per column gather from the staged tile / carry, store whole
//                           sector groups, save the new carry (in place: the per-column barrier
//                           separates the reads of the old carry from the writes of the new one)
// Hand-off through mbarriers: slots_ready (rankers -> movers), slots_free (movers -> rankers, as
// soon as the slot list sits in mover registers), flush_done at chunk ends, full/empty per ring
// stage and per pid buffer.
// Shared memory (one CTA per SM), T = 4096, E = num * (G - 1):
//   ring[S][T] u64 | mbarriers | carry[ncols][E] u64 | slotinfo[T+E] u32 | wpos kcnt binfo
//   bin_n wstart wdelta [nbp] u32 | scanw[64] | carryinfo[E] u16 | rank records [2][12800 B]
// ---------------------------------------------------------------------------
constexpr int kWsMoverWarps = 16, kWsRankWarps = 8;
constexpr int kWsMovers = kWsMoverWarps * 32, kWsRankers = kWsRankWarps * 32;
constexpr int kWsThreads = kWsMovers + kWsRankers + 128;  // + producer warpgroup (1 active warp)
constexpr int kWsG = 4;  // rows per write-combined group (32 B); 8 (64 B) measured 4.1-5.0 ms vs 3.09: spills, 3 ring stages
constexpr int kWsRankItems = 16;  // rows per ranker thread per tile: tile = 256 x 16 = 4096 rows (2048: no faster)

struct WsUnits {
  const uint64_t* src[kSwcMaxCols];
  uint64_t* dst[kSwcMaxCols];
  int32_t nunits;
};

// K4, the fused map epilogue: output unit u is not a copy of src[u] but an affine function of one or
// two staged input tiles, computed by the movers right after the gather and before the store:
//   mode 1 (float64): (a * x + b * y) + c, every operation rounded on its own (no FMA contraction), i.e.
//                     exactly what the expression evaluator (K8) gives for `x * a + y * b + c`
//   mode 2 (int64)  : a * x + b * y + c  (wrapping)
// src2 == nullptr: y does not exist (b ignored).  A two-operand unit occupies two ring stages.
struct WsMap {
  const uint64_t* src2[kSwcMaxCols];
  uint64_t a[kSwcMaxCols], b[kSwcMaxCols], c[kSwcMaxCols];
  int32_t mode[kSwcMaxCols];
};

__device__ __forceinline__ uint64_t ws_apply_map(int mode, bool two, uint64_t x, uint64_t y, uint64_t a, uint64_t b,
                                                 uint64_t c) {
  if (mode == 1) {
    double r = __dmul_rn(__longlong_as_double((long long)a), __longlong_as_double((long long)x));
    if (two) r = __dadd_rn(r, __dmul_rn(__longlong_as_double((long long)b), __longlong_as_double((long long)y)));
    return (uint64_t)__double_as_longlong(__dadd_rn(r, __longlong_as_double((long long)c)));
  }
  if (mode == 2) return a * x + (two ? b * y : 0ULL) + c;
  return x;
}

template <int G, int RI>
__host__ __device__ inline size_t ws_book_bytes(uint32_t num, int ncols) {
  constexpr size_t kT = (size_t)kWsRankers * RI;
  const size_t nbp = nb_padded(num);
  const size_t E = (size_t)num * (G - 1);
  size_t b = 64 * 8;                           // mbarriers
  b += (size_t)ncols * E * 8;                  // carry buffers (in place)
  b += (kT + E) * 4;                           // slotinfo
  b += 6 * nbp * 4 + 64 * 4;                   // per-partition arrays + scanw
  b += ((E * 2 + 15) / 16) * 16;               // carryinfo
  b += 2 * (size_t)kMetaBytes + 128;           // rank records (+ alignment slack)
  return b;
}

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {  // release.cta: publishes prior smem writes
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mover_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kWsMovers) : "memory"); }
__device__ __forceinline__ void ranker_sync() { asm volatile("bar.sync 2, %0;" ::"n"(kWsRankers) : "memory"); }

template <int kBits, int G, int kWsRankItems, bool kMap>
__global__ void __launch_bounds__(kWsThreads, 1)
fb_scatter_ws_kernel(WsUnits units, uint32_t num, ChunkGeom g, int nstages,
                     const uint8_t* __restrict__ meta,
                     const uint32_t* __restrict__ chunk_base, const int64_t* __restrict__ part_offsets,
                     const __grid_constant__ WsMap map) {
  constexpr uint32_t T = (uint32_t)kWsRankers * kWsRankItems;  // rows per tile
  static_assert(T == (uint32_t)kTile, "pass 1 ranks tiles of kTile rows");
  constexpr uint32_t GM = G - 1;
  constexpr uint32_t kStageBytes = T * 8;
  constexpr int kSlotRounds = ((int)T + (int)kSwcMaxNum * (G - 1) + kWsMovers - 1) / kWsMovers;
  constexpr int kEntryRoundsM = ((int)kSwcMaxNum * (G - 1) + kWsMovers - 1) / kWsMovers;
  constexpr int kEntryRoundsR = ((int)kSwcMaxNum * (G - 1) + kWsRankers - 1) / kWsRankers;
  extern __shared__ __align__(128) uint64_t smem64[];
  const uint32_t nbp = nb_padded(num);
  const uint32_t E = num * GM;
  const int ncols = units.nunits;
  uint64_t* ring = smem64;
  uint64_t* bars = ring + (size_t)nstages * T;
  uint64_t* carry = bars + 64;
  uint32_t* slotinfo = (uint32_t*)(carry + (size_t)ncols * E);
  uint32_t* wpos = slotinfo + T + E;
  uint32_t* kcnt = wpos + nbp;
  uint32_t* binfo = kcnt + nbp;
  uint32_t* bin_n = binfo + nbp;
  uint32_t* wstart = bin_n + nbp;
  uint32_t* wdelta = wstart + nbp;
  uint32_t* scanw = wdelta + nbp;  // [8,16) written per ranker warp, [40] W
  uint16_t* carryinfo = (uint16_t*)(scanw + 64);
  uint8_t* metabuf = (uint8_t*)(((uintptr_t)(carryinfo + E) + 127) & ~(uintptr_t)127);  // TMA dst

  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t bar_full = smem_u32(bars), bar_empty = smem_u32(bars + 16);
  const uint32_t bar_pid_full = smem_u32(bars + 32), bar_pid_empty = smem_u32(bars + 34);
  const uint32_t bar_slots_ready = smem_u32(bars + 36), bar_slots_free = smem_u32(bars + 37);
  const uint32_t bar_flush_done = smem_u32(bars + 38);
  // per column step: "all movers have read the old carry".  Two barriers used alternately: the wait
  // for step k happens during step k+1, after this warp's arrival for step k+1, so a single barrier
  // could run two phases ahead of a pending parity wait (deadlock); with two, at most one.
  const uint32_t bar_carry_read = smem_u32(bars + 40);

  if (threadIdx.x == 0) {
    for (int s = 0; s < nstages; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, kWsMoverWarps);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar_pid_full + 8 * i, 1);
      mbar_init(bar_pid_empty + 8 * i, kWsRankWarps);
    }
    mbar_init(bar_slots_ready, kWsRankWarps);
    mbar_init(bar_slots_free, kWsMoverWarps);
    mbar_init(bar_flush_done, kWsMoverWarps);
    mbar_init(bar_carry_read, kWsMoverWarps);
    mbar_init(bar_carry_read + 8, kWsMoverWarps);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (warp >= kWsMoverWarps + kWsRankWarps) {
    // ============================ producer =============================================
    if (warp == kWsMoverWarps + kWsRankWarps && lane == 0) {
      const uint64_t pol = l2_policy_evict_first();
      const uint32_t ring_s = smem_u32(ring), meta_s = smem_u32(metabuf);
      uint32_t s = 0, ph = 0, seq = 0;
      // pids of the very first tile
      int chunk = (int)blockIdx.x;
      int64_t r0 = 0, r1 = 0, t0 = 0;
      bool have = chunk < g.nchunks_full;
      if (have) { chunk_range(g, chunk, r0, r1); t0 = r0; }
      auto load_pid = [&](int64_t row0, uint32_t q) {
        const uint32_t b = q & 1, pp = (q >> 1) & 1;
        mbar_wait(bar_pid_empty + 8 * b, pp ^ 1);
        mbar_expect_tx(bar_pid_full + 8 * b, kMetaBytes);
        tma_load_1d(meta_s + b * kMetaBytes, meta + (size_t)(row0 / T) * kMetaBytes, kMetaBytes,
                    bar_pid_full + 8 * b, pol);
      };
      if (have) load_pid(t0, 0);
      while (have) {
        // next tile of this CTA's sequence (for the pid look-ahead)
        int nchunk = chunk;
        int64_t nr0 = r0, nr1 = r1, nt0 = t0 + T;
        bool nhave = true;
        if (nt0 >= r1) {
          nchunk = chunk + (int)gridDim.x;
          nhave = nchunk < g.nchunks_full;
          if (nhave) { chunk_range(g, nchunk, nr0, nr1); nt0 = nr0; }
        }
        if (nhave) load_pid(nt0, seq + 1);
        for (int u = 0; u < ncols; ++u) {
          mbar_wait(bar_empty + 8 * s, ph ^ 1);
          mbar_expect_tx(bar_full + 8 * s, kStageBytes);
          tma_load_1d(ring_s + s * kStageBytes, units.src[u] + t0, kStageBytes, bar_full + 8 * s, pol);
          if (++s == (uint32_t)nstages) { s = 0; ph ^= 1; }
          if constexpr (kMap) {
            if (map.src2[u] != nullptr) {  // second operand of a fused map: the next stage
              mbar_wait(bar_empty + 8 * s, ph ^ 1);
              mbar_expect_tx(bar_full + 8 * s, kStageBytes);
              tma_load_1d(ring_s + s * kStageBytes, map.src2[u] + t0, kStageBytes, bar_full + 8 * s, pol);
              if (++s == (uint32_t)nstages) { s = 0; ph ^= 1; }
            }
          }
        }
        chunk = nchunk; r0 = nr0; r1 = nr1; t0 = nt0; have = nhave;
        ++seq;
      }
    }
    return;
  }

  if (warp >= kWsMoverWarps) {
    // ============================ rankers (8 warps) ====================================
    const unsigned rw = warp - kWsMoverWarps;          // ranker warp 0..7
    const unsigned rtid = threadIdx.x - kWsMovers;     // 0..255
    uint32_t seq = 0, cseq = 0;
    for (int chunk = (int)blockIdx.x; chunk < g.nchunks_full; chunk += (int)gridDim.x, ++cseq) {
      int64_t r0, r1;
      chunk_range(g, chunk, r0, r1);
      if (cseq > 0) mbar_wait(bar_flush_done, (cseq - 1) & 1);  // movers flushed the previous chunk
      ranker_sync();
      for (uint32_t b = rtid; b < nbp; b += kWsRankers) {
        const uint32_t p0 = b < num ? (uint32_t)part_offsets[b] + chunk_base[(size_t)chunk * num + b] : 0u;
        wpos[b] = p0 & ~GM;
        kcnt[b] = (p0 & GM) | ((p0 & GM) << 8);
      }
      ranker_sync();
      for (int64_t t0 = r0; t0 < r1; t0 += T, ++seq) {
        const uint32_t pb = seq & 1, pph = (seq >> 1) & 1;
        mbar_wait(bar_pid_full + 8 * pb, pph);
        const uint8_t* __restrict__ rec = metabuf + pb * kMetaBytes;
        // rows of this thread: r * 256 + rtid; packed (partition id << 16) | rank in tile
        uint32_t pr[kWsRankItems];
#pragma unroll
        for (int r = 0; r < kWsRankItems; ++r) {
          const uint32_t row = r * kWsRankers + rtid;
          pr[r] = ((uint32_t)rec[row] << 16) | ((const uint16_t*)(rec + kMetaRank))[row];
        }
        // ---- per partition (thread b < num): tile count, rows to write, new pending state
        const uint32_t b = rtid;
        uint32_t n = 0, w = 0, kold = 0, phold = 0, wp_old = 0;
        if (b < num) n = ((const uint16_t*)(rec + kMetaCnt))[b];
        __syncwarp();
        if (lane == 0) mbar_arrive_relaxed(bar_pid_empty + 8 * pb);  // the record is in registers
        if (b < num) {
          const uint32_t kc = kcnt[b];
          kold = kc & 0xFFu;
          phold = kc >> 8;
          wp_old = wpos[b];
          const uint32_t end = wp_old + kold + n;
          const uint32_t aend = end & ~GM;
          if (aend > wp_old) {
            w = aend - wp_old;
            wpos[b] = aend;
            kcnt[b] = end - aend;  // phantoms are consumed by the first write
          } else {
            kcnt[b] = (kold + n) | (phold << 8);
          }
          binfo[b] = kold | (phold << 4) | (w << 8);
          bin_n[b] = n;
        }
        uint32_t xw = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const uint32_t yw = __shfl_up_sync(0xFFFFFFFFu, xw, o);
          if (lane >= (unsigned)o) xw += yw;
        }
        if (lane == 31) scanw[8 + rw] = xw;
        ranker_sync();  // B
        uint32_t bw = xw - w;
        {
          const uint32_t tw = lane < kWsRankWarps ? scanw[8 + lane] : 0;
#pragma unroll
          for (int wi = 0; wi < kWsRankWarps; ++wi) {
            const uint32_t vw = __shfl_sync(0xFFFFFFFFu, tw, wi);
            if ((unsigned)wi < rw) bw += vw;
          }
        }
        // ---- hand-off arrays may be rewritten once the movers hold the previous slot list
        if (seq > 0) mbar_wait(bar_slots_free, (seq - 1) & 1);
        if (b < num) {
          wstart[b] = bw;
          wdelta[b] = wp_old - bw;  // slot j lands at output row wdelta + j
        }
        if (rtid == kWsRankers - 1) scanw[40] = bw + w;  // W: slots to store this tile
        ranker_sync();  // C
        // ---- every new row / old carry entry finds its place
#pragma unroll
        for (int r = 0; r < kWsRankItems; ++r) {
          const uint32_t pb2 = pr[r] >> 16;
          const uint32_t bi = binfo[pb2];
          const uint32_t i = (bi & 0xFu) + (pr[r] & 0xFFFFu);
          const uint32_t ww = bi >> 8;
          const uint32_t row = r * kWsRankers + rtid;
          if (i < ww) slotinfo[wstart[pb2] + i] = (pb2 << 16) | row;
          else carryinfo[pb2 * GM + (i - ww)] = (uint16_t)row;
        }
#pragma unroll
        for (int q = 0; q < kEntryRoundsR; ++q) {
          const uint32_t e = q * kWsRankers + rtid;
          if (e < E) {
            const uint32_t eb = e / GM, i = e - eb * GM;
            const uint32_t bi = binfo[eb];
            const uint32_t ko = bi & 0xFu, po = (bi >> 4) & 0xFu, ww = bi >> 8;
            const uint32_t nn = bin_n[eb];
            const uint32_t desc = i < po ? 0xFFFFu : T + e;
            if (i < ko) {
              if (i < ww) slotinfo[wstart[eb] + i] = (eb << 16) | desc;
              else carryinfo[e] = (uint16_t)desc;
            }
            if (ww + i >= ko + nn) carryinfo[e] = 0xFFFFu;
          }
        }
        ranker_sync();  // D: the slot list of this tile is complete
        if (lane == 0) mbar_arrive(bar_slots_ready);
      }
    }
    return;
  }

  // ================================ movers (16 warps) ====================================
  uint32_t s = 0, ph = 0, seq = 0, astep = 0, wstep = 0;
  for (int chunk = (int)blockIdx.x; chunk < g.nchunks_full; chunk += (int)gridDim.x) {
    int64_t r0, r1;
    chunk_range(g, chunk, r0, r1);
    for (int64_t t0 = r0; t0 < r1; t0 += T, ++seq) {
      mbar_wait(bar_slots_ready, seq & 1);
      const uint32_t W = scanw[40];
      uint32_t srcd[kSlotRounds], dst[kSlotRounds];
#pragma unroll
      for (int k = 0; k < kSlotRounds; ++k) {
        const uint32_t j = k * kWsMovers + threadIdx.x;
        srcd[k] = 0xFFFFu;
        dst[k] = 0;
        if (j < W) {
          const uint32_t info = slotinfo[j];
          srcd[k] = info & 0xFFFFu;
          dst[k] = wdelta[info >> 16] + j;
        }
      }
      uint32_t csrc[kEntryRoundsM];
#pragma unroll
      for (int q = 0; q < kEntryRoundsM; ++q) {
        const uint32_t e = q * kWsMovers + threadIdx.x;
        csrc[q] = e < E ? (uint32_t)carryinfo[e] : 0xFFFFu;
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_slots_free);  // the slot list sits in registers now

      // The new carry of column u is written one step late (while column u+1 moves): by then every
      // mover has long finished reading the old carry of column u, so nobody waits at a barrier.
      uint64_t cv_prev[kEntryRoundsM];
      for (int u = 0; u < ncols; ++u) {
        mbar_wait(bar_full + 8 * s, ph);
        const uint64_t* __restrict__ st = ring + (size_t)s * T;
        uint64_t* __restrict__ out = units.dst[u];
        const uint64_t* __restrict__ cbuf = carry + (size_t)u * E;
        uint64_t v[kSlotRounds], cv[kEntryRoundsM];
        uint32_t s2 = s;
        bool two = false;
        if constexpr (kMap) {
          // fused map (K4): rows taken from the staged tile(s) are mapped here; carry entries already are
          // output values
          const int mode = map.mode[u];
          two = map.src2[u] != nullptr;
          const uint64_t* __restrict__ st2 = st;
          if (two) {
            s2 = s + 1 == (uint32_t)nstages ? 0 : s + 1;
            mbar_wait(bar_full + 8 * s2, s2 == 0 ? ph ^ 1 : ph);
            st2 = ring + (size_t)s2 * T;
          }
          const uint64_t ma = map.a[u], mb = map.b[u], mc = map.c[u];
#pragma unroll
          for (int k = 0; k < kSlotRounds; ++k)
            if (srcd[k] != 0xFFFFu)
              v[k] = srcd[k] < T ? ws_apply_map(mode, two, st[srcd[k]], st2[srcd[k]], ma, mb, mc) : cbuf[srcd[k] - T];
#pragma unroll
          for (int q = 0; q < kEntryRoundsM; ++q)
            if (csrc[q] != 0xFFFFu)
              cv[q] = csrc[q] < T ? ws_apply_map(mode, two, st[csrc[q]], st2[csrc[q]], ma, mb, mc) : cbuf[csrc[q] - T];
        } else {
#pragma unroll
          for (int k = 0; k < kSlotRounds; ++k)
            if (srcd[k] != 0xFFFFu) v[k] = srcd[k] < T ? st[srcd[k]] : cbuf[srcd[k] - T];
#pragma unroll
          for (int q = 0; q < kEntryRoundsM; ++q)
            if (csrc[q] != 0xFFFFu) cv[q] = csrc[q] < T ? st[csrc[q]] : cbuf[csrc[q] - T];
        }
#pragma unroll
        for (int k = 0; k < kSlotRounds; ++k)
          if (srcd[k] != 0xFFFFu) out[dst[k]] = v[k];
        // all my reads of the stage and of the old carry have completed (their values were
        // consumed by the stores above / are in cv): release the stage, publish "carry read"
        __syncwarp();
        if (lane == 0) {
          mbar_arrive_relaxed(bar_empty + 8 * s);
          if (kMap && two) mbar_arrive_relaxed(bar_empty + 8 * s2);
          mbar_arrive_relaxed(bar_carry_read + 8 * (astep & 1));
        }
        ++astep;
        if (++s == (uint32_t)nstages) { s = 0; ph ^= 1; }
        if (kMap && two) {
          if (++s == (uint32_t)nstages) { s = 0; ph ^= 1; }
        }
        if (u > 0) {  // write the previous column's new carry
          mbar_wait(bar_carry_read + 8 * (wstep & 1), (wstep >> 1) & 1);
          ++wstep;
          uint64_t* __restrict__ pbuf = carry + (size_t)(u - 1) * E;
#pragma unroll
          for (int q = 0; q < kEntryRoundsM; ++q) {
            const uint32_t e = q * kWsMovers + threadIdx.x;
            if (csrc[q] != 0xFFFFu) pbuf[e] = cv_prev[q];
          }
        }
#pragma unroll
        for (int q = 0; q < kEntryRoundsM; ++q) cv_prev[q] = cv[q];
      }
      {  // the last column's new carry
        mbar_wait(bar_carry_read + 8 * (wstep & 1), (wstep >> 1) & 1);
        ++wstep;
        uint64_t* __restrict__ pbuf = carry + (size_t)(ncols - 1) * E;
#pragma unroll
        for (int q = 0; q < kEntryRoundsM; ++q) {
          const uint32_t e = q * kWsMovers + threadIdx.x;
          if (csrc[q] != 0xFFFFu) pbuf[e] = cv_prev[q];
        }
      }
    }
    // ---- chunk end: flush the pending rows (partial sector groups)
    mover_sync();
    for (int u = 0; u < ncols; ++u) {
      uint64_t* __restrict__ out = units.dst[u];
      const uint64_t* __restrict__ cbuf = carry + (size_t)u * E;
#pragma unroll
      for (int q = 0; q < kEntryRoundsM; ++q) {
        const uint32_t e = q * kWsMovers + threadIdx.x;
        if (e < E) {
          const uint32_t b = e / GM, i = e - b * GM;
          const uint32_t kc = kcnt[b];
          if (i < (kc & 0xFFu) && i >= (kc >> 8)) out[wpos[b] + i] = cbuf[e];
        }
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(bar_flush_done);  // rankers may start the next chunk
  }
}

// ---------------------------------------------------------------------------
// validity bitmap <-> byte mask
// ---------------------------------------------------------------------------
__global__ void fb_bits_to_bytes_kernel(const uint8_t* __restrict__ bits, int64_t bit_offset,
                                        int64_t nrows, uint8_t* __restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < nrows; i += stride) {
    int64_t j = i + bit_offset;
    out[i] = (bits[j >> 3] >> (j & 7)) & 1;
  }
}

__global__ void fb_bytes_to_bits_kernel(const uint8_t* __restrict__ bytes, int64_t nrows,
                                        uint8_t* __restrict__ out, unsigned long long* null_count) {
  // one thread per output byte
  int64_t nbytes = (nrows + 7) >> 3;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  unsigned long long nulls = 0;
  for (; i < nbytes; i += stride) {
    uint8_t v = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      int64_t r = i * 8 + k;
      if (r < nrows) {
        if (bytes[r]) v |= (uint8_t)(1u << k);
        else ++nulls;
      }
    }
    out[i] = v;
  }
  if (null_count != nullptr && nulls) atomicAdd(null_count, nulls);
}

inline int bits_for(uint32_t num) { return num <= 16 ? 4 : (num <= 256 ? 8 : 10); }

#define FB_DISPATCH_SB(single, bits, LAUNCH)                 \
  do {                                                       \
    if (single) {                                            \
      if (bits == 4) LAUNCH(true, 4);                        \
      else if (bits == 8) LAUNCH(true, 8);                   \
      else LAUNCH(true, 10);                                 \
    } else {                                                 \
      if (bits == 4) LAUNCH(false, 4);                       \
      else if (bits == 8) LAUNCH(false, 8);                  \
      else LAUNCH(false, 10);                                \
    }                                                        \
  } while (0)

template <typename K>
cudaError_t optin(K kernel, size_t bytes) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

// opt in to > 48 KB of dynamic shared memory, once per device
cudaError_t ensure_smem_optin(int dev) {
  static std::mutex mu;
  static uint64_t done = 0;
  std::lock_guard<std::mutex> lock(mu);
  if (dev >= 0 && dev < 64 && (done >> dev) & 1) return cudaSuccess;
  const size_t sc = scatter_smem_bytes(FB_MAX_PARTITIONS);
  const size_t hs = (size_t)kHistWarps * FB_MAX_PARTITIONS * sizeof(uint32_t);
  cudaError_t e = cudaSuccess;
#define FB_OPTIN(S, B)                                                   \
  do {                                                                   \
    if (e == cudaSuccess) e = optin(fb_scatter_kernel<S, B, true>, sc);  \
    if (e == cudaSuccess) e = optin(fb_scatter_kernel<S, B, false>, sc); \
    if (e == cudaSuccess) e = optin(fb_hist_kernel<S, B>, hs);           \
  } while (0)
  {
    int smem_max = 0;
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (e == cudaSuccess) e = optin(fb_scatter_ws_kernel<4, kWsG, kWsRankItems, false>, (size_t)smem_max);
    if (e == cudaSuccess) e = optin(fb_scatter_ws_kernel<8, kWsG, kWsRankItems, false>, (size_t)smem_max);
    if (e == cudaSuccess) e = optin(fb_scatter_ws_kernel<4, kWsG, kWsRankItems, true>, (size_t)smem_max);
    if (e == cudaSuccess) e = optin(fb_scatter_ws_kernel<8, kWsG, kWsRankItems, true>, (size_t)smem_max);
  }
  FB_OPTIN(true, 4); FB_OPTIN(true, 8); FB_OPTIN(true, 10);
  FB_OPTIN(false, 4); FB_OPTIN(false, 8); FB_OPTIN(false, 10);
#undef FB_OPTIN
  if (e == cudaSuccess && dev >= 0 && dev < 64) done |= (1ull << dev);
  return e;
}

bool single_u64_key(int nkeys, const int32_t* widths, const uint8_t* const* valid) {
  return nkeys == 1 && widths[0] == 8 && (valid == nullptr || valid[0] == nullptr);
}

int fill_keys(FbKeys& k, int nkeys, const void* const* ptrs, const int32_t* widths,
              const uint8_t* const* valid) {
  FB_CHECK(nkeys >= 1 && nkeys <= FB_MAX_KEYS, "nkeys=%d out of range [1,%d]", nkeys, FB_MAX_KEYS);
  memset(&k, 0, sizeof(k));
  k.nkeys = nkeys;
  k.digit_shift = -1;
  for (int i = 0; i < nkeys; ++i) {
    FB_CHECK(widths[i] == 1 || widths[i] == 2 || widths[i] == 4 || widths[i] == 8,
             "key %d has unsupported width %d", i, widths[i]);
    FB_CHECK(ptrs[i] != nullptr, "key %d pointer is NULL", i);
    k.ptr[i] = ptrs[i];
    k.width[i] = widths[i];
    k.valid[i] = valid ? valid[i] : nullptr;
  }
  return 0;
}

struct PlanLayout {
  size_t hist_bytes;     // uint32 [nchunks][num]
  size_t pid_offset;     // rank records, kMetaBytes per full tile (num <= 256), 256-byte aligned
  size_t total_bytes;
};

PlanLayout plan_layout(const ChunkGeom& g, uint32_t num) {
  PlanLayout l;
  l.hist_bytes = (((size_t)g.nchunks * num * sizeof(uint32_t)) + 255) & ~(size_t)255;
  l.pid_offset = l.hist_bytes + 256;
  l.total_bytes = l.pid_offset + (num <= kSwcMaxNum ? (size_t)(g.full_rows / kTile) * kMetaBytes : 0) + 256;
  return l;
}

}  // namespace

extern "C" {

size_t fb_partition_scratch_bytes(int dev, int64_t nrows, uint32_t num_partitions) {
  if (nrows < 0 || num_partitions == 0) return 0;
  ChunkGeom g = make_geom(dev, nrows);
  return plan_layout(g, num_partitions).total_bytes;
}

int fb_partition_ids(int dev, void* stream, int64_t nrows, int nkeys, const void* const* key_ptrs,
                     const int32_t* key_widths, const uint8_t* const* key_valid,
                     uint32_t num_partitions, uint32_t* out_pids) {
  FB_CHECK(nrows >= 0, "nrows < 0");
  FB_CHECK(num_partitions >= 1, "num_partitions must be >= 1");
  if (nrows == 0) return 0;
  FbDeviceGuard guard(dev);
  FB_CHECK(guard.ok, "cannot select device %d", dev);
  FbKeys k;
  if (int rc = fill_keys(k, nkeys, key_ptrs, key_widths, key_valid)) return rc;
  FbDiv dv = fb_make_div(num_partitions);
  int64_t blocks = (nrows + 255) / 256;
  int64_t maxb = (int64_t)fb_sm_count(dev) * 16;
  if (blocks > maxb) blocks = maxb;
  cudaStream_t st = (cudaStream_t)stream;
  if (single_u64_key(nkeys, key_widths, key_valid))
    fb_pid_kernel<true><<<(unsigned)blocks, 256, 0, st>>>(k, dv, nrows, out_pids);
  else
    fb_pid_kernel<false><<<(unsigned)blocks, 256, 0, st>>>(k, dv, nrows, out_pids);
  FB_CUDA(cudaGetLastError());
  return 0;
}

int fb_row_hash64(int dev, void* stream, int64_t nrows, int nkeys, const void* const* key_ptrs,
                  const int32_t* key_widths, const uint8_t* const* key_valid, uint64_t* out_hash) {
  FB_CHECK(nrows >= 0, "nrows < 0");
  if (nrows == 0) return 0;
  FbDeviceGuard guard(dev);
  FB_CHECK(guard.ok, "cannot select device %d", dev);
  FbKeys k;
  if (int rc = fill_keys(k, nkeys, key_ptrs, key_widths, key_valid)) return rc;
  int64_t blocks = (nrows + 255) / 256;
  int64_t maxb = (int64_t)fb_sm_count(dev) * 16;
  if (blocks > maxb) blocks = maxb;
  fb_row_hash_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(k, nrows, out_hash);
  FB_CUDA(cudaGetLastError());
  return 0;
}

static int plan_impl(int dev, void* stream, int64_t nrows, const FbKeys& k, bool single,
                     uint32_t num_partitions, void* scratch, size_t scratch_bytes,
                     int64_t* out_part_offsets) {
  FB_CHECK(nrows >= 0, "nrows < 0");
  FB_CHECK(nrows < ((int64_t)1 << 32), "nrows=%lld exceeds the 2^32-1 rows one call handles",
           (long long)nrows);
  FB_CHECK(num_partitions >= 1 && num_partitions <= FB_MAX_PARTITIONS,
           "num_partitions=%u out of range [1,%d]", num_partitions, FB_MAX_PARTITIONS);
  FB_CHECK(out_part_offsets != nullptr, "out_part_offsets is NULL");
  FbDeviceGuard guard(dev);
  FB_CHECK(guard.ok, "cannot select device %d", dev);
  cudaStream_t st = (cudaStream_t)stream;
  if (nrows == 0) {
    FB_CUDA(cudaMemsetAsync(out_part_offsets, 0, sizeof(int64_t) * ((size_t)num_partitions + 1), st));
    return 0;
  }
  ChunkGeom g = make_geom(dev, nrows);
  PlanLayout l = plan_layout(g, num_partitions);
  FB_CHECK(scratch != nullptr && scratch_bytes >= l.total_bytes,
           "scratch too small: need %zu bytes, got %zu", l.total_bytes, scratch_bytes);
  FB_CHECK((uintptr_t)scratch % 16 == 0, "scratch must be 16-byte aligned (rank records are stored in 16-byte words)");
  FbDiv dv = fb_make_div(num_partitions);
  uint32_t* hist = (uint32_t*)scratch;
  size_t smem = (size_t)kHistWarps * num_partitions * sizeof(uint32_t);
  FB_CUDA(ensure_smem_optin(dev));
  const int bits = bits_for(num_partitions);
  // num <= 256: full tiles are ranked completely (fb_rank_kernel); the tail chunk and larger
  // partition counts only need the histogram
  int hist_chunk0 = 0;
  if (num_partitions <= kSwcMaxNum && g.nchunks_full > 0) {
    uint8_t* meta = (uint8_t*)scratch + l.pid_offset;
    const bool pow2 = (num_partitions & (num_partitions - 1)) == 0;
#define FB_LAUNCH_RANK(S, B, P) \
  fb_rank_kernel<S, B, P><<<g.nchunks_full, kRankBlock, 0, st>>>(k, dv, num_partitions, g, hist, meta)
    if (single && pow2) {
      if (bits == 4) FB_LAUNCH_RANK(true, 4, true);
      else FB_LAUNCH_RANK(true, 8, true);
    } else if (single) {
      if (bits == 4) FB_LAUNCH_RANK(true, 4, false);
      else FB_LAUNCH_RANK(true, 8, false);
    } else {
      if (bits == 4) FB_LAUNCH_RANK(false, 4, false);
      else FB_LAUNCH_RANK(false, 8, false);
    }
#undef FB_LAUNCH_RANK
    FB_CUDA(cudaGetLastError());
    hist_chunk0 = g.nchunks_full;
  }
  if (hist_chunk0 < g.nchunks) {
#define FB_LAUNCH_HIST(S, B)                                                                       \
  fb_hist_kernel<S, B><<<g.nchunks - hist_chunk0, kHistBlock, smem, st>>>(k, dv, num_partitions, g, \
                                                                          hist_chunk0, hist)
    FB_DISPATCH_SB(single, bits, FB_LAUNCH_HIST);
#undef FB_LAUNCH_HIST
    FB_CUDA(cudaGetLastError());
  }
  fb_scan_chunks_kernel<<<num_partitions, 256, 0, st>>>(hist, num_partitions, g.nchunks, out_part_offsets);
  FB_CUDA(cudaGetLastError());
  fb_scan_parts_kernel<<<1, 1024, 0, st>>>(out_part_offsets, num_partitions);
  FB_CUDA(cudaGetLastError());
  return 0;
}

int fb_partition_plan(int dev, void* stream, int64_t nrows, int nkeys, const void* const* key_ptrs,
                      const int32_t* key_widths, const uint8_t* const* key_valid,
                      uint32_t num_partitions, void* scratch, size_t scratch_bytes,
                      int64_t* out_part_offsets) {
  FbKeys k;
  if (nrows == 0) {  // empty tables have NULL column pointers: nothing to read, offsets are all zero
    memset(&k, 0, sizeof(k));
    k.nkeys = 1;
    k.digit_shift = -1;
    return plan_impl(dev, stream, 0, k, false, num_partitions, scratch, scratch_bytes, out_part_offsets);
  }
  if (int rc = fill_keys(k, nkeys, key_ptrs, key_widths, key_valid)) return rc;
  return plan_impl(dev, stream, nrows, k, single_u64_key(nkeys, key_widths, key_valid), num_partitions,
                   scratch, scratch_bytes, out_part_offsets);
}

// Rows of the partial tail tile of the mapped units, evaluated into tail_tmp[c][0 .. nrows - full_rows): the
// generic scatter kernel then moves them like any column.
__global__ void fb_map_tail_kernel(int ncols, const void* const* __restrict__ x_ptrs, const fb_map_unit* __restrict__ maps,
                                   int64_t row0, int64_t nrows, uint64_t* __restrict__ tmp) {
  const int64_t n = nrows - row0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n * ncols; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i / n);
    const int64_t r = row0 + i % n;
    const fb_map_unit m = maps[c];
    const uint64_t x = ((const uint64_t*)x_ptrs[c])[r];
    const uint64_t y = m.src2 != nullptr ? ((const uint64_t*)m.src2)[r] : 0;
    tmp[(size_t)c * kTile + (size_t)(i % n)] = ws_apply_map(m.mode, m.src2 != nullptr, x, y, m.a, m.b, m.c);
  }
}

static int apply_impl(int dev, void* stream, int64_t nrows, const FbKeys& k, bool single,
                      uint32_t num_partitions, const void* scratch, size_t scratch_bytes,
                      const int64_t* part_offsets, int ncols, const void* const* col_ptrs,
                      const int32_t* col_widths, void* const* out_col_ptrs, int sm_reserve = 0,
                      const fb_map_unit* maps = nullptr, void* tail_tmp = nullptr, int cols_per_launch_req = 0) {
  FB_CHECK(nrows >= 0 && nrows < ((int64_t)1 << 32), "nrows out of range");
  FB_CHECK(num_partitions >= 1 && num_partitions <= FB_MAX_PARTITIONS,
           "num_partitions=%u out of range [1,%d]", num_partitions, FB_MAX_PARTITIONS);
  FB_CHECK(ncols >= 0, "ncols < 0");
  if (nrows == 0 || ncols == 0) return 0;
  FbDeviceGuard guard(dev);
  FB_CHECK(guard.ok, "cannot select device %d", dev);
  ChunkGeom g = make_geom(dev, nrows);
  PlanLayout l = plan_layout(g, num_partitions);
  FB_CHECK(scratch != nullptr && scratch_bytes >= l.total_bytes, "scratch too small");
  FbDiv dv = fb_make_div(num_partitions);
  cudaStream_t st = (cudaStream_t)stream;
  const size_t smem = scatter_smem_bytes(num_partitions);
  FB_CUDA(ensure_smem_optin(dev));
  const int bits = bits_for(num_partitions);

  for (int c = 0; c < ncols; ++c) {
    const int w = col_widths[c];
    FB_CHECK(w == 1 || w == 2 || w == 4 || w == 8, "column %d has unsupported width %d", c, w);
    FB_CHECK(col_ptrs[c] != nullptr && out_col_ptrs[c] != nullptr, "column %d pointer is NULL", c);
  }

  // generic kernel over chunks [chunk0, chunk0 + nch) for the columns listed in idx[0..n)
  const void* const* gen_src = col_ptrs;
  auto launch_generic = [&](const int* idx, int n, int chunk0, int nch) -> int {
    for (int c0 = 0; c0 < n && nch > 0; c0 += FB_MAX_COLS) {
      FbCols cols;
      memset(&cols, 0, sizeof(cols));
      cols.ncols = n - c0 < FB_MAX_COLS ? n - c0 : FB_MAX_COLS;
      bool all8 = true;
      for (int c = 0; c < cols.ncols; ++c) {
        cols.src[c] = gen_src[idx[c0 + c]];
        cols.dst[c] = out_col_ptrs[idx[c0 + c]];
        cols.width[c] = col_widths[idx[c0 + c]];
        all8 = all8 && cols.width[c] == 8;
      }
#define FB_LAUNCH_SCATTER(S, B)                                                                        \
  do {                                                                                                 \
    if (all8)                                                                                          \
      fb_scatter_kernel<S, B, true><<<nch, kBlock, smem, st>>>(k, dv, num_partitions, g, chunk0,       \
                                                               (const uint32_t*)scratch, part_offsets, cols); \
    else                                                                                               \
      fb_scatter_kernel<S, B, false><<<nch, kBlock, smem, st>>>(k, dv, num_partitions, g, chunk0,      \
                                                                (const uint32_t*)scratch, part_offsets, cols); \
  } while (0)
      FB_DISPATCH_SB(single, bits, FB_LAUNCH_SCATTER);
#undef FB_LAUNCH_SCATTER
      FB_CUDA(cudaGetLastError());
    }
    return 0;
  };

  // ---- split the columns: fast path (warp-specialised TMA ring + write combining; reads the rank
  //      records written by pass 1, so any key shape qualifies) vs generic.  8-byte columns, num <= 256.
  const bool fast_ok = num_partitions <= kSwcMaxNum && g.nchunks_full > 0;
  if (maps != nullptr) {  // fused map epilogue (K4): every unit must qualify for the fast kernel
    FB_CHECK(num_partitions <= kSwcMaxNum, "fused map needs num_partitions <= %u", kSwcMaxNum);
    FB_CHECK(tail_tmp != nullptr || g.full_rows == nrows, "fused map: tail_tmp is NULL");
    for (int c = 0; c < ncols; ++c) {
      FB_CHECK(col_widths[c] == 8 && (uintptr_t)col_ptrs[c] % 16 == 0, "fused map: column %d is not an aligned 8-byte column", c);
      FB_CHECK(maps[c].mode >= 0 && maps[c].mode <= 2, "fused map: column %d has mode %d", c, maps[c].mode);
      FB_CHECK(maps[c].src2 == nullptr || (maps[c].mode != 0 && (uintptr_t)maps[c].src2 % 16 == 0),
               "fused map: bad second operand of column %d", c);
    }
  }
  int* fast_idx = (int*)alloca(sizeof(int) * (size_t)ncols);
  int* gen_idx = (int*)alloca(sizeof(int) * (size_t)ncols);
  int nfast = 0, ngen = 0;
  for (int c = 0; c < ncols; ++c) {
    if (fast_ok && col_widths[c] == 8 && (uintptr_t)col_ptrs[c] % 16 == 0) fast_idx[nfast++] = c;
    else gen_idx[ngen++] = c;
  }
  if (int rc = launch_generic(gen_idx, ngen, 0, g.nchunks)) return rc;

  if (nfast > 0) {
    int smem_max = 0;
    FB_CUDA(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    int grid = fb_sm_count(dev) < g.nchunks_full ? fb_sm_count(dev) : g.nchunks_full;
    // sm_reserve: SMs left free for kernels that must co-run with this persistent one (the
    // multi-GPU barrier / pull kernels: a scatter CTA owns the whole register file of its SM)
    if (sm_reserve > 0 && grid > fb_sm_count(dev) - sm_reserve) grid = fb_sm_count(dev) - sm_reserve;
    if (grid < 1) grid = 1;
    const uint8_t* pid_plane = (const uint8_t*)scratch + l.pid_offset;  // rank records of pass 1
    // measured (100 M rows x 8 cols, columns per launch): 8 -> 3.45 ms, 4 -> 3.10, 3 -> 3.21, 2 -> 3.33,
    // 1 -> 4.59 (fewer open write streams: half-written lines meet their other half while still in L2;
    // a launch costs ~0.15 ms of ramp + rank-record traffic).  Groups of at most 4, evenly sized.
    const int ngroups = (nfast + 3) / 4;
    int cols_per_launch = (nfast + ngroups - 1) / ngroups;
    if (cols_per_launch_req >= 1 && cols_per_launch_req <= kSwcMaxCols) cols_per_launch = cols_per_launch_req;
    for (int c0 = 0; c0 < nfast; c0 += cols_per_launch) {
      const int nb = nfast - c0 < cols_per_launch ? nfast - c0 : cols_per_launch;
      WsUnits wu;
      memset(&wu, 0, sizeof(wu));
      wu.nunits = nb;
      for (int c = 0; c < nb; ++c) {
        wu.src[c] = (const uint64_t*)col_ptrs[fast_idx[c0 + c]];
        wu.dst[c] = (uint64_t*)out_col_ptrs[fast_idx[c0 + c]];
      }
      const size_t book = ws_book_bytes<kWsG, kWsRankItems>(num_partitions, nb);
      const size_t stage_bytes = (size_t)kWsRankers * kWsRankItems * 8;
      int nstages = (int)(((size_t)smem_max - book) / stage_bytes);
      if (nstages > 16) nstages = 16;
      FB_CHECK(nstages >= 2, "not enough shared memory for the TMA ring (%d stages)", nstages);
      const size_t tsmem = (size_t)nstages * stage_bytes + book;
      WsMap wm;
      memset(&wm, 0, sizeof(wm));
      if (maps != nullptr) {
        for (int c = 0; c < nb; ++c) {
          const fb_map_unit& m = maps[fast_idx[c0 + c]];
          wm.src2[c] = (const uint64_t*)m.src2;
          wm.a[c] = m.a; wm.b[c] = m.b; wm.c[c] = m.c;
          wm.mode[c] = m.mode;
        }
        if (bits == 4)
          fb_scatter_ws_kernel<4, kWsG, kWsRankItems, true><<<grid, kWsThreads, tsmem, st>>>(
              wu, num_partitions, g, nstages, pid_plane, (const uint32_t*)scratch, part_offsets, wm);
        else
          fb_scatter_ws_kernel<8, kWsG, kWsRankItems, true><<<grid, kWsThreads, tsmem, st>>>(
              wu, num_partitions, g, nstages, pid_plane, (const uint32_t*)scratch, part_offsets, wm);
      } else if (bits == 4) {
        fb_scatter_ws_kernel<4, kWsG, kWsRankItems, false><<<grid, kWsThreads, tsmem, st>>>(
            wu, num_partitions, g, nstages, pid_plane, (const uint32_t*)scratch, part_offsets, wm);
      } else {
        fb_scatter_ws_kernel<8, kWsG, kWsRankItems, false><<<grid, kWsThreads, tsmem, st>>>(
            wu, num_partitions, g, nstages, pid_plane, (const uint32_t*)scratch, part_offsets, wm);
      }
      FB_CUDA(cudaGetLastError());
    }
    // the partial tail tile of the fast columns
    if (maps == nullptr)
      if (int rc = launch_generic(fast_idx, nfast, g.nchunks_full, g.nchunks - g.nchunks_full)) return rc;
  }
  if (maps != nullptr && g.full_rows < nrows) {
    // fused map: the tail rows are mapped into tail_tmp (device arrays of pointers / descriptors live in
    // its first bytes) and the generic kernel reads them through shifted column bases
    FB_CHECK(ncols <= kSwcMaxCols * 8, "fused map: too many columns (%d)", ncols);
    uint8_t* base = (uint8_t*)tail_tmp;
    const size_t hdr = (((size_t)ncols * (sizeof(void*) + sizeof(fb_map_unit))) + 255) & ~(size_t)255;
    FB_CUDA(cudaMemcpyAsync(base, col_ptrs, sizeof(void*) * (size_t)ncols, cudaMemcpyHostToDevice, st));
    FB_CUDA(cudaMemcpyAsync(base + sizeof(void*) * (size_t)ncols, maps, sizeof(fb_map_unit) * (size_t)ncols,
                            cudaMemcpyHostToDevice, st));
    uint64_t* vals = (uint64_t*)(base + hdr);
    fb_map_tail_kernel<<<32, 256, 0, st>>>(ncols, (const void* const*)base,
                                           (const fb_map_unit*)(base + sizeof(void*) * (size_t)ncols), g.full_rows,
                                           nrows, vals);
    FB_CUDA(cudaGetLastError());
    const void** shifted = (const void**)alloca(sizeof(void*) * (size_t)ncols);
    int* all_idx = (int*)alloca(sizeof(int) * (size_t)ncols);
    for (int c = 0; c < ncols; ++c) {
      shifted[c] = (const uint8_t*)(vals + (size_t)c * kTile) - (size_t)g.full_rows * 8;
      all_idx[c] = c;
    }
    gen_src = shifted;
    if (int rc = launch_generic(all_idx, ncols, g.nchunks_full, g.nchunks - g.nchunks_full)) return rc;
  }
  return 0;
}

int fb_partition_apply(int dev, void* stream, int64_t nrows, int nkeys, const void* const* key_ptrs,
                       const int32_t* key_widths, const uint8_t* const* key_valid,
                       uint32_t num_partitions, const void* scratch, size_t scratch_bytes,
                       const int64_t* part_offsets, int ncols, const void* const* col_ptrs,
                       const int32_t* col_widths, void* const* out_col_ptrs) {
  if (nrows == 0 || ncols == 0) return 0;
  FbKeys k;
  if (int rc = fill_keys(k, nkeys, key_ptrs, key_widths, key_valid)) return rc;
  return apply_impl(dev, stream, nrows, k, single_u64_key(nkeys, key_widths, key_valid), num_partitions,
                    scratch, scratch_bytes, part_offsets, ncols, col_ptrs, col_widths, out_col_ptrs);
}

int fb_partition_apply_ex(int dev, void* stream, int64_t nrows, int nkeys, const void* const* key_ptrs,
                          const int32_t* key_widths, const uint8_t* const* key_valid,
                          uint32_t num_partitions, const void* scratch, size_t scratch_bytes,
                          const int64_t* part_offsets, int ncols, const void* const* col_ptrs,
                          const int32_t* col_widths, void* const* out_col_ptrs, int sm_reserve,
                          int cols_per_launch) {
  if (nrows == 0 || ncols == 0) return 0;
  FB_CHECK(sm_reserve >= 0, "sm_reserve < 0");
  FbKeys k;
  if (int rc = fill_keys(k, nkeys, key_ptrs, key_widths, key_valid)) return rc;
  return apply_impl(dev, stream, nrows, k, single_u64_key(nkeys, key_widths, key_valid), num_partitions,
                    scratch, scratch_bytes, part_offsets, ncols, col_ptrs, col_widths, out_col_ptrs, sm_reserve,
                    nullptr, nullptr, cols_per_launch);
}

size_t fb_partition_map_tail_bytes(int ncols) {
  if (ncols < 0) return 0;
  return ((((size_t)ncols * (sizeof(void*) + sizeof(fb_map_unit))) + 255) & ~(size_t)255) + (size_t)ncols * kTile * 8;
}

int fb_partition_apply_map(int dev, void* stream, int64_t nrows, int nkeys, const void* const* key_ptrs,
                           const int32_t* key_widths, const uint8_t* const* key_valid,
                           uint32_t num_partitions, const void* scratch, size_t scratch_bytes,
                           const int64_t* part_offsets, int ncols, const void* const* col_ptrs,
                           void* const* out_col_ptrs, const fb_map_unit* maps, void* tail_tmp, int sm_reserve) {
  if (nrows == 0 || ncols == 0) return 0;
  FB_CHECK(maps != nullptr, "maps is NULL");
  FB_CHECK(ncols <= FB_MAX_COLS, "ncols=%d > %d", ncols, FB_MAX_COLS);
  FbKeys k;
  if (int rc = fill_keys(k, nkeys, key_ptrs, key_widths, key_valid)) return rc;
  int32_t widths[FB_MAX_COLS];
  for (int c = 0; c < ncols; ++c) widths[c] = 8;
  return apply_impl(dev, stream, nrows, k, single_u64_key(nkeys, key_widths, key_valid), num_partitions,
                    scratch, scratch_bytes, part_offsets, ncols, col_ptrs, widths, out_col_ptrs, sm_reserve, maps,
                    tail_tmp);
}

int fb_radix_pass(int dev, void* stream, int64_t nrows, const void* sort_key_u64, int shift, int ncols,
                  const void* const* col_ptrs, const int32_t* col_widths, void* const* out_col_ptrs,
                  void* scratch, size_t scratch_bytes, int64_t* d_offsets /*257*/) {
  FB_CHECK(shift >= 0 && shift <= 56, "shift out of range");
  if (nrows == 0) return 0;
  const void* kp[1] = {sort_key_u64};
  const int32_t kw[1] = {8};
  FbKeys k;
  if (int rc = fill_keys(k, 1, kp, kw, nullptr)) return rc;
  k.digit_shift = shift;
  if (int rc = plan_impl(dev, stream, nrows, k, false, 256, scratch, scratch_bytes, d_offsets)) return rc;
  return apply_impl(dev, stream, nrows, k, false, 256, scratch, scratch_bytes, d_offsets, ncols, col_ptrs,
                    col_widths, out_col_ptrs);
}

int fb_partition_cols(int dev, void* stream, int64_t nrows, int ncols, const void* const* col_ptrs,
                      const int32_t* col_widths, const int32_t* key_col_idx, int nkeys,
                      const uint8_t* const* key_valid, uint32_t num_partitions,
                      void* const* out_col_ptrs, int64_t* out_part_offsets, void* scratch,
                      size_t scratch_bytes) {
  FB_CHECK(nkeys >= 1 && nkeys <= FB_MAX_KEYS, "nkeys=%d out of range [1,%d]", nkeys, FB_MAX_KEYS);
  const void* kp[FB_MAX_KEYS];
  int32_t kw[FB_MAX_KEYS];
  for (int i = 0; i < nkeys; ++i) {
    FB_CHECK(key_col_idx[i] >= 0 && key_col_idx[i] < ncols, "key column index %d out of range", key_col_idx[i]);
    kp[i] = col_ptrs[key_col_idx[i]];
    kw[i] = col_widths[key_col_idx[i]];
  }
  if (int rc = fb_partition_plan(dev, stream, nrows, nkeys, kp, kw, key_valid, num_partitions, scratch,
                                 scratch_bytes, out_part_offsets))
    return rc;
  return fb_partition_apply(dev, stream, nrows, nkeys, kp, kw, key_valid, num_partitions, scratch,
                            scratch_bytes, out_part_offsets, ncols, col_ptrs, col_widths, out_col_ptrs);
}

int fb_bits_to_bytes(int dev, void* stream, const uint8_t* bits, int64_t bit_offset, int64_t nrows,
                     uint8_t* out_bytes) {
  if (nrows <= 0) return 0;
  FbDeviceGuard guard(dev);
  FB_CHECK(guard.ok, "cannot select device %d", dev);
  int64_t blocks = (nrows + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  fb_bits_to_bytes_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(bits, bit_offset, nrows, out_bytes);
  FB_CUDA(cudaGetLastError());
  return 0;
}

int fb_bytes_to_bits(int dev, void* stream, const uint8_t* bytes, int64_t nrows, uint8_t* out_bits,
                     int64_t* out_null_count) {
  FbDeviceGuard guard(dev);
  FB_CHECK(guard.ok, "cannot select device %d", dev);
  cudaStream_t st = (cudaStream_t)stream;
  if (out_null_count) FB_CUDA(cudaMemsetAsync(out_null_count, 0, sizeof(int64_t), st));
  if (nrows <= 0) return 0;
  int64_t nbytes = (nrows + 7) / 8;
  int64_t blocks = (nbytes + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  fb_bytes_to_bits_kernel<<<(unsigned)blocks, 256, 0, st>>>(bytes, nrows, out_bits,
                                                           (unsigned long long*)out_null_count);
  FB_CUDA(cudaGetLastError());
  return 0;
}

}  // extern "C"
