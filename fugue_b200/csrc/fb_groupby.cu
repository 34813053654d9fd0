// K6: hash group-by with aggregation on sm_100a.
//
// Replaces the arithmetic behind ExecutionEngine.aggregate / SQL GROUP BY:
//   fugue/execution/execution_engine.py:889-939 (aggregate -> select -> SQL text)
//   fugue/column/sql.py:275-334               (SELECT keys, AGG(..) .. GROUP BY keys)
//   fugue/execution/native_execution_engine.py:59-66 (QPDPandasEngine.select -> qpd -> pandas
//                                                     groupby(dropna=False).agg)
// NULL key is a group of its own (fugue_test/execution_suite.py:195-200); NULL values are
// skipped by SUM/MIN/MAX/COUNT(col) and counted by COUNT(*) (SQL semantics).
//
// Design: open-addressing hash table in HBM, one 32-byte-aligned slot per group:
//   word 0            key (8 bytes; EMPTY = all ones, claimed with atomicCAS)
//   word 1 .. naggs   accumulators (8 bytes each), updated with L2 atomics (RED.ADD.F64 /
//                     RED.ADD.64 / RED.MIN/MAX.S64; f64 min/max on an order-preserving int code)
// so one row touches exactly one sector for (key, SUM, COUNT).  Rows whose key equals the EMPTY
// pattern and rows with a NULL key use two dedicated slots after the table.  Linear probing;
// a probe sequence longer than kMaxProbe raises the overflow flag and the host retries with a
// larger table.  Warp-level pre-merge: lanes of a warp that hold the same key (ballot match on
// the hash bits, verified on the key) elect one leader per key for the slot claim, so hot keys
// cost one CAS per warp instead of 32.
// Algorithmic bytes: 8 (key) + 8 per value column per row; the table traffic is random-access
// (one 32 B sector per row when the table exceeds L2).
#include "fb_common.cuh"

namespace {

constexpr uint64_t kEmpty = ~0ULL;
constexpr int kMaxProbe = 4096;

enum : int32_t {
  kSumF64 = FB_AGG_SUM_F64,
  kSumI64 = FB_AGG_SUM_I64,
  kCount = FB_AGG_COUNT,
  kMinI64 = FB_AGG_MIN_I64,
  kMaxI64 = FB_AGG_MAX_I64,
  kMinF64 = FB_AGG_MIN_F64,
  kMaxF64 = FB_AGG_MAX_F64,
};

struct AggSpec {
  const uint64_t* val[FB_MAX_AGGS];   // 8-byte value column (NULL for COUNT(*))
  const uint8_t* valid[FB_MAX_AGGS];  // byte mask or NULL
  int32_t op[FB_MAX_AGGS];
  int32_t naggs;
};

__host__ __device__ inline int slot_words(int naggs) { return (1 + naggs + 3) & ~3; }

// order-preserving map double <-> int64 (so that signed integer min/max order doubles)
__device__ __forceinline__ long long f64_to_ordered(uint64_t bits) {
  long long b = (long long)bits;
  return b >= 0 ? b : (long long)(bits ^ 0x7FFFFFFFFFFFFFFFULL);
}
__device__ __forceinline__ uint64_t ordered_to_f64(long long o) {
  return o >= 0 ? (uint64_t)o : ((uint64_t)o ^ 0x7FFFFFFFFFFFFFFFULL);
}

// The f64 identities are the ends of the ordered code (IEEE total order: -NaN < -inf < ... < +inf < +NaN),
// not +-inf: MIN over {+NaN} must stay +NaN.  An identity never reaches the output - a group either has a
// non-NULL value or its hidden COUNT makes the result NULL.
__device__ __forceinline__ uint64_t identity_of(int op) {
  switch (op) {
    case kMinI64:
    case kMinF64: return (uint64_t)0x7FFFFFFFFFFFFFFFLL;
    case kMaxI64:
    case kMaxF64: return (uint64_t)0x8000000000000000ULL;
    default: return 0;  // sums and counts (0.0 == bit pattern 0)
  }
}

// initialises slots [slot0, slot0 + nslots); status is reset when it is passed
constexpr int64_t kL2BatchBytes = 32ll << 20;  // table bytes worked on at a time (B200 L2: 126 MB)

__global__ void fb_groupby_init_kernel(uint64_t* __restrict__ table_all, int64_t slot0, int64_t nslots, int words,
                                       AggSpec spec, int64_t* __restrict__ status) {
  uint64_t* __restrict__ table = table_all + slot0 * words;
  const int64_t total = nslots * words;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int w = (int)(i % words);
    uint64_t v = 0;
    if (w == 0) v = kEmpty;
    else if (w <= spec.naggs) v = identity_of(spec.op[w - 1]);
    table[i] = v;
  }
  if (status != nullptr && blockIdx.x == 0 && threadIdx.x < 4) status[threadIdx.x] = 0;
}

__device__ __forceinline__ void apply_aggs(uint64_t* __restrict__ slot, const AggSpec& spec, int64_t row) {
#pragma unroll 1
  for (int a = 0; a < spec.naggs; ++a) {
    const int op = spec.op[a];
    if (spec.valid[a] != nullptr && spec.valid[a][row] == 0) continue;  // NULL value: skipped
    if (op == kCount) {
      atomicAdd((unsigned long long*)(slot + 1 + a), 1ULL);
      continue;
    }
    const uint64_t bits = spec.val[a][row];
    switch (op) {
      case kSumF64: atomicAdd((double*)(slot + 1 + a), __longlong_as_double((long long)bits)); break;
      case kSumI64: atomicAdd((unsigned long long*)(slot + 1 + a), (unsigned long long)bits); break;
      case kMinI64: atomicMin((long long*)(slot + 1 + a), (long long)bits); break;
      case kMaxI64: atomicMax((long long*)(slot + 1 + a), (long long)bits); break;
      case kMinF64: atomicMin((long long*)(slot + 1 + a), f64_to_ordered(bits)); break;
      case kMaxF64: atomicMax((long long*)(slot + 1 + a), f64_to_ordered(bits)); break;
      default: break;
    }
  }
}

// slot of `key` (inserting it if absent); -1 on overflow.  With num_parts > 0 the table is cut
// into num_parts equal regions and a key lives in the region of its partition id (the same
// hash % num_parts as the partitioner): on hash-partitioned input the kernel then sweeps the
// table region by region and the atomics stay L2-resident instead of going to HBM.
__device__ __forceinline__ int64_t find_or_insert(uint64_t* __restrict__ table, int words, int64_t mask,
                                                  uint64_t key, const FbDiv& dv, int64_t region_base_shift) {
  int64_t base = 0;
  uint64_t h = fb_fmix64(key);
  if (region_base_shift >= 0) {
    base = (int64_t)fb_fastmod(fb_hash_single_u64(key), dv) << region_base_shift;
    h >>= 7;
  }
  int64_t s = (int64_t)(h & (uint64_t)mask);
#pragma unroll 1
  for (int probe = 0; probe < kMaxProbe; ++probe) {
    uint64_t* slot = table + (base + s) * words;
    uint64_t cur = *(volatile uint64_t*)slot;
    if (cur == key) return base + s;
    if (cur == kEmpty) {
      const uint64_t old = atomicCAS((unsigned long long*)slot, (unsigned long long)kEmpty,
                                     (unsigned long long)key);
      if (old == kEmpty || old == key) return base + s;
    }
    s = (s + 1) & mask;
  }
  return -1;
}

__global__ void __launch_bounds__(256)
fb_groupby_kernel(const uint64_t* __restrict__ keys, const uint8_t* __restrict__ key_valid, int64_t nrows,
                  uint64_t* __restrict__ table, int64_t capacity, int words, AggSpec spec,
                  int64_t* __restrict__ status, FbDiv dv, int64_t region_shift,
                  const int64_t* __restrict__ part_off, int p0, int p1) {
  // region_shift < 0: one region = the whole table; else region size = 1 << region_shift
  // part_off != nullptr: only the rows of hash partitions [p0, p1) (one launch per batch of regions)
  const int64_t mask = region_shift >= 0 ? (((int64_t)1 << region_shift) - 1) : capacity - 1;
  const unsigned lane = threadIdx.x & 31;
  const unsigned lt = fb_lanemask_lt();
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t row_lo = part_off != nullptr ? part_off[p0] : 0;
  const int64_t row_hi = part_off != nullptr ? part_off[p1] : nrows;
  const int64_t nround = (row_hi - row_lo + stride - 1) / stride;
  for (int64_t it = 0; it < nround; ++it) {
    const int64_t row = row_lo + it * stride + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool ok = row < row_hi;
    uint64_t key = 0;
    int64_t s = -2;
    bool special = false;
    if (ok) {
      key = keys[row];
      if (key_valid != nullptr && key_valid[row] == 0) { s = capacity + 1; special = true; }  // NULL group
      else if (key == kEmpty) { s = capacity; special = true; }                             // EMPTY-valued key
    }
    // warp pre-merge: one leader per distinct key does the probe, the others reuse its slot
    const bool need = ok && !special;
    const unsigned need_mask = __ballot_sync(0xFFFFFFFFu, need);
    unsigned peers = need_mask;
    if (need) {
      const uint32_t h = (uint32_t)(fb_fmix64(key) >> 20);
#pragma unroll
      for (int b = 0; b < 6; ++b) {
        const bool bit = (h >> b) & 1u;
        const unsigned bal = __ballot_sync(need_mask, bit);
        peers &= bit ? bal : ~bal;
      }
    }
    int leader = need ? (__ffs(peers) - 1) : (int)lane;
    const uint64_t lkey = __shfl_sync(0xFFFFFFFFu, key, leader);
    const bool follow = need && leader != (int)lane && lkey == key;
    if (need && !follow) s = find_or_insert(table, words, mask, key, dv, region_shift);
    const int64_t ls = __shfl_sync(0xFFFFFFFFu, s, leader);
    if (follow) s = ls;
    if (ok) {
      if (s < 0) {
        status[0] = 1;  // overflow: the host retries with a larger table
      } else {
        if (special) table[s * words] = 0;  // mark the dedicated slot as used (any value != EMPTY)
        apply_aggs(table + s * words, spec, row);
      }
    }
    (void)lt;
  }
}

// ---------------------------------------------------------------------------------------------------
// Lean variant of fb_groupby_kernel for hash-partitioned input and at most four aggregates (the shape of
// SELECT key, SUM(v), COUNT(*) ... GROUP BY key): ONE hash per row (the partitioner's; region = partition
// id, slot from its upper bits), the aggregate descriptors in registers, the loop over aggregates
// unrolled.  The generic kernel spends ~660 thread instructions per row and is issue-bound (ncu: 70 %
// issue-active, profiles/r2_groupby_notes.md); this one leaves the L2 atomic units as the limit.
// ---------------------------------------------------------------------------------------------------
template <int NAGG>
struct LeanAggs {
  const uint64_t* val[NAGG];
  const uint8_t* valid[NAGG];
  int32_t op[NAGG];
};

template <int NAGG>
__global__ void __launch_bounds__(256)
fb_groupby_lean_kernel(const uint64_t* __restrict__ keys, const uint8_t* __restrict__ key_valid, int64_t nrows,
                       uint64_t* __restrict__ table, int64_t capacity, const LeanAggs<NAGG> aggs,
                       int64_t* __restrict__ status, uint32_t parts_mask, int region_shift) {
  constexpr int words = (1 + NAGG + 3) & ~3;
  const uint32_t mask = (1u << region_shift) - 1u;
  const unsigned lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t nround = (nrows + stride - 1) / stride;
  for (int64_t it = 0; it < nround; ++it) {
    const int64_t row = it * stride + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool ok = row < nrows;
    uint64_t key = ok ? keys[row] : 0;
    int64_t s = -2;
    bool special = false;
    if (ok) {
      if (key_valid != nullptr && key_valid[row] == 0) { s = capacity + 1; special = true; }  // NULL group
      else if (key == kEmpty) { s = capacity; special = true; }                             // EMPTY-valued key
    }
    const uint64_t h = fb_hash_single_u64(key);
    // warp pre-merge on 6 hash bits (verified on the key): one prober per distinct key per warp, so that a hot
    // key costs one probe + 32 updates instead of 32 serialised probes
    const bool need = ok && !special;
    const unsigned need_mask = __ballot_sync(0xFFFFFFFFu, need);
    unsigned peers = need_mask;
    if (need) {
      const uint32_t hb = (uint32_t)(h >> 40);
#pragma unroll
      for (int b = 0; b < 6; ++b) {
        const bool bit = (hb >> b) & 1u;
        const unsigned bal = __ballot_sync(need_mask, bit);
        peers &= bit ? bal : ~bal;
      }
    }
    const int leader = need ? (__ffs(peers) - 1) : (int)lane;
    const uint64_t lkey = __shfl_sync(0xFFFFFFFFu, key, leader);
    const bool follow = need && leader != (int)lane && lkey == key;
    if (need && !follow) {
      const int64_t base = (int64_t)((uint32_t)h & parts_mask) << region_shift;
      uint32_t o = (uint32_t)(h >> 10) & mask;
      s = -1;
#pragma unroll 1
      for (int probe = 0; probe < kMaxProbe; ++probe) {
        uint64_t* slot = table + (base + o) * words;
        uint64_t cur = *(volatile uint64_t*)slot;
        if (cur == kEmpty) {
          cur = atomicCAS((unsigned long long*)slot, (unsigned long long)kEmpty, (unsigned long long)key);
          if (cur == kEmpty) cur = key;
        }
        if (cur == key) { s = base + o; break; }
        o = (o + 1) & mask;
      }
    }
    const int64_t ls = __shfl_sync(0xFFFFFFFFu, s, leader);
    if (follow) s = ls;
    if (ok) {
      if (s < 0) {
        status[0] = 1;  // overflow: the host retries with a larger table
      } else {
        uint64_t* slot = table + s * words;
        if (special) slot[0] = 0;  // mark the dedicated slot as used (any value != EMPTY)
#pragma unroll
        for (int a = 0; a < NAGG; ++a) {
          if (aggs.valid[a] != nullptr && aggs.valid[a][row] == 0) continue;  // NULL value: skipped
          const int op = aggs.op[a];
          if (op == kCount) {
            atomicAdd((unsigned long long*)(slot + 1 + a), 1ULL);
            continue;
          }
          const uint64_t bits = aggs.val[a][row];
          switch (op) {
            case kSumF64: atomicAdd((double*)(slot + 1 + a), __longlong_as_double((long long)bits)); break;
            case kSumI64: atomicAdd((unsigned long long*)(slot + 1 + a), (unsigned long long)bits); break;
            case kMinI64: atomicMin((long long*)(slot + 1 + a), (long long)bits); break;
            case kMaxI64: atomicMax((long long*)(slot + 1 + a), (long long)bits); break;
            case kMinF64: atomicMin((long long*)(slot + 1 + a), f64_to_ordered(bits)); break;
            case kMaxF64: atomicMax((long long*)(slot + 1 + a), f64_to_ordered(bits)); break;
            default: break;
          }
        }
      }
    }
  }
}

template <int NAGG>
void launch_lean(const uint64_t* keys, const uint8_t* key_valid, int64_t nrows, uint64_t* table, int64_t capacity,
                 const AggSpec& spec, int64_t* status, uint32_t num_parts, int region_shift, int grid,
                 cudaStream_t st) {
  LeanAggs<NAGG> la;
  for (int a = 0; a < NAGG; ++a) {
    la.val[a] = spec.val[a];
    la.valid[a] = spec.valid[a];
    la.op[a] = spec.op[a];
  }
  fb_groupby_lean_kernel<NAGG><<<grid, 256, 0, st>>>(keys, key_valid, nrows, table, capacity, la, status, num_parts - 1,
                                                     region_shift);
}

__global__ void __launch_bounds__(256)
fb_groupby_extract_kernel(const uint64_t* __restrict__ table, int64_t capacity, int words, AggSpec spec,
                          uint64_t* __restrict__ out_keys, uint8_t* __restrict__ out_key_valid,
                          uint64_t* const* __restrict__ out_aggs, int64_t* __restrict__ status) {
  const unsigned lane = threadIdx.x & 31;
  const int64_t nslots = capacity + 2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t nround = (nslots + stride - 1) / stride;
  for (int64_t it = 0; it < nround; ++it) {
    const int64_t s = it * stride + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool used = s < nslots && table[s * words] != kEmpty;
    const unsigned m = __ballot_sync(0xFFFFFFFFu, used);
    if (m == 0) continue;
    long long base = 0;
    if (lane == (unsigned)(__ffs(m) - 1))
      base = (long long)atomicAdd((unsigned long long*)&status[1], (unsigned long long)__popc(m));
    base = __shfl_sync(0xFFFFFFFFu, base, __ffs(m) - 1);
    if (used) {
      const int64_t o = base + __popc(m & fb_lanemask_lt());
      const uint64_t* slot = table + s * words;
      out_keys[o] = s < capacity ? slot[0] : (s == capacity ? kEmpty : 0ULL);
      if (out_key_valid != nullptr) out_key_valid[o] = s == capacity + 1 ? 0 : 1;
      for (int a = 0; a < spec.naggs; ++a) {
        uint64_t v = slot[1 + a];
        if (spec.op[a] == kMinF64 || spec.op[a] == kMaxF64) v = ordered_to_f64((long long)v);
        out_aggs[a][o] = v;
      }
    }
  }
}

int fill_spec(AggSpec& spec, int naggs, const void* const* val_ptrs, const uint8_t* const* val_valid,
              const int32_t* ops) {
  FB_CHECK(naggs >= 0 && naggs <= FB_MAX_AGGS, "naggs=%d out of range [0,%d]", naggs, FB_MAX_AGGS);
  memset(&spec, 0, sizeof(spec));
  spec.naggs = naggs;
  for (int a = 0; a < naggs; ++a) {
    FB_CHECK(ops[a] >= FB_AGG_SUM_F64 && ops[a] <= FB_AGG_MAX_F64, "unknown aggregate op %d", ops[a]);
    FB_CHECK(ops[a] == FB_AGG_COUNT || (val_ptrs != nullptr && val_ptrs[a] != nullptr),
             "aggregate %d needs a value column", a);
    spec.op[a] = ops[a];
    spec.val[a] = val_ptrs ? (const uint64_t*)val_ptrs[a] : nullptr;
    spec.valid[a] = val_valid ? val_valid[a] : nullptr;
  }
  return 0;
}

}  // namespace

extern "C" {

size_t fb_groupby_table_bytes(int64_t capacity, int naggs) {
  if (capacity <= 0 || naggs < 0) return 0;
  return (size_t)(capacity + 2) * slot_words(naggs) * sizeof(uint64_t);
}

int fb_groupby_u64(int dev, void* stream, int64_t nrows, const void* keys, const uint8_t* key_valid,
                   int naggs, const void* const* val_ptrs, const uint8_t* const* val_valid,
                   const int32_t* agg_ops, int64_t capacity, uint32_t num_parts, void* table,
                   int64_t* d_status, const int64_t* d_part_offsets) {
  FB_CHECK(nrows >= 0, "nrows < 0");
  FB_CHECK(capacity >= 2 && (capacity & (capacity - 1)) == 0, "capacity must be a power of two >= 2");
  FB_CHECK(table != nullptr && d_status != nullptr, "table/status is NULL");
  FbDeviceGuard guard(dev);
  FB_CHECK(guard.ok, "cannot select device %d", dev);
  AggSpec spec;
  if (int rc = fill_spec(spec, naggs, val_ptrs, val_valid, agg_ops)) return rc;
  int64_t region_shift = -1;
  if (num_parts > 1) {
    FB_CHECK((num_parts & (num_parts - 1)) == 0 && (int64_t)num_parts * 2 <= capacity,
             "num_parts must be a power of two <= capacity / 2");
    region_shift = 0;
    while (((int64_t)num_parts << region_shift) < capacity) ++region_shift;
  }
  const FbDiv dv = fb_make_div(num_parts > 1 ? num_parts : 1);
  cudaStream_t st = (cudaStream_t)stream;
  const int words = slot_words(naggs);
  const int sms = fb_sm_count(dev);
  if (nrows > 0) FB_CHECK(keys != nullptr, "keys is NULL");
  if (num_parts > 1 && d_part_offsets != nullptr && nrows > 0) {
    // batches of regions small enough to stay in L2 between their initialisation and the last
    // atomic on them: a table that is initialised as a whole is back in HBM before it is used,
    // and every probe / atomic then costs a random DRAM sector read plus a write-back
    // (measured: 3.4 ms for 125 M rows into 10 M groups; batched: see profiles/r1_notes.md)
    const int64_t region_bytes = ((int64_t)1 << region_shift) * words * (int64_t)sizeof(uint64_t);
    int64_t per = kL2BatchBytes / region_bytes;
    if (per < 1) per = 1;
    fb_groupby_init_kernel<<<1, 64, 0, st>>>((uint64_t*)table, capacity, 2, words, spec, d_status);  // special slots
    FB_CUDA(cudaGetLastError());
    for (int64_t p0 = 0; p0 < (int64_t)num_parts; p0 += per) {
      const int64_t p1 = p0 + per < (int64_t)num_parts ? p0 + per : (int64_t)num_parts;
      const int64_t nslots = (p1 - p0) << region_shift;
      int64_t ib = (nslots * words + 256 * 8 - 1) / (256 * 8);
      if (ib > sms * 8) ib = sms * 8;
      fb_groupby_init_kernel<<<(unsigned)ib, 256, 0, st>>>((uint64_t*)table, p0 << region_shift, nslots, words, spec,
                                                          nullptr);
      const int64_t est = nrows / num_parts * (p1 - p0) * 5 / 4 + 256;
      int64_t gb = (est + 255) / 256;
      if (gb > sms * 8) gb = sms * 8;
      fb_groupby_kernel<<<(unsigned)gb, 256, 0, st>>>((const uint64_t*)keys, key_valid, nrows, (uint64_t*)table,
                                                     capacity, words, spec, d_status, dv, region_shift,
                                                     d_part_offsets, (int)p0, (int)p1);
    }
    FB_CUDA(cudaGetLastError());
    return 0;
  }
  fb_groupby_init_kernel<<<sms * 8, 256, 0, st>>>((uint64_t*)table, 0, capacity + 2, words, spec, d_status);
  FB_CUDA(cudaGetLastError());
  if (nrows > 0 && num_parts > 1 && naggs >= 1 && naggs <= 4 && region_shift >= 1 && region_shift < 31) {
    // hash-partitioned input, few aggregates: the lean kernel (the find-or-insert of the generic kernel
    // hashes with fb_fmix64(key) >> 7; here the slot comes from the partitioner's hash - a table is only
    // ever read back by the extract pass, which does not hash)
    const uint64_t* k64 = (const uint64_t*)keys;
    uint64_t* t64 = (uint64_t*)table;
    switch (naggs) {
      case 1: launch_lean<1>(k64, key_valid, nrows, t64, capacity, spec, d_status, num_parts, (int)region_shift, sms * 8, st); break;
      case 2: launch_lean<2>(k64, key_valid, nrows, t64, capacity, spec, d_status, num_parts, (int)region_shift, sms * 8, st); break;
      case 3: launch_lean<3>(k64, key_valid, nrows, t64, capacity, spec, d_status, num_parts, (int)region_shift, sms * 8, st); break;
      default: launch_lean<4>(k64, key_valid, nrows, t64, capacity, spec, d_status, num_parts, (int)region_shift, sms * 8, st); break;
    }
    FB_CUDA(cudaGetLastError());
    return 0;
  }
  if (nrows > 0) {
    fb_groupby_kernel<<<sms * 8, 256, 0, st>>>((const uint64_t*)keys, key_valid, nrows, (uint64_t*)table,
                                              capacity, words, spec, d_status, dv, region_shift, nullptr, 0, 0);
    FB_CUDA(cudaGetLastError());
  }
  return 0;
}

int fb_groupby_extract(int dev, void* stream, int64_t capacity, int naggs, const int32_t* agg_ops,
                       const void* table, void* out_keys, uint8_t* out_key_valid,
                       void* const* d_out_aggs, int64_t* d_status) {
  FB_CHECK(capacity >= 2 && (capacity & (capacity - 1)) == 0, "capacity must be a power of two >= 2");
  FbDeviceGuard guard(dev);
  FB_CHECK(guard.ok, "cannot select device %d", dev);
  AggSpec spec;
  memset(&spec, 0, sizeof(spec));
  FB_CHECK(naggs >= 0 && naggs <= FB_MAX_AGGS, "naggs out of range");
  spec.naggs = naggs;
  for (int a = 0; a < naggs; ++a) spec.op[a] = agg_ops[a];
  const int sms = fb_sm_count(dev);
  fb_groupby_extract_kernel<<<sms * 8, 256, 0, (cudaStream_t)stream>>>(
      (const uint64_t*)table, capacity, slot_words(naggs), spec, (uint64_t*)out_keys, out_key_valid,
      (uint64_t* const*)d_out_aggs, d_status);
  FB_CUDA(cudaGetLastError());
  return 0;
}

}  // extern "C"
