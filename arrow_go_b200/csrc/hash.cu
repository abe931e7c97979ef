// hash.cu — is_in and unique for fixed-width columns on sm_100a (SURVEY §8f rank 3).
//
// Replaces, for 1/2/4/8-byte values, the memo-table kernels of the reference:
//   is_in   arrow/compute/internal/kernels/scalar_set_lookup.go:112-413 (SetLookupState.Init builds a memo table of
//           the value set keyed by the RAW BYTES of a value — floats compare by bit pattern: NaN == NaN of the same
//           payload, -0.0 != +0.0; isInKernelExec :373-413 writes a data bit and a validity bit per row by the
//           NullMatchingBehavior table restated in is_in_kernel below);
//   unique  arrow/compute/internal/kernels/vector_hash.go (the distinct values in order of FIRST appearance, a null
//           kept once at the position of its first appearance).
// Both sit on the same open-addressing table: 16-byte slots {64-bit key = the value's bytes zero-extended, lowest row
// that carried the key}, linear probing from an even slot (so a probe can always look at an aligned pair), load factor
// <= 0.5, keys inserted with atomicCAS, first rows with atomicMin.  The first row is all `unique` needs: a row is
// emitted iff it is the first row of its key, and the emitted rows are compacted in row order by the filter kernel
// (filter.cu) — so the output order is the reference's and does not depend on the order in which threads reached the
// table.
//   is_in : value sets up to 4096 entries are probed in shared memory (at most 8192 key slots = 64 KB, load factor <= 1/4
//           for sets up to 2048 values, two slots per 128-bit read); 1- and 2-byte values skip hashing altogether:
//           the set becomes a 256 / 65536-bit membership bitmap.  Larger sets are probed in HBM / L2.
//   unique: a column of more than 2M rows first runs against a 4M-slot table that stays L2-resident (64 MB); only when
//           more than 2M distinct values turn up does the insert raise an overflow word, and the full-size table
//           (2n slots) is cleared and filled by kernels that test that word first — the choice is made on the device,
//           the call stays stream-ordered.  Each warp also keeps the last keys it met in a small shared-memory cache:
//           a key met at a lower row of the same warp cannot be a first appearance, so low-cardinality columns
//           (the usual dictionary-encoding case) hardly touch the table at all.
//   dictionary_encode (kernels/vector_hash.go:144-241 dictionaryEncodeAction over doAppendNumeric :359-385) follows
//           the same table policy as unique (ag_unique_set_policy) and the same insert + mark passes; then the
//           first rows are ranked (an exclusive scan of popc(keep) per tile), the finalize pass writes each distinct
//           value to dict[rank] and stores the rank in the slot's spare word, and one streaming pass writes an int32
//           index per row (one probe returns key + first row + rank in a 16-byte load; a per-warp (key, rank)
//           cache keeps low-cardinality columns off the table).  Ranks are positions of first rows, so the output
//           does not depend on the order in which threads reached the table.
// Roofline: HBM, 8 B/row read once per pass (is_in: one pass; unique: insert + mark + compaction; dictionary_encode:
// insert + mark + encode, which also writes 4 B/row).
#include "common.cuh"

namespace ag {

ag_status filter_primitive_dev(int bit_width, const void* vals, const uint8_t* vvalid, int64_t voff, const uint8_t* mask,
                               const uint8_t* mvalid, int64_t moff, int64_t n, int null_selection, void* out, uint8_t* out_valid,
                               int64_t capacity, int64_t* d_out_len, cudaStream_t st);

constexpr int kHThreads = 256;
constexpr int kHWarps = kHThreads / 32;
constexpr int kHUnroll = 4;                 // 32-row groups a warp has in flight
constexpr unsigned long long kEmptyKey = 0xffffffffffffffffull;
constexpr unsigned kNoRow = 0xffffffffu;
constexpr unsigned kNoCap = 0xffffffffu;

// `rank`: unused by is_in / unique; dictionary_encode's finalize pass stores the key's dictionary position there
struct alignas(16) Slot { unsigned long long key; unsigned first; unsigned rank; };

struct HashTable {
  Slot* slots;                // cleared to all-ones: key = kEmptyKey (free), first = kNoRow
  unsigned long long mask;    // slots - 1
  int shift;                  // 64 - log2(slots)
  unsigned cap;               // distinct keys after which an insert raises special[3] and stops (kNoCap: never)
  unsigned* special;          // [0] lowest row whose key is the all-ones pattern (cannot live in `slots`), [1] lowest NULL row,
                              // [2] distinct keys inserted, [3] overflow word (0xffffffff after the clear = not raised),
                              // [4] / [5] dictionary_encode: ranks of the all-ones key / of the null entry
};

// multiplicative (Fibonacci) hash of the folded key, forced even: every probe sequence starts on an aligned slot pair
__device__ __forceinline__ unsigned long long hash_slot(unsigned long long key, int shift) {
  const unsigned long long x = key ^ (key >> 32);
  return ((x * 0x9E3779B97F4A7C15ull) >> shift) & ~1ull;
}
__device__ __forceinline__ bool overflowed(const HashTable& t) { return *reinterpret_cast<volatile unsigned*>(&t.special[3]) == 1u; }

template <typename V>
__device__ __forceinline__ unsigned long long raw_key(const V* __restrict__ vals, int64_t i) {
  return (unsigned long long)vals[i];
}

// lower `*p` to `row` (rows arrive roughly in increasing order, so after the first few rows of a key the word already
// holds a lower row and a plain load replaces the atomic: 100M rows over 100 keys would otherwise serialise 100M atomics
// on 100 addresses)
__device__ __forceinline__ void lower_row(unsigned* p, unsigned seen, unsigned row) {
  if (seen > row) atomicMin(p, row);
}

// returns true when this call created the key's slot
__device__ __forceinline__ bool table_insert(const HashTable& t, unsigned long long key, unsigned row) {
  unsigned long long h = hash_slot(key, t.shift);
  unsigned probes = 0;
  while (true) {
    Slot* s = t.slots + h;
    const ulonglong2 raw = __ldcg(reinterpret_cast<const ulonglong2*>(s));   // key and first row in one L2 request
    unsigned long long cur = raw.x;
    unsigned seen = (unsigned)raw.y;
    bool made = false;
    if (cur == kEmptyKey) {
      cur = atomicCAS(&s->key, kEmptyKey, key);
      if (cur == kEmptyKey) { made = true; seen = kNoRow; cur = key; }
      else if (cur == key) seen = kNoRow;     // somebody else created it just now: its first row is not in `raw`
    }
    if (cur == key) { lower_row(&s->first, seen, row); return made; }
    h = (h + 1) & t.mask;
    // a capped table can fill up completely while the inserts that were in flight when the cap was crossed finish
    if (t.cap != kNoCap && ((++probes & 7u) == 0u)) {
      if (overflowed(t)) return false;
      // a probe this long at load factor <= 1/2 means the table has filled up behind the counter (the lanes that
      // created the last keys report them only after their warp step, and a lane spinning here would keep its own
      // warp from ever reporting): raise the word from here
      if (probes >= 1024u) { *reinterpret_cast<volatile unsigned*>(&t.special[3]) = 1u; return false; }
    }
  }
}
// lowest row that carried `key`, kNoRow when absent (the table is complete: plain cached loads)
__device__ __forceinline__ unsigned table_first_row(const HashTable& t, unsigned long long key) {
  unsigned long long h = hash_slot(key, t.shift);
  while (true) {
    const ulonglong2 raw = *reinterpret_cast<const ulonglong2*>(t.slots + h);
    if (raw.x == key) return (unsigned)raw.y;
    if (raw.x == kEmptyKey) return kNoRow;
    h = (h + 1) & t.mask;
  }
}

// Per-warp cache of keys already met (direct-mapped, 256 entries).  A warp walks its rows in increasing order, so a hit
// means: this key sits at a lower row that this warp has already sent to the table.
constexpr int kWarpCacheSlots = 256;
__device__ __forceinline__ int warp_cache_slot(unsigned long long key) {
  return (int)(((key ^ (key >> 32)) * 0x9E3779B97F4A7C15ull) >> 56);
}

// `run_if`: NULL, or a device word the kernel tests first (the full-size pass of `unique` runs only after an overflow)
template <typename V>
__global__ void __launch_bounds__(kHThreads)
hash_insert_kernel(const V* __restrict__ vals, const uint8_t* __restrict__ valid, int64_t off, int64_t n, const HashTable t,
                   const unsigned* __restrict__ run_if) {
  __shared__ unsigned long long s_cache[kHWarps][kWarpCacheSlots];
  if (run_if && *run_if != 1u) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long* cache = s_cache[warp];
  for (int i = lane; i < kWarpCacheSlots; i += 32) cache[i] = kEmptyKey;
  __syncwarp();
  const int64_t n_words = (n + 31) >> 5;
  const int64_t warp0 = ((int64_t)blockIdx.x * kHThreads + threadIdx.x) >> 5;
  const int64_t warps = ((int64_t)gridDim.x * kHThreads) >> 5;
  for (int64_t w0 = warp0 * kHUnroll; w0 < n_words; w0 += warps * kHUnroll) {
    if (__any_sync(0xffffffffu, t.cap != kNoCap && overflowed(t))) return;   // the small table is being abandoned (warp-uniform exit)
    V x[kHUnroll];
    int kind[kHUnroll];                                  // 0 nothing, 1 value, 2 null
    if (!valid && ((w0 + kHUnroll) << 5) <= n) {         // interior, no nulls: unconditional loads
      const V* __restrict__ p = vals + off + (w0 << 5) + lane;
#pragma unroll
      for (int k = 0; k < kHUnroll; ++k) { x[k] = __ldcs(p + 32 * k); kind[k] = 1; }
    } else {
#pragma unroll
      for (int k = 0; k < kHUnroll; ++k) {
        const int64_t i = ((w0 + k) << 5) + lane;
        kind[k] = i < n ? ((valid && !bit_is_set(valid, off + i)) ? 2 : 1) : 0;
        x[k] = kind[k] == 1 ? __ldcs(vals + off + i) : V(0);
      }
    }
#pragma unroll
    for (int k = 0; k < kHUnroll; ++k) {
      const unsigned row = (unsigned)(((w0 + k) << 5) + lane);
      const unsigned long long key = (unsigned long long)x[k];
      const int cs = warp_cache_slot(key);
      const bool ones = sizeof(V) == 8 && key == kEmptyKey;     // narrower values zero-extend: never all ones
      if (kind[k] == 2) lower_row(&t.special[1], *reinterpret_cast<volatile unsigned*>(&t.special[1]), row);
      else if (kind[k] == 1 && ones) lower_row(&t.special[0], *reinterpret_cast<volatile unsigned*>(&t.special[0]), row);
      const bool go = kind[k] == 1 && !ones && cache[cs] != key;
      __syncwarp();
      bool made = false;
      if (go) { made = table_insert(t, key, row); atomicExch(&cache[cs], key); }   // several lanes may share a slot: one whole key wins
      __syncwarp();
      if (t.cap != kNoCap) {
        // distinct keys so far, one atomic per warp step (a column of all-distinct values would otherwise put 2M
        // atomics on one word before the cap stops it: 2.9 ms).  special[2] is cleared to 0xffffffff = count - 1.
        const unsigned m = __ballot_sync(0xffffffffu, made);
        if (lane == 0 && m) {
          const unsigned c = (unsigned)__popc(m);
          if (atomicAdd(&t.special[2], c) + 1u + c > t.cap) *reinterpret_cast<volatile unsigned*>(&t.special[3]) = 1u;
        }
      }
    }
  }
}

__global__ void __launch_bounds__(kHThreads)
table_clear_kernel(uint4* __restrict__ p, int64_t n16, const unsigned* __restrict__ run_if) {
  if (run_if && *run_if != 1u) return;
  const uint4 ones = make_uint4(0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu);
  for (int64_t i = (int64_t)blockIdx.x * kHThreads + threadIdx.x; i < n16; i += (int64_t)gridDim.x * kHThreads) p[i] = ones;
}

// isInKernelExec (scalar_set_lookup.go:373-413), per row:
//   valid value : in the set -> (true, valid); else INCONCLUSIVE with a null in the set -> (false, null); else (false, valid)
//   null        : MATCH with a null in the set -> (true, valid); SKIP, or MATCH without one -> (false, valid); else (false, null)
constexpr int kIsInSmemSlots = 8192;   // 64 KB of keys
enum { kMemberTable = 0, kMemberSmem = 1, kMemberBitmap = 2 };

// membership bitmap of a 1- or 2-byte value set: bit v of `bits`; a null in the set lowers special[1]
template <typename V>
__global__ void __launch_bounds__(kHThreads)
set_bitmap_kernel(const V* __restrict__ set, const uint8_t* __restrict__ valid, int64_t off, int64_t n, unsigned* __restrict__ bits,
                  unsigned* __restrict__ special) {
  for (int64_t i = (int64_t)blockIdx.x * kHThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kHThreads) {
    if (valid && !bit_is_set(valid, off + i)) atomicMin(&special[1], (unsigned)i);
    else { const unsigned v = (unsigned)set[off + i]; atomicOr(&bits[v >> 5], 1u << (v & 31)); }
  }
}

template <typename V, int kMember>
__global__ void __launch_bounds__(kHThreads)
is_in_kernel(const V* __restrict__ vals, const uint8_t* __restrict__ valid, int64_t off, int64_t n, const HashTable t,
             const unsigned* __restrict__ set_bits, int null_behavior, uint32_t* __restrict__ out_data, uint32_t* __restrict__ out_valid,
             unsigned long long* __restrict__ null_count) {
  extern __shared__ __align__(16) unsigned long long s_keys[];   // kMemberSmem: the table's keys; kMemberBitmap: the bitmap words
  constexpr int kBitWords = sizeof(V) == 1 ? 8 : 2048;
  if (kMember == kMemberSmem) {
    // the column streams through L1 and would keep evicting a table that lives in global memory
    for (unsigned i = threadIdx.x; i <= (unsigned)t.mask; i += kHThreads) s_keys[i] = t.slots[i].key;
    __syncthreads();
  } else if (kMember == kMemberBitmap) {
    unsigned* sb = reinterpret_cast<unsigned*>(s_keys);
    for (int i = threadIdx.x; i < kBitWords; i += kHThreads) sb[i] = set_bits[i];
    __syncthreads();
  }
  const bool set_has_null = t.special[1] != kNoRow;
  const bool set_has_ones = t.special[0] != kNoRow;
  auto member = [&](unsigned long long key) -> bool {
    if (kMember == kMemberBitmap) {
      const unsigned* sb = reinterpret_cast<const unsigned*>(s_keys);
      return (sb[(unsigned)key >> 5] >> ((unsigned)key & 31)) & 1u;
    }
    if (sizeof(V) == 8 && key == kEmptyKey) return set_has_ones;      // narrower values zero-extend: never all ones
    unsigned long long h = hash_slot(key, t.shift);
    while (true) {
      unsigned long long k0, k1;
      if (kMember == kMemberSmem) {
        const ulonglong2 pr = *reinterpret_cast<const ulonglong2*>(s_keys + h);   // h is even: one aligned pair
        k0 = pr.x; k1 = pr.y;
      } else {
        k0 = t.slots[h].key; k1 = t.slots[h + 1].key;                             // same 32-byte sector
      }
      if (k0 == key || k1 == key) return true;
      if (k0 == kEmptyKey || k1 == kEmptyKey) return false;
      h = (h + 2) & t.mask;
    }
  };
  const int lane = threadIdx.x & 31;
  const int64_t n_words = (n + 31) >> 5;
  const int64_t warp0 = ((int64_t)blockIdx.x * kHThreads + threadIdx.x) >> 5;
  const int64_t warps = ((int64_t)gridDim.x * kHThreads) >> 5;
  unsigned long long nulls = 0;
  const bool miss_is_null = null_behavior == AG_NULL_INCONCLUSIVE && set_has_null;
  for (int64_t w0 = warp0 * kHUnroll; w0 < n_words; w0 += warps * kHUnroll) {
    if (!valid && ((w0 + kHUnroll) << 5) <= n) {
      // interior, no input nulls: no range tests, no masks; word k of the step is stored by lane k
      // (profile: the edge handling below was half of the 112 instructions per row of this kernel)
      const V* __restrict__ p = vals + off + (w0 << 5) + lane;
      V x[kHUnroll];
#pragma unroll
      for (int k = 0; k < kHUnroll; ++k) x[k] = __ldcs(p + 32 * k);
      uint32_t mine = 0;
#pragma unroll
      for (int k = 0; k < kHUnroll; ++k) {
        const uint32_t dbits = __ballot_sync(0xffffffffu, member((unsigned long long)x[k]));
        if (lane == k) mine = dbits;
      }
      if (lane < kHUnroll) {
        out_data[w0 + lane] = mine;
        if (out_valid) out_valid[w0 + lane] = miss_is_null ? mine : 0xffffffffu;
        if (miss_is_null) nulls += __popc(~mine);
      }
      continue;
    }
    V x[kHUnroll];
    bool have[kHUnroll], isnull[kHUnroll];
#pragma unroll
    for (int k = 0; k < kHUnroll; ++k) {   // independent loads first: 4 rows in flight per lane
      const int64_t i = ((w0 + k) << 5) + lane;
      have[k] = i < n;
      isnull[k] = have[k] && valid && !bit_is_set(valid, off + i);
      x[k] = (have[k] && !isnull[k]) ? __ldcs(vals + off + i) : V(0);
    }
#pragma unroll
    for (int k = 0; k < kHUnroll; ++k) {
      const int64_t w = w0 + k;
      if (w >= n_words) break;   // warp-uniform
      bool d = false, v = true;
      if (have[k]) {
        if (isnull[k]) {
          if (null_behavior == AG_NULL_MATCH && set_has_null) d = true;
          else if (null_behavior == AG_NULL_SKIP || (null_behavior == AG_NULL_MATCH && !set_has_null)) d = false;
          else v = false;
        } else if (member((unsigned long long)x[k])) {
          d = true;
        } else if (null_behavior == AG_NULL_INCONCLUSIVE && set_has_null) {
          v = false;
        }
      }
      const uint32_t dbits = __ballot_sync(0xffffffffu, d);
      const uint32_t vbits = __ballot_sync(0xffffffffu, v);
      if (lane == 0) {
        const int64_t rem = n - (w << 5);
        const uint32_t m = rem >= 32 ? 0xffffffffu : bit_range_mask(0, (int)rem);
        bitmap_store32_masked(out_data + w, dbits, m);
        if (out_valid) bitmap_store32_masked(out_valid + w, vbits, m);
        nulls += __popc(~vbits & m);
      }
    }
  }
  if (lane < kHUnroll && nulls && null_count) atomicAdd(null_count, nulls);
}

// the table that holds the complete result: `big` is the full-size table of an overflowed call (slots == NULL when the
// call has only one table)
__device__ __forceinline__ HashTable complete_table(const HashTable& small_t, const HashTable& big_t) {
  const bool use_big = big_t.slots && overflowed(small_t);
  HashTable t;
  t.slots = use_big ? big_t.slots : small_t.slots;
  t.mask = use_big ? big_t.mask : small_t.mask;
  t.shift = use_big ? big_t.shift : small_t.shift;
  t.cap = kNoCap;
  t.special = use_big ? big_t.special : small_t.special;
  return t;
}

// unique: row i is kept iff it is the first row of its key (or, with `count_null`, the first null row; dictionary_encode's
// mask mode gives nulls no dictionary entry).
template <typename V>
__global__ void __launch_bounds__(kHThreads)
unique_mark_kernel(const V* __restrict__ vals, const uint8_t* __restrict__ valid, int64_t off, int64_t n, const HashTable small_t,
                   const HashTable big_t, bool count_null, uint32_t* __restrict__ keep) {
  __shared__ unsigned long long s_cache[kHWarps][kWarpCacheSlots];
  const HashTable t = complete_table(small_t, big_t);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long* cache = s_cache[warp];
  for (int i = lane; i < kWarpCacheSlots; i += 32) cache[i] = kEmptyKey;
  __syncwarp();
  const unsigned first_ones = t.special[0], first_null = t.special[1];
  const int64_t n_words = (n + 31) >> 5;
  const int64_t warp0 = ((int64_t)blockIdx.x * kHThreads + threadIdx.x) >> 5;
  const int64_t warps = ((int64_t)gridDim.x * kHThreads) >> 5;
  for (int64_t w0 = warp0 * kHUnroll; w0 < n_words; w0 += warps * kHUnroll) {
    V x[kHUnroll];
    int kind[kHUnroll];
    if (!valid && ((w0 + kHUnroll) << 5) <= n) {         // interior, no nulls: unconditional loads
      const V* __restrict__ p = vals + off + (w0 << 5) + lane;
#pragma unroll
      for (int k = 0; k < kHUnroll; ++k) { x[k] = __ldcs(p + 32 * k); kind[k] = 1; }
    } else {
#pragma unroll
      for (int k = 0; k < kHUnroll; ++k) {
        const int64_t i = ((w0 + k) << 5) + lane;
        kind[k] = i < n ? ((valid && !bit_is_set(valid, off + i)) ? 2 : 1) : 0;
        x[k] = kind[k] == 1 ? __ldcs(vals + off + i) : V(0);
      }
    }
#pragma unroll
    for (int k = 0; k < kHUnroll; ++k) {
      const int64_t w = w0 + k;
      if (w >= n_words) break;   // warp-uniform
      const unsigned row = (unsigned)((w << 5) + lane);
      const unsigned long long key = (unsigned long long)x[k];
      const int cs = warp_cache_slot(key);
      const bool ones = sizeof(V) == 8 && key == kEmptyKey;
      bool kp = false;
      if (kind[k] == 2) kp = count_null && first_null == row;
      else if (kind[k] == 1 && ones) kp = first_ones == row;
      const bool go = kind[k] == 1 && !ones && cache[cs] != key;   // a cached key sits at a lower row: not first
      __syncwarp();
      if (go) { kp = table_first_row(t, key) == row; atomicExch(&cache[cs], key); }
      __syncwarp();
      const uint32_t bits = __ballot_sync(0xffffffffu, kp);
      if (lane == 0) keep[w] = bits;
    }
  }
}

struct TableMem {
  void* block = nullptr;
  size_t bytes = 0;
  HashTable t{};
  // slots = the power of two >= max(2 * entries, min_slots)
  ag_status alloc(int64_t entries, unsigned long long min_slots, unsigned cap, cudaStream_t st) {
    unsigned long long slots = 1024;
    while (slots < (unsigned long long)entries * 2 || slots < min_slots) slots <<= 1;
    int bits = 0;
    while ((1ull << bits) < slots) ++bits;
    bytes = slots * sizeof(Slot) + 64;
    AG_TRY(dev_alloc_async(&block, bytes, st));
    t.slots = reinterpret_cast<Slot*>(block);
    t.special = reinterpret_cast<unsigned*>(reinterpret_cast<char*>(block) + slots * sizeof(Slot));
    t.mask = slots - 1;
    t.shift = 64 - bits;
    t.cap = cap;
    return AG_OK;
  }
  // every key free, every first row = none, special = {none, none, 0xffffffff (the counter: +1 per key wraps to 0 first), not raised}
  ag_status clear(cudaStream_t st, const unsigned* run_if = nullptr) {
    if (!run_if) { AG_CUDA_TRY(cudaMemsetAsync(block, 0xff, bytes, st)); return AG_OK; }
    table_clear_kernel<<<grid_for((int64_t)(bytes / 16), kHThreads * 8, 8), kHThreads, 0, st>>>(reinterpret_cast<uint4*>(block), (int64_t)(bytes / 16), run_if);
    return check_launch("table_clear_kernel");
  }
  void release(cudaStream_t st) { if (block) cudaFreeAsync(block, st); block = nullptr; }
};

template <typename V>
static ag_status is_in_t(const void* vals, const uint8_t* valid, int64_t off, int64_t n, const void* set, const uint8_t* set_valid, int64_t set_off,
                         int64_t set_n, int null_behavior, uint8_t* out_data, uint8_t* out_valid, int64_t* d_null_count, cudaStream_t st) {
  constexpr bool kSmall = sizeof(V) <= 2;
  TableMem tm;
  // 1-/2-byte values: a 1024-slot block whose first 8 KB hold the membership bitmap (zeroed), `special` behind it as usual
  // others: load factor <= 1/4 while the table still fits the shared-memory copy (a 1000-value set: 4096 slots = 32 KB,
  // six blocks per SM), <= 1/2 beyond
  unsigned long long min_slots = 1024;
  if (!kSmall) { while (min_slots < (unsigned long long)set_n * 4 && min_slots < (unsigned long long)kIsInSmemSlots) min_slots <<= 1; }
  AG_TRY(tm.alloc(kSmall ? 0 : set_n, min_slots, kNoCap, st));
  ag_status rc = tm.clear(st);
  unsigned* bits = reinterpret_cast<unsigned*>(tm.block);
  do {
    if (rc != AG_OK) break;
    if (kSmall && cudaMemsetAsync(bits, 0, 8192, st) != cudaSuccess) { rc = cuda_fail(cudaGetLastError(), "memset", __FILE__, __LINE__); break; }
    if (set_n > 0) {
      if constexpr (kSmall) set_bitmap_kernel<V><<<grid_for(set_n, kHThreads, 8), kHThreads, 0, st>>>(reinterpret_cast<const V*>(set), set_valid, set_off, set_n, bits, tm.t.special);
      else hash_insert_kernel<V><<<grid_for(set_n, kHThreads * kHUnroll, 8), kHThreads, 0, st>>>(reinterpret_cast<const V*>(set), set_valid, set_off, set_n, tm.t, nullptr);
      if ((rc = check_launch("is_in set kernel")) != AG_OK) break;
    }
    if (d_null_count && cudaMemsetAsync(d_null_count, 0, 8, st) != cudaSuccess) { rc = cuda_fail(cudaGetLastError(), "memset", __FILE__, __LINE__); break; }
    uint32_t* od = reinterpret_cast<uint32_t*>(out_data);
    uint32_t* ov = reinterpret_cast<uint32_t*>(out_valid);
    unsigned long long* nc = reinterpret_cast<unsigned long long*>(d_null_count);
    const V* v = reinterpret_cast<const V*>(vals);
    if constexpr (kSmall) {
      is_in_kernel<V, kMemberBitmap><<<grid_for(n, kHThreads * kHUnroll, 8), kHThreads, 8192, st>>>(v, valid, off, n, tm.t, bits, null_behavior, od, ov, nc);
    } else if (tm.t.mask < (unsigned long long)kIsInSmemSlots) {
      const int smem = (int)((tm.t.mask + 1) * 8);
      static std::atomic<unsigned> attr_set{0u};   // per V, one bit per device
      if ((rc = ensure_dynamic_smem((const void*)is_in_kernel<V, kMemberSmem>, kIsInSmemSlots * 8, &attr_set)) != AG_OK) break;
      const int per_sm = smem > 32768 ? 3 : (smem > 16384 ? 6 : 8);
      is_in_kernel<V, kMemberSmem><<<grid_for(n, kHThreads * kHUnroll, per_sm), kHThreads, smem, st>>>(v, valid, off, n, tm.t, nullptr, null_behavior, od, ov, nc);
    } else {
      is_in_kernel<V, kMemberTable><<<grid_for(n, kHThreads * kHUnroll, 8), kHThreads, 0, st>>>(v, valid, off, n, tm.t, nullptr, null_behavior, od, ov, nc);
    }
    rc = check_launch("is_in_kernel");
  } while (0);
  tm.release(st);
  return rc;
}

ag_status is_in_dev(int bit_width, const void* vals, const uint8_t* valid, int64_t off, int64_t n, const void* set, const uint8_t* set_valid,
                    int64_t set_off, int64_t set_n, int null_behavior, uint8_t* out_data, uint8_t* out_valid, int64_t* d_null_count, cudaStream_t st) {
  if (n < 0 || set_n < 0 || off < 0 || set_off < 0) AG_FAIL(AG_ERR_INVALID, "is_in: negative length or offset");
  if (null_behavior < 0 || null_behavior > 3) AG_FAIL(AG_ERR_INVALID, "is_in: bad null matching behaviour %d", null_behavior);
  if (n == 0) return AG_OK;
  if (!vals || !out_data || (set_n > 0 && !set)) AG_FAIL(AG_ERR_INVALID, "is_in: NULL values / value set / output");
  if ((reinterpret_cast<uintptr_t>(out_data) & 3) || (reinterpret_cast<uintptr_t>(out_valid) & 3)) AG_FAIL(AG_ERR_INVALID, "is_in: output bitmaps must be 4-byte aligned");
  if (set_n >= (1ll << 31)) AG_FAIL(AG_ERR_NOT_IMPLEMENTED, "is_in: value set too large");
  switch (bit_width) {
    case 8: return is_in_t<uint8_t>(vals, valid, off, n, set, set_valid, set_off, set_n, null_behavior, out_data, out_valid, d_null_count, st);
    case 16: return is_in_t<uint16_t>(vals, valid, off, n, set, set_valid, set_off, set_n, null_behavior, out_data, out_valid, d_null_count, st);
    case 32: return is_in_t<uint32_t>(vals, valid, off, n, set, set_valid, set_off, set_n, null_behavior, out_data, out_valid, d_null_count, st);
    case 64: return is_in_t<unsigned long long>(vals, valid, off, n, set, set_valid, set_off, set_n, null_behavior, out_data, out_valid, d_null_count, st);
    default: AG_FAIL(AG_ERR_NOT_IMPLEMENTED, "is_in: fixed-width values of 1/2/4/8 bytes only (got %d bits)", bit_width);
  }
}

// columns above `small_rows` try a table of `small_slots` slots (4M x 16 B = 64 MB: L2-resident) first
static std::atomic<long long> g_unique_small_rows{1ll << 21};
static std::atomic<long long> g_unique_small_slots{1ll << 22};

// Insert pass of unique / dictionary_encode: every key's lowest row, in the small table or (after an overflow, decided
// on the device) in the full-size one, plus the first-row bitmap `keep` (n/32 words) for the mark pass.
struct FirstRowTables {
  TableMem small_t, big_t;
  uint32_t* keep = nullptr;
  template <typename V>
  ag_status build(const V* v, const uint8_t* valid, int64_t off, int64_t n, int grid, cudaStream_t st) {
    const bool two = n > g_unique_small_rows.load(std::memory_order_relaxed);
    const unsigned long long small_slots = (unsigned long long)g_unique_small_slots.load(std::memory_order_relaxed);
    if (two) AG_TRY(small_t.alloc(0, small_slots, (unsigned)(small_slots / 2), st));
    else AG_TRY(small_t.alloc(n, 1024, kNoCap, st));
    AG_TRY(small_t.clear(st));
    if (two) AG_TRY(big_t.alloc(n, 1024, kNoCap, st));
    AG_TRY(dev_alloc_async((void**)&keep, (size_t)((n + 31) / 32) * 4 + 64, st));
    hash_insert_kernel<V><<<grid, kHThreads, 0, st>>>(v, valid, off, n, small_t.t, nullptr);
    AG_TRY(check_launch("hash_insert_kernel"));
    if (two) {
      const unsigned* raised = small_t.t.special + 3;
      AG_TRY(big_t.clear(st, raised));
      hash_insert_kernel<V><<<grid, kHThreads, 0, st>>>(v, valid, off, n, big_t.t, raised);
      AG_TRY(check_launch("hash_insert_kernel"));
    }
    return AG_OK;
  }
  void release(cudaStream_t st) {
    if (keep) cudaFreeAsync(keep, st);
    keep = nullptr;
    small_t.release(st);
    big_t.release(st);
  }
};

template <typename V>
static ag_status unique_t(int bit_width, const void* vals, const uint8_t* valid, int64_t off, int64_t n, void* out, uint8_t* out_valid,
                          int64_t capacity, int64_t* d_out_len, cudaStream_t st) {
  FirstRowTables tabs;
  ag_status rc = AG_OK;
  do {
    const V* v = reinterpret_cast<const V*>(vals);
    const int grid = grid_for(n, kHThreads * kHUnroll, 8);
    if ((rc = tabs.build(v, valid, off, n, grid, st)) != AG_OK) break;
    uint32_t* keep = tabs.keep;
    unique_mark_kernel<V><<<grid, kHThreads, 0, st>>>(v, valid, off, n, tabs.small_t.t, tabs.big_t.t, true, keep);
    if ((rc = check_launch("unique_mark_kernel")) != AG_OK) break;
    if (out_valid) {
      if (cudaMemsetAsync(out_valid, 0, (size_t)((capacity + 31) / 32) * 4, st) != cudaSuccess) { rc = cuda_fail(cudaGetLastError(), "memset", __FILE__, __LINE__); break; }
    }
    rc = filter_primitive_dev(bit_width, vals, valid, off, reinterpret_cast<const uint8_t*>(keep), nullptr, 0, n, AG_DROP_NULLS, out, out_valid,
                              capacity, d_out_len, st);
  } while (0);
  tabs.release(st);
  return rc;
}

ag_status unique_dev(int bit_width, const void* vals, const uint8_t* valid, int64_t off, int64_t n, void* out, uint8_t* out_valid, int64_t capacity,
                     int64_t* d_out_len, cudaStream_t st) {
  if (n < 0 || off < 0 || capacity < 0) AG_FAIL(AG_ERR_INVALID, "unique: negative length or offset");
  if (!d_out_len) AG_FAIL(AG_ERR_INVALID, "unique: NULL length word");
  if (n == 0) { AG_CUDA_TRY(cudaMemsetAsync(d_out_len, 0, sizeof(int64_t), st)); return AG_OK; }
  if (!vals || (!out && capacity > 0)) AG_FAIL(AG_ERR_INVALID, "unique: NULL values/output");
  if (valid && !out_valid && capacity > 0) AG_FAIL(AG_ERR_INVALID, "unique: an input with a validity bitmap needs an output validity bitmap");
  if (n >= (1ll << 31)) AG_FAIL(AG_ERR_NOT_IMPLEMENTED, "unique: more than 2^31-1 rows per call");
  switch (bit_width) {
    case 8: return unique_t<uint8_t>(bit_width, vals, valid, off, n, out, out_valid, capacity, d_out_len, st);
    case 16: return unique_t<uint16_t>(bit_width, vals, valid, off, n, out, out_valid, capacity, d_out_len, st);
    case 32: return unique_t<uint32_t>(bit_width, vals, valid, off, n, out, out_valid, capacity, d_out_len, st);
    case 64: return unique_t<unsigned long long>(bit_width, vals, valid, off, n, out, out_valid, capacity, d_out_len, st);
    default: AG_FAIL(AG_ERR_NOT_IMPLEMENTED, "unique: fixed-width values of 1/2/4/8 bytes only (got %d bits)", bit_width);
  }
}

// ---- dictionary_encode: rank + finalize + encode passes after unique's insert + mark ------------------------------------
constexpr int kRankWordsPerThread = 8;
constexpr int kRankTileWords = kHThreads * kRankWordsPerThread;   // keep words (65536 rows) per rank tile

// exclusive prefix of `x` over the block; *total = the block's sum
template <int kThreads>
__device__ __forceinline__ unsigned block_exclusive_scan(unsigned x, unsigned* total) {
  __shared__ unsigned s_warp[kThreads / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned inc = x;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned y = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += y;
  }
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    unsigned w = lane < kThreads / 32 ? s_warp[lane] : 0u;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned y = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += y;
    }
    if (lane < kThreads / 32) s_warp[lane] = w;
  }
  __syncthreads();
  const unsigned base = warp ? s_warp[warp - 1] : 0u;
  *total = s_warp[kThreads / 32 - 1];
  __syncthreads();   // s_warp is reused by the next call
  return base + inc - x;
}

// number of first rows per rank tile
__global__ void __launch_bounds__(kHThreads)
dict_rank_count_kernel(const uint32_t* __restrict__ keep, int64_t n_words, unsigned* __restrict__ tile_sums) {
  const int64_t w0 = (int64_t)blockIdx.x * kRankTileWords + (int64_t)threadIdx.x * kRankWordsPerThread;
  unsigned c = 0;
#pragma unroll
  for (int k = 0; k < kRankWordsPerThread; ++k) c += w0 + k < n_words ? __popc(keep[w0 + k]) : 0u;
  unsigned total;
  block_exclusive_scan<kHThreads>(c, &total);
  if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}

// tile_sums -> exclusive tile offsets (in place); counts[0] = dictionary length
constexpr int kRankScanThreads = 1024;
__global__ void __launch_bounds__(kRankScanThreads)
dict_rank_scan_kernel(unsigned* __restrict__ tile_sums, int64_t tiles, long long* __restrict__ counts) {
  unsigned carry = 0;
  for (int64_t b = 0; b < tiles; b += kRankScanThreads) {
    const int64_t i = b + threadIdx.x;
    const unsigned x = i < tiles ? tile_sums[i] : 0u;
    unsigned total;
    const unsigned ex = block_exclusive_scan<kRankScanThreads>(x, &total);
    if (i < tiles) tile_sums[i] = carry + ex;
    carry += total;
  }
  if (threadIdx.x == 0) counts[0] = (long long)carry;
}

// slot of a key that is in the table
__device__ __forceinline__ Slot* table_slot(const HashTable& t, unsigned long long key) {
  unsigned long long h = hash_slot(key, t.shift);
  while (true) {
    const unsigned long long k = t.slots[h].key;
    if (k == key) return t.slots + h;
    if (k == kEmptyKey) return nullptr;
    h = (h + 1) & t.mask;
  }
}

// one lane per first row: dict[rank] = its value, the rank goes to the key's slot (or special[4] / special[5])
template <typename V>
__global__ void __launch_bounds__(kHThreads)
dict_finalize_kernel(const V* __restrict__ vals, const uint8_t* __restrict__ valid, int64_t off, const HashTable small_t,
                     const HashTable big_t, const uint32_t* __restrict__ keep, int64_t n_words, const unsigned* __restrict__ tile_off,
                     V* __restrict__ dict, uint32_t* __restrict__ dict_valid, int64_t dict_capacity) {
  const HashTable t = complete_table(small_t, big_t);
  const int64_t w0 = (int64_t)blockIdx.x * kRankTileWords + (int64_t)threadIdx.x * kRankWordsPerThread;
  uint32_t words[kRankWordsPerThread];
  unsigned c = 0;
#pragma unroll
  for (int k = 0; k < kRankWordsPerThread; ++k) {
    words[k] = w0 + k < n_words ? keep[w0 + k] : 0u;
    c += __popc(words[k]);
  }
  unsigned total;
  unsigned rank = tile_off[blockIdx.x] + block_exclusive_scan<kHThreads>(c, &total);
#pragma unroll
  for (int k = 0; k < kRankWordsPerThread; ++k) {
    uint32_t bits = words[k];
    while (bits) {
      const int64_t row = ((w0 + k) << 5) + (__ffs(bits) - 1);
      bits &= bits - 1;
      const bool is_null = valid && !bit_is_set(valid, off + row);
      const V x = is_null ? V(0) : vals[off + row];
      if ((int64_t)rank < dict_capacity) {
        dict[rank] = x;
        if (is_null && dict_valid) atomicAnd(&dict_valid[rank >> 5], ~(1u << (rank & 31)));
      }
      const unsigned long long key = (unsigned long long)x;
      if (is_null) t.special[5] = rank;
      else if (sizeof(V) == 8 && key == kEmptyKey) t.special[4] = rank;
      else table_slot(t, key)->rank = rank;
      ++rank;
    }
  }
}

// rank of a key that is in the table: key, first row and rank arrive in one 16-byte load
__device__ __forceinline__ unsigned table_rank(const HashTable& t, unsigned long long key) {
  unsigned long long h = hash_slot(key, t.shift);
  while (true) {
    const ulonglong2 raw = *reinterpret_cast<const ulonglong2*>(t.slots + h);
    if (raw.x == key) return (unsigned)(raw.y >> 32);
    if (raw.x == kEmptyKey) return 0u;
    h = (h + 1) & t.mask;
  }
}

// one int32 index per row.  Mask mode: a null row gets index 0 and a cleared validity bit; encode mode: the null entry's
// rank.  The table is read-only here, so a per-warp cache of (key, rank) pairs is always right.
template <typename V>
__global__ void __launch_bounds__(kHThreads)
dict_encode_kernel(const V* __restrict__ vals, const uint8_t* __restrict__ valid, int64_t off, int64_t n, const HashTable small_t,
                   const HashTable big_t, bool mask_nulls, int32_t* __restrict__ indices, uint32_t* __restrict__ indices_valid,
                   unsigned long long* __restrict__ null_count) {
  __shared__ unsigned long long s_key[kHWarps][kWarpCacheSlots];
  __shared__ unsigned s_rank[kHWarps][kWarpCacheSlots];
  const HashTable t = complete_table(small_t, big_t);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long* ckey = s_key[warp];
  unsigned* crank = s_rank[warp];
  for (int i = lane; i < kWarpCacheSlots; i += 32) ckey[i] = kEmptyKey;
  __syncwarp();
  const unsigned ones_rank = t.special[4], null_rank = mask_nulls ? 0u : t.special[5];
  const int64_t n_words = (n + 31) >> 5;
  const int64_t warp0 = ((int64_t)blockIdx.x * kHThreads + threadIdx.x) >> 5;
  const int64_t warps = ((int64_t)gridDim.x * kHThreads) >> 5;
  unsigned long long nulls = 0;
  for (int64_t w0 = warp0 * kHUnroll; w0 < n_words; w0 += warps * kHUnroll) {
    V x[kHUnroll];
    int kind[kHUnroll];                                  // 0 nothing, 1 value, 2 null
    if (!valid && ((w0 + kHUnroll) << 5) <= n) {
      const V* __restrict__ p = vals + off + (w0 << 5) + lane;
#pragma unroll
      for (int k = 0; k < kHUnroll; ++k) { x[k] = __ldcs(p + 32 * k); kind[k] = 1; }
    } else {
#pragma unroll
      for (int k = 0; k < kHUnroll; ++k) {
        const int64_t i = ((w0 + k) << 5) + lane;
        kind[k] = i < n ? ((valid && !bit_is_set(valid, off + i)) ? 2 : 1) : 0;
        x[k] = kind[k] == 1 ? __ldcs(vals + off + i) : V(0);
      }
    }
#pragma unroll
    for (int k = 0; k < kHUnroll; ++k) {
      const int64_t w = w0 + k;
      if (w >= n_words) break;   // warp-uniform
      const unsigned long long key = (unsigned long long)x[k];
      const int cs = warp_cache_slot(key);
      const bool ones = sizeof(V) == 8 && key == kEmptyKey;
      unsigned idx = kind[k] == 2 ? null_rank : ones_rank;
      bool miss = false;
      if (kind[k] == 1 && !ones) {
        if (ckey[cs] == key) idx = crank[cs];
        else miss = true;
      }
      __syncwarp();
      if (miss) { idx = table_rank(t, key); atomicExch(&ckey[cs], key); }   // several lanes may share a slot: one whole key wins
      __syncwarp();
      if (miss && ckey[cs] == key) crank[cs] = idx;                        // every lane holding the winning key writes the same rank
      __syncwarp();
      if (kind[k] != 0) __stcs(indices + (w << 5) + lane, (int32_t)idx);
      if (indices_valid) {
        const uint32_t vbits = __ballot_sync(0xffffffffu, kind[k] == 1 || (kind[k] == 2 && !mask_nulls));
        if (lane == 0) {
          indices_valid[w] = vbits;
          const int64_t rem = n - (w << 5);
          nulls += __popc(~vbits & (rem >= 32 ? 0xffffffffu : bit_range_mask(0, (int)rem)));
        }
      }
    }
  }
  if (lane == 0 && nulls) atomicAdd(null_count, nulls);
}

template <typename V>
static ag_status dictionary_encode_t(const void* vals, const uint8_t* valid, int64_t off, int64_t n, int null_encoding, int32_t* indices,
                                     uint8_t* indices_valid, void* dict, uint8_t* dict_valid, int64_t dict_capacity, int64_t* d_counts,
                                     cudaStream_t st) {
  FirstRowTables tabs;
  unsigned* tile_off = nullptr;
  ag_status rc = AG_OK;
  const bool mask_nulls = null_encoding == AG_NULL_ENCODING_MASK;
  do {
    const V* v = reinterpret_cast<const V*>(vals);
    const int grid = grid_for(n, kHThreads * kHUnroll, 8);
    const int64_t n_words = (n + 31) / 32;
    const int64_t tiles = (n_words + kRankTileWords - 1) / kRankTileWords;
    if (cudaMemsetAsync(d_counts, 0, 2 * sizeof(int64_t), st) != cudaSuccess) { rc = cuda_fail(cudaGetLastError(), "memset", __FILE__, __LINE__); break; }
    if ((rc = tabs.build(v, valid, off, n, grid, st)) != AG_OK) break;
    if ((rc = dev_alloc_async((void**)&tile_off, (size_t)tiles * 4 + 64, st)) != AG_OK) break;
    unique_mark_kernel<V><<<grid, kHThreads, 0, st>>>(v, valid, off, n, tabs.small_t.t, tabs.big_t.t, !mask_nulls, tabs.keep);
    if ((rc = check_launch("unique_mark_kernel")) != AG_OK) break;
    dict_rank_count_kernel<<<(unsigned)tiles, kHThreads, 0, st>>>(tabs.keep, n_words, tile_off);
    if ((rc = check_launch("dict_rank_count_kernel")) != AG_OK) break;
    dict_rank_scan_kernel<<<1, kRankScanThreads, 0, st>>>(tile_off, tiles, reinterpret_cast<long long*>(d_counts));
    if ((rc = check_launch("dict_rank_scan_kernel")) != AG_OK) break;
    if (dict_valid && dict_capacity > 0) {
      if (cudaMemsetAsync(dict_valid, 0xff, (size_t)((dict_capacity + 31) / 32) * 4, st) != cudaSuccess) { rc = cuda_fail(cudaGetLastError(), "memset", __FILE__, __LINE__); break; }
    }
    dict_finalize_kernel<V><<<(unsigned)tiles, kHThreads, 0, st>>>(v, valid, off, tabs.small_t.t, tabs.big_t.t, tabs.keep, n_words, tile_off,
                                                                  reinterpret_cast<V*>(dict), reinterpret_cast<uint32_t*>(dict_valid), dict_capacity);
    if ((rc = check_launch("dict_finalize_kernel")) != AG_OK) break;
    dict_encode_kernel<V><<<grid, kHThreads, 0, st>>>(v, valid, off, n, tabs.small_t.t, tabs.big_t.t, mask_nulls, indices,
                                                      reinterpret_cast<uint32_t*>(indices_valid), reinterpret_cast<unsigned long long*>(d_counts + 1));
    rc = check_launch("dict_encode_kernel");
  } while (0);
  if (tile_off) cudaFreeAsync(tile_off, st);
  tabs.release(st);
  return rc;
}

ag_status dictionary_encode_dev(int bit_width, const void* vals, const uint8_t* valid, int64_t off, int64_t n, int null_encoding, int32_t* indices,
                                uint8_t* indices_valid, void* dict, uint8_t* dict_valid, int64_t dict_capacity, int64_t* d_counts, cudaStream_t st) {
  if (n < 0 || off < 0 || dict_capacity < 0) AG_FAIL(AG_ERR_INVALID, "dictionary_encode: negative length, offset or capacity");
  if (null_encoding != AG_NULL_ENCODING_MASK && null_encoding != AG_NULL_ENCODING_ENCODE)
    AG_FAIL(AG_ERR_INVALID, "dictionary_encode: invalid null encoding behavior %d", null_encoding);
  if (!d_counts) AG_FAIL(AG_ERR_INVALID, "dictionary_encode: NULL counts word");
  if (n == 0) { AG_CUDA_TRY(cudaMemsetAsync(d_counts, 0, 2 * sizeof(int64_t), st)); return AG_OK; }
  if (!vals || !indices || (!dict && dict_capacity > 0)) AG_FAIL(AG_ERR_INVALID, "dictionary_encode: NULL values / indices / dictionary");
  if (valid && null_encoding == AG_NULL_ENCODING_MASK && !indices_valid)
    AG_FAIL(AG_ERR_INVALID, "dictionary_encode: an input with a validity bitmap needs an indices validity bitmap in mask mode");
  if (valid && null_encoding == AG_NULL_ENCODING_ENCODE && !dict_valid && dict_capacity > 0)
    AG_FAIL(AG_ERR_INVALID, "dictionary_encode: an input with a validity bitmap needs a dictionary validity bitmap in encode mode");
  if ((reinterpret_cast<uintptr_t>(indices) & 3) || (reinterpret_cast<uintptr_t>(indices_valid) & 3) || (reinterpret_cast<uintptr_t>(dict_valid) & 3))
    AG_FAIL(AG_ERR_INVALID, "dictionary_encode: indices and bitmaps must be 4-byte aligned");
  if (n >= (1ll << 31)) AG_FAIL(AG_ERR_NOT_IMPLEMENTED, "dictionary_encode: more than 2^31-1 rows per call");
  switch (bit_width) {
    case 8: return dictionary_encode_t<uint8_t>(vals, valid, off, n, null_encoding, indices, indices_valid, dict, dict_valid, dict_capacity, d_counts, st);
    case 16: return dictionary_encode_t<uint16_t>(vals, valid, off, n, null_encoding, indices, indices_valid, dict, dict_valid, dict_capacity, d_counts, st);
    case 32: return dictionary_encode_t<uint32_t>(vals, valid, off, n, null_encoding, indices, indices_valid, dict, dict_valid, dict_capacity, d_counts, st);
    case 64: return dictionary_encode_t<unsigned long long>(vals, valid, off, n, null_encoding, indices, indices_valid, dict, dict_valid, dict_capacity, d_counts, st);
    default: AG_FAIL(AG_ERR_NOT_IMPLEMENTED, "dictionary_encode: fixed-width values of 1/2/4/8 bytes only (got %d bits)", bit_width);
  }
}

}  // namespace ag

using namespace ag;

extern "C" ag_status ag_is_in_dev(int bit_width, const void* d_vals, const uint8_t* d_valid, int64_t offset, int64_t n, const void* d_set,
                                  const uint8_t* d_set_valid, int64_t set_offset, int64_t set_n, int null_behavior, uint8_t* d_out_data,
                                  uint8_t* d_out_valid, int64_t* d_null_count, ag_stream_t s) {
  AG_TRY(ensure_init());
  return is_in_dev(bit_width, d_vals, d_valid, offset, n, d_set, d_set_valid, set_offset, set_n, null_behavior, d_out_data, d_out_valid, d_null_count,
                   resolve_stream(s));
}

extern "C" ag_status ag_unique_set_policy(int64_t small_rows, int64_t small_slots) {
  if (small_rows < 0 || small_slots < 0) AG_FAIL(AG_ERR_INVALID, "ag_unique_set_policy: negative argument");
  if (small_slots && (small_slots < 1024 || small_slots > (1ll << 31) || (small_slots & (small_slots - 1))))
    AG_FAIL(AG_ERR_INVALID, "ag_unique_set_policy: small_slots must be a power of two in [1024, 2^31]");
  g_unique_small_rows.store(small_rows ? small_rows : (1ll << 21), std::memory_order_relaxed);
  g_unique_small_slots.store(small_slots ? small_slots : (1ll << 22), std::memory_order_relaxed);
  return AG_OK;
}

extern "C" ag_status ag_unique_dev(int bit_width, const void* d_vals, const uint8_t* d_valid, int64_t offset, int64_t n, void* d_out,
                                   uint8_t* d_out_valid, int64_t capacity, int64_t* d_out_len, ag_stream_t s) {
  AG_TRY(ensure_init());
  return unique_dev(bit_width, d_vals, d_valid, offset, n, d_out, d_out_valid, capacity, d_out_len, resolve_stream(s));
}

extern "C" ag_status ag_dictionary_encode_dev(int bit_width, const void* d_vals, const uint8_t* d_valid, int64_t offset, int64_t n, int null_encoding,
                                              int32_t* d_indices, uint8_t* d_indices_valid, void* d_dict, uint8_t* d_dict_valid,
                                              int64_t dict_capacity, int64_t* d_counts, ag_stream_t s) {
  AG_TRY(ensure_init());
  return dictionary_encode_dev(bit_width, d_vals, d_valid, offset, n, null_encoding, d_indices, d_indices_valid, d_dict, d_dict_valid,
                               dict_capacity, d_counts, resolve_stream(s));
}
