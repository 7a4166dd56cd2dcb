// probe.cuh -- seq.kmer.pos: match query windows against the index.
//
// Replaces seq_kmer_positions (src/kmer_pos.c:110-136).  kmer_pos/kh_get (:55-60) is one random DRAM
// probe per query window in the reference and stays one here: the distinct keys are put (once per
// index, on first use) into an open-addressing table of 16-byte slots {key, first position slot,
// count}, two slots per 32-byte sector, load <= 0.5, so a lookup is one sector read in the common
// case and needs no second access for the list length.  pair_positions_push (:101-108) becomes a count
// pass, a chained 64-bit scan and a load-balanced emit, so rows come out ordered by query position then
// index position exactly as the reference pushes them.
#pragma once
#include "common.cuh"
#include "lookback.cuh"
#include "windows.cuh"
#include "csr.cuh"

namespace kmg {

struct QueryStats {
  uint64_t H;   // query windows that hit
  uint64_t M;   // result rows
};

// ---- key table -------------------------------------------------------------------------------------------
// slot = uint4 {key lo, key hi, start, count}; count == 0 marks an empty slot (a stored k-mer has >= 1
// position).  Two slots form a 32-byte bucket = one memory request; a key lives in the first bucket at or
// after its home bucket that had room, so a bucket with an empty slot ends the search.  Measured on B200
// (tools/micro/gups.cu, profiles/): a random read costs a whole 128-byte line of DRAM traffic whatever its
// size and the rate is bound by requests, 46 G/s for 32-byte requests = HBM peak in lines; an overflow
// bucket is in the same line three times out of four and then comes from L2.
constexpr int BUCKET_SLOTS = 2;

__device__ __forceinline__ uint64_t hash64(uint64_t x) {
  x ^= x >> 33; x *= 0xff51afd7ed558ccdULL;
  x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL;
  x ^= x >> 33;
  return x;
}

// Home bucket of a key.  hbits == 0: hash64(key) & (nb - 1), nb a power of two (table of an index in ascending key order,
// filled by 128-bit CAS).  hbits > 0: floor(low hbits bits of mix64(key) / 2^hbits * nb), any nb: MONOTONE in the order of a
// grouped index (records sorted on those bits), so its table is written front to back by a streaming kernel.
struct KeyHash {
  uint4 *slots;
  uint64_t nb;      // buckets
  int hbits;
  __device__ __forceinline__ uint64_t bucket(uint64_t key) const {
    const uint64_t h = hash64(key);                        // == mix64(key)
    return hbits ? __umul64hi(h << (64 - hbits), nb) : (h & (nb - 1));
  }
  __device__ __forceinline__ uint64_t next(uint64_t b) const { return b + 1 == nb ? 0 : b + 1; }
};

// compare a 16-byte slot with all-zero and swap `desired` in (one 128-bit CAS, sm_90+); true if it was empty
__device__ __forceinline__ bool claim_slot(uint4 *slot, uint4 desired) {
  uint64_t olo, ohi;
  const uint64_t dlo = (uint64_t)desired.x | ((uint64_t)desired.y << 32), dhi = (uint64_t)desired.z | ((uint64_t)desired.w << 32);
  asm volatile(
      "{\n\t.reg .b128 cmp, val, old;\n\t"
      "mov.b128 cmp, {%3, %3};\n\t"
      "mov.b128 val, {%4, %5};\n\t"
      "atom.relaxed.gpu.global.cas.b128 old, [%2], cmp, val;\n\t"
      "mov.b128 {%0, %1}, old;\n\t}"
      : "=l"(olo), "=l"(ohi) : "l"(slot), "l"((uint64_t)0), "l"(dlo), "l"(dhi) : "memory");
  return olo == 0 && ohi == 0;
}

// skip_home: the home bucket is known to be full (overflow of the streamed build): start at the next one
__device__ __forceinline__ void cas_insert(const KeyHash &kh, uint64_t key, uint32_t start, uint32_t count, uint64_t b, bool skip_home) {
  const uint4 rec = make_uint4((uint32_t)key, (uint32_t)(key >> 32), start, count);
  if (skip_home) b = kh.next(b);
  bool placed = false;
  while (!placed) {
#pragma unroll
    for (int j = 0; j < BUCKET_SLOTS; ++j)
      if (!placed) placed = claim_slot(kh.slots + b * BUCKET_SLOTS + j, rec);
    b = kh.next(b);
  }
}

// Slot payloads {z, w} (w != 0: the slot is taken).  Position index: {first position slot, list length}.
struct IndexPayload {
  const uint32_t *ustart;
  __device__ __forceinline__ uint2 operator()(uint64_t u) const { const uint32_t s = ustart[u]; return make_uint2(s, ustart[u + 1] - s); }
};
// Count table (U x source_n matrix): {row u, count} with one column (a k-mer in the table was counted, so count >= 1),
// {row u, 1} with several (the lookup then gathers the row).
struct CountPayload {
  const int32_t *counts;
  int source_n;
  __device__ __forceinline__ uint2 operator()(uint64_t u) const { return make_uint2((uint32_t)u, source_n == 1 ? (uint32_t)counts[u] : 1u); }
};

// Distinct keys only: one 128-bit CAS claims a slot and fills it (a stored slot is never all-zero: w >= 1).
// overflow_only (tables written by hash_stream_kernel): insert only a bucket's third and later k-mers, found by the same
// test as there (the two k-mers before it share its home bucket).
template <class Payload>
__global__ void hash_insert_kernel(const uint64_t *__restrict__ ukeys, const Payload pay, uint64_t U, KeyHash kh,
                                   const bool overflow_only) {
  for (uint64_t u = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; u < U; u += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t key = ukeys[u];
    const uint64_t b = kh.bucket(key);
    if (overflow_only) {
      if (u < 2) continue;
      if (kh.bucket(ukeys[u - 1]) != b || kh.bucket(ukeys[u - 2]) != b) continue;
    }
    const uint2 p = pay(u);
    cas_insert(kh, key, p.x, p.y, b, overflow_only);
  }
}

// The overflow phase of a streamed table (hash_stream_kernel below): a bucket's third and later k-mers, ~7 % of all, each
// placed by 128-bit CAS in the first bucket after its home that has room.  A CAS is a ~1.5 us round trip and a k-mer needs
// about two, so the cost is latency x (k-mers per thread in flight): a thread owns ITEMS consecutive k-mers and issues the
// CAS of ALL its pending ones back to back before looking at any result (one k-mer per thread, 93 % of the lanes idle in
// every round: 5.8 ms for 230 M k-mers; this way: see profiles/r02_notes.md).
template <int ITEMS>
__global__ void __launch_bounds__(256)
hash_overflow_kernel(const uint64_t *__restrict__ ukeys, const uint32_t *__restrict__ ustart, uint64_t U, KeyHash kh) {
  const uint64_t u0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * ITEMS;
  if (u0 >= U) return;
  uint64_t key[ITEMS], cur[ITEMS];                         // cur: the bucket tried next
  uint32_t st[ITEMS], cn[ITEMS], slot = 0;                  // slot: bit i = which of the bucket's two slots item i tries next
  uint32_t pend = 0;
  uint64_t bm2 = u0 >= 2 ? kh.bucket(ukeys[u0 - 2]) : ~uint64_t(0), bm1 = u0 >= 1 ? kh.bucket(ukeys[u0 - 1]) : ~uint64_t(0);
#pragma unroll
  for (int i = 0; i < ITEMS; ++i) {
    const uint64_t u = u0 + i;
    key[i] = u < U ? ukeys[u] : 0;
    const uint64_t b = kh.bucket(key[i]);
    if (u < U && u >= 2 && bm1 == b && bm2 == b) {         // the two k-mers before it share its home bucket: it did not fit
      pend |= 1u << i;
      cur[i] = kh.next(b);
      st[i] = ustart[u];
      cn[i] = ustart[u + 1] - st[i];
    }
    bm2 = bm1; bm1 = b;
  }
  while (pend) {
    uint64_t olo[ITEMS], ohi[ITEMS];
#pragma unroll
    for (int i = 0; i < ITEMS; ++i) {
      if ((pend >> i) & 1u) {
        uint4 *sl = kh.slots + cur[i] * BUCKET_SLOTS + ((slot >> i) & 1u);
        const uint64_t dlo = key[i], dhi = (uint64_t)st[i] | ((uint64_t)cn[i] << 32);
        asm volatile(
            "{\n\t.reg .b128 cmp, val, old;\n\t"
            "mov.b128 cmp, {%3, %3};\n\t"
            "mov.b128 val, {%4, %5};\n\t"
            "atom.relaxed.gpu.global.cas.b128 old, [%2], cmp, val;\n\t"
            "mov.b128 {%0, %1}, old;\n\t}"
            : "=l"(olo[i]), "=l"(ohi[i]) : "l"(sl), "l"((uint64_t)0), "l"(dlo), "l"(dhi) : "memory");
      }
    }
#pragma unroll
    for (int i = 0; i < ITEMS; ++i) {
      if ((pend >> i) & 1u) {
        if (olo[i] == 0 && ohi[i] == 0) pend &= ~(1u << i);          // the slot was empty: it is ours now
        else if ((slot >> i) & 1u) { slot &= ~(1u << i); cur[i] = kh.next(cur[i]); }
        else slot |= 1u << i;
      }
    }
  }
}

// Table of a grouped index, written front to back (no memset, no atomics): the k-mers come in ascending home-bucket order,
// so the first k-mer of a bucket (its leader) writes the whole 32-byte bucket -- itself, the next k-mer if it shares the
// bucket, else an empty slot -- and zero-fills the empty buckets before it.  A bucket's third and later k-mers (~10 % at
// one k-mer per bucket on average) are CAS-inserted afterwards by hash_insert_kernel(overflow_only), which places each in
// the first bucket after its home that has room: exactly the table the all-CAS build gives up to slot order.
// The buckets after the last k-mer's are zeroed by the caller.
__global__ void hash_stream_kernel(const uint64_t *__restrict__ ukeys, const uint32_t *__restrict__ ustart, uint64_t U, KeyHash kh,
                                   uint64_t *last_bucket) {
  const uint4 zero = make_uint4(0, 0, 0, 0);
  for (uint64_t u = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; u < U; u += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t key = ukeys[u];
    const uint64_t b = kh.bucket(key);
    const int64_t bp1 = u > 0 ? (int64_t)kh.bucket(ukeys[u - 1]) : -1;
    if (bp1 != (int64_t)b) {                               // leader of bucket b
      const uint32_t s0 = ustart[u], s1 = ustart[u + 1];
      uint4 second = zero;
      if (u + 1 < U) {
        const uint64_t kn = ukeys[u + 1];
        if (kh.bucket(kn) == b) second = make_uint4((uint32_t)kn, (uint32_t)(kn >> 32), s1, ustart[u + 2] - s1);
      }
      kh.slots[b * BUCKET_SLOTS] = make_uint4((uint32_t)key, (uint32_t)(key >> 32), s0, s1 - s0);
      kh.slots[b * BUCKET_SLOTS + 1] = second;
      for (int64_t g = bp1 + 1; g < (int64_t)b; ++g) { kh.slots[g * BUCKET_SLOTS] = zero; kh.slots[g * BUCKET_SLOTS + 1] = zero; }
    }
    if (u + 1 == U) *last_bucket = b;
  }
}

// (start, count) of `key`, or count 0.  s0, s1: the key's home bucket `b`, already loaded.
__device__ __forceinline__ uint2 resolve_key(const KeyHash &kh, uint64_t key, uint64_t b, uint4 s0, uint4 s1) {
  const uint32_t klo = (uint32_t)key, khi = (uint32_t)(key >> 32);
  while (true) {
    if (s0.w != 0 && s0.x == klo && s0.y == khi) return make_uint2(s0.z, s0.w);
    if (s1.w != 0 && s1.x == klo && s1.y == khi) return make_uint2(s1.z, s1.w);
    if (s0.w == 0 || s1.w == 0) return make_uint2(0u, 0u);
    b = kh.next(b);
    ld_stream_sector(kh.slots + b * BUCKET_SLOTS, s0, s1);
  }
}

// ---- pass 1: look every query window up; write (first position slot, count) per window, count 0 = no hit ----
//   FROM_SEQ: windows of the query sequence;  else: pre-encoded keys.
// A thread owns ITEMS consecutive windows (keys roll from one to the next) and has BATCH table requests in
// flight at a time; there is no block-wide step after the tile is packed, so the kernel runs at the
// random-access rate of HBM.
template <int THREADS, int ITEMS, bool FROM_SEQ>
__global__ void __launch_bounds__(THREADS, 4)
probe_lookup_kernel(const SeqView sv, const uint64_t *__restrict__ keys_in, int64_t n_in, const uint64_t *__restrict__ n_dev,
                    const KeyHash kh, uint2 *__restrict__ found, const bool mixed = false) {
  constexpr int TILE = THREADS * ITEMS;
  __shared__ TileCodes<FROM_SEQ ? TILE : 16> tc;
  const unsigned tid = threadIdx.x;
  const int64_t q0 = (int64_t)blockIdx.x * TILE;
  const int64_t total = FROM_SEQ ? sv.nstarts : (n_dev ? min((int64_t)*n_dev, n_in) : n_in);   // the count may only exist on the device
  if (q0 >= total) return;
  const int t0 = tid * ITEMS;
  bool special = false;
  if constexpr (FROM_SEQ) special = tile_pack<TILE, THREADS>(sv, q0, tc);
  constexpr int BATCH = 4;
  static_assert(ITEMS % BATCH == 0, "items in batches");
  uint64_t key = 0;
  const uint64_t kmask = key_mask(FROM_SEQ ? sv.k : 32);
#pragma unroll
  for (int i0 = 0; i0 < ITEMS; i0 += BATCH) {
    uint4 s0[BATCH], s1[BATCH];
    uint64_t kk[BATCH], home[BATCH];
    bool ok[BATCH];
#pragma unroll
    for (int j = 0; j < BATCH; ++j) {
      const int i = i0 + j;
      if constexpr (FROM_SEQ) {
        if (i == 0) key = tile_key<TILE>(tc, t0, sv.k);
        else {                                            // roll in the base at tile position t0 + i + k - 1
          const int p = t0 + i + sv.k - 1;
          const uint32_t code = (tc.codes[p >> 4] >> (30 - 2 * (p & 15))) & 3u;
          key = ((key << 2) | code) & kmask;
        }
        ok[j] = tile_valid<TILE>(sv, tc, q0, t0 + i, special);
      } else {
        ok[j] = q0 + t0 + i < total;
        key = ok[j] ? ld_stream_u64(keys_in + q0 + t0 + i) : 0;
        if (mixed) key = unmix64(key);                      // records of a grouped sharded index carry mix64(key)
      }
      kk[j] = key;
      home[j] = kh.bucket(key);
      if (ok[j]) ld_stream_sector(kh.slots + home[j] * BUCKET_SLOTS, s0[j], s1[j]);
    }
    uint2 r[BATCH];
#pragma unroll
    for (int j = 0; j < BATCH; ++j) r[j] = ok[j] ? resolve_key(kh, kk[j], home[j], s0[j], s1[j]) : make_uint2(0u, 0u);
    if (q0 + t0 + i0 + BATCH <= total) {                  // 32 contiguous bytes per thread
      uint4 *dst = reinterpret_cast<uint4 *>(found + q0 + t0 + i0);
      dst[0] = make_uint4(r[0].x, r[0].y, r[1].x, r[1].y);
      dst[1] = make_uint4(r[2].x, r[2].y, r[3].x, r[3].y);
    } else {
#pragma unroll
      for (int j = 0; j < BATCH; ++j)
        if (q0 + t0 + i0 + j < total) found[q0 + t0 + i0 + j] = r[j];
    }
  }
}

// ---- seq.kmer.depth: per-window counts of the query's k-mers ------------------------------------------------
// Reverse complement of a k-mer key in code space: the k 2-bit codes reversed and each complemented as code ^ 2
// (A0 <-> T2, C1 <-> G3).  Complement all codes, reverse the 64 bits (which also swaps the two bits of every code), swap
// them back, drop the 64 - 2k bits that were above the key.
__device__ __forceinline__ uint64_t revcomp_key(uint64_t key, int k) {
  uint64_t x = __brevll(key ^ 0xAAAAAAAAAAAAAAAAull);
  x = ((x >> 1) & 0x5555555555555555ull) | ((x & 0x5555555555555555ull) << 1);
  return x >> (64 - 2 * k);
}

// Windows [first, first + rows) of the query into out[0, rows * cols): row r = window first + r, cols = source_n with
// MULTI (the k-mer's row of the count matrix, gathered through the slot's row number) else 1 (the slot's count field:
// a position list's length or a one-column count).  A window the window rule drops gets INT32_MIN (R's NA_integer_) in
// every column, an absent k-mer 0.  BOTH: count(key) + count(revcomp(key)), a palindrome once, saturated at INT32_MAX.
// A chunk may start at any window; tile_pack needs 16-aligned tile starts, so tiles start at `first` rounded down to
// 16 and windows in front of the chunk are encoded (the keys roll through them) but neither looked up nor written.
// The lookup is probe_lookup_kernel's: BATCH sectors in flight per thread (twice as many with BOTH), then resolve.
// nb == 0: an empty table, nothing is looked up.  Blocks per SM: the most whose register share holds the variant
// without spills (ptxas: 62 registers forward / one column, ~70 forward / gathered, ~120 both strands).
template <int THREADS, int ITEMS, bool BOTH, bool MULTI>
__global__ void __launch_bounds__(THREADS, BOTH ? 2 : (MULTI ? 3 : 4))
depth_lookup_kernel(const SeqView sv, int64_t first, int64_t rows, const KeyHash kh, const int32_t *__restrict__ counts,
                    const int source_n, int32_t *__restrict__ out) {
  constexpr int TILE = THREADS * ITEMS, BATCH = 4;
  static_assert(ITEMS % BATCH == 0, "items in batches");
  __shared__ TileCodes<TILE> tc;
  const int64_t q0 = (first & ~int64_t(15)) + (int64_t)blockIdx.x * TILE, end = first + rows;
  if (q0 >= end) return;
  const int t0 = threadIdx.x * ITEMS;
  const bool special = tile_pack<TILE, THREADS>(sv, q0, tc);
  const bool have = kh.nb != 0;
  const int cols = MULTI ? source_n : 1;
  const uint64_t kmask = key_mask(sv.k);
  uint64_t key = 0;
#pragma unroll
  for (int i0 = 0; i0 < ITEMS; i0 += BATCH) {
    uint4 s0[BATCH], s1[BATCH], c0[BATCH], c1[BATCH];
    uint64_t kk[BATCH], home[BATCH], rk[BATCH], rhome[BATCH];
    bool ok[BATCH], in[BATCH], pal[BATCH];
#pragma unroll
    for (int j = 0; j < BATCH; ++j) {
      const int i = i0 + j;
      if (i == 0) key = tile_key<TILE>(tc, t0, sv.k);
      else {                                              // roll in the base at tile position t0 + i + k - 1
        const int p = t0 + i + sv.k - 1;
        key = ((key << 2) | ((tc.codes[p >> 4] >> (30 - 2 * (p & 15))) & 3u)) & kmask;
      }
      const int64_t q = q0 + t0 + i;
      in[j] = q >= first && q < end;
      ok[j] = in[j] && tile_valid<TILE>(sv, tc, q0, t0 + i, special);
      kk[j] = key;
      home[j] = kh.bucket(key);
      if (ok[j] && have) ld_stream_sector(kh.slots + home[j] * BUCKET_SLOTS, s0[j], s1[j]);
      if constexpr (BOTH) {
        rk[j] = revcomp_key(key, sv.k);
        pal[j] = rk[j] == key;
        rhome[j] = kh.bucket(rk[j]);
        if (ok[j] && have && !pal[j]) ld_stream_sector(kh.slots + rhome[j] * BUCKET_SLOTS, c0[j], c1[j]);
      }
    }
    uint2 f[BATCH], r[BATCH];
#pragma unroll
    for (int j = 0; j < BATCH; ++j) {
      f[j] = ok[j] && have ? resolve_key(kh, kk[j], home[j], s0[j], s1[j]) : make_uint2(0u, 0u);
      r[j] = make_uint2(0u, 0u);
      if constexpr (BOTH) if (ok[j] && have && !pal[j]) r[j] = resolve_key(kh, rk[j], rhome[j], c0[j], c1[j]);
    }
    int32_t *dst = out + (q0 + t0 + i0 - first) * cols;   // row of window j: dst + j * cols (only rows of the chunk are touched)
    for (int s = 0; s < cols; ++s) {
      int32_t v[BATCH];
#pragma unroll
      for (int j = 0; j < BATCH; ++j) {
        uint64_t c = (uint64_t)f[j].y + r[j].y;
        if constexpr (MULTI) c = (f[j].y ? (uint32_t)__ldg(counts + (uint64_t)f[j].x * cols + s) : 0u) +
                                 (uint64_t)(r[j].y ? (uint32_t)__ldg(counts + (uint64_t)r[j].x * cols + s) : 0u);
        v[j] = ok[j] ? (int32_t)(c < (uint64_t)INT32_MAX ? c : (uint64_t)INT32_MAX) : INT32_MIN;
      }
#pragma unroll
      for (int j = 0; j < BATCH; ++j)
        if (in[j]) dst[j * cols + s] = v[j];
    }
  }
}

// ---- pass 2: ordered compaction of the hits + chained 64-bit scan of their row counts --------------------
//   coordinate i of a hit: FROM_SEQ: 1-based END of the window (src/kmer_pos.c:127,132: `i` is one past the
//   window); else the record's own i.
//   max_count: a window whose k-mer has more positions is a miss (dot plots drop repeats); UINT32_MAX = no limit.
template <int THREADS, int ITEMS, bool FROM_SEQ>
__global__ void __launch_bounds__(THREADS)
probe_compact_kernel(const uint2 *__restrict__ found, int64_t coord0, const int32_t *__restrict__ i_in, int64_t n_in,
                     const uint64_t *__restrict__ n_dev, int32_t *__restrict__ hit_i, uint32_t *__restrict__ hit_start,
                     uint64_t *__restrict__ row_off, QueryStats *qs, Pair64 *status, uint32_t *ticket, const uint32_t max_count) {
  constexpr int TILE = THREADS * ITEMS, WARPS = THREADS / 32;
  static_assert(ITEMS % 2 == 0, "pairs of windows are read as one 16-byte word");
  static_assert(TILE <= 4096, "rows inside a tile: at most TILE * (2^32 - 1) < 2^48");
  __shared__ uint32_t s_tile, s_wh[WARPS];
  __shared__ uint64_t s_wr[WARPS], s_bh, s_br;
  __shared__ int32_t st_i[TILE];
  __shared__ uint32_t st_start[TILE], st_row[TILE];
  __shared__ uint16_t st_row_hi[TILE];
  const unsigned tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  if (tid == 0) s_tile = atomicAdd(ticket, 1u);
  __syncthreads();
  const uint32_t tile = s_tile;
  const int64_t q0 = (int64_t)tile * TILE;
  const int64_t total = n_dev ? min((int64_t)*n_dev, n_in) : n_in;
  if (q0 >= total) return;
  const int64_t t0 = q0 + (int64_t)tid * ITEMS;
  uint2 f[ITEMS];
  if (t0 + ITEMS <= total) {
#pragma unroll
    for (int i = 0; i < ITEMS; i += 2) {
      const uint4 v = ld_stream_u4(reinterpret_cast<const uint4 *>(found + t0 + i));
      f[i] = make_uint2(v.x, v.y); f[i + 1] = make_uint2(v.z, v.w);
    }
  } else {
#pragma unroll
    for (int i = 0; i < ITEMS; ++i) f[i] = t0 + i < total ? found[t0 + i] : make_uint2(0u, 0u);
  }
#pragma unroll
  for (int i = 0; i < ITEMS; ++i) if (f[i].y > max_count) f[i].y = 0;
  uint32_t hmine = 0;
  uint64_t rmine = 0;
#pragma unroll
  for (int i = 0; i < ITEMS; ++i) { hmine += f[i].y != 0; rmine += f[i].y; }
  const uint32_t hincl = warp_incl_scan(hmine);
  const uint64_t rincl = warp_incl_scan64(rmine);
  if (lane == 31) { s_wh[warp] = hincl; s_wr[warp] = rincl; }
  __syncthreads();
  uint64_t bh = 0, br = 0, th = 0, tr = 0;
#pragma unroll
  for (int w = 0; w < WARPS; ++w) {
    if (w < (int)warp) { bh += s_wh[w]; br += s_wr[w]; }
    th += s_wh[w]; tr += s_wr[w];
  }
  if (warp == 0) {
    uint64_t ea, eb;
    pair_lookback(status, tile, th, tr, ea, eb);
    if (lane == 0) { s_bh = ea; s_br = eb; }
  }
  __syncthreads();
  // stage the tile's hits in shared memory in order, then write them out coalesced
  {
    uint32_t hl = (uint32_t)bh + (hincl - hmine);        // index among the tile's hits
    uint64_t rl = br + (rincl - rmine);                  // rows before it inside the tile
#pragma unroll
    for (int i = 0; i < ITEMS; ++i) {
      if (f[i].y) {
        st_i[hl] = FROM_SEQ ? (int32_t)(coord0 + t0 + i) : i_in[t0 + i];
        st_start[hl] = f[i].x;
        st_row[hl] = (uint32_t)rl;                       // < TILE * 2^32 / ... : rows inside a tile fit 44 bits; low 32 here, high below
        st_row_hi[hl] = (uint16_t)(rl >> 32);
        ++hl;
        rl += f[i].y;
      }
    }
  }
  __syncthreads();
  const uint64_t gh = s_bh, gr = s_br;
  for (uint32_t idx = tid; idx < (uint32_t)th; idx += THREADS) {
    hit_i[gh + idx] = st_i[idx];
    hit_start[gh + idx] = st_start[idx];
    row_off[gh + idx] = gr + (((uint64_t)st_row_hi[idx] << 32) | st_row[idx]);
  }
  if (q0 + TILE >= total && tid == 0) { qs->H = s_bh + th; qs->M = s_br + tr; }
}

// (A fused lookup + compaction kernel was measured in round 2 and dropped: keeping a thread's eight (slot, count) pairs in
// registers through a ticket-ordered chained scan costs the latency-bound lookups more -- 29 KB of staging per block, spills
// at 64 registers -- than the 16 bytes per window of HBM traffic it saves: 3.57 ms against 2.73 + 0.62; profiles/r02_notes.md.)

// Emit rows [first, first+nrows): row r belongs to hit h = largest h with row_off[h] <= r; it pairs
// the hit's query coordinate with the (r - row_off[h])-th position of its k-mer.
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
probe_emit_kernel(const int32_t *__restrict__ hit_i, const uint32_t *__restrict__ hit_start,
                  const uint64_t *__restrict__ row_off, uint64_t H, const uint32_t *__restrict__ pos, uint64_t first,
                  uint64_t nrows, const uint64_t *__restrict__ blk_first, int2 *__restrict__ out) {
  constexpr int PER = 8, T = THREADS * PER;
  __shared__ __align__(16) uint8_t s_flag[T];
  __shared__ __align__(16) uint32_t s_seg[T];
  __shared__ uint32_t s_warp[THREADS / 32];
  __shared__ uint64_t s_first;
  const uint64_t b0 = (uint64_t)blockIdx.x * T;
  if (b0 >= nrows) return;
  const uint64_t r0 = first + b0;
  const uint64_t h0 = block_segments<THREADS, PER, uint64_t>(row_off, H, r0, blk_first[blockIdx.x], s_flag, s_seg, s_warp, &s_first);
#pragma unroll
  for (int j = 0; j < PER; ++j) {
    const uint32_t s = j * THREADS + threadIdx.x;
    if (b0 + s >= nrows) continue;
    const uint64_t h = h0 + s_seg[s];
    const uint64_t within = r0 + s - row_off[h];
    out[b0 + s] = make_int2(hit_i[h], (int)pos[hit_start[h] + within]);
  }
}

// ---- reverse complement of a query on the device (SURVEY.md 8f rank 2) ---------------------------------------
// Every dot plot in the reference's notebook probes the index twice, with the query and with
// reverseComplement(query) made on the host (test.R:43-52,73).  out[i] = comp(in[L-1-i]) with the IUPAC
// complement (A<->T, C<->G, R<->Y, K<->M, B<->V, D<->H; S, W, N and every other byte unchanged; case kept),
// so probing `out` equals seq.kmer.pos on the host-made reverse complement, byte for byte.
__device__ __forceinline__ uint8_t dna_complement(uint8_t c) {
  const uint8_t up = c & 0xDFu, lower = c & 0x20u;
  uint8_t r;
  switch (up) {
    case 'A': r = 'T'; break;  case 'T': r = 'A'; break;  case 'C': r = 'G'; break;  case 'G': r = 'C'; break;
    case 'R': r = 'Y'; break;  case 'Y': r = 'R'; break;  case 'K': r = 'M'; break;  case 'M': r = 'K'; break;
    case 'B': r = 'V'; break;  case 'V': r = 'B'; break;  case 'D': r = 'H'; break;  case 'H': r = 'D'; break;
    default: return c;
  }
  return (uint8_t)(r | lower);       // c & 0xDF matched a letter, so c is that letter in either case
}
__global__ void revcomp_kernel(const uint8_t *__restrict__ in, int64_t L, uint8_t *__restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < L; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = dna_complement(in[L - 1 - i]);
}

// ---- kmer.pairs(a, b): positions of the k-mers two indexes share ----------------------------------------------
// kmer_pair_pos (src/kmer_hash.c:1174-1203): for every k-mer of `a` that `b` also holds, rows (a_pos, b_pos),
// a position outer, b position inner.  a's distinct keys are looked up in b's key table (probe_lookup_kernel,
// record source); this kernel compacts the shared ones in a's order and scans their row counts ca * cb.
// max_count: a k-mer with more positions in either index is not shared (UINT32_MAX = no limit).
template <int THREADS, int ITEMS>
__global__ void __launch_bounds__(THREADS)
join_compact_kernel(const uint2 *__restrict__ found, const uint32_t *__restrict__ ustart_a, uint64_t U,
                    uint32_t *__restrict__ hit_astart, uint32_t *__restrict__ hit_bstart, uint32_t *__restrict__ hit_cb,
                    uint64_t *__restrict__ row_off, QueryStats *qs, Pair64 *status, uint32_t *ticket, const uint32_t max_count) {
  constexpr int TILE = THREADS * ITEMS, WARPS = THREADS / 32;
  __shared__ uint32_t s_tile, s_wh[WARPS];
  __shared__ uint64_t s_wr[WARPS], s_bh, s_br;
  const unsigned tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  if (tid == 0) s_tile = atomicAdd(ticket, 1u);
  __syncthreads();
  const uint32_t tile = s_tile;
  const uint64_t q0 = (uint64_t)tile * TILE;
  if (q0 >= U) return;
  const uint64_t t0 = q0 + (uint64_t)tid * ITEMS;
  uint2 f[ITEMS];
  uint32_t as[ITEMS + 1];
#pragma unroll
  for (int i = 0; i <= ITEMS; ++i) as[i] = t0 + i <= U ? ustart_a[t0 + i] : 0;
  uint32_t hmine = 0;
  uint64_t rmine = 0, rows[ITEMS];
#pragma unroll
  for (int i = 0; i < ITEMS; ++i) {
    f[i] = t0 + i < U ? found[t0 + i] : make_uint2(0u, 0u);
    if (f[i].y > max_count || as[i + 1] - as[i] > max_count) f[i].y = 0;
    rows[i] = f[i].y ? (uint64_t)(as[i + 1] - as[i]) * f[i].y : 0;
    hmine += f[i].y != 0;
    rmine += rows[i];
  }
  const uint32_t hincl = warp_incl_scan(hmine);
  const uint64_t rincl = warp_incl_scan64(rmine);
  if (lane == 31) { s_wh[warp] = hincl; s_wr[warp] = rincl; }
  __syncthreads();
  uint64_t bh = 0, br = 0, th = 0, tr = 0;
#pragma unroll
  for (int w = 0; w < WARPS; ++w) {
    if (w < (int)warp) { bh += s_wh[w]; br += s_wr[w]; }
    th += s_wh[w]; tr += s_wr[w];
  }
  if (warp == 0) {
    uint64_t ea, eb;
    pair_lookback(status, tile, th, tr, ea, eb);
    if (lane == 0) { s_bh = ea; s_br = eb; }
  }
  __syncthreads();
  uint64_t h = s_bh + bh + (hincl - hmine);
  uint64_t r = s_br + br + (rincl - rmine);
#pragma unroll
  for (int i = 0; i < ITEMS; ++i) {
    if (f[i].y) {
      hit_astart[h] = as[i];
      hit_bstart[h] = f[i].x;
      hit_cb[h] = f[i].y;
      row_off[h] = r;
      ++h;
      r += rows[i];
    }
  }
  if (q0 + TILE >= U && tid == 0) { qs->H = s_bh + th; qs->M = s_br + tr; }
}

template <int THREADS>
__global__ void __launch_bounds__(THREADS)
join_emit_kernel(const uint32_t *__restrict__ hit_astart, const uint32_t *__restrict__ hit_bstart,
                 const uint32_t *__restrict__ hit_cb, const uint64_t *__restrict__ row_off, uint64_t H,
                 const uint32_t *__restrict__ pos_a, const uint32_t *__restrict__ pos_b, uint64_t first, uint64_t nrows,
                 const uint64_t *__restrict__ blk_first, int2 *__restrict__ out) {
  constexpr int PER = 8, T = THREADS * PER;
  __shared__ __align__(16) uint8_t s_flag[T];
  __shared__ __align__(16) uint32_t s_seg[T];
  __shared__ uint32_t s_warp[THREADS / 32];
  __shared__ uint64_t s_first;
  const uint64_t b0 = (uint64_t)blockIdx.x * T;
  if (b0 >= nrows) return;
  const uint64_t r0 = first + b0;
  const uint64_t h0 = block_segments<THREADS, PER, uint64_t>(row_off, H, r0, blk_first[blockIdx.x], s_flag, s_seg, s_warp, &s_first);
#pragma unroll
  for (int j = 0; j < PER; ++j) {
    const uint32_t s = j * THREADS + threadIdx.x;
    if (b0 + s >= nrows) continue;
    const uint64_t h = h0 + s_seg[s];
    const uint64_t within = r0 + s - row_off[h];
    const uint32_t cb = hit_cb[h];
    const uint64_t ia = within / cb;                       // a position outer, b position inner (src/kmer_hash.c:1190-1195)
    out[b0 + s] = make_int2((int)pos_a[hit_astart[h] + ia], (int)pos_b[hit_bstart[h] + (within - ia * cb)]);
  }
}

// ---- dot plots: the rows of a probe or a join counted into an nx x ny image -----------------------------------------
// One axis of the image: a coordinate v is in the window iff 0 <= v - lo < range, and goes to bin floor((v - lo) * n / range).
// (v - lo) * n < 2^31 * 2^31, so the quotient is exact from the host's inv = floor((2^64 - 1) / range): umulhi(p, inv) is
// the quotient or one less (inv > 2^64 / range - 1 and p < 2^62), and one compare corrects it.
struct DotAxis {
  uint64_t lo, range, inv;
  uint32_t n;
};
constexpr uint32_t DOT_NONE = 0xFFFFFFFFu;

__device__ __forceinline__ uint32_t dot_bin(const DotAxis &a, uint32_t v) {
  const uint64_t d = (uint64_t)v - a.lo;                  // wraps to >= 2^63 below the window
  if (d >= a.range) return DOT_NONE;
  const uint64_t p = d * a.n;
  uint64_t q = __umul64hi(p, a.inv);
  if ((q + 1) * a.range <= p) ++q;
  return (uint32_t)q;
}

// Row sources: (x, y) of the within-th row of hit h.  A probe pairs the hit's query coordinate with the within-th position
// of its k-mer (probe_emit_kernel); a join takes a's positions outer and b's inner (join_emit_kernel), with a 32-bit
// division whenever the row number within the hit fits 32 bits.
struct ProbeRows {
  const int32_t *hit_i;
  const uint32_t *hit_start, *pos;
  __device__ __forceinline__ uint2 operator()(uint64_t h, uint64_t within) const {
    return make_uint2((uint32_t)hit_i[h], pos[hit_start[h] + within]);
  }
};
struct JoinRows {
  const uint32_t *hit_astart, *hit_bstart, *hit_cb, *pos_a, *pos_b;
  __device__ __forceinline__ uint2 operator()(uint64_t h, uint64_t within) const {
    const uint32_t cb = hit_cb[h];
    const uint64_t ia = within <= 0xFFFFFFFFull ? (uint64_t)((uint32_t)within / cb) : within / cb;
    return make_uint2(pos_a[hit_astart[h] + ia], pos_b[hit_bstart[h] + (within - ia * cb)]);
  }
};

// Rows [first, first + nrows) into the image img[bx + by * nx] (u64 counts), balanced by rows like the emit kernels
// (block_segments).  Lanes of a warp hold consecutive rows, which along a diagonal or inside one hit mostly share a bin:
// every run of equal bins among the lanes (compared with lane - 1) is summed by its first lane, which issues one 64-bit
// atomic for the run.  Rows outside the window are dropped.
template <int THREADS, class Rows>
__global__ void __launch_bounds__(THREADS)
dotplot_bin_kernel(const Rows rows, const uint64_t *__restrict__ row_off, uint64_t H, uint64_t first, uint64_t nrows,
                   const uint64_t *__restrict__ blk_first, const DotAxis ax, const DotAxis ay, unsigned long long *__restrict__ img) {
  constexpr int PER = 8, T = THREADS * PER;
  __shared__ __align__(16) uint8_t s_flag[T];
  __shared__ __align__(16) uint32_t s_seg[T];
  __shared__ uint32_t s_warp[THREADS / 32];
  __shared__ uint64_t s_first;
  const uint64_t b0 = (uint64_t)blockIdx.x * T;
  if (b0 >= nrows) return;
  const uint64_t r0 = first + b0;
  const uint64_t h0 = block_segments<THREADS, PER, uint64_t>(row_off, H, r0, blk_first[blockIdx.x], s_flag, s_seg, s_warp, &s_first);
  uint32_t bins[PER];                                     // all rows' loads first, then the atomics: the loads overlap
#pragma unroll
  for (int j = 0; j < PER; ++j) {
    const uint32_t s = j * THREADS + threadIdx.x;
    bins[j] = DOT_NONE;
    if (b0 + s < nrows) {                                 // every lane stays for the warp-wide run detection below
      const uint64_t h = h0 + s_seg[s];
      const uint2 xy = rows(h, r0 + s - row_off[h]);
      const uint32_t bx = dot_bin(ax, xy.x), by = dot_bin(ay, xy.y);
      if (bx != DOT_NONE && by != DOT_NONE) bins[j] = bx + by * ax.n;
    }
  }
  const unsigned lane = lane_id();
#pragma unroll
  for (int j = 0; j < PER; ++j) {
    const uint32_t bin = bins[j];
    const uint32_t prev = __shfl_up_sync(FULL, bin, 1);
    const bool head = lane == 0 || bin != prev;
    const uint32_t heads = __ballot_sync(FULL, head);
    if (head && bin != DOT_NONE) {
      const uint32_t later = lane == 31 ? 0u : heads & (0xFFFFFFFFu << (lane + 1));
      const uint32_t run = (later ? (uint32_t)__ffs(later) - 1 : 32u) - lane;
      atomicAdd(img + bin, (unsigned long long)run);
    }
  }
}

// u64 counts -> doubles (exact below 2^53)
__global__ void dotplot_finish_kernel(const unsigned long long *__restrict__ img, uint64_t n, double *__restrict__ out) {
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
    out[i] = (double)img[i];
}

}  // namespace kmg
