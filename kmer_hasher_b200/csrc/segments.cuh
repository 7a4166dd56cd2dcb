// segments.cuh -- match segments: maximal diagonal runs of a probe's rows (seq.kmer.segments).
//
// A run is a maximal sequence of rows (i + t, j + t), t = 0 .. n-1, of one probe.  The probe's hits are its query windows
// in ascending i, each with the sorted position list of its k-mer, so the row (i, j) of hit h continues a run from the row
// (i - 1, j - 1) iff hit h - 1 has i - 1 and j - 1 is in its list, and likewise forward.  segments_mark_kernel finds the
// rows that start a run and the rows that end one and compacts both in row order; the ends are then sorted by diagonal
// (kmg_build_records, stable, so i ascends inside a diagonal) and segments_pair_kernel pairs each start with the first end
// of its diagonal at or after it: runs of one diagonal do not overlap, so its k-th start and k-th end belong together.
// ANTI (kmer.pairs.segments with the reverse complement): runs are antiparallel, rows (i + t, j - t); the row (i, j)
// continues one from (i - 1, j + 1) and into (i + 1, j - 1), and a run's anti-diagonal is i + j.  The rows of a hit
// still ascend in j, so the starts still come out in (i, j) order.
#pragma once
#include "common.cuh"
#include "csr.cuh"
#include "lookback.cuh"

namespace kmg {

// Is v in the ascending list p[0, n)?  p[g] is read first: copies of a repeat tend to keep their order from one k-mer's
// list to the next, so the neighbour of the row at rank g of its list is often at rank g of the neighbouring list; a
// miss still halves the range of the lower-bound search.
__device__ __forceinline__ bool sorted_has(const uint32_t *__restrict__ p, uint32_t n, uint32_t v, uint32_t g) {
  uint32_t lo = 0, len = n;
  if (g < n) {
    const uint32_t x = __ldg(p + g);
    if (x == v) return true;
    if (x < v) { lo = g + 1; len = n - g - 1; } else len = g;
  }
  while (len > 0) {
    const uint32_t half = len >> 1;
    if (__ldg(p + lo + half) < v) { lo += half + 1; len -= half + 1; } else len = half;
  }
  return lo < n && __ldg(p + lo) == v;
}

// The key of the diagonal (i - j + 2^31) or, with ANTI, of the anti-diagonal (i + j) of the row (i, j): below 2^32 either way.
template <bool ANTI>
__device__ __forceinline__ uint64_t segment_key(int64_t i, int64_t j) {
  return (uint64_t)(ANTI ? i + j : i - j + (int64_t(1) << 31));
}

// Rows [first, first + nrows) of a probe (hits hit_i / hit_start / row_off[0, H), M rows in all), balanced by rows like
// probe_emit_kernel.  Writes the run starts as (i, j) and the run ends as (segment_key(i, j), i), each in row order, from
// the bases (base_s, base_e) on; entries at or past `cap` are counted but not written.  tot: (starts, ends) of the slice.
// Tiles take their number from `ticket` so that the chained scan of their counts (pair_lookback) cannot deadlock.
template <int THREADS, bool ANTI>
__global__ void __launch_bounds__(THREADS)
segments_mark_kernel(const int32_t *__restrict__ hit_i, const uint32_t *__restrict__ hit_start, const uint64_t *__restrict__ row_off,
                     uint64_t H, uint64_t M, const uint32_t *__restrict__ pos, uint64_t first, uint64_t nrows,
                     const uint64_t *__restrict__ blk_first, Pair64 *status, uint32_t *ticket, uint64_t base_s, uint64_t base_e,
                     uint64_t cap, int2 *__restrict__ starts, uint64_t *__restrict__ end_key, uint32_t *__restrict__ end_i,
                     uint64_t *tot) {
  constexpr int PER = 8, T = THREADS * PER, WARPS = THREADS / 32;
  static_assert(PER * WARPS == 64, "the block scan below gives each lane of one warp two (round, warp) counts");
  __shared__ __align__(16) uint8_t s_flag[T];
  __shared__ __align__(16) uint32_t s_seg[T];
  __shared__ uint32_t s_warp[WARPS], s_tile;
  __shared__ uint64_t s_first;
  __shared__ uint32_t s_cs[PER * WARPS], s_ce[PER * WARPS];   // per (round, warp): counts, then exclusive offsets
  __shared__ uint64_t s_bs, s_be;
  const unsigned tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  if (tid == 0) s_tile = atomicAdd(ticket, 1u);
  __syncthreads();
  const uint32_t tile = s_tile;
  const uint64_t b0 = (uint64_t)tile * T;
  if (b0 >= nrows) return;
  const uint64_t r0 = first + b0;
  const uint64_t h0 = block_segments<THREADS, PER, uint64_t>(row_off, H, r0, blk_first[tile], s_flag, s_seg, s_warp, &s_first);
  int32_t vi[PER];
  uint32_t vj[PER], ms[PER], me[PER];
#pragma unroll
  for (int r = 0; r < PER; ++r) {
    const uint32_t s = r * THREADS + tid;
    bool st = false, en = false;
    vi[r] = 0; vj[r] = 0;
    if (b0 + s < nrows) {
      const uint64_t h = h0 + s_seg[s];
      const uint64_t o = row_off[h], within = r0 + s - o;
      const uint64_t o1 = h + 1 < H ? row_off[h + 1] : M;
      const int32_t i = hit_i[h];
      const uint32_t hs = hit_start[h];
      const uint32_t j = pos[hs + within];
      bool pred = false, succ = false;
      if constexpr (!ANTI) {
        if (h > 0 && hit_i[h - 1] == i - 1 && j > 0) {
          const uint32_t ps = hit_start[h - 1];
          if (ps == hs) pred = within > 0 && pos[hs + within - 1] == j - 1;     // the same list: j - 1 would sit just before j
          else pred = sorted_has(pos + ps, (uint32_t)(o - row_off[h - 1]), j - 1, (uint32_t)within);
        }
        if (h + 1 < H && hit_i[h + 1] == i + 1) {
          const uint32_t ns = hit_start[h + 1];
          if (ns == hs) succ = within + 1 < o1 - o && pos[hs + within + 1] == j + 1;
          else succ = sorted_has(pos + ns, (uint32_t)((h + 2 < H ? row_off[h + 2] : M) - o1), j + 1, (uint32_t)within);
        }
      } else {                                            // (i - 1, j + 1) and (i + 1, j - 1); positions are >= 1
        if (h > 0 && hit_i[h - 1] == i - 1) {
          const uint32_t ps = hit_start[h - 1];
          if (ps == hs) pred = within + 1 < o1 - o && pos[hs + within + 1] == j + 1;
          else pred = sorted_has(pos + ps, (uint32_t)(o - row_off[h - 1]), j + 1, (uint32_t)within);
        }
        if (h + 1 < H && hit_i[h + 1] == i + 1) {
          const uint32_t ns = hit_start[h + 1];
          if (ns == hs) succ = within > 0 && pos[hs + within - 1] == j - 1;
          else succ = sorted_has(pos + ns, (uint32_t)((h + 2 < H ? row_off[h + 2] : M) - o1), j - 1, (uint32_t)within);
        }
      }
      st = !pred; en = !succ;
      vi[r] = i; vj[r] = j;
    }
    ms[r] = __ballot_sync(FULL, st);
    me[r] = __ballot_sync(FULL, en);
    if (lane == 0) { s_cs[r * WARPS + warp] = __popc(ms[r]); s_ce[r * WARPS + warp] = __popc(me[r]); }
  }
  __syncthreads();
  if (warp == 0) {                                        // rows in order: round, then warp, then lane
    const uint32_t a0 = s_cs[2 * lane], a1 = s_cs[2 * lane + 1], e0 = s_ce[2 * lane], e1 = s_ce[2 * lane + 1];
    const uint32_t ai = warp_incl_scan(a0 + a1), ei = warp_incl_scan(e0 + e1);
    const uint32_t at = __shfl_sync(FULL, ai, 31), et = __shfl_sync(FULL, ei, 31);
    s_cs[2 * lane] = ai - a0 - a1; s_cs[2 * lane + 1] = ai - a1;
    s_ce[2 * lane] = ei - e0 - e1; s_ce[2 * lane + 1] = ei - e1;
    uint64_t xs, xe;
    pair_lookback(status, tile, at, et, xs, xe);
    if (lane == 0) {
      s_bs = base_s + xs; s_be = base_e + xe;
      if (b0 + T >= nrows) { tot[0] = xs + at; tot[1] = xe + et; }
    }
  }
  __syncthreads();
  const uint64_t bs = s_bs, be = s_be;
  const unsigned lt = lanemask_lt();
#pragma unroll
  for (int r = 0; r < PER; ++r) {
    if (ms[r] >> lane & 1u) {
      const uint64_t at = bs + s_cs[r * WARPS + warp] + __popc(ms[r] & lt);
      if (at < cap) starts[at] = make_int2(vi[r], (int32_t)vj[r]);
    }
    if (me[r] >> lane & 1u) {
      const uint64_t at = be + s_ce[r * WARPS + warp] + __popc(me[r] & lt);
      if (at < cap) {
        end_key[at] = segment_key<ANTI>(vi[r], (int64_t)vj[r]);
        end_i[at] = (uint32_t)vi[r];
      }
    }
  }
}

// Pair the starts [0, R0) with the ends sorted by diagonal, or anti-diagonal with ANTI (dkeys[0, U) ascending, the ends'
// i in ei[dstart[u], dstart[u+1]) ascending): n = (first end i >= i on the start's diagonal) - i + 1.  The runs with
// n >= min_rows go to out as (i, j, n) triples in the starts' order (a chained scan, tiles numbered by `ticket`).
// tot: (runs kept, sum of n over all runs); a start without an end adds 0 to the sum, which the host checks against the
// probe's row count.
template <int THREADS, int ITEMS, bool ANTI>
__global__ void __launch_bounds__(THREADS)
segments_pair_kernel(const int2 *__restrict__ starts, uint64_t R0, const uint64_t *__restrict__ dkeys, uint64_t U,
                     const uint32_t *__restrict__ dstart, const uint32_t *__restrict__ ei, uint32_t min_rows, Pair64 *status,
                     uint32_t *ticket, int32_t *__restrict__ out, uint64_t *tot) {
  constexpr int TILE = THREADS * ITEMS, WARPS = THREADS / 32;
  __shared__ uint32_t s_tile, s_wk[WARPS];
  __shared__ uint64_t s_wn[WARPS], s_bk;
  const unsigned tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  if (tid == 0) s_tile = atomicAdd(ticket, 1u);
  __syncthreads();
  const uint32_t tile = s_tile;
  const uint64_t q0 = (uint64_t)tile * TILE;
  if (q0 >= R0) return;
  const uint64_t t0 = q0 + (uint64_t)tid * ITEMS;
  int2 v[ITEMS];
  uint32_t n[ITEMS];
  uint32_t kmine = 0;
  uint64_t nmine = 0;
#pragma unroll
  for (int t = 0; t < ITEMS; ++t) {
    n[t] = 0;
    v[t] = make_int2(0, 0);
    if (t0 + t >= R0) continue;
    v[t] = starts[t0 + t];
    const uint64_t key = segment_key<ANTI>(v[t].x, v[t].y);
    uint64_t lo = 0, len = U;                             // the diagonal: lower bound of key in dkeys
    while (len > 0) {
      const uint64_t half = len >> 1;
      if (__ldg(dkeys + lo + half) < key) { lo += half + 1; len -= half + 1; } else len = half;
    }
    if (lo < U && __ldg(dkeys + lo) == key) {
      const uint32_t e0 = __ldg(dstart + lo), e1 = __ldg(dstart + lo + 1);
      uint32_t a = e0, m = e1 - e0;                       // the first end at or after the start
      while (m > 0) {
        const uint32_t half = m >> 1;
        if (__ldg(ei + a + half) < (uint32_t)v[t].x) { a += half + 1; m -= half + 1; } else m = half;
      }
      if (a < e1) n[t] = __ldg(ei + a) - (uint32_t)v[t].x + 1;
    }
    nmine += n[t];
    kmine += n[t] != 0 && n[t] >= min_rows;
  }
  const uint32_t kincl = warp_incl_scan(kmine);
  const uint64_t nw = warp_sum64(nmine);
  if (lane == 31) s_wk[warp] = kincl;
  if (lane == 0) s_wn[warp] = nw;
  __syncthreads();
  uint64_t bk = 0, tk = 0, tn = 0;
#pragma unroll
  for (int w = 0; w < WARPS; ++w) {
    if (w < (int)warp) bk += s_wk[w];
    tk += s_wk[w]; tn += s_wn[w];
  }
  if (warp == 0) {
    uint64_t xk, xn;
    pair_lookback(status, tile, tk, tn, xk, xn);
    if (lane == 0) {
      s_bk = xk;
      if (q0 + TILE >= R0) { tot[0] = xk + tk; tot[1] = xn + tn; }
    }
  }
  __syncthreads();
  uint64_t at = s_bk + bk + (kincl - kmine);
#pragma unroll
  for (int t = 0; t < ITEMS; ++t) {
    if (n[t] != 0 && n[t] >= min_rows) {
      out[3 * at] = v[t].x; out[3 * at + 1] = v[t].y; out[3 * at + 2] = (int32_t)n[t];
      ++at;
    }
  }
}

// 32-bit words in[0, n) -> out (emit of the finished (i, j, n) triples into a stream_rows chunk)
__global__ void segments_emit_kernel(const int32_t *__restrict__ in, uint64_t n, int32_t *__restrict__ out) {
  for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < n; w += (uint64_t)gridDim.x * blockDim.x)
    out[w] = ld_stream_u32(reinterpret_cast<const uint32_t *>(in) + w);
}

}  // namespace kmg
