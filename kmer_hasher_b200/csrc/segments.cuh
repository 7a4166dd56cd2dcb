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

// ---- chains: runs joined across mismatches and short indels (kmg_chains_begin) ------------------------------------
// A run s = (i, j, n) ends at (I, J) = (i + n - 1, j + n - 1), or (i + n - 1, j - n + 1) with ANTI.  For a pair (s, t) the
// gaps are gq = i_t - I_s - 1 and gr = j_t - J_s - 1 (ANTI: J_s - j_t - 1); gq - gr = key_t - key_s (segment_key).  t may
// follow s iff 0 <= gq, gr <= G and |gq - gr| <= W; the cost (max(gq, gr), |gq - gr|, gq) is compared lexicographically.
// succ(s) and pred(t) are the least-cost partners; s -> t is a link iff succ(s) = t and pred(t) = s, and a chain is a
// maximal path of links.  The runs are viewed by diagonal (kmg_build_records over the keys, run numbers as payload: i
// ascends inside a diagonal, and the runs of one diagonal are disjoint, so their last rows ascend too).

// Key and run number of every run, the records of the diagonal sort.
template <bool ANTI>
__global__ void chains_keys_kernel(const int32_t *__restrict__ rows, uint64_t R, uint64_t *__restrict__ key, uint32_t *__restrict__ run) {
  for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < R; r += (uint64_t)gridDim.x * blockDim.x) {
    key[r] = segment_key<ANTI>(rows[3 * r], rows[3 * r + 1]);
    run[r] = (uint32_t)r;
  }
}

// In diagonal order p: the first and last row's i of run order[p], so the link searches read contiguous arrays.
__global__ void chains_gather_kernel(const int32_t *__restrict__ rows, const uint32_t *__restrict__ order, uint64_t R,
                                     uint32_t *__restrict__ si, uint32_t *__restrict__ sI) {
  for (uint64_t p = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < R; p += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t r = __ldg(order + p);
    const uint32_t i = (uint32_t)__ldg(rows + 3 * r), n = (uint32_t)__ldg(rows + 3 * r + 2);
    si[p] = i;
    sI[p] = i + n - 1;
  }
}

// The cost of a candidate as one word: max(gq, gr) < 2^31, then |delta| <= 1024, then gq -- which, for a fixed max and
// |delta|, is smaller exactly when delta < 0 (gq = max - |delta|) than when delta > 0 (gq = max).
__device__ __forceinline__ uint64_t chain_cost(int64_t gq, int64_t delta) {
  const int64_t gr = gq - delta, ad = delta < 0 ? -delta : delta;
  return (uint64_t)(gq > gr ? gq : gr) << 12 | (uint64_t)ad << 1 | (uint64_t)(delta > 0);
}

// One thread per run s (run order): succ[s] and pred[s] (run numbers, -1 for none), visiting only the occupied diagonals
// of [key - W, key + W] (dkeys[0, U) ascending, run order[dstart[u], dstart[u+1]) on diagonal u, si / sI in that order).
// On diagonal key + delta the best successor is the first run with i >= I + 1 + max(0, delta) (the least gq there), the
// best predecessor on diagonal key - delta the last run with I <= i - 1 - max(0, delta).  Either must also have
// gq <= G + min(0, delta), which is gr <= G.
// nsum: the n of all runs.
template <bool ANTI>
__global__ void __launch_bounds__(256)
chains_link_kernel(const int32_t *__restrict__ rows, uint64_t R, const uint64_t *__restrict__ dkeys, uint64_t U,
                   const uint32_t *__restrict__ dstart, const uint32_t *__restrict__ order, const uint32_t *__restrict__ si,
                   const uint32_t *__restrict__ sI, uint32_t G, uint32_t W, int32_t *__restrict__ succ,
                   int32_t *__restrict__ pred, unsigned long long *nsum) {
  const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint64_t mine = 0;
  if (s < R) {
    const int64_t i = rows[3 * s], j = rows[3 * s + 1], n = rows[3 * s + 2];
    const int64_t I = i + n - 1;
    const uint64_t key = segment_key<ANTI>(i, j);
    mine = (uint64_t)n;
    uint64_t lo = 0, len = U;                             // the first occupied diagonal at or after key - W
    const uint64_t k0 = key > W ? key - W : 0;
    while (len > 0) {
      const uint64_t half = len >> 1;
      if (__ldg(dkeys + lo + half) < k0) { lo += half + 1; len -= half + 1; } else len = half;
    }
    uint64_t bs = ~uint64_t(0), bp = ~uint64_t(0);
    int32_t vs = -1, vp = -1;
    for (uint64_t u = lo; u < U; ++u) {
      const uint64_t ku = __ldg(dkeys + u);
      if (ku > key + W) break;
      const uint32_t e0 = __ldg(dstart + u), e1 = __ldg(dstart + u + 1);
      {                                                   // successor on this diagonal: delta = ku - key
        const int64_t delta = (int64_t)ku - (int64_t)key;
        const int64_t thr = I + 1 + (delta > 0 ? delta : 0);
        if (thr <= INT32_MAX) {
          uint32_t a = e0, m = e1 - e0;                     // the first run with i >= thr
          while (m > 0) {
            const uint32_t half = m >> 1;
            if ((int64_t)__ldg(si + a + half) < thr) { a += half + 1; m -= half + 1; } else m = half;
          }
          if (a < e1) {
            const int64_t gq = (int64_t)__ldg(si + a) - I - 1;
            if (gq <= (int64_t)G + (delta < 0 ? delta : 0)) {
              const uint64_t c = chain_cost(gq, delta);
              if (c < bs) { bs = c; vs = (int32_t)__ldg(order + a); }
            }
          }
        }
      }
      {                                                   // predecessor on this diagonal: delta = key - ku
        const int64_t delta = (int64_t)key - (int64_t)ku;
        const int64_t thr = i - 1 - (delta > 0 ? delta : 0);
        if (thr >= 1) {
          uint32_t a = e0, m = e1 - e0;                     // the first run with I > thr; the one before it is the candidate
          while (m > 0) {
            const uint32_t half = m >> 1;
            if ((int64_t)__ldg(sI + a + half) <= thr) { a += half + 1; m -= half + 1; } else m = half;
          }
          if (a > e0) {
            const int64_t gq = i - (int64_t)__ldg(sI + a - 1) - 1;
            if (gq <= (int64_t)G + (delta < 0 ? delta : 0)) {
              const uint64_t c = chain_cost(gq, delta);
              if (c < bp) { bp = c; vp = (int32_t)__ldg(order + a - 1); }
            }
          }
        }
      }
    }
    succ[s] = vs;
    pred[s] = vp;
  }
  const uint64_t w = warp_sum64(mine);
  if ((threadIdx.x & 31u) == 0 && w) atomicAdd(nsum, (unsigned long long)w);
}

// head[t] = pred[t] when the link is mutual (succ[pred[t]] = t), else t: a chain's first run points to itself.
__global__ void chains_heads_kernel(const int32_t *__restrict__ succ, const int32_t *__restrict__ pred, uint64_t R,
                                    int32_t *__restrict__ head) {
  for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < R; t += (uint64_t)gridDim.x * blockDim.x) {
    const int32_t p = pred[t];
    head[t] = p >= 0 && __ldg(succ + p) == (int32_t)t ? p : (int32_t)t;
  }
}

// One round of pointer jumping, in place: head[t] = head[head[t]].  A value read mid-round is still an earlier run of the
// same chain, so the rounds stay correct and needed ones only fewer; *changed is set while a pointer still moved.
__global__ void chains_jump_kernel(int32_t *head, uint64_t R, uint32_t *changed) {
  bool moved = false;
  for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < R; t += (uint64_t)gridDim.x * blockDim.x) {
    const int32_t h = head[t], hh = head[h];
    if (hh != h) { head[t] = hh; moved = true; }
  }
  if (__any_sync(FULL, moved) && (threadIdx.x & 31u) == 0) *changed = 1u;
}

// Every run that is not a chain's first adds (n << 32 | 1) into nm[head] and its packed last row (I << 32 | J) into
// last[head] by atomic max: along a chain I strictly increases, so the max is the last run's in either orientation.
template <bool ANTI>
__global__ void chains_aggregate_kernel(const int32_t *__restrict__ rows, const int32_t *__restrict__ head, uint64_t R,
                                        unsigned long long *nm, unsigned long long *last) {
  for (uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; t < R; t += (uint64_t)gridDim.x * blockDim.x) {
    const int32_t h = head[t];
    if (h == (int32_t)t) continue;
    const uint32_t i = (uint32_t)rows[3 * t], j = (uint32_t)rows[3 * t + 1], n = (uint32_t)rows[3 * t + 2];
    const uint32_t J = ANTI ? j - n + 1 : j + n - 1;
    atomicAdd(nm + h, (unsigned long long)n << 32 | 1ull);
    atomicMax(last + h, (unsigned long long)(i + n - 1) << 32 | J);
  }
}

// The chains, first runs in run order ((i, j) order), with n >= min_rows, as (i, j, I, J, n, m) into out (a chained scan,
// tiles numbered by `ticket`).  The scan carries (kept + 2^31 * m, n): both kept and the m of all chains stay below 2^31.
// tot: (chains kept, sum of m, sum of n) over all chains, which the host checks against R and the runs' sum of n.
template <int THREADS, int ITEMS, bool ANTI>
__global__ void __launch_bounds__(THREADS)
chains_compact_kernel(const int32_t *__restrict__ rows, const int32_t *__restrict__ head, const unsigned long long *__restrict__ nm,
                      const unsigned long long *__restrict__ last, uint64_t R, uint32_t min_rows, Pair64 *status,
                      uint32_t *ticket, int32_t *__restrict__ out, uint64_t *tot) {
  constexpr int TILE = THREADS * ITEMS, WARPS = THREADS / 32;
  __shared__ uint32_t s_tile, s_wk[WARPS];
  __shared__ uint64_t s_wm[WARPS], s_wn[WARPS], s_bk;
  const unsigned tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  if (tid == 0) s_tile = atomicAdd(ticket, 1u);
  __syncthreads();
  const uint32_t tile = s_tile;
  const uint64_t q0 = (uint64_t)tile * TILE;
  if (q0 >= R) return;
  const uint64_t t0 = q0 + (uint64_t)tid * ITEMS;
  uint32_t kmine = 0;
  uint64_t mmine = 0, nmine = 0;
  uint32_t keep = 0;                                      // bit t: item t is a kept chain
#pragma unroll
  for (int t = 0; t < ITEMS; ++t) {
    if (t0 + t >= R || head[t0 + t] != (int32_t)(t0 + t)) continue;
    const unsigned long long a = nm[t0 + t];
    const uint64_t n = (uint64_t)(uint32_t)rows[3 * (t0 + t) + 2] + (a >> 32);
    mmine += 1 + (a & 0xffffffffull);
    nmine += n;
    if (n >= min_rows) { keep |= 1u << t; ++kmine; }
  }
  const uint32_t kincl = warp_incl_scan(kmine);
  const uint64_t mw = warp_sum64(mmine), nw = warp_sum64(nmine);
  if (lane == 31) s_wk[warp] = kincl;
  if (lane == 0) { s_wm[warp] = mw; s_wn[warp] = nw; }
  __syncthreads();
  uint64_t bk = 0, tk = 0, tm = 0, tn = 0;
#pragma unroll
  for (int w = 0; w < WARPS; ++w) {
    if (w < (int)warp) bk += s_wk[w];
    tk += s_wk[w]; tm += s_wm[w]; tn += s_wn[w];
  }
  if (warp == 0) {
    uint64_t xa, xn;
    pair_lookback(status, tile, tk + (tm << 31), tn, xa, xn);
    if (lane == 0) {
      s_bk = xa & 0x7fffffffull;
      if (q0 + TILE >= R) { tot[0] = (xa & 0x7fffffffull) + tk; tot[1] = (xa >> 31) + tm; tot[2] = xn + tn; }
    }
  }
  __syncthreads();
  uint64_t at = s_bk + bk + (kincl - kmine);
#pragma unroll
  for (int t = 0; t < ITEMS; ++t) {
    if (!(keep >> t & 1u)) continue;
    const uint64_t r = t0 + t;
    const int32_t i = rows[3 * r], j = rows[3 * r + 1], n = rows[3 * r + 2];
    const unsigned long long a = nm[r];
    const unsigned long long own = (unsigned long long)(uint32_t)(i + n - 1) << 32 | (uint32_t)(ANTI ? j - n + 1 : j + n - 1);
    const unsigned long long l = last[r] > own ? last[r] : own;   // last[r] is 0 for a chain of one
    int32_t *o = out + 6 * at;
    o[0] = i; o[1] = j; o[2] = (int32_t)(l >> 32); o[3] = (int32_t)(uint32_t)l;
    o[4] = (int32_t)((uint64_t)(uint32_t)n + (a >> 32)); o[5] = (int32_t)(1 + (a & 0xffffffffull));
    ++at;
  }
}

}  // namespace kmg
