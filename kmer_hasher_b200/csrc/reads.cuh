// reads.cuh -- FASTA / FASTQ text -> sequences, parsed on the device (SURVEY.md 8f rank 4).
//
// The reference reads sequence files with klib's kseq.h over zlib (src/kseq.h, used by kmer_reader_read,
// src/kmer_reader.c:41-77): a record starts at a line that begins with '>' (FASTA) or '@' (FASTQ), its name is the
// header up to the first white space, its sequence is the following line(s) with the line ends removed (a trailing '\r'
// too, kseq.h:141).  Here the host only inflates the file (zlib) and uploads the text; the lines are found, classified
// and packed on the device:
//   nl_scan_kernel      positions of all '\n' (ordered compaction, chained scan) + newlines before every 16-byte block
//   line_info_kernel    per line: sequence bytes it contributes, whether it is a header
//   line_scan_kernel    exclusive scans of both (chained scan): where every line's bases go, which record it belongs to
//   record_kernel       per header line: the record's offset in the packed sequence buffer and its name
//   pack_kernel         copies the sequence bytes; records are laid out back to back with ONE separator byte ('N', a window
//                       breaker) between them, so the whole buffer is also a valid input for counting all records at once
// FASTA may be multi-line with any line length (a 250 Mbp chromosome on one line is fine: the copy is parallel over
// bytes, not lines).  FASTQ must be the usual four-line form (checked on the device; multi-line FASTQ is refused).
#pragma once
#include "common.cuh"
#include "lookback.cuh"

namespace kmg {

enum : uint8_t { LINE_OTHER = 0, LINE_HEADER = 1, LINE_SEQ = 2 };

struct ReadsInfo {
  uint64_t n_newlines, n_lines, n_records, total_bases;
  uint32_t bad;        // != 0: not a well-formed four-line FASTQ / sequence before the first header
  uint32_t pad;
};

__device__ __forceinline__ uint32_t newline_mask16(uint4 v) {          // bit j set: byte j of the 16 is '\n'
  auto m4 = [](uint32_t x) { uint32_t e = __vcmpeq4(x, 0x0A0A0A0Au) & 0x01010101u; return ((e * 0x01020408u) >> 24) & 0xFu; };
  return m4(v.x) | (m4(v.y) << 4) | (m4(v.z) << 8) | (m4(v.w) << 12);
}

// number of '\n' in the text (sizes the position list exactly)
__global__ void nl_count_kernel(const uint8_t *__restrict__ text, uint64_t n, unsigned long long *count) {
  const uint64_t nblocks = (n + 15) / 16;
  uint64_t c = 0;
  for (uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; b < nblocks; b += (uint64_t)gridDim.x * blockDim.x) {
    uint32_t m = newline_mask16(ld_stream_u4(reinterpret_cast<const uint4 *>(text) + b));
    const uint64_t left = n - b * 16;
    if (left < 16) m &= (1u << left) - 1;
    c += __popc(m);
  }
  c = warp_sum64(c);
  if (lane_id() == 0 && c) atomicAdd(count, (unsigned long long)c);
}

// text is readable (zero padded) up to a multiple of 64 bytes.  A thread owns 4 consecutive 16-byte blocks.
template <int THREADS>
__global__ void __launch_bounds__(THREADS)
nl_scan_kernel(const uint8_t *__restrict__ text, uint64_t n, uint64_t *__restrict__ nl, uint32_t *__restrict__ blk_nl,
               Pair64 *status, uint32_t *ticket, ReadsInfo *info) {
  constexpr int WARPS = THREADS / 32, PER = 4;
  __shared__ uint32_t s_tile, s_w[WARPS];
  __shared__ uint64_t s_base;
  const unsigned tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  if (tid == 0) s_tile = atomicAdd(ticket, 1u);
  __syncthreads();
  const uint32_t tile = s_tile;
  const uint64_t b0 = ((uint64_t)tile * THREADS + tid) * PER;            // first 16-byte block of this thread
  const uint64_t nblocks = (n + 15) / 16;
  if ((uint64_t)tile * THREADS * PER >= nblocks) return;
  uint32_t m[PER], c = 0;
#pragma unroll
  for (int j = 0; j < PER; ++j) {
    m[j] = 0;
    if (b0 + j < nblocks) {
      m[j] = newline_mask16(ld_stream_u4(reinterpret_cast<const uint4 *>(text) + b0 + j));
      const uint64_t left = n - (b0 + j) * 16;                            // bytes of the block that exist
      if (left < 16) m[j] &= (1u << left) - 1;
    }
    c += __popc(m[j]);
  }
  const uint32_t incl = warp_incl_scan(c);
  if (lane == 31) s_w[warp] = incl;
  __syncthreads();
  uint32_t wb = 0, tot = 0;
#pragma unroll
  for (int w = 0; w < WARPS; ++w) { if (w < (int)warp) wb += s_w[w]; tot += s_w[w]; }
  if (warp == 0) {
    uint64_t ea, eb;
    pair_lookback(status, tile, tot, 0, ea, eb);
    if (lane == 0) s_base = ea;
  }
  __syncthreads();
  uint64_t at = s_base + wb + (incl - c);
#pragma unroll
  for (int j = 0; j < PER; ++j) {
    if (b0 + j < nblocks) blk_nl[b0 + j] = (uint32_t)at;
    uint32_t mm = m[j];
    while (mm) { const int bit = __ffs(mm) - 1; mm &= mm - 1; nl[at++] = (b0 + j) * 16 + bit; }
  }
  if ((uint64_t)(tile + 1) * THREADS * PER >= nblocks && tid == 0) {      // last tile
    const uint64_t nnl = s_base + tot;
    info->n_newlines = nnl;
    info->n_lines = nnl + ((n > 0 && text[n - 1] != '\n') ? 1 : 0);
  }
}

__device__ __forceinline__ void line_bounds(const uint64_t *nl, uint64_t nnl, uint64_t n, uint64_t i, const uint8_t *text, uint64_t &start,
                                            uint64_t &end) {
  start = i == 0 ? 0 : nl[i - 1] + 1;
  end = i < nnl ? nl[i] : n;
  if (end > start && text[end - 1] == '\r') --end;                        // Windows line ends (kseq.h:141)
}

// per line: bytes of sequence it holds, header flag.  fastq: the four-line form is enforced.
__global__ void line_info_kernel(const uint8_t *__restrict__ text, uint64_t n, const uint64_t *__restrict__ nl, const ReadsInfo *info,
                                 bool fastq, uint64_t *__restrict__ seq_len, uint8_t *__restrict__ kind, ReadsInfo *out) {
  const uint64_t nnl = info->n_newlines, nlines = info->n_lines;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nlines; i += (uint64_t)gridDim.x * blockDim.x) {
    uint64_t s, e;
    line_bounds(nl, nnl, n, i, text, s, e);
    uint8_t kd = LINE_OTHER;
    uint64_t len = 0;
    if (fastq) {
      const int t = (int)(i & 3);
      if (e == s && i + 4 > nlines && t == 0) { /* trailing blank line */ }
      else if (t == 0) { kd = LINE_HEADER; if (e == s || text[s] != '@') out->bad = 1; }
      else if (t == 1) { kd = LINE_SEQ; len = e - s; }
      else if (t == 2) { if (e == s || text[s] != '+') out->bad = 1; }
      else {                                                               // quality: as long as the sequence line
        uint64_t ps, pe;
        line_bounds(nl, nnl, n, i - 2, text, ps, pe);
        if (pe - ps != e - s) out->bad = 1;
      }
    } else if (e > s) {
      if (text[s] == '>') kd = LINE_HEADER;
      else { kd = LINE_SEQ; len = e - s; }
    }
    seq_len[i] = len;
    kind[i] = kd;
  }
}

// exclusive scans over the lines: sequence bytes before (a) and headers before (b)
template <int THREADS, int ITEMS>
__global__ void __launch_bounds__(THREADS)
line_scan_kernel(const uint64_t *__restrict__ seq_len, const uint8_t *__restrict__ kind, ReadsInfo *info, uint64_t *__restrict__ seq_before,
                 uint64_t *__restrict__ hdr_before, Pair64 *status, uint32_t *ticket) {
  constexpr int TILE = THREADS * ITEMS, WARPS = THREADS / 32;
  __shared__ uint32_t s_tile;
  __shared__ uint64_t s_wa[WARPS], s_wb[WARPS], s_ba, s_bb;
  const unsigned tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
  if (tid == 0) s_tile = atomicAdd(ticket, 1u);
  __syncthreads();
  const uint32_t tile = s_tile;
  const uint64_t nlines = info->n_lines;
  const uint64_t q0 = (uint64_t)tile * TILE;
  if (q0 >= nlines) { if (nlines == 0 && tile == 0 && tid == 0) { info->n_records = 0; info->total_bases = 0; } return; }
  const uint64_t i0 = q0 + (uint64_t)tid * ITEMS;
  uint64_t a[ITEMS], suma = 0, sumb = 0;
  uint8_t h[ITEMS];
#pragma unroll
  for (int j = 0; j < ITEMS; ++j) {
    a[j] = i0 + j < nlines ? seq_len[i0 + j] : 0;
    h[j] = i0 + j < nlines ? (kind[i0 + j] == LINE_HEADER) : 0;
    suma += a[j]; sumb += h[j];
  }
  const uint64_t ia = warp_incl_scan64(suma), ib = warp_incl_scan64(sumb);
  if (lane == 31) { s_wa[warp] = ia; s_wb[warp] = ib; }
  __syncthreads();
  uint64_t ba = 0, bb = 0, ta = 0, tb = 0;
#pragma unroll
  for (int w = 0; w < WARPS; ++w) { if (w < (int)warp) { ba += s_wa[w]; bb += s_wb[w]; } ta += s_wa[w]; tb += s_wb[w]; }
  if (warp == 0) {
    uint64_t ea, eb;
    pair_lookback(status, tile, ta, tb, ea, eb);
    if (lane == 0) { s_ba = ea; s_bb = eb; }
  }
  __syncthreads();
  uint64_t ra = s_ba + ba + (ia - suma), rb = s_bb + bb + (ib - sumb);
#pragma unroll
  for (int j = 0; j < ITEMS; ++j) {
    if (i0 + j < nlines) { seq_before[i0 + j] = ra; hdr_before[i0 + j] = rb; }
    ra += a[j]; rb += h[j];
  }
  if (q0 + TILE >= nlines && tid == 0) { info->total_bases = s_ba + ta; info->n_records = s_bb + tb; }
}

// per header line: where the record's bases start in the packed buffer (bases before + one separator per earlier record)
// and its name (header text after '>' / '@' up to the first white space)
__global__ void record_kernel(const uint8_t *__restrict__ text, uint64_t n, const uint64_t *__restrict__ nl, const ReadsInfo *info,
                              const uint8_t *__restrict__ kind, const uint64_t *__restrict__ seq_before, const uint64_t *__restrict__ hdr_before,
                              uint64_t *__restrict__ rec_off, uint64_t *__restrict__ name_pos, uint32_t *__restrict__ name_len) {
  const uint64_t nnl = info->n_newlines, nlines = info->n_lines;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nlines; i += (uint64_t)gridDim.x * blockDim.x) {
    if (kind[i] != LINE_HEADER) continue;
    uint64_t s, e;
    line_bounds(nl, nnl, n, i, text, s, e);
    const uint64_t r = hdr_before[i];
    rec_off[r] = seq_before[i] + r;
    uint64_t p = s + 1;
    while (p < e && text[p] != ' ' && text[p] != '\t') ++p;
    name_pos[r] = s + 1;
    name_len[r] = (uint32_t)(p - s - 1);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) rec_off[info->n_records] = info->total_bases + info->n_records;   // one past the last separator
}

// copy the sequence bytes into the packed buffer, one 16-byte block of text per thread step
__global__ void pack_kernel(const uint8_t *__restrict__ text, uint64_t n, const uint64_t *__restrict__ nl, const uint32_t *__restrict__ blk_nl,
                            const ReadsInfo *info, const uint8_t *__restrict__ kind, const uint64_t *__restrict__ seq_before,
                            const uint64_t *__restrict__ hdr_before, uint8_t *__restrict__ seq, ReadsInfo *out) {
  const uint64_t nblocks = (n + 15) / 16;
  for (uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; b < nblocks; b += (uint64_t)gridDim.x * blockDim.x) {
    uint64_t line = blk_nl[b];
    const uint4 v = ld_stream_u4(reinterpret_cast<const uint4 *>(text) + b);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    bool is_seq = kind[line] == LINE_SEQ;
    uint64_t start = line == 0 ? 0 : nl[line - 1] + 1;
    uint64_t base = is_seq ? seq_before[line] + hdr_before[line] - 1 : 0;      // hdr_before >= 1 for a sequence line of a record
    if (is_seq && hdr_before[line] == 0) { out->bad = 1; is_seq = false; }      // sequence before the first header
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const uint64_t p = b * 16 + j;
      if (p >= n) break;
      const uint8_t c = (uint8_t)(w[j >> 2] >> (8 * (j & 3)));
      if (c == '\n') {
        ++line;
        if (p + 1 < n) {
          is_seq = kind[line] == LINE_SEQ;
          start = p + 1;
          if (is_seq && hdr_before[line] == 0) { out->bad = 1; is_seq = false; }
          base = is_seq ? seq_before[line] + hdr_before[line] - 1 : 0;
        }
      } else if (is_seq && !(c == '\r' && (p + 1 == n || text[p + 1] == '\n'))) {
        seq[base + (p - start)] = c;                                    // as line_bounds: only a line's final '\r' is dropped
      }
    }
  }
}

// separators between records ('N': no window spans two records); lengths
__global__ void record_finish_kernel(const ReadsInfo *info, const uint64_t *__restrict__ rec_off, uint8_t *__restrict__ seq) {
  const uint64_t nrec = info->n_records;
  for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < nrec; r += (uint64_t)gridDim.x * blockDim.x)
    seq[rec_off[r + 1] - 1] = 'N';
}

// Counting every record at once (count.kmers over a character vector, src/kmer_hash.c:580-587): the packed buffer is one
// sequence whose records are separated by breakers, with two corrections so that it yields exactly the windows the reference
// takes record by record: records of length <= k are skipped there (:582-583) -> blanked with 'N'; and a record whose last
// N-free run is exactly k long loses that window (the end-of-string rule, src/kmer_pos.c:81-83 = src/kmer_hash.c:238-239)
// -> its last base becomes 'N', which removes that window and no other.
__global__ void mask_for_counting_kernel(const ReadsInfo *info, const uint64_t *__restrict__ rec_off, int k, uint8_t *__restrict__ seq) {
  const uint64_t nrec = info->n_records;
  for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < nrec; r += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t o = rec_off[r], len = rec_off[r + 1] - 1 - o;
    if (len <= (uint64_t)k) { for (uint64_t j = 0; j < len; ++j) seq[o + j] = 'N'; continue; }
    bool clean = true;                                                    // last k bases free of breakers?
    for (int j = 0; j < k && clean; ++j) clean = (seq[o + len - 1 - j] | 0x20) != 'n';
    if (clean && (seq[o + len - 1 - k] | 0x20) == 'n') seq[o + len - 1] = 'N';
  }
}

}  // namespace kmg
