/*
 * kmergpu.h -- C ABI of libkmergpu, the B200 (sm_100a) k-mer position index that stands in
 * for kmer_hasheR's khash/kvec engine.
 *
 * This is the drop-in boundary.  The reference's R glue (src/kmer_hash.c) calls plain C
 * functions of src/kmer_pos.c to build, read and probe the index; a maintainer replaces those
 * calls by the functions below (see INTEGRATION.md and kmer_hasher_b200/rglue/kmer_hash.c).
 * Citations are file:line in the reference checkout.
 *
 * Conventions
 *   - every function returns KMG_OK (0) or a negative kmg_status; it never throws, aborts,
 *     exits or longjmps.  kmg_last_error() gives the message for the calling thread.
 *   - `seq`, `q` and every output pointer may address pageable host memory, pinned host memory
 *     (kmg_host_alloc) or device memory of the current device; the library looks the pointer up.
 *   - sequences are byte strings with an explicit length (the reference scans for the NUL of an
 *     R CHARSXP, which cannot contain one).
 *   - all coordinates are 1-based 32-bit ints exactly as the reference returns them.
 *   - the reference orders k-mers by khash bucket, which is not semantic; here they are ordered by
 *     ascending 2-bit key (KMG_ORDER_SORTED) or by a mix of the key (KMG_ORDER_GROUPED, the faster
 *     build), see kmg_build_ordered.
 */
#ifndef KMERGPU_H
#define KMERGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KMG_MAX_K 32 /* MAX_K, src/kmer_util.h:12 */

typedef enum {
  KMG_OK = 0,
  KMG_ERR_ARG = -1,    /* NULL / negative / inconsistent argument                        */
  KMG_ERR_K = -2,      /* k outside [1,32]            (guard of src/kmer_hash.c:515)      */
  KMG_ERR_RANGE = -3,  /* a size does not fit the reference's `int` coordinates/extents  */
  KMG_ERR_CUDA = -4,   /* CUDA runtime error; message carries the CUDA error string       */
  KMG_ERR_NOMEM = -5,  /* host or device allocation failed                                */
  KMG_ERR_NODEV = -6,  /* no usable sm_100 device                                         */
  KMG_ERR_UNSTABLE = -7 /* (builds from records) the always-on check found a position list not ascending: the
                          one-atomic sort variant's hardware assumption failed; it is now disabled: rebuild */
} kmg_status;

typedef struct kmg_index kmg_index; /* replaces khash_ptr            (src/kmer_pos.h:43-48)  */
typedef struct kmg_query kmg_query; /* replaces the kmer_ppos result (src/kmer_pos.h:41)     */
typedef struct kmg_join kmg_join;   /* the result of kmer.pairs      (src/kmer_hash.c:1177)   */

/* ---- library / device -------------------------------------------------------------------- */
const char *kmg_last_error(void);
int kmg_version(void);
int kmg_device_count(int *n);
int kmg_set_device(int device);          /* device used by this thread's subsequent calls      */
int kmg_set_stream(void *cuda_stream);   /* run this thread's work on a caller stream (0 = own)  */
void *kmg_host_alloc(size_t bytes);      /* pinned host memory: full-speed PCIe for in/outputs   */
void kmg_host_free(void *p);

/* ---- make.kmer.hash ------------------------------------------------------------------------
 * kmg_build replaces   seq_to_hash(seq, k, hash)              src/kmer_pos.c:66-98
 *   (and through it    init_kmer / skip_n                     src/kmer_util.c:4-32,
 *                      kmer_h_insert / kh_put / kv_push       src/kmer_pos.c:36-50)
 * as called from       make_kmer_h_index                      src/kmer_hash.c:524-527.
 * It indexes every window the reference would insert (see DESIGN.md "window rule"), position =
 * 1-based start.  The length guard `length(seq) <= k` (src/kmer_hash.c:519) belongs to the
 * glue, as in the reference: like the C core, kmg_build accepts any len >= 0.
 * sort_kmer_pos (src/kmer_pos.c:21-33, do.sort) has no counterpart: lists are always ascending.
 */
int kmg_build(const char *seq, int64_t len, int k, kmg_index **out);   /* = kmg_build_ordered(..., KMG_ORDER_GROUPED, ...) */

/* The order of the k-mers in an index (and so the meaning of the k-mer number i) is not semantic: the
 * reference's is its hash table's bucket order.  KMG_ORDER_SORTED: ascending 2-bit key (A<C<T<G, first base
 * most significant), ceil(2k/8) radix passes.  KMG_ORDER_GROUPED: the records are sorted on 32 bits (40 beyond
 * 400 M records) of a bijective mix of the key, which tells almost all k-mers of a genome apart in 4 passes; the
 * few groups in which k-mers that share those bits interleave are partitioned afterwards.  k-mers then come in the
 * order of those bits; used when it saves passes (k >= 21), otherwise the build is sorted.  Everything else
 * (positions ascending per k-mer, counts, pairs, probes) is identical; kmg_index_order tells which. */
#define KMG_ORDER_GROUPED 0
#define KMG_ORDER_SORTED 1
int kmg_build_ordered(const char *seq, int64_t len, int k, int order, kmg_index **out);
int kmg_index_order(const kmg_index *idx);

/* replaces clear_kmer_h (src/kmer_pos.c:10-19) + the finaliser body (src/kmer_hash.c:56-66).
 * NULL is accepted. */
int kmg_free(kmg_index *idx);

/* U = distinct k-mers (kh_size, src/kmer_hash.c:1090), N = indexed windows = rows of `pos`,
 * P = sum n(n-1)/2 = rows of `pair.pos`.  Any pointer may be NULL; P is computed (one sweep of the index, then
 * cached) the first time it is asked for, so callers that do not emit pairs pass NULL (the reference, too, walks the
 * lists for pairs only under opt.flag 4, src/kmer_hash.c:1113). */
int kmg_sizes(const kmg_index *idx, uint64_t *U, uint64_t *N, uint64_t *P);
int kmg_index_k(const kmg_index *idx);   /* khash_ptr.k, src/kmer_pos.h:45 */

/* ---- kmer.pos: the four fields of kmer_positions, src/kmer_hash.c:1054-1147 --------------------
 * Each writes directly into the caller's (R-allocated) buffer; the glue sizes it from kmg_sizes
 * first, so nothing is staged twice (the reference's kvec + memcpy, :1127-1140).           */
int kmg_kmers_u64(const kmg_index *idx, uint64_t *keys /* U */);
/* flag 1: U strings of k upper-case bases + NUL, stride k+1 (kmer_seq, src/kmer_hash.c:123-133) */
int kmg_kmers_ascii(const kmg_index *idx, char *buf /* U*(k+1) */);
/* flag 8: list lengths (src/kmer_hash.c:1103-1104) */
int kmg_counts(const kmg_index *idx, int32_t *counts /* U */);
/* flag 2: column-major 2 x N = interleaved (i,pos) (src/kmer_hash.c:1109-1112) */
int kmg_positions(const kmg_index *idx, int32_t *out /* 2N */);
/* flag 4: column-major 3 x P = interleaved (i,x,y), x<y, x slowest (src/kmer_hash.c:1113-1120).
 * kmg_pairs_chunk writes rows [first, first+n) so > 2^31-row results can be streamed. */
int kmg_pairs(const kmg_index *idx, int32_t *out /* 3P */);
int kmg_pairs_chunk(const kmg_index *idx, uint64_t first, uint64_t n, int32_t *out /* 3n */);
/* The same two with the k-mer number offset by i_base: the owners of a sharded index each write their slice of ONE
 * caller matrix with global k-mer numbers (i_base = distinct k-mers of the owners before; SURVEY.md 8e "Extraction"). */
int kmg_positions_base(const kmg_index *idx, uint64_t i_base, int32_t *out);
int kmg_pairs_chunk_base(const kmg_index *idx, uint64_t i_base, uint64_t first, uint64_t n, int32_t *out);

/* ---- seq.kmer.pos --------------------------------------------------------------------------
 * kmg_query_begin + kmg_query_emit replace seq_kmer_positions  src/kmer_pos.c:110-136
 *   (kmer_pos lookup :55-60, pair_positions_push :101-108) as called from
 *   sequence_kmer_positions, src/kmer_hash.c:1166-1170.
 * begin encodes the query with its own k (never compared with the index's k, as in the
 * reference), matches it and reports M = number of (i,j) rows; emit writes them: i = 1-based END
 * of the query k-mer, j = 1-based start in the index, ordered by i then j.  k <= 32 is accepted;
 * the reference's R-level limit k <= 31 (src/kmer_hash.c:1163) is the glue's business. */
int kmg_query_begin(const kmg_index *idx, const char *q, int64_t qlen, int k, kmg_query **st,
                    uint64_t *M);
/* the same probe with reverseComplement(q) taken on the device (every dot plot of test.R:43-52,73 probes
 * both strands; the reference's users make the reverse complement on the host): IUPAC complement, case
 * kept, N and every other byte unchanged; i is a coordinate of the reverse-complemented string. */
int kmg_query_begin_rc(const kmg_index *idx, const char *q, int64_t qlen, int k, kmg_query **st,
                       uint64_t *M);
int kmg_query_emit(kmg_query *st, int32_t *out /* 2M */);
int kmg_query_emit_chunk(kmg_query *st, uint64_t first, uint64_t n, int32_t *out /* 2n */);
int kmg_query_free(kmg_query *st);

/* ---- kmer.pairs ----------------------------------------------------------------------------------
 * kmg_join_begin + kmg_join_emit replace kmer_pair_pos, src/kmer_hash.c:1174-1203 (kmer_hash.R:30-34):
 * for every k-mer of index `a` that index `b` also holds, the rows (a_pos, b_pos), a position outer,
 * b position inner (:1190-1195).  The reference walks a's hash buckets without kh_exist and crashes
 * (test.R:330-331); this is its evident intent, with a's k-mers taken in a's own k-mer order (kmg_index_order).  Keys
 * are compared as raw 2-bit codes, whatever k each index was built with, as kh_get does (:1185).
 * Both indexes must be on the same device.  M = number of rows. */
int kmg_join_begin(const kmg_index *a, const kmg_index *b, kmg_join **st, uint64_t *M);
int kmg_join_emit(kmg_join *st, int32_t *out /* 2M */);
int kmg_join_emit_chunk(kmg_join *st, uint64_t first, uint64_t n, int32_t *out /* 2n */);
int kmg_join_free(kmg_join *st);

/* ---- dot plots: seq.kmer.pos / kmer.pairs rows counted into an image on the device (additive) -----------------------
 * What a dot plot draws is the 2-D histogram of those rows, which needs nx*ny counts instead of M rows: no 2^31-1 row
 * limit and no transfer of the rows.  kmg_query_dotplot bins the rows kmg_query_begin (rc = 0) or kmg_query_begin_rc
 * (rc = 1) + kmg_query_emit give for (idx, q, qlen, k), x = i (1-based END of the query window; with rc = 1 a coordinate
 * of the reverse-complemented string), y = j (1-based start in the index).  kmg_join_dotplot bins the rows of
 * kmg_join_begin + kmg_join_emit, x = position in a, y = position in b (same device).
 * max_count: 0 = no limit; else a k-mer with more than max_count positions in the index (in a join: in either index)
 * adds no rows -- how dot plots suppress repeats.
 * Windows are half-open, 0 <= x0 < x1 <= 2^31 (y alike): a row counts iff x0 <= x < x1 and y0 <= y < y1, into bin
 * bx = floor((x - x0) * nx / (x1 - x0)), by likewise (exact integer arithmetic).  out: nx*ny doubles, column-major,
 * out[bx + by*nx] (an R matrix with nx rows); every cell is written (exact below 2^53), nothing else is touched; device,
 * pinned or pageable memory.  An empty index, query or intersection gives an all-zero image.
 * KMG_ERR_ARG: NULL handle or out, nx or ny < 1, an empty or out-of-range window, rc not 0/1; KMG_ERR_RANGE: nx*ny >
 * INT32_MAX, or the query length check of kmg_query_begin; KMG_ERR_K as there. */
int kmg_query_dotplot(const kmg_index *idx, const char *q, int64_t qlen, int k, int rc, int64_t x0, int64_t x1, int nx,
                      int64_t y0, int64_t y1, int ny, uint32_t max_count, double *out /* nx*ny */);
int kmg_join_dotplot(const kmg_index *a, const kmg_index *b, int64_t x0, int64_t x1, int nx, int64_t y0, int64_t y1, int ny,
                     uint32_t max_count, double *out /* nx*ny */);

/* ---- match segments: maximal diagonal runs of seq.kmer.pos rows, found on the device (additive) ---------------------
 * S = the rows kmg_query_begin (rc = 0) or kmg_query_begin_rc (rc = 1) + kmg_query_emit give for (idx, q, qlen, k): i =
 * 1-based END of the query window (with rc = 1 a coordinate of the reverse-complemented string), j = 1-based start in the
 * index.  max_count > 0: k-mers with more than max_count positions in the index add no rows (as kmg_query_dotplot).
 * A run is a maximal sequence of rows (i+t, j+t), t = 0..n-1, all in S: (i-1, j-1) and (i+n, j+n) are not in S.  Every
 * row is in exactly one run, so the n of all runs sum to |S|.  When the query's k is the index's, a run of n rows means
 * query bases [i-k+1, i+n-1] equal index bases [j, j+n+k-2] in 2-bit code (the window rule of the index aside).
 * kmg_segments_begin finds the runs with n >= min_rows (0 and 1: every run) and reports their number R; emit writes them
 * as interleaved int32 (i, j, n), column-major 3 x R like kmg_pairs, ordered by (i, j) of their first row (the order of
 * the rows of kmg_query_emit), into device, pinned or pageable memory; emit_chunk writes runs [first, first+n).  The
 * handle holds only the 12 R bytes of the result.  An empty index, query or intersection gives R = 0.
 * KMG_ERR_ARG: NULL handle/st/out, rc not 0/1, runs outside [0, R); KMG_ERR_K and the query length check (KMG_ERR_RANGE)
 * of kmg_query_begin; KMG_ERR_RANGE: more than 2^31 - 1 runs before the min_rows filter. */
typedef struct kmg_segments kmg_segments;
int kmg_segments_begin(const kmg_index *idx, const char *q, int64_t qlen, int k, int rc, uint32_t max_count,
                       uint32_t min_rows, kmg_segments **st, uint64_t *R);
int kmg_segments_emit(kmg_segments *st, int32_t *out /* 3R */);
int kmg_segments_emit_chunk(kmg_segments *st, uint64_t first, uint64_t n, int32_t *out /* 3n */);
int kmg_segments_free(kmg_segments *st);   /* NULL accepted */
/* kmer.pairs.segments: the runs of a join, for two indexes on one device (a == b allowed), x = 1-based position in a,
 * y = 1-based position in b.  rc = 0: S = the rows kmg_join_begin + kmg_join_emit give (keys compared as raw 2-bit codes,
 * whatever k each index has), runs (x+t, y+t) as above.  rc = 1: S = the rows (x, y) where b's k-mer at y is the code-space
 * reverse complement of a's k-mer at x (codes reversed, each code ^ 2; needs one k, else KMG_ERR_K), and a run is
 * antiparallel: rows (x+t, y-t), t = 0..n-1, all in S, (x-1, y+1) and (x+n, y-n) not in S.  max_count > 0: a k-mer with
 * more than max_count positions in either index adds no rows (rc = 1: a's k-mer in a, its reverse complement in b).
 * min_rows, R, the (x, y, n) triples of each run's first (smallest x) row ordered by (x, y), the handle and its emit /
 * emit_chunk / free are those of kmg_segments_begin.  With one k, forward: a[x, x+n+k-2] equals b[y, y+n+k-2] in 2-bit
 * code; rc = 1: a[x, x+n+k-2] is the code-space reverse complement of b[y-n+1, y+k-1] (the window rule aside).  An empty
 * index or no shared k-mer gives R = 0.  KMG_ERR_ARG: NULL a, b or st, rc not 0/1, indexes on different devices;
 * KMG_ERR_RANGE: more than 2^31 - 1 runs before the min_rows filter. */
int kmg_join_segments_begin(const kmg_index *a, const kmg_index *b, int rc, uint32_t max_count,
                            uint32_t min_rows, kmg_segments **st, uint64_t *R);

/* ---- chains: match segments joined across mismatches and short indels, found on the device (additive) ---------------
 * Input: the R runs a kmg_segments handle holds (after its own max_count and min_rows).  A run s = (i, j, n) has its first
 * row (i, j) and its last row (I, J) = (i+n-1, j+n-1), or (i+n-1, j-n+1) for antiparallel runs (kmg_join_segments_begin
 * with rc = 1).  For an ordered pair (s, t): gq = i_t - I_s - 1, gr = j_t - J_s - 1 (antiparallel: J_s - j_t - 1); gq - gr
 * is the difference of the two runs' diagonal keys (i - j, or i + j antiparallel).  t may follow s iff 0 <= gq <= G,
 * 0 <= gr <= G and |gq - gr| <= W (G = max_gap, W = max_shift): runs that overlap in either coordinate never follow one
 * another.  The cost c(s, t) = (max(gq, gr), |gq - gr|, gq) is compared lexicographically; succ(s) is the t of least cost
 * that may follow s, pred(t) the s of least cost that t may follow (both unique when they exist).  s -> t is a link iff
 * succ(s) = t and pred(t) = s, and a chain is a maximal path of links (a run without one is a chain of one).  Per chain:
 * (i, j) = first row of its first run, (I, J) = last row of its last run, n = the sum of its runs' n, m = its number of
 * runs; interleaved int32 (i, j, I, J, n, m), column-major 6 x C, ordered by (i, j), only chains with n >= min_rows (0 and
 * 1 keep all).  Before that filter the m sum to R and the n to the runs' n.  G = 0 gives the runs themselves (m = 1).  An
 * isolated substitution leaves gq = gr = k on one diagonal, a 1-base indel (k, k-1) or (k-1, k), so G >= k bridges
 * isolated differences and W is the longest indel bridged.  Bases covered, for one k: seq.kmer.segments query
 * [i-k+1, I], index [j, J+k-1]; a forward join a [i, I+k-1], b [j, J+k-1]; an antiparallel join a [i, I+k-1], b [J, j+k-1].
 * kmg_chains_begin leaves seg unchanged (it can still be emitted, and is freed by its owner); the chains handle holds
 * only the 24 C bytes of the result; emit / emit_chunk write to device, pinned or pageable memory like
 * kmg_segments_emit.  C may be NULL; an empty handle gives C = 0.  KMG_ERR_ARG: NULL seg or st, max_gap >= 2^31,
 * max_shift > max_gap or > 1024 (the search visits every occupied diagonal of the band), seg on another device than the
 * calling thread, chains outside [0, C). */
typedef struct kmg_chains kmg_chains;
int kmg_chains_begin(const kmg_segments *seg, uint32_t max_gap, uint32_t max_shift, uint32_t min_rows,
                     kmg_chains **st, uint64_t *C);
int kmg_chains_emit(kmg_chains *st, int32_t *out /* 6C */);
int kmg_chains_emit_chunk(kmg_chains *st, uint64_t first, uint64_t n, int32_t *out /* 6n */);
int kmg_chains_free(kmg_chains *st);   /* NULL accepted */

/* ---- sharded build (one process per GPU; the exchange itself is the host's NCCL all-to-all) ----
 * A rank holds bytes [g0,g1) of a global sequence of length L in device memory at d_seq (d_seq[0]
 * is byte g0) and owns the window starts [s0,s1), g0 <= max(s0-1,0), g1 >= min(L, s1+k-1).
 * kmg_shard_sample    : n evenly spaced window keys of the shard (for splitter selection).
 * kmg_shard_partition : encodes the shard's windows and groups the (key,pos) records by owner
 *                       (owner r holds keys in [splitters[r-1], splitters[r])), keeping sequence
 *                       order inside each group; pos is global and 1-based.  counts[nparts] is host.
 * kmg_build_records   : builds an index from device records (e.g. the concatenation, in source
 *                       rank order, of what the all-to-all delivered).  Input arrays are consumed
 *                       as scratch but stay owned by the caller.
 */
int kmg_shard_sample(const void *d_seq, int64_t g0, int64_t g1, int64_t L, int64_t s0, int64_t s1,
                     int k, int n, uint64_t *d_samples);
int kmg_shard_partition(const void *d_seq, int64_t g0, int64_t g1, int64_t L, int64_t s0,
                        int64_t s1, int k, const uint64_t *splitters /* host, nparts-1 */,
                        int nparts, uint64_t *d_keys, uint32_t *d_pos, uint64_t *counts);
int kmg_build_records(uint64_t *d_keys, uint32_t *d_pos, int64_t n, int k, kmg_index **out);
/* match pre-encoded query records (key, i) against the index: rows (i,j) ordered as given */
int kmg_query_records(const kmg_index *idx, const uint64_t *d_keys, const int32_t *d_i, int64_t n,
                      kmg_query **st, uint64_t *M);

/* ---- sharded build over peer memory (NVLink): the fused partition + exchange -----------------------
 * The partitioning pass writes every record straight into the arrays of the GPU that owns its key
 * range (peer memory mapped with kmg_ipc_open), so there is no staging copy and no all-to-all; the
 * host only all-gathers the G x G count matrix and issues one barrier.  No call below synchronises
 * with the host except kmg_build_received / kmg_query_received (they read the result's sizes).
 * kmg_shard_open    : aligned, padded device copy of a rank's bytes [g0,g1) (arguments as above).
 * kmg_shard_sample_keys / kmg_shard_count : splitter sample; counts[nparts] (device) of the shard's
 *                     records per owner for device-resident splitters.
 * kmg_shard_scatter : encodes the shard and writes owner b's records to peer_keys[b]/peer_pos[b]
 *                     (capacity records each) behind those of lower ranks; d_matrix[src][owner] is the
 *                     all-gathered count matrix (device).  pos_add is added to the 1-based start
 *                     (k-1 gives the reference's query coordinate).  d_info[0] = records this rank
 *                     receives, d_info[1] = 1 if an owner would overflow (its surplus is dropped and
 *                     kmg_build_received / kmg_query_received then fail with KMG_ERR_RANGE).
 * `order` (kmg_shard_pack, kmg_shard_open_packed, kmg_build_received; the same value on every rank):
 * with KMG_ORDER_GROUPED and k >= 21 the sample, the owner ranges and the exchanged records are those of
 * the mixed key (see kmg_build_ordered) and every owner builds a grouped index; query records scattered
 * from a shard opened that way carry the mix too (kmg_query_received: mixed = 1).
 */
typedef struct kmg_shard kmg_shard;
int kmg_shard_open(const void *d_seq, int64_t g0, int64_t g1, int64_t L, int64_t s0, int64_t s1,
                   int k, kmg_shard **out);
 /* halo + splitter sample in ONE exchange: every rank packs its first k-1 bytes, its last byte and
 * n_samples (a power of two <= 4096) ascending sample keys into kmg_shard_pack_bytes(n_samples) bytes;
 * the packs are all-gathered ([world][bytes]); kmg_shard_open_packed assembles the shard of `rank`
 * (its own bytes [rank*per, (rank+1)*per) of L, per = ceil(L/world), plus halo) and writes the
 * world-1 splitters (element j*total/world of all samples in ascending order) to d_splitters. */
int kmg_shard_pack_bytes(int n_samples);
int kmg_shard_pack(const void *d_own, int64_t n_own, int k, int n_samples, int order, void *d_pack);
int kmg_shard_open_packed(const void *d_own, int64_t n_own, int64_t L, int world, int rank, int k,
                          int n_samples, int order, const void *d_allpack, kmg_shard **out,
                          uint64_t *d_splitters);
int kmg_shard_close(kmg_shard *sh);
int kmg_shard_set_mixed(kmg_shard *sh, int mixed);   /* route by mix64(key): queries against a grouped sharded index */
int kmg_shard_windows(const kmg_shard *sh, int64_t *nstarts);
int kmg_shard_sample_keys(const kmg_shard *sh, int n, uint64_t *d_samples);
int kmg_shard_count(const kmg_shard *sh, const uint64_t *d_splitters, int nparts, uint64_t *d_counts);
int kmg_shard_scatter(const kmg_shard *sh, const uint64_t *d_splitters, int nparts, int rank,
                      void *const *peer_keys, void *const *peer_pos, uint64_t capacity,
                      const uint64_t *d_matrix, int32_t pos_add, uint64_t *d_info);
int kmg_build_received(uint64_t *d_keys, uint32_t *d_pos, uint64_t capacity, const uint64_t *d_info,
                       int k, int order, kmg_index **out);
int kmg_query_received(const kmg_index *idx, const uint64_t *d_keys, const int32_t *d_i,
                       uint64_t capacity, const uint64_t *d_info, int mixed, kmg_query **st,
                       uint64_t *M);
/* Region exchange (grouped order, k >= 21): owners are nparts EQUAL ranges of the mixed key -- uniform whatever the
 * sequence, so nothing is sampled, counted or exchanged before the scatter.  Every source rank has its own region of
 * region_cap slots in every owner's arrays (region r starts at r * region_cap); the scatter's last tile stores the number
 * of records this rank sent to owner b in peer_counts[b][rank].  The owner then builds from / probes its regions. */
int kmg_shard_scatter_ranges(const kmg_shard *sh, int nparts, int rank, void *const *peer_keys, void *const *peer_pos,
                             void *const *peer_counts, uint64_t region_cap, int32_t pos_add);
int kmg_build_regions(uint64_t *d_keys, uint32_t *d_pos, uint64_t region_cap, int nparts, const uint64_t *d_counts, int k,
                      kmg_index **out);
int kmg_query_regions(const kmg_index *idx, const uint64_t *d_keys, const int32_t *d_i, uint64_t region_cap, int nparts,
                      const uint64_t *d_counts, kmg_query **st, uint64_t *M);
/* device buffers other processes of the node can map (CUDA IPC); handle is 64 bytes */
int kmg_ipc_alloc(size_t bytes, void **dptr, void *handle);
int kmg_ipc_free(void *dptr);
int kmg_ipc_open(const void *handle, void **dptr);
int kmg_ipc_close(void *dptr);

/* ---- count.kmers (per-source k-mer counts) and spectra ---------------------------------------------------
 * kmg_count_add replaces  seq_to_counts / kmer_count_insert   src/kmer_hash.c:185-252
 * as called from          count_kmers                         src/kmer_hash.c:548-591  (count.kmers, kmer_hash.R:43-46).
 * The reference keeps source_n counters per distinct k-mer in the same hash type as the position index and bumps
 * column `source` once per window; the table is read back with kmer.pos (rows (i, count of source s)).  Here the
 * k-mers of a table are ordered by ascending key.  Spectra: spec[min(count, max_count)] += 1 per k-mer, as doubles
 * (count_spectrum, src/kmer_tree.c:85-99, the shape kmer_spectrum_* return, src/kmer_hash.c:975-1038). */
typedef struct kmg_counter kmg_counter;
int kmg_count_new(int k, int source_n, kmg_counter **out);
int kmg_count_add(kmg_counter *c, const char *seq, int64_t len, int source);
int kmg_count_sizes(const kmg_counter *c, uint64_t *U, int *source_n, int *k, uint64_t *new_total);
int kmg_count_kmers_u64(const kmg_counter *c, uint64_t *keys /* U */);
int kmg_count_kmers_ascii(const kmg_counter *c, char *buf /* U*(k+1) */);
int kmg_count_matrix(const kmg_counter *c, int32_t *out /* U*source_n, one row per k-mer */);
int kmg_count_positions(const kmg_counter *c, int32_t *out /* 2*U*source_n: rows (i, count) as kmer.pos(ptr, 2) gives */);
int kmg_count_spectrum(const kmg_counter *c, int source /* < 0: summed over sources */, uint32_t max_count, double *spec /* max_count+1 */);
int kmg_index_spectrum(const kmg_index *idx, uint32_t max_count, double *spec /* max_count+1 */);
int kmg_count_free(kmg_counter *c);

/* ---- seq.kmer.depth: per-window k-mer counts along a sequence (additive; the reference has it only for its suffix-hash
 * counter, seq_kmer_depth_sh) ------------------------------------------------------------------------------------------
 * For every window start r = 0 .. nwin-1 of q, nwin = max(0, qlen - k + 1) with k = the handle's own k, row r of `out` is
 * the count of the window's k-mer: source_n int32 per row for a count table (the k-mer's row of the count matrix), one
 * for a position index (the length of its position list).  Row r is the window at 1-based start r+1 (= i - k + 1 of
 * seq.kmer.pos).  A k-mer absent from the table gives 0; a window the window rule does not emit (an N/n inside, or the
 * end-of-string rule; exactly the windows make.kmer.hash skips) gives INT32_MIN = R's NA_integer_ in every column.
 * KMG_STRAND_BOTH: count(key) + count(rc(key)), rc = the reverse complement in code space (the k 2-bit codes reversed,
 * each complemented as code ^ 2: A<->T, C<->G); a palindrome (rc(key) == key, even k only) counts once; sums saturate at
 * INT32_MAX; validity is the forward window's.  For ACGT/acgt bytes rc(key) is the key of the same window in
 * kmg_query_begin_rc's string; for other non-N bytes it is not (that routine complements bytes IUPAC-style, R -> Y, this
 * complements the code the byte was given).  `q` and `out` may be host (pageable or pinned) or device memory.  The first
 * call on a count table builds its key table (cached; kmg_count_add drops it). */
#define KMG_STRAND_FORWARD 0
#define KMG_STRAND_BOTH 1
int kmg_count_depth(const kmg_counter *c, const char *q, int64_t qlen, int strands, int32_t *out /* nwin * source_n */);
int kmg_index_depth(const kmg_index *idx, const char *q, int64_t qlen, int strands, int32_t *out /* nwin */);

/* ---- FASTA / FASTQ ingestion (SURVEY.md 8f rank 4) ---------------------------------------------------------
 * Replaces, for the index path, what the reference does with klib's kseq.h over zlib (src/kseq.h; read loop
 * src/kmer_reader.c:41-77): the host inflates the file, the DEVICE finds and classifies the lines and packs the records'
 * sequences (csrc/reads.cuh).  Record names are the header up to the first white space; line ends (and a trailing CR)
 * are removed.  FASTA may be multi-line; FASTQ must be the four-line form.  An index is then built from a record without
 * the sequence ever being an R string (no 2^31-1 limit on the file, no host copy), and count.kmers can take a whole file. */
typedef struct kmg_reads kmg_reads;
int kmg_reads_open(const char *path, kmg_reads **out);                       /* plain or gz */
int kmg_reads_from_memory(const void *text, int64_t len, kmg_reads **out);   /* inflated file contents, host or device */
int kmg_reads_count(const kmg_reads *r, uint64_t *n_records, uint64_t *total_bases);
int kmg_reads_record(const kmg_reads *r, uint64_t i, int64_t *seq_len, char *name_buf, int name_cap);
int kmg_reads_sequence(const kmg_reads *r, uint64_t i, char *out /* seq_len bytes, host or device */);
int kmg_build_record(const kmg_reads *r, uint64_t i, int k, int order, kmg_index **out);  /* make.kmer.hash on record i */
int kmg_count_add_reads(kmg_counter *c, const kmg_reads *r, int source);     /* count.kmers over every record */
int kmg_reads_free(kmg_reads *r);

/* ---- instrumentation (bench.py / profiles) ------------------------------------------------------ */
int kmg_profile_enable(int on);          /* bracket every kernel with CUDA events               */
int kmg_profile_reset(void);
int kmg_profile_count(void);             /* number of distinct kernels seen                     */
int kmg_profile_get(int i, const char **name, double *total_ms, uint64_t *launches,
                    double *algo_bytes);
uint64_t kmg_launch_count(void);         /* kernels launched by this library since load         */
int kmg_selftest_lane_order(uint32_t *failures); /* precondition of the one-atomic rank variant (sort.cuh) */
int kmg_tune(const char *key, int value); /* tests and tuning runs: "sort_cfg" (rank variant: -1 auto, 0 bitmap, 3 one
                                            atomic, 4 unstable on purpose), "sort_shape" (-1 auto, 0..2), "hash_bits" (0 = from the
                                            record count), "hash_rb", "fix_cap", "reset_rank", "sort_dbg" (bit 2: generic write-out of
                                            the NVLink scatter, bit 3 / bit 4: keys / positions by register loads instead of the bulk copy), "sort_trace" */
int64_t kmg_tune_get(const char *key, int64_t arg); /* "rank_variant" in use on this device, "unstable_rebuilds" so far,
                                            "hash_bits" / "hash_rb" the grouped build picks for `arg` records */
int kmg_trim(void);                      /* return the library's cached (free) device blocks of this device to the driver */
uint64_t kmg_cached_bytes(void);         /* bytes held in that cache (KMERGPU_CACHE_MB caps it; default a quarter of the device) */

#ifdef __cplusplus
}
#endif
#endif /* KMERGPU_H */
