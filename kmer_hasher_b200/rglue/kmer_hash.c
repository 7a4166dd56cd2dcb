/*
 * kmer_hash.c -- R glue of the B200 k-mer position index: the drop-in replacement for the three
 * index entry points of the reference's src/kmer_hash.c.  It exports the same .Call names with the
 * same arity, argument types, return layouts, external-pointer tag and finaliser convention, so the
 * reference's kmer_hash.R (make.kmer.hash / kmer.pos / seq.kmer.pos, kmer_hash.R:5-28) works
 * unchanged when this file is built as src/kmer_hash.so.  All work is done by libkmergpu
 * (include/kmergpu.h); nothing here builds a hash table and there is no CPU path.
 *
 *   make_kmer_h_index(seq, k, do.sort)      replaces src/kmer_hash.c:506-540
 *   kmer_positions(ptr, opt.flag)           replaces src/kmer_hash.c:1054-1147
 *   sequence_kmer_positions(ptr, seq, k)    replaces src/kmer_hash.c:1151-1172
 *   kmer_pair_pos(ptr.a, ptr.b)             replaces src/kmer_hash.c:1174-1203 (which crashes: test.R:330-331)
 *   count_kmers(ptr, params, seq)           replaces src/kmer_hash.c:548-591 (count.kmers: per-source counts)
 *   sequence_kmer_depth(ptr, seq, strands)  additive: per-window counts of a sequence's k-mers (seq.kmer.depth)
 *   sequence_kmer_dotplot(ptr, seq, k, params), kmer_pair_dotplot(ptr.a, ptr.b, params)
 *                                           additive: binned dot plots of seq.kmer.pos / kmer.pairs rows
 *   R_init_kmer_hash                        replaces src/kmer_hash.c:1221-1224
 *
 * Differences a user can observe: k-mers come out in the order of a mix of their 2-bit key (ascending key
 * with do.sort = TRUE) instead of khash bucket order (not semantic); results too large for an R matrix raise a clean error before anything is
 * allocated (the reference overflows or leaks, README "pair.pos"); do.sort is a no-op (lists are
 * always ascending).  Set KMERGPU_ALLOW_K32=1 to lift the reference's k <= 31 limit of seq.kmer.pos
 * (its C core handles 32; the limit is only in its R entry, src/kmer_hash.c:1163).
 *
 * Built against R's headers on a machine with R, or against rstub/ (a minimal R C-API stand-in)
 * where R is absent, which is how tests/test_rglue.py drives it.
 */
#include <R.h>
#include <Rinternals.h>
#include <limits.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "kmergpu.h"

#define KMER_HASH_TAG "kmer_hash_250930" /* src/kmer_hash.c:22 */
enum { F_KMER = 1, F_POS = 2, F_PAIRS = 4, F_COUNT = 8 }; /* pos_opt_flags, src/kmer_hash.c:17 */
static const char *const field_names[4] = {"kmer", "pos", "pair.pos", "count"}; /* :18 */

/* what the external pointer addresses (the reference's khash_ptr, src/kmer_pos.h:43-48) */
typedef struct {
  kmg_index *index;     /* make.kmer.hash: positions */
  kmg_counter *counter; /* count.kmers: per-source counts (the reference keeps both kinds in the same khash type) */
  int k;
} kmer_handle;

/* Tag-checked unwrap that never raises: safe inside the finaliser. */
static kmer_handle *handle_or_null(SEXP ptr) {
  if (TYPEOF(ptr) != EXTPTRSXP) return NULL;
  SEXP tag = R_ExternalPtrTag(ptr);
  if (TYPEOF(tag) != STRSXP || length(tag) != 1 || strcmp(CHAR(STRING_ELT(tag, 0)), KMER_HASH_TAG) != 0) return NULL;
  return (kmer_handle *)R_ExternalPtrAddr(ptr);
}

/* The same with the reference's errors (extract_khash_ptr, src/kmer_hash.c:491-503). */
static kmer_handle *handle_or_error(SEXP ptr) {
  if (TYPEOF(ptr) != EXTPTRSXP) error("ptr_r should be an external pointer");
  kmer_handle *h = handle_or_null(ptr);
  if (!h) {
    SEXP tag = R_ExternalPtrTag(ptr);
    if (TYPEOF(tag) != STRSXP || length(tag) != 1 || strcmp(CHAR(STRING_ELT(tag, 0)), KMER_HASH_TAG) != 0)
      error("External pointer has incorrect tag");
    error("external pointer is NULL");
  }
  if (!h->index && !h->counter) error("the k-mer index has been released");
  return h;
}
static kmer_handle *index_handle_or_error(SEXP ptr) {
  kmer_handle *h = handle_or_error(ptr);
  if (!h->index) error("this external pointer holds k-mer counts (count.kmers), not a position index");
  return h;
}

/* Runs from the garbage collector or at exit: frees the device index once, tolerates a cleared
 * pointer, never calls error() (convention stated at src/kmer_hash.c:37-40). */
static void finalise_handle(SEXP ptr) {
  kmer_handle *h = handle_or_null(ptr);
  if (!h) return;
  if (h->index) {
    kmg_free(h->index);
    h->index = NULL;
  }
  if (h->counter) {
    kmg_count_free(h->counter);
    h->counter = NULL;
  }
  free(h);
  R_ClearExternalPtr(ptr);
}

SEXP make_kmer_h_index(SEXP seq_r, SEXP k_r, SEXP sort_pos_r) {
  if (TYPEOF(seq_r) != STRSXP || length(seq_r) < 1) error("seq_r should be a character vector of length at least one");
  if (TYPEOF(k_r) != INTSXP || length(k_r) < 1) error("k_r must be an integer vector of length at least one");
  if (TYPEOF(sort_pos_r) != INTSXP || length(sort_pos_r) < 1) error("sort_pos_r must be an integer vector of length at least one");
  const int k = INTEGER(k_r)[0];
  if (k < 1 || k > KMG_MAX_K) error("k must be a positive integer less than 1+MAX_K");
  SEXP s = STRING_ELT(seq_r, 0); /* like the reference, only the first element is indexed */
  const int len = length(s);
  if (len <= k) error("the length of the sequence must be at least k");

  kmer_handle *h = (kmer_handle *)calloc(1, sizeof *h);
  if (!h) error("out of memory");
  h->k = k;
  /* do.sort: position lists are always ascending, so there is nothing to sort there (src/kmer_pos.c:21-33 is a
   * no-op in the reference too); it selects the order of the k-mers instead: TRUE = ascending key, FALSE (the R
   * default) = the faster grouped build.  Neither order is semantic (the reference's is khash bucket order). */
  const int order = INTEGER(sort_pos_r)[0] ? KMG_ORDER_SORTED : KMG_ORDER_GROUPED;
  if (kmg_build_ordered(CHAR(s), (int64_t)len, k, order, &h->index) != KMG_OK) {
    free(h);
    error("make.kmer.hash failed: %s", kmg_last_error());
  }
  SEXP tag = PROTECT(allocVector(STRSXP, 1));
  SET_STRING_ELT(tag, 0, mkChar(KMER_HASH_TAG));
  SEXP ptr = PROTECT(R_MakeExternalPtr(h, tag, R_NilValue));
  R_RegisterCFinalizerEx(ptr, finalise_handle, TRUE);
  UNPROTECT(2);
  return ptr;
}

/* kmer.pos() of a count table: the reference's kmer_positions walks v.a[0..v.n) of every k-mer, and count.kmers
 * keeps the source_n counters there (src/kmer_hash.c:196-205), so "pos" = rows (i, count of source 0), (i, count of
 * source 1), ..., "count" = source_n for every k-mer, "pair.pos" = rows (i, c_a, c_b) for a < b, "kmer" as usual. */
static SEXP count_table_positions(kmer_handle *h, unsigned flag) {
  uint64_t U = 0;
  int sn = 0;
  if (kmg_count_sizes(h->counter, &U, &sn, NULL, NULL) != KMG_OK) error("kmer.pos failed: %s", kmg_last_error());
  const uint64_t N = U * (uint64_t)sn, P = U * (uint64_t)sn * (uint64_t)(sn - 1) / 2;
  if ((flag & (F_KMER | F_COUNT)) && U > (uint64_t)INT_MAX) error("%llu distinct k-mers do not fit an R vector", (unsigned long long)U);
  if ((flag & F_POS) && N > (uint64_t)INT_MAX) error("%llu rows do not fit an R matrix", (unsigned long long)N);
  if ((flag & F_PAIRS) && P > (uint64_t)INT_MAX) error("pair.pos would have %llu rows, more than an R matrix can hold (2^31-1)", (unsigned long long)P);
  SEXP ret = PROTECT(allocVector(VECSXP, 4));
  SEXP names = PROTECT(allocVector(STRSXP, 4));
  for (int i = 0; i < 4; ++i) SET_STRING_ELT(names, i, mkChar(field_names[i]));
  setAttrib(ret, R_NamesSymbol, names);
  UNPROTECT(1);
  const char *failed = NULL;
  if (flag & F_KMER) {
    const size_t stride = (size_t)h->k + 1;
    char *buf = R_alloc(U ? U : 1, (int)stride);
    if (kmg_count_kmers_ascii(h->counter, buf) != KMG_OK) failed = "kmer";
    else {
      SEXP kmers = allocVector(STRSXP, (R_xlen_t)U);
      SET_VECTOR_ELT(ret, 0, kmers);
      for (uint64_t u = 0; u < U; ++u) SET_STRING_ELT(kmers, (R_xlen_t)u, mkCharLen(buf + u * stride, h->k));
    }
  }
  if (!failed && (flag & F_POS)) {
    SEXP m = allocMatrix(INTSXP, 2, (int)N);
    SET_VECTOR_ELT(ret, 1, m);
    if (kmg_count_positions(h->counter, INTEGER(m)) != KMG_OK) failed = "pos";
  }
  if (!failed && (flag & F_PAIRS)) {
    SEXP m = allocMatrix(INTSXP, 3, (int)P);
    SET_VECTOR_ELT(ret, 2, m);
    int *mat = (int *)R_alloc(N ? N : 1, sizeof(int));
    if (kmg_count_matrix(h->counter, mat) != KMG_OK) failed = "pair.pos";
    else {
      int *o = INTEGER(m);
      for (uint64_t u = 0; u < U; ++u)
        for (int a = 0; a < sn; ++a)
          for (int b = a + 1; b < sn; ++b) { *o++ = (int)(u + 1); *o++ = mat[u * sn + a]; *o++ = mat[u * sn + b]; }
    }
  }
  if (!failed && (flag & F_COUNT)) {
    SEXP v = allocVector(INTSXP, (R_xlen_t)U);
    SET_VECTOR_ELT(ret, 3, v);
    int *o = INTEGER(v);
    for (uint64_t u = 0; u < U; ++u) o[u] = sn;
  }
  UNPROTECT(1);
  if (failed) error("kmer.pos failed while extracting %s: %s", failed, kmg_last_error());
  return ret;
}

/* count.kmers(seq, c(k, source, source_n), hash.ptr) -> .Call("count_kmers", hash.ptr, params, seq), kmer_hash.R:43-46;
 * replaces src/kmer_hash.c:548-591 (and seq_to_counts / kmer_count_insert, :185-252): every sequence longer than k adds
 * its windows to column `source` of the table; a NULL pointer makes a new table. */
SEXP count_kmers(SEXP hash_ptr_r, SEXP params_r, SEXP seq_r) {
  if (TYPEOF(seq_r) != STRSXP || length(seq_r) < 1) error("seq_r should be a character vector of length at least one");
  if (TYPEOF(params_r) != INTSXP || length(params_r) != 3) error("k_r must be an integer vector of length 3");
  const int *params = INTEGER(params_r);
  const int k = params[0], source = params[1], source_n = params[2];
  if (k < 1 || k > KMG_MAX_K) error("k must be a positive integer less than 1+MAX_K");
  if (source_n < 1 || source >= source_n || source < 0) error("source_n must be larger than 1 and larger than source");
  SEXP ptr_r = hash_ptr_r;
  kmer_handle *h = NULL;
  int protect_n = 0;
  if (ptr_r == R_NilValue) {
    h = (kmer_handle *)calloc(1, sizeof *h);
    if (!h) error("out of memory");
    h->k = k;
    if (kmg_count_new(k, source_n, &h->counter) != KMG_OK) {
      free(h);
      error("count.kmers failed: %s", kmg_last_error());
    }
    SEXP tag = PROTECT(allocVector(STRSXP, 1));
    SET_STRING_ELT(tag, 0, mkChar(KMER_HASH_TAG));
    ptr_r = PROTECT(R_MakeExternalPtr(h, tag, R_NilValue));
    R_RegisterCFinalizerEx(ptr_r, finalise_handle, TRUE);
    protect_n = 2;
  } else {
    h = handle_or_null(hash_ptr_r);
  }
  if (!h) error("failed to extract kmer_hash from external pointer");
  if (!h->counter) { UNPROTECT(protect_n); error("the external pointer holds a position index, not k-mer counts"); }
  if (h->k != k) { UNPROTECT(protect_n); error("mismatch between specified k and that given in the external pointer"); }
  int sn = 0;
  kmg_count_sizes(h->counter, NULL, &sn, NULL, NULL);
  if (sn != source_n) { UNPROTECT(protect_n); error("mismatch between specified source_n and that of the external pointer"); }
  for (int i = 0; i < length(seq_r); ++i) {
    SEXP s = STRING_ELT(seq_r, i);
    if (length(s) <= k) continue;                              /* as the reference: too short to hold a k-mer */
    if (kmg_count_add(h->counter, CHAR(s), (int64_t)length(s), source) != KMG_OK) {
      UNPROTECT(protect_n);
      error("count.kmers failed: %s", kmg_last_error());
    }
  }
  UNPROTECT(protect_n);
  return ptr_r;
}

SEXP kmer_positions(SEXP ptr_r, SEXP opt_flag_r) {
  kmer_handle *h = handle_or_error(ptr_r);
  if (TYPEOF(opt_flag_r) != INTSXP || length(opt_flag_r) != 1) error("opt_flag_r should be an integer vector of length 1");
  const unsigned flag = (unsigned)asInteger(opt_flag_r);
  if (h->counter) return count_table_positions(h, flag);

  uint64_t U = 0, N = 0, P = 0;
  /* P (rows of pair.pos) costs a sweep of the index the first time: asked for only under flag 4, as the reference only
   * walks the lists for pairs there (src/kmer_hash.c:1113) */
  if (kmg_sizes(h->index, &U, &N, (flag & F_PAIRS) ? &P : NULL) != KMG_OK) error("kmer.pos failed: %s", kmg_last_error());
  /* size checks BEFORE any allocation: R vectors/matrix extents are int */
  if ((flag & (F_KMER | F_COUNT)) && U > (uint64_t)INT_MAX) error("%llu distinct k-mers do not fit an R vector", (unsigned long long)U);
  if ((flag & F_POS) && N > (uint64_t)INT_MAX) error("%llu positions do not fit an R matrix", (unsigned long long)N);
  if ((flag & F_PAIRS) && P > (uint64_t)INT_MAX)
    error("pair.pos would have %llu rows, more than an R matrix can hold (2^31-1); index a shorter region", (unsigned long long)P);

  SEXP ret = PROTECT(allocVector(VECSXP, 4));
  SEXP names = PROTECT(allocVector(STRSXP, 4));
  for (int i = 0; i < 4; ++i) SET_STRING_ELT(names, i, mkChar(field_names[i]));
  setAttrib(ret, R_NamesSymbol, names);
  UNPROTECT(1);

  const char *failed = NULL;
  if (flag & F_KMER) {
    const size_t stride = (size_t)h->k + 1;
    char *buf = R_alloc(U ? U : 1, (int)stride);          /* transient: R reclaims it, also on error() */
    if (kmg_kmers_ascii(h->index, buf) != KMG_OK) failed = "kmer";
    else {
      SEXP kmers = allocVector(STRSXP, (R_xlen_t)U);
      SET_VECTOR_ELT(ret, 0, kmers);
      for (uint64_t u = 0; u < U; ++u) SET_STRING_ELT(kmers, (R_xlen_t)u, mkCharLen(buf + u * stride, h->k));
    }
  }
  if (!failed && (flag & F_POS)) {
    SEXP m = allocMatrix(INTSXP, 2, (int)N);          /* rows (i,pos); kmer.pos() transposes it */
    SET_VECTOR_ELT(ret, 1, m);
    if (kmg_positions(h->index, INTEGER(m)) != KMG_OK) failed = "pos";
  }
  if (!failed && (flag & F_PAIRS)) {
    SEXP m = allocMatrix(INTSXP, 3, (int)P);          /* rows (i,x,y) */
    SET_VECTOR_ELT(ret, 2, m);
    if (kmg_pairs(h->index, INTEGER(m)) != KMG_OK) failed = "pair.pos";
  }
  if (!failed && (flag & F_COUNT)) {
    SEXP v = allocVector(INTSXP, (R_xlen_t)U);
    SET_VECTOR_ELT(ret, 3, v);
    if (kmg_counts(h->index, INTEGER(v)) != KMG_OK) failed = "count";
  }
  UNPROTECT(1);
  if (failed) error("kmer.pos failed while extracting %s: %s", failed, kmg_last_error());
  return ret;
}

/* allocMatrix() can longjmp (allocation failure, interrupt) while a kmg_query / kmg_join holds device memory: the state is
 * parked in an external pointer whose finaliser releases it, so nothing leaks past an R error. */
static void finalise_query_guard(SEXP g) {
  kmg_query *q = (kmg_query *)R_ExternalPtrAddr(g);
  if (q) kmg_query_free(q);
  R_ClearExternalPtr(g);
}
static void finalise_join_guard(SEXP g) {
  kmg_join *j = (kmg_join *)R_ExternalPtrAddr(g);
  if (j) kmg_join_free(j);
  R_ClearExternalPtr(g);
}

SEXP sequence_kmer_positions(SEXP ptr_r, SEXP seq_r, SEXP k_r) {
  kmer_handle *h = index_handle_or_error(ptr_r);
  if (TYPEOF(seq_r) != STRSXP || length(seq_r) != 1) error("seq_r should be a single sequence");
  if (TYPEOF(k_r) != INTSXP || length(k_r) != 1) error("k should be an integer of length 1");
  const int k = INTEGER(k_r)[0];
  SEXP s = STRING_ELT(seq_r, 0);
  const char *allow = getenv("KMERGPU_ALLOW_K32");
  const int kmax = (allow && allow[0] == '1') ? 32 : 31;
  if (length(s) <= k || k > kmax || k < 1) error("the sequence should be longer than k and k should not be longer than 31");

  kmg_query *q = NULL;
  uint64_t M = 0;
  if (kmg_query_begin(h->index, CHAR(s), (int64_t)length(s), k, &q, &M) != KMG_OK) error("seq.kmer.pos failed: %s", kmg_last_error());
  if (M > (uint64_t)INT_MAX) {
    kmg_query_free(q);
    error("seq.kmer.pos would return %llu rows, more than an R matrix can hold (2^31-1)", (unsigned long long)M);
  }
  SEXP guard = PROTECT(R_MakeExternalPtr(q, R_NilValue, R_NilValue));
  R_RegisterCFinalizerEx(guard, finalise_query_guard, TRUE);
  SEXP m = PROTECT(allocMatrix(INTSXP, 2, (int)M)); /* rows (i,j); seq.kmer.pos() names and transposes */
  const int rc = kmg_query_emit(q, INTEGER(m));
  kmg_query_free(q);
  R_ClearExternalPtr(guard);
  UNPROTECT(2);
  if (rc != KMG_OK) error("seq.kmer.pos failed: %s", kmg_last_error());
  return m;
}

/* kmer.pairs(ptr.a, ptr.b) -> .Call("kmer_pair_pos", ...), kmer_hash.R:30-34; replaces src/kmer_hash.c:1174-1203:
 * rows (a, b) for every k-mer the two indexes share; kmer.pairs() names and transposes. */
SEXP kmer_pair_pos(SEXP ptr_a, SEXP ptr_b) {
  kmer_handle *a = index_handle_or_error(ptr_a);
  kmer_handle *b = index_handle_or_error(ptr_b);
  kmg_join *j = NULL;
  uint64_t M = 0;
  if (kmg_join_begin(a->index, b->index, &j, &M) != KMG_OK) error("kmer.pairs failed: %s", kmg_last_error());
  if (M > (uint64_t)INT_MAX) {
    kmg_join_free(j);
    error("kmer.pairs would return %llu rows, more than an R matrix can hold (2^31-1)", (unsigned long long)M);
  }
  SEXP guard = PROTECT(R_MakeExternalPtr(j, R_NilValue, R_NilValue));
  R_RegisterCFinalizerEx(guard, finalise_join_guard, TRUE);
  SEXP m = PROTECT(allocMatrix(INTSXP, 2, (int)M));
  const int rc = kmg_join_emit(j, INTEGER(m));
  kmg_join_free(j);
  R_ClearExternalPtr(guard);
  UNPROTECT(2);
  if (rc != KMG_OK) error("kmer.pairs failed: %s", kmg_last_error());
  return m;
}

/* ---- additive entry points: a sequence file instead of an R string (SURVEY.md 8f rank 4) ------------------------
 * make.kmer.hash.file(file, record, k, do.sort) and count.kmers.file(file, params, hash.ptr): the file is inflated on
 * the host and parsed on the device (kmg_reads_*), so the sequence never becomes an R CHARSXP (whose 2^31-1 byte limit
 * is what bounds make.kmer.hash in the reference).  record: 1-based record number. */
static SEXP new_tagged_pointer(kmer_handle *h) {
  SEXP tag = PROTECT(allocVector(STRSXP, 1));
  SET_STRING_ELT(tag, 0, mkChar(KMER_HASH_TAG));
  SEXP ptr = PROTECT(R_MakeExternalPtr(h, tag, R_NilValue));
  R_RegisterCFinalizerEx(ptr, finalise_handle, TRUE);
  UNPROTECT(2);
  return ptr;
}

SEXP make_kmer_h_index_file(SEXP file_r, SEXP record_r, SEXP k_r, SEXP sort_pos_r) {
  if (TYPEOF(file_r) != STRSXP || length(file_r) != 1) error("file_r should be a single file name");
  if (TYPEOF(record_r) != INTSXP || length(record_r) != 1) error("record_r should be a single integer");
  if (TYPEOF(k_r) != INTSXP || length(k_r) < 1) error("k_r must be an integer vector of length at least one");
  if (TYPEOF(sort_pos_r) != INTSXP || length(sort_pos_r) < 1) error("sort_pos_r must be an integer vector of length at least one");
  const int k = INTEGER(k_r)[0], rec = INTEGER(record_r)[0];
  if (k < 1 || k > KMG_MAX_K) error("k must be a positive integer less than 1+MAX_K");
  kmg_reads *rd = NULL;
  if (kmg_reads_open(CHAR(STRING_ELT(file_r, 0)), &rd) != KMG_OK) error("make.kmer.hash.file failed: %s", kmg_last_error());
  uint64_t nrec = 0;
  int64_t len = 0;
  kmg_reads_count(rd, &nrec, NULL);
  if (rec < 1 || (uint64_t)rec > nrec) { kmg_reads_free(rd); error("the file holds %llu records; record %d does not exist", (unsigned long long)nrec, rec); }
  kmg_reads_record(rd, (uint64_t)rec - 1, &len, NULL, 0);
  if (len <= k) { kmg_reads_free(rd); error("the length of the sequence must be at least k"); }
  kmer_handle *h = (kmer_handle *)calloc(1, sizeof *h);
  if (!h) { kmg_reads_free(rd); error("out of memory"); }
  h->k = k;
  const int rc = kmg_build_record(rd, (uint64_t)rec - 1, k, INTEGER(sort_pos_r)[0] ? KMG_ORDER_SORTED : KMG_ORDER_GROUPED, &h->index);
  kmg_reads_free(rd);
  if (rc != KMG_OK) { free(h); error("make.kmer.hash.file failed: %s", kmg_last_error()); }
  return new_tagged_pointer(h);
}

SEXP count_kmers_file(SEXP hash_ptr_r, SEXP params_r, SEXP file_r) {
  if (TYPEOF(file_r) != STRSXP || length(file_r) != 1) error("file_r should be a single file name");
  if (TYPEOF(params_r) != INTSXP || length(params_r) != 3) error("k_r must be an integer vector of length 3");
  const int *params = INTEGER(params_r);
  const int k = params[0], source = params[1], source_n = params[2];
  if (k < 1 || k > KMG_MAX_K) error("k must be a positive integer less than 1+MAX_K");
  if (source_n < 1 || source >= source_n || source < 0) error("source_n must be larger than 1 and larger than source");
  kmer_handle *h = NULL;
  SEXP ptr_r = hash_ptr_r;
  int fresh = 0;
  if (ptr_r == R_NilValue) {
    h = (kmer_handle *)calloc(1, sizeof *h);
    if (!h) error("out of memory");
    h->k = k;
    if (kmg_count_new(k, source_n, &h->counter) != KMG_OK) { free(h); error("count.kmers.file failed: %s", kmg_last_error()); }
    ptr_r = PROTECT(new_tagged_pointer(h));
    fresh = 1;
  } else {
    h = handle_or_null(hash_ptr_r);
    if (!h || !h->counter) error("failed to extract kmer counts from external pointer");
    int sn = 0;
    kmg_count_sizes(h->counter, NULL, &sn, NULL, NULL);
    if (h->k != k || sn != source_n) error("mismatch between specified k and that given in the external pointer");
  }
  kmg_reads *rd = NULL;
  int rc = kmg_reads_open(CHAR(STRING_ELT(file_r, 0)), &rd);
  if (rc == KMG_OK) {
    rc = kmg_count_add_reads(h->counter, rd, source);
    kmg_reads_free(rd);
  }
  if (fresh) UNPROTECT(1);
  if (rc != KMG_OK) error("count.kmers.file failed: %s", kmg_last_error());
  return ptr_r;
}

/* seq.kmer.depth(ptr, seq, both.strands) -> t(.Call("sequence_kmer_depth", ptr, as.character(seq), as.integer(both.strands)))
 * (additive; INTEGRATION.md): for every k-mer window of seq, the count of its k-mer in a count table (source_n rows, one
 * per source) or a position index (one row: the length of the position list).  Returns a source_n x nwin matrix, nwin =
 * length(seq) - k + 1 with the handle's k; NA for a window make.kmer.hash would skip (the library writes INT32_MIN, which
 * is NA_integer_). */
SEXP sequence_kmer_depth(SEXP ptr_r, SEXP seq_r, SEXP strands_r) {
  if (TYPEOF(seq_r) != STRSXP || length(seq_r) != 1) error("seq_r should be a single sequence");
  if (TYPEOF(strands_r) != INTSXP || length(strands_r) != 1 || (INTEGER(strands_r)[0] != 0 && INTEGER(strands_r)[0] != 1))
    error("both.strands should be TRUE or FALSE");
  kmer_handle *h = handle_or_error(ptr_r);
  const int strands = INTEGER(strands_r)[0] ? KMG_STRAND_BOTH : KMG_STRAND_FORWARD;
  int sn = 1;
  if (h->counter && kmg_count_sizes(h->counter, NULL, &sn, NULL, NULL) != KMG_OK) error("seq.kmer.depth failed: %s", kmg_last_error());
  SEXP s = STRING_ELT(seq_r, 0);
  const int len = length(s);
  if (len <= h->k) error("the sequence should be longer than k");
  const uint64_t nwin = (uint64_t)(len - h->k + 1);
  if (nwin * (uint64_t)sn > (uint64_t)INT_MAX)
    error("seq.kmer.depth would return %llu values, more than an R matrix can hold (2^31-1)", (unsigned long long)(nwin * (uint64_t)sn));
  SEXP m = PROTECT(allocMatrix(INTSXP, sn, (int)nwin));
  const int rc = h->counter ? kmg_count_depth(h->counter, CHAR(s), (int64_t)len, strands, INTEGER(m))
                            : kmg_index_depth(h->index, CHAR(s), (int64_t)len, strands, INTEGER(m));
  UNPROTECT(1);
  if (rc != KMG_OK) error("seq.kmer.depth failed: %s", kmg_last_error());
  return m;
}

/* seq.kmer.dotplot / kmer.pairs.dotplot (additive; INTEGRATION.md): the rows seq.kmer.pos or kmer.pairs would return,
 * counted into an nx x ny double matrix on the device, so neither the 2^31-1 row limit nor the transfer of the rows
 * applies.  Cell [bx, by] (1-based in R: [bx+1, by+1]) counts the rows with floor((x - x0) * nx / (x1 - x0)) = bx and
 * floor((y - y0) * ny / (y1 - y0)) = by, over the half-open windows [x0, x1) x [y0, y1); max.count > 0 drops the k-mers
 * with more positions. */
static void dotplot_bins(const int *p, int *nx, int *ny) {
  *nx = p[2];
  *ny = p[5];
  if (*nx < 1 || *ny < 1) error("bins must be positive");
  if ((int64_t)*nx * *ny > (int64_t)INT_MAX)
    error("a dot plot of %d x %d bins would have %lld cells, more than an R matrix can hold (2^31-1)", *nx, *ny, (long long)*nx * *ny);
}

/* params = as.integer(c(x0, x1, nx, y0, y1, ny, rc, max.count)) */
SEXP sequence_kmer_dotplot(SEXP ptr_r, SEXP seq_r, SEXP k_r, SEXP params_r) {
  kmer_handle *h = index_handle_or_error(ptr_r);
  if (TYPEOF(seq_r) != STRSXP || length(seq_r) != 1) error("seq_r should be a single sequence");
  if (TYPEOF(k_r) != INTSXP || length(k_r) != 1) error("k should be an integer of length 1");
  if (TYPEOF(params_r) != INTSXP || length(params_r) != 8) error("params should be an integer vector of length 8");
  const int k = INTEGER(k_r)[0];
  SEXP s = STRING_ELT(seq_r, 0);
  const char *allow = getenv("KMERGPU_ALLOW_K32");
  const int kmax = (allow && allow[0] == '1') ? 32 : 31;
  if (length(s) <= k || k > kmax || k < 1) error("the sequence should be longer than k and k should not be longer than 31");
  const int *p = INTEGER(params_r);
  if (p[6] != 0 && p[6] != 1) error("rc should be TRUE or FALSE");
  if (p[7] < 0) error("max.count should be 0 (no limit) or positive");
  int nx, ny;
  dotplot_bins(p, &nx, &ny);
  SEXP m = PROTECT(allocMatrix(REALSXP, nx, ny));
  const int rc = kmg_query_dotplot(h->index, CHAR(s), (int64_t)length(s), k, p[6], p[0], p[1], nx, p[3], p[4], ny, (uint32_t)p[7], REAL(m));
  UNPROTECT(1);
  if (rc != KMG_OK) error("seq.kmer.dotplot failed: %s", kmg_last_error());
  return m;
}

/* params = as.integer(c(a0, a1, nx, b0, b1, ny, max.count)): x = position in a, y = position in b */
SEXP kmer_pair_dotplot(SEXP ptr_a, SEXP ptr_b, SEXP params_r) {
  kmer_handle *a = index_handle_or_error(ptr_a);
  kmer_handle *b = index_handle_or_error(ptr_b);
  if (TYPEOF(params_r) != INTSXP || length(params_r) != 7) error("params should be an integer vector of length 7");
  const int *p = INTEGER(params_r);
  if (p[6] < 0) error("max.count should be 0 (no limit) or positive");
  int nx, ny;
  dotplot_bins(p, &nx, &ny);
  SEXP m = PROTECT(allocMatrix(REALSXP, nx, ny));
  const int rc = kmg_join_dotplot(a->index, b->index, p[0], p[1], nx, p[3], p[4], ny, (uint32_t)p[6], REAL(m));
  UNPROTECT(1);
  if (rc != KMG_OK) error("kmer.pairs.dotplot failed: %s", kmg_last_error());
  return m;
}

static const R_CallMethodDef call_methods[] = {
    {"make_kmer_h_index", (DL_FUNC)&make_kmer_h_index, 3},
    {"kmer_positions", (DL_FUNC)&kmer_positions, 2},
    {"sequence_kmer_positions", (DL_FUNC)&sequence_kmer_positions, 3},
    {"kmer_pair_pos", (DL_FUNC)&kmer_pair_pos, 2},
    {"count_kmers", (DL_FUNC)&count_kmers, 3},
    {"make_kmer_h_index_file", (DL_FUNC)&make_kmer_h_index_file, 4},
    {"count_kmers_file", (DL_FUNC)&count_kmers_file, 3},
    {"sequence_kmer_depth", (DL_FUNC)&sequence_kmer_depth, 3},
    {"sequence_kmer_dotplot", (DL_FUNC)&sequence_kmer_dotplot, 4},
    {"kmer_pair_dotplot", (DL_FUNC)&kmer_pair_dotplot, 3},
    {NULL, NULL, 0}};

void R_init_kmer_hash(DllInfo *info) { R_registerRoutines(info, NULL, call_methods, NULL, NULL); }
