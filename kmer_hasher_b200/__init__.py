"""kmer_hasher_b200 -- host-side mirror of kmer_hasheR's R API over libkmergpu (B200, sm_100a).

The three functions keep the names, argument meaning, error behaviour and return layouts of the
reference's R closures (kmer_hash.R:5-28 in the reference checkout):

    make.kmer.hash(seq, k, do.sort) -> make_kmer_hash(seq, k, do_sort)   external pointer -> KmerHash
    kmer.pos(ex.ptr, opt.flag)      -> kmer_pos(ex_ptr, opt_flag)        list(kmer,pos,pair.pos,count)
    seq.kmer.pos(ex.ptr, seq, k)    -> seq_kmer_pos(ex_ptr, seq, k)      matrix with columns i, j

R is not installed in the build image, so this Python layer plays the part of kmer_hash.R and the
SEXP glue (the C glue that a real R session loads is kmer_hasher_b200/rglue/kmer_hash.c).  All
work happens in the CUDA library; if it cannot be loaded the import of this module fails.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import KmgError, check

__all__ = ["KmerHash", "KmerCounts", "SequenceFile", "make_kmer_hash_file", "count_kmers_file", "make_kmer_hash", "kmer_pos", "seq_kmer_pos", "kmer_pairs", "count_kmers", "kmer_spectrum",
           "seq_kmer_depth", "seq_kmer_dotplot", "kmer_pairs_dotplot", "pinned_empty", "KmgError",
           "OPT_KMER", "OPT_POS", "OPT_PAIRS", "OPT_COUNT", "NA_INTEGER"]

# opt.flag bits, src/kmer_hash.c:17 (pos_opt_flags) in the reference
OPT_KMER, OPT_POS, OPT_PAIRS, OPT_COUNT = 1, 2, 4, 8
ORDER_GROUPED, ORDER_SORTED = 0, 1      # include/kmergpu.h
KMER_HASH_TAG = "kmer_hash_250930"      # src/kmer_hash.c:22
MAX_K = 32                              # src/kmer_util.h:12
INT_MAX = 2**31 - 1
NA_INTEGER = -2**31                     # R's NA_integer_: seq_kmer_depth's value for a window that is not a k-mer

_L = _lib.load()                        # loud failure when libkmergpu.so is absent


def _seq_buffer(seq):
    """(pointer, length, keepalive) of a str / bytes / uint8 array / torch CUDA tensor."""
    if isinstance(seq, str):
        seq = seq.encode("latin-1")
    if isinstance(seq, (bytes, bytearray)):
        b = bytes(seq)
        return C.cast(C.c_char_p(b), C.c_void_p), len(b), b
    if isinstance(seq, np.ndarray):
        a = np.ascontiguousarray(seq.view(np.uint8) if seq.dtype != np.uint8 else seq)
        return C.c_void_p(a.ctypes.data), a.size, a
    if hasattr(seq, "data_ptr"):        # torch tensor (host or device), uint8
        t = seq.contiguous()
        return C.c_void_p(t.data_ptr()), t.numel() * t.element_size(), t
    raise TypeError("seq must be str, bytes, a uint8 numpy array or a uint8 torch tensor")


class _Pinned:
    def __init__(self, nbytes):
        self.ptr = _L.kmg_host_alloc(max(int(nbytes), 1))
        if not self.ptr:
            raise MemoryError(_L.kmg_last_error().decode())

    def __del__(self):
        if getattr(self, "ptr", None) and _L is not None:      # _L is gone at interpreter shutdown
            _L.kmg_host_free(self.ptr)
            self.ptr = None


def pinned_empty(shape, dtype) -> np.ndarray:
    """A numpy array in page-locked host memory (full-speed PCIe target/source)."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    owner = _Pinned(n)
    raw = (C.c_char * max(n, 1)).from_address(owner.ptr)
    raw._owner = owner
    return np.frombuffer(raw, dtype=dtype, count=int(np.prod(shape))).reshape(shape)


def _out_ptr(arr):
    if arr is None:
        return None
    if isinstance(arr, np.ndarray):
        return C.c_void_p(arr.ctypes.data)
    return C.c_void_p(arr.data_ptr())   # torch tensor


class KmerHash:
    """What make.kmer.hash returns: an external pointer tagged "kmer_hash_250930" whose finaliser
    frees the index (make_kmer_h_index / finalise_khash_ptr, src/kmer_hash.c:531-537, 56-66)."""

    tag = KMER_HASH_TAG

    def __init__(self, handle: int, k: int):
        self._h = handle
        self.k = k

    @property
    def sizes(self):
        """(U, N, P); P -- rows of pair.pos -- costs a sweep of the index the first time (cached afterwards)"""
        U, N, P = C.c_uint64(), C.c_uint64(), C.c_uint64()
        check(_L.kmg_sizes(self._handle(), C.byref(U), C.byref(N), C.byref(P)))
        return U.value, N.value, P.value

    @property
    def sizes_un(self):
        """(U, N) only: what make.kmer.hash + kmer.pos without pair.pos need"""
        U, N = C.c_uint64(), C.c_uint64()
        check(_L.kmg_sizes(self._handle(), C.byref(U), C.byref(N), None))
        return U.value, N.value

    def _handle(self):
        if not self._h:
            raise ValueError("external pointer has been cleared")
        return self._h

    def free(self):
        if self._h:
            _L.kmg_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class KmerCounts(KmerHash):
    """What count.kmers returns: the same kind of external pointer (same tag) holding per-source counts instead of
    positions (count_kmers, src/kmer_hash.c:548-591)."""

    def __init__(self, handle: int, k: int, source_n: int):
        super().__init__(handle, k)
        self.source_n = source_n

    @property
    def sizes(self):
        U, nt = C.c_uint64(), C.c_uint64()
        check(_L.kmg_count_sizes(self._handle(), C.byref(U), None, None, C.byref(nt)))
        sn = self.source_n
        return U.value, U.value * sn, U.value * sn * (sn - 1) // 2

    @property
    def sizes_un(self):
        return self.sizes[:2]

    @property
    def kmer_count(self):
        """khash_ptr.kmer_count: k-mers that were new when added, summed over the calls"""
        nt = C.c_uint64()
        check(_L.kmg_count_sizes(self._handle(), None, None, None, C.byref(nt)))
        return nt.value

    def free(self):
        if self._h:
            _L.kmg_count_free(self._h)
            self._h = None


def _extract(ex_ptr) -> KmerHash:
    # extract_khash_ptr, src/kmer_hash.c:491-503
    if not isinstance(ex_ptr, KmerHash):
        raise TypeError("ptr_r should be an external pointer")
    if ex_ptr.tag != KMER_HASH_TAG:
        raise ValueError("External pointer has incorrect tag")
    return ex_ptr


def _extract_index(ex_ptr) -> KmerHash:
    ix = _extract(ex_ptr)
    if isinstance(ix, KmerCounts):
        raise ValueError("this external pointer holds k-mer counts (count.kmers), not a position index")
    return ix


def make_kmer_hash(seq, k, do_sort=False) -> KmerHash:
    """make.kmer.hash (kmer_hash.R:5-8 -> make_kmer_h_index, src/kmer_hash.c:506-540).

    `seq` may be a character vector: like the reference, only its first element is used.
    Position lists are always ascending, so the reference's `do.sort` has nothing to sort; here it selects
    the order of the K-MERS, which is not semantic (the reference's is hash-bucket order): do_sort=True gives
    ascending 2-bit key (KMG_ORDER_SORTED), the default the faster grouped build (KMG_ORDER_GROUPED: order of
    a mix of the key, used for k >= 21).  `kmer_pos(..., canonical=True)` re-orders any index by key.
    """
    if isinstance(seq, (list, tuple)):
        if len(seq) < 1:
            raise ValueError("seq_r should be a character vector of length at least one")
        seq = seq[0]
    k = int(k)
    order = ORDER_SORTED if int(do_sort) else ORDER_GROUPED
    if k < 1 or k > MAX_K:
        raise ValueError("k must be a positive integer less than 1+MAX_K")
    ptr, n, keep = _seq_buffer(seq)
    if n <= k:
        raise ValueError("the length of the sequence must be at least k")
    h = C.c_void_p()
    check(_L.kmg_build_ordered(ptr, n, k, order, C.byref(h)))
    del keep
    return KmerHash(h.value, k)


def _by_key(ix: "KmerHash"):
    """(order, rank): order[j] = index (0-based) of the k-mer with the j-th smallest key, rank = its inverse."""
    U = ix.sizes_un[0]
    keys = np.empty(U, np.uint64)
    check(_L.kmg_kmers_u64(ix._handle(), _out_ptr(keys)))
    order = np.argsort(keys, kind="stable")
    rank = np.empty(U, np.int64)
    rank[order] = np.arange(U)
    return keys, order, rank


def _renumber(rows: np.ndarray, rank: np.ndarray) -> np.ndarray:
    """Rows whose first column is a 1-based k-mer number: renumber by `rank` and group by the new number (stable)."""
    if len(rows) == 0:
        return rows
    new_i = rank[rows[:, 0].astype(np.int64) - 1] + 1
    o = np.argsort(new_i, kind="stable")
    out = rows[o].copy()
    out[:, 0] = new_i[o].astype(np.int32)
    return out


def kmer_pos(ex_ptr, opt_flag, out: dict | None = None, canonical: bool = False) -> dict:
    """kmer.pos (kmer_hash.R:10-21 -> kmer_positions, src/kmer_hash.c:1054-1147).

    Returns {"kmer", "pos", "pair.pos", "count"}; fields whose opt.flag bit is off are None.
    "pos" is an N x 2 int32 array with columns (i, pos) and "pair.pos" a P x 3 array with columns
    (i, x, y) -- the matrices R holds after kmer.pos's t().  k-mers come in the index's own order (see
    make_kmer_hash); `canonical=True` re-orders them by ascending key with i renumbered, the form in which
    results are compared with the reference (whose own order is its hash table's).
    `out` may supply preallocated (e.g. pinned) arrays under the same names.
    """
    ix = _extract(ex_ptr)
    opt_flag = int(opt_flag)
    if isinstance(ix, KmerCounts):
        return _count_table_pos(ix, opt_flag)
    out = out or {}
    U, N = ix.sizes_un
    P = ix.sizes[2] if opt_flag & OPT_PAIRS else 0
    h = ix._handle()
    res = {"kmer": None, "pos": None, "pair.pos": None, "count": None}
    if opt_flag & OPT_KMER:
        buf = out.get("kmer_buf")
        if buf is None:
            buf = np.empty(U * (ix.k + 1), np.uint8)
        check(_L.kmg_kmers_ascii(h, _out_ptr(buf)))
        res["kmer"] = np.ascontiguousarray(buf[:U * (ix.k + 1)].reshape(U, ix.k + 1)[:, :ix.k]).view(f"S{ix.k}").ravel()
    if opt_flag & OPT_POS:
        if N > INT_MAX:
            raise OverflowError("pos matrix extent exceeds int")
        a = out.get("pos")
        if a is None:
            a = np.empty((N, 2), np.int32)
        check(_L.kmg_positions(h, _out_ptr(a)))
        res["pos"] = a[:N]
    if opt_flag & OPT_PAIRS:
        if P > INT_MAX:
            raise OverflowError(f"pair.pos would need {P} rows; an R matrix extent is int "
                                "(use kmg_pairs_chunk to stream)")
        a = out.get("pair.pos")
        if a is None:
            a = np.empty((P, 3), np.int32)
        check(_L.kmg_pairs(h, _out_ptr(a)))
        res["pair.pos"] = a[:P]
    if opt_flag & OPT_COUNT:
        a = out.get("count")
        if a is None:
            a = np.empty(U, np.int32)
        check(_L.kmg_counts(h, _out_ptr(a)))
        res["count"] = a[:U]
    if canonical and _L.kmg_index_order(h) != ORDER_SORTED:
        _, order, rank = _by_key(ix)
        if res["kmer"] is not None:
            res["kmer"] = res["kmer"][order]
        if res["count"] is not None:
            res["count"] = np.asarray(res["count"])[order]
        if res["pos"] is not None:
            res["pos"] = _renumber(np.asarray(res["pos"]), rank)
        if res["pair.pos"] is not None:
            res["pair.pos"] = _renumber(np.asarray(res["pair.pos"]), rank)
    return res


def count_kmers(seq, params, hash_ptr: "KmerCounts | None" = None) -> KmerCounts:
    """count.kmers (kmer_hash.R:43-46 -> count_kmers, src/kmer_hash.c:548-591).

    params = (k, source, source_n).  Every sequence of `seq` (a string or a list of strings) that is longer than k
    adds one to column `source` of its k-mers' counters, window rule as in make.kmer.hash; `hash_ptr=None` makes a
    new table.  Read the table with kmer_pos(ptr, 1 + 2 + 8) as the reference does (test.R:340-347): "pos" holds
    rows (i, count of source 0), (i, count of source 1), ...; "count" is source_n for every k-mer.  k-mers come in
    ascending key order (the reference's is its hash table's)."""
    params = [int(p) for p in params]
    if len(params) != 3:
        raise ValueError("k_r must be an integer vector of length 3")
    k, source, source_n = params
    if k < 1 or k > MAX_K:
        raise ValueError("k must be a positive integer less than 1+MAX_K")
    if source_n < 1 or source >= source_n or source < 0:
        raise ValueError("source_n must be larger than 1 and larger than source")
    if isinstance(seq, (str, bytes, bytearray, np.ndarray)) or hasattr(seq, "data_ptr"):
        seq = [seq]
    if len(seq) < 1:
        raise ValueError("seq_r should be a character vector of length at least one")
    if hash_ptr is None:
        h = C.c_void_p()
        check(_L.kmg_count_new(k, source_n, C.byref(h)))
        hash_ptr = KmerCounts(h.value, k, source_n)
    else:
        if not isinstance(hash_ptr, KmerCounts):
            raise ValueError("failed to extract kmer_hash from external pointer")
        if hash_ptr.k != k:
            raise ValueError("mismatch between specified k and that given in the external pointer")
        if hash_ptr.source_n != source_n:
            raise ValueError("mismatch between specified source_n and that of the external pointer")
    for s in seq:
        ptr, n, keep = _seq_buffer(s)
        if n <= k:
            continue
        check(_L.kmg_count_add(hash_ptr._handle(), ptr, n, source))
        del keep
    return hash_ptr


def _count_table_pos(ct: KmerCounts, opt_flag: int) -> dict:
    U = ct.sizes[0]
    sn, h = ct.source_n, ct._handle()
    res = {"kmer": None, "pos": None, "pair.pos": None, "count": None}
    if opt_flag & OPT_KMER:
        buf = np.empty(U * (ct.k + 1), np.uint8)
        check(_L.kmg_count_kmers_ascii(h, _out_ptr(buf)))
        res["kmer"] = np.ascontiguousarray(buf.reshape(U, ct.k + 1)[:, :ct.k]).view(f"S{ct.k}").ravel()
    if opt_flag & OPT_POS:
        if U * sn > INT_MAX:
            raise OverflowError("pos matrix extent exceeds int")
        a = np.empty((U * sn, 2), np.int32)
        check(_L.kmg_count_positions(h, _out_ptr(a)))
        res["pos"] = a
    if opt_flag & OPT_PAIRS:
        m = np.empty((U, sn), np.int32)
        check(_L.kmg_count_matrix(h, _out_ptr(m)))
        ia, ib = np.triu_indices(sn, 1)
        rows = np.empty((U, len(ia), 3), np.int32)
        rows[:, :, 0] = np.arange(1, U + 1, dtype=np.int32)[:, None]
        rows[:, :, 1] = m[:, ia]
        rows[:, :, 2] = m[:, ib]
        res["pair.pos"] = rows.reshape(-1, 3)
    if opt_flag & OPT_COUNT:
        res["count"] = np.full(U, sn, np.int32)
    return res


class SequenceFile:
    """The records of a FASTA / FASTQ file (plain or gz), parsed on the device and kept there (kmg_reads_*): what the
    reference gets from kseq_read (src/kmer_reader.c:41-77) -- names up to the first white space, sequences with the line
    ends removed -- without the sequences ever becoming host strings."""

    def __init__(self, path_or_text):
        h = C.c_void_p()
        if isinstance(path_or_text, (bytes, bytearray, np.ndarray)) or hasattr(path_or_text, "data_ptr"):
            ptr, n, keep = _seq_buffer(path_or_text)
            check(_L.kmg_reads_from_memory(ptr, n, C.byref(h)))
        else:
            check(_L.kmg_reads_open(str(path_or_text).encode(), C.byref(h)))
        self._h = h.value
        n, tot = C.c_uint64(), C.c_uint64()
        check(_L.kmg_reads_count(self._h, C.byref(n), C.byref(tot)))
        self.n_records, self.total_bases = n.value, tot.value

    def record(self, i: int):
        """(name, sequence length) of record i"""
        ln, buf = C.c_int64(), C.create_string_buffer(4096)
        check(_L.kmg_reads_record(self._h, i, C.byref(ln), buf, 4096))
        return buf.value.decode("latin-1"), ln.value

    def sequence(self, i: int) -> bytes:
        _, ln = self.record(i)
        out = np.empty(max(ln, 1), np.uint8)
        check(_L.kmg_reads_sequence(self._h, i, _out_ptr(out)))
        return out[:ln].tobytes()

    def names(self):
        return [self.record(i)[0] for i in range(self.n_records)]

    def free(self):
        if self._h:
            _L.kmg_reads_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def make_kmer_hash_file(file, k, record=0, do_sort=False) -> KmerHash:
    """make.kmer.hash on one record of a FASTA / FASTQ file (by number or by name): the sequence goes file -> device
    -> index, never through a host string.  `file` is a path or an open SequenceFile."""
    sf = file if isinstance(file, SequenceFile) else SequenceFile(file)
    try:
        if isinstance(record, str):
            names = sf.names()
            if record not in names:
                raise KeyError(f"no record named {record!r}")
            record = names.index(record)
        k = int(k)
        if k < 1 or k > MAX_K:
            raise ValueError("k must be a positive integer less than 1+MAX_K")
        if sf.record(record)[1] <= k:
            raise ValueError("the length of the sequence must be at least k")
        h = C.c_void_p()
        check(_L.kmg_build_record(sf._h, record, k, ORDER_SORTED if int(do_sort) else ORDER_GROUPED, C.byref(h)))
        return KmerHash(h.value, k)
    finally:
        if not isinstance(file, SequenceFile):
            sf.free()


def count_kmers_file(file, params, hash_ptr: "KmerCounts | None" = None) -> KmerCounts:
    """count.kmers over every record of a FASTA / FASTQ file: as count_kmers(list of the records' sequences, params,
    hash_ptr) -- records no longer than k are skipped, every record keeps the reference's end-of-string rule -- but the
    whole file is counted by ONE index build on the device."""
    params = [int(p) for p in params]
    if len(params) != 3:
        raise ValueError("k_r must be an integer vector of length 3")
    k, source, source_n = params
    sf = file if isinstance(file, SequenceFile) else SequenceFile(file)
    try:
        if hash_ptr is None:
            if k < 1 or k > MAX_K:
                raise ValueError("k must be a positive integer less than 1+MAX_K")
            if source_n < 1 or source >= source_n or source < 0:
                raise ValueError("source_n must be larger than 1 and larger than source")
            h = C.c_void_p()
            check(_L.kmg_count_new(k, source_n, C.byref(h)))
            hash_ptr = KmerCounts(h.value, k, source_n)
        elif not isinstance(hash_ptr, KmerCounts) or hash_ptr.k != k or hash_ptr.source_n != source_n:
            raise ValueError("mismatch between specified k and that given in the external pointer")
        if source < 0 or source >= source_n:
            raise ValueError("source_n must be larger than 1 and larger than source")
        check(_L.kmg_count_add_reads(hash_ptr._handle(), sf._h, source))
        return hash_ptr
    finally:
        if not isinstance(file, SequenceFile):
            sf.free()


def kmer_spectrum(ptr, max_count: int, source: "int | None" = None) -> np.ndarray:
    """k-mer count spectrum: spec[c] = number of k-mers seen c times, counts >= max_count pooled in spec[max_count];
    doubles, like the reference's kmer.spec.* (count_spectrum, src/kmer_tree.c:85-99; src/kmer_hash.c:975-1038).
    `ptr` is a count table (count_kmers; `source` picks a column, None sums them) or a position index
    (make_kmer_hash; a k-mer's count is the length of its position list)."""
    ix = _extract(ptr)
    max_count = int(max_count)
    if max_count < 1 or max_count > (1 << 30):
        raise ValueError("Unsuitable value of max_count")
    spec = np.zeros(max_count + 1, np.float64)
    sp = spec.ctypes.data_as(C.POINTER(C.c_double))
    if isinstance(ix, KmerCounts):
        check(_L.kmg_count_spectrum(ix._handle(), -1 if source is None else int(source), max_count, sp))
    else:
        check(_L.kmg_index_spectrum(ix._handle(), max_count, sp))
    return spec


def kmer_keys(ex_ptr, canonical: bool = False) -> np.ndarray:
    """The distinct k-mers as uint64 keys in the index's order, or ascending with canonical=True (not part of
    the R API; used by tests)."""
    ix = _extract(ex_ptr)
    U, _ = ix.sizes_un
    a = np.empty(U, np.uint64)
    if isinstance(ix, KmerCounts):
        check(_L.kmg_count_kmers_u64(ix._handle(), _out_ptr(a)))
        return a
    check(_L.kmg_kmers_u64(ix._handle(), _out_ptr(a)))
    return np.sort(a) if canonical else a


def seq_kmer_pos(ex_ptr, seq, k, *, allow_k32: bool = False, out: np.ndarray | None = None,
                 reverse_complement: bool = False) -> np.ndarray:
    """seq.kmer.pos (kmer_hash.R:23-28 -> sequence_kmer_positions, src/kmer_hash.c:1151-1172).

    M x 2 int32 array, columns (i, j): i = 1-based END of the query k-mer, j = 1-based start in the
    index; rows ordered by i then j.  The reference's R entry rejects k > 31
    (src/kmer_hash.c:1163) although its C core handles k = 32; `allow_k32=True` lifts that guard.
    `reverse_complement=True` probes reverseComplement(seq) instead, made on the device: the second half
    of every dot plot in the reference's notebook (test.R:43-52,73); i then refers to that string.
    """
    ix = _extract_index(ex_ptr)
    if isinstance(seq, (list, tuple)):
        if len(seq) != 1:
            raise ValueError("seq_r should be a single sequence")
        seq = seq[0]
    k = int(k)
    ptr, n, keep = _seq_buffer(seq)
    if n <= k or k > (32 if allow_k32 else 31):
        raise ValueError("the sequence should be longer than k and k should not be longer than 31")
    st, M = C.c_void_p(), C.c_uint64()
    begin = _L.kmg_query_begin_rc if reverse_complement else _L.kmg_query_begin
    check(begin(ix._handle(), ptr, n, k, C.byref(st), C.byref(M)))
    try:
        if M.value > INT_MAX:
            raise OverflowError(f"{M.value} result rows exceed an R matrix extent")
        a = out if out is not None else np.empty((M.value, 2), np.int32)
        check(_L.kmg_query_emit(st, _out_ptr(a)))
    finally:
        _L.kmg_query_free(st)
    del keep
    return a[:M.value]


def seq_kmer_depth(ptr, seq, *, both_strands: bool = False, out=None):
    """seq.kmer.depth (additive; the R closure is in INTEGRATION.md): for every k-mer window of `seq`, how often its k-mer
    was counted.  `ptr` is a count table (count_kmers: one column per source) or a position index (make_kmer_hash: one
    column, the length of the k-mer's position list); k is the handle's own.

    Returns an (nwin, source_n) int32 array, nwin = len(seq) - k + 1, row r = the window at 1-based start r + 1.  An absent
    k-mer gives 0; a window make.kmer.hash would skip (an N/n in it, or the end-of-string rule) gives NA_INTEGER in every
    column.  `both_strands=True` adds the count of the reverse complement (code space: A<->T, C<->G; a palindrome counts
    once; saturating at 2^31 - 1).  `seq` is a str, bytes, uint8 numpy array or uint8 torch tensor (host or device);
    `out` may supply the result array (numpy, pinned or a torch device tensor) of at least nwin * source_n int32."""
    ix = _extract(ptr)
    if isinstance(seq, (list, tuple)):
        if len(seq) != 1:
            raise ValueError("seq_r should be a single sequence")
        seq = seq[0]
    counts = isinstance(ix, KmerCounts)
    cols = ix.source_n if counts else 1
    p, n, keep = _seq_buffer(seq)
    if n <= ix.k:
        raise ValueError("the sequence should be longer than k")
    nwin = n - ix.k + 1
    if nwin * cols > INT_MAX:
        raise OverflowError(f"{nwin * cols} values exceed an R matrix extent")
    if out is None:
        out = np.empty((nwin, cols), np.int32)
    else:
        size = out.nbytes if isinstance(out, np.ndarray) else out.numel() * out.element_size()
        if size < 4 * nwin * cols:
            raise ValueError(f"out holds {size} bytes; the depth needs {4 * nwin * cols}")
    depth = _L.kmg_count_depth if counts else _L.kmg_index_depth
    check(depth(ix._handle(), p, n, int(bool(both_strands)), _out_ptr(out)))
    del keep
    return out


def kmer_pairs(ptr_a, ptr_b, *, out: np.ndarray | None = None) -> np.ndarray:
    """kmer.pairs (kmer_hash.R:30-34 -> kmer_pair_pos, src/kmer_hash.c:1174-1203).

    M x 2 int32 array, columns (a, b): for every k-mer that both indexes hold, each of its 1-based
    positions in `ptr_a` paired with each of its positions in `ptr_b` (a position outer, b position
    inner), k-mers of `ptr_a` in ascending key order.  (The reference's own routine crashes on its
    bucket walk, test.R:330-331; this is its evident intent.)
    """
    a, b = _extract_index(ptr_a), _extract_index(ptr_b)
    st, M = C.c_void_p(), C.c_uint64()
    check(_L.kmg_join_begin(a._handle(), b._handle(), C.byref(st), C.byref(M)))
    try:
        if M.value > INT_MAX:
            raise OverflowError(f"{M.value} result rows exceed an R matrix extent")
        r = out if out is not None else np.empty((M.value, 2), np.int32)
        check(_L.kmg_join_emit(st, _out_ptr(r)))
    finally:
        _L.kmg_join_free(st)
    return r[:M.value]


def _dotplot_args(bins, ranges, max_count, out):
    """(nx, ny, (x0, x1), (y0, y1), max_count, out) checked; `out` allocated column-major when None."""
    nx, ny = (int(b) for b in bins)
    if nx < 1 or ny < 1:
        raise ValueError("bins must be positive")
    if nx * ny > INT_MAX:
        raise OverflowError(f"a dot plot of {nx} x {ny} bins has more than 2^31 - 1 cells")
    win = []
    for name, r in zip(("x", "y"), ranges):
        lo, hi = (int(v) for v in r)
        if not 0 <= lo < hi <= 2**31:
            raise ValueError(f"{name} range [{lo}, {hi}) must satisfy 0 <= start < end <= 2^31")
        win.append((lo, hi))
    max_count = int(max_count)
    if not 0 <= max_count < 2**32:
        raise ValueError("max_count must be 0 (no limit) or a positive 32-bit count")
    if out is None:
        out = np.empty((nx, ny), np.float64, order="F")
    else:
        size = out.nbytes if isinstance(out, np.ndarray) else out.numel() * out.element_size()
        if size < 8 * nx * ny:
            raise ValueError(f"out holds {size} bytes; the image needs {8 * nx * ny}")
    return nx, ny, win[0], win[1], max_count, out


def seq_kmer_dotplot(ptr, seq, k, *, y_range, bins=(1000, 1000), x_range=None, reverse_complement=False, max_count=0,
                     allow_k32=False, out=None):
    """seq.kmer.dotplot (additive; the R closure is in INTEGRATION.md): the rows seq_kmer_pos(ptr, seq, k,
    reverse_complement=...) would return, counted on the device into an nx x ny image -- x = i (1-based END of the query
    window, of the reverse-complemented string with reverse_complement=True), y = j (1-based start in the index).

    x_range = (x0, x1) and y_range = (y0, y1) are half-open windows (0 <= start < end <= 2^31; x_range defaults to
    (1, len(seq) + 1), the index's length is not recorded so y_range is required); a row counts into bin
    (floor((x - x0) * nx / (x1 - x0)), floor((y - y0) * ny / (y1 - y0))) if it lies in both windows.  max_count > 0 drops
    the k-mers with more positions in the index.  Returns a float64 (nx, ny) array in column-major order (the bytes of the
    R matrix); `out` may supply it (numpy, pinned or a torch device tensor of at least nx * ny float64)."""
    ix = _extract_index(ptr)
    if isinstance(seq, (list, tuple)):
        if len(seq) != 1:
            raise ValueError("seq_r should be a single sequence")
        seq = seq[0]
    k = int(k)
    p, n, keep = _seq_buffer(seq)
    if n <= k or k > (32 if allow_k32 else 31):
        raise ValueError("the sequence should be longer than k and k should not be longer than 31")
    nx, ny, (x0, x1), (y0, y1), mc, out = _dotplot_args(bins, (x_range if x_range is not None else (1, n + 1), y_range),
                                                        max_count, out)
    check(_L.kmg_query_dotplot(ix._handle(), p, n, k, int(bool(reverse_complement)), x0, x1, nx, y0, y1, ny, mc, _out_ptr(out)))
    del keep
    return out


def kmer_pairs_dotplot(ptr_a, ptr_b, *, a_range, b_range, bins=(1000, 1000), max_count=0, out=None):
    """kmer.pairs.dotplot (additive; INTEGRATION.md): the rows kmer_pairs(ptr_a, ptr_b) would return, counted on the device
    into an nx x ny image, x = position in ptr_a over the half-open a_range, y = position in ptr_b over b_range; binning,
    max_count (here: more positions in either index), result and `out` as in seq_kmer_dotplot."""
    a, b = _extract_index(ptr_a), _extract_index(ptr_b)
    nx, ny, (x0, x1), (y0, y1), mc, out = _dotplot_args(bins, (a_range, b_range), max_count, out)
    check(_L.kmg_join_dotplot(a._handle(), b._handle(), x0, x1, nx, y0, y1, ny, mc, _out_ptr(out)))
    return out


def profile(enable: bool | None = None, reset: bool = False) -> dict:
    """Per-kernel CUDA-event totals recorded by the library: {name: (ms, launches, algo_bytes)}."""
    if enable is not None:
        check(_L.kmg_profile_enable(int(enable)))
    res = {}
    for i in range(_L.kmg_profile_count()):
        name, ms, n, b = C.c_char_p(), C.c_double(), C.c_uint64(), C.c_double()
        check(_L.kmg_profile_get(i, C.byref(name), C.byref(ms), C.byref(n), C.byref(b)))
        res[name.value.decode()] = (ms.value, n.value, b.value)
    if reset:
        check(_L.kmg_profile_reset())
    return res


def launch_count() -> int:
    return int(_L.kmg_launch_count())
