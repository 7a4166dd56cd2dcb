"""Every emitter past its chunk boundaries.

An emitter writes rows through stream_rows (csrc/api.cu): into a device buffer in one launch; into pinned host memory
in 256 MiB device chunks, two device buffers taking turns; into pageable host memory over 8 MiB in 64 MiB chunks through
three pinned staging slots.  Each chunk's launch gets its first row and must write its own rows only.  Here each output
is produced all three ways and must be the same bytes; the launch counts from kh.profile prove the chunked paths ran;
the device output is checked against the oracle (or, at the largest size, against properties every correct result has).

Chunks reached (device / pinned / pageable):
  kmg_kmers_ascii      k = 32, ~10 M k-mers, 33-byte rows         1 / 2 / 5
  kmg_counts           ~69 M k-mers, 4-byte rows                  1 / 2 / 5
  kmg_positions_base   ~70 M rows of 8 bytes, i_base = 12345      1 / 3 / 9
  kmg_pairs_chunk      ~46 M rows of 12 bytes from row 1,234,567  1 / 3 / 9
  kmg_query_emit_chunk ~37 M rows of 8 bytes from row 777,777     1 / 2 / 5
  kmg_join_emit_chunk  ~37 M rows of 8 bytes from row 555,555     1 / 2 / 5
The count table's two emitters (kmg_count_positions, kmg_count_kmers_ascii) are run the same three ways in
test_counts_oracle_gpu.py::test_large_count_table_across_chunks.  No pinned output here exceeds 600 MB.
"""
import numpy as np
import pytest

from conftest import random_dna

CHUNK_BYTES = 256 << 20                    # device chunk of a pinned destination
STAGE_BYTES = 64 << 20                     # staged chunk of a pageable destination over 8 MiB


def within(c):
    """For counts c: 0..c[0]-1, 0..c[1]-1, ... concatenated."""
    c = np.asarray(c, np.int64)
    return np.arange(int(c.sum()), dtype=np.int64) - np.repeat(np.cumsum(c) - c, c)


def probe_rows(e, qkeys, qstart, k):
    """seq.kmer.pos rows (i = 1-based end of the query window, j = index position) from a canonical extraction
    `e = extract(2 | 8)` and the query's window stream (oracle.windows): windows in order, positions ascending."""
    keys, cnt, pos = e["keys"], e["count"].astype(np.int64), e["pos"].reshape(-1, 2)[:, 1]
    start = np.concatenate([[0], np.cumsum(cnt)])
    idx = np.minimum(np.searchsorted(keys, qkeys), max(len(keys) - 1, 0))
    hit = (keys[idx] == qkeys) if len(keys) else np.zeros(len(qkeys), bool)
    c = np.where(hit, cnt[idx], 0)
    rows = np.empty((int(c.sum()), 2), np.int32)
    rows[:, 0] = np.repeat(qstart.astype(np.int64) + k - 1, c)
    rows[:, 1] = pos[np.repeat(start[idx], c) + within(c)]
    return rows


def join_rows(ea, eb):
    """kmer.pairs rows (a position, b position) from two canonical extractions: k-mers of a in ascending key order, a
    position outer, b position inner (vectorised oracle.pairs_join)."""
    ca, cb = ea["count"].astype(np.int64), eb["count"].astype(np.int64)
    pa, pb = ea["pos"].reshape(-1, 2)[:, 1], eb["pos"].reshape(-1, 2)[:, 1]
    sa, sb = np.cumsum(ca) - ca, np.cumsum(cb) - cb
    idx = np.minimum(np.searchsorted(eb["keys"], ea["keys"]), len(eb["keys"]) - 1)
    u = np.nonzero(eb["keys"][idx] == ea["keys"])[0]
    v = idx[u]
    a_at = np.repeat(sa[u], ca[u]) + within(ca[u])         # every a position of a shared k-mer
    nb, b0 = np.repeat(cb[v], ca[u]), np.repeat(sb[v], ca[u])
    rows = np.empty((int(nb.sum()), 2), np.int32)
    rows[:, 0] = pa[np.repeat(a_at, nb)]
    rows[:, 1] = pb[np.repeat(b0, nb) + within(nb)]
    return rows


def test_row_restatements_match_the_oracle(oracle):
    """probe_rows == oracle query, join_rows == oracle.pairs_join (CPU)."""
    import oracle as oracle_mod
    a = random_dna(30_000, 1, p_n=0.002)
    b = random_dna(20_000, 2, p_n=0.002)
    b[5_000:9_000] = a[1_000:5_000]
    for k in (5, 8, 13):
        oa, ob = oracle.build(a, k), oracle.build(b, k)
        ea, eb = oa.extract(2 | 8), ob.extract(2 | 8)
        qk, qs = oracle.windows(b, k)
        assert np.array_equal(probe_rows(ea, qk, qs, k).ravel(), oa.query(b, k))
        assert np.array_equal(join_rows(ea, eb).ravel(), oracle_mod.pairs_join(ea, eb))


@pytest.fixture(scope="module")
def kh():
    import kmer_hasher_b200 as kh
    return kh


def chunks(rows, row_bytes, chunk_bytes):
    return -(-rows // (chunk_bytes // row_bytes))


def three_ways(kh, name, emit, rows, row_bytes, dtype, width):
    """Run `emit(out_pointer)` into a device tensor, pinned memory and pageable memory; require one launch of kernel
    `name`, the pinned and the staged chunk counts, and the same bytes all three ways.  Returns the rows."""
    import torch
    nbytes = rows * row_bytes
    assert nbytes > (8 << 20)
    kh.profile(enable=True, reset=True)
    try:
        dev = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        emit(dev.data_ptr())
        torch.cuda.synchronize()
        assert kh.profile(reset=True)[name][1] == 1
        base = dev.cpu().numpy()
        del dev
        pin = kh.pinned_empty(nbytes, np.uint8)
        emit(pin.ctypes.data)
        n_pin = chunks(rows, row_bytes, CHUNK_BYTES)
        assert kh.profile(reset=True)[name][1] == n_pin >= 2, name
        assert np.array_equal(pin, base), name
        del pin
        page = np.empty(nbytes, np.uint8)
        emit(page.ctypes.data)
        n_page = chunks(rows, row_bytes, STAGE_BYTES)
        assert kh.profile(reset=True)[name][1] == n_page >= 3, name
        assert np.array_equal(page, base), name
        del page
    finally:
        kh.profile(enable=False, reset=True)
    return base.view(dtype).reshape(rows, width)


@pytest.mark.gpu
def test_kmers_ascii_across_chunks(kh, oracle):
    from kmer_hasher_b200 import _lib
    L = _lib.load()
    k = 32
    s = random_dna(10_000_000, 32)
    ix = kh.make_kmer_hash(s, k, do_sort=True)
    U = ix.sizes_un[0]
    got = three_ways(kh, "kmers_ascii", lambda p: _lib.check(L.kmg_kmers_ascii(ix._handle(), p)), U, k + 1, np.uint8, k + 1)
    assert np.array_equal(got.ravel(), oracle.build(s, k).extract(1)["kmer"])
    ix.free()


@pytest.mark.gpu
def test_counts_and_positions_across_chunks(kh):
    """70 Mbp, k = 32, the grouped build: counts and positions (with a k-mer number offset) in the index's own order,
    checked by the properties of test_full_size_properties."""
    from kmer_hasher_b200 import _lib
    L = _lib.load()
    k, i_base = 32, 12345
    s = random_dna(70_000_000, 70)
    s[20_000_000:21_000_000] = s[:1_000_000]               # a million k-mers with two positions
    ix = kh.make_kmer_hash(s, k)
    U, N = ix.sizes_un
    assert N == len(s) - k + 1 and U > (CHUNK_BYTES // 4)
    cnt = three_ways(kh, "counts", lambda p: _lib.check(L.kmg_counts(ix._handle(), p)), U, 4, np.int32, 1).ravel()
    cnt = cnt.astype(np.int64)
    assert cnt.sum() == N and cnt.min() >= 1 and (cnt == 2).sum() >= 999_000
    pos = three_ways(kh, "positions", lambda p: _lib.check(L.kmg_positions_base(ix._handle(), i_base, p)), N, 8, np.int32, 2)
    assert np.array_equal(pos[:, 0], np.repeat(np.arange(i_base + 1, i_base + U + 1, dtype=np.int32), cnt))
    p = pos[:, 1]
    assert np.array_equal(np.bincount(p, minlength=N + 1)[1:], np.ones(N, np.int64))   # every window exactly once
    same = pos[1:, 0] == pos[:-1, 0]
    assert np.all(p[1:][same] > p[:-1][same])              # ascending inside each k-mer
    keys = kh.kmer_keys(ix)
    code = ((s >> 1) & 3).astype(np.uint64)
    sel = np.random.default_rng(0).integers(0, N, 200_000)
    want = np.zeros(len(sel), np.uint64)
    for j in range(k):
        want = (want << np.uint64(2)) | code[p[sel].astype(np.int64) - 1 + j]
    assert np.array_equal(want, keys[pos[sel, 0] - i_base - 1])
    ix.free()


@pytest.fixture(scope="module")
def k11(kh, oracle):
    """A 20 Mbp index at k = 11 (about 4.8 positions per k-mer, 48 M pair rows) and an 8 Mbp query / second index."""
    k = 11
    a = random_dna(20_000_000, 111)
    q = random_dna(8_000_000, 112)
    ia = kh.make_kmer_hash(a, k, do_sort=True)
    oa = oracle.build(a, k)
    yield k, a, q, ia, oa
    ia.free(); oa.close()


@pytest.mark.gpu
def test_pairs_chunk_across_chunks(kh, k11):
    from kmer_hasher_b200 import _lib
    L = _lib.load()
    k, a, q, ia, oa = k11
    P = ia.sizes[2]
    assert P == oa.P
    first = 1_234_567
    n = P - first
    got = three_ways(kh, "pairs", lambda p: _lib.check(L.kmg_pairs_chunk(ia._handle(), first, n, p)), n, 12, np.int32, 3)
    assert np.array_equal(got.ravel(), oa.extract(4, with_keys=False)["pair_pos"][3 * first:])


@pytest.mark.gpu
def test_query_emit_chunk_across_chunks(kh, oracle, k11):
    import ctypes as C
    from kmer_hasher_b200 import _lib
    L = _lib.load()
    k, a, q, ia, oa = k11
    st, M = C.c_void_p(), C.c_uint64()
    _lib.check(L.kmg_query_begin(ia._handle(), q.ctypes.data, len(q), k, C.byref(st), C.byref(M)))
    try:
        first = 777_777
        n = M.value - first
        got = three_ways(kh, "probe_emit", lambda p: _lib.check(L.kmg_query_emit_chunk(st, first, n, p)), n, 8, np.int32, 2)
    finally:
        L.kmg_query_free(st)
    qk, qs = oracle.windows(q, k)
    want = probe_rows(oa.extract(2 | 8), qk, qs, k)
    assert len(want) == M.value
    assert np.array_equal(got, want[first:])


@pytest.mark.gpu
def test_join_emit_chunk_across_chunks(kh, oracle, k11):
    import ctypes as C
    from kmer_hasher_b200 import _lib
    L = _lib.load()
    k, a, q, ia, oa = k11
    ib = kh.make_kmer_hash(q, k)
    st, M = C.c_void_p(), C.c_uint64()
    _lib.check(L.kmg_join_begin(ia._handle(), ib._handle(), C.byref(st), C.byref(M)))
    try:
        first = 555_555
        n = M.value - first
        got = three_ways(kh, "join_emit", lambda p: _lib.check(L.kmg_join_emit_chunk(st, first, n, p)), n, 8, np.int32, 2)
    finally:
        L.kmg_join_free(st)
    want = join_rows(oa.extract(2 | 8), oracle.build(q, k).extract(2 | 8))
    assert len(want) == M.value
    assert np.array_equal(got, want[first:])
    ib.free()
