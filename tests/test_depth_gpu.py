"""seq.kmer.depth (kmg_count_depth / kmg_index_depth, seq_kmer_depth, .Call("sequence_kmer_depth")) against a restatement.

`expected_depth` restates the result from the plain-C oracle: `oracle.build(query, k).extract(2)` lists exactly the windows
the window rule emits (1-based starts) with their k-mer numbers, its keys turn those into keys, and the table side is a
count matrix -- the restated count table of `expected_counts`, or the list lengths of an index (`extract(8)`).  Every
other window is NA.  `revcomp_keys` restates the reverse complement in code space.
"""
import ctypes as C
import hashlib

import numpy as np
import pytest

from conftest import random_dna
from test_counts_oracle_gpu import _oracle, expected_counts
from test_extraction_chunks_gpu import three_ways

NA = -2**31
INT_MAX = 2**31 - 1
CODE = {ord("A"): 0, ord("C"): 1, ord("T"): 2, ord("G"): 3}


def revcomp_keys(keys, k):
    """Reverse complement of 2-bit keys in code space: codes reversed, each complemented as code ^ 2 (A0<->T2, C1<->G3)."""
    keys = np.asarray(keys, np.uint64)
    out = np.zeros_like(keys)
    for j in range(k):                                     # the last code of the key becomes the first of its complement
        out = (out << np.uint64(2)) | (((keys >> np.uint64(2 * j)) & np.uint64(3)) ^ np.uint64(2))
    return out


def _as_bytes(q):
    return q.encode("latin-1") if isinstance(q, str) else (q.tobytes() if isinstance(q, np.ndarray) else bytes(q))


def expected_depth(table_keys, matrix, query, k, both):
    """nwin x source_n int32: row r = window at 0-based start r; the k-mer's row of `matrix` (rows in ascending
    `table_keys` order, 0 if absent), plus its reverse complement's row (once for a palindrome) with `both`, saturated
    at INT32_MAX; NA for a window the window rule does not emit."""
    q = _as_bytes(query)
    m = np.asarray(matrix, np.int64)
    m = m[:, None] if m.ndim == 1 else m
    nwin = max(0, len(q) - k + 1)
    out = np.full((nwin, m.shape[1]), NA, np.int64)
    if nwin == 0:
        return out.astype(np.int32)
    e = _oracle().build(q, k, guard=False).extract(2)
    pos = e["pos"].reshape(-1, 2).astype(np.int64)
    wkeys = e["keys"][pos[:, 0] - 1]

    def lookup(x):
        if len(table_keys) == 0:
            return np.zeros((len(x), m.shape[1]), np.int64)
        idx = np.minimum(np.searchsorted(table_keys, x), len(table_keys) - 1)
        return np.where((table_keys[idx] == x)[:, None], m[idx], 0)

    v = lookup(wkeys)
    if both:
        rk = revcomp_keys(wkeys, k)
        v = v + np.where((rk != wkeys)[:, None], lookup(rk), 0)
    out[pos[:, 1] - 1] = np.minimum(v, INT_MAX)
    return out.astype(np.int32)


def encode(s):
    """2-bit key of an ACGT string (first base most significant)."""
    key = 0
    for c in s.encode():
        key = (key << 2) | CODE[c]
    return key


def revcomp_str(s):
    return s[::-1].translate(str.maketrans("ACGT", "TGCA"))


def test_revcomp_keys_by_hand():
    assert revcomp_keys([encode("AACC")], 4).tolist() == [250] and encode("AACC") == 5 and encode("GGTT") == 250
    assert encode("ACGT") == 30 and revcomp_keys([30], 4).tolist() == [30]          # its own reverse complement
    assert revcomp_keys([0, 1, 2, 3], 1).tolist() == [2, 3, 0, 1]                   # A->T, C->G, T->A, G->C
    assert revcomp_keys([0], 32).tolist() == [0xAAAAAAAAAAAAAAAA]                    # A^32 -> T^32
    rng = np.random.default_rng(5)
    for k in (1, 2, 7, 31, 32):
        strs = ["".join(rng.choice(list("ACGT"), k)) for _ in range(50)]
        keys = np.array([encode(s) for s in strs], np.uint64)
        assert revcomp_keys(keys, k).tolist() == [encode(revcomp_str(s)) for s in strs]
        assert np.array_equal(revcomp_keys(revcomp_keys(keys, k), k), keys)


# Table: count.kmers("ACGTT", k = 2) = AC, CG, GT, TT once each (A0 C1 T2 G3).  CG is a palindrome; rc(AC) = GT.
HAND_TABLE = (["ACGTT"], 0)
HAND = {
    # query: (forward, both strands); GN and NC contain an N; the last window GT of ACNGT is freshly primed after
    # the N and ends the string (end-of-string rule), so it is NA too
    "ACGNCGT": ([1, 1, NA, NA, 1, 1], [2, 1, NA, NA, 1, 2]),
    "ACNGT": ([1, NA, NA, NA], [2, NA, NA, NA]),
    "AATT": ([0, 0, 1], [1, 0, 1]),                         # AA absent (its rc TT counted), AT absent palindrome
}


def test_expected_depth_by_hand():
    keys, m = expected_counts([HAND_TABLE], 2, 1)
    assert keys.tolist() == [1, 7, 10, 14]
    for q, (fwd, both) in HAND.items():
        assert expected_depth(keys, m, q, 2, False).ravel().tolist() == fwd, q
        assert expected_depth(keys, m, q, 2, True).ravel().tolist() == both, q
    assert expected_depth(keys, m, "ACG", 3, False).tolist() == [[NA]]          # length k: one window, dropped
    assert expected_depth(keys, m, "", 2, False).shape == (0, 1)


def test_python_guards_on_cpu():
    """seq_kmer_depth checks its arguments before the handle is used (the handle here was never made)."""
    import kmer_hasher_b200 as kh
    assert kh.NA_INTEGER == NA
    ct = kh.KmerCounts(None, 4, 3)
    with pytest.raises(TypeError, match="external pointer"):
        kh.seq_kmer_depth("not a pointer", "ACGTACGT")
    with pytest.raises(ValueError, match="single sequence"):
        kh.seq_kmer_depth(ct, ["ACGTAC", "ACGTAC"])
    with pytest.raises(ValueError, match="longer than k"):
        kh.seq_kmer_depth(ct, "ACGT")
    with pytest.raises(ValueError, match="out holds 32 bytes; the depth needs 36"):
        kh.seq_kmer_depth(ct, "ACGTAC", out=np.empty(8, np.int32))
    with pytest.raises(ValueError, match="cleared"):
        kh.seq_kmer_depth(ct, ["ACGTAC"], out=np.empty((3, 3), np.int32))
    ix = kh.KmerHash(None, 31)
    with pytest.raises(ValueError, match="longer than k"):
        kh.seq_kmer_depth(ix, "A" * 31)


def test_glue_registration_and_argument_errors_on_cpu():
    from rsession import RError, RSession
    R = RSession()
    with pytest.raises(RError, match="Incorrect number of arguments"):
        R.call("sequence_kmer_depth", R.integer(1), R.character("ACGT"))
    with pytest.raises(RError, match="single sequence"):
        R.call("sequence_kmer_depth", R.integer(1), R.character("ACGT", "ACGT"), R.integer(0))
    with pytest.raises(RError, match="single sequence"):
        R.call("sequence_kmer_depth", R.integer(1), R.integer(1), R.integer(0))
    with pytest.raises(RError, match="both.strands should be TRUE or FALSE"):
        R.call("sequence_kmer_depth", R.integer(1), R.character("ACGT"), R.integer(2))
    with pytest.raises(RError, match="both.strands should be TRUE or FALSE"):
        R.call("sequence_kmer_depth", R.integer(1), R.character("ACGT"), R.character("1"))
    with pytest.raises(RError, match="ptr_r should be an external pointer"):
        R.call("sequence_kmer_depth", R.integer(1), R.character("ACGT"), R.integer(1))
    assert R.stub.rstub_protect_depth() == 0


# ---- on the GPU ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def kh():
    import kmer_hasher_b200 as kh
    return kh


def _lib():
    from kmer_hasher_b200 import _lib as lib
    return lib, lib.load()


@pytest.mark.gpu
def test_hand_cases_on_the_device(kh):
    ct = kh.count_kmers(HAND_TABLE[0], (2, 0, 1))
    for q, (fwd, both) in HAND.items():
        assert kh.seq_kmer_depth(ct, q).ravel().tolist() == fwd, q
        assert kh.seq_kmer_depth(ct, q, both_strands=True).ravel().tolist() == both, q
    ix = kh.make_kmer_hash("ACGTT", 2)
    for q, (fwd, both) in HAND.items():
        assert kh.seq_kmer_depth(ix, q).ravel().tolist() == fwd, q
        assert kh.seq_kmer_depth(ix, q, both_strands=True).ravel().tolist() == both, q
    ct.free(); ix.free()


def _palindrome(k, seed):
    rng = np.random.default_rng(seed)
    half = "".join(rng.choice(list("ACGT"), k // 2))
    return half + revcomp_str(half)


def _table_batches(k, sn):
    """Batches (sequences, source) into sn sources: a mixed sequence, one without A (with an even-k palindrome), a mix of
    known and new k-mers."""
    base = random_dna(30_000, 300 + k, p_n=0.002, p_lower=0.2, p_other=0.005, n_runs=2)
    no_a = np.frombuffer(b"CGT", np.uint8)[np.random.default_rng(k).integers(0, 3, 8_000)].copy()
    pal = (_palindrome(k, k) * 3) if k % 2 == 0 else "ACGT" * 8
    return [([base], 0 % sn), ([no_a, pal], 1 % sn), ([base[10_000:18_000].copy(), random_dna(4_000, 400 + k)], 2 % sn)]


def _queries(k, base):
    pal = _palindrome(k, k) if k % 2 == 0 else "ACGT"
    shared = base[2_000:14_000].copy()
    return {
        "mixed": random_dna(12_000, 500 + k, p_n=0.003, p_lower=0.3, p_other=0.01, n_runs=2),
        "shared": shared,
        "none": np.full(k + 300, ord("A"), np.uint8),       # A^k: no table sequence of these seeds holds it at k >= 11
        "palindromes": np.frombuffer((pal + "N" + pal + pal + "acgtN" + "ACGT" * k).encode(), np.uint8).copy(),
        "tail": np.concatenate([random_dna(300, 600 + k), np.frombuffer(b"N", np.uint8), shared[:k].copy()]),
    }


def _raw_depth(kh, ptr, q, strands, cols):
    """kmg_*_depth through the C ABI (lengths the Python guard refuses); returns the rows."""
    lib, L = _lib()
    b = _as_bytes(q)
    nwin = max(0, len(b) - ptr.k + 1)
    out = np.full((max(nwin, 1), cols), 12345, np.int32)
    fn = L.kmg_count_depth if isinstance(ptr, kh.KmerCounts) else L.kmg_index_depth
    lib.check(fn(ptr._handle(), b if b else None, len(b), strands, out.ctypes.data if nwin else None))
    if nwin == 0:
        assert (out == 12345).all()                        # nothing written
    return out[:nwin]


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 11, 16, 21, 31, 32])
def test_count_table_depth_matches_the_restatement(kh, k):
    """source_n 1, 2 and 3 built by several batches; queries with N/n, N runs, lower case, IUPAC bytes, shared and
    unshared k-mers, palindromes, the end-of-string rule, length k and 0; both strands."""
    for sn in (1, 2, 3):
        batches = _table_batches(k, sn)
        ptr = None
        for seqs, source in batches:
            ptr = kh.count_kmers(seqs, (k, source, sn), ptr)
        keys, m = expected_counts(batches, k, sn)
        assert ptr.sizes[0] == len(keys)
        for name, q in _queries(k, batches[0][0][0]).items():
            for both in (False, True):
                got = kh.seq_kmer_depth(ptr, q, both_strands=both)
                want = expected_depth(keys, m, q, k, both)
                assert got.shape == (len(q) - k + 1, sn) and np.array_equal(got, want), (name, sn, both)
                if name == "tail":
                    assert (got[-1] == NA).all()
                if name == "none" and k >= 11 and not both:
                    assert (got == 0).all()
                if name == "shared":                       # every valid window was counted into source 0
                    assert (got[got[:, 0] != NA, 0] > 0).all()
        for strands in (0, 1):
            one = _raw_depth(kh, ptr, batches[0][0][0][:k].copy(), strands, sn)
            assert one.shape == (1, sn) and (one == NA).all()  # one window, dropped by the end-of-string rule
            assert _raw_depth(kh, ptr, b"", strands, sn).shape == (0, sn)
        ptr.free()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 11, 16, 21, 31, 32])
def test_index_depth_matches_the_restatement(kh, k):
    """Depth against a position index = the length of the k-mer's position list; a sorted index and (k >= 21) a grouped
    one, whose key table is streamed."""
    batches = _table_batches(k, 1)
    seq = batches[0][0][0]
    e = _oracle().build(seq, k).extract(8)
    for do_sort in (True, False):
        ix = kh.make_kmer_hash(seq, k, do_sort=do_sort)
        assert kh._L.kmg_index_order(ix._handle()) == (1 if do_sort or k < 21 else 0)
        for name, q in _queries(k, seq).items():
            for both in (False, True):
                got = kh.seq_kmer_depth(ix, q, both_strands=both)
                assert got.shape == (len(q) - k + 1, 1)
                assert np.array_equal(got, expected_depth(e["keys"], e["count"], q, k, both)), (name, do_sort, both)
        one = _raw_depth(kh, ix, seq[:k].copy(), 1, 1)
        assert one.tolist() == [[NA]]
        ix.free()


@pytest.mark.gpu
def test_empty_table_still_writes_every_row(kh):
    ct = kh.count_kmers([np.full(50, ord("N"), np.uint8)], (5, 0, 2))         # U = 0: no key table
    assert ct.sizes[0] == 0
    q = "ACGTACGTNNACGTACGTAC"
    for both in (False, True):
        got = kh.seq_kmer_depth(ct, q, both_strands=both)
        assert np.array_equal(got, expected_depth(np.empty(0, np.uint64), np.zeros((0, 2)), q, 5, both))
    ct.free()


@pytest.mark.gpu
def test_depth_after_more_batches_sees_the_new_table(kh, tmp_path):
    """The key table is cached by the first depth call: counting another batch must drop it (count_kmers and
    count_kmers_file)."""
    k, sn = 21, 2
    a = random_dna(40_000, 71, p_n=0.001)
    b = random_dna(30_000, 72)
    b[:10_000] = a[5_000:15_000]
    q = np.concatenate([a[:20_000], b[:20_000]])
    batches = [([a], 0)]
    ptr = kh.count_kmers([a], (k, 0, sn))
    for both in (False, True):
        assert np.array_equal(kh.seq_kmer_depth(ptr, q, both_strands=both), expected_depth(*expected_counts(batches, k, sn), q, k, both))
    ptr = kh.count_kmers([b], (k, 1, sn), ptr)
    batches.append(([b], 1))
    for both in (False, True):
        assert np.array_equal(kh.seq_kmer_depth(ptr, q, both_strands=both), expected_depth(*expected_counts(batches, k, sn), q, k, both))
    recs = [random_dna(5_000, 80 + i) for i in range(3)] + [a[30_000:36_000].copy()]
    path = tmp_path / "reads.fa"
    path.write_bytes(b"".join(b">r%d\n" % i + r.tobytes() + b"\n" for i, r in enumerate(recs)))
    ptr = kh.count_kmers_file(str(path), (k, 0, sn), ptr)
    batches.append((recs, 0))
    q2 = np.concatenate([q, recs[1], recs[3]])
    for both in (False, True):
        assert np.array_equal(kh.seq_kmer_depth(ptr, q2, both_strands=both), expected_depth(*expected_counts(batches, k, sn), q2, k, both))
    ptr.free()


@pytest.mark.gpu
def test_depth_across_chunks(kh):
    """source_n = 3, 23 M windows of 12 bytes: one launch into device memory, 2 chunks of 22,369,621 windows into pinned
    memory, 5 staged chunks of 5,592,405 into pageable memory -- chunk starts that are not multiples of 16.  The query is
    a device tensor."""
    import torch
    lib, L = _lib()
    k, sn = 31, 3
    q = random_dna(23_000_000, 2300, p_n=0.0001)
    batches = [([q[:8_000_000].copy()], 0), ([q[4_000_000:12_000_000].copy()], 1),
               ([q[10_000_000:11_000_000].copy(), random_dna(2_000_000, 2301)], 2)]
    ptr = None
    for seqs, source in batches:
        ptr = kh.count_kmers(seqs, (k, source, sn), ptr)
    nwin = len(q) - k + 1
    assert nwin * 12 > (256 << 20) and (64 << 20) // 12 % 16 != 0 and (256 << 20) // 12 % 16 != 0
    dq = torch.from_numpy(q).cuda()
    h = ptr._handle()
    got = three_ways(kh, "depth_lookup", lambda p: lib.check(L.kmg_count_depth(h, C.c_void_p(dq.data_ptr()), len(q), 0, C.c_void_p(p))),
                     nwin, 12, np.int32, sn)
    keys, m = expected_counts(batches, k, sn)
    want = expected_depth(keys, m, q, k, False)
    assert np.array_equal(got, want)
    assert (got[:4_000_000, 0] > 0).sum() > 3_900_000 and (got[4_000_000:8_000_000, :2] > 0).all(axis=1).sum() > 3_900_000
    ptr.free()


@pytest.mark.gpu
def test_caller_memory_and_frees(kh):
    """A device tensor allocated before a depth call is unchanged by it; a table freed right after a depth call gives all
    its device memory back (after kmg_trim)."""
    import torch
    lib, L = _lib()
    warm = kh.count_kmers([random_dna(10_000, 1)], (21, 0, 2))
    kh.seq_kmer_depth(warm, random_dna(1_000, 2))
    warm.free()
    sentinel = torch.randint(-2**31, 2**31 - 1, (16 << 20,), dtype=torch.int32, device="cuda")
    sha = hashlib.sha256(sentinel.cpu().numpy().tobytes()).hexdigest()
    seq = random_dna(6_000_000, 3)
    q = random_dna(3_000_000, 4)
    q[:1_000_000] = seq[:1_000_000]
    torch.cuda.synchronize()
    lib.check(L.kmg_trim())
    free0 = torch.cuda.mem_get_info()[0]
    ct = kh.count_kmers([seq], (21, 1, 2))
    ix = kh.make_kmer_hash(seq, 21)
    dout = torch.empty((len(q) - 20, 2), dtype=torch.int32, device="cuda")
    kh.seq_kmer_depth(ct, q, both_strands=True, out=dout)
    d1 = kh.seq_kmer_depth(ix, q, both_strands=True)
    torch.cuda.synchronize()
    assert np.array_equal(dout.cpu().numpy()[:, 1], d1[:, 0]) and (d1[:1_000_000] > 0).sum() > 999_000
    assert hashlib.sha256(sentinel.cpu().numpy().tobytes()).hexdigest() == sha
    held = torch.cuda.mem_get_info()[0]
    assert free0 - held > 16 * (8 << 20)                   # the key tables alone: 2^24 slots of 16 bytes each
    ct.free(); ix.free()
    del dout
    torch.cuda.empty_cache()
    lib.check(L.kmg_trim())
    assert torch.cuda.mem_get_info()[0] >= free0 - (2 << 20)


@pytest.mark.gpu
def test_c_abi_guards(kh):
    lib, L = _lib()
    ct = kh.count_kmers(["ACGTACGTAC"], (4, 0, 2))
    h = ct._handle()
    q = b"ACGTACGTAC"
    out = np.empty((7, 2), np.int32)
    assert L.kmg_count_depth(h, q, len(q), 2, out.ctypes.data) == -1
    assert L.kmg_count_depth(h, q, len(q), -1, out.ctypes.data) == -1
    assert L.kmg_count_depth(h, q, len(q), 0, None) == -1
    assert L.kmg_count_depth(h, q, 2**31 - 1, 0, out.ctypes.data) == -3                # qlen + 1 > INT32_MAX
    assert L.kmg_count_depth(h, None, 5, 0, out.ctypes.data) == -1
    assert L.kmg_count_depth(None, q, len(q), 0, out.ctypes.data) == -1
    assert L.kmg_count_depth(h, q, 3, 0, None) == 0                                     # no window: nothing to write
    assert L.kmg_count_depth(h, q, len(q), 1, out.ctypes.data) == 0
    ix = kh.make_kmer_hash(q, 4)
    assert L.kmg_index_depth(ix._handle(), q, len(q), 3, out.ctypes.data) == -1
    assert L.kmg_index_depth(ix._handle(), q, 2**31 - 1, 0, out.ctypes.data) == -3
    ct.free(); ix.free()


@pytest.mark.gpu
def test_r_glue_depth(oracle):
    """.Call("sequence_kmer_depth") on a count table and an index: t() of the source_n x nwin matrix equals the
    restatement, NA included; sizes are checked before anything is allocated."""
    from rsession import RError, RSession
    R = RSession()
    k, sn = 16, 3
    seqs = [random_dna(20_000, 90 + i, p_n=0.002) for i in range(3)]
    ptr = R.nil
    for i, s in enumerate(seqs):
        ptr = R.call("count_kmers", ptr, R.integer(k, i, sn), R.character(s))
    q = np.concatenate([seqs[0][:5_000], random_dna(3_000, 95, p_n=0.01, p_lower=0.3), seqs[2][:2_000]])
    keys, m = expected_counts([([s], i) for i, s in enumerate(seqs)], k, sn)
    ix = R.make_kmer_hash(seqs[1], k)
    e = oracle.build(seqs[1], k).extract(8)
    for both in (0, 1):
        for p, cols, want in ((ptr, sn, expected_depth(keys, m, q, k, both)), (ix, 1, expected_depth(e["keys"], e["count"], q, k, both))):
            r = R.call("sequence_kmer_depth", p, R.character(q), R.integer(both))
            assert R.dims(r) == (cols, len(q) - k + 1)
            got = R.ints(r).reshape(len(q) - k + 1, cols)
            R.stub.rstub_release(r)
            assert np.array_equal(got, want) and (got == NA).any()
    with pytest.raises(RError, match="the sequence should be longer than k"):
        R.call("sequence_kmer_depth", ptr, R.character("ACGT" * 4), R.integer(0))
    wide = R.call("count_kmers", R.nil, R.integer(k, 0, 1000), R.character(seqs[0]))
    long_seq, forward = R.character(np.full(2_200_000, ord("A"), np.uint8)), R.integer(0)
    live = R.stub.rstub_live_objects()
    with pytest.raises(RError, match="more than an R matrix can hold"):
        R.call("sequence_kmer_depth", wide, long_seq, forward)
    assert R.stub.rstub_live_objects() == live                                          # refused before allocating
    assert R.stub.rstub_protect_depth() == 0
    for p in (ptr, ix, wide):
        R.stub.rstub_finalize(p)
