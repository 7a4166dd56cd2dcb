"""Match segments of a join (kmg_join_segments_begin, kmer_pairs_segments, .Call("kmer_pair_segments")) against the runs of
the oracle's kmer.pairs rows.

Forward: `runs_of(pairs_join(ea, eb))` (test_segments_gpu.py).  Reverse complement: the rows are `pairs_join` with a's keys
replaced by their code-space reverse complements, and the antiparallel runs (x + t, y - t) are `runs_of` over (x, -y),
mapped back and ordered by (x, y) (`anti_runs`).  Where max_count drops k-mers the rows come from the vectorised
`join_rows` over extractions without them.  Cross-checks with seq.kmer.segments tie both strands to the query path.
"""
import ctypes as C
import hashlib

import numpy as np
import pytest

import oracle as oracle_mod
from conftest import random_dna
from test_dotplot_gpu import _pair, host_revcomp, without_repeats
from test_extraction_chunks_gpu import join_rows
from test_segments_gpu import runs_of, runs_torch

INTSXP = 13


def revcomp_keys(keys, k):
    """Code-space reverse complement of 2-bit keys: the k codes reversed, each code ^ 2."""
    keys = np.asarray(keys, np.uint64)
    out = np.zeros_like(keys)
    for t in range(k):
        code = (keys >> np.uint64(2 * t)) & np.uint64(3)
        out = (out << np.uint64(2)) | (code ^ np.uint64(2))
    return out


def rc_extraction(e, k):
    """The extraction `e` with every key replaced by its reverse complement (a's side of the antiparallel join)."""
    return dict(e, keys=revcomp_keys(e["keys"], k))


def anti_runs(rows, min_rows=1):
    """(R, 3) (x, y, n): the maximal antiparallel runs (x + t, y - t) of the (x, y) rows, first row = smallest x, ordered
    by (x, y), n >= min_rows."""
    r = np.asarray(rows, np.int64).reshape(-1, 2) * np.array([1, -1])
    out = runs_of(r, min_rows)
    out[:, 1] = -out[:, 1]
    return out[np.lexsort((out[:, 1], out[:, 0]))]


def test_revcomp_and_anti_runs_by_hand():
    # ACG (codes 0 1 3) -> reverse complement CGT (1 3 2)
    assert revcomp_keys([0b000111], 3).tolist() == [0b011110]
    assert revcomp_keys(revcomp_keys([12345, 0, 2**62 - 1], 31), 31).tolist() == [12345, 0, 2**62 - 1]
    rows = [(3, 9), (4, 8), (5, 7), (5, 20), (6, 6), (7, 1), (8, 2)]   # one run of 4, two single rows off it, two singles
    assert anti_runs(rows).tolist() == [[3, 9, 4], [5, 20, 1], [7, 1, 1], [8, 2, 1]]
    assert anti_runs(rows, 2).tolist() == [[3, 9, 4]]
    assert anti_runs(np.empty((0, 2), np.int32)).shape == (0, 3)


def test_python_guards_on_cpu():
    import kmer_hasher_b200 as kh
    ix = kh.KmerHash(None, 5)
    with pytest.raises(TypeError, match="external pointer"):
        kh.kmer_pairs_segments("not a pointer", ix)
    with pytest.raises(ValueError, match="count.kmers"):
        kh.kmer_pairs_segments(ix, kh.KmerCounts(None, 5, 2))
    with pytest.raises(ValueError, match="count.kmers"):
        kh.kmer_pairs_segments(kh.KmerCounts(None, 5, 2), ix)
    for bad in (-1, 2**32):
        with pytest.raises(ValueError, match="max_count"):
            kh.kmer_pairs_segments(ix, ix, max_count=bad)
        with pytest.raises(ValueError, match="min_rows"):
            kh.kmer_pairs_segments(ix, ix, min_rows=bad)
    with pytest.raises(ValueError, match="cleared"):
        kh.kmer_pairs_segments(ix, ix)


def test_glue_registration_and_argument_errors_on_cpu():
    from rsession import RError, RSession
    R = RSession()
    with pytest.raises(RError, match="Incorrect number of arguments"):
        R.call("kmer_pair_segments", R.integer(1), R.integer(2))
    with pytest.raises(RError, match="ptr_r should be an external pointer"):
        R.call("kmer_pair_segments", R.integer(1), R.integer(2), R.integer(0, 0, 1))
    assert R.stub.rstub_protect_depth() == 0


# ---- on the GPU ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def kh():
    import kmer_hasher_b200 as kh
    return kh


def _lib():
    from kmer_hasher_b200 import _lib as lib
    return lib, lib.load()


def _begin(L, a, b, rc=0, mc=0, mr=1):
    """kmg_join_segments_begin -> (return code, handle, R)"""
    st, R = C.c_void_p(), C.c_uint64()
    rv = L.kmg_join_segments_begin(a, b, rc, mc, mr, C.byref(st), C.byref(R))
    return rv, st, R.value


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 5, 8, 11, 16, 21, 27, 31, 32])
def test_join_segments_match_oracle_runs(kh, oracle, k):
    """_pair inputs (N runs, lower case, IUPAC, a shared stretch, a reverse-complemented one, an internal repeat); two
    indexes and a self join; sorted and grouped builds of each side; both strands; min_rows 0, 1, 3 and 20."""
    s, q = _pair(k, 4000 + k)
    es, eq = oracle.build(s, k).extract(2 | 8), oracle.build(q, k).extract(2 | 8)
    for sort_a, sort_b in ((True, False), (False, True)):
        ia, ib = kh.make_kmer_hash(s, k, do_sort=sort_a), kh.make_kmer_hash(q, k, do_sort=sort_b)
        for (pa, pb), (ea, eb) in (((ia, ib), (es, eq)), ((ib, ia), (eq, es)), ((ia, ia), (es, es))):
            for rc in (False, True):
                rows = oracle_mod.pairs_join(rc_extraction(ea, k) if rc else ea, eb)
                restate = anti_runs if rc else runs_of
                want = restate(rows)
                assert want[:, 2].sum() * 2 == len(rows) and (len(want) > 0 or (rc and pa is pb))
                got = kh.kmer_pairs_segments(pa, pb, reverse_complement=rc)
                assert got.dtype == np.int32 and np.array_equal(got, want), (sort_a, sort_b, rc)
                if k >= 8 and pa is not pb:
                    assert want[:, 2].max() > 20                 # the shared stretches give long runs on both strands
                for mr in (0, 3, 20):
                    got = kh.kmer_pairs_segments(pa, pb, reverse_complement=rc, min_rows=mr)
                    assert np.array_equal(got, restate(rows, mr)), (sort_a, sort_b, rc, mr)
        ia.free(); ib.free()


@pytest.mark.gpu
def test_different_k(kh, oracle):
    """Indexes of different k join on raw 2-bit keys, as kmer.pairs does; the reverse complement needs one k."""
    lib, L = _lib()
    s, q = _pair(11, 61)
    ea, eb = oracle.build(s, 11).extract(2 | 8), oracle.build(q, 13).extract(2 | 8)
    ia, ib = kh.make_kmer_hash(s, 11), kh.make_kmer_hash(q, 13)
    rows = oracle_mod.pairs_join(ea, eb)
    assert len(rows) > 0
    assert np.array_equal(kh.kmer_pairs_segments(ia, ib), runs_of(rows))
    assert np.array_equal(kh.kmer_pairs_segments(ia, ib, min_rows=2), runs_of(rows, 2))
    assert _begin(L, ia._handle(), ib._handle(), rc=1)[0] == -2
    with pytest.raises(lib.KmgError, match="one k"):
        kh.kmer_pairs_segments(ia, ib, reverse_complement=True)
    ia.free(); ib.free()


def _cross_inputs(seed, k):
    """(A, b): random ACGT / acgt / N strings whose ends have N-free runs longer than k (the end-of-string rule and IUPAC
    bytes are where the byte-level reverse complement of seq.kmer.segments legitimately differs); b shares stretches of
    A on both strands."""
    A = random_dna(40_000, seed, p_n=0.003, p_lower=0.2)
    b = random_dna(30_000, seed + 1, p_n=0.003, p_lower=0.2)
    for x in (A, b):
        x[:2 * k] = random_dna(2 * k, seed + 2)
        x[-2 * k:] = random_dna(2 * k, seed + 3)
    b[1_000:6_000] = A[10_000:15_000]
    b[8_000:12_000] = np.frombuffer(host_revcomp(A[20_000:24_000]), np.uint8)
    return A, b


def _query_equivalents(kh, ib, A, k, min_rows=1):
    """(forward, rc) segments of kmer_pairs_segments(index(A), ib) restated from seq_kmer_segments(ib, A, k)."""
    L = len(A)
    f = kh.seq_kmer_segments(ib, A, k, min_rows=min_rows, allow_k32=True).astype(np.int64)
    f[:, 0] -= k - 1
    r = kh.seq_kmer_segments(ib, A, k, reverse_complement=True, min_rows=min_rows, allow_k32=True).astype(np.int64)
    i, j, n = r[:, 0], r[:, 1], r[:, 2]
    r = np.stack([L - i - n + 2, j + n - 1, n], 1)
    return f, r[np.lexsort((r[:, 1], r[:, 0]))]


@pytest.mark.gpu
@pytest.mark.parametrize("k", [7, 16, 31])
def test_cross_check_with_query_segments(kh, k):
    A, b = _cross_inputs(100 + k, k)
    ia, ib = kh.make_kmer_hash(A, k), kh.make_kmer_hash(b, k, do_sort=True)
    for mr in (1, 12):
        f, r = _query_equivalents(kh, ib, A, k, mr)
        assert len(f) > 0 and len(r) > 0
        assert np.array_equal(kh.kmer_pairs_segments(ia, ib, min_rows=mr), f), mr
        assert np.array_equal(kh.kmer_pairs_segments(ia, ib, reverse_complement=True, min_rows=mr), r), mr
    ia.free(); ib.free()


@pytest.mark.gpu
def test_test_fa_self(kh, test_fa):
    """test.fa against itself at k = 16 (~29 M rows, the top k-mer has 2,188 positions), both strands, against the query
    path."""
    k = 16
    ix = kh.make_kmer_hash(test_fa, k)
    f, r = _query_equivalents(kh, ix, test_fa, k)
    assert f[:, 2].sum() > 25_000_000
    assert np.array_equal(kh.kmer_pairs_segments(ix, ix), f)
    assert np.array_equal(kh.kmer_pairs_segments(ix, ix, reverse_complement=True), r)
    ix.free()


@pytest.mark.gpu
@pytest.mark.parametrize("mc", [0, 3])
def test_row_totals(kh, mc):
    """With min_rows 0 the n of all runs sum to kmg_join_begin's M and to the 1 x 1 kmer_pairs_dotplot total."""
    lib, L = _lib()
    k = 15
    s, q = _pair(k, 5)
    s = np.concatenate([s, s[:5_000], s[2_000:4_000]])        # repeated stretches: lists of 2 and 3 positions
    ia, ib = kh.make_kmer_hash(s, k), kh.make_kmer_hash(q, k, do_sort=True)
    for pa, pb in ((ia, ib), (ib, ia), (ia, ia)):
        got = kh.kmer_pairs_segments(pa, pb, max_count=mc, min_rows=0)
        total = kh.kmer_pairs_dotplot(pa, pb, a_range=(0, 2**31), b_range=(0, 2**31), bins=(1, 1), max_count=mc)[0, 0]
        assert got[:, 2].astype(np.int64).sum() == total > 0
        if mc == 0:
            st, M = C.c_void_p(), C.c_uint64()
            lib.check(L.kmg_join_begin(pa._handle(), pb._handle(), C.byref(st), C.byref(M)))
            L.kmg_join_free(st)
            assert got[:, 2].astype(np.int64).sum() == M.value
    ia.free(); ib.free()


@pytest.mark.gpu
def test_max_count(kh, oracle):
    """max_count equals the runs of the rows without the k-mers too long in either index (the repeats of
    test_dotplot_gpu's max_count test), both strands, with and without min_rows."""
    k = 11
    s, q = _pair(k, 77)
    s = s.copy()
    for at in (12_000, 13_000, 14_000, 15_000, 16_000):
        s[at:at + 400] = s[7_000:7_400]
    for at in (18_000, 18_500):
        s[at:at + 100] = s[8_000:8_100]
    es, eq = oracle.build(s, k).extract(2 | 8), oracle.build(q, k).extract(2 | 8)
    longest = int(es["count"].max())
    assert longest >= 6
    ia, ib = kh.make_kmer_hash(s, k, do_sort=True), kh.make_kmer_hash(q, k)
    for (pa, pb), (ea, eb) in (((ia, ib), (es, eq)), ((ib, ia), (eq, es)), ((ia, ia), (es, es))):
        for rc in (False, True):
            xa = rc_extraction(ea, k) if rc else ea
            sizes = []
            for mc in (1, 2, 3, longest - 1, longest, 2**32 - 1):
                rows = join_rows(without_repeats(xa, mc), without_repeats(eb, mc))
                for mr in (1, 15):
                    got = kh.kmer_pairs_segments(pa, pb, reverse_complement=rc, max_count=mc, min_rows=mr)
                    assert np.array_equal(got, (anti_runs if rc else runs_of)(rows, mr)), (rc, mc, mr)
                sizes.append(len(rows))
            if not rc and pa is not ib:                         # the repeated stretches are shared forward
                assert sizes[0] < sizes[2] < sizes[3] < sizes[4]
    ia.free(); ib.free()


@pytest.mark.gpu
def test_more_than_2_31_rows(kh):
    """A 50,000-base homopolymer: its N positions are 1..N.  Forward self join: N^2 ~ 2.5 * 10^9 rows, one run per
    diagonal d, x from max(1, 1 + d) to min(N, N + d).  "A"*n against "T"*n with rc: every (x, y) is a row and each
    anti-diagonal x + y = t holds one antiparallel run, x from max(1, t - N) to min(N, t - 1)."""
    k, n = 16, 50_000
    N = n - k + 1
    ia, it = kh.make_kmer_hash("A" * n, k, do_sort=True), kh.make_kmer_hash("T" * n, k)
    assert ia.sizes_un == (1, N) and N * N > 2**31
    d = np.arange(1 - N, N, dtype=np.int64)
    x0, x1 = np.maximum(1, 1 + d), np.minimum(N, N + d)
    want = np.stack([x0, x0 - d, x1 - x0 + 1], 1)
    want = want[np.lexsort((want[:, 1], want[:, 0]))]
    assert want[:, 2].sum() == N * N
    assert np.array_equal(kh.kmer_pairs_segments(ia, ia), want)
    assert np.array_equal(kh.kmer_pairs_segments(ia, ia, min_rows=40_000), want[want[:, 2] >= 40_000])
    assert len(kh.kmer_pairs_segments(ia, ia, max_count=N - 1)) == 0
    t = np.arange(2, 2 * N + 1, dtype=np.int64)
    x0, x1 = np.maximum(1, t - N), np.minimum(N, t - 1)
    want = np.stack([x0, t - x0, x1 - x0 + 1], 1)
    want = want[np.lexsort((want[:, 1], want[:, 0]))]
    assert want[:, 2].sum() == N * N
    assert np.array_equal(kh.kmer_pairs_segments(ia, it, reverse_complement=True), want)
    assert np.array_equal(kh.kmer_pairs_segments(ia, it, reverse_complement=True, min_rows=40_000), want[want[:, 2] >= 40_000])
    assert len(kh.kmer_pairs_segments(ia, it, reverse_complement=True, max_count=N - 1)) == 0
    assert len(kh.kmer_pairs_segments(ia, it)) == 0               # forward: nothing shared
    ia.free(); it.free()


@pytest.mark.gpu
def test_output_memory_kinds_and_chunks(kh):
    """A random 30 Mbp self join at k = 12: ~40 M runs (480 MB).  The same bytes into a device tensor, pinned memory (2
    chunks) and pageable memory (7 or more chunks), guard bytes untouched; emit_chunk windows agree with the full emit;
    the result equals the runs of the library's own kmer.pairs rows, restated on the device."""
    import torch
    lib, L = _lib()
    k, n, G = 12, 30_000_000, 16
    s = random_dna(n, 4343)
    ix = kh.make_kmer_hash(s, k)
    rv, st, R = _begin(L, ix._handle(), ix._handle())
    lib.check(rv)
    try:
        pin_rows, stage_rows = (256 << 20) // 12, (64 << 20) // 12
        assert R > pin_rows
        kh.profile(enable=True, reset=True)
        dev = torch.full((3 * R + 2 * G,), -7, dtype=torch.int32, device="cuda")
        lib.check(L.kmg_segments_emit(st, C.c_void_p(dev[G:].data_ptr())))
        torch.cuda.synchronize()
        assert kh.profile(reset=True)["segments_emit"][1] == 1
        pin = kh.pinned_empty(3 * R + 2 * G, np.int32)
        page = np.empty(3 * R + 2 * G, np.int32)
        for buf, chunks in ((pin, -(-R // pin_rows)), (page, -(-R // stage_rows))):
            buf[:] = -7
            lib.check(L.kmg_segments_emit(st, C.c_void_p(buf[G:].ctypes.data)))
            assert kh.profile(reset=True)["segments_emit"][1] == chunks >= 2
        kh.profile(enable=False, reset=True)
        d = dev.cpu().numpy()
        for buf in (d, pin, page):
            assert (buf[:G] == -7).all() and (buf[-G:] == -7).all()
        assert np.array_equal(pin, d) and np.array_equal(page, d)
        runs = d[G:-G].reshape(R, 3)
        for a, b in ((0, 1), (1, 12_345_679), (12_345_679, R - 3), (R - 3, R)):
            part = np.full(3 * (b - a) + 2 * G, -7, np.int32)
            lib.check(L.kmg_segments_emit_chunk(st, a, b - a, C.c_void_p(part[G:].ctypes.data)))
            assert (part[:G] == -7).all() and (part[-G:] == -7).all() and np.array_equal(part[G:-G].reshape(-1, 3), runs[a:b])
        pd = torch.full((3 * 1000 + 2 * G,), -7, dtype=torch.int32, device="cuda")
        lib.check(L.kmg_segments_emit_chunk(st, R - 1000, 1000, C.c_void_p(pd[G:].data_ptr())))
        p = pd.cpu().numpy()
        assert (p[:G] == -7).all() and (p[-G:] == -7).all() and np.array_equal(p[G:-G].reshape(-1, 3), runs[R - 1000:])
    finally:
        L.kmg_segments_free(st)
    assert (runs[:, 2] > n // 2).sum() == 1                   # the main diagonal is one run
    rows = torch.from_numpy(kh.kmer_pairs(ix, ix)).cuda()
    want = runs_torch(rows)
    del rows
    assert want.shape[0] == R
    assert torch.equal(torch.from_numpy(runs).cuda().to(torch.int64), want)
    ix.free()


@pytest.mark.gpu
def test_empty_cases(kh):
    lib, L = _lib()
    empty = kh.make_kmer_hash("N" * 50, 5)                     # U = 0
    assert empty.sizes_un == (0, 0)
    ia, ic = kh.make_kmer_hash("A" * 50, 5), kh.make_kmer_hash("C" * 50, 5)
    for pa, pb in ((empty, ia), (ia, empty), (empty, empty), (ia, ic), (ic, ia)):   # no shared k-mer on either strand
        for rc in (False, True):
            assert kh.kmer_pairs_segments(pa, pb, reverse_complement=rc).shape == (0, 3)
    assert kh.kmer_pairs_segments(ia, ia, min_rows=100).shape == (0, 3)     # every run filtered out
    o = np.full(6, -1, np.int32)
    rv, st, R = _begin(L, empty._handle(), ia._handle())
    assert rv == 0 and R == 0
    assert L.kmg_segments_emit(st, o.ctypes.data) == 0 and L.kmg_segments_emit(st, None) == 0
    assert L.kmg_segments_free(st) == 0
    assert (o == -1).all()
    empty.free(); ia.free(); ic.free()


@pytest.mark.gpu
def test_c_abi_guards(kh):
    lib, L = _lib()
    ia, ib = kh.make_kmer_hash("ACGTACGTACGGTACCA", 5), kh.make_kmer_hash("TGGTACCGTACGTACGT", 5)
    a, b = ia._handle(), ib._handle()
    for rc in (0, 1):
        rv, st, R = _begin(L, a, b, rc=rc)
        assert rv == 0 and R > 0
        o = np.full(3 * R + 8, -1, np.int32)
        assert L.kmg_segments_emit_chunk(st, 0, R + 1, o.ctypes.data) == -1 and (o == -1).all()
        assert L.kmg_segments_emit(st, o.ctypes.data) == 0 and (o[3 * R:] == -1).all() and (o[:3 * R] != -1).all()
        assert L.kmg_segments_free(st) == 0
    assert _begin(L, None, b)[0] == -1 and _begin(L, a, None)[0] == -1 and _begin(L, None, None)[0] == -1
    assert L.kmg_join_segments_begin(a, b, 0, 0, 1, None, None) == -1
    assert _begin(L, a, b, rc=2)[0] == -1 and _begin(L, a, b, rc=-1)[0] == -1
    st, R = C.c_void_p(), C.c_uint64()
    assert L.kmg_join_segments_begin(a, b, 0, 0, 1, C.byref(st), None) == 0    # R may be NULL
    L.kmg_segments_free(st)
    ia.free(); ib.free()


@pytest.mark.gpu
def test_nothing_else_changes(kh):
    """No device memory is kept (after kmg_trim), a caller's device tensor is untouched, and both indexes read the same
    before and after."""
    import torch
    lib, L = _lib()
    k = 21
    s = random_dna(2_000_000, 11, p_n=0.001)
    q = random_dna(1_000_000, 12)
    q[:300_000] = s[500_000:800_000]
    ia, ib = kh.make_kmer_hash(s, k), kh.make_kmer_hash(q, k, do_sort=True)
    kh.kmer_pairs_segments(ia, ib)                              # warm: key table built
    before = [kh.kmer_pos(x, 2 | 8) for x in (ia, ib)]
    sentinel = torch.randint(-2**31, 2**31 - 1, (4 << 20,), dtype=torch.int32, device="cuda")
    sha = hashlib.sha256(sentinel.cpu().numpy().tobytes()).hexdigest()
    torch.cuda.synchronize()
    lib.check(L.kmg_trim())
    free0 = torch.cuda.mem_get_info()[0]
    for rc in (False, True):
        for mc in (0, 10):
            got = kh.kmer_pairs_segments(ia, ib, reverse_complement=rc, max_count=mc, min_rows=5)
            if not rc:                                          # the shared stretch, up to the first N of s in it
                assert got[0, :2].tolist() == [500_001, 1] and got[0, 2] > 100
    rv, st, R = _begin(L, ia._handle(), ib._handle())
    lib.check(rv)
    L.kmg_segments_free(st)                                     # freed without an emit
    lib.check(L.kmg_trim())
    assert torch.cuda.mem_get_info()[0] >= free0 - (2 << 20)
    assert hashlib.sha256(sentinel.cpu().numpy().tobytes()).hexdigest() == sha
    for x, b in zip((ia, ib), before):
        after = kh.kmer_pos(x, 2 | 8)
        assert np.array_equal(b["pos"], after["pos"]) and np.array_equal(b["count"], after["count"])
    ia.free(); ib.free()


@pytest.mark.gpu
def test_r_glue_join_segments(oracle):
    """.Call("kmer_pair_segments"): a 3 x R INTSXP matrix whose transpose (kmer.pairs.segments) equals the runs; argument
    guards; count tables refused; PROTECT balanced."""
    from rsession import RError, RSession
    R = RSession()
    k = 13
    s, q = _pair(k, 555)
    pa, pb = R.make_kmer_hash(s, k), R.make_kmer_hash(q, k)
    ea, eb = oracle.build(s, k).extract(2 | 8), oracle.build(q, k).extract(2 | 8)
    for rc in (0, 1):
        xa = rc_extraction(ea, k) if rc else ea
        for mc, mr in ((0, 1), (0, 12), (3, 0)):
            rows = join_rows(without_repeats(xa, mc), without_repeats(eb, mc))
            r = R.call("kmer_pair_segments", pa, pb, R.integer(rc, mc, mr))
            want = (anti_runs if rc else runs_of)(rows, mr)
            assert R.typeof(r) == INTSXP and R.dims(r) == (3, len(want))
            got = R.ints(r).reshape(-1, 3)                      # column-major 3 x R: t(m) has columns a, b, n
            R.stub.rstub_release(r)
            assert np.array_equal(got, want), (rc, mc, mr)
    with pytest.raises(RError, match="params should be an integer vector of length 3"):
        R.call("kmer_pair_segments", pa, pb, R.integer(0, 0))
    with pytest.raises(RError, match="rc should be TRUE or FALSE"):
        R.call("kmer_pair_segments", pa, pb, R.integer(2, 0, 1))
    with pytest.raises(RError, match="max.count should be 0"):
        R.call("kmer_pair_segments", pa, pb, R.integer(0, -1, 1))
    with pytest.raises(RError, match="min.rows should be 0 or positive"):
        R.call("kmer_pair_segments", pa, pb, R.integer(0, 0, -1))
    p11 = R.make_kmer_hash(s, 11)
    with pytest.raises(RError, match="kmer.pairs.segments failed: .*one k"):
        R.call("kmer_pair_segments", p11, pb, R.integer(1, 0, 1))
    ct = R.call("count_kmers", R.nil, R.integer(k, 0, 1), R.character(s))
    for x, y in ((ct, pb), (pa, ct)):
        with pytest.raises(RError, match="holds k-mer counts"):
            R.call("kmer_pair_segments", x, y, R.integer(0, 0, 1))
    assert R.stub.rstub_protect_depth() == 0
    for p in (pa, pb, p11, ct):
        R.stub.rstub_finalize(p)


def _c4():
    import torch
    from kmer_hasher_b200 import synth
    seq = synth.config_c3()
    q = synth.config_c4_query(seq, 100_000_000)
    return torch.from_numpy(seq).cuda(), torch.from_numpy(q).cuda()


@pytest.mark.gpu
def test_c4_full_size(kh):
    """The config-4 query built as a k = 32 index, joined with the config-3 index: equal to seq_kmer_segments on the device
    with x = i - k + 1; 22,878,529 runs holding 459,931,872 rows."""
    import torch
    dseq, dq = _c4()
    k = 32
    ic, iq = kh.make_kmer_hash(dseq, k), kh.make_kmer_hash(dq, k)
    del dseq
    R = 22_878_529
    want = kh.seq_kmer_segments(ic, dq, k, allow_k32=True, out=torch.empty((R, 3), dtype=torch.int32, device="cuda"))
    want[:, 0] -= k - 1
    got = kh.kmer_pairs_segments(iq, ic, out=torch.empty((R, 3), dtype=torch.int32, device="cuda"))
    assert int(got[:, 2].sum(dtype=torch.int64)) == 459_931_872
    assert torch.equal(got, want)
    ic.free(); iq.free()


@pytest.mark.gpu
def test_c5_self_join(kh):
    """The config-5 self join at k = 12: the n sum to the join's 2.98 * 10^9 rows, and the runs equal seq_kmer_segments of
    the sequence against its own index, shifted to x = i - k + 1."""
    import torch
    from kmer_hasher_b200 import synth
    lib, L = _lib()
    k = 12
    s5 = synth.config_c5()
    ds = torch.from_numpy(s5).cuda()
    ix = kh.make_kmer_hash(ds, k)
    st, M = C.c_void_p(), C.c_uint64()
    lib.check(L.kmg_join_begin(ix._handle(), ix._handle(), C.byref(st), C.byref(M)))
    L.kmg_join_free(st)
    M = M.value
    assert M > 2_900_000_000
    rv, sg, R = _begin(L, ix._handle(), ix._handle())
    lib.check(rv)
    try:
        got = torch.empty((R, 3), dtype=torch.int32, device="cuda")
        lib.check(L.kmg_segments_emit(sg, C.c_void_p(got.data_ptr())))
    finally:
        L.kmg_segments_free(sg)
    assert int(got[:, 2].sum(dtype=torch.int64)) == M
    want = kh.seq_kmer_segments(ix, ds, k, out=torch.empty((R, 3), dtype=torch.int32, device="cuda"))
    want[:, 0] -= k - 1
    assert torch.equal(got, want)
    ix.free()
