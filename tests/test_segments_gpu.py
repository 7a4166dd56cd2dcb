"""Match segments (kmg_segments_begin / emit / emit_chunk / free, seq_kmer_segments, .Call("sequence_kmer_segments")) against
the maximal diagonal runs of the oracle's rows.

`runs_of` restates a segment list from rows: sort the (i, j) rows by (i - j, i), split where the diagonal changes or i does
not step by 1, order the runs by (i, j) of their first row, keep those with n >= min_rows.  The rows come from the plain-C
oracle (`oracle.build(...).query(...)`) or, where max_count drops k-mers, from the row restatement of
test_extraction_chunks_gpu.py over an extraction without those k-mers.  At sizes where the oracle would be slow the rows
come from the library's own seq.kmer.pos on the device, and `runs_torch` restates the runs there.
"""
import ctypes as C
import hashlib

import numpy as np
import pytest

from conftest import random_dna
from test_dotplot_gpu import _pair, host_revcomp, without_repeats
from test_extraction_chunks_gpu import probe_rows

INT_MAX = 2**31 - 1
INTSXP = 13


def runs_of(rows, min_rows=1):
    """(R, 3) int64 (i, j, n): the maximal diagonal runs of the (i, j) rows, ordered by (i, j), n >= min_rows."""
    r = np.asarray(rows, np.int64).reshape(-1, 2)
    if len(r) == 0:
        return np.empty((0, 3), np.int64)
    i, j = r[:, 0], r[:, 1]
    o = np.lexsort((i, i - j))
    i, j = i[o], j[o]
    d = i - j
    head = np.ones(len(i), bool)
    head[1:] = (d[1:] != d[:-1]) | (i[1:] != i[:-1] + 1)
    at = np.flatnonzero(head)
    n = np.diff(np.append(at, len(i)))
    out = np.stack([i[at], j[at], n], 1)
    out = out[np.lexsort((out[:, 1], out[:, 0]))]
    return out[out[:, 2] >= max(min_rows, 1)]


def runs_torch(rows):
    """runs_of on the device: rows an (M, 2) int32 CUDA tensor; returns an (R, 3) int64 CUDA tensor."""
    import torch
    i = rows[:, 0].to(torch.int64)
    key = (i - rows[:, 1].to(torch.int64)) * 2**32 + i          # (diagonal, i): i < 2^31, so the order is that of the pair
    del i
    key = torch.sort(key).values
    d, i = key >> 32, key & 0xFFFFFFFF                          # the shift floors: d back for negative diagonals too
    del key
    head = torch.ones(len(d), dtype=torch.bool, device=d.device)
    head[1:] = (d[1:] != d[:-1]) | (i[1:] != i[:-1] + 1)
    at = torch.nonzero(head).flatten()
    del head
    n = torch.diff(torch.cat([at, torch.tensor([len(d)], device=d.device)]))
    i0, d0 = i[at], d[at]
    del d, i
    j0 = i0 - d0
    o = torch.sort(i0 * 2**32 + j0).indices
    return torch.stack([i0[o], j0[o], n[o]], 1)


def test_runs_of_by_hand():
    # one diagonal broken by a missing row; a crossing diagonal; a window with many j (a repeated k-mer)
    rows = [(5, 1), (6, 2), (8, 4), (9, 5), (10, 6),            # d = 4: runs (5,1,2) and (8,4,3)
            (6, 9), (7, 8), (8, 7),                             # anti-diagonal crossing it: three one-row runs
            (12, 3), (12, 20), (12, 40), (13, 21), (13, 41), (14, 42)]   # i = 12 with three j
    want = [(5, 1, 2), (6, 9, 1), (7, 8, 1), (8, 4, 3), (8, 7, 1), (12, 3, 1), (12, 20, 2), (12, 40, 3)]
    got = runs_of(rows)
    assert got.tolist() == [list(w) for w in want]
    assert got[:, 2].sum() == len(rows)
    assert runs_of(rows, 2).tolist() == [[5, 1, 2], [8, 4, 3], [12, 20, 2], [12, 40, 3]]
    assert runs_of(rows, 3).tolist() == [[8, 4, 3], [12, 40, 3]]
    assert runs_of(rows, 0).tolist() == got.tolist()
    assert runs_of(np.empty((0, 2), np.int32)).shape == (0, 3)
    assert runs_of([(3, 3)]).tolist() == [[3, 3, 1]]
    # order by (i, j) of the first row, not by diagonal; rows given in any order
    shuffled = np.array(rows)[np.random.default_rng(1).permutation(len(rows))]
    assert runs_of(shuffled).tolist() == got.tolist()


def test_python_guards_on_cpu():
    """The Python entry checks its arguments before the handle is used (these handles were never made)."""
    import kmer_hasher_b200 as kh
    ix = kh.KmerHash(None, 5)
    with pytest.raises(TypeError, match="external pointer"):
        kh.seq_kmer_segments("not a pointer", "ACGTACGT", 5)
    with pytest.raises(ValueError, match="count.kmers"):
        kh.seq_kmer_segments(kh.KmerCounts(None, 5, 2), "ACGTACGT", 5)
    with pytest.raises(ValueError, match="longer than k"):
        kh.seq_kmer_segments(ix, "ACGTA", 5)
    with pytest.raises(ValueError, match="longer than k"):
        kh.seq_kmer_segments(ix, "A" * 40, 32)
    with pytest.raises(ValueError, match="single sequence"):
        kh.seq_kmer_segments(ix, ["ACGTACGT", "ACGTACGT"], 5)
    for bad in (-1, 2**32):
        with pytest.raises(ValueError, match="max_count"):
            kh.seq_kmer_segments(ix, "ACGTACGT", 5, max_count=bad)
        with pytest.raises(ValueError, match="min_rows"):
            kh.seq_kmer_segments(ix, "ACGTACGT", 5, min_rows=bad)
    with pytest.raises(ValueError, match="cleared"):
        kh.seq_kmer_segments(ix, "ACGTACGT", 5)


def test_glue_registration_and_argument_errors_on_cpu():
    from rsession import RError, RSession
    R = RSession()
    with pytest.raises(RError, match="Incorrect number of arguments"):
        R.call("sequence_kmer_segments", R.integer(1), R.character("ACGT"), R.integer(2))
    with pytest.raises(RError, match="ptr_r should be an external pointer"):
        R.call("sequence_kmer_segments", R.integer(1), R.character("ACGT"), R.integer(2), R.integer(0, 0, 1))
    assert R.stub.rstub_protect_depth() == 0


# ---- on the GPU ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def kh():
    import kmer_hasher_b200 as kh
    return kh


def _lib():
    from kmer_hasher_b200 import _lib as lib
    return lib, lib.load()


def _begin(L, h, q, k, rc=0, mc=0, mr=1, qlen=None):
    """kmg_segments_begin -> (return code, handle, R)"""
    st, R = C.c_void_p(), C.c_uint64()
    rv = L.kmg_segments_begin(h, q, len(q) if qlen is None else qlen, k, rc, mc, mr, C.byref(st), C.byref(R))
    return rv, st, R.value


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 5, 8, 11, 16, 21, 27, 31, 32])
def test_segments_match_oracle_runs(kh, oracle, k):
    """N runs, lower case, IUPAC bytes, a shared stretch, a reverse-complemented one and an internal repeat (_pair); both
    strands, sorted and grouped indexes, min_rows 1 and a filter."""
    s, q = _pair(k, 2000 + k)
    o = oracle.build(s, k)
    for rc in (False, True):
        rows = o.query(host_revcomp(q) if rc else q, k)
        want = runs_of(rows)
        assert len(want) > 0 and want[:, 2].sum() * 2 == len(rows)
        assert want[:, 2].max() > 20                             # the shared stretches give long runs
        for do_sort in (True, False):
            ix = kh.make_kmer_hash(s, k, do_sort=do_sort)
            got = kh.seq_kmer_segments(ix, q, k, reverse_complement=rc, allow_k32=True)
            assert got.dtype == np.int32 and got.shape == want.shape
            assert np.array_equal(got, want), (rc, do_sort)
            for mr in (0, 3, 20):
                got = kh.seq_kmer_segments(ix, q, k, reverse_complement=rc, min_rows=mr, allow_k32=True)
                assert np.array_equal(got, runs_of(rows, mr)), (rc, do_sort, mr)
            ix.free()


@pytest.mark.gpu
def test_bases_of_a_run(kh, oracle):
    """With the index's k, a run of n rows means query bases [i-k+1, i+n-1] equal index bases [j, j+n+k-2] (2-bit code)."""
    k = 13
    s, q = _pair(k, 91)
    ix = kh.make_kmer_hash(s, k)
    got = kh.seq_kmer_segments(ix, q, k, min_rows=10)
    assert len(got) > 0
    code = lambda b: (np.asarray(b, np.uint8) >> 1) & 3
    for i, j, n in got[:200]:
        assert np.array_equal(code(q[i - k:i + n - 1]), code(s[j - 1:j + n + k - 2])), (i, j, n)
    ix.free()


@pytest.mark.gpu
def test_max_count(kh, oracle):
    """max_count equals the runs of the oracle's rows without the over-long k-mers (the repeats of test_dotplot_gpu's
    max_count test: 400 bases six times, 100 bases three times), with and without min_rows."""
    k = 11
    s, q = _pair(k, 77)
    s = s.copy()
    for at in (12_000, 13_000, 14_000, 15_000, 16_000):
        s[at:at + 400] = s[7_000:7_400]
    for at in (18_000, 18_500):
        s[at:at + 100] = s[8_000:8_100]
    o = oracle.build(s, k)
    e = o.extract(2 | 8)
    longest = int(e["count"].max())
    assert longest >= 6
    for rc in (False, True):
        qq = host_revcomp(q) if rc else q
        qk, qs = oracle.windows(qq, k)
        for do_sort in (True, False):
            ix = kh.make_kmer_hash(s, k, do_sort=do_sort)
            sizes = []
            for mc in (1, 2, 3, longest - 1, longest, 2**32 - 1):
                rows = probe_rows(without_repeats(e, mc), qk, qs, k)
                for mr in (1, 15):
                    got = kh.seq_kmer_segments(ix, q, k, reverse_complement=rc, max_count=mc, min_rows=mr)
                    assert np.array_equal(got, runs_of(rows, mr)), (rc, do_sort, mc, mr)
                sizes.append(len(rows))
            if not rc:                                          # the repeated stretches are shared forward
                assert sizes[0] < sizes[2] < sizes[3] < sizes[4]
            ix.free()


@pytest.mark.gpu
@pytest.mark.parametrize("mc", [0, 3])
def test_row_totals(kh, mc):
    """With min_rows <= 1 the n of all runs sum to M of the probe, and to the total of seq_kmer_dotplot over full windows
    with the same max_count."""
    lib, L = _lib()
    k = 15
    s, q = _pair(k, 5)
    s = np.concatenate([s, s[:5_000], s[2_000:4_000]])        # repeated stretches: lists of 2 and 3 positions
    ix = kh.make_kmer_hash(s, k)
    for rc in (0, 1):
        got = kh.seq_kmer_segments(ix, q, k, reverse_complement=rc, max_count=mc, min_rows=0)
        total = kh.seq_kmer_dotplot(ix, q, k, y_range=(0, 2**31), x_range=(0, 2**31), bins=(1, 1), reverse_complement=rc,
                                    max_count=mc)[0, 0]
        assert got[:, 2].astype(np.int64).sum() == total
        if mc == 0:
            st, M = C.c_void_p(), C.c_uint64()
            begin = L.kmg_query_begin_rc if rc else L.kmg_query_begin
            lib.check(begin(ix._handle(), bytes(q), len(q), k, C.byref(st), C.byref(M)))
            L.kmg_query_free(st)
            assert got[:, 2].astype(np.int64).sum() == M.value
    ix.free()


@pytest.mark.gpu
def test_test_fa_self(kh, oracle, test_fa):
    """test.fa against itself at k = 16: the top k-mer has 2,188 positions (telomeric repeats), ~29 M rows."""
    k = 16
    ix = kh.make_kmer_hash(test_fa, k)
    rows = oracle.build(test_fa, k).query(test_fa, k)
    assert len(rows) // 2 > 25_000_000
    want = runs_of(rows)
    got = kh.seq_kmer_segments(ix, test_fa, k)
    assert np.array_equal(got, want)
    assert (want[:, 0] == want[:, 1] + k - 1).sum() >= 1 and want[:, 2].max() >= len(test_fa) // 100
    got = kh.seq_kmer_segments(ix, test_fa, k, min_rows=25)
    assert np.array_equal(got, runs_of(rows, 25))
    ix.free()


@pytest.mark.gpu
def test_more_than_2_31_rows(kh, oracle):
    """A 50,000-base homopolymer against itself: (n - k + 1)^2 ~ 2.5 * 10^9 rows over several 2^30-row slices.  Query ends
    I and index positions J are contiguous ranges, so each diagonal d holds one run, from i = max(I0, J0 + d) to
    min(I1, J1 + d)."""
    lib, L = _lib()
    k, n = 16, 50_000
    s = "A" * n
    ix = kh.make_kmer_hash(s, k, do_sort=True)
    _, N = ix.sizes_un
    qk, qs = oracle.windows(s, k)
    I = (qs + k - 1).astype(np.int64)
    J = oracle.build(s, k).extract(2)["pos"].reshape(-1, 2)[:, 1].astype(np.int64)
    assert len(J) == N and len(I) * N > 2**31
    assert np.array_equal(I, np.arange(I[0], I[-1] + 1)) and np.array_equal(J, np.arange(J[0], J[-1] + 1))
    d = np.arange(I[0] - J[-1], I[-1] - J[0] + 1)
    i0 = np.maximum(I[0], J[0] + d)
    i1 = np.minimum(I[-1], J[-1] + d)
    want = np.stack([i0, i0 - d, i1 - i0 + 1], 1)
    want = want[np.lexsort((want[:, 1], want[:, 0]))]
    assert want[:, 2].sum() == len(I) * N
    got = kh.seq_kmer_segments(ix, s, k)
    assert np.array_equal(got, want)
    assert np.array_equal(kh.seq_kmer_segments(ix, s, k, min_rows=40_000), want[want[:, 2] >= 40_000])
    assert len(kh.seq_kmer_segments(ix, s, k, max_count=N - 1)) == 0
    ix.free()


@pytest.mark.gpu
def test_output_memory_kinds_and_chunks(kh):
    """A random 30 Mbp self query at k = 12: ~40 M runs, mostly of one row (480 MB).  The same bytes into a device tensor,
    pinned memory (2 chunks) and pageable memory (the staged path, 7 or more chunks), guard bytes untouched; emit_chunk windows
    agree with the full emit; the device result equals the runs of the library's own seq.kmer.pos rows."""
    import torch
    lib, L = _lib()
    k, n, G = 12, 30_000_000, 16
    s = random_dna(n, 4242)
    ix = kh.make_kmer_hash(s, k)
    rv, st, R = _begin(L, ix._handle(), s.tobytes(), k)
    lib.check(rv)
    try:
        pin_rows, stage_rows = (256 << 20) // 12, (64 << 20) // 12     # rows per pinned / staged chunk
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
    rows = torch.from_numpy(kh.seq_kmer_pos(ix, s, k)).cuda()
    want = runs_torch(rows)
    del rows
    assert want.shape[0] == R
    assert torch.equal(torch.from_numpy(runs).cuda().to(torch.int64), want)
    ix.free()


@pytest.mark.gpu
def test_empty_cases(kh):
    lib, L = _lib()
    ix = kh.make_kmer_hash("N" * 50, 5)                        # U = 0
    assert ix.sizes_un == (0, 0)
    assert kh.seq_kmer_segments(ix, "ACGTACGTAC", 5).shape == (0, 3)
    ix2 = kh.make_kmer_hash("ACGTACGTACGGT", 5)
    assert kh.seq_kmer_segments(ix2, "NNNNNNNN", 5).shape == (0, 3)        # no windows
    assert kh.seq_kmer_segments(ix2, "TTTTTTTTTT", 5).shape == (0, 3)      # nothing shared
    assert kh.seq_kmer_segments(ix2, "ACGTACGTACGGT", 5, min_rows=100).shape == (0, 3)   # every run filtered out
    o = np.full(6, -1, np.int32)
    for q in (b"ACGT", b""):                                    # qlen < k
        rv, st, R = _begin(L, ix2._handle(), q, 5)
        assert rv == 0 and R == 0
        assert L.kmg_segments_emit(st, o.ctypes.data) == 0 and L.kmg_segments_emit(st, None) == 0
        assert L.kmg_segments_free(st) == 0
    assert (o == -1).all()
    ix.free(); ix2.free()


@pytest.mark.gpu
def test_c_abi_guards(kh):
    lib, L = _lib()
    ix = kh.make_kmer_hash("ACGTACGTACGGTACCA", 5)
    h = ix._handle()
    q = b"ACGTACGTAC"
    rv, st, R = _begin(L, h, q, 5)
    assert rv == 0 and R > 0
    o = np.full(3 * R + 8, -1, np.int32)
    p = o.ctypes.data
    assert L.kmg_segments_emit(None, p) == -1
    assert L.kmg_segments_emit(st, None) == -1
    assert L.kmg_segments_emit_chunk(st, 0, R + 1, p) == -1
    assert L.kmg_segments_emit_chunk(st, R + 1, 0, p) == -1
    assert L.kmg_segments_emit_chunk(st, 1, R, p) == -1
    assert L.kmg_segments_emit_chunk(None, 0, 1, p) == -1
    assert (o == -1).all()
    assert L.kmg_segments_emit_chunk(st, R, 0, p) == 0
    assert L.kmg_segments_emit(st, p) == 0 and (o[3 * R:] == -1).all() and (o[:3 * R] != -1).all()
    assert L.kmg_segments_free(st) == 0
    assert L.kmg_segments_free(None) == 0
    assert _begin(L, None, q, 5)[0] == -1
    assert L.kmg_segments_begin(h, q, len(q), 5, 0, 0, 1, None, None) == -1
    assert _begin(L, h, q, 0)[0] == -2 and _begin(L, h, q, 33)[0] == -2
    assert _begin(L, h, q, 5, rc=2)[0] == -1 and _begin(L, h, q, 5, rc=-1)[0] == -1
    assert _begin(L, h, q, 5, qlen=2**31 - 1)[0] == -3
    assert _begin(L, h, None, 5, qlen=10)[0] == -1
    ix.free()


@pytest.mark.gpu
def test_nothing_else_changes(kh):
    """No device memory is kept (after kmg_trim), a caller's device tensor is untouched, and the index reads the same
    before and after."""
    import torch
    lib, L = _lib()
    k = 21
    s = random_dna(2_000_000, 11, p_n=0.001)
    q = random_dna(1_000_000, 12)
    q[:300_000] = s[500_000:800_000]
    ix = kh.make_kmer_hash(s, k)
    kh.seq_kmer_segments(ix, q, k)                              # warm: key table built
    before = kh.kmer_pos(ix, 2 | 8)
    sentinel = torch.randint(-2**31, 2**31 - 1, (4 << 20,), dtype=torch.int32, device="cuda")
    sha = hashlib.sha256(sentinel.cpu().numpy().tobytes()).hexdigest()
    torch.cuda.synchronize()
    lib.check(L.kmg_trim())
    free0 = torch.cuda.mem_get_info()[0]
    for rc in (False, True):
        for mc in (0, 10):
            got = kh.seq_kmer_segments(ix, q, k, reverse_complement=rc, max_count=mc, min_rows=5)
            if not rc:                                          # the shared stretch, up to the index's first N in it
                assert got[0, :2].tolist() == [k, 500_001] and got[0, 2] > 100
    rv, st, R = _begin(L, ix._handle(), bytes(q), k)
    lib.check(rv)
    L.kmg_segments_free(st)                                     # freed without an emit
    lib.check(L.kmg_trim())
    assert torch.cuda.mem_get_info()[0] >= free0 - (2 << 20)
    assert hashlib.sha256(sentinel.cpu().numpy().tobytes()).hexdigest() == sha
    after = kh.kmer_pos(ix, 2 | 8)
    assert np.array_equal(before["pos"], after["pos"]) and np.array_equal(before["count"], after["count"])
    ix.free()


@pytest.mark.gpu
def test_r_glue_segments(oracle):
    """.Call("sequence_kmer_segments"): a 3 x R INTSXP matrix equal to the runs of the oracle's rows; the guards of
    seq.kmer.pos; count tables refused."""
    from rsession import RError, RSession
    R = RSession()
    k = 13
    s, q = _pair(k, 555)
    ix = R.make_kmer_hash(s, k)
    o = oracle.build(s, k)
    e = o.extract(2 | 8)
    for rc in (0, 1):
        qq = host_revcomp(q) if rc else q
        for mc, mr in ((0, 1), (0, 12), (3, 0)):
            rows = o.query(qq, k) if mc == 0 else probe_rows(without_repeats(e, mc), *oracle.windows(qq, k), k)
            r = R.call("sequence_kmer_segments", ix, R.character(q), R.integer(k), R.integer(rc, mc, mr))
            want = runs_of(rows, mr)
            assert R.typeof(r) == INTSXP and R.dims(r) == (3, len(want))
            got = R.ints(r).reshape(-1, 3)
            R.stub.rstub_release(r)
            assert np.array_equal(got, want), (rc, mc, mr)
    with pytest.raises(RError, match="the sequence should be longer than k and k should not be longer than 31"):
        R.call("sequence_kmer_segments", ix, R.character(q), R.integer(32), R.integer(0, 0, 1))
    with pytest.raises(RError, match="the sequence should be longer than k"):
        R.call("sequence_kmer_segments", ix, R.character("ACGT"), R.integer(k), R.integer(0, 0, 1))
    with pytest.raises(RError, match="single sequence"):
        R.call("sequence_kmer_segments", ix, R.character(q, q), R.integer(k), R.integer(0, 0, 1))
    with pytest.raises(RError, match="params should be an integer vector of length 3"):
        R.call("sequence_kmer_segments", ix, R.character(q), R.integer(k), R.integer(0, 0))
    with pytest.raises(RError, match="rc should be TRUE or FALSE"):
        R.call("sequence_kmer_segments", ix, R.character(q), R.integer(k), R.integer(2, 0, 1))
    with pytest.raises(RError, match="max.count should be 0"):
        R.call("sequence_kmer_segments", ix, R.character(q), R.integer(k), R.integer(0, -1, 1))
    with pytest.raises(RError, match="min.rows should be 0 or positive"):
        R.call("sequence_kmer_segments", ix, R.character(q), R.integer(k), R.integer(0, 0, -1))
    ct = R.call("count_kmers", R.nil, R.integer(k, 0, 1), R.character(s))
    with pytest.raises(RError, match="holds k-mer counts"):
        R.call("sequence_kmer_segments", ct, R.character(q), R.integer(k), R.integer(0, 0, 1))
    assert R.stub.rstub_protect_depth() == 0
    for p in (ix, ct):
        R.stub.rstub_finalize(p)


@pytest.mark.gpu
def test_c4_full_size(kh):
    """Config 4: the 100 Mbp query against the 250 Mbp config-3 index at k = 32.  The forward segments equal the runs of
    the 459,931,872 rows kmg_query_emit writes to device memory, restated on the device; their n sum to that count."""
    import torch
    from kmer_hasher_b200 import synth
    lib, L = _lib()
    seq = synth.config_c3()
    q = synth.config_c4_query(seq, 100_000_000)
    dseq, dq = torch.from_numpy(seq).cuda(), torch.from_numpy(q).cuda()
    del seq
    k = 32
    ix = kh.make_kmer_hash(dseq, k)
    del dseq
    st, M = C.c_void_p(), C.c_uint64()
    lib.check(L.kmg_query_begin(ix._handle(), C.c_void_p(dq.data_ptr()), len(q), k, C.byref(st), C.byref(M)))
    M = M.value
    assert M == 459_931_872
    rows = torch.empty((M, 2), dtype=torch.int32, device="cuda")
    try:
        lib.check(L.kmg_query_emit(st, C.c_void_p(rows.data_ptr())))
    finally:
        L.kmg_query_free(st)
    want = runs_torch(rows)
    del rows
    torch.cuda.empty_cache()
    rv, sg, R = _begin(L, ix._handle(), C.c_void_p(dq.data_ptr()), k, qlen=len(q))
    lib.check(rv)
    try:
        got = torch.empty((R, 3), dtype=torch.int32, device="cuda")
        lib.check(L.kmg_segments_emit(sg, C.c_void_p(got.data_ptr())))
    finally:
        L.kmg_segments_free(sg)
    assert R == want.shape[0] and int(got[:, 2].sum(dtype=torch.int64)) == M
    assert torch.equal(got.to(torch.int64), want)
    long_ = kh.seq_kmer_segments(ix, dq, k, min_rows=20, allow_k32=True, out=torch.empty((R, 3), dtype=torch.int32, device="cuda"))
    keep = want[:, 2] >= 20
    assert torch.equal(long_[:int(keep.sum())].to(torch.int64), want[keep])
    ix.free()
