"""Dot plots (kmg_query_dotplot / kmg_join_dotplot, seq_kmer_dotplot / kmer_pairs_dotplot, .Call("sequence_kmer_dotplot")
and .Call("kmer_pair_dotplot")) against integer binning of the oracle's rows.

A dot plot is the 2-D histogram of the rows seq.kmer.pos or kmer.pairs returns.  `bin_rows` restates it with np.bincount on
bx + by * nx; the rows come from the plain-C oracle (`oracle.build(...).query(...)`, `oracle.pairs_join`) or, where a
max_count drops k-mers, from the row restatements of test_extraction_chunks_gpu.py over an extraction without those
k-mers.  Reverse-complement queries are complemented on the host (IUPAC, case kept).
"""
import ctypes as C
import hashlib

import numpy as np
import pytest

import oracle as oracle_mod
from conftest import random_dna
from test_extraction_chunks_gpu import join_rows, probe_rows

INT_MAX = 2**31 - 1
TOP = 2**31
REALSXP = 14
IUPAC = bytes.maketrans(b"ACGTRYKMBVDHacgtrykmbvdh", b"TGCAYRMKVBHDtgcayrmkvbhd")


def bin_rows(rows, xr, yr, nx, ny):
    """Column-major nx * ny float64 histogram of (x, y) rows over the half-open windows xr, yr (exact integer bins)."""
    rows = np.asarray(rows, np.int64).reshape(-1, 2)
    x, y = rows[:, 0], rows[:, 1]
    (x0, x1), (y0, y1) = xr, yr
    keep = (x >= x0) & (x < x1) & (y >= y0) & (y < y1)
    bx = (x[keep] - x0) * nx // (x1 - x0)
    by = (y[keep] - y0) * ny // (y1 - y0)
    return np.bincount(bx + by * nx, minlength=nx * ny).astype(np.float64)


def host_revcomp(q):
    b = q.encode("latin-1") if isinstance(q, str) else (q.tobytes() if isinstance(q, np.ndarray) else bytes(q))
    return b[::-1].translate(IUPAC)


def without_repeats(e, max_count):
    """The extraction `e` (extract(2 | 8)) without the k-mers that have more than max_count positions (0: unchanged)."""
    if not max_count:
        return e
    cnt = e["count"].astype(np.int64)
    keep = cnt <= max_count
    pos = e["pos"].reshape(-1, 2)[np.repeat(keep, cnt)]
    return dict(keys=e["keys"][keep], count=e["count"][keep], pos=pos.ravel())


def test_bin_rows_by_hand():
    rows = [(1, 1), (2, 5), (3, 9), (9, 9), (10, 1), (0, 4), (4, 10)]
    # x window [1, 10) in 4 bins: 9 coordinates, bins {1,2,3}, {4,5}, {6,7}, {8,9} -> floor((x-1)*4/9)
    # y window [1, 10) in 2 bins: {1..5}, {6..9}; x = 10, x = 0 and y = 10 fall outside
    img = bin_rows(rows, (1, 10), (1, 10), 4, 2).reshape(2, 4)      # [by, bx]
    assert img.tolist() == [[2, 0, 0, 0], [1, 0, 0, 1]]
    assert bin_rows(rows, (0, TOP), (0, TOP), 1, 1).tolist() == [7]
    assert bin_rows(rows, (5, 8), (0, 3), 3, 3).tolist() == [0] * 9   # a window that holds no row
    assert bin_rows(np.empty((0, 2), np.int32), (0, 5), (0, 5), 2, 3).tolist() == [0] * 6
    # more bins than coordinates: x in [2, 4) over 5 bins -> x = 2 to bin 0, x = 3 to bin floor(5/2) = 2
    assert bin_rows([(2, 0), (3, 0)], (2, 4), (0, 1), 5, 1).tolist() == [1, 0, 1, 0, 0]
    assert host_revcomp("ACgtRYKMBDHVNnS-") == b"-SnNBDHVKMRYacGT"


def test_python_guards_on_cpu():
    """The Python entries check their arguments before the handle is used (these handles were never made)."""
    import kmer_hasher_b200 as kh
    ix = kh.KmerHash(None, 5)
    ok = dict(y_range=(1, 100))
    with pytest.raises(TypeError, match="external pointer"):
        kh.seq_kmer_dotplot("not a pointer", "ACGTACGT", 5, **ok)
    with pytest.raises(ValueError, match="count.kmers"):
        kh.seq_kmer_dotplot(kh.KmerCounts(None, 5, 2), "ACGTACGT", 5, **ok)
    with pytest.raises(ValueError, match="longer than k"):
        kh.seq_kmer_dotplot(ix, "ACGTA", 5, **ok)
    with pytest.raises(ValueError, match="longer than k"):
        kh.seq_kmer_dotplot(ix, "A" * 40, 32, **ok)
    with pytest.raises(ValueError, match="bins must be positive"):
        kh.seq_kmer_dotplot(ix, "ACGTACGT", 5, bins=(0, 3), **ok)
    with pytest.raises(OverflowError, match="2\\^31 - 1 cells"):
        kh.seq_kmer_dotplot(ix, "ACGTACGT", 5, bins=(65536, 32768), **ok)
    for bad in ((5, 5), (-1, 3), (0, TOP + 1)):
        with pytest.raises(ValueError, match="y range"):
            kh.seq_kmer_dotplot(ix, "ACGTACGT", 5, y_range=bad)
        with pytest.raises(ValueError, match="x range"):
            kh.seq_kmer_dotplot(ix, "ACGTACGT", 5, x_range=bad, **ok)
        with pytest.raises(ValueError, match="x range"):
            kh.kmer_pairs_dotplot(ix, ix, a_range=bad, b_range=(0, 9))
    with pytest.raises(ValueError, match="max_count"):
        kh.seq_kmer_dotplot(ix, "ACGTACGT", 5, max_count=-1, **ok)
    with pytest.raises(ValueError, match="max_count"):
        kh.kmer_pairs_dotplot(ix, ix, a_range=(0, 9), b_range=(0, 9), max_count=2**32)
    with pytest.raises(ValueError, match="out holds 48 bytes; the image needs 64"):
        kh.seq_kmer_dotplot(ix, "ACGTACGT", 5, bins=(2, 4), out=np.empty(6), **ok)
    with pytest.raises(ValueError, match="cleared"):
        kh.seq_kmer_dotplot(ix, "ACGTACGT", 5, bins=(2, 4), x_range=(0, TOP), y_range=(0, TOP))
    with pytest.raises(ValueError, match="cleared"):
        kh.kmer_pairs_dotplot(ix, ix, a_range=(0, 9), b_range=(0, 9))


def test_glue_registration_and_argument_errors_on_cpu():
    from rsession import RError, RSession
    R = RSession()
    with pytest.raises(RError, match="Incorrect number of arguments"):
        R.call("sequence_kmer_dotplot", R.integer(1), R.character("ACGT"), R.integer(2))
    with pytest.raises(RError, match="Incorrect number of arguments"):
        R.call("kmer_pair_dotplot", R.integer(1), R.integer(1))
    with pytest.raises(RError, match="ptr_r should be an external pointer"):
        R.call("sequence_kmer_dotplot", R.integer(1), R.character("ACGT"), R.integer(2), R.integer(0, 5, 1, 0, 5, 1, 0, 0))
    with pytest.raises(RError, match="ptr_r should be an external pointer"):
        R.call("kmer_pair_dotplot", R.integer(1), R.integer(1), R.integer(0, 5, 1, 0, 5, 1, 0))
    assert R.stub.rstub_protect_depth() == 0


# ---- on the GPU ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def kh():
    import kmer_hasher_b200 as kh
    return kh


def _lib():
    from kmer_hasher_b200 import _lib as lib
    return lib, lib.load()


def _pair(k, seed):
    """(index sequence, query): random, with N runs, lower case and IUPAC bytes; the query shares two stretches of the index
    (one of them reverse-complemented) and repeats one of its own."""
    n = 3_000 if k < 8 else 20_000
    s = random_dna(n, seed, p_n=0.002, p_lower=0.2, p_other=0.005, n_runs=2)
    q = random_dna(n // 2, seed + 1, p_n=0.002, p_lower=0.2, p_other=0.005, n_runs=1)
    q[100:100 + n // 5] = s[n // 3:n // 3 + n // 5]
    q[len(q) - n // 6:] = np.frombuffer(host_revcomp(s[n // 2:n // 2 + n // 6]), np.uint8)
    q[n // 4:n // 4 + 200] = q[100:300]
    return s, q


def _grids(ls, lq):
    """(x window, y window, nx, ny): the full plot, a ragged grid, a zoom that cuts rows on all four sides."""
    return [((1, lq + 1), (1, ls + 1), 40, 30),
            ((0, TOP), (0, TOP), 7, 3),
            ((lq // 7, lq // 7 + 1_013), (ls // 5, ls // 5 + 2_011), 17, 23)]


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 5, 11, 16, 21, 31, 32])
def test_query_dotplot_matches_binned_oracle_rows(kh, oracle, k):
    s, q = _pair(k, 1000 + k)
    o = oracle.build(s, k)
    for rc in (False, True):
        qq = host_revcomp(q) if rc else q
        rows = o.query(qq, k)
        assert len(rows) > 0
        for do_sort in (True, False):
            ix = kh.make_kmer_hash(s, k, do_sort=do_sort)
            for xr, yr, nx, ny in _grids(len(s), len(q)):
                got = kh.seq_kmer_dotplot(ix, q, k, x_range=xr, y_range=yr, bins=(nx, ny), reverse_complement=rc,
                                          allow_k32=True)
                assert got.shape == (nx, ny) and got.flags.f_contiguous
                assert np.array_equal(got.ravel(order="F"), bin_rows(rows, xr, yr, nx, ny)), (rc, do_sort, xr, nx)
            ix.free()


@pytest.fixture(scope="module")
def k11(oracle):
    k = 11
    s, q = _pair(k, 77)
    o = oracle.build(s, k)
    return k, s, q, o.query(q, k), o.extract(2 | 8)


@pytest.mark.gpu
def test_grids(kh, k11):
    """1 x 1; more bins than coordinates (empty bins); ranges that are not multiples of the bin count; zooms cutting rows
    at every edge; windows that hold no row; the window's end at 2^31."""
    k, s, q, rows, _ = k11
    r = rows.reshape(-1, 2)
    ix = kh.make_kmer_hash(s, k)
    xmid, ymid = int(np.median(r[:, 0])), int(np.median(r[:, 1]))
    cases = [((1, len(q) + 1), (1, len(s) + 1), 1, 1),
             ((xmid, xmid + 50), (ymid, ymid + 40), 150, 97),       # more bins than coordinates
             ((1, 10_008), (3, 20_004), 97, 89),
             ((0, 9_973), (1, 19_997), 1_000, 3),
             ((xmid - 777, xmid + 1_001), (ymid - 1_234, ymid + 999), 13, 11),
             ((len(q) + 1, len(q) + 5_000), (1, len(s) + 1), 10, 10),  # no row
             ((1, len(q) + 1), (len(s) + 1, TOP), 10, 10),            # no row
             ((TOP - 1, TOP), (0, TOP), 2, 2),                          # no row, the last coordinate
             ((0, TOP), (0, TOP), 1_000, 1_000)]
    for xr, yr, nx, ny in cases:
        want = bin_rows(r, xr, yr, nx, ny)
        got = kh.seq_kmer_dotplot(ix, q, k, x_range=xr, y_range=yr, bins=(nx, ny))
        assert np.array_equal(got.ravel(order="F"), want), (xr, yr, nx, ny)
    inside = bin_rows(r, cases[4][0], cases[4][1], 1, 1)[0]
    assert 0 < inside < len(r)                                     # the zoom did cut rows
    assert (bin_rows(r, *cases[1]) == 0).any()                     # and the fine grid has empty bins
    assert kh.seq_kmer_dotplot(ix, q, k, y_range=(1, len(s) + 1), bins=(1, 1))[0, 0] == len(r)
    ix.free()


@pytest.mark.gpu
def test_max_count(kh, oracle, k11):
    """max_count equals the oracle's rows without the over-long k-mers.  The index repeats two stretches the query shares
    (400 bases six times, 100 bases three times), so its lists are long enough for every limit below to drop rows."""
    k, s, q, _, _ = k11
    s = s.copy()
    for at in (12_000, 13_000, 14_000, 15_000, 16_000):
        s[at:at + 400] = s[7_000:7_400]
    for at in (18_000, 18_500):
        s[at:at + 100] = s[8_000:8_100]
    o = oracle.build(s, k)
    rows, e = o.query(q, k), o.extract(2 | 8)
    qk, qs = oracle.windows(q, k)
    ix = kh.make_kmer_hash(s, k, do_sort=True)
    full = ((1, len(q) + 1), (1, len(s) + 1), 64, 48)
    longest = int(e["count"].max())
    assert longest >= 6
    assert np.array_equal(probe_rows(e, qk, qs, k).ravel(), rows)
    sizes = []
    for mc in (1, 2, 3, longest - 1, longest, longest + 1, 2**32 - 1):
        want_rows = probe_rows(without_repeats(e, mc), qk, qs, k)
        got = kh.seq_kmer_dotplot(ix, q, k, x_range=full[0], y_range=full[1], bins=full[2:], max_count=mc)
        assert np.array_equal(got.ravel(order="F"), bin_rows(want_rows, *full)), mc
        assert got.sum() == len(want_rows)
        sizes.append(len(want_rows))
        if mc >= longest:
            assert len(want_rows) * 2 == len(rows)
    assert sizes[0] < sizes[2] < sizes[3] < sizes[4]                    # the limits below the longest list drop rows
    one = kh.seq_kmer_dotplot(ix, q, k, y_range=(1, len(s) + 1), bins=(1, 1), max_count=1)[0, 0]
    assert one == sizes[0] < len(rows) // 2
    ix.free()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [5, 13, 21])
def test_join_dotplot(kh, oracle, k):
    """Two different indexes and an index with itself, with and without max_count."""
    s, q = _pair(k, 300 + k)
    q = q.copy()
    oa, ob = oracle.build(s, k), oracle.build(q, k)
    ea, eb = oa.extract(2 | 8), ob.extract(2 | 8)
    ia, ib = kh.make_kmer_hash(s, k, do_sort=True), kh.make_kmer_hash(q, k)
    for (pa, pb), (xa, xb), (la, lb) in (((ia, ib), (ea, eb), (len(s), len(q))), ((ia, ia), (ea, ea), (len(s), len(s))),
                                         ((ib, ib), (eb, eb), (len(q), len(q)))):
        rows = oracle_mod.pairs_join(xa, xb)
        assert len(rows) > 0
        for xr, yr, nx, ny in [((1, la + 1), (1, lb + 1), 50, 31), ((la // 3, la // 3 + 997), (0, TOP), 9, 4)]:
            got = kh.kmer_pairs_dotplot(pa, pb, a_range=xr, b_range=yr, bins=(nx, ny))
            assert np.array_equal(got.ravel(order="F"), bin_rows(rows, xr, yr, nx, ny))
            for mc in (1, 2, 5):
                want = join_rows(without_repeats(xa, mc), without_repeats(xb, mc))
                got = kh.kmer_pairs_dotplot(pa, pb, a_range=xr, b_range=yr, bins=(nx, ny), max_count=mc)
                assert np.array_equal(got.ravel(order="F"), bin_rows(want, xr, yr, nx, ny)), mc
    ia.free(); ib.free()


@pytest.mark.gpu
def test_load_balance_test_fa(kh, oracle, test_fa):
    """test.fa against itself at k = 16: the top k-mer has 2,188 positions, ~29 M rows."""
    k = 16
    ix = kh.make_kmer_hash(test_fa, k)
    assert int(kh.kmer_pos(ix, 8)["count"].max()) == 2_188
    rows = oracle.build(test_fa, k).query(test_fa, k)
    assert len(rows) // 2 > 25_000_000
    L = len(test_fa)
    for xr, yr, nx, ny in [((1, L + 1), (1, L + 1), 1_000, 1_000), ((1, L + 1), (1, L + 1), 61, 7),
                           ((20_000, 30_000), (5_000, 45_000), 333, 250)]:
        got = kh.seq_kmer_dotplot(ix, test_fa, k, x_range=xr, y_range=yr, bins=(nx, ny))
        assert np.array_equal(got.ravel(order="F"), bin_rows(rows, xr, yr, nx, ny)), (nx, ny)
    ix.free()


@pytest.mark.gpu
def test_more_than_2_31_rows(kh, oracle):
    """Self dot plot of a 50,000-base homopolymer: (n - k + 1)^2 ~ 2.5 * 10^9 rows, checked analytically: every query
    window pairs with every indexed position, so the image is the outer product of the two coordinates' histograms."""
    k, n = 16, 50_000
    s = "A" * n
    ix = kh.make_kmer_hash(s, k, do_sort=True)
    _, N = ix.sizes_un
    qk, qs = oracle.windows(s, k)
    ipos = oracle.build(s, k).extract(2)["pos"].reshape(-1, 2)[:, 1]
    assert len(ipos) == N and len(qs) * N > 2**31
    xr, yr, nx, ny = (0, n + 2), (1, n - 3), 7, 5
    hx = bin_rows(np.stack([qs + k - 1, np.zeros_like(qs) + 1], 1), xr, (0, 2), nx, 1)
    hy = bin_rows(np.stack([np.zeros_like(ipos) + 1, ipos], 1), (0, 2), yr, 1, ny)
    want = np.outer(hx, hy).ravel(order="F")
    got = kh.seq_kmer_dotplot(ix, s, k, x_range=xr, y_range=yr, bins=(nx, ny))
    assert np.array_equal(got.ravel(order="F"), want) and got.sum() > 2**31
    hxa = bin_rows(np.stack([ipos, np.zeros_like(ipos) + 1], 1), xr, (0, 2), nx, 1)
    got = kh.kmer_pairs_dotplot(ix, ix, a_range=xr, b_range=yr, bins=(nx, ny))
    assert np.array_equal(got.ravel(order="F"), np.outer(hxa, hy).ravel(order="F"))
    assert kh.kmer_pairs_dotplot(ix, ix, a_range=xr, b_range=yr, bins=(nx, ny), max_count=N - 1).sum() == 0
    ix.free()


@pytest.mark.gpu
def test_output_memory_kinds_and_guards(kh, k11):
    """The same bytes into a device tensor, pinned memory and pageable memory (8.8 MB: the staged path), with guard bytes
    around the image untouched and every cell written."""
    import torch
    k, s, q, rows, _ = k11
    ix = kh.make_kmer_hash(s, k)
    nx, ny, G = 1_100, 1_000, 64
    args = dict(x_range=(1, len(q) + 1), y_range=(1, len(s) + 1), bins=(nx, ny))
    want = bin_rows(rows, args["x_range"], args["y_range"], nx, ny)
    assert 8 * nx * ny > (8 << 20)
    dev = torch.full((nx * ny + 2 * G,), -7.0, dtype=torch.float64, device="cuda")
    kh.seq_kmer_dotplot(ix, q, k, out=dev[G:-G], **args)
    d = dev.cpu().numpy()
    pin = kh.pinned_empty(nx * ny + 2 * G, np.float64)
    page = np.empty(nx * ny + 2 * G, np.float64)
    for buf in (pin, page):
        buf[:] = -7.0
        kh.seq_kmer_dotplot(ix, q, k, out=buf[G:-G], **args)
    for buf in (d, pin, page):
        assert (buf[:G] == -7.0).all() and (buf[-G:] == -7.0).all()
        assert np.array_equal(buf[G:-G], want)
    jd = torch.full((7 * 5 + 2 * G,), -7.0, dtype=torch.float64, device="cuda")
    kh.kmer_pairs_dotplot(ix, ix, a_range=(1, len(s) + 1), b_range=(1, len(s) + 1), bins=(7, 5), out=jd[G:-G])
    j = jd.cpu().numpy()
    assert (j[:G] == -7.0).all() and (j[-G:] == -7.0).all() and j[G:-G].sum() > 0 and (j[G:-G] >= 0).all()
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
    kh.seq_kmer_dotplot(ix, q, k, y_range=(1, len(s) + 1))                # warm: key table built
    before = kh.kmer_pos(ix, 2 | 8)
    sentinel = torch.randint(-2**31, 2**31 - 1, (4 << 20,), dtype=torch.int32, device="cuda")
    sha = hashlib.sha256(sentinel.cpu().numpy().tobytes()).hexdigest()
    torch.cuda.synchronize()
    lib.check(L.kmg_trim())
    free0 = torch.cuda.mem_get_info()[0]
    for rc in (False, True):
        kh.seq_kmer_dotplot(ix, q, k, y_range=(1, len(s) + 1), reverse_complement=rc, max_count=10)
    img = kh.kmer_pairs_dotplot(ix, ix, a_range=(1, len(s) + 1), b_range=(1, len(s) + 1), bins=(500, 500))
    assert np.trace(img) >= ix.sizes_un[1] - 1                   # the diagonal: every position pairs with itself
    lib.check(L.kmg_trim())
    assert torch.cuda.mem_get_info()[0] >= free0 - (2 << 20)
    assert hashlib.sha256(sentinel.cpu().numpy().tobytes()).hexdigest() == sha
    after = kh.kmer_pos(ix, 2 | 8)
    assert np.array_equal(before["pos"], after["pos"]) and np.array_equal(before["count"], after["count"])
    ix.free()


@pytest.mark.gpu
def test_empty_cases(kh):
    ix = kh.make_kmer_hash("N" * 50, 5)                        # U = 0
    assert ix.sizes_un == (0, 0)
    out = np.full((3, 4), -1.0, order="F")
    assert (kh.seq_kmer_dotplot(ix, "ACGTACGTAC", 5, y_range=(0, 60), bins=(3, 4), out=out) == 0).all()
    ix2 = kh.make_kmer_hash("ACGTACGTACGGT", 5)
    out[:] = -1
    assert (kh.seq_kmer_dotplot(ix2, "NNNNNNNN", 5, y_range=(0, 60), bins=(3, 4), out=out) == 0).all()   # no windows
    out[:] = -1
    assert (kh.seq_kmer_dotplot(ix2, "TTTTTTTTTT", 5, y_range=(0, 60), bins=(3, 4), out=out) == 0).all()  # nothing shared
    out[:] = -1
    assert (kh.kmer_pairs_dotplot(ix, ix2, a_range=(0, 60), b_range=(0, 60), bins=(3, 4), out=out) == 0).all()
    lib, L = _lib()
    o = np.full(12, -1.0)
    assert L.kmg_query_dotplot(ix2._handle(), b"ACGT", 4, 5, 0, 0, 60, 3, 0, 60, 4, 0, o.ctypes.data) == 0   # qlen < k
    assert (o == 0).all()
    ix.free(); ix2.free()


@pytest.mark.gpu
def test_c_abi_guards(kh):
    lib, L = _lib()
    ix = kh.make_kmer_hash("ACGTACGTACGGTACCA", 5)
    h = ix._handle()
    q = b"ACGTACGTAC"
    o = np.full(64, -1.0)
    p = o.ctypes.data

    def qd(*, ix=h, q=q, qlen=len(q), k=5, rc=0, x=(0, 20), nx=3, y=(0, 20), ny=4, mc=0, out=p):
        return L.kmg_query_dotplot(ix, q, qlen, k, rc, x[0], x[1], nx, y[0], y[1], ny, mc, out)

    def jd(*, a=h, b=h, x=(0, 20), nx=3, y=(0, 20), ny=4, mc=0, out=p):
        return L.kmg_join_dotplot(a, b, x[0], x[1], nx, y[0], y[1], ny, mc, out)

    assert qd() == 0 and jd() == 0 and o[:12].sum() > 0 and (o[12:] == -1).all()
    for f in (qd, jd):
        for bad in (dict(out=None), dict(nx=0), dict(ny=-1), dict(x=(5, 5)), dict(x=(6, 5)), dict(x=(-1, 5)),
                    dict(y=(0, TOP + 1)), dict(y=(TOP, TOP + 1))):
            assert f(**bad) == -1, (f.__name__, bad)
        assert f(nx=65536, ny=32768) == -3
    assert qd(ix=None) == -1 and jd(a=None) == -1 and jd(b=None) == -1
    assert qd(rc=2) == -1 and qd(rc=-1) == -1
    assert qd(k=0) == -2 and qd(k=33) == -2
    assert qd(qlen=2**31 - 1) == -3
    assert qd(q=None) == -1
    assert (o[12:] == -1).all()
    ix.free()


@pytest.mark.gpu
def test_r_glue_dotplot(oracle):
    """.Call("sequence_kmer_dotplot") and .Call("kmer_pair_dotplot"): nx x ny REALSXP matrices equal to the binned oracle
    rows; the guards of seq.kmer.pos; count tables refused; over-size refused before anything is allocated."""
    from rsession import RError, RSession
    R = RSession()
    R.stub.REAL.restype, R.stub.REAL.argtypes = C.POINTER(C.c_double), [C.c_void_p]

    def reals(x):
        n = R.stub.Rf_length(x)
        return np.ctypeslib.as_array(R.stub.REAL(x), shape=(n,)).copy()

    k = 13
    s, q = _pair(k, 555)
    ix = R.make_kmer_hash(s, k)
    o = oracle.build(s, k)
    for rc in (0, 1):
        rows = o.query(host_revcomp(q) if rc else q, k)
        for mc in (0, 3):
            if mc:
                qk, qs = oracle.windows(host_revcomp(q) if rc else q, k)
                rows = probe_rows(without_repeats(o.extract(2 | 8), mc), qk, qs, k)
            r = R.call("sequence_kmer_dotplot", ix, R.character(q), R.integer(k), R.integer(1, len(q) + 1, 37, 1, len(s) + 1, 29, rc, mc))
            assert R.typeof(r) == REALSXP and R.dims(r) == (37, 29)
            got = reals(r)
            R.stub.rstub_release(r)
            assert np.array_equal(got, bin_rows(rows, (1, len(q) + 1), (1, len(s) + 1), 37, 29)), (rc, mc)
    ib = R.make_kmer_hash(q, k)
    e_s, e_q = o.extract(2 | 8), oracle.build(q, k).extract(2 | 8)
    r = R.call("kmer_pair_dotplot", ix, ib, R.integer(0, len(s) + 2, 11, 1, len(q) + 1, 13, 0))
    assert R.typeof(r) == REALSXP and R.dims(r) == (11, 13)
    assert np.array_equal(reals(r), bin_rows(oracle_mod.pairs_join(e_s, e_q), (0, len(s) + 2), (1, len(q) + 1), 11, 13))
    R.stub.rstub_release(r)
    good = R.integer(1, 100, 5, 1, 100, 5, 0, 0)
    with pytest.raises(RError, match="the sequence should be longer than k and k should not be longer than 31"):
        R.call("sequence_kmer_dotplot", ix, R.character(q), R.integer(32), good)
    with pytest.raises(RError, match="the sequence should be longer than k"):
        R.call("sequence_kmer_dotplot", ix, R.character("ACGT"), R.integer(k), good)
    with pytest.raises(RError, match="params should be an integer vector of length 8"):
        R.call("sequence_kmer_dotplot", ix, R.character(q), R.integer(k), R.integer(1, 100, 5))
    with pytest.raises(RError, match="params should be an integer vector of length 7"):
        R.call("kmer_pair_dotplot", ix, ix, good)
    with pytest.raises(RError, match="rc should be TRUE or FALSE"):
        R.call("sequence_kmer_dotplot", ix, R.character(q), R.integer(k), R.integer(1, 100, 5, 1, 100, 5, 2, 0))
    with pytest.raises(RError, match="max.count should be 0"):
        R.call("kmer_pair_dotplot", ix, ix, R.integer(1, 100, 5, 1, 100, 5, -1))
    with pytest.raises(RError, match="bins must be positive"):
        R.call("kmer_pair_dotplot", ix, ix, R.integer(1, 100, 0, 1, 100, 5, 0))
    with pytest.raises(RError, match="seq.kmer.dotplot failed: .*x window"):
        R.call("sequence_kmer_dotplot", ix, R.character(q), R.integer(k), R.integer(100, 100, 5, 1, 100, 5, 0, 0))
    with pytest.raises(RError, match="kmer.pairs.dotplot failed: .*y window"):
        R.call("kmer_pair_dotplot", ix, ix, R.integer(1, 100, 5, -5, 100, 5, 0))
    ct = R.call("count_kmers", R.nil, R.integer(k, 0, 1), R.character(s))
    with pytest.raises(RError, match="holds k-mer counts"):
        R.call("sequence_kmer_dotplot", ct, R.character(q), R.integer(k), good)
    with pytest.raises(RError, match="holds k-mer counts"):
        R.call("kmer_pair_dotplot", ix, ct, R.integer(1, 100, 5, 1, 100, 5, 0))
    big_q, big_s, big_p = R.character(q), R.integer(k), R.integer(1, 100, 65536, 1, 100, 32768, 0, 0)
    big_j = R.integer(1, 100, 65536, 1, 100, 32768, 0)
    live = R.stub.rstub_live_objects()
    with pytest.raises(RError, match="more than an R matrix can hold"):
        R.call("sequence_kmer_dotplot", ix, big_q, big_s, big_p)
    with pytest.raises(RError, match="more than an R matrix can hold"):
        R.call("kmer_pair_dotplot", ix, ix, big_j)
    assert R.stub.rstub_live_objects() == live                                     # refused before allocating
    assert R.stub.rstub_protect_depth() == 0
    for p in (ix, ib, ct):
        R.stub.rstub_finalize(p)
