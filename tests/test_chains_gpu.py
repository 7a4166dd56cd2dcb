"""Chains (kmg_chains_begin / emit / emit_chunk / free, seq_kmer_chains, kmer_pairs_chains, .Call("sequence_kmer_chains") and
.Call("kmer_pair_chains")) against a numpy restatement of the chaining rules over the runs of the oracle's rows.

`chains_of` follows the rules of include/kmergpu.h literally: for every run, on each diagonal key + delta (|delta| <= W),
the first run at or after the successor threshold and the last run ending before the predecessor threshold (searchsorted
over the runs sorted by (diagonal, i)); the least cost packed into one int64; mutual links; heads by pointer jumping;
n and m by bincount.  `chains_brute` restates it again over all pairs, for small inputs.
"""
import ctypes as C
import hashlib

import numpy as np
import pytest

import oracle as oracle_mod
from conftest import random_dna
from test_dotplot_gpu import _pair, host_revcomp, without_repeats
from test_extraction_chunks_gpu import probe_rows
from test_join_segments_gpu import anti_runs, rc_extraction
from test_segments_gpu import runs_of

INTSXP = 13
I31 = 2**31


def _cost(gq, gr, delta):
    """(max(gq, gr), |delta|, gq) as one int64: for a fixed max and |delta| the smaller gq is the negative delta."""
    return (np.maximum(gq, gr) << 12) | (np.abs(delta) << 1) | (delta > 0)


def chains_of(runs, max_gap, max_shift, anti=False, min_rows=1):
    """(C, 6) int64 (i, j, I, J, n, m): the chains of the (i, j, n) runs, ordered by (i, j), n >= min_rows."""
    r = np.asarray(runs, np.int64).reshape(-1, 3)
    R = len(r)
    if R == 0:
        return np.empty((0, 6), np.int64)
    r = r[np.lexsort((r[:, 1], r[:, 0]))]
    i, j, n = r[:, 0], r[:, 1], r[:, 2]
    I = i + n - 1
    J = j - n + 1 if anti else j + n - 1
    key = i + j if anti else i - j + I31                         # below 2^32: (key << 31) | i stays below 2^63
    o = np.lexsort((i, key))                                    # the diagonal view: queries made in it come sorted,
    sk, si, sI = key[o], i[o], I[o]                             # which keeps searchsorted fast
    P1, P2 = (sk << 31) | si, (sk << 31) | sI                   # runs of one diagonal are disjoint: both ascend
    G, W = int(max_gap), int(max_shift)
    NONE = np.iinfo(np.int64).max
    bs, bp = np.full(R, NONE), np.full(R, NONE)
    vs, vp = np.full(R, -1), np.full(R, -1)                     # in the diagonal view
    for d in range(-W, W + 1):
        # successor on diagonal key + d: the first run with i >= I + 1 + max(0, d)
        tk, thr = sk + d, sI + 1 + max(d, 0)
        ok = (tk >= 0) & (tk < 2**32) & (thr < I31)
        at = np.searchsorted(P1, (np.clip(tk, 0, 2**32 - 1) << 31) | np.minimum(thr, I31 - 1))
        a = np.minimum(at, R - 1)
        gq = si[a] - sI - 1
        ok &= (at < R) & (sk[a] == tk) & (gq <= G + min(d, 0))
        c = _cost(gq, gq - d, d)
        b = ok & (c < bs)
        bs[b], vs[b] = c[b], a[b]
        # predecessor on diagonal key - d: the last run with I <= i - 1 - max(0, d)
        pk, thr = sk - d, si - 1 - max(d, 0)
        ok = (pk >= 0) & (pk < 2**32) & (thr >= 1)
        at = np.searchsorted(P2, (np.clip(pk, 0, 2**32 - 1) << 31) | np.maximum(thr, 0), side="right") - 1
        a = np.maximum(at, 0)
        gq = si - sI[a] - 1
        ok &= (at >= 0) & (sk[a] == pk) & (gq <= G + min(d, 0))
        c = _cost(gq, gq - d, d)
        b = ok & (c < bp)
        bp[b], vp[b] = c[b], a[b]
    del P1, P2, bs, bp
    run_vs, run_vp = np.full(R, -1), np.full(R, -1)             # back to run numbers
    run_vs[o] = np.where(vs >= 0, o[np.maximum(vs, 0)], -1)
    run_vp[o] = np.where(vp >= 0, o[np.maximum(vp, 0)], -1)
    vs, vp = run_vs, run_vp
    return _assemble(r, I, J, vs, vp, min_rows)


def _assemble(r, I, J, vs, vp, min_rows):
    """Mutual links of succ / pred, heads by pointer jumping, per-chain sums: the chains in run order."""
    R = len(r)
    ar = np.arange(R)
    linked_in = (vp >= 0) & (vs[np.maximum(vp, 0)] == ar)
    head = np.where(linked_in, vp, ar)
    while True:
        nxt = head[head]
        if np.array_equal(nxt, head):
            break
        head = nxt
    n = np.bincount(head, weights=r[:, 2], minlength=R).astype(np.int64)
    m = np.bincount(head, minlength=R).astype(np.int64)
    tail = ~((vs >= 0) & linked_in[np.maximum(vs, 0)] & (vp[np.maximum(vs, 0)] == ar))
    lastI, lastJ = np.zeros(R, np.int64), np.zeros(R, np.int64)
    lastI[head[tail]], lastJ[head[tail]] = I[tail], J[tail]
    h = head == ar
    out = np.stack([r[h, 0], r[h, 1], lastI[h], lastJ[h], n[h], m[h]], 1)
    return out[out[:, 4] >= max(min_rows, 1)]


def chains_brute(runs, max_gap, max_shift, anti=False, min_rows=1):
    """chains_of by an all-pairs search (small inputs only)."""
    r = np.asarray(runs, np.int64).reshape(-1, 3)
    if len(r) == 0:
        return np.empty((0, 6), np.int64)
    r = r[np.lexsort((r[:, 1], r[:, 0]))]
    i, j, n = r[:, 0], r[:, 1], r[:, 2]
    I = i + n - 1
    J = j - n + 1 if anti else j + n - 1
    gq = i[None, :] - I[:, None] - 1                            # [s, t]
    gr = (J[:, None] - j[None, :] - 1) if anti else (j[None, :] - J[:, None] - 1)
    may = (gq >= 0) & (gr >= 0) & (gq <= max_gap) & (gr <= max_gap) & (np.abs(gq - gr) <= max_shift)
    c = np.where(may, _cost(gq, gr, gq - gr), np.iinfo(np.int64).max)
    vs = np.where(may.any(1), c.argmin(1), -1)
    vp = np.where(may.any(0), c.argmin(0), -1)
    return _assemble(r, I, J, vs, vp, min_rows)


# ---- the restatement by hand ---------------------------------------------------------------------------------------
def test_substitution_bridged_at_k():
    k = 5
    runs = [(10, 1, 6), (21, 12, 4)]                            # one base differs: gq = gr = k on one diagonal
    assert chains_of(runs, k, 0).tolist() == [[10, 1, 24, 15, 10, 2]]
    assert chains_of(runs, k - 1, 0).tolist() == [[10, 1, 15, 6, 6, 1], [21, 12, 24, 15, 4, 1]]


def test_one_base_indels_need_a_shift():
    k = 5
    ins = [(10, 1, 6), (21, 11, 4)]                             # (gq, gr) = (k, k - 1)
    dele = [(10, 1, 6), (20, 12, 4)]                            # (k - 1, k)
    for runs, end in ((ins, [24, 14]), (dele, [23, 15])):
        assert chains_of(runs, k, 0)[:, 5].tolist() == [1, 1]
        assert chains_of(runs, k, 1).tolist() == [[10, 1] + end + [10, 2]]


def test_tie_break_levels():
    s = (10, 1, 6)                                              # I = 15, J = 6
    # level 1: max(gq, gr) 3 (delta 1) beats 4 (delta 0); the loser is a chain of its own
    assert chains_of([s, (20, 11, 3), (19, 9, 3)], 10, 2).tolist() == [[10, 1, 21, 11, 9, 2], [20, 11, 22, 13, 3, 1]]
    # level 2: max 4 both, |delta| 0 beats 1
    assert chains_of([s, (20, 11, 3), (19, 11, 3)], 10, 2).tolist() == [[10, 1, 22, 13, 9, 2], [19, 11, 21, 13, 3, 1]]
    # level 3: max 4 and |delta| 1 both, gq 3 (delta -1) beats gq 4 (delta +1)
    assert chains_of([s, (20, 10, 3), (19, 11, 3)], 10, 2).tolist() == [[10, 1, 21, 13, 9, 2], [20, 10, 22, 12, 3, 1]]


def test_competing_predecessors_link_once():
    # s1 and s2 both have t as their least-cost successor; pred(t) = s1, so s2 -> t is not a link
    runs = [(10, 1, 6), (11, 1, 5), (21, 12, 4)]
    assert chains_of(runs, 10, 2).tolist() == [[10, 1, 24, 15, 10, 2], [11, 1, 15, 5, 5, 1]]


def test_overlapping_runs_refused():
    runs = [(10, 1, 6), (14, 6, 5), (17, 5, 3)]                 # overlap in the query; overlap in the index
    assert chains_of(runs, 100, 3)[:, 5].tolist() == [1, 1, 1]


def test_antiparallel():
    k = 5
    runs = [(10, 100, 6), (21, 89, 4)]                          # I = 15, J = 95; gq = gr = 5 on one anti-diagonal
    assert chains_of(runs, k, 0, anti=True).tolist() == [[10, 100, 24, 86, 10, 2]]
    assert chains_of(runs, k, 0).tolist() == [[10, 100, 15, 105, 6, 1], [21, 89, 24, 92, 4, 1]]
    assert chains_of([(10, 100, 6), (21, 90, 4)], k, 1, anti=True).tolist() == [[10, 100, 24, 87, 10, 2]]


def test_gap_zero_is_the_runs():
    rng = np.random.default_rng(5)
    rows = np.unique(rng.integers(1, 60, (900, 2)), axis=0)
    for anti, restate in ((False, runs_of), (True, anti_runs)):
        runs = restate(rows)
        got = chains_of(runs, 0, 0, anti=anti)
        I, J = runs[:, 0] + runs[:, 2] - 1, runs[:, 1] - runs[:, 2] + 1 if anti else runs[:, 1] + runs[:, 2] - 1
        assert np.array_equal(got, np.stack([runs[:, 0], runs[:, 1], I, J, runs[:, 2], np.ones(len(runs), np.int64)], 1))


@pytest.mark.parametrize("seed", range(6))
def test_restatement_equals_all_pairs(seed):
    rng = np.random.default_rng(seed)
    rows = np.unique(rng.integers(1, 120, (2500, 2)), axis=0)
    for anti, restate in ((False, runs_of), (True, anti_runs)):
        runs = restate(rows)
        for G, W, mr in ((0, 0, 1), (3, 0, 1), (5, 2, 1), (12, 4, 3), (40, 40, 1)):
            want = chains_brute(runs, G, W, anti, mr)
            got = chains_of(runs, G, W, anti, mr)
            assert np.array_equal(got, want), (anti, G, W, mr)
            if mr == 1:
                assert got[:, 5].sum() == len(runs) and got[:, 4].sum() == runs[:, 2].sum()
        assert (chains_of(runs, 40, 40, anti)[:, 5] > 1).any()


def test_python_guards_on_cpu():
    import kmer_hasher_b200 as kh
    ix = kh.KmerHash(None, 5)
    for call in (lambda **kw: kh.seq_kmer_chains(ix, "ACGTACGT", 5, **kw), lambda **kw: kh.kmer_pairs_chains(ix, ix, **kw)):
        for G, W in ((-1, 0), (2**31, 0)):
            with pytest.raises(ValueError, match="max_gap"):
                call(max_gap=G, max_shift=W)
        for G, W in ((5, 6), (5, -1), (2000, 1025)):
            with pytest.raises(ValueError, match="max_shift"):
                call(max_gap=G, max_shift=W)
        with pytest.raises(ValueError, match="min_rows"):
            call(max_gap=5, max_shift=1, min_rows=-1)
        with pytest.raises(ValueError, match="min_rows"):
            call(max_gap=5, max_shift=1, min_run=2**32)
        with pytest.raises(ValueError, match="max_count"):
            call(max_gap=5, max_shift=1, max_count=-1)
        with pytest.raises(ValueError, match="cleared"):
            call(max_gap=5, max_shift=1)
    with pytest.raises(TypeError):
        kh.seq_kmer_chains(ix, "ACGTACGT", 5)                   # max_gap and max_shift have no default
    with pytest.raises(ValueError, match="count.kmers"):
        kh.seq_kmer_chains(kh.KmerCounts(None, 5, 2), "ACGTACGT", 5, max_gap=5, max_shift=1)
    with pytest.raises(ValueError, match="count.kmers"):
        kh.kmer_pairs_chains(ix, kh.KmerCounts(None, 5, 2), max_gap=5, max_shift=1)
    with pytest.raises(ValueError, match="longer than k"):
        kh.seq_kmer_chains(ix, "ACGTA", 5, max_gap=5, max_shift=1)


def test_glue_registration_and_argument_errors_on_cpu():
    from rsession import RError, RSession
    R = RSession()
    with pytest.raises(RError, match="Incorrect number of arguments"):
        R.call("sequence_kmer_chains", R.integer(1), R.character("ACGT"), R.integer(2))
    with pytest.raises(RError, match="Incorrect number of arguments"):
        R.call("kmer_pair_chains", R.integer(1), R.integer(2))
    with pytest.raises(RError, match="ptr_r should be an external pointer"):
        R.call("sequence_kmer_chains", R.integer(1), R.character("ACGT"), R.integer(2), R.integer(0, 0, 1, 5, 1, 1))
    with pytest.raises(RError, match="ptr_r should be an external pointer"):
        R.call("kmer_pair_chains", R.integer(1), R.integer(2), R.integer(0, 0, 1, 5, 1, 1))
    assert R.stub.rstub_protect_depth() == 0


# ---- on the GPU ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def kh():
    import kmer_hasher_b200 as kh
    return kh


def _lib():
    from kmer_hasher_b200 import _lib as lib
    return lib, lib.load()


def _chains_begin(L, seg, G, W, mr=1):
    """kmg_chains_begin -> (return code, handle, C)"""
    st, Cn = C.c_void_p(), C.c_uint64()
    rv = L.kmg_chains_begin(seg, G, W, mr, C.byref(st), C.byref(Cn))
    return rv, st, Cn.value


PARAMS = ((0, 0, 1, 1), (None, 1, 1, 1), (None, 3, 1, 30), (100, 4, 1, 1), (100, 4, 5, 40), (1000, 16, 1, 0))


def _gw(G, W, k):
    """(G, W) of a PARAMS entry for this k: None is 2k, and W never exceeds G."""
    G = 2 * k if G is None else G
    return G, min(W, G)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 5, 8, 11, 16, 21, 27, 31, 32])
def test_chains_match_oracle(kh, oracle, k):
    """_pair inputs: the query on both strands and the join forward and antiparallel, sorted and grouped builds, several
    (G, W, min_run, min_rows), and max_count through the oracle's rows without the repeated k-mers."""
    s, q = _pair(k, 7000 + k)
    o = oracle.build(s, k)
    es, eq = o.extract(2 | 8), oracle.build(q, k).extract(2 | 8)
    for do_sort in (True, False):
        ix, iq = kh.make_kmer_hash(s, k, do_sort=do_sort), kh.make_kmer_hash(q, k, do_sort=not do_sort)
        for rc in (False, True):
            rows = o.query(host_revcomp(q) if rc else q, k)
            for G, W, mrun, mr in PARAMS:
                G, W = _gw(G, W, k)
                want = chains_of(runs_of(rows, mrun), G, W, min_rows=mr)
                got = kh.seq_kmer_chains(ix, q, k, max_gap=G, max_shift=W, reverse_complement=rc, min_run=mrun,
                                         min_rows=mr, allow_k32=True)
                assert got.dtype == np.int32 and np.array_equal(got, want), (do_sort, rc, G, W, mrun, mr)
            jrows = oracle_mod.pairs_join(rc_extraction(es, k) if rc else es, eq)
            restate = anti_runs if rc else runs_of
            for G, W, mrun, mr in PARAMS:
                G, W = _gw(G, W, k)
                want = chains_of(restate(jrows, mrun), G, W, anti=rc, min_rows=mr)
                got = kh.kmer_pairs_chains(ix, iq, max_gap=G, max_shift=W, reverse_complement=rc, min_run=mrun, min_rows=mr)
                assert np.array_equal(got, want), (do_sort, rc, G, W, mrun, mr)
        if k in (11, 21):
            qk, qs = oracle.windows(q, k)
            for mc in (1, 3):
                rows = probe_rows(without_repeats(es, mc), qk, qs, k)
                for G, W, mrun, mr in PARAMS[1:4]:
                    G, W = _gw(G, W, k)
                    got = kh.seq_kmer_chains(ix, q, k, max_gap=G, max_shift=W, max_count=mc, min_run=mrun, min_rows=mr)
                    assert np.array_equal(got, chains_of(runs_of(rows, mrun), G, W, min_rows=mr)), (mc, G, W)
        ix.free(); iq.free()


@pytest.mark.gpu
def test_gap_zero_is_the_segments_and_invariants(kh):
    k = 15
    s, q = _pair(k, 31)
    s = np.concatenate([s, s[:5_000], s[2_000:4_000]])
    ix = kh.make_kmer_hash(s, k)
    for rc in (False, True):
        seg = kh.seq_kmer_segments(ix, q, k, reverse_complement=rc, min_rows=0).astype(np.int64)
        got = kh.seq_kmer_chains(ix, q, k, max_gap=0, max_shift=0, reverse_complement=rc, min_rows=0)
        want = np.stack([seg[:, 0], seg[:, 1], seg[:, 0] + seg[:, 2] - 1, seg[:, 1] + seg[:, 2] - 1, seg[:, 2],
                         np.ones(len(seg), np.int64)], 1)
        assert np.array_equal(got, want)
        for G, W in ((k, 1), (3 * k, 3), (500, 20)):
            got = kh.seq_kmer_chains(ix, q, k, max_gap=G, max_shift=W, reverse_complement=rc, min_rows=0).astype(np.int64)
            assert got[:, 5].sum() == len(seg) and got[:, 4].sum() == seg[:, 2].sum()
            assert len(got) < len(seg)
    jseg = kh.kmer_pairs_segments(ix, ix, reverse_complement=True).astype(np.int64)
    got = kh.kmer_pairs_chains(ix, ix, max_gap=0, max_shift=0, reverse_complement=True)
    assert np.array_equal(got, np.stack([jseg[:, 0], jseg[:, 1], jseg[:, 0] + jseg[:, 2] - 1, jseg[:, 1] - jseg[:, 2] + 1,
                                         jseg[:, 2], np.ones(len(jseg), np.int64)], 1))
    ix.free()


def _planted(seed, k):
    """(index, query, blocks): the query holds 5-10 copies of 10-50 kb index blocks between unrelated random stretches,
    each with substitutions every 100-200 bases and a few 1-3 base indels.  blocks: (query start, query end, index start,
    index offset change at the end), 0-based half-open query range."""
    rng = np.random.default_rng(seed)
    s = random_dna(3_000_000, seed)
    parts, blocks, at = [random_dna(int(rng.integers(2_000, 6_000)), seed + 1)], [], None
    at = len(parts[0])
    nb = int(rng.integers(5, 11))
    starts = rng.choice(np.arange(0, len(s) - 60_000, 60_000), nb, replace=False)
    for b in range(nb):
        ln = int(rng.integers(10_000, 50_001))
        src = s[starts[b]:starts[b] + ln + 10]
        out, p, shift, ev = [], 0, 0, 0
        nxt = min(int(rng.integers(100, 200)), ln)
        indels = set(rng.choice(np.arange(5, ln // 150), 3, replace=False).tolist())
        while p < ln:
            if nxt > p:
                out.append(src[p:nxt]); p = nxt
                continue
            if ev in indels and p + 3 < ln:
                L = int(rng.integers(1, 4))
                if rng.integers(0, 2):                          # insertion into the query
                    out.append(np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, L)]); shift += L
                else:                                           # deletion from the query
                    p += L; shift -= L
            else:                                               # substitution
                out.append(np.frombuffer(b"ACGT", np.uint8)[[(("ACGT".index(chr(src[p])) + int(rng.integers(1, 4))) % 4)]])
                p += 1
            ev += 1
            nxt = min(p + int(rng.integers(100, 200)), ln)
        blk = np.concatenate(out)
        parts.append(blk)
        blocks.append((at, at + len(blk), int(starts[b]), shift))
        at += len(blk)
        gap = random_dna(int(rng.integers(1_000, 5_000)), seed + 10 + b)
        parts.append(gap)
        at += len(gap)
    return s, np.concatenate(parts), blocks


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [3, 4])
def test_planted_blocks(kh, seed):
    """With G = 3k and W = 3 each planted block gives one chain holding most of its rows, starting and ending on the
    planted diagonals near the planted ends; no chain reaches into two blocks; the chains equal chains_of(segments)."""
    k = 21
    s, q, blocks = _planted(seed, k)
    ix = kh.make_kmer_hash(s, k)
    seg = kh.seq_kmer_segments(ix, q, k)
    got = kh.seq_kmer_chains(ix, q, k, max_gap=3 * k, max_shift=3).astype(np.int64)
    assert np.array_equal(got, chains_of(seg, 3 * k, 3))
    qs, qe = got[:, 0] - k + 1, got[:, 2]                      # 1-based query bases covered
    for q0, q1, s0, shift in blocks:
        inside = (qe >= q0 + 1) & (qs <= q1)
        big = inside & (got[:, 4] > 1_000)
        assert big.sum() == 1, (q0, q1, got[inside][:5])
        c = got[big][0]
        ln = q1 - q0
        assert c[4] >= 0.7 * ln and c[5] > 20
        assert q0 + 1 - 10 <= c[0] - k + 1 <= q0 + 1 + 200 and q1 - 200 <= c[2] <= q1 + 10
        assert (c[1] - 1) - (c[0] - k) == s0 - q0                 # the planted diagonal at the start
        assert (c[3] - 1) - (c[2] - k) == s0 - q0 - shift         # and at the end, after the indels
        assert ((qs >= q0 + 1 - 10) & (qe <= q1 + 10) | ~inside).all()
    ix.free()


@pytest.mark.gpu
def test_output_memory_kinds_and_chunks(kh):
    """A random 30 Mbp self query at k = 12 (~40 M runs) chained at G = 24, W = 2: the same bytes into a device tensor,
    pinned memory and pageable memory, guard bytes untouched; emit_chunk windows agree; Σ m = R and Σ n = the runs' n."""
    import torch
    lib, L = _lib()
    k, n, Gd = 12, 30_000_000, 16
    s = random_dna(n, 4243)
    ix = kh.make_kmer_hash(s, k)
    seg, R = C.c_void_p(), C.c_uint64()
    lib.check(L.kmg_segments_begin(ix._handle(), s.tobytes(), n, k, 0, 0, 1, C.byref(seg), C.byref(R)))
    rv, st, Cn = _chains_begin(L, seg, 24, 2, 0)
    try:
        lib.check(rv)
        runs = torch.empty((R.value, 3), dtype=torch.int32, device="cuda")
        lib.check(L.kmg_segments_emit(seg, C.c_void_p(runs.data_ptr())))
        L.kmg_segments_free(seg)
        seg = None
        assert Cn > (256 << 20) // 24
        kh.profile(enable=True, reset=True)
        dev = torch.full((6 * Cn + 2 * Gd,), -7, dtype=torch.int32, device="cuda")
        lib.check(L.kmg_chains_emit(st, C.c_void_p(dev[Gd:].data_ptr())))
        torch.cuda.synchronize()
        assert kh.profile(reset=True)["chains_emit"][1] == 1
        pin = kh.pinned_empty(6 * Cn + 2 * Gd, np.int32)
        page = np.empty(6 * Cn + 2 * Gd, np.int32)
        for buf in (pin, page):
            buf[:] = -7
            lib.check(L.kmg_chains_emit(st, C.c_void_p(buf[Gd:].ctypes.data)))
            assert kh.profile(reset=True)["chains_emit"][1] >= 2
        kh.profile(enable=False, reset=True)
        d = dev.cpu().numpy()
        for buf in (d, pin, page):
            assert (buf[:Gd] == -7).all() and (buf[-Gd:] == -7).all()
        assert np.array_equal(pin, d) and np.array_equal(page, d)
        ch = d[Gd:-Gd].reshape(Cn, 6)
        for a, b in ((0, 1), (1, 7_654_321), (7_654_321, Cn - 3), (Cn - 3, Cn)):
            part = np.full(6 * (b - a) + 2 * Gd, -7, np.int32)
            lib.check(L.kmg_chains_emit_chunk(st, a, b - a, C.c_void_p(part[Gd:].ctypes.data)))
            assert (part[:Gd] == -7).all() and (part[-Gd:] == -7).all() and np.array_equal(part[Gd:-Gd].reshape(-1, 6), ch[a:b])
        pd = torch.full((6 * 1000 + 2 * Gd,), -7, dtype=torch.int32, device="cuda")
        lib.check(L.kmg_chains_emit_chunk(st, Cn - 1000, 1000, C.c_void_p(pd[Gd:].data_ptr())))
        p = pd.cpu().numpy()
        assert (p[:Gd] == -7).all() and (p[-Gd:] == -7).all() and np.array_equal(p[Gd:-Gd].reshape(-1, 6), ch[Cn - 1000:])
    finally:
        L.kmg_chains_free(st)
        if seg is not None:
            L.kmg_segments_free(seg)
    assert ch[:, 5].astype(np.int64).sum() == R.value and ch[:, 4].astype(np.int64).sum() == int(runs[:, 2].sum(dtype=torch.int64))
    assert Cn <= R.value
    o = np.lexsort((ch[:, 1], ch[:, 0]))
    assert np.array_equal(o, np.arange(Cn))                      # ordered by (i, j)
    ix.free()


@pytest.mark.gpu
def test_empty_cases(kh):
    lib, L = _lib()
    ix = kh.make_kmer_hash("N" * 50, 5)
    assert kh.seq_kmer_chains(ix, "ACGTACGTAC", 5, max_gap=10, max_shift=2).shape == (0, 6)
    assert kh.kmer_pairs_chains(ix, ix, max_gap=10, max_shift=2).shape == (0, 6)
    ix2 = kh.make_kmer_hash("ACGTACGTACGGT", 5)
    assert kh.seq_kmer_chains(ix2, "TTTTTTTTTT", 5, max_gap=10, max_shift=2).shape == (0, 6)
    assert kh.seq_kmer_chains(ix2, "ACGTACGTACGGT", 5, max_gap=10, max_shift=2, min_rows=100).shape == (0, 6)
    assert kh.seq_kmer_chains(ix2, "ACGTACGTACGGT", 5, max_gap=10, max_shift=2, min_run=100).shape == (0, 6)
    seg, R = C.c_void_p(), C.c_uint64()
    lib.check(L.kmg_segments_begin(ix2._handle(), b"ACGT", 4, 5, 0, 0, 1, C.byref(seg), C.byref(R)))
    assert R.value == 0
    rv, st, Cn = _chains_begin(L, seg, 10, 2)
    assert rv == 0 and Cn == 0
    o = np.full(6, -1, np.int32)
    assert L.kmg_chains_emit(st, o.ctypes.data) == 0 and L.kmg_chains_emit(st, None) == 0 and (o == -1).all()
    assert L.kmg_chains_free(st) == 0
    st = C.c_void_p()
    assert L.kmg_chains_begin(seg, 10, 2, 1, C.byref(st), None) == 0   # C may be NULL
    assert L.kmg_chains_free(st) == 0 and L.kmg_segments_free(seg) == 0
    ix.free(); ix2.free()


@pytest.mark.gpu
def test_c_abi_guards_and_segments_unaffected(kh):
    lib, L = _lib()
    k = 13
    s, q = _pair(k, 17)
    ix = kh.make_kmer_hash(s, k)
    seg, R = C.c_void_p(), C.c_uint64()
    lib.check(L.kmg_segments_begin(ix._handle(), bytes(q), len(q), k, 0, 0, 1, C.byref(seg), C.byref(R)))
    R = R.value
    before = np.full(3 * R, -1, np.int32)
    lib.check(L.kmg_segments_emit(seg, before.ctypes.data))
    for G, W in ((2**31, 0), (2**32 - 1, 0), (5, 6), (2000, 1025)):
        assert _chains_begin(L, seg, G, W)[0] == -1
    assert _chains_begin(L, None, 10, 2)[0] == -1
    assert L.kmg_chains_begin(seg, 10, 2, 1, None, None) == -1
    rv, st, Cn = _chains_begin(L, seg, 2**31 - 1, 1024)           # the largest accepted band
    lib.check(rv)
    L.kmg_chains_free(st)
    rv, st, Cn = _chains_begin(L, seg, 3 * k, 2)
    lib.check(rv)
    assert 0 < Cn < R
    o = np.full(6 * Cn + 8, -1, np.int32)
    p = o.ctypes.data
    assert L.kmg_chains_emit(None, p) == -1
    assert L.kmg_chains_emit(st, None) == -1
    assert L.kmg_chains_emit_chunk(st, 0, Cn + 1, p) == -1
    assert L.kmg_chains_emit_chunk(st, Cn + 1, 0, p) == -1
    assert L.kmg_chains_emit_chunk(st, 1, Cn, p) == -1
    assert L.kmg_chains_emit_chunk(None, 0, 1, p) == -1
    assert (o == -1).all()
    assert L.kmg_chains_emit_chunk(st, Cn, 0, p) == 0
    assert L.kmg_chains_emit(st, p) == 0 and (o[6 * Cn:] == -1).all()
    assert np.array_equal(o[:6 * Cn].reshape(-1, 6), chains_of(before.reshape(-1, 3), 3 * k, 2))
    assert L.kmg_chains_free(st) == 0 and L.kmg_chains_free(None) == 0
    after = np.full(3 * R, -1, np.int32)
    lib.check(L.kmg_segments_emit(seg, after.ctypes.data))     # the segments handle emits the same runs
    assert np.array_equal(before, after)
    L.kmg_segments_free(seg)
    ix.free()


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
    q[400_000:410_000] = s[900_000:910_000]
    q[405_000] = ord("A") if q[405_000] != ord("A") else ord("C")   # one substitution
    ix, iq = kh.make_kmer_hash(s, k), kh.make_kmer_hash(q, k, do_sort=True)
    kh.seq_kmer_chains(ix, q, k, max_gap=3 * k, max_shift=3)    # warm: key tables built
    kh.kmer_pairs_chains(iq, ix, max_gap=3 * k, max_shift=3)
    before = [kh.kmer_pos(x, 2 | 8) for x in (ix, iq)]
    sentinel = torch.randint(-2**31, 2**31 - 1, (4 << 20,), dtype=torch.int32, device="cuda")
    sha = hashlib.sha256(sentinel.cpu().numpy().tobytes()).hexdigest()
    torch.cuda.synchronize()
    lib.check(L.kmg_trim())
    free0 = torch.cuda.mem_get_info()[0]
    for rc in (False, True):
        got = kh.seq_kmer_chains(ix, q, k, max_gap=3 * k, max_shift=3, reverse_complement=rc, min_rows=100)
        jg = kh.kmer_pairs_chains(iq, ix, max_gap=3 * k, max_shift=3, reverse_complement=rc, min_rows=100)
        if not rc:                                              # the two shared stretches, each one chain
            big = got[got[:, 4] > 9_000].astype(np.int64)
            assert len(big) == 2 and big[0, :2].tolist() == [k, 500_001] and 400_000 + k - 10 <= big[1, 0] <= 400_000 + k + 100
            assert ((big[:, 1] - 1) - (big[:, 0] - k) == 500_000).all()   # the shared diagonal (flank bases may match by chance)
            assert len(jg) == len(got) and np.array_equal(jg[:, 0] + k - 1, got[:, 0])
    lib.check(L.kmg_trim())
    assert torch.cuda.mem_get_info()[0] >= free0 - (2 << 20)
    assert hashlib.sha256(sentinel.cpu().numpy().tobytes()).hexdigest() == sha
    for x, b in zip((ix, iq), before):
        a = kh.kmer_pos(x, 2 | 8)
        assert np.array_equal(b["pos"], a["pos"]) and np.array_equal(b["count"], a["count"])
    ix.free(); iq.free()


@pytest.mark.gpu
def test_r_glue_chains(oracle):
    """.Call("sequence_kmer_chains") and .Call("kmer_pair_chains"): 6 x C INTSXP matrices equal to chains_of over the
    oracle's runs; argument messages; count tables refused; PROTECT balanced."""
    from rsession import RError, RSession
    R = RSession()
    k = 13
    s, q = _pair(k, 556)
    ix, iq = R.make_kmer_hash(s, k), R.make_kmer_hash(q, k)
    o = oracle.build(s, k)
    es, eq = o.extract(2 | 8), oracle.build(q, k).extract(2 | 8)
    for rc in (0, 1):
        rows = o.query(host_revcomp(q) if rc else q, k)
        jrows = oracle_mod.pairs_join(rc_extraction(es, k) if rc else es, eq)
        for mrun, G, W, mr in ((1, 0, 0, 1), (1, 3 * k, 3, 1), (4, 100, 4, 30)):
            r = R.call("sequence_kmer_chains", ix, R.character(q), R.integer(k), R.integer(rc, 0, mrun, G, W, mr))
            want = chains_of(runs_of(rows, mrun), G, W, min_rows=mr)
            assert R.typeof(r) == INTSXP and R.dims(r) == (6, len(want))
            got = R.ints(r).reshape(-1, 6)
            R.stub.rstub_release(r)
            assert np.array_equal(got, want), (rc, mrun, G, W, mr)
            r = R.call("kmer_pair_chains", ix, iq, R.integer(rc, 0, mrun, G, W, mr))
            want = chains_of((anti_runs if rc else runs_of)(jrows, mrun), G, W, anti=bool(rc), min_rows=mr)
            assert R.typeof(r) == INTSXP and R.dims(r) == (6, len(want))
            got = R.ints(r).reshape(-1, 6)
            R.stub.rstub_release(r)
            assert np.array_equal(got, want), (rc, mrun, G, W, mr)
    args = lambda *p: (ix, R.character(q), R.integer(k), R.integer(*p))
    with pytest.raises(RError, match="params should be an integer vector of length 6"):
        R.call("sequence_kmer_chains", *args(0, 0, 1))
    with pytest.raises(RError, match="params should be an integer vector of length 6"):
        R.call("kmer_pair_chains", ix, iq, R.integer(0, 0, 1, 5, 1))
    for p, msg in (((2, 0, 1, 5, 1, 1), "rc should be TRUE or FALSE"), ((0, -1, 1, 5, 1, 1), "max.count should be 0"),
                   ((0, 0, -1, 5, 1, 1), "min.run should be 0 or positive"), ((0, 0, 1, -5, 0, 1), "max.gap should be 0"),
                   ((0, 0, 1, 5, 6, 1), "max.shift should be between"), ((0, 0, 1, 5000, 1025, 1), "max.shift should be between"),
                   ((0, 0, 1, 5, 1, -1), "min.rows should be 0 or positive")):
        with pytest.raises(RError, match=msg):
            R.call("sequence_kmer_chains", *args(*p))
        with pytest.raises(RError, match=msg):
            R.call("kmer_pair_chains", ix, iq, R.integer(*p))
    with pytest.raises(RError, match="the sequence should be longer than k and k should not be longer than 31"):
        R.call("sequence_kmer_chains", ix, R.character(q), R.integer(32), R.integer(0, 0, 1, 5, 1, 1))
    with pytest.raises(RError, match="single sequence"):
        R.call("sequence_kmer_chains", ix, R.character(q, q), R.integer(k), R.integer(0, 0, 1, 5, 1, 1))
    ct = R.call("count_kmers", R.nil, R.integer(k, 0, 1), R.character(s))
    with pytest.raises(RError, match="holds k-mer counts"):
        R.call("sequence_kmer_chains", ct, R.character(q), R.integer(k), R.integer(0, 0, 1, 5, 1, 1))
    with pytest.raises(RError, match="holds k-mer counts"):
        R.call("kmer_pair_chains", ix, ct, R.integer(0, 0, 1, 5, 1, 1))
    assert R.stub.rstub_protect_depth() == 0
    for p in (ix, iq, ct):
        R.stub.rstub_finalize(p)


@pytest.mark.gpu
def test_c4_full_size(kh):
    """Config 4 (the 100 Mbp query against the 250 Mbp config-3 index, k = 32) at G = 100, W = 4, both strands: Σ m = R and
    Σ n = the runs' rows (22,878,529 runs of 459,931,872 rows forward), and the chains equal chains_of over the GPU's own
    runs."""
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
    for rc in (0, 1):
        seg, R = C.c_void_p(), C.c_uint64()
        lib.check(L.kmg_segments_begin(ix._handle(), C.c_void_p(dq.data_ptr()), len(q), k, rc, 0, 1, C.byref(seg), C.byref(R)))
        R = R.value
        runs = np.empty((R, 3), np.int32)
        try:
            lib.check(L.kmg_segments_emit(seg, runs.ctypes.data))
            rv, st, Cn = _chains_begin(L, seg, 100, 4)
            lib.check(rv)
            got = np.empty((Cn, 6), np.int32)
            try:
                lib.check(L.kmg_chains_emit(st, got.ctypes.data))
            finally:
                L.kmg_chains_free(st)
        finally:
            L.kmg_segments_free(seg)
        M = int(runs[:, 2].astype(np.int64).sum())
        if not rc:
            assert (R, M) == (22_878_529, 459_931_872)
        assert got[:, 5].astype(np.int64).sum() == R and got[:, 4].astype(np.int64).sum() == M
        assert Cn < R
        assert np.array_equal(got, chains_of(runs, 100, 4)), rc
        del runs, got
    ix.free()
