"""The retry of segments and chains after an unstable sort, and the device memory it takes and gives back.

Segments and chains sort their runs by diagonal with kmg_build_records; when a sort pass ranks equal keys out of order
(rank variant 4, "unstable on purpose", as in test_parity_gpu.py::test_unstable_sort_is_caught_and_rebuilt) the build
reports KMG_ERR_UNSTABLE, the device is switched to the bitmap variant and kmg_segments_begin / kmg_join_segments_begin /
kmg_chains_begin run once more.  The result must be that of a stable sort, and once every handle is freed and kmg_trim
has run the device must have back what it had before.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import random_dna

pytestmark = pytest.mark.gpu

K = 12
G, W = 3 * K, 4                 # chains: bridge substitutions and shifts of up to 4 bases


@pytest.fixture(scope="module")
def kh():
    import kmer_hasher_b200 as kh
    return kh


def _lib():
    from kmer_hasher_b200 import _lib as lib
    return lib, lib.load()


def tandem(seed, unit=37, copies=400, flank=3000):
    """Random flanks around `copies` copies of one random unit, one substitution in each copy: every diagonal between two
    copies is cut into many runs, so the sorts by diagonal see long stretches of equal keys."""
    rng = np.random.default_rng(seed)
    rep = np.tile(random_dna(unit, seed + 1), copies)
    at = np.arange(copies) * unit + rng.integers(0, unit, copies)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    rep[at] = acgt[(np.searchsorted(acgt, rep[at]) + rng.integers(1, 4, copies)) % 4]
    return np.concatenate([random_dna(flank, seed + 2), rep, random_dna(flank, seed + 3)])


def revcomp(s):
    return np.frombuffer(s[::-1].tobytes().translate(bytes.maketrans(b"ACGT", b"TGCA")), np.uint8).copy()


def _free_after_trim(lib, L):
    import torch
    torch.cuda.synchronize()
    lib.check(L.kmg_trim())
    return torch.cuda.mem_get_info()[0]


def _unstable(lib, L, call):
    """call() with the sort variant that is unstable on purpose; its first sort must fail and be redone."""
    before = L.kmg_tune_get(b"unstable_rebuilds", 0)
    try:
        lib.check(L.kmg_tune(b"reset_rank", 0))
        lib.check(L.kmg_tune(b"sort_cfg", 4))
        got = call()
        assert L.kmg_tune_get(b"rank_variant", 0) == 0          # demoted to the bitmap variant, override dropped
    finally:
        lib.check(L.kmg_tune(b"sort_cfg", -1))
        lib.check(L.kmg_tune(b"reset_rank", 0))               # the self-test decides again
    assert L.kmg_tune_get(b"unstable_rebuilds", 0) > before, "no unstable sort was caught: the retry did not run"
    return got


def _same_after_retry(lib, L, call):
    """call() with the default variant, then with the unstable one: the same rows, and no device memory kept."""
    want = call()
    free0 = _free_after_trim(lib, L)
    got = _unstable(lib, L, call)
    assert got.shape == want.shape and np.array_equal(got, want)
    assert _free_after_trim(lib, L) >= free0 - (2 << 20)
    return want


def _indexes(kh, case):
    """(query index a, index b, query sequence, reverse_complement) of a case"""
    seq = tandem(11)
    b = kh.make_kmer_hash(seq, K)
    if case == "seq":
        return b, b, seq, False
    if case == "pairs":
        return b, b, None, False
    return kh.make_kmer_hash(revcomp(seq), K), b, None, True


def _free(a, b):
    a.free()
    if b is not a:
        b.free()


@pytest.mark.parametrize("case", ["seq", "pairs", "pairs_rc"])
def test_segments_retry(kh, case):
    lib, L = _lib()
    a, b, q, rc = _indexes(kh, case)
    try:
        if q is not None:
            call = lambda: kh.seq_kmer_segments(b, q, K)
        else:
            call = lambda: kh.kmer_pairs_segments(a, b, reverse_complement=rc)
        runs = _same_after_retry(lib, L, call)
        assert len(runs) > 10_000
    finally:
        _free(a, b)


def _segments_handle(lib, L, a, b, q, rc):
    """A segments handle made with the default variant, through the C API"""
    st, R = C.c_void_p(), C.c_uint64()
    if q is not None:
        lib.check(L.kmg_segments_begin(b._handle(), C.c_void_p(q.ctypes.data), q.size, K, 0, 0, 1, C.byref(st), C.byref(R)))
    else:
        lib.check(L.kmg_join_segments_begin(a._handle(), b._handle(), int(rc), 0, 1, C.byref(st), C.byref(R)))
    return st


def _chains(lib, L, seg):
    """kmg_chains_begin over the segments handle seg (which stays), emitted and freed"""
    st, Cn = C.c_void_p(), C.c_uint64()
    lib.check(L.kmg_chains_begin(seg, G, W, 1, C.byref(st), C.byref(Cn)))
    try:
        out = np.empty((Cn.value, 6), np.int32)
        lib.check(L.kmg_chains_emit(st, C.c_void_p(out.ctypes.data)))
    finally:
        L.kmg_chains_free(st)
    return out


@pytest.mark.parametrize("case", ["seq", "pairs", "pairs_rc"])
def test_chains_retry(kh, case):
    """The segments are made with the default variant, so that the sort that fails is chains' own sort by diagonal."""
    lib, L = _lib()
    a, b, q, rc = _indexes(kh, case)
    seg = _segments_handle(lib, L, a, b, q, rc)
    try:
        chains = _same_after_retry(lib, L, lambda: _chains(lib, L, seg))
        assert 0 < len(chains) and (chains[:, 5] > 1).any()     # some chains join several runs
        if q is not None:
            assert np.array_equal(chains, kh.seq_kmer_chains(b, q, K, max_gap=G, max_shift=W))
        else:
            assert np.array_equal(chains, kh.kmer_pairs_chains(a, b, max_gap=G, max_shift=W, reverse_complement=rc))
    finally:
        L.kmg_segments_free(seg)
        _free(a, b)
