"""count.kmers, spectra and kmer.pos of a count table against a restatement built from the plain-C oracle.

A count is the length of a sequence's position list (test_oracle.py::test_restated_count_kmers_is_pinned_to_seq_to_hash
pins this against the reference engine), so `expected_counts` restates a whole table from `oracle.build(seq, k)` of
every sequence: the union of the keys and a U x source_n matrix of summed list lengths.  Everything that kmer.pos,
kmer_count and the spectra return follows from that matrix, and is compared exactly.
"""
import ctypes as C
import hashlib

import numpy as np
import pytest

from conftest import random_dna

_ORACLE = []


def _oracle():
    if not _ORACLE:
        from oracle import Oracle
        _ORACLE.append(Oracle())
    return _ORACLE[0]


def expected_counts(batches, k, source_n):
    """(keys, m): ascending distinct keys and the U x source_n int64 count matrix after count.kmers of every batch.
    A batch is (list of sequences, source); sequences no longer than k are skipped, as count.kmers skips them."""
    keys, cols, cnts = [], [], []
    for seqs, source in batches:
        for s in seqs:
            if len(s) <= k:
                continue
            e = _oracle().build(s, k).extract(8)
            keys.append(e["keys"])
            cnts.append(e["count"].astype(np.int64))
            cols.append(np.full(len(e["keys"]), source, np.int64))
    if not keys:
        return np.empty(0, np.uint64), np.zeros((0, source_n), np.int64)
    allk = np.concatenate(keys)
    srt = np.sort(allk)                                    # the union of the keys (np.unique, without its slow path)
    ukeys = srt[np.concatenate([[True], srt[1:] != srt[:-1]])]
    m = np.zeros((len(ukeys), source_n), np.int64)
    np.add.at(m, (np.searchsorted(ukeys, allk), np.concatenate(cols)), np.concatenate(cnts))
    return ukeys, m


def decode_kmers(keys, k):
    """U x k uint8 k-mer strings of 2-bit keys, alphabet A, C, T, G (the reference's decoder)."""
    out = np.empty((len(keys), k), np.uint8)
    alphabet = np.frombuffer(b"ACTG", np.uint8)
    for j in range(k):
        out[:, j] = alphabet[((keys >> np.uint64(2 * (k - 1 - j))) & np.uint64(3)).astype(np.int64)]
    return out


def expected_kmer_pos(keys, m, k, flag=15):
    """What kmer_pos(count table, flag) must return, from the restated table (fields not asked for are None)."""
    U, sn = m.shape
    res = {"kmer": None, "pos": None, "pair.pos": None, "count": None}
    if flag & 1:
        res["kmer"] = decode_kmers(keys, k)
    if flag & 2:
        res["pos"] = np.empty((U * sn, 2), np.int32)
        res["pos"][:, 0] = np.repeat(np.arange(1, U + 1, dtype=np.int32), sn)
        res["pos"][:, 1] = m.ravel()
    if flag & 4:
        ia, ib = np.triu_indices(sn, 1)
        pairs = np.empty((U, len(ia), 3), np.int32)
        pairs[:, :, 0] = np.arange(1, U + 1, dtype=np.int32)[:, None]
        pairs[:, :, 1] = m[:, ia]
        pairs[:, :, 2] = m[:, ib]
        res["pair.pos"] = pairs.reshape(-1, 3)
    if flag & 8:
        res["count"] = np.full(U, sn, np.int32)
    return res


def spectrum(col, max_count):
    return np.bincount(np.minimum(col, max_count), minlength=max_count + 1).astype(np.float64)


def test_expected_counts_by_hand():
    """k = 2 (codes A0 C1 T2 G3): ACGT -> AC CG GT into source 0; ACAC -> AC CA AC into source 1; NN and AC (length
    <= k) are skipped."""
    keys, m = expected_counts([(["ACGT", "AC"], 0), (["ACAC", "NN"], 1)], 2, 2)
    assert keys.tolist() == [1, 4, 7, 14]                  # AC, CA, CG, GT
    assert m.tolist() == [[1, 2], [0, 1], [1, 0], [1, 0]]
    e = expected_kmer_pos(keys, m, 2)
    assert [bytes(r).decode() for r in e["kmer"]] == ["AC", "CA", "CG", "GT"]
    assert e["pos"].tolist() == [[1, 1], [1, 2], [2, 0], [2, 1], [3, 1], [3, 0], [4, 1], [4, 0]]
    assert e["pair.pos"].tolist() == [[1, 1, 2], [2, 0, 1], [3, 1, 0], [4, 1, 0]]
    assert e["count"].tolist() == [2, 2, 2, 2]
    assert spectrum(m[:, 1], 1).tolist() == [2.0, 2.0] and spectrum(m.sum(1), 2).tolist() == [0.0, 3.0, 1.0]
    # end-of-string rule: a last N-free run of exactly k gives no window
    keys, m = expected_counts([(["ACNGT"], 0)], 2, 1)
    assert keys.tolist() == [1] and m.tolist() == [[1]]


@pytest.fixture(scope="module")
def kh():
    import kmer_hasher_b200 as kh
    return kh


def check_table(kh, ptr, keys, m, k):
    """kmer_pos(ptr, 15), kmer_keys, sizes and kmer_count of a count table against the restatement."""
    U, sn = m.shape
    assert ptr.sizes[0] == U
    assert ptr.kmer_count == U                             # every distinct k-mer was new exactly once
    assert np.array_equal(kh.kmer_keys(ptr), keys)
    got, want = kh.kmer_pos(ptr, 15), expected_kmer_pos(keys, m, k)
    assert np.array_equal(got["kmer"].view(np.uint8).reshape(U, k), want["kmer"])
    assert np.array_equal(got["pos"], want["pos"])
    assert np.array_equal(got["pair.pos"], want["pair.pos"])
    assert np.array_equal(got["count"], want["count"])


def check_spectra(kh, ptr, m):
    U, sn = m.shape
    for source in list(range(sn)) + [None]:
        col = m.sum(1) if source is None else m[:, source]
        top = int(col.max())                               # 0 for a column no batch went into
        for max_count in sorted({1, max(top, 1), max(top - 1, 1), 1 << 20}):
            assert np.array_equal(kh.kmer_spectrum(ptr, max_count, source), spectrum(col, max_count)), (source, max_count)


def _scenario(k, sn):
    """Batches (sequences, source) for one table: sources in a scrambled order, a batch of only new k-mers, one of only
    known k-mers, an all-N sequence longer than k, sequences of length k and k+1, a last N-free run of exactly k, lower
    case and IUPAC bytes, and a second batch into a filled column."""
    rng = np.random.default_rng(1000 * k + sn)
    src = [int(x) for x in rng.permutation(max(sn, 6)) % sn]
    mixed = random_dna(40_000, k, p_n=0.002, p_lower=0.3, p_other=0.01, n_runs=3)
    poly_a = np.full(k + 7, ord("A"), np.uint8)
    no_a = np.frombuffer(b"CGT", np.uint8)[rng.integers(0, 3, 30_000)].copy()    # no window equals A^k: all new
    tail = np.concatenate([random_dna(300, k + 1), np.frombuffer(b"N", np.uint8), random_dna(k, k + 2)])
    return [
        ([poly_a], src[0]),
        ([no_a], src[1]),                                                        # only new k-mers
        ([mixed, random_dna(k, 7), random_dna(k + 1, 8), tail], src[2]),
        ([np.full(k + 20, ord("N"), np.uint8), np.full(k + 3, ord("n"), np.uint8)], src[3]),   # U == 0
        ([mixed[5_000:25_000].copy(), no_a[:1000].copy()], src[4]),              # only known k-mers
        ([random_dna(20_000, 50 + k, p_lower=0.5), mixed[:7_000].copy()], src[5]),
    ]


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 5, 11, 16, 20, 21, 27, 31, 32])
def test_count_table_matches_the_restatement(kh, k):
    """1 to 8 sort passes in the batch build and in the merge's record build, both sides of the grouped threshold (k = 21;
    count tables are key-ordered all the same), source_n 1, 2, 3 and 7."""
    for sn in (1, 2, 3, 7):
        batches = _scenario(k, sn)
        ptr = None
        for i, (seqs, source) in enumerate(batches):
            before = ptr.kmer_count if ptr is not None else 0
            ptr = kh.count_kmers(seqs, (k, source, sn), ptr)
            keys, m = expected_counts(batches[:i + 1], k, sn)
            if i in (3, 4):                                # the all-N batch and the batch of known k-mers add nothing
                assert ptr.kmer_count == before
            check_table(kh, ptr, keys, m, k)
        check_spectra(kh, ptr, m)
        if sn >= 2 and k >= 11:                            # some column misses k-mers the others hold: spec[0] > 0
            assert (m == 0).any(axis=0).any()
            assert any(kh.kmer_spectrum(ptr, 3, s)[0] > 0 for s in range(sn))
        with pytest.raises(kh.KmgError):
            kh.kmer_spectrum(ptr, 5, sn)
        ptr.free()


@pytest.mark.gpu
def test_twenty_merges_into_one_table(kh):
    """Twenty successive batches into one table (every merge reuses arena blocks the previous one gave back)."""
    k, sn = 21, 3
    base = random_dna(200_000, 5, p_n=0.001, p_lower=0.2)
    batches = []
    ptr = None
    for i in range(20):
        a = int((i * 7919) % 150_000)
        seqs = [base[a:a + 30_000 + 1000 * i].copy(), random_dna(5_000 + 300 * i, 300 + i)]
        batches.append((seqs, (i * 2) % sn))
        ptr = kh.count_kmers(seqs, (k, (i * 2) % sn, sn), ptr)
        if i % 5 == 4:
            keys, m = expected_counts(batches, k, sn)
            check_table(kh, ptr, keys, m, k)
    check_spectra(kh, ptr, m)
    ptr.free()


# ---- a large table: extraction in many chunks ----------------------------------------------------------------------
STAGE_ROWS_POS = (64 << 20) // 8           # pageable destinations over 8 MiB: 64 MiB staged chunks
PINNED_ROWS_POS = (256 << 20) // 8         # pinned destinations: 256 MiB device chunks


def _chunks(rows, per):
    return -(-rows // per)


@pytest.fixture(scope="module")
def big():
    """About 10.5 M distinct 31-mers over 7 sources (73 M cells): batch j holds 1.5 Mbp of its own and 100 kbp of
    batch j-1, so some k-mers are counted in two columns."""
    k, sn = 31, 7
    own = [random_dna(1_500_000, 7000 + j) for j in range(sn)]
    batches = [([own[j]] + ([own[j - 1][:100_000].copy()] if j else []), (3 * j + 2) % sn) for j in range(sn)]
    keys, m = expected_counts(batches, k, sn)
    return k, sn, batches, keys, m


@pytest.mark.gpu
def test_large_count_table_across_chunks(kh, big):
    """kmg_count_positions and kmg_count_kmers_ascii into a device tensor (one launch), pinned memory (256 MiB chunks)
    and pageable memory (64 MiB staged chunks); all equal to the restatement.  The count matrix, a device tensor and an
    index allocated before the extractions must be unchanged by them: a chunk writes its own rows and nothing else."""
    import torch
    from kmer_hasher_b200 import _lib
    L = _lib.load()
    k, sn, batches, keys, m = big
    U = len(keys)
    cells = U * sn
    assert U >= 9_000_000 and _chunks(cells, STAGE_ROWS_POS) >= 3 and _chunks(cells, PINNED_ROWS_POS) >= 2
    ptr = None
    for seqs, source in batches:
        ptr = kh.count_kmers(seqs, (k, source, sn), ptr)
    assert ptr.sizes[0] == U and ptr.kmer_count == U
    assert np.array_equal(kh.kmer_keys(ptr), keys)

    def matrix():
        a = np.empty((U, sn), np.int32)
        _lib.check(L.kmg_count_matrix(ptr._handle(), a.ctypes.data))
        return a

    m_before = matrix()
    assert np.array_equal(m_before, m)
    sentinel = torch.randint(-2**31, 2**31 - 1, (32 << 20,), dtype=torch.int32, device="cuda")
    sentinel_sha = hashlib.sha256(sentinel.cpu().numpy().tobytes()).hexdigest()
    small_seq = random_dna(300_000, 4242, p_n=0.001)
    small = kh.make_kmer_hash(small_seq, 21)
    small_before = kh.kmer_pos(small, 2 | 8)

    want = expected_kmer_pos(keys, m, k, 1 | 2)
    stride = k + 1
    kh.profile(enable=True, reset=True)
    try:
        dpos = torch.empty((cells, 2), dtype=torch.int32, device="cuda")
        _lib.check(L.kmg_count_positions(ptr._handle(), C.c_void_p(dpos.data_ptr())))
        torch.cuda.synchronize()
        assert kh.profile(reset=True)["count_rows"][1] == 1
        assert np.array_equal(dpos.cpu().numpy(), want["pos"])
        del dpos

        pin = kh.pinned_empty((cells, 2), np.int32)
        _lib.check(L.kmg_count_positions(ptr._handle(), pin.ctypes.data))
        assert kh.profile(reset=True)["count_rows"][1] == _chunks(cells, PINNED_ROWS_POS)
        assert np.array_equal(pin, want["pos"])
        del pin

        got = kh.kmer_pos(ptr, 2)["pos"]                   # pageable numpy
        assert kh.profile(reset=True)["count_rows"][1] == _chunks(cells, STAGE_ROWS_POS)
        assert np.array_equal(got, want["pos"])
        del got

        kmers = np.zeros((U, stride), np.uint8)
        kmers[:, :k] = want["kmer"]
        dk = torch.empty(U * stride, dtype=torch.uint8, device="cuda")
        _lib.check(L.kmg_count_kmers_ascii(ptr._handle(), C.c_void_p(dk.data_ptr())))
        torch.cuda.synchronize()
        assert kh.profile(reset=True)["kmers_ascii"][1] == 1
        assert np.array_equal(dk.cpu().numpy().reshape(U, stride), kmers)
        del dk
        pk = kh.pinned_empty(U * stride, np.uint8)
        _lib.check(L.kmg_count_kmers_ascii(ptr._handle(), pk.ctypes.data))
        assert kh.profile(reset=True)["kmers_ascii"][1] == _chunks(U * stride, 256 << 20) >= 2
        assert np.array_equal(pk.reshape(U, stride), kmers)
        del pk
        got = kh.kmer_pos(ptr, 1)["kmer"]                  # pageable numpy
        assert kh.profile(reset=True)["kmers_ascii"][1] == _chunks(U, (64 << 20) // stride) >= 3
        assert np.array_equal(got.view(np.uint8).reshape(U, k), want["kmer"])
        del got
    finally:
        kh.profile(enable=False, reset=True)
    assert np.array_equal(matrix(), m_before)
    assert hashlib.sha256(sentinel.cpu().numpy().tobytes()).hexdigest() == sentinel_sha
    small_after = kh.kmer_pos(small, 2 | 8)
    assert np.array_equal(small_after["pos"], small_before["pos"]) and np.array_equal(small_after["count"], small_before["count"])
    small.free(); ptr.free()


@pytest.mark.gpu
def test_large_count_table_through_the_r_glue(big):
    """.Call("count_kmers") batch by batch, then kmer.pos(ptr, 2) into the matrix R allocates (pageable): 73 M cells,
    nine staged chunks."""
    from rsession import RSession
    k, sn, batches, keys, m = big
    R = RSession()
    ptr = R.nil
    for seqs, source in batches:
        ptr = R.call("count_kmers", ptr, R.integer(k, source, sn), R.character(*seqs))
    got = R.kmer_pos(ptr, 2)
    assert got["pos"].shape == (len(keys) * sn, 2) and len(keys) * sn > 16_000_000
    assert np.array_equal(got["pos"][:, 1], m.ravel())
    assert np.array_equal(got["pos"][:, 0], np.repeat(np.arange(1, len(keys) + 1, dtype=np.int32), sn))
    assert got["kmer"] is None and got["pair.pos"] is None and got["count"] is None
    R.stub.rstub_finalize(ptr)
