"""The device FASTA / FASTQ parser (csrc/reads.cuh) and counting from files, against what the test wrote.

What a test writes is itself the expected parse: names up to the first space or tab, sequences with the line ends
removed (test_reads_gpu.py::test_reference_reader_reads_what_was_written pins that reading against kseq).  Counts and
indexes built from a file are compared with the oracle restatement of the same records as strings.
"""
import numpy as np
import pytest

from conftest import random_dna
from test_counts_oracle_gpu import check_table, expected_counts
from test_reads_gpu import _records, _write_fasta, _write_fastq

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def kh():
    import kmer_hasher_b200 as kh
    return kh


def check_parse(sf, names, seqs, sample=None):
    """n_records, total_bases, names and record lengths of every record; the bases of every record (or of `sample`)."""
    assert sf.n_records == len(names)
    assert sf.total_bases == sum(len(s) for s in seqs)
    assert sf.names() == names
    assert [sf.record(i)[1] for i in range(sf.n_records)] == [len(s) for s in seqs]
    for i in range(len(seqs)) if sample is None else sample:
        assert sf.sequence(i) == seqs[i], i


def _write(fmt, path, recs):
    if fmt == "fa60":
        return _write_fasta(path, recs, 60)
    if fmt == "fa_crlf_oneline":
        return _write_fasta(path, recs, 0, crlf=True)
    if fmt == "fa_gz_blank":
        return _write_fasta(path, recs, 80, gz=True, blank=True)
    return _write_fastq(path, recs, gz=fmt.endswith("gz"))


@pytest.mark.parametrize("fmt", ["fa60", "fa_crlf_oneline", "fa_gz_blank", "fq", "fq_gz"])
def test_device_parser_reads_what_was_written(kh, tmp_path, fmt):
    recs = _records()
    p = str(tmp_path / ("reads." + fmt))
    text = _write(fmt, p, recs)
    names, seqs = [r[0] for r in recs], [r[2].tobytes() for r in recs]
    for src in (p, np.frombuffer(text, np.uint8)):         # the file, and the (inflated) text from memory
        sf = kh.SequenceFile(src)
        check_parse(sf, names, seqs)
        sf.free()


# (text, names, sequences): FASTA / FASTQ record edges
EDGES = [
    (b">a\n>b\nACGT\n", ["a", "b"], [b"", b"ACGT"]),                                   # a header right after a header
    (b">a\nACGT\n>b", ["a", "b"], [b"ACGT", b""]),                                     # last header without newline
    (b">a\nAC\nGT", ["a"], [b"ACGT"]),                                                 # no final newline
    (b">a x\nAC\n\nGT\n\n\n>b\tc\n\nTT\n\n", ["a", "b"], [b"ACGT", b"TT"]),               # blank lines between / inside
    (b">\n>\nAC\n", ["", ""], [b"", b"AC"]),                                           # empty names
    (b">a y\r\nAC\r\nGT\r\n>b\r\nTT\r\n", ["a", "b"], [b"ACGT", b"TT"]),                # CRLF throughout
    (b">a\r\nAC\r\r\nGT\r\n", ["a"], [b"AC\rGT"]),                                      # "\r\r\n": only the last '\r' goes
    (b">a\nAC\rGT\nT\rT\n\rA\n", ["a"], [b"AC\rGTT\rT\rA"]),                             # interior '\r' in sequence lines
    (b">a\nACGT\r", ["a"], [b"ACGT"]),                                                 # a final '\r' with no '\n'
    (b"@r1 c\r\nACGT\r\n+\r\nIIII\r\n@r2\r\nA\rG\r\n+\r\nIII\r\n", ["r1", "r2"], [b"ACGT", b"A\rG"]),   # CRLF FASTQ
]


def test_record_edges(kh, tmp_path):
    for j, (text, names, seqs) in enumerate(EDGES):
        p = str(tmp_path / f"edge{j}")
        with open(p, "wb") as fh:
            fh.write(text)
        for src in (p, np.frombuffer(text, np.uint8)):
            sf = kh.SequenceFile(src)
            check_parse(sf, names, seqs)
            sf.free()
    # the same records again inside larger text: the packed buffer comes from reused (not zeroed) device memory, so
    # a byte the parser counts but does not write shows up as a wrong base
    big = random_dna(3_000_000, 77).tobytes()
    for text, names, seqs in EDGES[6:8]:
        sf = kh.SequenceFile(np.frombuffer(text + b">pad\n" + big + b"\n", np.uint8))
        check_parse(sf, names + ["pad"], seqs + [big])
        sf.free()


def test_tile_and_size_edges(kh, tmp_path):
    """Text over many 16 KiB nl_scan tiles with lines across tile boundaries (width 61) and many 2048-line line_scan
    tiles; one 20 Mbp single-line record; 200 k FASTQ reads; text over 8 MiB from pageable memory (staged upload) and
    as a device tensor (names read from device memory)."""
    import torch
    rng = np.random.default_rng(5)
    recs = [(f"s{i}", "c", random_dna(int(rng.integers(1, 40_000)), 500 + i, p_n=0.001, p_lower=0.1)) for i in range(60)]
    p = str(tmp_path / "tiles.fa")
    text = _write_fasta(p, recs, 61)
    assert len(text) > 20 * 16384 and text.count(b"\n") > 5 * 2048
    sf = kh.SequenceFile(p)
    check_parse(sf, [r[0] for r in recs], [r[2].tobytes() for r in recs])
    sf.free()

    long = random_dna(20_000_000, 6, p_n=0.0001)
    p = str(tmp_path / "long.fa")
    text = _write_fasta(p, [("chrL", "one line", long), ("after", "", long[:1000].copy())], 0)
    for src in (p, np.frombuffer(text, np.uint8), torch.from_numpy(np.frombuffer(text, np.uint8).copy()).cuda()):
        sf = kh.SequenceFile(src)
        check_parse(sf, ["chrL", "after"], [long.tobytes(), long[:1000].tobytes()])
        sf.free()

    n = 200_000
    lens = rng.integers(50, 151, n)
    pool = random_dna(int(lens.sum()), 9, p_n=0.002)
    offs = np.concatenate([[0], np.cumsum(lens)])
    reads = [(f"read{i}", "x" if i % 3 == 0 else "", pool[offs[i]:offs[i + 1]]) for i in range(n)]
    p = str(tmp_path / "reads.fq")
    text = _write_fastq(p, reads)
    assert len(text) > (8 << 20)
    names, seqs = [r[0] for r in reads], [r[2].tobytes() for r in reads]
    sample = sorted(set(rng.integers(0, n, 300).tolist()) | {0, 1, n // 2, n - 1})
    for src in (p, np.frombuffer(text, np.uint8), torch.from_numpy(np.frombuffer(text, np.uint8).copy()).cuda()):
        sf = kh.SequenceFile(src)                          # file; pageable text over 8 MiB; device text
        check_parse(sf, names, seqs, sample)
        sf.free()


def _counting_records(k, seed):
    """Records at the edges mask_for_counting_kernel handles: length <= k, exactly k+1, k+1 with a leading N, a last
    N-free run of exactly k and of exactly k+1, all N, empty."""
    N, n = np.frombuffer(b"N", np.uint8), np.frombuffer(b"n", np.uint8)
    r = lambda L, s: random_dna(L, seed * 100 + s)
    return [("mixed", "", random_dna(60_000, seed, p_n=0.002, p_lower=0.3, p_other=0.01, n_runs=4)),
            ("short", "", r(max(1, k - 1), 1)), ("exact_k", "", r(k, 2)), ("k_plus_1", "", r(k + 1, 3)),
            ("N_k", "", np.concatenate([N, r(k, 4)])), ("empty", "", np.empty(0, np.uint8)),
            ("run_k", "", np.concatenate([r(40, 5), N, r(k, 6)])), ("run_k1", "", np.concatenate([r(40, 7), n, r(k + 1, 8)])),
            ("allN", "", np.full(k + 5, ord("N"), np.uint8)), ("alln", "", np.full(2 * k + 3, ord("n"), np.uint8)),
            ("k_plus_1b", "", r(k + 1, 9)), ("last", "", np.concatenate([r(3_000, 10), N, r(k, 11)]))]


@pytest.mark.parametrize("k", [1, 12, 21, 32])
def test_count_kmers_file_matches_the_restatement(kh, tmp_path, k):
    recs = _counting_records(k, 31 + k)
    recs2 = [(f"q{i}", "", random_dna(k + 1 + 13 * i, 700 + i, p_n=0.01)) for i in range(150)] + \
            [(f"z{i}", "", r[2]) for i, r in enumerate(_counting_records(k, 90 + k)) if len(r[2])]
    p, p2 = str(tmp_path / "a.fa"), str(tmp_path / "b.fq")
    _write_fasta(p, recs, 70)
    _write_fastq(p2, recs2)
    sn = 3
    ct = kh.count_kmers_file(p, (k, 2, sn))
    keys, m = expected_counts([([r[2] for r in recs], 2)], k, sn)
    check_table(kh, ct, keys, m, k)
    ct = kh.count_kmers_file(p2, (k, 0, sn), ct)          # a second file into another column
    keys, m = expected_counts([([r[2] for r in recs], 2), ([r[2] for r in recs2], 0)], k, sn)
    check_table(kh, ct, keys, m, k)
    ct.free()


def test_index_of_a_file_record(kh, oracle, tmp_path):
    """make_kmer_hash_file on the first, a middle and the last record == make.kmer.hash of the same string."""
    recs = _records()
    p = str(tmp_path / "genome.fa.gz")
    _write_fasta(p, recs, 70, gz=True)
    for k in (12, 21, 32):
        for rec in (0, 3, len(recs) - 1):
            seq = recs[rec][2]
            ix = kh.make_kmer_hash_file(p, k, record=rec if rec else recs[0][0])
            want = oracle.build(seq, k).extract(2 | 8)
            got = kh.kmer_pos(ix, 2 | 8, canonical=True)
            assert np.array_equal(kh.kmer_keys(ix, canonical=True), want["keys"])
            assert np.array_equal(got["count"], want["count"]) and np.array_equal(got["pos"].ravel(), want["pos"])
            ix.free()
