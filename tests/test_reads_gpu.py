"""FASTA / FASTQ ingestion (SURVEY.md 8f rank 4): the device parser (csrc/reads.cuh) against the reference's own reader
(klib kseq.h over zlib, unmodified, through oracle/ref_fasta.c), then index builds and counts fed from the file."""
import gzip
import os

import numpy as np
import pytest

from conftest import random_dna


def _write_fasta(path, records, width, crlf=False, gz=False, blank=False):
    nl = "\r\n" if crlf else "\n"
    out = []
    for name, comment, seq in records:
        out.append(f">{name}{(' ' + comment) if comment else ''}{nl}")
        s = seq.tobytes().decode("latin-1")
        if width:
            for a in range(0, len(s), width):
                out.append(s[a:a + width] + nl)
            if blank:
                out.append(nl)
        else:
            out.append(s + nl)
    text = "".join(out).encode("latin-1")
    if text.endswith(b"\n") and not crlf and len(records) % 2 == 0:
        text = text[:-1]                                          # files without a final newline happen
    with (gzip.open if gz else open)(path, "wb") as fh:
        fh.write(text)
    return text


def _write_fastq(path, records, gz=False):
    rng = np.random.default_rng(1)
    out = []
    for name, comment, seq in records:
        q = bytes(rng.integers(33, 74, len(seq)).astype(np.uint8))
        q = b"@" + q[1:] if len(q) else q                        # a quality line may start with '@' or '>'
        out.append(b"@" + name.encode() + (b" " + comment.encode() if comment else b"") + b"\n" + seq.tobytes() + b"\n+\n" + q + b"\n")
    text = b"".join(out)
    with (gzip.open if gz else open)(path, "wb") as fh:
        fh.write(text)
    return text


def _records():
    from kmer_hasher_b200 import synth
    recs = [("chr1", "the first one", synth.config_c3(200_000, tail_k=21)),
            ("short", "", random_dna(15, 3)),                     # shorter than k: skipped by count.kmers
            ("exactk", "len == k", random_dna(21, 4)),
            ("scaf_2", "has\ttabs", random_dna(70_001, 5, p_n=0.002, p_lower=0.3)),
            ("quirk", "", np.concatenate([random_dna(500, 6), np.frombuffer(b"N", np.uint8), random_dna(21, 7)])),   # last run exactly k
            ("tail", "", random_dna(3_333, 8))]
    # a '\r' inside a sequence line is sequence (only a line's final '\r' is a line end): here never the last byte of a
    # line at the widths written (60, 80, one line), once the first byte of a 60-wide line
    recs[-1][2][[100, 120, 241]] = ord("\r")
    return recs


def test_reference_reader_reads_what_was_written(reference, tmp_path):
    """the kseq-based oracle itself, on files written here (CPU)"""
    recs = _records()
    for i, (kw, writer) in enumerate([(dict(width=60), _write_fasta), (dict(width=0, crlf=True), _write_fasta),
                                      (dict(width=80, gz=True, blank=True), _write_fasta), (dict(gz=False), _write_fastq),
                                      (dict(gz=True), _write_fastq)]):
        p = str(tmp_path / f"f{i}")
        writer(p, recs, **kw)
        names, seqs = reference.parse_reads(p)
        assert names == [r[0] for r in recs]
        assert seqs == [r[2].tobytes() for r in recs]


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["fa60", "fa_crlf_oneline", "fa_gz_blank", "fq", "fq_gz"])
def test_device_parser_matches_kseq(reference, tmp_path, fmt):
    import kmer_hasher_b200 as kh
    recs = _records()
    p = str(tmp_path / ("reads." + fmt))
    if fmt == "fa60":
        text = _write_fasta(p, recs, 60)
    elif fmt == "fa_crlf_oneline":
        text = _write_fasta(p, recs, 0, crlf=True)
    elif fmt == "fa_gz_blank":
        text = _write_fasta(p, recs, 80, gz=True, blank=True)
    else:
        text = _write_fastq(p, recs, gz=fmt.endswith("gz"))
    names, seqs = reference.parse_reads(p)
    sf = kh.SequenceFile(p)
    assert sf.n_records == len(names) and sf.total_bases == sum(len(s) for s in seqs)
    assert sf.names() == names
    for i, s in enumerate(seqs):
        assert sf.record(i)[1] == len(s) and sf.sequence(i) == s
    sf2 = kh.SequenceFile(np.frombuffer(text, np.uint8))           # the same from memory (already inflated)
    assert sf2.n_records == sf.n_records and sf2.sequence(3) == seqs[3]
    sf.free(); sf2.free()


@pytest.mark.gpu
def test_index_and_counts_from_a_file(reference, oracle, tmp_path):
    import kmer_hasher_b200 as kh
    recs = _records()
    p = str(tmp_path / "genome.fa.gz")
    _write_fasta(p, recs, 70, gz=True)
    k = 21
    # make.kmer.hash on a record of the file == make.kmer.hash on that sequence
    for rec in (0, "scaf_2"):
        seq = recs[0][2] if rec == 0 else recs[3][2]
        ix = kh.make_kmer_hash_file(p, k, record=rec)
        want = oracle.build(seq, k).extract(2 | 8)
        got = kh.kmer_pos(ix, 2 | 8, canonical=True)
        assert np.array_equal(kh.kmer_keys(ix, canonical=True), want["keys"])
        assert np.array_equal(got["count"], want["count"]) and np.array_equal(got["pos"].ravel(), want["pos"])
        ix.free()
    with pytest.raises(ValueError):
        kh.make_kmer_hash_file(p, k, record="short")
    # count.kmers over the whole file == the reference's count.kmers over the records' strings (short records skipped,
    # every record with its own end-of-string rule), and a second file into another column
    p2 = str(tmp_path / "reads.fq")
    recs2 = [(f"r{i}", "", random_dna(40 + 7 * i, 100 + i, p_n=0.01)) for i in range(300)]
    recs2[5] = ("r5", "", np.concatenate([random_dna(30, 9), np.frombuffer(b"n", np.uint8), random_dna(k, 10)]))
    _write_fastq(p2, recs2)
    ct = kh.count_kmers_file(p, (k, 0, 2))
    ct = kh.count_kmers_file(p2, (k, 1, 2), ct)
    ref = reference.count_kmers([r[2] for r in recs], k, 0, 2)
    ref = reference.count_kmers([r[2] for r in recs2], k, 1, 2, ref)
    want = ref.extract(2 | 8)
    got = kh.kmer_pos(ct, 2 | 8)
    assert ct.sizes[0] == ref.U and ct.kmer_count == ref.new_kmers
    assert np.array_equal(kh.kmer_keys(ct), want["keys"]) and np.array_equal(got["pos"].ravel(), want["pos"])
    ct.free(); ref.close()
    # through the R glue
    from rsession import RSession, RError
    R = RSession()
    ptr = R.call("make_kmer_h_index_file", R.character(p), R.integer(4), R.integer(k), R.integer(1))
    got = R.kmer_pos(ptr, 2 | 8)
    want = oracle.build(recs[3][2], k).extract(2 | 8)
    assert np.array_equal(got["pos"].ravel(), want["pos"]) and np.array_equal(got["count"], want["count"])
    with pytest.raises(RError, match="does not exist"):
        R.call("make_kmer_h_index_file", R.character(p), R.integer(99), R.integer(k), R.integer(0))
    cp = R.call("count_kmers_file", R.nil, R.integer(k, 0, 1), R.character(p2))
    ref = reference.count_kmers([r[2] for r in recs2], k, 0, 1)
    assert np.array_equal(R.kmer_pos(cp, 2)["pos"].ravel(), ref.extract(2)["pos"])
    R.stub.rstub_finalize(ptr); R.stub.rstub_finalize(cp)


@pytest.mark.gpu
def test_malformed_files_are_refused(tmp_path):
    import kmer_hasher_b200 as kh
    from kmer_hasher_b200 import KmgError
    for name, text in (("multi.fq", b"@r1\nACGT\nACGT\n+\nIIII\nIIII\n"), ("noheader.fa", b"ACGT\n>x\nACGT\n"),
                       ("qual.fq", b"@r1\nACGT\n+\nIII\n"), ("binary", b"\x1f\x00garbage")):
        p = str(tmp_path / name)
        open(p, "wb").write(text)
        with pytest.raises(KmgError):
            kh.SequenceFile(p)
    with pytest.raises(KmgError):
        kh.SequenceFile(str(tmp_path / "does_not_exist.fa"))
    open(str(tmp_path / "empty.fa"), "wb").write(b"")
    assert kh.SequenceFile(str(tmp_path / "empty.fa")).n_records == 0
