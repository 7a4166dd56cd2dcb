import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def oracle():
    from oracle import Oracle
    return Oracle()


@pytest.fixture(scope="session")
def reference():
    from oracle import Reference
    if not Reference.available():
        pytest.skip("reference engine oracle/_ref/libkmer_ref.so not built (make -C oracle REF=<kmer_hasheR checkout>)")
    return Reference()


@pytest.fixture(scope="session")
def test_fa():
    """The reference's test.fa (config 1 fixture), as one upper-case string of 59,940 bases."""
    with open(os.path.join(GOLDEN, "test_fa.seq")) as fh:
        return fh.read().strip()


@pytest.fixture(scope="session")
def golden():
    import json
    with open(os.path.join(GOLDEN, "golden.json")) as fh:
        return json.load(fh)


def sha(a) -> str:
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def random_dna(n, seed, p_n=0.0, p_lower=0.0, p_other=0.0, n_runs=0):
    """ACGT with optional isolated N/n, lower case, other IUPAC bytes and runs of N."""
    rng = np.random.default_rng(seed)
    s = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)].copy()
    if p_other:
        m = rng.random(n) < p_other
        s[m] = np.frombuffer(b"RYKMSWBDHVU-*", np.uint8)[rng.integers(0, 13, int(m.sum()))]
    if p_lower:
        m = rng.random(n) < p_lower
        s[m] |= 0x20
    if p_n:
        m = rng.random(n) < p_n
        s[m] = np.where(rng.random(int(m.sum())) < 0.5, ord("N"), ord("n"))
    for _ in range(n_runs):
        a = int(rng.integers(0, n))
        s[a:a + int(rng.integers(1, 200))] = ord("N")
    return s
