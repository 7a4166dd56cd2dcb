"""The 32-bit edges: an index of 2^31 - 1 windows, probes whose index positions and query ends lie near 2^31, and row
streams whose 64-bit row numbers pass 2^32 -- every output compared in full, on the device.

The reference for the large cases is a restatement in plain int64 torch, independent of the library's kernels:

  window_keys     the 2-bit key ((c >> 1) & 3, first base most significant) of every window and its validity: no N/n
                  inside (a cumulative sum of breakers, not a loop over k) and not the end-of-string rule's window (a
                  final N-free run of exactly k bases loses its window, SURVEY.md A.3)
  check_index     a complete check of an index in its own order: rows grouped by i with counts as the list lengths,
                  positions ascending inside each k-mer, the positions exactly the valid windows (each once), every row's
                  window key equal to its k-mer's key, the keys distinct, and (U, N, P) as kmg_sizes reports them; these
                  pin the index down uniquely.  It returns the verified index in ascending key order (`Verified`)
  expected_rows   the seq.kmer.pos rows of a query, from the verified index by searchsorted + repeat_interleave; with it
                  the depth on one and both strands, the join rows of two verified indexes, and the diagonal runs

The restatement is checked against the plain-C oracle at a few hundred kb (CPU tests, no GPU), and the checker against
deliberately corrupted arrays, which it must reject naming the row.  Where the inputs are homopolymers every output has a
closed form, computed in Python integers.  Everything works in slices of 2^26 rows so that temporaries stay bounded.
"""
import ctypes as C
import time

import numpy as np
import pytest
import torch

from conftest import random_dna
from test_chains_gpu import chains_of
from test_dotplot_gpu import IUPAC, host_revcomp
from test_join_segments_gpu import anti_runs, revcomp_keys
from test_segments_gpu import runs_of

INT32_MAX = 2**31 - 1
SIGN = -2**63                      # xor with it turns the unsigned order of 64-bit keys into the signed one
SLICE = 1 << 26
NA = -2**31
KMG_ERR_RANGE = -3


def _first_bad(ok, base=0):
    """None when the bool tensor `ok` holds everywhere, else base + the index of its first False."""
    if bool(ok.all()):
        return None
    return base + int(torch.nonzero(~ok)[0, 0])


def _require(ok, base, what):
    bad = _first_bad(ok, base)
    assert bad is None, f"{what}: row {bad}"


def _is_breaker(b):
    return (b | 0x20) == ord("n")


# ---- the restatement ------------------------------------------------------------------------------------------------
def window_keys(seq, k):
    """(keys, valid) of every window start 0 .. len(seq) - k of the uint8 tensor seq: int64 2-bit keys (the unsigned key's
    bits) and whether make.kmer.hash emits the window."""
    L = seq.numel()
    n = L - k + 1
    dev = seq.device
    keys = torch.empty(max(n, 0), dtype=torch.int64, device=dev)
    valid = torch.empty(max(n, 0), dtype=torch.bool, device=dev)
    for a in range(0, n, SLICE):
        b = min(n, a + SLICE)
        part = seq[a:b + k - 1]
        code = ((part >> 1) & 3).to(torch.int64)
        w = torch.zeros(b - a, dtype=torch.int64, device=dev)
        for t in range(k):
            w = (w << 2) | code[t:t + b - a]
        keys[a:b] = w
        del code, w
        cs = torch.zeros(part.numel() + 1, dtype=torch.int32, device=dev)
        cs[1:] = torch.cumsum(_is_breaker(part).to(torch.int32), 0, dtype=torch.int32)
        valid[a:b] = cs[k:k + b - a] == cs[:b - a]
        del cs
    if n >= 1 and bool(valid[n - 1]) and (n == 1 or bool(_is_breaker(seq[n - 2]))):
        valid[n - 1] = False                                   # freshly primed and ending at the terminator
    return keys, valid


def revcomp_keys_t(keys, k):
    """Code-space reverse complement of int64 keys: the k codes reversed, each code ^ 2."""
    out = torch.zeros_like(keys)
    for t in range(k):
        out = (out << 2) | (((keys >> (2 * t)) & 3) ^ 2)
    return out


class Verified:
    """An index checked by check_index, held in ascending key order: skf = key ^ SIGN (ascending as int64), sstart and
    scount = where each k-mer's positions begin in `pos` (the index's own row order) and how many there are."""

    def __init__(self, k, skf, sstart, scount, pos, sizes, snum=None):
        self.k, self.skf, self.sstart, self.scount, self.pos, self.sizes = k, skf, sstart, scount, pos, sizes
        self.snum = snum                                       # with keep_order: each k-mer's number in the index's order

    def lookup(self, keys):
        """(hit, u): whether each key is in the index and, where it is, its rank."""
        U = self.skf.numel()
        kf = keys ^ SIGN
        u = torch.searchsorted(self.skf, kf).clamp_(max=max(U - 1, 0))
        hit = self.skf[u] == kf if U else torch.zeros_like(kf, dtype=torch.bool)
        return hit, u


def check_index(seq, k, arrays, sorted_build, wk=None, valid=None, keep_order=False):
    """Assert that arrays = {keys: [U] int64, pos: [N, 2] int32 rows (i, pos), counts: [U] int32, sizes: (U, N, P) of
    kmg_sizes}, an index in its own order, is the index of the windows of `seq` at k.  Returns a Verified.  The arrays are
    taken out of the dict, so that they are freed as soon as they are no longer needed.  keep_order: also keep each k-mer's
    number in the index's own order (kmer.pairs walks its first index in that order)."""
    keys, pos, counts, sizes = (arrays.pop(n) for n in ("keys", "pos", "counts", "sizes"))
    dev = keys.device
    U, N, P = sizes
    assert keys.numel() == U and counts.numel() == U and tuple(pos.shape) == (N, 2), "array sizes differ from (U, N)"
    if wk is None:
        wk, valid = window_keys(seq, k)
    nst = wk.numel()
    _require(counts >= 1, 0, "a k-mer without positions (k-mer number)")
    ends = torch.cumsum(counts, 0, dtype=torch.int64)
    assert int(ends[-1]) == N if U else N == 0, f"counts sum to {int(ends[-1]) if U else 0}, not N = {N}"
    assert P == int(sum(int((c * (c - 1)).sum()) for c in (counts[a:a + SLICE].to(torch.int64) for a in range(0, U, SLICE)))) // 2, "P"
    ends = ends.to(torch.int32)                                # <= N <= INT32_MAX
    seen = torch.zeros(nst, dtype=torch.bool, device=dev)
    for a in range(0, N, SLICE):
        b = min(N, a + SLICE)
        i, p = pos[a:b, 0], pos[a:b, 1]
        u = torch.searchsorted(ends, torch.arange(a, b, device=dev, dtype=torch.int32), right=True, out_int32=True)
        _require(i == u + 1, a, "rows not grouped by k-mer number or a count differs from its list length")
        del u
        _require((p >= 1) & (p <= nst), a, "position outside the sequence")
        lo = max(a - 1, 0)
        ii, pp = pos[lo:b, 0], pos[lo:b, 1]
        _require((ii[1:] != ii[:-1]) | (pp[1:] > pp[:-1]), lo + 1, "positions not ascending inside a k-mer")
        w = (p - 1).to(torch.int64)
        _require(valid[w], a, "position of a window make.kmer.hash does not emit")
        _require(wk[w] == keys[(i - 1).to(torch.int64)], a, "window key differs from the k-mer's key")
        seen[w] = True
        del w
    assert int(valid.sum()) == N, f"{int(valid.sum())} valid windows, N = {N}"
    for a in range(0, nst, SLICE):
        _require(seen[a:a + SLICE] == valid[a:a + SLICE], a, "valid window missing from the positions (window)")
    del seen
    posj = pos[:, 1].clone()
    del pos
    starts = ends - counts
    del ends
    if sorted_build:
        for a in range(0, U, SLICE):
            kf = keys[max(a - 1, 0):a + SLICE] ^ SIGN
            _require(kf[1:] > kf[:-1], max(a - 1, 0) + 1, "keys not strictly ascending (k-mer number)")
        return Verified(k, keys ^ SIGN, starts, counts, posj, sizes,
                        torch.arange(U, device=dev, dtype=torch.int32) if keep_order else None)
    # grouped: sort by key one bucket of the top four key bits at a time (bounded temporaries), then strictly ascending
    skf = torch.empty_like(keys)
    sstart, scount = torch.empty_like(counts), torch.empty_like(counts)
    snum = torch.empty_like(counts) if keep_order else None
    shift = max(2 * k - 4, 0)
    bucket = torch.empty(U, dtype=torch.uint8, device=dev)
    for a in range(0, U, SLICE):
        bucket[a:a + SLICE] = ((keys[a:a + SLICE] >> shift) & 15).to(torch.uint8)
    at = 0
    for v in range(16):
        idx = torch.nonzero(bucket == v).flatten()
        if idx.numel() == 0:
            continue
        s, o = torch.sort(keys[idx] ^ SIGN)
        _require(s[1:] > s[:-1], at + 1, "duplicated key (rank)")
        idx = idx[o]
        m = idx.numel()
        skf[at:at + m], sstart[at:at + m], scount[at:at + m] = s, starts[idx], counts[idx]
        if keep_order:
            snum[at:at + m] = idx.to(torch.int32)
        at += m
        del idx, s, o
    assert at == U
    del keys, counts, starts, bucket
    return Verified(k, skf, sstart, scount, posj, sizes, snum)


def expected_rows(qkeys, qvalid, k, ix: Verified):
    """(M, 2) int32 rows (i, j) of seq.kmer.pos: i = 1-based end of the query window, j = the k-mer's positions in
    ascending order, rows ordered by (i, j)."""
    hit, u = ix.lookup(qkeys)
    hit &= qvalid
    c = torch.where(hit, ix.scount[u], 0).to(torch.int64)
    M = int(c.sum())
    w = torch.nonzero(c).flatten()
    cw, uw = c[w], u[w]
    del c, hit, u
    first = torch.cumsum(cw, 0) - cw
    rows = torch.empty((M, 2), dtype=torch.int32, device=qkeys.device)
    rows[:, 0] = torch.repeat_interleave(w + k, cw).to(torch.int32)
    src = torch.repeat_interleave(ix.sstart[uw].to(torch.int64) - first, cw) + torch.arange(M, device=qkeys.device)
    rows[:, 1] = ix.pos[src]
    return rows


def expected_depth(qkeys, qvalid, k, ix: Verified, both):
    """seq.kmer.depth of an index: the count of each window's k-mer (0 when absent), with `both` plus its reverse
    complement's (once for a palindrome), saturated at INT32_MAX; NA where the window is not emitted."""
    hit, u = ix.lookup(qkeys)
    d = torch.where(hit, ix.scount[u], 0).to(torch.int64)
    if both:
        rk = revcomp_keys_t(qkeys, k)
        hit, u = ix.lookup(rk)
        d += torch.where(hit & (rk != qkeys), ix.scount[u], 0)
    return torch.where(qvalid, d.clamp(max=INT32_MAX), NA).to(torch.int32)


def join_rows(a: Verified, b: Verified, rc=False):
    """(M, 2) int32 rows (x, y) of kmer.pairs(a, b): for every k-mer of a (with rc: its reverse complement) that b holds,
    each position in a paired with each position in b, x outer, y inner; a's k-mers in a's own order when a was verified
    with keep_order, else in ascending key order."""
    bkeys = b.skf ^ SIGN
    ak = revcomp_keys_t(bkeys, b.k) if rc else bkeys           # the key of a that pairs with each key of b
    hit, ua = a.lookup(ak)
    del ak
    vb = torch.nonzero(hit).flatten()
    ua = ua[vb]
    if a.snum is not None or rc:                               # order the shared keys by a's k-mer number or a's rank
        o = torch.argsort(a.snum[ua] if a.snum is not None else ua)
        ua, vb = ua[o], vb[o]
    ca, cb = a.scount[ua].to(torch.int64), b.scount[vb].to(torch.int64)
    cnt = ca * cb
    M = int(cnt.sum())
    first = torch.cumsum(cnt, 0) - cnt
    g = torch.repeat_interleave(torch.arange(len(cnt), device=cnt.device), cnt)
    t = torch.arange(M, device=cnt.device) - first[g]
    rows = torch.empty((M, 2), dtype=torch.int32, device=cnt.device)
    rows[:, 0] = a.pos[a.sstart[ua].to(torch.int64)[g] + t // cb[g]]
    rows[:, 1] = b.pos[b.sstart[vb].to(torch.int64)[g] + t % cb[g]]
    return rows


def runs_dev(rows, anti=False):
    """(R, 3) int64 (i, j, n): the maximal runs (i + t, j + t) -- anti: (i + t, j - t) -- of the (M, 2) rows, first row the
    smallest i, ordered by (i, j).  Diagonal keys i - j + 2^31 and i + j are below 2^32, i below 2^31: key * 2^31 + i fits."""
    i = rows[:, 0].to(torch.int64)
    j = rows[:, 1].to(torch.int64)
    d = i + j if anti else i - j + 2**31
    key = torch.sort(d * 2**31 + i).values
    del d, j
    d, i = key >> 31, key & (2**31 - 1)
    del key
    head = torch.ones(len(d), dtype=torch.bool, device=d.device)
    head[1:] = (d[1:] != d[:-1]) | (i[1:] != i[:-1] + 1)
    at = torch.nonzero(head).flatten()
    n = torch.diff(torch.cat([at, torch.tensor([len(d)], device=d.device)]))
    i0, d0 = i[at], d[at]
    j0 = d0 - i0 if anti else i0 - d0 + 2**31
    o = torch.sort(i0 * 2**31 + j0).indices
    return torch.stack([i0[o], j0[o], n[o]], 1)


def bin_counts(x, y, xr, nx, yr, ny):
    """float64 nx * ny image (column-major, flattened) of the points (x, y) in the half-open windows: bin
    floor((v - lo) * n / (hi - lo)) in int64."""
    (x0, x1), (y0, y1) = xr, yr
    x, y = x.to(torch.int64), y.to(torch.int64)
    keep = (x >= x0) & (x < x1) & (y >= y0) & (y < y1)
    bx = (x[keep] - x0) * nx // (x1 - x0)
    by = (y[keep] - y0) * ny // (y1 - y0)
    return torch.bincount(bx + by * nx, minlength=nx * ny).to(torch.float64)


def assert_rows_equal(got, want, what="rows", base=0):
    """Complete comparison of two row arrays (torch), naming the first differing row."""
    assert tuple(got.shape) == tuple(want.shape), f"{what}: shape {tuple(got.shape)} != {tuple(want.shape)}"
    eq = (got == want)
    if eq.dim() > 1:
        eq = eq.all(1)
    bad = _first_bad(eq, base)
    if bad is not None:
        r = bad - base
        raise AssertionError(f"{what}: row {bad} is {got[r].tolist()}, expected {want[r].tolist()}")


def unrank_pair(t, n):
    """Pair t (0-based) of a list of n positions enumerated (0,1),(0,2)..(0,n-1),(1,2)..: (a, b) in Python integers.
    Rows before first index j: S(j) = j(2n - j - 1)/2."""
    lo, hi = 0, n - 2
    while lo < hi:                                             # the last j with S(j) <= t
        mid = (lo + hi + 1) // 2
        if mid * (2 * n - mid - 1) // 2 <= t:
            lo = mid
        else:
            hi = mid - 1
    return lo, lo + 1 + t - lo * (2 * n - lo - 1) // 2


def _mutated(src, rng):
    """src with a substitution every 100-200 bases and a few 1-3 base indels."""
    out, p, ev, ln = [], 0, 0, len(src)
    indels = set(rng.choice(np.arange(5, ln // 150), 6, replace=False).tolist())
    nxt = int(rng.integers(100, 200))
    while p < ln:
        if nxt > p:
            out.append(src[p:min(nxt, ln)]); p = min(nxt, ln)
            continue
        if ev in indels and p + 3 < ln:
            L = int(rng.integers(1, 4))
            if rng.integers(0, 2):
                out.append(np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, L)])
            else:
                p += L
        else:
            c = src[p] & 0xDF
            out.append(np.array([ord("A") if c != ord("A") else ord("C")], np.uint8))
            p += 1
        ev += 1
        nxt = p + int(rng.integers(100, 200))
    return np.concatenate(out)


# ---- CPU: the restatement against the oracle, and the checker against corrupted arrays -------------------------------
def _cpu_inputs():
    """A few hundred kb with isolated and run N/n, lower case, IUPAC bytes, and the end-of-string cases of
    test_tile_boundaries (a final run of exactly k, of k + 1, breakers at both ends)."""
    s = random_dna(300_000, 71, p_n=0.002, p_lower=0.1, p_other=0.002, n_runs=5)
    return np.concatenate([s, s[1_000:3_000], np.frombuffer(b"CA" * 300, np.uint8), s[50_000:50_400], s[1_500:2_200],
                           random_dna(5_000, 72)])


def _oracle_arrays(oracle, seq, k, permute_seed=None):
    """(keys, pos, counts, sizes) of the oracle's index as torch tensors; with permute_seed the k-mers in a random order
    (i renumbered, rows regrouped), as a grouped build would hold them."""
    o = oracle.build(seq, k)
    e = o.extract(2 | 8)
    keys = torch.from_numpy(e["keys"].view(np.int64).copy())
    cnt = torch.from_numpy(e["count"].copy())
    pos = torch.from_numpy(e["pos"].reshape(-1, 2).copy())
    if permute_seed is not None:
        U = len(keys)
        perm = torch.from_numpy(np.random.default_rng(permute_seed).permutation(U))
        rank = torch.empty_like(perm)
        rank[perm] = torch.arange(U)
        new_i = rank[pos[:, 0].to(torch.int64) - 1]
        order = torch.sort(new_i, stable=True).indices
        pos = torch.stack([new_i[order].to(torch.int32) + 1, pos[order, 1]], 1)
        keys, cnt = keys[perm], cnt[perm]
    return dict(keys=keys, pos=pos, counts=cnt, sizes=(o.U, o.N, o.P))


@pytest.mark.parametrize("k", [1, 5, 15, 16, 31, 32])
def test_window_keys_match_oracle(oracle, k):
    s = _cpu_inputs()
    variants = [s, s.copy(), s.copy(), s.copy()]
    variants[1][0], variants[1][-1] = ord("N"), ord("n")
    variants[2][len(s) - k - 1] = ord("N")                     # final run of exactly k: its window dropped
    variants[3][len(s) - k - 2] = ord("N")                     # final run of k + 1: two windows, both kept
    for t in variants + [np.frombuffer(b"acgt" * 3, np.uint8)[:k + 1].copy()]:
        if len(t) <= k:
            continue
        keys, valid = window_keys(torch.from_numpy(t), k)
        ok, op = oracle.windows(t, k)
        w = torch.nonzero(valid).flatten().numpy()
        assert np.array_equal(w + 1, op)
        assert np.array_equal(keys.numpy()[w].view(np.uint64), ok)
    if k >= 2:
        t = variants[2]
        assert not bool(window_keys(torch.from_numpy(t), k)[1][-1])


@pytest.mark.parametrize("k", [5, 15, 32])
def test_check_index_accepts_the_oracle_index(oracle, k):
    s = _cpu_inputs()
    st = torch.from_numpy(s)
    want = oracle.build(s, k).extract(2 | 8)
    for seed in (None, 3):
        v = check_index(st, k, _oracle_arrays(oracle, s, k, seed), sorted_build=seed is None)
        assert np.array_equal((v.skf ^ SIGN).numpy().view(np.uint64), want["keys"])
        assert np.array_equal(v.scount.numpy(), want["count"])
        rows = want["pos"].reshape(-1, 2)[:, 1]
        c = v.scount.to(torch.int64)
        src = torch.repeat_interleave(v.sstart.to(torch.int64) - (torch.cumsum(c, 0) - c), c) + torch.arange(int(c.sum()))
        assert np.array_equal(v.pos[src].numpy(), rows)


@pytest.mark.parametrize("k", [9, 15, 32])
def test_expected_rows_and_depth_match_oracle(oracle, k):
    s = _cpu_inputs()
    q = np.concatenate([s[100_000:160_000], random_dna(20_000, 5, p_n=0.001), _mutated(s[200_000:260_000],
                                                                                         np.random.default_rng(1))])
    o = oracle.build(s, k)
    v = check_index(torch.from_numpy(s), k, _oracle_arrays(oracle, s, k, 9), sorted_build=False)
    for rc in (False, True):
        qq = np.frombuffer(host_revcomp(q), np.uint8) if rc else q
        qk, qv = window_keys(torch.from_numpy(qq.copy()), k)
        rows = expected_rows(qk, qv, k, v)
        assert np.array_equal(rows.numpy().ravel(), o.query(qq, k))
        assert np.array_equal(runs_dev(rows).numpy(), runs_of(rows.numpy()))
    from test_depth_gpu import expected_depth as depth_np
    e = o.extract(2 | 8)
    qk, qv = window_keys(torch.from_numpy(q), k)
    for both in (False, True):
        assert np.array_equal(expected_depth(qk, qv, k, v, both).numpy(), depth_np(e["keys"], e["count"], q, k, both)[:, 0])


@pytest.mark.parametrize("k", [9, 15])
def test_join_rows_match_oracle(oracle, k):
    import oracle as oracle_mod
    from test_join_segments_gpu import rc_extraction
    s = _cpu_inputs()
    q = np.concatenate([s[50_000:90_000], np.frombuffer(host_revcomp(s[150_000:170_000]), np.uint8), random_dna(10_000, 2)])
    va = check_index(torch.from_numpy(s), k, _oracle_arrays(oracle, s, k, 4), sorted_build=False)
    vb = check_index(torch.from_numpy(q), k, _oracle_arrays(oracle, q, k), sorted_build=True)
    ea, eb = oracle.build(s, k).extract(2 | 8), oracle.build(q, k).extract(2 | 8)
    assert np.array_equal(join_rows(va, vb).numpy().ravel(), oracle_mod.pairs_join(ea, eb))
    rc = join_rows(va, vb, rc=True)
    want = oracle_mod.pairs_join(rc_extraction(ea, k), eb)
    assert len(want) > 1000 and np.array_equal(rc.numpy().ravel(), want)
    assert np.array_equal(runs_dev(rc, anti=True).numpy(), anti_runs(want))
    # a in its own (permuted) k-mer order, as kmer.pairs walks a grouped index
    arr = _oracle_arrays(oracle, s, k, 4)
    own = dict(keys=arr["keys"].numpy().view(np.uint64), count=arr["counts"].numpy(), pos=arr["pos"].numpy().ravel())
    vo = check_index(torch.from_numpy(s), k, arr, sorted_build=False, keep_order=True)
    assert np.array_equal(join_rows(vo, vb).numpy().ravel(), oracle_mod.pairs_join(own, eb))
    assert np.array_equal(join_rows(vo, vb, rc=True).numpy().ravel(), oracle_mod.pairs_join(rc_extraction(own, k), eb))


def test_revcomp_and_unranking_restatements():
    rng = np.random.default_rng(2)
    keys = rng.integers(0, 2**63, 1000, dtype=np.int64)
    for k in (1, 7, 31, 32):
        kk = keys & ((1 << (2 * k)) - 1) if k < 32 else keys
        got = revcomp_keys_t(torch.from_numpy(kk), k).numpy().view(np.uint64)
        assert np.array_equal(got, revcomp_keys(kk.view(np.uint64), k))
    for n in (2, 3, 7, 50):
        pairs = [(a, b) for a in range(n) for b in range(a + 1, n)]
        assert [unrank_pair(t, n) for t in range(len(pairs))] == pairs


def _corrupt_cases(keys, pos, cnt, sizes, k):
    """(name, keys, pos, counts, sizes) of one corruption each."""
    U, N, P = sizes
    c = cnt.to(torch.int64)
    u2 = int(torch.nonzero(c >= 2)[len(torch.nonzero(c >= 2)) // 2, 0])     # a k-mer with several positions
    r2 = int(torch.cumsum(c, 0)[u2] - c[u2])                                    # its first row
    r = N // 2
    out = []
    p = pos.clone(); p[r, 1] += 1
    out.append(("position off by one", keys, p, cnt, sizes))
    p = pos.clone(); p[[r2, r2 + 1], 1] = p[[r2 + 1, r2], 1]
    out.append(("two rows of one k-mer swapped", keys, p, cnt, sizes))
    kk = keys.clone(); kk[U // 3] = kk[U // 3 + 1]
    out.append(("duplicated key", kk, pos, cnt, sizes))
    cc = cnt.clone(); cc[u2] += 1; cc[u2 + 1] -= 1 if int(cc[u2 + 1]) > 1 else 0
    out.append(("count off by one", keys, pos, cc, (U, N, P) if int(cc.sum()) == N else sizes))
    cc = cnt.clone(); cc[u2] -= 1; cc[u2 - 1] += 1
    out.append(("count off by one, the sum kept", keys, pos, cc, sizes))
    p = pos.clone(); p[r, 1] ^= -2**31
    out.append(("position bit 31 flipped", keys, p, cnt, sizes))
    p = pos.clone(); p[r, 0] ^= -2**31
    out.append(("k-mer number bit 31 flipped", keys, p, cnt, sizes))
    kk = keys.clone(); kk[U // 2] ^= 1 << 32 if k > 16 else 1 << 31
    out.append(("key bit 32 (31) flipped", kk, pos, cnt, sizes))
    out.append(("N off by one", keys, pos[:-1], cnt, (U, N - 1, P)))
    out.append(("P off by one", keys, pos, cnt, (U, N, P + 1)))
    return out


@pytest.mark.parametrize("k", [11, 32])
@pytest.mark.parametrize("grouped", [False, True])
def test_checker_rejects_corrupted_indexes(oracle, k, grouped):
    s = _cpu_inputs()
    st = torch.from_numpy(s)
    base = _oracle_arrays(oracle, s, k, 8 if grouped else None)
    check_index(st, k, dict(base), sorted_build=not grouped)
    wk, valid = window_keys(st, k)
    for name, keys, pos, cnt, sizes in _corrupt_cases(base["keys"], base["pos"], base["counts"], base["sizes"], k):
        with pytest.raises(AssertionError) as e:
            check_index(st, k, dict(keys=keys, pos=pos, counts=cnt, sizes=sizes), sorted_build=not grouped, wk=wk, valid=valid)
        msg = str(e.value)
        assert "row" in msg or "N =" in msg or msg.startswith("P") or "sizes" in msg, (name, msg)


def test_row_comparison_rejects_corrupted_rows(oracle):
    k = 15
    s = _cpu_inputs()
    v = check_index(torch.from_numpy(s), k, _oracle_arrays(oracle, s, k), sorted_build=True)
    qk, qv = window_keys(torch.from_numpy(s[:80_000].copy()), k)
    want = expected_rows(qk, qv, k, v)
    M = len(want)
    assert_rows_equal(want.clone(), want)
    r = M // 2
    same_i = torch.nonzero(want[1:, 0] == want[:-1, 0]).flatten()
    cases = []
    g = want.clone(); g[r, 1] += 1; cases.append(g)
    g = want.clone(); g[r, 0] -= 1; cases.append(g)
    t = int(same_i[len(same_i) // 2])
    g = want.clone(); g[[t, t + 1]] = g[[t + 1, t]]; cases.append(g)
    g = want.clone(); g[r, 1] ^= -2**31; cases.append(g)
    g = want.clone(); g[r, 0] ^= 1 << 30; cases.append(g)
    for g in cases:
        with pytest.raises(AssertionError, match=r"row \d+"):
            assert_rows_equal(g, want)
    with pytest.raises(AssertionError, match="shape"):
        assert_rows_equal(want[:-1], want)
    # depth and images: one value off
    d = expected_depth(qk, qv, k, v, True)
    e = d.clone(); e[len(e) // 3] += 1
    with pytest.raises(AssertionError, match=r"row \d+"):
        assert_rows_equal(e, d, "depth")
    runs = runs_dev(want)
    rr = runs.clone(); rr[len(rr) // 2, 2] += 2**32
    with pytest.raises(AssertionError, match=r"row \d+"):
        assert_rows_equal(rr, runs, "runs")


# ---- on the GPU ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def kh():
    import kmer_hasher_b200 as kh
    return kh


def _L():
    from kmer_hasher_b200 import _lib
    return _lib, _lib.load()


def _log(what, t0):
    torch.cuda.synchronize()
    print(f"  {what}: {time.time() - t0:.1f} s, peak {torch.cuda.max_memory_allocated() / 2**30:.1f} GiB allocated by torch, "
          f"{torch.cuda.mem_get_info()[0] / 2**30:.1f} GiB free on the device")


def index_arrays(kh, ix):
    """(keys int64 [U], pos int32 [N, 2], counts int32 [U], sizes) of an index, written by the C ABI into device tensors."""
    lib, L = _L()
    U, N, P = ix.sizes
    keys = torch.empty(U, dtype=torch.int64, device="cuda")
    lib.check(L.kmg_kmers_u64(ix._handle(), C.c_void_p(keys.data_ptr())))
    cnt = torch.empty(U, dtype=torch.int32, device="cuda")
    pos = torch.empty((N, 2), dtype=torch.int32, device="cuda")
    kh.kmer_pos(ix, 2 | 8, out={"pos": pos, "count": cnt})
    return dict(keys=keys, pos=pos, counts=cnt, sizes=(U, N, P))


def verify(kh, seq, k, ix, wk=None, valid=None, keep_order=False):
    lib, L = _L()
    arrays = index_arrays(kh, ix)
    lib.check(L.kmg_trim())
    return check_index(seq, k, arrays, L.kmg_index_order(ix._handle()) == 1, wk, valid, keep_order)


def _trim():
    lib, L = _L()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    lib.check(L.kmg_trim())


def _emit_chunked(emit, st, M, want, what, step=1 << 27):
    """Rows [0, M) through the chunk entry into a device buffer, compared with `want` chunk by chunk."""
    lib, _ = _L()
    buf = torch.empty((min(step, max(M, 1)), want.shape[1]), dtype=torch.int32, device="cuda")
    for a in range(0, M, step):
        n = min(step, M - a)
        lib.check(emit(st, a, n, C.c_void_p(buf.data_ptr())))
        assert_rows_equal(buf[:n], want[a:a + n], what, a)


def _emit_at(emit, st, first, n, width=2):
    lib, _ = _L()
    buf = torch.empty((n, width), dtype=torch.int32, device="cuda")
    lib.check(emit(st, first, n, C.c_void_p(buf.data_ptr())))
    return buf


# ---- 4. row streams past 2^32: a homopolymer against itself, closed forms --------------------------------------------
@pytest.mark.gpu
def test_row_streams_past_2_32(kh):
    """A 96,000-base homopolymer at k = 16: N = 95,985 windows, (i, j) rows M = N^2 = 9.2 * 10^9 and pair rows
    P = N(N - 1)/2 = 4.6 * 10^9, both past 2^32.  Row r of seq.kmer.pos is (k + r // N, 1 + r % N), of kmer.pairs
    (1 + r // N, 1 + r % N); every dot plot cell, run and chain has a closed form."""
    lib, L = _L()
    t0 = time.time()
    k, n = 16, 96_000
    s = b"A" * n
    N = n - k + 1
    ix = kh.make_kmer_hash(s, k, do_sort=True)
    assert ix.sizes == (1, N, N * (N - 1) // 2)
    M = N * N
    firsts = [0, 2**31 - 3, 2**32 - 5, 2**32 - 1, 2**32, 2**32 + 7 * N + 3, 2 * 2**32 + 11, M - 6]

    def check_chunks(st, I0):
        for f in firsts:
            nrow = min(6, M - f)
            got = _emit_at(L.kmg_query_emit_chunk if I0 == k else L.kmg_join_emit_chunk, st, f, nrow).cpu().tolist()
            assert got == [[I0 + (r // N), 1 + r % N] for r in range(f, f + nrow)], f
        big = _emit_at(L.kmg_query_emit_chunk if I0 == k else L.kmg_join_emit_chunk, st, 2**32 - 2**20, 2**21)
        r = torch.arange(2**32 - 2**20, 2**32 + 2**20, device="cuda", dtype=torch.int64)
        assert_rows_equal(big, torch.stack([I0 + r // N, 1 + r % N], 1).to(torch.int32), "rows across 2^32", 2**32 - 2**20)

    st, Mv = C.c_void_p(), C.c_uint64()
    lib.check(L.kmg_query_begin(ix._handle(), s, n, k, C.byref(st), C.byref(Mv)))
    try:
        assert Mv.value == M
        check_chunks(st, k)
    finally:
        L.kmg_query_free(st)
    st = C.c_void_p()
    lib.check(L.kmg_join_begin(ix._handle(), ix._handle(), C.byref(st), C.byref(Mv)))
    try:
        assert Mv.value == M
        check_chunks(st, 1)
    finally:
        L.kmg_join_free(st)
    # pair triples (1, a + 1, b + 1) around 2^32 and at the end
    P = N * (N - 1) // 2
    for f in (2**32 - 3, 2**32, 2**32 + 1, P - 4):
        got = _emit_at(lambda st_, a, m, o: L.kmg_pairs_chunk(ix._handle(), a, m, o), None, f, 4, 3).cpu().tolist()
        assert got == [[1, a + 1, b + 1] for a, b in (unrank_pair(t, N) for t in range(f, f + 4))], f

    # dot plots: cell (x, y) = (#I in bin x) * (#J in bin y); the total is N^2 > 2^32
    def per_bin(vals_lo, vals_hi, lo, hi, nb):
        c = [0] * nb
        for v in range(max(vals_lo, lo), min(vals_hi, hi - 1) + 1):
            c[(v - lo) * nb // (hi - lo)] += 1
        return np.array(c, np.float64)

    for xr, yr, nx, ny in (((1, n + 1), (1, N + 1), 37, 53), ((9_000, 90_001), (5, 2**31), 101, 7)):
        got = kh.seq_kmer_dotplot(ix, s, k, x_range=xr, y_range=yr, bins=(nx, ny))
        want = np.outer(per_bin(k, n, *xr, nx), per_bin(1, N, *yr, ny))
        assert np.array_equal(got, want), (xr, yr)
        got = kh.kmer_pairs_dotplot(ix, ix, a_range=xr, b_range=yr, bins=(nx, ny))
        assert np.array_equal(got, np.outer(per_bin(1, N, *xr, nx), per_bin(1, N, *yr, ny))), (xr, yr)
    assert kh.seq_kmer_dotplot(ix, s, k, y_range=(1, N + 1), bins=(1, 1))[0, 0] == M > 2**32

    # segments: one run per diagonal (query) / per diagonal and anti-diagonal (join with the T homopolymer's index)
    I0, J0, J1 = k, 1, N
    d = np.arange(I0 - J1, n - J0 + 1)
    i0, i1 = np.maximum(I0, J0 + d), np.minimum(n, J1 + d)
    qruns = np.stack([i0, i0 - d, i1 - i0 + 1], 1)
    qruns = qruns[np.lexsort((qruns[:, 1], qruns[:, 0]))]
    assert qruns[:, 2].sum() == M
    assert np.array_equal(kh.seq_kmer_segments(ix, s, k), qruns)
    for mr in (2, N - 1, N, N + 1):
        assert np.array_equal(kh.seq_kmer_segments(ix, s, k, min_rows=mr), qruns[qruns[:, 2] >= mr]), mr
    assert np.array_equal(kh.seq_kmer_segments(ix, s, k, max_count=N), qruns)
    assert len(kh.seq_kmer_segments(ix, s, k, max_count=N - 1)) == 0
    d = np.arange(1 - N, N)
    x0 = np.maximum(1, 1 + d)
    jruns = np.stack([x0, x0 - d, N - np.abs(d)], 1)
    jruns = jruns[np.lexsort((jruns[:, 1], jruns[:, 0]))]
    assert np.array_equal(kh.kmer_pairs_segments(ix, ix), jruns)
    it = kh.make_kmer_hash(b"T" * n, k, do_sort=True)
    sm = np.arange(2, 2 * N + 1)                               # antiparallel: x + y = sm, first row the smallest x
    x0 = np.maximum(1, sm - N)
    aruns = np.stack([x0, sm - x0, np.minimum(N, sm - 1) - x0 + 1], 1)
    aruns = aruns[np.lexsort((aruns[:, 1], aruns[:, 0]))]
    assert aruns[:, 2].sum() == M
    assert np.array_equal(kh.kmer_pairs_segments(ix, it, reverse_complement=True), aruns)
    assert len(kh.kmer_pairs_segments(ix, ix, reverse_complement=True)) == 0
    assert np.array_equal(kh.kmer_pairs_segments(ix, it, reverse_complement=True, min_rows=N), aruns[aruns[:, 2] >= N])

    # chains over those runs (G > 0): against chains_of
    for G, W in ((3 * k, 3), (100, 4), (N, 2)):
        assert np.array_equal(kh.seq_kmer_chains(ix, s, k, max_gap=G, max_shift=W), chains_of(qruns, G, W)), (G, W)
        assert np.array_equal(kh.kmer_pairs_chains(ix, ix, max_gap=G, max_shift=W), chains_of(jruns, G, W)), (G, W)
        assert np.array_equal(kh.kmer_pairs_chains(ix, it, max_gap=G, max_shift=W, reverse_complement=True),
                              chains_of(aruns, G, W, anti=True)), (G, W)
    ix.free(); it.free()
    _log("row streams past 2^32", t0)


# ---- 2. an index at the top of the range -----------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("k", [12, 32])
def test_top_homopolymer_index(kh, k):
    """INT32_MAX + k - 1 bases of A: one k-mer with INT32_MAX positions 1 .. N (one bin, one group, one list), checked in
    closed form; pair triples at a dozen row numbers over [0, P), P = N(N - 1)/2 ~ 2.3 * 10^18, against the unranking in
    Python integers; one base more is refused with KMG_ERR_RANGE before anything stays allocated."""
    lib, L = _L()
    t0 = time.time()
    _trim()
    torch.cuda.reset_peak_memory_stats()
    N = INT32_MAX
    seq = torch.full((N + k,), ord("A"), dtype=torch.uint8, device="cuda")     # one byte more than the largest index
    # one window too many: refused, and nothing stays allocated
    lib.check(L.kmg_trim())
    cached0, free0 = L.kmg_cached_bytes(), torch.cuda.mem_get_info()[0]
    h = C.c_void_p()
    assert L.kmg_build_ordered(C.c_void_p(seq.data_ptr()), N + k, k, 1, C.byref(h)) == KMG_ERR_RANGE and not h.value
    assert L.kmg_build_ordered(C.c_void_p(seq.data_ptr()), N + k, k, 0, C.byref(h)) == KMG_ERR_RANGE and not h.value
    lib.check(L.kmg_trim())
    assert L.kmg_cached_bytes() == cached0 and torch.cuda.mem_get_info()[0] >= free0 - (2 << 20)
    ix = kh.make_kmer_hash(seq[:N + k - 1], k, do_sort=k < 21)
    assert L.kmg_index_order(ix._handle()) == (1 if k < 21 else 0)
    P = N * (N - 1) // 2
    assert ix.sizes == (1, N, P)
    _trim()
    a = index_arrays(kh, ix)
    keys, pos, cnt = a.pop("keys"), a.pop("pos"), a.pop("counts")
    assert keys.tolist() == [0] and cnt.tolist() == [N]
    for a in range(0, N, SLICE):
        b = min(N, a + SLICE)
        _require(pos[a:b, 0] == 1, a, "k-mer number")
        _require(pos[a:b, 1] == torch.arange(a + 1, b + 1, device="cuda", dtype=torch.int32), a, "position")
    del keys, pos, cnt
    spec = kh.kmer_spectrum(ix, 1 << 30)
    assert spec[-1] == 1 and spec.sum() == 1
    spec = kh.kmer_spectrum(ix, 7)
    assert spec.tolist() == [0] * 7 + [1]
    # pair triples: boundaries of j(2n - j - 1)/2, the first row of the last j, P - 1
    S = lambda j: j * (2 * N - j - 1) // 2
    firsts = [0, 1, N - 2, N - 1, S(2**20), S(2**30) - 1, S(2**30), 2**32, 2**60 + 12345, P // 2, S(N - 3), S(N - 2) - 1,
              S(N - 2), P - 1]
    for f in firsts:
        m = min(4, P - f)
        got = _emit_at(lambda st_, a, n_, o: L.kmg_pairs_chunk(ix._handle(), a, n_, o), None, f, m, 3).cpu().tolist()
        assert got == [[1, a + 1, b + 1] for a, b in (unrank_pair(t, N) for t in range(f, f + m))], f
    assert unrank_pair(P - 1, N) == (N - 2, N - 1)
    ix.free()
    del seq
    _trim()
    _log(f"homopolymer index of 2^31 - 1 windows at k = {k}", t0)


def _big_sequence():
    """INT32_MAX + 31 bases (nstarts = INT32_MAX at k = 32): repeats, tandem arrays, lower case, N runs, and breakers just
    below and above 2^30 and 2^31 - 2^20."""
    from kmer_hasher_b200 import synth
    L = INT32_MAX + 31
    s = synth.generate(L, 0x1E32, repeat=0.02, tandem=0.005, homo=0.0005, lower=0.2, n_gaps=8, gap_min=10, gap_max=5000,
                       n_single=3000, tandem_len_min=100, tandem_len_max=2000, homo_len_max=60)
    for p in (2**30 - 40, 2**30 - 1, 2**30 + 1, 2**30 + 33, 2**31 - 2**20 - 40, 2**31 - 2**20 - 1, 2**31 - 2**20 + 2):
        s[p] = ord("N") if p & 1 else ord("n")
    return s


@pytest.fixture(scope="module")
def big_seq():
    s = _big_sequence()
    return s, torch.from_numpy(s).cuda()


@pytest.mark.gpu
def test_top_index_sorted_k16(kh, big_seq):
    """The sorted build (32-bit keys) of the first INT32_MAX + 15 bases (nstarts = INT32_MAX): checked completely; its
    spectrum."""
    t0 = time.time()
    _trim()
    torch.cuda.reset_peak_memory_stats()
    k = 16
    dseq = big_seq[1][:INT32_MAX + k - 1]
    ix = kh.make_kmer_hash(dseq, k, do_sort=True)
    _log("k = 16 build", t0)
    v = verify(kh, dseq, k, ix)
    assert v.sizes[1] > 2**31 - 2**25 and int(v.pos.max()) > 2**31 - 2**20
    _check_spectrum(kh, ix, v)
    ix.free()
    del v
    _trim()
    _log("k = 16 index of 2^31 - 16 windows, checked", t0)


def _check_spectrum(kh, ix, v):
    for mc in (3, 1000, 1 << 20):
        assert np.array_equal(kh.kmer_spectrum(ix, mc), _spectrum_of(v.scount, mc)), mc


@pytest.fixture(scope="module")
def big32(kh, big_seq):
    """The grouped build at k = 32 of the whole sequence (nstarts = INT32_MAX), its window keys and the verified index."""
    t0 = time.time()
    _trim()
    torch.cuda.reset_peak_memory_stats()
    s, dseq = big_seq
    k = 32
    ix = kh.make_kmer_hash(dseq, k)
    _log("k = 32 grouped build", t0)
    wk, valid = window_keys(dseq, k)
    assert wk.numel() == INT32_MAX
    v = verify(kh, dseq, k, ix, wk, valid)
    _log("k = 32 index of 2^31 - 1 windows, checked", t0)
    # The library's key table for probing 2^31 k-mers takes 85 GB of the device: keep only what the probe tests compare
    # with -- the verified index restricted to the query's k-mers and their reverse complements, the spectrum, and the
    # self depth's expected values -- so that it fits beside the index.
    spec = {mc: kh.kmer_spectrum(ix, mc) for mc in (3, 1000, 1 << 20)}
    want_spec = {mc: _spectrum_of(v.scount, mc) for mc in spec}
    top = int(v.pos.max())
    q = torch.from_numpy(_query(s)).cuda()
    qk, qv = window_keys(q, k)
    keys = torch.cat([qk[qv], revcomp_keys_t(qk[qv], k)])
    sub = restrict(v, keys)
    del q, qk, qv, keys
    nwin = INT32_MAX - 1 - k + 1                               # windows of the longest query, seq[:INT32_MAX - 1]
    qvalid = valid[:nwin].clone()
    if bool(qvalid[-1]) and bool(_is_breaker(dseq[nwin - 2])):
        qvalid[-1] = False                                     # the query's own end-of-string rule
    depth = [torch.empty(nwin, dtype=torch.int32, device="cuda") for _ in range(2)]
    for a in range(0, nwin, SLICE):
        b = min(nwin, a + SLICE)
        for both in (0, 1):
            depth[both][a:b] = expected_depth(wk[a:b], qvalid[a:b], k, v, bool(both))
    del v, wk, valid, qvalid
    _trim()
    _log("k = 32 expected values kept", t0)
    yield dict(ix=ix, sub=sub, k=k, spec=spec, want_spec=want_spec, top=top, depth=depth)
    ix.free()
    _trim()


def _spectrum_of(counts, mc):
    hist = torch.bincount(counts.to(torch.int64).clamp(max=mc), minlength=mc + 1).cpu().numpy()
    return hist.astype(np.float64)


def restrict(v: Verified, keys):
    """The verified index cut down to those of `keys` it holds (every position of each)."""
    hit, u = v.lookup(keys)
    u = torch.unique(u[hit])                                   # ascending rank = ascending key
    c = v.scount[u].to(torch.int64)
    first = torch.cumsum(c, 0) - c
    src = torch.repeat_interleave(v.sstart[u].to(torch.int64) - first, c) + torch.arange(int(c.sum()), device=c.device)
    return Verified(v.k, v.skf[u], first.to(torch.int32), v.scount[u], v.pos[src], v.sizes,
                    None if v.snum is None else v.snum[u])


@pytest.mark.gpu
def test_top_index_grouped_k32(kh, big32):
    """The grouped build of INT32_MAX windows at k = 32, checked completely (in the fixture); its spectrum."""
    L = _L()[1]
    assert L.kmg_index_order(big32["ix"]._handle()) == 0
    assert big32["top"] == INT32_MAX                            # the highest position is there
    for mc, got in big32["spec"].items():
        assert np.array_equal(got, big32["want_spec"][mc]), mc


def _query(s):
    """A 16 Mbp slice from the top of the index (positions up to INT32_MAX), an 8 Mbp top slice with substitutions every
    100-200 bases and a few short indels, and 2 Mbp of unrelated sequence."""
    rng = np.random.default_rng(31)
    L = len(s)
    return np.concatenate([s[L - 2**24:], _mutated(s[L - 2**25:L - 2**25 + 2**23], rng), random_dna(2_000_000, 77)])


def _revcomp_dev(q):
    tab = torch.from_numpy(np.frombuffer(bytes(range(256)).translate(IUPAC), np.uint8).copy()).cuda()
    return tab[q.flip(0).to(torch.int64)]


@pytest.mark.gpu
def test_probes_at_high_coordinates(kh, big_seq, big32):
    """seq.kmer.pos (whole and through kmg_query_emit_chunk), seq.kmer.depth on one and both strands, seq.kmer.dotplot
    over the top 2^25 and the whole range, seq.kmer.segments and seq.kmer.chains of a query against the index verified
    above, forward and reverse-complemented, every output against the restatement."""
    lib, L = _L()
    t0 = time.time()
    torch.cuda.reset_peak_memory_stats()
    s, _ = big_seq
    ix, v, k = big32["ix"], big32["sub"], big32["k"]
    q = _query(s)
    dq = torch.from_numpy(q).cuda()
    nq = len(q)
    for rc in (False, True):
        qq = _revcomp_dev(dq) if rc else dq
        qk, qv = window_keys(qq, k)
        want = expected_rows(qk, qv, k, v)
        M = len(want)
        assert int(want[:, 1].max()) > 2**31 - 2**20
        got = torch.empty((M, 2), dtype=torch.int32, device="cuda")
        kh.seq_kmer_pos(ix, dq, k, allow_k32=True, reverse_complement=rc, out=got)
        assert_rows_equal(got, want, f"seq.kmer.pos rc={rc}")
        del got
        st, Mv = C.c_void_p(), C.c_uint64()
        begin = L.kmg_query_begin_rc if rc else L.kmg_query_begin
        lib.check(begin(ix._handle(), C.c_void_p(dq.data_ptr()), nq, k, C.byref(st), C.byref(Mv)))
        try:
            assert Mv.value == M
            _emit_chunked(L.kmg_query_emit_chunk, st, M, want, f"kmg_query_emit_chunk rc={rc}", step=(1 << 24) + 7)
        finally:
            L.kmg_query_free(st)
        if not rc:                                             # depth is of the forward windows
            for both in (False, True):
                got = torch.empty(nq - k + 1, dtype=torch.int32, device="cuda")
                kh.seq_kmer_depth(ix, dq, both_strands=both, out=got)
                assert_rows_equal(got, expected_depth(qk, qv, k, v, both), f"depth both={both}")
        for yr, bins in (((2**31 - 2**25, 2**31), (1000, 1000)), ((0, 2**31), (997, 1009))):
            got = kh.seq_kmer_dotplot(ix, dq, k, y_range=yr, bins=bins, reverse_complement=rc, allow_k32=True)
            wimg = bin_counts(want[:, 0], want[:, 1], (1, nq + 1), bins[0], yr, bins[1]).cpu().numpy()
            assert np.array_equal(got.ravel(order="F"), wimg), (rc, yr)
        runs = runs_dev(want)
        del want
        seg = kh.seq_kmer_segments(ix, dq, k, reverse_complement=rc, allow_k32=True)
        assert_rows_equal(torch.from_numpy(seg).cuda().to(torch.int64), runs, f"segments rc={rc}")
        rn = runs.cpu().numpy()
        for G, W in ((3 * k, 3), (100, 4)):
            got = kh.seq_kmer_chains(ix, dq, k, max_gap=G, max_shift=W, reverse_complement=rc, allow_k32=True)
            want_c = chains_of(rn, G, W)
            assert np.array_equal(got, want_c), (rc, G, W)
        del runs, qk, qv
    _trim()
    _log("probes at high coordinates", t0)


@pytest.mark.gpu
def test_self_depth_longest_query(kh, big_seq, big32):
    """seq.kmer.depth of seq[:INT32_MAX - 1], the longest query accepted, against the index of the whole sequence:
    exactly counts[rank(window key)], NA where the window is not emitted; a query of INT32_MAX bases is refused."""
    lib, L = _L()
    t0 = time.time()
    torch.cuda.reset_peak_memory_stats()
    _, dseq = big_seq
    ix, k = big32["ix"], big32["k"]
    depth = big32.pop("depth")                                 # needed here only: freed for the join that follows
    _trim()
    nq = INT32_MAX - 1
    nwin = nq - k + 1
    out = torch.empty(nwin + 1, dtype=torch.int32, device="cuda")
    p = C.c_void_p(dseq.data_ptr())
    assert L.kmg_index_depth(ix._handle(), p, INT32_MAX, 0, C.c_void_p(out.data_ptr())) == KMG_ERR_RANGE
    st, Mv = C.c_void_p(), C.c_uint64()
    assert L.kmg_query_begin(ix._handle(), p, INT32_MAX, k, C.byref(st), C.byref(Mv)) == KMG_ERR_RANGE
    for both in (0, 1):
        lib.check(L.kmg_index_depth(ix._handle(), p, nq, both, C.c_void_p(out.data_ptr())))
        assert_rows_equal(out[:nwin], depth[both], f"self depth both={both}")
    _log("self depth over 2^31 - 2 bases", t0)


@pytest.mark.gpu
def test_join_at_high_coordinates(kh, big_seq, big32):
    """The same query as an index of its own (verified like the big one) joined with the big index, so that the positions
    in the second index reach INT32_MAX: kmer.pairs through kmg_join_emit_chunk, kmer.pairs.dotplot, and
    kmer.pairs.segments / kmer.pairs.chains on both strands.  (The query's index comes first: a join keeps per-k-mer
    arrays of its first index, 50 GB for the big one, which does not fit beside its 85 GB key table.)"""
    lib, L = _L()
    t0 = time.time()
    torch.cuda.reset_peak_memory_stats()
    _trim()
    s, _ = big_seq
    ix, v, k = big32["ix"], big32["sub"], big32["k"]
    q = _query(s)
    dq = torch.from_numpy(q).cuda()
    iq = kh.make_kmer_hash(dq, k)
    vq = verify(kh, dq, k, iq, keep_order=True)
    want = join_rows(vq, v)
    M = len(want)
    st, Mv = C.c_void_p(), C.c_uint64()
    lib.check(L.kmg_join_begin(iq._handle(), ix._handle(), C.byref(st), C.byref(Mv)))
    try:
        assert Mv.value == M
        _emit_chunked(L.kmg_join_emit_chunk, st, M, want, "kmg_join_emit_chunk", step=(1 << 24) + 5)
    finally:
        L.kmg_join_free(st)
    for ar, br, bins in (((1, len(q) + 1), (2**31 - 2**25, 2**31), (700, 1000)), ((0, 2**31), (0, 2**31), (1009, 997))):
        got = kh.kmer_pairs_dotplot(iq, ix, a_range=ar, b_range=br, bins=bins)
        assert np.array_equal(got.ravel(order="F"), bin_counts(want[:, 0], want[:, 1], ar, bins[0], br, bins[1]).cpu().numpy())
    for rc in (False, True):
        rows = join_rows(vq, v, rc=rc) if rc else want
        runs = runs_dev(rows, anti=rc)
        del rows
        seg = kh.kmer_pairs_segments(iq, ix, reverse_complement=rc)
        assert_rows_equal(torch.from_numpy(seg).cuda().to(torch.int64), runs, f"join segments rc={rc}")
        rn = runs.cpu().numpy()
        for G, W in ((3 * k, 3), (100, 4)):
            got = kh.kmer_pairs_chains(iq, ix, max_gap=G, max_shift=W, reverse_complement=rc)
            assert np.array_equal(got, chains_of(rn, G, W, anti=rc)), (rc, G, W)
        del runs
    iq.free()
    _log("join at high coordinates", t0)
