"""Dot plots on BASELINE configs 4 and 5: seq.kmer.dotplot of the 100 Mbp C4 query against the 250 Mbp C3 index (k = 32,
grouped) at 1000 x 1000 over the full ranges, forward and reverse complement, zoomed to a 1 Mbp x 1 Mbp window, and at
64 x 64; kmer.pairs.dotplot of the 40 Mbp C5 index (k = 12) with itself, with and without max_count = 100.

For each workload: the median call time into a device-resident image (CUDA events, REPS calls), the dotplot_bin kernel's
time and its algorithmic bytes over that time (4 bytes of position per row, 8 for a join, plus the 8-byte-per-cell image),
and for comparison the rows emitted in the same run by kmg_query_begin + kmg_query_emit (kmg_join_begin + kmg_join_emit)
into device memory and into pageable host memory -- what an R user gets today (skipped over 2^31 - 1 rows, which no R
matrix can hold).  The card's name and power limit are read at the start.
usage: python tools/dotplotbench.py [L] [Lq] [L5]"""
import ctypes as C
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import kmer_hasher_b200 as kh
from kmer_hasher_b200 import _lib, synth

L = int(sys.argv[1]) if len(sys.argv) > 1 else 250_000_000
Lq = int(sys.argv[2]) if len(sys.argv) > 2 else 100_000_000
L5 = int(sys.argv[3]) if len(sys.argv) > 3 else 40_000_000
REPS = 7
lib = _lib.load()


def card():
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:                                 # the numbers below are still printed, marked as such
        pl = f"unknown ({e})"
    return f"{torch.cuda.get_device_name(0)}, power limit / max SM clock: {pl}"


def timed(fn):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); fn(); b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b)


def median_ms(fn):
    fn()
    t = sorted(timed(fn) for _ in range(REPS))
    return t[len(t) // 2]


def kernels(fn, names):
    """per-call ms and algorithmic bytes of the named kernels over REPS profiled calls"""
    kh.profile(enable=True, reset=True)
    for _ in range(REPS):
        fn()
    torch.cuda.synchronize()
    p = kh.profile(reset=True)
    kh.profile(enable=False)
    return {n: (p[n][0] / REPS, p[n][2] / REPS, p[n][1] / REPS) for n in names if n in p}


def rows_compare(begin, emit, free, M_expected=None):
    """(begin + emit into device, begin + emit into pageable) in ms; pageable is None over 2^31 - 1 rows"""
    st, M = C.c_void_p(), C.c_uint64()
    _lib.check(begin(C.byref(st), C.byref(M)))
    M = M.value
    free(st)
    dev = torch.empty(2 * max(M, 1), dtype=torch.int32, device="cuda")

    def run(ptr):
        s2, m2 = C.c_void_p(), C.c_uint64()
        _lib.check(begin(C.byref(s2), C.byref(m2)))
        _lib.check(emit(s2, C.c_void_p(ptr)))
        free(s2)
    t_dev = median_ms(lambda: run(dev.data_ptr()))
    del dev
    torch.cuda.empty_cache()
    t_page = None
    if M <= 2**31 - 1:
        page = np.empty(2 * max(M, 1), np.int32)
        page[::1024] = 0                                   # fault the pages in once, as R's allocMatrix result is
        run(page.ctypes.data)
        ts = []
        for _ in range(3):
            t0 = time.perf_counter(); run(page.ctypes.data); ts.append((time.perf_counter() - t0) * 1e3)
        t_page = sorted(ts)[1]
        del page
    return M, t_dev, t_page


def report(name, call, M, rb, cells, cmp):
    ms = median_ms(call)
    kt = kernels(call, ["dotplot_bin", "dotplot_finish", "probe_lookup", "probe_compact", "probe_lookup_rec", "join_compact",
                        "segment_starts", "revcomp"])
    kb, bb, nb = kt.get("dotplot_bin", (0.0, 0.0, 0))
    parts = ", ".join(f"{n} {v[0]:.3f}" for n, v in kt.items())
    _, t_dev, t_page = cmp
    print(f"{name:34s} rows {M:>13,d} | call {ms:8.2f} ms | dotplot_bin {kb:8.3f} ms ({nb:.0f} launches) "
          f"{bb / kb / 1e6 if kb else 0:7.0f} GB/s ({rb} B/row + image), {M / kb / 1e6 if kb else 0:6.1f} G rows/s"
          f" | rows instead: begin+emit device {t_dev:8.2f} ms, pageable "
          f"{'%8.2f ms' % t_page if t_page is not None else '(over 2^31-1 rows: no R matrix)'}")
    print(f"{'':34s} kernels per call (ms): {parts}")


print(card())
seq = synth.config_c3(L)
q = synth.config_c4_query(seq, Lq)
dseq, dq = torch.from_numpy(seq).cuda(), torch.from_numpy(q).cuda()
k = 32
ix = kh.make_kmer_hash(dseq, k)
h = ix._handle()
img = torch.empty(1000 * 1000, dtype=torch.float64, device="cuda")
qp = C.c_void_p(dq.data_ptr())


def qdot(rc, xr, yr, nx, ny, mc=0):
    return lambda: _lib.check(lib.kmg_query_dotplot(h, qp, Lq, k, rc, xr[0], xr[1], nx, yr[0], yr[1], ny, mc, C.c_void_p(img.data_ptr())))


cmp = {}
for rc in (0, 1):
    begin = lib.kmg_query_begin_rc if rc else lib.kmg_query_begin
    cmp[rc] = rows_compare(lambda st, M, b=begin: b(h, qp, Lq, k, st, M), lib.kmg_query_emit, lib.kmg_query_free)
full_x, full_y = (1, Lq + 1), (1, L + 1)
for rc in (0, 1):
    M = cmp[rc][0]
    report(f"C4 1000x1000 full {'rc ' if rc else 'fwd'}", qdot(rc, full_x, full_y, 1000, 1000), M, 4, 10**6, cmp[rc])
# zoom: a 1 Mbp x 1 Mbp window around the densest 1 Mbp cell of a 100 x 250 coarse plot of the forward rows
coarse = torch.empty(100 * 250, dtype=torch.float64, device="cuda")
_lib.check(lib.kmg_query_dotplot(h, qp, Lq, k, 0, 1, Lq + 1, 100, 1, L + 1, 250, 0, C.c_void_p(coarse.data_ptr())))
cell = int(torch.argmax(coarse).item())
zx0, zy0 = 1 + (cell % 100) * (Lq // 100), 1 + (cell // 100) * (L // 250)
zx, zy = (zx0, zx0 + 1_000_000), (zy0, zy0 + 1_000_000)
zoom_rows = int(coarse[cell].item())
print(f"zoom window x [{zx[0]}, {zx[1]}), y [{zy[0]}, {zy[1]}) (densest coarse cell, {zoom_rows:,d} rows in its 1 Mbp x 1 Mbp)")
report("C4 1000x1000 zoom 1 Mbp fwd", qdot(0, zx, zy, 1000, 1000), cmp[0][0], 4, 10**6, cmp[0])
report("C4 64x64 full fwd (small image)", qdot(0, full_x, full_y, 64, 64), cmp[0][0], 4, 64 * 64, cmp[0])
report("C4 1000x1000 full fwd max_count 100", qdot(0, full_x, full_y, 1000, 1000, 100), cmp[0][0], 4, 10**6, cmp[0])
ix.free()
del dseq, dq, coarse
torch.cuda.empty_cache()
lib.kmg_trim()

s5 = synth.config_c5(L5)
ds5 = torch.from_numpy(s5).cuda()
ix5 = kh.make_kmer_hash(ds5, 12)
h5 = ix5._handle()
for mc in (0, 100):
    st0, M0 = C.c_void_p(), C.c_uint64()
    if mc == 0:
        cmpj = rows_compare(lambda st, M: lib.kmg_join_begin(h5, h5, st, M), lib.kmg_join_emit, lib.kmg_join_free)
    else:                                                  # no row path has a max_count: rows of the limited join, counted
        z = torch.empty(1, dtype=torch.float64, device="cuda")
        _lib.check(lib.kmg_join_dotplot(h5, h5, 0, 2**31, 1, 0, 2**31, 1, mc, C.c_void_p(z.data_ptr())))
        cmpj = (int(z.item()), float("nan"), None)
    call = lambda mc=mc: _lib.check(lib.kmg_join_dotplot(h5, h5, 1, L5 + 1, 1000, 1, L5 + 1, 1000, mc, C.c_void_p(img.data_ptr())))
    report(f"C5 self join 1000x1000 max_count {mc}", call, cmpj[0], 8, 10**6, cmpj)
ix5.free()
lib.kmg_trim()
