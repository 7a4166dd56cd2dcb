"""Match segments on BASELINE config 4: seq.kmer.segments of the 100 Mbp C4 query against the 250 Mbp C3 index (k = 32,
grouped), forward and reverse complement, max_count 0 and 100, min_rows 1 and 20.

For each workload: R (runs returned) and the sum of their n; the median of REPS calls of begin + emit into a device
tensor (CUDA events); the per-kernel times of kmg_profile_* over REPS profiled calls; and for comparison the rows emitted
in the same run by kmg_query_begin + kmg_query_emit into device memory and into pageable host memory -- what an R user
gets from seq.kmer.pos today.  The card's name and power limit are read at the start.
usage: python tools/segmentbench.py [L] [Lq]"""
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
REPS = 7
lib = _lib.load()
KERNELS = ["probe_lookup", "probe_compact", "revcomp", "segment_starts", "segments_mark", "hist_rec", "scan_hist",
           "sort_pass_hist", "sort_pass", "rle", "segments_pair", "segments_emit"]


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


def rows_compare(begin, emit, free):
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


def profiled(fn):
    """per-call ms and launches of every kernel over REPS profiled calls"""
    kh.profile(enable=True, reset=True)
    for _ in range(REPS):
        fn()
    torch.cuda.synchronize()
    p = kh.profile(reset=True)
    kh.profile(enable=False)
    return {n: (v[0] / REPS, v[1] / REPS) for n, v in p.items()}


print(card())
seq = synth.config_c3(L)
q = synth.config_c4_query(seq, Lq)
dseq, dq = torch.from_numpy(seq).cuda(), torch.from_numpy(q).cuda()
k = 32
ix = kh.make_kmer_hash(dseq, k)
h = ix._handle()
qp = C.c_void_p(dq.data_ptr())

cmp = {}
for rc in (0, 1):
    begin = lib.kmg_query_begin_rc if rc else lib.kmg_query_begin
    cmp[rc] = rows_compare(lambda st, M, b=begin: b(h, qp, Lq, k, st, M), lib.kmg_query_emit, lib.kmg_query_free)
    print(f"C4 rows {'rc ' if rc else 'fwd'}: M {cmp[rc][0]:,d}; begin+emit into device {cmp[rc][1]:.2f} ms, "
          f"into pageable {cmp[rc][2]:.2f} ms")

for rc in (0, 1):
    for mc in (0, 100):
        for mr in (1, 20):
            st, R = C.c_void_p(), C.c_uint64()
            _lib.check(lib.kmg_segments_begin(h, qp, Lq, k, rc, mc, mr, C.byref(st), C.byref(R)))
            R = R.value
            out = torch.empty((max(R, 1), 3), dtype=torch.int32, device="cuda")
            _lib.check(lib.kmg_segments_emit(st, C.c_void_p(out.data_ptr())))
            lib.kmg_segments_free(st)
            rows = int(out[:R, 2].sum(dtype=torch.int64))

            def call(rc=rc, mc=mc, mr=mr, out=out):
                s2, r2 = C.c_void_p(), C.c_uint64()
                _lib.check(lib.kmg_segments_begin(h, qp, Lq, k, rc, mc, mr, C.byref(s2), C.byref(r2)))
                _lib.check(lib.kmg_segments_emit(s2, C.c_void_p(out.data_ptr())))
                lib.kmg_segments_free(s2)
            ms = median_ms(call)
            kt = profiled(call)
            parts = ", ".join(f"{n} {kt[n][0]:.3f}" + (f" (x{kt[n][1]:.0f})" if kt[n][1] > 1 else "") for n in KERNELS if n in kt)
            other = sum(v[0] for n, v in kt.items() if n not in KERNELS)
            M, t_dev, t_page = cmp[rc]
            print(f"C4 segments {'rc ' if rc else 'fwd'} max_count {mc:3d} min_rows {mr:2d}: R {R:>12,d}, sum n {rows:>13,d}"
                  f" | call {ms:7.2f} ms ({ms / t_dev:.2f}x rows into device {t_dev:.2f} ms; rows into pageable {t_page:.1f} ms)")
            print(f"{'':8s}kernels per call (ms): {parts}" + (f", other {other:.3f}" if other else ""))
            del out
            torch.cuda.empty_cache()
ix.free()
lib.kmg_trim()
