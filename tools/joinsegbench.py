"""Match segments of joins (kmer.pairs.segments): the 100 Mbp C4 query built as a k = 32 index against the 250 Mbp C3 index,
and the 40 Mbp C5 index (k = 12) with itself, each forward and reverse complement, C5 with max_count 0 and 100.

For each workload: R and the sum of n; the median of REPS calls of kmg_join_segments_begin + emit into a device tensor
(CUDA events); the per-kernel times of kmg_profile_* over REPS profiled calls, with the bytes prof_bytes assigns to the
kernels of the join probe (last_pos, revcomp_keys, join_scatter, probe_compact); kmg_join_begin + kmg_join_emit into
device memory in the same run (forward only: the join has no reverse complement).  For C4 forward, also seq.kmer.segments
of the same pair (the C4 query against the C3 index), which must return the same runs shifted by k - 1.
The card's name and power limit are read at the start.
usage: python tools/joinsegbench.py [L3] [Lq] [L5]"""
import ctypes as C
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import kmer_hasher_b200 as kh
from kmer_hasher_b200 import _lib, synth

L3 = int(sys.argv[1]) if len(sys.argv) > 1 else 250_000_000
Lq = int(sys.argv[2]) if len(sys.argv) > 2 else 100_000_000
L5 = int(sys.argv[3]) if len(sys.argv) > 3 else 40_000_000
REPS = 7
lib = _lib.load()
KERNELS = ["last_pos", "revcomp_keys", "probe_lookup_rec", "segment_starts", "join_scatter", "probe_compact", "segments_mark",
           "hist_rec", "scan_hist", "sort_pass_hist", "sort_pass", "rle", "segments_pair", "segments_emit"]
PROBE = ["last_pos", "revcomp_keys", "join_scatter", "probe_compact"]


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


def profiled(fn):
    """per-call (ms, launches, bytes) of every kernel over REPS profiled calls"""
    kh.profile(enable=True, reset=True)
    for _ in range(REPS):
        fn()
    torch.cuda.synchronize()
    p = kh.profile(reset=True)
    kh.profile(enable=False)
    return {n: (v[0] / REPS, v[1] / REPS, v[2] / REPS) for n, v in p.items()}


def segments(begin):
    """(R, sum n, device result) of one call of `begin(st, R)` + emit"""
    st, R = C.c_void_p(), C.c_uint64()
    _lib.check(begin(C.byref(st), C.byref(R)))
    R = R.value
    out = torch.empty((max(R, 1), 3), dtype=torch.int32, device="cuda")
    _lib.check(lib.kmg_segments_emit(st, C.c_void_p(out.data_ptr())))
    lib.kmg_segments_free(st)
    return R, int(out[:R, 2].sum(dtype=torch.int64)), out[:R]


def call_of(begin, out):
    def call():
        st, R = C.c_void_p(), C.c_uint64()
        _lib.check(begin(C.byref(st), C.byref(R)))
        _lib.check(lib.kmg_segments_emit(st, C.c_void_p(out.data_ptr())))
        lib.kmg_segments_free(st)
    return call


def join_rows_ms(a, b):
    """(M, kmg_join_begin + kmg_join_emit into device memory in ms)"""
    st, M = C.c_void_p(), C.c_uint64()
    _lib.check(lib.kmg_join_begin(a, b, C.byref(st), C.byref(M)))
    lib.kmg_join_free(st)
    M = M.value
    dev = torch.empty(2 * max(M, 1), dtype=torch.int32, device="cuda")

    def run():
        s2, m2 = C.c_void_p(), C.c_uint64()
        _lib.check(lib.kmg_join_begin(a, b, C.byref(s2), C.byref(m2)))
        _lib.check(lib.kmg_join_emit(s2, C.c_void_p(dev.data_ptr())))
        lib.kmg_join_free(s2)
    t = median_ms(run)
    del dev
    torch.cuda.empty_cache()
    return M, t


def report(name, begin, rows=None, ref=None):
    R, n, res = segments(begin)
    out = torch.empty((max(R, 1), 3), dtype=torch.int32, device="cuda")
    call = call_of(begin, out)
    ms = median_ms(call)
    kt = profiled(call)
    parts = ", ".join(f"{k} {kt[k][0]:.3f}" + (f" (x{kt[k][1]:.0f})" if kt[k][1] > 1 else "") for k in KERNELS if k in kt)
    other = sum(v[0] for k, v in kt.items() if k not in KERNELS)
    rate = ", ".join(f"{k} {kt[k][2] / 1e6:.0f} MB = {kt[k][2] / kt[k][0] / 1e6:.0f} GB/s" for k in PROBE if k in kt and kt[k][0] > 0)
    line = f"{name}: R {R:>12,d}, sum n {n:>14,d} | call {ms:8.2f} ms"
    if rows:
        line += f" | join rows M {rows[0]:,d}, begin+emit into device {rows[1]:.2f} ms"
    if ref:
        line += f" | seq.kmer.segments of the same pair {ref:.2f} ms ({ms / ref:.2f}x)"
    print(line)
    print(f"{'':8s}kernels per call (ms): {parts}" + (f", other {other:.3f}" if other else ""))
    print(f"{'':8s}join probe bytes (prof_bytes): {rate}")
    del out
    torch.cuda.empty_cache()
    return R, n, res


print(card())
seq = synth.config_c3(L3)
q = synth.config_c4_query(seq, Lq)
dseq, dq = torch.from_numpy(seq).cuda(), torch.from_numpy(q).cuda()
del seq
k = 32
ic, iq = kh.make_kmer_hash(dseq, k), kh.make_kmer_hash(dq, k)
del dseq
hc, hq = ic._handle(), iq._handle()
qp = C.c_void_p(dq.data_ptr())

# the same pair through the query path: C4 query against the C3 index
sq_begin = lambda st, R: lib.kmg_segments_begin(hc, qp, Lq, k, 0, 0, 1, st, R)
Rq, nq, resq = segments(sq_begin)
outq = torch.empty((max(Rq, 1), 3), dtype=torch.int32, device="cuda")
t_query = median_ms(call_of(sq_begin, outq))
del outq
print(f"C4 seq.kmer.segments fwd (query against the C3 index): R {Rq:,d}, sum n {nq:,d}, call {t_query:.2f} ms")
rows = join_rows_ms(hq, hc)
for rc in (0, 1):
    R, n, res = report(f"C4 join segments {'rc ' if rc else 'fwd'} (C4 index x C3 index)",
                       lambda st, R_, rc=rc: lib.kmg_join_segments_begin(hq, hc, rc, 0, 1, st, R_),
                       rows if rc == 0 else None, t_query if rc == 0 else None)
    if rc == 0:
        resq[:, 0] -= k - 1
        print(f"{'':8s}equal to seq.kmer.segments shifted by k - 1: {R == Rq and torch.equal(res, resq)}")
    del res
del resq
ic.free(); iq.free()
del dq
lib.kmg_trim()
torch.cuda.empty_cache()

s5 = synth.config_c5(L5)
d5 = torch.from_numpy(s5).cuda()
del s5
k = 12
i5 = kh.make_kmer_hash(d5, k)
del d5
h5 = i5._handle()
rows5 = join_rows_ms(h5, h5)
for rc in (0, 1):
    for mc in (0, 100):
        R, n, res = report(f"C5 self join segments {'rc ' if rc else 'fwd'} max_count {mc:3d}",
                           lambda st, R_, rc=rc, mc=mc: lib.kmg_join_segments_begin(h5, h5, rc, mc, 1, st, R_),
                           rows5 if rc == 0 and mc == 0 else None)
        del res
i5.free()
lib.kmg_trim()
