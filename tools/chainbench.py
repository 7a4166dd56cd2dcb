"""Chains (seq.kmer.chains, kmer.pairs.chains): the 100 Mbp C4 query against the 250 Mbp C3 index at k = 32, forward and
reverse complement, and the 40 Mbp C5 index (k = 12) joined with itself, forward and antiparallel; (G, W) in (0, 0),
(100, 4), (1000, 16), each with min_run 1 and 20.

For each workload: the chain count C, sum n and sum m; the median of REPS calls of segments begin + chains begin + emit
into a device tensor (CUDA events); the segments call alone (begin + emit) in the same run; the per-kernel times of the
chaining kernels from kmg_profile_* over REPS profiled calls.  The card's name and power limit are read at the start.
usage: python tools/chainbench.py [L3] [Lq] [L5]"""
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
CHAIN = ["chains_keys", "hist_rec", "scan_hist", "sort_pass_hist", "sort_pass", "rle", "chains_gather", "chains_link",
         "chains_heads", "chains_jump", "chains_aggregate", "chains_compact", "chains_emit"]
BANDS = ((0, 0), (100, 4), (1000, 16))


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
    """per-call (ms, launches) of every kernel over REPS profiled calls"""
    kh.profile(enable=True, reset=True)
    for _ in range(REPS):
        fn()
    torch.cuda.synchronize()
    p = kh.profile(reset=True)
    kh.profile(enable=False)
    return {n: (v[0] / REPS, v[1] / REPS) for n, v in p.items()}


def seg_call(begin, out):
    def call():
        st, R = C.c_void_p(), C.c_uint64()
        _lib.check(begin(C.byref(st), C.byref(R)))
        _lib.check(lib.kmg_segments_emit(st, C.c_void_p(out.data_ptr())))
        lib.kmg_segments_free(st)
    return call


def chain_call(begin, G, W, out, chains_only_prof=False):
    def call():
        st, R = C.c_void_p(), C.c_uint64()
        _lib.check(begin(C.byref(st), C.byref(R)))
        ch, Cn = C.c_void_p(), C.c_uint64()
        try:
            if chains_only_prof:
                kh.profile(enable=True)
            _lib.check(lib.kmg_chains_begin(st, G, W, 1, C.byref(ch), C.byref(Cn)))
            _lib.check(lib.kmg_chains_emit(ch, C.c_void_p(out.data_ptr())))
            if chains_only_prof:
                torch.cuda.synchronize()
                kh.profile(enable=False)
        finally:
            lib.kmg_chains_free(ch)
            lib.kmg_segments_free(st)
    return call


def chain_kernels(begin, G, W, out):
    """per-call times of the chaining kernels only (the profile is on during kmg_chains_begin + emit alone)"""
    kh.profile(enable=False, reset=True)
    call = chain_call(begin, G, W, out, True)
    for _ in range(REPS):
        call()
    p = kh.profile(reset=True)
    return {n: (v[0] / REPS, v[1] / REPS) for n, v in p.items()}


def workload(name, begin):
    st, R = C.c_void_p(), C.c_uint64()
    _lib.check(begin(C.byref(st), C.byref(R)))
    R = R.value
    lib.kmg_segments_free(st)
    sout = torch.empty((max(R, 1), 3), dtype=torch.int32, device="cuda")
    t_seg = median_ms(seg_call(begin, sout))
    del sout
    cout = torch.empty((max(R, 1), 6), dtype=torch.int32, device="cuda")
    print(f"{name}: segments R {R:,d}, segments begin + emit {t_seg:.2f} ms")
    for G, W in BANDS:
        st, Rr = C.c_void_p(), C.c_uint64()
        _lib.check(begin(C.byref(st), C.byref(Rr)))
        ch, Cn = C.c_void_p(), C.c_uint64()
        _lib.check(lib.kmg_chains_begin(st, G, W, 1, C.byref(ch), C.byref(Cn)))
        Cn = Cn.value
        _lib.check(lib.kmg_chains_emit(ch, C.c_void_p(cout.data_ptr())))
        lib.kmg_chains_free(ch)
        lib.kmg_segments_free(st)
        sn = int(cout[:Cn, 4].sum(dtype=torch.int64))
        sm = int(cout[:Cn, 5].sum(dtype=torch.int64))
        ms = median_ms(chain_call(begin, G, W, cout))
        kt = chain_kernels(begin, G, W, cout)
        parts = ", ".join(f"{k} {kt[k][0]:.3f}" + (f" (x{kt[k][1]:.0f})" if kt[k][1] > 1 else "") for k in CHAIN if k in kt)
        tot = sum(v[0] for v in kt.values())
        print(f"    G {G:4d} W {W:2d}: C {Cn:>12,d}, sum n {sn:>14,d}, sum m {sm:>12,d} | segments + chains + emit {ms:8.2f} ms"
              f" = {ms / t_seg:.3f}x the segments call (+{ms - t_seg:.2f} ms)")
        print(f"{'':8s}chaining kernels per call (ms, {tot:.3f} in all): {parts}")
    del cout
    torch.cuda.empty_cache()


print(card())
seq = synth.config_c3(L3)
q = synth.config_c4_query(seq, Lq)
dseq, dq = torch.from_numpy(seq).cuda(), torch.from_numpy(q).cuda()
del seq
k = 32
ic = kh.make_kmer_hash(dseq, k)
del dseq
hc, qp = ic._handle(), C.c_void_p(dq.data_ptr())
for rc in (0, 1):
    for mr in (1, 20):
        workload(f"C4 seq.kmer.chains {'rc ' if rc else 'fwd'} min_run {mr:2d}",
                 lambda st, R, rc=rc, mr=mr: lib.kmg_segments_begin(hc, qp, Lq, k, rc, 0, mr, st, R))
ic.free()
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
for rc in (0, 1):
    for mr in (1, 20):
        workload(f"C5 self kmer.pairs.chains {'anti' if rc else 'fwd '} min_run {mr:2d}",
                 lambda st, R, rc=rc, mr=mr: lib.kmg_join_segments_begin(h5, h5, rc, 0, mr, st, R))
i5.free()
lib.kmg_trim()
