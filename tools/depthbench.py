"""seq.kmer.depth on BASELINE config 4: the 100 Mbp C4 query against the 250 Mbp C3 sequence at k = 32, counted into a
one-column table (kmg_count_add), into a three-column table, and indexed (make.kmer.hash, grouped).  For each, forward
and both strands: the first call (it builds the key table), the steady-state call into a device-resident output (CUDA
events, median of REPS), windows/s, and the depth_lookup kernel's time and its line traffic (128 bytes per table request,
plus one line per window and strand for the row gather of a multi-column table) as a share of the measured HBM copy
bandwidth.  The C4 probe_lookup kernel is timed in the same run for comparison.
usage: python tools/depthbench.py [L] [Lq]"""
import ctypes as C
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import kmer_hasher_b200 as kh
from kmer_hasher_b200 import _lib, synth

L = int(sys.argv[1]) if len(sys.argv) > 1 else 250_000_000
Lq = int(sys.argv[2]) if len(sys.argv) > 2 else 100_000_000
k, REPS = 32, 7
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


def copy_bandwidth():
    """GB/s of a device-to-device copy of 4 GiB (read + write), best of 5: the HBM bandwidth the kernels are compared to."""
    x = torch.empty(1 << 32, dtype=torch.uint8, device="cuda")
    y = torch.empty_like(x)
    y.copy_(x)
    best = min(timed(lambda: y.copy_(x)) for _ in range(5))
    del x, y
    torch.cuda.empty_cache()
    return 2 * (1 << 32) / best / 1e6


print(card())
bw = copy_bandwidth()
print(f"device-to-device copy: {bw:.0f} GB/s")
seq = synth.config_c3(L)
q = synth.config_c4_query(seq, Lq)
dseq, dq = torch.from_numpy(seq).cuda(), torch.from_numpy(q).cuda()
nwin = Lq - k + 1


def run(name, ptr, cols, depth_fn):
    out = torch.empty((nwin, cols), dtype=torch.int32, device="cuda")
    h = ptr._handle()
    for strands in (0, 1):
        call = lambda: _lib.check(depth_fn(h, C.c_void_p(dq.data_ptr()), Lq, strands, C.c_void_p(out.data_ptr())))
        first = timed(call) if strands == 0 else None
        times = sorted(timed(call) for _ in range(REPS))
        kh.profile(enable=True, reset=True)
        for _ in range(REPS):
            call()
        torch.cuda.synchronize()
        ms, n, _ = kh.profile(reset=True)["depth_lookup"]
        kh.profile(enable=False)
        kms = ms / n
        lines = (2 if strands else 1) * (2 if cols > 1 else 1) * nwin * 128
        na = int((out[:, 0] == kh.NA_INTEGER).sum())
        hits = int((out[:, 0] > 0).sum())
        tag = f"{name:28s} {'both' if strands else 'fwd ':4s}"
        print(f"{tag} first call {first:7.2f} ms (key table build included)" if first is not None else f"{tag} first call    (table cached)",
              f"| steady {times[len(times) // 2]:6.2f} ms (min {times[0]:.2f}) = {nwin / times[len(times) // 2] / 1e6:6.2f} G windows/s"
              f" | depth_lookup {kms:6.3f} ms, lines {lines / kms / 1e6:6.0f} GB/s = {lines / kms / 1e6 / bw:.2f} of the copy"
              f" | hits {hits}, NA {na}")
    del out


ct1 = kh.count_kmers([dseq], (k, 0, 1))
print(f"count table, one source: U = {ct1.sizes[0]}")
run("count table, source_n = 1", ct1, 1, lib.kmg_count_depth)
ct1.free()
ct3 = kh.count_kmers([dseq], (k, 0, 3))
ct3 = kh.count_kmers([dq], (k, 1, 3), ct3)
ct3 = kh.count_kmers([dseq[:100_000_000]], (k, 2, 3), ct3)
print(f"count table, three sources: U = {ct3.sizes[0]}")
run("count table, source_n = 3", ct3, 3, lib.kmg_count_depth)
ct3.free()
ix = kh.make_kmer_hash(dseq, k)
run("position index (grouped)", ix, 1, lib.kmg_index_depth)

# the probe's lookup kernel on the same index, table already built
st, M = C.c_void_p(), C.c_uint64()
_lib.check(lib.kmg_query_begin(ix._handle(), dq.data_ptr(), Lq, k, C.byref(st), C.byref(M)))
lib.kmg_query_free(st)
kh.profile(enable=True, reset=True)
for _ in range(REPS):
    _lib.check(lib.kmg_query_begin(ix._handle(), dq.data_ptr(), Lq, k, C.byref(st), C.byref(M)))
    lib.kmg_query_free(st)
torch.cuda.synchronize()
ms, n, _ = kh.profile(reset=True)["probe_lookup"]
kh.profile(enable=False)
print(f"probe_lookup (seq.kmer.pos, same index and query): {ms / n:.3f} ms, lines {nwin * 128 / (ms / n) / 1e6:.0f} GB/s = "
      f"{nwin * 128 / (ms / n) / 1e6 / bw:.2f} of the copy")
ix.free()
lib.kmg_trim()
