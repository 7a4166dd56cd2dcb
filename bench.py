#!/usr/bin/env python
"""bench.py -- k-mers indexed/s and queried/s of the B200 k-mer position index (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c3k32|c3|c2]
                    [--scaling strong|weak] [--dump-outputs DIR]

A step = one pass of the hot path over one synthetic sequence.  The default workload is BASELINE.json's target
configuration, `c3k32`: ONE 250 Mbp synthetic chromosome with N gaps, k=32, make.kmer.hash + kmer.pos(2|8)
(index + counts + positions); `c3` is BASELINE config 3 (the same sequence at k=21), `c2` config 2 (40 Mbp, k=32).

  N=1   `value` times the step with the sequence and the outputs resident in HBM; `e2e` times the same calls
        through the public API with pinned HOST buffers (sequence in, pos/count matrices out), copies inside the
        timed region; `e2e_pageable` the same with ordinary (pageable) host arrays, which is what R's allocVector
        hands the glue.  `probe` is BASELINE config 4 on the same index: seq.kmer.pos of a 100 Mbp query (diverged
        copies of index segments + 20 % unrelated), kmg_query_begin AND kmg_query_emit, device-resident and e2e.
  N>1   strong scaling (default): the SAME sequence cut into N shards with k-1 bases of overlap, (key,pos) records
        written straight into the key-range owners' arrays over NVLink by the partitioning pass, per-owner sort + CSR,
        per-owner kmer.pos(2|8); `--scaling weak` gives every rank its own L-base shard of an N*L sequence instead.
        The sharded index is checked against committed digests of the reference's output (`parity_checked`).
--impl reference times the reference's own C (oracle/_ref, single-threaded like the reference) on the host cores for
the same metric on a bounded prefix of the same sequence.
--dump-outputs DIR (N=1) writes the pos and count matrices of the last timed step to DIR/pos.npy and DIR/count.npy,
each a fixed, seeded sample of 2^20 rows (see dump_rows), so that two builds can be compared output for output.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    "c3k32": dict(L=250_000_000, k=32, gen="c3", Lq=100_000_000, golden="c3k32",
                  name="c3k32: synthetic 250 Mbp chromosome with N gaps, k=32, make.kmer.hash + kmer.pos(2|8)"),
    "c3": dict(L=250_000_000, k=21, gen="c3", Lq=100_000_000, golden="c3",
               name="c3: synthetic 250 Mbp chromosome with N gaps, k=21, make.kmer.hash + kmer.pos(2|8)"),
    "c2": dict(L=40_000_000, k=32, gen="c2", Lq=10_000_000, golden="c2",
               name="c2: synthetic 40 Mbp repeat-rich, k=32, make.kmer.hash + kmer.pos(2|8)"),
}
METRIC = "kmers_indexed_per_s"


def load_synth():
    """The synthetic generator WITHOUT importing the kmer_hasher_b200 package (whose __init__ dlopens libkmergpu.so):
    the reference arm must not load the product."""
    spec = importlib.util.spec_from_file_location("_kmer_synth", os.path.join(ROOT, "kmer_hasher_b200", "synth.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def gen_sequence(w: dict, L: int, out=None):
    synth = load_synth()
    return synth.config_c2(L, out=out) if w["gen"] == "c2" else synth.config_c3(L, out=out)


def config_of(w: dict, k: int, L: int) -> dict:
    """Identical on both arms (ours / reference)."""
    return {"workload": w["name"], "k": k, "bases": L}


def ncu_profile(name: str):
    """Facts from the committed `ncu --set full` capture of a kernel (profiles/r02_ncu_<name>.json), if any."""
    path = os.path.join(ROOT, "profiles", f"r02_ncu_{name}.json")
    if os.path.exists(path):
        return json.load(open(path))
    return None


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock + throttle reasons sampled through NVML while the timed region runs."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz, self._stop = [], set(), None, threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # noqa: BLE001
            self.nv, self.err = None, repr(e)
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake": 0x80, "sync_boost": 0x10, "app_clocks": 0x2}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for n, bit in names.items():
                    if r & bit:
                        self.reasons.add(n)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.005)

    def __enter__(self):
        if self.nv:
            self.t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self.nv:
            self.t.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------------------
# reference arm: the reference's own C on the host cores
# ---------------------------------------------------------------------------------------------------------
def cpu_reference(k: int, seq: np.ndarray, probe_seq=None):
    """Times seq_to_hash + the kmer_positions(2|8) loop of the unmodified reference engine on `seq`
    (and seq_kmer_positions of `probe_seq` if given)."""
    from oracle import Reference
    ref = Reference()
    s = np.where(seq == 0, ord("A"), seq).astype(np.uint8)
    ix = ref.build(s, k)
    e = ix.extract_raw(2 | 8)
    n = ix.N
    t_build, t_ext = ix.build_seconds, e["seconds"]
    del e
    probe = None
    if probe_seq is not None:
        rows = ix.query(probe_seq, k, want_rows=False)
        probe = (len(probe_seq) - k + 1, ix.query_seconds, int(rows))
    ix.close()
    return n, t_build, t_ext, probe


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = WORKLOADS[args.workload]
    k, L = w["k"], w["L"]
    steps, warm = args.steps, args.warmup
    # bound each step so the whole run stays within a few minutes (~4.5 M k-mers/s on one core)
    budget = 150.0 * 4.0e6
    sample = int(min(L, max(2_000_000, budget / max(1, steps + warm))))
    seq = np.ascontiguousarray(gen_sequence(w, L)[:sample])
    times = []
    n = 0
    for i in range(warm + steps):
        n, tb, te, _ = cpu_reference(k, seq)
        if i >= warm:
            times.append(tb + te)
    t = float(np.mean(times))
    val = n / t
    sample_desc = (f"first {sample} bases of the workload's sequence per step; reference seq_to_hash + kmer_positions(2|8) loop "
                   f"(oracle/_ref = /root/reference/src/kmer_pos.c + kmer_util.c, gcc -O2), 1 thread: the reference path is single-threaded")
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "k-mers/s", "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": 1e3 * t, "higher_is_better": True,
            "scaling": args.scaling if args.gpus > 1 else "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": config_of(w, k, L),
            "cpu_baseline": {"value": val, "unit": "k-mers/s", "cores": 1, "kind": "reference", "sample": sample_desc},
            "e2e": {"value": val, "unit": "k-mers/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    import kmer_hasher_b200 as kh
    from kmer_hasher_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch N>1 with: python -m torch.distributed.run --nproc-per-node N bench.py --gpus N")
    torch.cuda.set_device(local)
    _lib.check(_lib.load().kmg_set_device(local))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    stream = torch.cuda.current_stream()
    _lib.check(_lib.load().kmg_set_stream(stream.cuda_stream))

    w = WORKLOADS[args.workload]
    k, L = w["k"], w["L"]
    steps, warm = args.steps, max(args.warmup, 3)
    hbm_peak, peak_src = peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if world == 1:
        line = bench_single(args, kh, torch, w, k, L, steps, warm, hbm_peak, peak_src, local)
    else:
        from kmer_hasher_b200 import dist as kdist
        line = kdist.bench_sharded(args, w, k, L, steps, warm, hbm_peak, peak_src, barrier)
    if rank == 0 and line is not None:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def timed(torch, fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


DUMP_ROWS = 1 << 20     # rows sampled from each output: 24 MB of .npy files for pos + count


def dump_rows(n: int) -> np.ndarray:
    """The rows of an n-row output that --dump-outputs keeps: all of them, or DUMP_ROWS distinct ones in ascending order,
    the same for every run with the same n."""
    return np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))


def dump_outputs(torch, out_dir: str, outputs: dict) -> None:
    """Writes `name.npy`: the rows `dump_rows` picks from each device array, as float64 (it holds every int32 exactly)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in outputs.items():
        rows = torch.from_numpy(dump_rows(a.shape[0])).to(a.device)
        np.save(os.path.join(out_dir, f"{name}.npy"), a[rows].cpu().numpy().astype(np.float64))


def index_leg(kh, torch, seq_dev, k, steps, warm):
    """build + kmer.pos(2|8), everything resident in HBM: (ms per step, N, U)."""
    ix = kh.make_kmer_hash(seq_dev, k)
    U, N = ix.sizes_un
    ix.free()
    pos_dev = torch.empty((N, 2), dtype=torch.int32, device="cuda")
    cnt_dev = torch.empty(U, dtype=torch.int32, device="cuda")

    def step():
        h = kh.make_kmer_hash(seq_dev, k)
        kh.kmer_pos(h, 2 | 8, out={"pos": pos_dev, "count": cnt_dev})
        h.free()
    for _ in range(warm):
        step()
    return step, N, U, (pos_dev, cnt_dev)


def probe_leg(kh, torch, _lib, w, seq_pin, seq_dev, k, steps, hbm_peak):
    """BASELINE config 4: seq.kmer.pos of a query made of diverged copies of index segments + 20 % unrelated sequence.
    Times kmg_query_begin (encode + table lookups + ordered compaction + 64-bit scan) AND kmg_query_emit (rows)."""
    import ctypes as C
    synth = load_synth()
    Lb = _lib.load()
    Lq = w["Lq"]
    q_pin = kh.pinned_empty(Lq, np.uint8)
    synth.config_c4_query(np.asarray(seq_pin), Lq, out=q_pin)
    q_dev = torch.from_numpy(np.asarray(q_pin)).cuda()
    st, M = C.c_void_p(), C.c_uint64()
    # first probe of a fresh index: includes building the key table (once per index)
    h = kh.make_kmer_hash(seq_dev, k)
    U = h.sizes_un[0]

    def begin(qptr):
        _lib.check(Lb.kmg_query_begin(h._handle(), qptr, Lq, k, C.byref(st), C.byref(M)))
    ms_first = timed(torch, lambda: begin(q_dev.data_ptr()), 1)
    Lb.kmg_query_free(st)
    h.free()                                  # its 9 GB key table goes back to the library's arena ...
    h = kh.make_kmer_hash(seq_dev, k)
    ms_first_warm = timed(torch, lambda: begin(q_dev.data_ptr()), 1)   # ... so this first probe of a NEW index allocates nothing
    Lb.kmg_query_free(st)
    begin(q_dev.data_ptr())
    rows_n = int(M.value)
    Lb.kmg_query_free(st)
    if rows_n > 2**31 - 1:               # more rows than an R matrix holds: seq.kmer.pos refuses (the glue checks M first)
        ms_b = timed(torch, lambda: (begin(q_dev.data_ptr()), Lb.kmg_query_free(st)), max(3, steps // 2))
        h.free()
        return {"metric": "kmers_queried_per_s", "value": None, "unit": "k-mers/s", "rows": rows_n, "ms_begin": ms_b,
                "first_probe_ms": ms_first, "first_probe_warm_ms": ms_first_warm, "note": "this query has more result rows than an R matrix can hold (2^31-1): seq.kmer.pos "
                "refuses it, so only kmg_query_begin (match + count + scan) is timed and no throughput with emission is claimed"}
    rows_dev = torch.empty((max(rows_n, 1), 2), dtype=torch.int32, device="cuda")
    rows_pin = kh.pinned_empty((max(rows_n, 1), 2), np.int32)
    n_rep = max(3, steps // 2)
    t_begin, t_emit = [0.0], [0.0]

    def dev_step():
        t_begin[0] += timed(torch, lambda: begin(q_dev.data_ptr()), 1)
        t_emit[0] += timed(torch, lambda: _lib.check(Lb.kmg_query_emit(st, rows_dev.data_ptr())), 1)
        Lb.kmg_query_free(st)

    def e2e_step():
        begin(q_pin.ctypes.data)
        _lib.check(Lb.kmg_query_emit(st, rows_pin.ctypes.data))
        Lb.kmg_query_free(st)
    for _ in range(2):
        dev_step()
    t_begin[0] = t_emit[0] = 0.0
    kh.profile(enable=True, reset=True)
    kh.profile(reset=True)
    for _ in range(n_rep):
        dev_step()
    prof = kh.profile(enable=False)
    kh.profile(reset=True)
    ms_b, ms_e = t_begin[0] / n_rep, t_emit[0] / n_rep
    e2e_step()
    ms_e2e = timed(torch, e2e_step, max(2, n_rep // 2))
    h.free()
    Nq = Lq - k + 1
    merge_bytes = Lq + 32 * Nq + 8 * U + 12 * rows_n                 # SURVEY.md 8d: seq.kmer.pos total
    ncu = ncu_profile("probe_match") or ncu_profile("probe_lookup")
    kern = {n: {"ms": v[0] / n_rep, "launches": v[1] / n_rep} for n, v in sorted(prof.items())}
    lookup_ms = sum(v["ms"] for n, v in kern.items() if n.startswith("probe_match") or n.startswith("probe_lookup"))
    roof = {"bound": "hbm", "what": "kmg_query_begin + kmg_query_emit, device-resident",
            "survey_merge_bytes": int(merge_bytes), "achieved": merge_bytes / ((ms_b + ms_e) * 1e-3) / 1e9, "peak": hbm_peak,
            "unit": "GB/s", "frac": merge_bytes / ((ms_b + ms_e) * 1e-3) / 1e9 / hbm_peak,
            "note": "graded denominator = SURVEY.md 8d's sort-merge formulation (Lq + 32 Nq + 8 U + 12 M); the shipped probe is one "
                    "random table access per window, which moves a whole 128-byte line of HBM per lookup",
            "lookup_line_bytes": int(128 * Nq), "lookup_line_GBps": 128 * Nq / (lookup_ms * 1e-3) / 1e9 if lookup_ms else None,
            "lookup_line_frac": 128 * Nq / (lookup_ms * 1e-3) / 1e9 / hbm_peak if lookup_ms else None,
            "ncu_dram_bytes_lookup": ncu["traffic_bytes_per_launch"] if ncu else None,
            "ncu_source": ncu["source"] if ncu else None}
    return {"metric": "kmers_queried_per_s", "value": Nq / ((ms_b + ms_e) * 1e-3), "unit": "k-mers/s",
            "config": f"c4: {Lq} bp query (diverged copies of index segments + 20 % unrelated) vs the {w['L']} bp index, k={k}, (i,j) rows emitted",
            "query_kmers": Nq, "rows": rows_n, "ms_begin": ms_b, "ms_emit": ms_e,
            "first_probe_ms": ms_first, "first_probe_what": "kmg_query_begin on a fresh index: includes building its key table (once per index) "
            "and, the very first time in a process, cudaMalloc of the table's 9 GB",
            "first_probe_warm_ms": ms_first_warm, "first_probe_warm_what": "the same on the next fresh index (the table's memory comes from the library's arena)",
            "e2e": {"value": Nq / (ms_e2e * 1e-3), "unit": "k-mers/s", "ms": ms_e2e, "h2d_bytes": Lq, "d2h_bytes": 8 * rows_n,
                    "what": "pinned host query in, (i,j) rows into a pinned host matrix"},
            "rows_per_s": rows_n / (ms_e * 1e-3) if ms_e else None, "roofline": roof, "kernels": kern}


def bench_single(args, kh, torch, w, k, L, steps, warm, hbm_peak, peak_src, dev):
    from kmer_hasher_b200 import _lib
    # ---- inputs: pinned host copy and a device-resident copy -------------------------------------------
    seq_pin = kh.pinned_empty(L, np.uint8)
    gen_sequence(w, L, out=seq_pin)
    seq_dev = torch.from_numpy(np.asarray(seq_pin)).cuda()
    step_device, N, U, (pos_dev, cnt_dev) = index_leg(kh, torch, seq_dev, k, steps, warm)
    pos_pin = kh.pinned_empty((N, 2), np.int32)
    cnt_pin = kh.pinned_empty(U, np.int32)

    def step_e2e():
        h = kh.make_kmer_hash(seq_pin, k)
        kh.kmer_pos(h, 2 | 8, out={"pos": pos_pin, "count": cnt_pin})
        h.free()

    kh.profile(enable=True, reset=True)
    kh.profile(reset=True)
    l0 = kh.launch_count()
    with ClockSampler(dev) as clk:
        ms = timed(torch, step_device, steps)
    launches = kh.launch_count() - l0
    prof = kh.profile(enable=False)
    kh.profile(reset=True)
    if args.dump_outputs:
        dump_outputs(torch, args.dump_outputs, {"pos": pos_dev, "count": cnt_dev})

    for _ in range(warm):
        step_e2e()
    ms_e2e = timed(torch, step_e2e, steps)

    # the same through ordinary pageable host arrays: what the R glue gets from allocVector / CHAR()
    e2e_pageable = None
    if not args.no_pageable:
        seq_pg = np.array(seq_pin, copy=True)
        pos_pg, cnt_pg = np.empty((N, 2), np.int32), np.empty(U, np.int32)
        pos_pg.fill(0); cnt_pg.fill(0)                            # touch the pages (R zero-fills nothing, but maps them)

        def step_pg():
            h = kh.make_kmer_hash(seq_pg, k)
            kh.kmer_pos(h, 2 | 8, out={"pos": pos_pg, "count": cnt_pg})
            h.free()
        step_pg()
        pg = sorted(timed(torch, step_pg, 1) for _ in range(max(5, steps // 4)))    # host memcpy threads share the box: per-step times, median
        ms_pg = pg[len(pg) // 2]
        e2e_pageable = {"value": N / (ms_pg * 1e-3), "unit": "k-mers/s", "ms_per_step": ms_pg, "vs_pinned": ms_pg / ms_e2e,
                        "ms_min": pg[0], "ms_max": pg[-1], "steps": len(pg),
                        "what": "same calls, pageable numpy arrays in and out (the R glue's INTEGER(allocMatrix) / CHAR memory); median step"}
        del seq_pg, pos_pg, cnt_pg

    probe = None if args.no_probe else probe_leg(kh, torch, _lib, w, seq_pin, seq_dev, k, steps, hbm_peak)

    # ---- roofline of the dominant kernel ---------------------------------------------------------------------
    dom = max(prof.items(), key=lambda kv: kv[1][0]) if prof else None
    roof = None
    if dom:
        name, (tms, nl, bytes_) = dom
        ach = bytes_ / (tms * 1e-3) / 1e9 if tms > 0 else 0.0
        ncu = ncu_profile("sort_pass") if name.startswith("sort_pass") else None
        roof = {"bound": "hbm", "kernel": name, "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                "traffic": ncu["traffic_bytes_per_launch"] if ncu else None, "traffic_source": ncu["source"] if ncu else None,
                "peak_source": peak_src, "launches": int(nl),
                "avg_launch_ms": tms / max(nl, 1), "algo_bytes_per_launch": bytes_ / max(nl, 1)}
    kernels = {n: {"ms_per_step": v[0] / steps, "launches_per_step": v[1] / steps,
                   "GBps": (v[2] / (v[0] * 1e-3) / 1e9 if v[0] > 0 else None)} for n, v in sorted(prof.items())}
    step_bytes = sum(v[2] for v in prof.values()) / steps
    kern_ms = sum(v[0] for v in prof.values()) / steps

    # ---- CPU baseline beside it (rank 0, bounded sample) --------------------------------------------------------
    cpu = None
    if not args.no_cpu:
        from oracle import Reference
        if not Reference.available():
            print("bench.py: cpu_baseline not measured: the reference engine (oracle/_ref) is not built", file=sys.stderr)
        else:
            sample = min(L, args.cpu_sample)
            n_cpu, tb, te, pr = cpu_reference(k, np.ascontiguousarray(np.asarray(seq_pin)[:sample]))
            cpu = {"value": n_cpu / (tb + te), "unit": "k-mers/s", "cores": 1, "kind": "reference",
                   "sample": f"first {sample} bases of the same sequence; reference seq_to_hash {tb:.2f}s + kmer_positions(2|8) loop {te:.2f}s, "
                             f"gcc -O2, 1 thread (the reference path is single-threaded); host has {os.cpu_count()} cores",
                   "build_only_value": n_cpu / tb}

    # ---- secondary workloads: the other BASELINE configs of this path, value only ---------------------------------
    secondary = {}
    if not args.no_secondary:
        for name in ("c3", "c2"):
            if name == args.workload:
                continue
            w2 = WORKLOADS[name]
            if w2["gen"] == w["gen"] and w2["L"] == L:
                sdev = seq_dev
            else:
                sdev = torch.from_numpy(gen_sequence(w2, w2["L"])).cuda()
            st2, N2, U2, keep = index_leg(kh, torch, sdev, w2["k"], steps, warm)
            ms2 = timed(torch, st2, max(5, steps // 2))
            secondary[name] = {"workload": w2["name"], "value": N2 / (ms2 * 1e-3), "unit": "k-mers/s", "ms_per_step": ms2,
                               "kmers": int(N2), "distinct": int(U2)}
            del keep, sdev

    R_key = (2 * k + 7) // 8
    survey_bytes = L + (36 + 24 * R_key) * N + 20 * U + (12 * U + 12 * N) + 8 * U
    step_roof = {"bound": "hbm", "what": "build + kmer.pos(2|8), all kernels of the step",
                 "algorithmic_bytes_as_built": int(step_bytes), "achieved": step_bytes / (ms * 1e-3) / 1e9,
                 "frac": step_bytes / (ms * 1e-3) / 1e9 / hbm_peak, "peak": hbm_peak, "unit": "GB/s",
                 "kernel_ms_sum": kern_ms,
                 "survey_formula_bytes": int(survey_bytes), "survey_formula_frac": survey_bytes / (ms * 1e-3) / 1e9 / hbm_peak,
                 "note": "frac = bytes the launched kernels must move (their own algorithmic bytes, summed) / step time; survey_formula_* "
                         f"charges SURVEY.md 8d's {R_key}-pass LSD sort by key although the grouped build runs fewer passes: equivalent "
                         "work, not a kernel efficiency"}
    h2d = L
    d2h = 8 * N + 4 * U
    cfg = config_of(w, k, L)
    hb = _lib.load().kmg_tune_get(b"hash_bits", int(N)) if k >= 21 else 0
    detail = {"kmers": int(N), "distinct": int(U),
              "kmer_order": (f"grouped (make.kmer.hash default for k >= 21: {hb // 8} radix passes on {hb} bits of a mix of the key, groups in "
                             "which k-mers sharing those bits interleave fixed up; do.sort=TRUE gives ascending keys)") if k >= 21 else "ascending key",
              "l2": "inputs_exceed_l2 (keys 8N + pos 4N bytes per pass >> 126 MB)"}
    return {"metric": METRIC, "value": N / (ms * 1e-3), "unit": "k-mers/s", "n_gpus": 1, "steps": steps,
            "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic", "config": cfg, "detail": detail,
            "e2e": {"value": N / (ms_e2e * 1e-3), "unit": "k-mers/s", "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "ms_per_step": ms_e2e,
                    "what": "make_kmer_hash(pinned host seq) + kmer_pos(2|8) into pinned host arrays"},
            "e2e_pageable": e2e_pageable,
            "gpu_launches": int(launches), "clocks": clk.summary(), "roofline": roof, "step_roofline": step_roof,
            "cpu_baseline": cpu, "probe": probe, "secondary": secondary, "kernels": kernels}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3k32", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"], help="N>1: one sequence cut N ways (default) or N times the sequence")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-probe", action="store_true")
    ap.add_argument("--no-pageable", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--cpu-sample", type=int, default=60_000_000)
    ap.add_argument("--dump-outputs", metavar="DIR", help="N=1: write the last timed step's outputs to DIR/pos.npy "
                    "and DIR/count.npy (the same seeded sample of 2^20 rows in every run)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.gpus != 1):
        ap.error("--dump-outputs needs --impl ours --gpus 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
