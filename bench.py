#!/usr/bin/env python3
"""bench.py — merged postings/s of segment compaction on B200 (BASELINE.json configs[1]:
"compaction of 64 segments, 1M terms, 100M postings on 1 B200"), one JSON line on stdout.

A step = ONE compaction (ii2_merge_dev: k-way term merge + per-term union/dedup + removed
filter + intcomp encode, shard.go:158-212) of all resident segments of this rank's shard range.
  value      whole-job merged INPUT postings/s, segments resident in HBM, CUDA-event timed
  e2e        the same through the host-buffer C-ABI call ii2_merge (what cgo calls from
             Shard.Merge): pinned host inputs -> H2D -> kernels -> D2H of the new segment
  roofline   the dominant kernel's algorithmic bytes / its CUDA-event time vs measured HBM peak
  cpu_baseline  the CPU oracle (C restatement of the Go path) on a bounded sample, rank 0, N=1
  range_read_us  BASELINE configs[2] (N=1): term-range reads over 256 resident segments with the
             5 % removed filter, a single term and ranges of 0.1 / 1 / 10 / 100 % of the term
             space, median / p99 us
Multi-GPU: shards are independent (shard.go:19-20) -> one process per GPU, each compacting its
own term range, no data-path collective; `value` is weak scaling (every rank its own C2 shard
range).  `strong` (N > 1, BASELINE configs[4]): ONE synthetic index partitioned by the reference's
shardKey rule (shard.go:362-378) into contiguous shard-key ranges, build (ii2_ingest) + merge
timed per rank, with the imbalance of the partition; `cross_shard_read` gathers a read that spans
all ranks through the library's own NCCL exchange (ii2_read_gather) and checks it.
`--impl reference` times the CPU oracle with all host threads (InvertedIndex.Merge's worker
pool over shards, inverted_index.go:83-103) on bounded samples of the SAME workload.
`--dump-outputs DIR` writes the merged segment of the last timed step (rank 0) as .npy files;
the inputs depend only on the arguments, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the (possibly read-only) tree

import numpy as np  # noqa: E402

from inverted_index_2_b200 import synth  # noqa: E402
from inverted_index_2_b200.flat import FlatSegment  # noqa: E402

METRIC = "merged postings/s"
UNIT = "postings/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--terms", type=int, default=1_000_000)
    ap.add_argument("--segments", type=int, default=64)
    ap.add_argument("--postings", type=int, default=100_000_000)
    ap.add_argument("--removed-frac", type=float, default=0.05)
    ap.add_argument("--cpu-seconds", type=float, default=15.0,
                    help="target CPU time of the bounded cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-range-read", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--strong-postings", type=int, default=1_000_000_000,
                    help="total postings of the ONE index of the strong-scaling leg (N > 1)")
    ap.add_argument("--strong-cap", type=int, default=250_000_000,
                    help="postings one rank holds at most in the strong leg (host RAM / time)")
    ap.add_argument("--verify", action="store_true",
                    help="check the full-size result against an independent numpy union")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the merged segment of the last timed step to DIR/<name>.npy "
                         f"(float32 / float64; an array of more than {DUMP_CAP} values as a "
                         "seeded sample of them)")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs dumps the GPU merge (--impl ours)")
    return a


def workload_name(a):
    return (f"compaction of {a.segments} segments, {a.terms} terms, {a.postings} postings, "
            f"{a.removed_frac:g} of the id universe removed (synthetic terms.1m stand-in)")


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# --------------------------------------------------------------------------- CPU legs
def slice_prefix(w: synth.Workload, n_terms: int, first: int = 0) -> list[FlatSegment]:
    """Segments restricted to global term ids [first, first+n_terms) — a term-range shard."""
    out = []
    for seg, ids in zip(w.segments, w.seg_term_ids):
        a, b = np.searchsorted(ids, [first, first + n_terms])
        toff = seg.term_off[a:b + 1]
        poff = seg.post_off[a:b + 1]
        out.append(FlatSegment(seg.term_bytes[int(toff[0]):int(toff[-1])].copy(),
                               (toff - toff[0]).astype(np.uint32), seg.mode,
                               post=seg.post[int(poff[0]):int(poff[-1])].copy(),
                               post_off=(poff - poff[0]).astype(np.uint64)))
    return out


def cpu_rate_single(w: synth.Workload, target_s: float):
    """One oracle thread = one Shard.Merge (single goroutine per shard, shard.go:168-212)."""
    from oracle import orc
    n_terms = len(w.term_off) - 1
    probe = min(n_terms, 2000)
    segs = slice_prefix(w, probe)
    t0 = time.perf_counter()
    r = orc.merge(segs, w.removed, decoded=False)
    dt = max(time.perf_counter() - t0, 1e-4)
    rate = r.postings_in / dt
    want = int(min(n_terms, max(probe, probe * target_s / dt)))
    segs = slice_prefix(w, want)
    t0 = time.perf_counter()
    r = orc.merge(segs, w.removed, decoded=False)
    dt = time.perf_counter() - t0
    return r.postings_in / dt, f"first {want} of {n_terms} terms over all {len(w.segments)} " \
                               f"segments ({r.postings_in} postings, {dt:.1f} s, 1 thread)"


def cpu_step_parallel(shards, removed, threads):
    """All shards merged by `threads` workers (InvertedIndex.Merge, inverted_index.go:83-103)."""
    from concurrent.futures import ThreadPoolExecutor

    from oracle import orc
    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:  # ctypes releases the GIL inside orc_merge
        n = sum(r.postings_in for r in ex.map(lambda s: orc.merge(s, removed, decoded=False), shards))
    return n, time.perf_counter() - t0


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import orc
    orc.lib()
    cores = os.cpu_count() or 1
    # the SAME workload as the GPU arm (config.workload names it); every step merges a bounded
    # sample of it: the first `step_terms` terms, cut into term-range shards
    w = synth.make_workload(a.terms, a.segments, a.postings, removed_frac=a.removed_frac)
    n_terms = len(w.term_off) - 1
    # calibrate one shard, then size a step to ~10 s of wall time on all cores
    probe = slice_prefix(w, 1000)
    t0 = time.perf_counter()
    r = orc.merge(probe, w.removed, decoded=False)
    per_term = (time.perf_counter() - t0) / 1000
    budget = 240.0 / max(1, a.steps + a.warmup)
    step_terms = int(min(n_terms, max(cores * 200, min(10.0, budget) * cores / per_term)))
    per_shard = max(1, step_terms // (cores * 4))
    shards = [slice_prefix(w, per_shard, f) for f in range(0, step_terms - per_shard + 1, per_shard)]
    for _ in range(min(a.warmup, 1)):
        cpu_step_parallel(shards[:cores], w.removed, cores)
    tot_n = tot_t = 0
    for _ in range(a.steps):
        n, dt = cpu_step_parallel(shards, w.removed, cores)
        tot_n += n
        tot_t += dt
    value = tot_n / tot_t
    sample = (f"first {len(shards) * per_shard} of {n_terms} terms of the workload as {len(shards)} "
              f"term-range shards x {per_shard} terms over all {a.segments} segments "
              f"({tot_n // a.steps} postings per step), {cores} threads; inputs are decoded lists "
              f"(the input-side intcomp decode of file/reader.go:100 is not in the timed region, "
              f"as in the GPU arm's `value`)")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * tot_t / a.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32",
        "data": "synthetic",
        "config": {"workload": workload_name(a), "per_gpu": True,
                   "l2": "inputs (>= 1.3 GB per step) larger than the 126 MB L2"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, dev: int):
        self.dev, self.proc, self.lines = dev, None, []
        self.nv, self.nv_samples, self.nv_stop = None, [], threading.Event()

    def _nvml_index(self) -> int:
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        ids = [x.strip() for x in vis.split(",") if x.strip()]
        if ids and all(x.isdigit() for x in ids) and self.dev < len(ids):
            return int(ids[self.dev])
        return self.dev

    def _nvml_loop(self, h):
        import pynvml as nv
        bits = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self.nv_stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.nv_samples.append((float(sm), float(mx), [k for k, b in bits.items() if r & b]))
            except Exception:
                break
            time.sleep(0.002)

    def start(self):
        # the timed region of the default run is ~30 ms: an in-process NVML poll every 2 ms sees
        # it (the library calls release the GIL); nvidia-smi -lms 100 stays as the fallback
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self._nvml_index())
            self.nv = threading.Thread(target=self._nvml_loop, args=(h,), daemon=True)
            self.nv.start()
            return
        except Exception:
            self.nv = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.dev)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nv is not None:
            self.nv_stop.set()
            self.nv.join(timeout=2)
            if self.nv_samples:
                sm = [x[0] for x in self.nv_samples]
                return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(x[1] for x in self.nv_samples),
                        "reasons": sorted({r for x in self.nv_samples for r in x[2]}),
                        "samples": len(sm), "source": "NVML, 2 ms poll over the timed region"}
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML sample"], "samples": 0}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 6:
                continue
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except ValueError:
                continue
            for nm, v in zip(names, p[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}



# --------------------------------------------------------------------------- extra legs
def range_read_leg(eng, a):
    """BASELINE configs[2]: term-range reads over 256 resident segments, 5 % of the id universe
    removed (read + merge-style filter, quirk Q2), a single term and ranges of 0.1 / 1 / 10 / 100 %
    of the term space at 16 random positions (4 for the full range); wall clock per call,
    microseconds."""
    import torch
    w = synth.make_workload(a.terms, 256, a.postings, seed=0xC3, presence=0.125,
                            removed_frac=a.removed_frac)
    dsegs = [eng.upload(s) for s in w.segments]
    drem = eng.upload_removed(w.removed)
    n = len(w.term_off) - 1
    rng = np.random.default_rng(3)
    out = {}
    for frac in (0.0, 0.001, 0.01, 0.1, 1.0):  # 0 = a single term (min == max)
        span = max(1, int(n * frac))
        lat, info = [], None
        for _ in range(16 if frac < 1 else 4):
            lo = int(rng.integers(0, n - span + 1))
            tlo = synth.term_at(w.term_bytes, w.term_off, lo)
            thi = synth.term_at(w.term_bytes, w.term_off, lo + span - 1)
            ts = []
            for rep in range(4):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                r = eng.read_range_dev(dsegs, tlo, thi, drem)
                torch.cuda.synchronize()
                if rep:  # the first call of a position warms the caches
                    ts.append(time.perf_counter() - t0)
                info = r.info()
                r.release()
            lat.append(float(np.median(ts)))
        out["one_term" if frac == 0 else f"{frac:g}"] = {"median_us": 1e6 * float(np.median(lat)), "p99_us": 1e6 * float(np.max(lat)),
                            "terms": int(info.terms_count), "postings_in": int(info.postings_in),
                            "postings_out": int(info.postings_out)}
    for d in dsegs:
        d.release()
    drem.release()
    return {"workload": f"256 resident segments, {a.terms} terms, {w.postings_in} postings, "
                        f"{a.removed_frac:g} of the id universe removed; ii2_read_range_dev, "
                        f"wall clock per call", "by_range_fraction": out}


def strong_leg(eng, a, world, rank, dist, torch, barrier):
    """BASELINE configs[4]: ONE index partitioned by the reference's shardKey rule into contiguous
    shard-key ranges (one per rank): build (ii2_ingest of this rank's share of 64 documents) +
    merge (64 resident segments holding this rank's share of the postings), max over ranks."""
    import ctypes as C

    from inverted_index_2_b200 import _abi as A
    from inverted_index_2_b200 import sharded
    tb, off = synth.make_terms(a.terms, 0x1EE7)
    keys = sharded.shard_keys_of_sorted(tb, off)
    weights = np.bincount(keys, minlength=sharded.N_SHARD_KEYS).astype(np.float64)
    bounds = sharded.partition_shard_keys(weights, world)
    lo, hi = (int(x) for x in np.searchsorted(keys, [bounds[rank], bounds[rank + 1]]))
    n_mine, n_terms = hi - lo, len(off) - 1
    total = int(min(a.strong_postings, a.strong_cap * world))
    mine = synth.gather_terms(tb, off, np.arange(lo, hi))
    # (max_len 512: lists of ~31 values on average are not clipped, so the requested total is met)
    w = synth.make_workload(n_mine, a.segments, int(total * n_mine / n_terms), terms=mine,
                            seed=0xC5 + rank, removed_frac=a.removed_frac, max_len=512)
    dsegs = [eng.upload(s) for s in w.segments]
    drem = eng.upload_removed(w.removed)
    # ---- build: 64 documents, each holding a random half of this rank's terms, unsorted
    rng = np.random.default_rng(0xB1D + rank)
    ndocs = 64
    docs = (A.DocView * ndocs)()
    keep, doc_terms = [], 0
    for d in range(ndocs):
        ids = np.nonzero(rng.random(n_mine) < 0.5)[0]
        rng.shuffle(ids)
        dtb, doff = synth.gather_terms(mine[0], mine[1], ids)
        dtb = np.concatenate([dtb, np.zeros(8, dtype=np.uint8)])
        keep.append((dtb, doff))
        docs[d].n_terms = len(ids)
        docs[d].term_bytes = A.np_ptr(dtb, A.u8p)
        docs[d].term_off = A.np_ptr(doff, A.u32p)
        docs[d].value = d + 1
        doc_terms += len(ids)
    out = A.MergeOut()

    def build():
        eng._check(eng.lib.ii2_ingest(docs, ndocs, None, 0, 0, C.byref(out)), "ingest")
        t = int(out.terms_count)
        eng.lib.ii2_merge_out_free(C.byref(out))
        return t
    build()
    barrier()
    t0 = time.perf_counter()
    built_terms = build()
    torch.cuda.synchronize()
    build_s = time.perf_counter() - t0
    # ---- merge
    for _ in range(2):
        eng.merge_dev(dsegs, drem, encode=True).release()
    barrier()
    t0 = time.perf_counter()
    steps = max(1, min(a.steps, 5))
    for _ in range(steps):
        r = eng.merge_dev(dsegs, drem, encode=True)
        n_in = int(r.info().postings_in)
        r.release()
    torch.cuda.synchronize()
    merge_s = (time.perf_counter() - t0) / steps
    t = torch.tensor([build_s, merge_s], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    cnt = torch.tensor([float(n_in), float(doc_terms), float(n_mine)], device="cuda", dtype=torch.float64)
    allc = [torch.zeros_like(cnt) for _ in range(world)]
    dist.all_gather(allc, cnt)
    per_rank = [int(c[0].item()) for c in allc]
    tot_in, tot_docs = sum(per_rank), sum(int(c[1].item()) for c in allc)
    res = {"index": f"{n_terms} terms, {tot_in} postings in {a.segments} segments, partitioned by shardKey "
                    f"(shard.go:362-378) into {world} contiguous key ranges",
           "scaling": "strong", "total_postings": tot_in,
           "requested_postings": int(a.strong_postings), "shard_key_bounds": [int(x) for x in bounds],
           "live_shard_keys": int((weights > 0).sum()),
           "postings_per_rank": per_rank, "terms_per_rank": [int(c[2].item()) for c in allc],
           "imbalance_max_over_mean": max(per_rank) / (tot_in / world),
           "merge": {"ms_per_step": 1e3 * float(t[1].item()), "postings_per_s": tot_in / float(t[1].item()),
                     "api": "ii2_merge_dev on resident segments, wall clock, max over ranks"},
           "build": {"ms": 1e3 * float(t[0].item()), "doc_terms": tot_docs, "documents_per_rank": ndocs,
                     "doc_terms_per_s": tot_docs / float(t[0].item()),
                     "api": "ii2_ingest (host documents -> sorted, deduped, merged segment)"}}
    return res, w, dsegs, drem, built_terms


def cross_shard_read(eng, w, dsegs, world, rank, dist, torch, barrier, stream):
    """A read that spans every rank: each rank reads 1 % of its terms, the library's own NCCL
    exchange (ii2_read_gather, csrc/comm.cu) concatenates the results in rank order on rank 0;
    checked there against the ranks' local results."""
    import hashlib
    nt = len(w.term_off) - 1
    lo_t = synth.term_at(w.term_bytes, w.term_off, nt // 2)
    hi_t = synth.term_at(w.term_bytes, w.term_off, nt // 2 + max(1, nt // 100))

    def one(check):
        r = eng.read_range_dev(dsegs, lo_t, hi_t, None)
        g = eng.read_gather(r, 0)
        out = None
        if check:
            loc = r.download_read()
            dig = hashlib.sha256(b"".join(x.tobytes() for x in (loc.term_bytes, loc.term_off, loc.post,
                                                               loc.post_off))).hexdigest()
            sizes = (loc.n_terms, len(loc.term_bytes), len(loc.post))
            every = [None] * world
            dist.all_gather_object(every, (dig, sizes))
            if rank == 0:
                got = g.download_read()
                ok, t0, b0, p0 = True, 0, 0, 0
                for dg, (nt_r, nb_r, np_r) in every:
                    toff = (got.term_off[t0:t0 + nt_r + 1].astype(np.int64) - b0).astype(np.uint32)
                    poff = (got.post_off[t0:t0 + nt_r + 1] - np.uint64(p0)).astype(np.uint64)
                    part = hashlib.sha256(b"".join(x.tobytes() for x in (
                        got.term_bytes[b0:b0 + nb_r], toff, got.post[p0:p0 + np_r], poff))).hexdigest()
                    ok = ok and part == dg
                    t0, b0, p0 = t0 + nt_r, b0 + nb_r, p0 + np_r
                ok = ok and got.n_terms == t0 and len(got.post) == p0
                out = (bool(ok), int(got.n_terms), int(len(got.post)))
        g.release()
        r.release()
        return out
    checked = one(True)
    one(False)
    barrier()
    t0 = time.perf_counter()
    reps = 10
    for _ in range(reps):
        one(False)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / reps
    t = torch.tensor([dt], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    res = {"range": "1% of every rank's terms", "us_per_read": 1e6 * float(t.item()),
           "collective": "ii2_read_gather: one ncclAllGather of a 32-byte size record + one group of "
                         "ncclSend/ncclRecv straight into the root's result, offsets rebased by a kernel"}
    if checked is not None:
        res.update({"verified": checked[0], "gathered_terms": checked[1], "gathered_postings": checked[2]})
    return res


# --------------------------------------------------------------------------- GPU arm
def pin(arr: np.ndarray):
    """Copy into page-locked host memory (torch owns it); returns (numpy view, keep-alive)."""
    import torch
    t = torch.from_numpy(np.ascontiguousarray(arr)).pin_memory()
    return t.numpy(), t


# values kept per dumped array: the default workload's merged segment is ~300 MB; sampled, its
# dump (values + sample positions) is ~30 MB and stays below 64 MB for any workload
DUMP_CAP = 1 << 19


def dump_outputs(out_dir: str, m) -> None:
    """Writes the merged segment `m` (what ii2_result_download_merge hands a caller) as .npy
    files that two builds can compare value for value.  Integer arrays are stored exactly as
    float64 (bytes as float32); an array longer than DUMP_CAP is replaced by the values at
    DUMP_CAP positions drawn with a fixed seed from its length, and `<name>_idx.npy` holds those
    positions, so equal lengths give equal positions."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"term_bytes": m.term_bytes, "term_off": m.term_off, "val_off": m.val_off,
              "val_bytes": m.val_bytes,
              "min_term": np.frombuffer(m.min_term or b"", dtype=np.uint8),
              "max_term": np.frombuffer(m.max_term or b"", dtype=np.uint8),
              "counts": np.array([m.terms_count, m.terms_merged, m.postings_in, m.postings_out,
                                  m.val_size], dtype=np.uint64)}
    for seed, (name, arr) in enumerate(arrays.items()):
        if len(arr) > DUMP_CAP:
            idx = np.sort(np.random.default_rng(seed).choice(len(arr), DUMP_CAP, replace=False))
            np.save(os.path.join(out_dir, f"{name}_idx.npy"), idx.astype(np.float64))
            arr = arr[idx]
        np.save(os.path.join(out_dir, f"{name}.npy"),
                arr.astype(np.float32 if arr.dtype == np.uint8 else np.float64))


def run_ours(a):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from inverted_index_2_b200.engine import Engine
    eng = Engine(local)
    stream = torch.cuda.Stream()
    eng.set_stream(stream.cuda_stream)

    # this rank's term-range shard: its own term set and postings (weak scaling)
    w = synth.make_workload(a.terms, a.segments, a.postings, removed_frac=a.removed_frac,
                            seed=0xC2 + 1000 * rank, terms_seed=0x1EE7 + rank)
    dsegs = [eng.upload(s) for s in w.segments]
    drem = eng.upload_removed(w.removed)
    eng.sync()

    def step(keep=False):
        """One compaction; the result stays on the device (returned) only when `keep`."""
        res = eng.merge_dev(dsegs, drem, encode=True)
        info = res.info()
        out = (int(info.postings_in), int(info.postings_out), int(info.terms_count),
               int(info.term_bytes), int(info.val_size))
        if keep:
            return out, res
        res.release()
        return out, None

    for _ in range(a.warmup):
        step()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    clocks = ClockSampler(local)
    eng.prof_enable(True)
    barrier()
    clocks.start()
    l0 = eng.kernel_launches()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for i in range(a.steps):
        stats, last = step(keep=bool(a.dump_outputs) and i == a.steps - 1)
    ev1.record(stream)
    barrier()
    launches = eng.kernel_launches() - l0
    clk = clocks.stop()
    prof = eng.prof_read()
    eng.prof_enable(False)
    ms = ev0.elapsed_time(ev1)
    n_in, n_out, t_out, t_out_bytes, val_size = stats
    if last is not None:
        if rank == 0:
            dump_outputs(a.dump_outputs, last.download_merge(decoded=False))
        last.release()
    if world > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        tot = torch.tensor([n_in], device="cuda", dtype=torch.float64)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        total_in = float(tot.item())
    else:
        total_in = float(n_in)
    value = total_in * a.steps / (ms * 1e-3)

    # ---- roofline of the dominant kernel (per launch, live CUDA events) ----
    t_in = w.term_instances
    t_in_bytes = int(sum(int(s.term_off[-1]) for s in w.segments))
    n_groups = int(prof_terms) if (prof_terms := stats[2]) else 0  # distinct terms ~ terms out
    # K1b (grouping): term bytes, term and posting offsets and the postings themselves in (the
    # sources of every term are copied into its gather slot), gather slots + a 32 B record per
    # distinct term out
    k1b_bytes = (t_in_bytes + 4 * (t_in + a.segments) + 8 * (t_in + a.segments) + 4 * n_in
                 + 4 * n_in + 32 * n_groups)
    # K2b (union + dedup + filter + encode): records + gather slots + the removed bitmap in,
    # records + the `_val` staging stream out
    k2b_bytes = 32 * n_groups + 4 * n_in + len(w.removed) // 8 + 32 * n_groups + val_size
    # K12f (one bucket from its inputs to its finished output): term bytes, both offset arrays,
    # postings and the removed bitmap in; the merged terms, their offsets and the `_val` words out
    k12f_bytes = (t_in_bytes + 12 * (t_in + a.segments) + 4 * n_in + len(w.removed) // 8
                  + val_size + t_out_bytes + 12 * t_out)
    alg = {
        "k12f_bucket": k12f_bytes,
        "k1b_group": k1b_bytes,
        "k2b_union": k2b_bytes,
        # K6: records + staged `_val` words + surviving term bytes in; the new segment out
        "k6_emit": 32 * n_groups + val_size + t_out_bytes + val_size + t_out_bytes + 12 * t_out,
    }
    # dram__bytes_read.sum + dram__bytes_write.sum per launch from the `ncu --set full` capture
    # of this command (profiles/r03_ncu_full_metrics.csv; the fused kernel:
    # profiles/r02_ncu_k12f_2cta_metrics.csv); only valid for the default workload
    ncu_traffic = {"k12f_bucket": 1230.4e6 + 253.7e6, "k1b_group": 1278.1e6 + 456.8e6,
                   "k2b_union": 493.7e6 + 308.4e6, "k6_emit": 521.4e6 + 297.9e6}
    traffic_src = {"k12f_bucket": "ncu --set full, profiles/r02_ncu_k12f_2cta_metrics.csv"}
    default_workload = (a.terms, a.segments, a.postings, a.removed_frac) == \
        (1_000_000, 64, 100_000_000, 0.05) and world == 1
    peak, peak_src = peaks()
    roof = None
    if prof:
        top = max((e for e in prof if e["name"] in alg), key=lambda e: e["ms"])
        per_launch_ms = top["ms"] / max(1, top["count"])
        b = alg.get(top["name"])
        if b is not None and per_launch_ms > 0:
            ach = b / (per_launch_ms * 1e-3) / 1e9
            roof = {"bound": "hbm", "kernel": top["name"], "achieved": ach, "peak": peak,
                    "unit": "GB/s", "frac": ach / peak,
                    "traffic": ncu_traffic.get(top["name"]) if default_workload else None,
                    "traffic_source": traffic_src.get(top["name"],
                                                      "ncu --set full, profiles/r03_ncu_full_metrics.csv"),
                    "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": b, "ms_per_launch": per_launch_ms}
    pipeline_bytes = synth.algorithmic_bytes(n_in, n_out, t_in, t_in_bytes, a.segments, t_out,
                                             t_out_bytes, len(w.removed))
    pipe = {"algorithmic_bytes_per_step": pipeline_bytes,
            "achieved_gbs": pipeline_bytes / (ms * 1e-3 / a.steps) / 1e9}
    pipe["frac_of_peak"] = pipe["achieved_gbs"] / peak

    # ---- end to end through the host-buffer C-ABI call (rank-local, same workload) ----
    e2e = e2e_decoded = None
    if not a.no_e2e:
        keep, hsegs = [], []
        for s in w.segments:
            arrs = {}
            for f in ("term_bytes", "term_off", "post", "post_off"):
                arrs[f], k = pin(getattr(s, f))
                keep.append(k)
            hsegs.append(FlatSegment(arrs["term_bytes"], arrs["term_off"], s.mode, post=arrs["post"],
                                     post_off=arrs["post_off"]))
        hrem, k = pin(w.removed)
        keep.append(k)
        h2d = sum(x.term_bytes.nbytes + x.term_off.nbytes + x.post.nbytes + x.post_off.nbytes
                  for x in hsegs) + hrem.nbytes
        import ctypes as C

        from inverted_index_2_b200 import _abi as A
        from inverted_index_2_b200.flat import views_array
        arr = views_array(hsegs)
        out = A.MergeOut()

        def e2e_step():
            eng._check(eng.lib.ii2_merge(arr, len(hsegs), A.np_ptr(hrem, A.u32p), len(hrem), 0,
                                         C.byref(out)), "merge")
            d2h = (int(out.val_size) + 8 * int(out.terms_count) + 4 * (int(out.terms_count) + 1) +
                   int(out.term_off[int(out.terms_count)]))
            eng.lib.ii2_merge_out_free(C.byref(out))
            return d2h
        e_steps = max(1, min(a.steps, 5))

        def time_e2e(step_fn):
            for _ in range(2):
                d2h_ = step_fn()
            barrier()
            t0 = time.perf_counter()
            for _ in range(e_steps):
                step_fn()
            torch.cuda.synchronize()
            dt_ = time.perf_counter() - t0
            if world > 1:
                t_ = torch.tensor([dt_], device="cuda", dtype=torch.float64)
                dist.all_reduce(t_, op=dist.ReduceOp.MAX)
                dt_ = float(t_.item())
            return dt_, d2h_
        dt, d2h = time_e2e(e2e_step)
        e2e_dec = {"value": total_in * e_steps / dt, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                   "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * dt / e_steps,
                   "steps": e_steps, "api": "ii2_merge, II2_SEG_DECODED views (pinned decoded lists)"}
        # the call a Go host makes (INTEGRATION.md seam 1): `_val` views — the mmap of <key>_val
        # and the FST outputs of every term (file/reader.go:50-52,79-100), here as 32-bit word
        # offsets — staged per term range, decoded on the device, merged, new segment back
        vsegs = []
        for s_, hs in zip(w.segments, hsegs):
            words, woff = eng.intcomp_encode_batch(s_.post, s_.post_off)
            vb, k1 = pin(words.view(np.uint8))
            vo, k2 = pin(woff[:-1].astype(np.uint32))
            keep += [k1, k2]
            vsegs.append(FlatSegment(hs.term_bytes, hs.term_off, A.II2_SEG_VAL, val_bytes=vb,
                                     val_size=int(woff[-1]) * 4, val_woff32=vo))
        h2d_v = sum(x.term_bytes.nbytes + x.term_off.nbytes + x.val_bytes.nbytes + x.val_woff32.nbytes
                    for x in vsegs) + hrem.nbytes
        varr = views_array(vsegs)

        def e2e_val_step():
            eng._check(eng.lib.ii2_merge(varr, len(vsegs), A.np_ptr(hrem, A.u32p), len(hrem), 0,
                                         C.byref(out)), "merge")
            d2h_ = (int(out.val_size) + 8 * int(out.terms_count) + 4 * (int(out.terms_count) + 1) +
                    int(out.term_off[int(out.terms_count)]))
            eng.lib.ii2_merge_out_free(C.byref(out))
            return d2h_
        dtv, d2hv = time_e2e(e2e_val_step)
        e2e = {"value": total_in * e_steps / dtv, "unit": UNIT, "h2d_bytes_per_step": int(h2d_v),
               "d2h_bytes_per_step": int(d2hv), "ms_per_step": 1e3 * dtv / e_steps, "steps": e_steps,
               "api": "ii2_merge, II2_SEG_VAL views (pinned `_val` bytes + 32-bit FST word offsets): "
                      "H2D + device decode + merge + D2H of the new segment"}
        e2e_decoded = e2e_dec

    # ---- N > 1: the exchange behind the C-ABI, the strong-scaling leg, the cross-shard read ----
    xread = strong = None
    if world > 1:
        from inverted_index_2_b200 import sharded
        sharded.comm_init_from_torch(eng)
        xw, xsegs = w, dsegs
        if not a.no_strong:
            strong, sw, ssegs, srem, _ = strong_leg(eng, a, world, rank, dist, torch, barrier)
            xw, xsegs = sw, ssegs  # the read spans the ONE index: rank order == term order
        xread = cross_shard_read(eng, xw, xsegs, world, rank, dist, torch, barrier, stream)
        xread["index"] = "strong-leg index (one index, shardKey ranges)" if strong else "per-rank sets"
        eng.comm_shutdown()

    rread = None
    if world == 1 and rank == 0 and not a.no_range_read:
        rread = range_read_leg(eng, a)

    verified = None
    if a.verify and rank == 0:
        res = eng.merge_dev(dsegs, drem, encode=True, decoded=True).download_merge(decoded=True)
        terms, vals, poff = w.expected_union(w.removed)
        etb, eoff = synth.gather_terms(w.term_bytes, w.term_off, terms)
        verified = bool(np.array_equal(res.post, vals) and np.array_equal(res.post_off, poff) and
                        np.array_equal(res.term_bytes, etb) and np.array_equal(res.term_off, eoff))

    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        v, sample = cpu_rate_single(w, a.cpu_seconds)
        cpu = {"value": v, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": ms / a.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": workload_name(a), "per_gpu": True,
                       "l2": "inputs (>= 1.3 GB per step) larger than the 126 MB L2",
                       "postings_in": n_in, "postings_out": n_out, "terms_out": t_out,
                       "term_instances": t_in},
            "roofline": roof, "pipeline": pipe, "cpu_baseline": cpu, "e2e": e2e,
            "e2e_decoded": e2e_decoded,
            "gpu_launches": int(launches), "clocks": clk,
            "kernels": prof,
        }
        if verified is not None:
            line["verified_full_size"] = verified
        if xread is not None:
            line["cross_shard_read"] = xread
        if strong is not None:
            line["strong"] = strong
        if rread is not None:
            line["range_read_us"] = {k2: v["median_us"] for k2, v in rread["by_range_fraction"].items()}
            line["range_read"] = rread
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    a = parse()
    # exactly ONE line on stdout: libraries that write to file descriptor 1 (NCCL prints its
    # version banner there when NCCL_DEBUG is set) are pointed at stderr for the duration of the
    # run; the JSON line goes to the real stdout
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    out = os.fdopen(real, "w")
    global print
    _print = print

    def print(*args, **kw):  # noqa: A001 - only the JSON lines are printed in this module
        kw.setdefault("file", out)
        _print(*args, **kw)
        out.flush()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
