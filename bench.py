#!/usr/bin/env python
"""bench.py -- BASELINE.json's headline metric on B200, plus one short leg per other BASELINE config.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c2null|c1|c4|c5]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Headline (BASELINE.json configs[1] / [2], SURVEY.md 8(d) "C2/C3"): a 1 B-row table of 8 int8 columns in 32
hash-distributed columnar shards (stripe 150 000, chunk group 10 000, compression none, no NULLs), query
    SELECT key, sum(v), count(*) FROM t WHERE f < 50 GROUP BY key          -- 1 M groups
One step = one execution of that query over all shards: per-shard fused scan+filter+partial aggregate on the
GPU that owns the shard (shard s -> rank s mod N), then the coordinator combine (cg_comm_combine: ncclReduce
over NVLink at N > 1) and the compaction of the result rows.

  value   rows/s with the shards resident in HBM when the timed region starts
  e2e     rows/s through the C-ABI call on HOST page images (cg_scan_relation): pinned staging
          + cudaMemcpyAsync + kernel + device->host fetch of the result, all timed
  parity_full_size   every one of the 1 M groups of the combined result against the CPU oracle, at every N
  extra   short legs of the other BASELINE configs on the same N GPUs, each with rows/s, the roofline
          fraction of its dominant kernel, a bit-exact check against the oracle, sampled clocks, a CPU arm:
            c2null  C2 with 5 % NULLs in v            c1  4 shards, 10 M rows, sum(a) WHERE b < k
            c4      hash repartition of two 256 M-row tables + merge-side join
            c5      TPC-H Q1 + Q6 on a synthetic lineitem at SF100
  --impl reference  the CPU restatement of the reference's path (oracle/, one pinned thread per shard, shards
          written by the oracle's own row-at-a-time writer: nothing of citus_b200 is loaded) on the box's host
          cores -- NOT PostgreSQL/Citus, which cannot be built here
  --dump-outputs DIR  after the timed steps of the headline, the result rows of its last step as DIR/<name>.npy
          (see dump_c2_result); the inputs are seeded, so two builds can be compared output for output
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 20260922
NSHARDS = 32
STRIPE_ROWS = 150_000
CHUNK_ROWS = 10_000
NKEYS = 1_000_000
C2_COLUMNS = [(8, 0, 0, NKEYS, 0), (8, 0, 0, 100, 0), (8, 0, -10**9, 10**9, 0)] + [(8, 0, 0, 1 << 40, 0)] * 5
C2_QUALS = [(1, "<", 50)]
C2_GROUP = [0]
C2_BYTES_PER_ROW = 24.375                     # SURVEY.md 8(d): 3 projected int8 columns x (8 + 1/8)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=5)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--workload", default="c2", choices=["c2", "c2null", "c1", "c4", "c5"],
                   help="c2 = the headline (default; the other configs follow as short legs under `extra`); "
                        "any other value runs that leg alone and prints it as the line")
    p.add_argument("--no-extra", action="store_true", help="headline only")
    p.add_argument("--rows", type=int, default=1_000_000_000)
    p.add_argument("--resident", default="all", choices=["all", "projected"],
                   help="stage all 8 columns in HBM (default) or only the 3 the query reads")
    p.add_argument("--e2e-steps", type=int, default=5)
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-cpu", action="store_true")
    p.add_argument("--pageable", action="store_true", help="e2e from pageable host pages (host de-framing) instead of pinned pages (DMA)")
    p.add_argument("--gen-threads", type=int, default=0)
    p.add_argument("--compression", default="none", choices=["none", "lz4", "zstd"],
                   help="columnar.compression of the synthetic shards (BASELINE configs use none; lz4/zstd exercise the GPU decoders)")
    p.add_argument("--no-numa-bind", action="store_true", help="do not pin the rank to the CPUs of its GPU's NUMA node")
    p.add_argument("--leg-steps", type=int, default=5)
    p.add_argument("--leg-timeout", type=float, default=240.0, help="deadline in seconds for each extra leg")
    p.add_argument("--dump-outputs", metavar="DIR", help="write the result rows of the headline's last timed step as DIR/<name>.npy")
    a = p.parse_args()
    if a.steps < 1 or a.warmup < 0:
        p.error("--steps must be at least 1 and --warmup at least 0")
    if a.dump_outputs and (a.impl != "ours" or a.workload != "c2"):
        p.error("--dump-outputs writes the headline's result: it needs --impl ours and --workload c2")
    return a


class ClockSampler(threading.Thread):
    """samples SM clock and throttle reasons of one GPU during a timed region (NVML)"""

    BITS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"),
            (0x80, "hw_power_brake"))

    def __init__(self, index):
        super().__init__(daemon=True)
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.stop_flag = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:          # noqa
            log("clock sampling unavailable:", e)

    def sample_once(self):
        if not self.ok:
            return
        nv = self.nv
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            try:
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception:
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            for bit, name in self.BITS:
                if r & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def run(self):
        while self.ok and not self.stop_flag.is_set():
            self.sample_once()
            time.sleep(0.002)

    def result(self):
        self.stop_flag.set()
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": []}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": float(self.max_mhz),
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------- CPU arm (oracle)
CPU_SLICE = (0, 1)        # (rank, world): every rank pins its oracle threads inside its own slice of the cores


def pinned_cpus(nthreads):
    """one CPU per thread out of this process's affinity mask (SMT siblings are usually the second half of the
    numbering, so the picks come from the first half: distinct cores), inside this rank's slice of them"""
    cpus = sorted(os.sched_getaffinity(0))
    half = cpus[: max(len(cpus) // 2, 1)]
    r, w = CPU_SLICE
    per = max(len(half) // w, 1)
    mine = half[r * per:(r + 1) * per] or half
    if nthreads >= len(mine):
        return mine
    stride = len(mine) / nthreads
    return [mine[int(i * stride)] for i in range(nthreads)]


def run_pinned(work, items, nthreads):
    """work(item) for every item on `nthreads` threads, thread i pinned to one CPU (the oracle releases the GIL
    inside its C calls)"""
    cpus = pinned_cpus(nthreads)
    pending = list(items)
    lock = threading.Lock()
    errors = []

    def loop(i):
        try:
            os.sched_setaffinity(0, {cpus[i % len(cpus)]})
        except OSError:
            pass
        while True:
            with lock:
                if not pending:
                    return
                it = pending.pop(0)
            try:
                work(it)
            except Exception as e:          # noqa
                errors.append(e)
                return

    ths = [threading.Thread(target=loop, args=(i,)) for i in range(min(nthreads, max(len(pending), 1)))]
    t0 = time.time()
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    if errors:
        raise errors[0]
    return time.time() - t0


def oracle_attach(orc, rel, attlen, nstripes=None, atttype=None):
    v = rel.view
    return orc.Table.attach_view(v.pages, v.nblocks, C.cast(v.stripes, C.c_void_p), v.nstripes if nstripes is None else nstripes,
                                 C.cast(v.nodes, C.c_void_p), v.nnodes, attlen, atttype, chunk_row_limit=CHUNK_ROWS)


def cpu_scan(rels, attlen, quals, group, oaggs, nthreads, budget_s=20.0, full=False):
    """the oracle's restatement of the reference path over product-written shard images, one pinned thread per shard
    (the reference fans one task per shard out over <= citus.max_adaptive_executor_pool_size connections).
    Returns (rows, seconds, {shard: Result}, sample description, stripes used per shard)."""
    from oracle import oracle as orc
    orc.build()
    shard_ids = sorted(rels)
    total_stripes = rels[shard_ids[0]].view.nstripes
    use = total_stripes
    if not full:
        probe = min(3, total_stripes)
        t0 = time.time()
        oracle_attach(orc, rels[shard_ids[0]], attlen, probe).scan(quals, group, oaggs)
        per_stripe = (time.time() - t0) / probe
        waves = -(-len(shard_ids) // nthreads)
        if per_stripe * total_stripes * waves > budget_s:
            use = max(1, int(budget_s / (per_stripe * waves)))
    results = {}

    def work(s):
        results[s] = oracle_attach(orc, rels[s], attlen, min(use, rels[s].view.nstripes)).scan(quals, group, oaggs)

    secs = run_pinned(work, shard_ids, nthreads)
    rows = sum(r.rows_scanned for r in results.values())
    sample = (f"{len(shard_ids)} shards x {use}/{total_stripes} stripes = {rows} rows, one pinned thread per shard "
              f"({min(nthreads, len(shard_ids))} threads)")
    return rows, secs, results, sample, use


def dense_from_oracle(results, nkeys, sum_agg=0, count_agg=1):
    """dense [nkeys] arrays (sum as int64, count) of the merged oracle results; NULL-group entry last"""
    S = np.zeros(nkeys + 1, np.int64)
    Cn = np.zeros(nkeys + 1, np.int64)
    Nn = np.zeros(nkeys + 1, np.int64)           # non-NULL inputs of the sum
    for r in results.values():
        a = r.export_arrays()
        k = np.where(a["key_nulls"] != 0, nkeys, a["keys"])
        lo = a["sum_lo"][:, sum_agg].view(np.int64)
        assert np.array_equal(a["sum_hi"][:, sum_agg], lo >> 63), "oracle sum does not fit int64"
        np.add.at(S, k, lo)
        np.add.at(Cn, k, a["count"][:, count_agg])
        np.add.at(Nn, k, a["count"][:, sum_agg])
    return S, Cn, Nn


def dense_from_gpu(fetch, nkeys, sum_agg=0, count_agg=1):
    S = np.zeros(nkeys + 1, np.int64)
    Cn = np.zeros(nkeys + 1, np.int64)
    Nn = np.zeros(nkeys + 1, np.int64)
    n = fetch["n"]
    k = np.where(fetch["key_nulls"][:n] != 0, nkeys, fetch["keys"][:n])
    lo = fetch["sum_lo"][:n, sum_agg].view(np.int64)
    assert np.array_equal(fetch["sum_hi"][:n, sum_agg], lo >> 63)
    assert np.unique(k).shape[0] == n, "duplicate group in the result"
    S[k] = lo
    Cn[k] = fetch["count"][:n, count_agg]
    Nn[k] = fetch["count"][:n, sum_agg]
    return S, Cn, Nn


def dump_c2_result(out_dir, fetch, sum_agg=0, count_agg=1):
    """the rows of SELECT key, sum(v), count(*) ... GROUP BY key as the caller receives them (cg_partial_fetch), ordered
    by key with the NULL group last, one .npy per column: key, key_is_null, sum_v (NaN where sum(v) is NULL),
    count_star.  float64 holds every key, count and sum exactly (|value| < 2^53 is checked); 28 bytes per group, 28 MB
    for the headline's 1 M groups."""
    n = fetch["n"]
    kn = fetch["key_nulls"][:n] != 0
    keys = np.where(kn, 0, fetch["keys"][:n])
    lo = fetch["sum_lo"][:n, sum_agg].view(np.int64)
    assert np.array_equal(fetch["sum_hi"][:n, sum_agg], lo >> 63), "sum does not fit int64"
    exact = 1 << 53
    assert np.abs(keys).max(initial=0) < exact and np.abs(lo).max(initial=0) < exact, "not exact in float64"
    order = np.lexsort((keys, kn))
    cols = {"key": keys.astype(np.float64), "key_is_null": kn.astype(np.float32),
            "sum_v": np.where(fetch["count"][:n, sum_agg] > 0, lo.astype(np.float64), np.nan),
            "count_star": fetch["count"][:n, count_agg].astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in cols.items():
        np.save(os.path.join(out_dir, name + ".npy"), a[order])
    log(f"wrote {n} result rows ({sum(a.nbytes for a in cols.values()) / 1e6:.1f} MB) to {out_dir}")


def reduce_host_arrays(arrays, world):
    """sum of numpy int64 arrays over ranks to rank 0 (gloo; bookkeeping of the parity check, not the product path)"""
    if world == 1:
        return arrays
    import torch
    import torch.distributed as dist
    out = []
    for a in arrays:
        t = torch.from_numpy(np.ascontiguousarray(a))
        dist.reduce(t, dst=0, op=dist.ReduceOp.SUM)
        out.append(t.numpy())
    return out


# ----------------------------------------------------------------------------- reference arm
def run_reference(args, rank, world):
    """bench.py --impl reference: the CPU restatement of the reference's path on the host cores.  Loads nothing of
    citus_b200: the shards are written by the oracle's own row-at-a-time writer from the same counter-based
    synthetic rows (tests/test_host_cabi.py checks the two writers byte for byte)."""
    if rank != 0:
        return
    from oracle import oracle as orc
    orc.build()
    rows_per_shard = args.rows // NSHARDS
    ncpu = len(os.sched_getaffinity(0))
    nthreads = min(NSHARDS, max(1, ncpu // 2))
    attlen = [c[0] for c in C2_COLUMNS]
    oaggs = [orc.sum_(2), orc.count_star()]
    # calibrate on a two-stripe shard, then size every step to a bounded sample of the workload
    probe = orc.Table(attlen, stripe_row_limit=STRIPE_ROWS, chunk_row_limit=CHUNK_ROWS)
    probe.generate(C2_COLUMNS, 2 * STRIPE_ROWS, SEED, 0)
    t0 = time.time()
    probe.scan(C2_QUALS, C2_GROUP, oaggs)
    per_stripe = (time.time() - t0) / 2
    total_stripes = -(-rows_per_shard // STRIPE_ROWS)
    waves = -(-NSHARDS // nthreads)
    budget = min(12.0, 100.0 / max(args.warmup + args.steps, 1))
    use = total_stripes
    if per_stripe * total_stripes * waves > budget:
        use = max(1, int(budget / (per_stripe * waves)))
    sample_rows = min(rows_per_shard, use * STRIPE_ROWS)
    tables = {}

    def gen(s):
        t = orc.Table(attlen, stripe_row_limit=STRIPE_ROWS, chunk_row_limit=CHUNK_ROWS)
        t.generate(C2_COLUMNS, sample_rows, SEED, s * rows_per_shard)
        tables[s] = t

    gsecs = run_pinned(gen, range(NSHARDS), nthreads)
    log(f"reference arm: oracle writer produced {NSHARDS} shards x {sample_rows} rows in {gsecs:.1f}s")
    times, rows = [], 0
    for i in range(args.warmup + args.steps):
        results = {}

        def work(s):
            results[s] = tables[s].scan(C2_QUALS, C2_GROUP, oaggs)

        secs = run_pinned(work, range(NSHARDS), nthreads)
        rows = sum(r.rows_scanned for r in results.values())
        if i >= args.warmup:
            times.append(secs)
    secs = float(np.mean(times))
    value = rows / secs
    sample = (f"{NSHARDS} shards x {use}/{total_stripes} stripes = {rows} rows per step, one pinned thread per shard "
              f"({nthreads} threads); shards written by the oracle writer")
    emit({
        "impl": "reference", "metric": "rows/sec scan+GROUP BY over 1B-row columnar shards", "value": value,
        "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": secs * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "int64", "data": "synthetic", "config": c2_config(args, f"shard s -> GPU s mod {args.gpus}"),
        "reference_arm": "host cores, one pinned thread per shard: the reference's own parallelism for this workload -- one backend per "
                         "shard task, and a columnar scan is not parallel-aware (columnar_customscan.c:365-366, 417-421, 1337)",
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": nthreads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "CPU restatement of the reference path (oracle/oracle.c): PostgreSQL/Citus cannot be built here",
    })


def c2_config(args, where, nulls=False):
    return {"workload": "C2: 32 columnar shards, 1B rows x 8 int8 cols, WHERE f<50 GROUP BY key (1M keys), sum(v), count(*)"
                        + (" -- 5% NULLs in v" if nulls else ""),
            "rows": args.rows, "shards": NSHARDS, "stripe_row_limit": STRIPE_ROWS, "chunk_group_row_limit": CHUNK_ROWS,
            "groups": NKEYS, "selectivity": 0.5, "compression": args.compression, "parallelism": where,
            "l2_policy": "inputs (24.4 GB/step) are far larger than the 126 MB L2; no explicit flush"}


# ----------------------------------------------------------------------------- GPU arm: shared plumbing
class Env:
    """one rank's view of the run: device, library stream, communicator, timing helpers"""

    def __init__(self, args, rank, world, local_rank):
        import torch
        from citus_b200 import build
        self.args, self.rank, self.world, self.local_rank = args, rank, world, local_rank
        self.torch = torch
        if world > 1:
            import torch.distributed as dist
            dist.init_process_group("gloo")            # bootstrap + parity bookkeeping only; the data path is cg_comm_*
            self.dist = dist
        if rank == 0:
            build.build()
        if world > 1:
            self.dist.barrier()
        from citus_b200 import capi, columnar as cg, distributed as cgd
        self.capi, self.cg, self.cgd = capi, cg, cgd
        global CPU_SLICE
        CPU_SLICE = (rank, world)
        self.ncpu = len(os.sched_getaffinity(0))
        torch.cuda.set_device(local_rank)
        cg.init(local_rank)
        self.numa_node = -1 if args.no_numa_bind else cg.numa_bind()
        # one non-default torch stream for everything: the library's kernels and collectives, and the events that time them
        torch.cuda.set_stream(torch.cuda.Stream())
        cg.use_torch_stream()
        cgd.init(rank, world)
        self.peak, self.peak_src = measured_peak()

    def barrier(self):
        self.cgd.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        return self.cgd.allreduce([int(ms * 1e6)], "max")[0] / 1e6 if self.world > 1 else ms

    def sum_over_ranks(self, values):
        return self.cgd.allreduce([int(v) for v in values], "sum") if self.world > 1 else [int(v) for v in values]

    def timed(self, step, steps, warmup, profile=True):
        """`warmup` untimed steps, then exactly `steps` timed ones between barriers; CUDA events on the launching
        stream, max over ranks; clocks sampled while the GPU is inside the steps.
        Returns (ms per step, clocks, launches, scan launches, scan kernel ms total, last step() result)."""
        torch, capi = self.torch, self.capi
        for _ in range(warmup):
            step()
        self.barrier()
        sampler = ClockSampler(self.local_rank)
        sampler.start()
        if profile:
            capi.check(capi.lib().cg_profile_begin())
        before = capi.lib().cg_kernel_launches()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = None
        for _ in range(steps):
            out = step()
        e1.record()
        sampler.sample_once()
        while not e1.query():
            sampler.sample_once()
        self.barrier()
        clocks = sampler.result()
        launches = capi.lib().cg_kernel_launches() - before
        nscan, ktotal, kmax = C.c_int32(), C.c_double(), C.c_double()
        if profile:
            capi.check(capi.lib().cg_profile_collect(C.byref(nscan), C.byref(ktotal), C.byref(kmax)))
        ms = self.max_over_ranks(e0.elapsed_time(e1) / steps)
        return ms, clocks, int(launches), int(nscan.value), float(ktotal.value), out


def make_partial(env, rels, quals, group, aggs, total_rows, expected_groups=0, columns=None):
    """plan constants from the skip lists (key range, |term| bounds), agreed over the ranks, and the group table.
    A rank that owns no shard of the relation (world > shard count) still builds the same table and takes part in
    every collective: `columns` (the generator's column list) gives it the column descriptors."""
    cg = env.cg
    desc = cg.make_desc(quals, group, aggs, expected_groups=expected_groups)
    two = len(group) == 2
    lows, highs, bounds = None, None, [0] * len(aggs)
    for rel in rels.values():
        a, b, bs, _ = cg.relation_bounds(rel, desc)
        bounds = [max(x, y) for x, y in zip(bounds, bs)]
        if a > b:
            continue
        lo = [_s32(a), _s32(a >> 32)] if two else [a]          # two group columns travel packed (low 32 bits: the first)
        hi = [_s32(b), _s32(b >> 32)] if two else [b]
        lows = lo if lows is None else [min(x, y) for x, y in zip(lows, lo)]
        highs = hi if highs is None else [max(x, y) for x, y in zip(highs, hi)]
    ncomp = 2 if two else 1
    none = -(1 << 62)
    if env.world > 1:                      # identical table layout on every rank
        r = env.cgd.allreduce([(-x if lows else none) for x in (lows or [0] * ncomp)] +
                              [(x if highs else none) for x in (highs or [0] * ncomp)] + bounds, "max")
        lows = [-x for x in r[:ncomp]] if r[0] != none else None
        highs = r[ncomp:2 * ncomp] if r[0] != none else None
        bounds = r[2 * ncomp:]
    if lows is None:
        kmin, kmax = 0, -1
    elif two:
        kmin = _s64((lows[0] & 0xffffffff) | ((lows[1] & 0xffffffff) << 32))
        kmax = _s64((highs[0] & 0xffffffff) | ((highs[1] & 0xffffffff) << 32))
    else:
        kmin, kmax = lows[0], highs[0]
    for a, b in zip(aggs, bounds):
        a.term_abs_bound = b
    desc = cg.make_desc(quals, group, aggs, expected_groups=expected_groups)
    coldescs = next(iter(rels.values())).column_descs() if rels else [(c[0], 0) for c in columns]
    return cg.GpuColumnarAgg(desc, coldescs, kmin, kmax, total_rows), desc


def _s32(x):
    x &= 0xffffffff
    return x - (1 << 32) if x & 0x80000000 else x


def _s64(x):
    x &= (1 << 64) - 1
    return x - (1 << 64) if x & (1 << 63) else x


def roofline_of(env, algo_bytes_per_launch, nscan, ktotal_ms, steps, ms_per_step, kernel):
    avg_kernel_ms = ktotal_ms / max(nscan, 1)
    achieved = algo_bytes_per_launch / (avg_kernel_ms / 1e3) / 1e9 if avg_kernel_ms > 0 else 0.0
    return {"bound": "hbm", "achieved": achieved, "peak": env.peak, "unit": "GB/s", "frac": achieved / env.peak, "traffic": None,
            "kernel": kernel, "bytes_per_launch": algo_bytes_per_launch, "avg_launch_ms": avg_kernel_ms,
            "peak_source": env.peak_src, "kernel_share_of_step": (ktotal_ms / steps / ms_per_step) if ms_per_step > 0 else None}


def generate_shards(env, columns, shard_ids, rows_per_shard, seed, compression="none"):
    cg = env.cg
    threads = env.args.gen_threads or max(4, min(64, env.ncpu // max(env.world, 1)))
    cg.set_writer_compression(compression)
    t0 = time.time()
    try:
        rels = {s: cg.Relation.generate(columns, rows_per_shard, seed=seed, first_row=s * rows_per_shard,
                                        stripe_row_limit=STRIPE_ROWS, chunk_row_limit=CHUNK_ROWS, nthreads=threads) for s in shard_ids}
    finally:
        cg.set_writer_compression("none")
    log(f"rank {env.rank}: generated {len(shard_ids)} shards x {rows_per_shard} rows in {time.time() - t0:.1f}s")
    return rels


def sample_parity(env, rels, my_shards, attlen, quals, group, aggs, oaggs, nstripes, total_rows, budget_s=6.0):
    """bit-exact check of a leg on a bounded sample: the first `nstripes` stripes of every local shard through the GPU
    path (staged separately) against the oracle on the same stripes; every group, every aggregate.  Also times the
    oracle (the leg's CPU arm).  Returns (bit_exact, groups compared on rank 0, cpu rows, cpu secs, threads)."""
    from oracle import oracle as orc
    cg = env.cg
    orc.build()
    nthreads = max(1, min(len(my_shards), (env.ncpu // 2) // max(env.world, 1))) if my_shards else 1
    prefixes = {s: rels[s].prefix(min(nstripes, rels[s].view.nstripes)) for s in my_shards}
    results = {}

    def work(s):
        results[s] = oracle_attach(orc, prefixes[s], attlen).scan(quals, group, oaggs)

    secs = run_pinned(work, list(my_shards), nthreads) if my_shards else 0.0
    rows = sum(r.rows_scanned for r in results.values())
    ok = True
    ncompared = 0
    for s in my_shards:                                   # per shard: the GPU partial of this sample against the oracle's
        part, _ = make_partial(_Solo(env), {s: prefixes[s]}, quals, group, aggs, total_rows)
        sh = cg.Shard(prefixes[s])
        part.scan_shard(sh, want_stats=False)
        got = part.groups()
        want = results[s].groups()
        if not group:
            got = {0: list(got.values())[0]}
            want = {0: want.get(0, [dict(sum=0, count=0)] * len(aggs))}
        if set(got) != set(want):
            ok = False
        else:
            for k in want:
                for i, a in enumerate(aggs):
                    g, w = got[k][i], want[k][i]
                    if g["count"] != w["count"] or (a.kind == 2 and not a.is_float and w["count"] and g["sum"] != w["sum"]):
                        ok = False
        ncompared += len(want)
        sh.free()
        part.free()
    flags = env.sum_over_ranks([0 if ok else 1, ncompared, rows, int(secs * 1e6), nthreads])
    secs_max = env.cgd.allreduce([int(secs * 1e6)], "max")[0] / 1e6 if env.world > 1 else secs
    return flags[0] == 0, flags[1], flags[2], secs_max, flags[4]


class _Solo:
    """a world-of-one view of env for plan constants that must not be agreed across ranks (per-shard parity partials)"""

    def __init__(self, env):
        self.cg, self.cgd, self.world = env.cg, env.cgd, 1


# ----------------------------------------------------------------------------- headline: C2
def run_c2(env, args, nulls=False, headline=True):
    cg, cgd, capi, torch = env.cg, env.cgd, env.capi, env.torch
    rank, world = env.rank, env.world
    rows_per_shard = args.rows // NSHARDS
    total_rows = rows_per_shard * NSHARDS
    my_shards = cgd.shards_of_rank(NSHARDS, rank, world)
    columns = list(C2_COLUMNS)
    if nulls:
        columns[2] = (8, 0, -10**9, 10**9, 50000)            # 5 % NULLs in v (SURVEY.md 8(d))
    rels = generate_shards(env, columns, my_shards, rows_per_shard, SEED, args.compression if headline else "none")
    aggs = [cg.sum_(2), cg.count_star()]
    partial, desc = make_partial(env, rels, C2_QUALS, C2_GROUP, aggs, total_rows, columns=columns)
    nw, ops, dense, cap = partial.layout()
    log(f"rank {rank}: group table dense={dense} capacity={cap} words={nw}")
    t0 = time.time()
    stage_cols = None if (args.resident == "all" and headline) else [0, 1, 2]
    shards = {s: cg.Shard(rels[s], stage_cols) for s in my_shards}
    resident = sum(sh.device_bytes for sh in shards.values())
    log(f"rank {rank}: staged {len(shards)} shards, {resident / 1e9:.1f} GB resident in {time.time() - t0:.1f}s")
    out_keys = torch.empty(NKEYS + 2, dtype=torch.int64, device="cuda")
    out_nulls = torch.empty(NKEYS + 2, dtype=torch.uint8, device="cuda")
    out_words = torch.empty((NKEYS + 2) * nw, dtype=torch.int64, device="cuda")
    state = {"unpacked": False}

    def step():
        status = 0
        try:
            partial.reset()
            for s in my_shards:
                partial.scan_shard(shards[s], want_stats=False)
        except capi.CitusGpuError as e:
            status = e.code
            log(f"rank {rank}: scan failed: {e}")
        cgd.combine_partials(partial, dst=0, local_status=status)
        retry, n = 0, 0
        if rank == 0:
            try:
                n = partial.export_device(out_keys.data_ptr(), out_nulls.data_ptr(), out_words.data_ptr(), NKEYS + 2)
            except capi.CitusGpuError as e:
                if e.code != capi.CG_ERETRY_UNPACKED:
                    raise
                retry = 1
        return n, retry

    def checked_step():
        """outside the timed loop: a packed-accumulator overflow (detected exactly on the root) makes EVERY rank switch
        to the two-word path and run the query again"""
        n, retry = step()
        if world > 1:
            retry = cgd.allreduce([retry], "max")[0]
        if retry and not state["unpacked"]:
            log("packed accumulators overflowed: every rank falls back to the two-word path")
            partial.reset()
            partial.set_packing(False)
            state["unpacked"] = True
            n, _ = step()
        return n

    # algorithmic bytes per launch (one instrumented pass) and the overflow check before anything is timed
    partial.reset()
    algo_bytes, rows_scanned = [], 0
    for s in my_shards:
        st = partial.scan_shard(shards[s], want_stats=True)
        algo_bytes.append(st.bytes_scanned)
        rows_scanned += st.rows_scanned
    assert rows_scanned == rows_per_shard * len(my_shards)
    checked_step()

    steps, warmup = (args.steps, args.warmup) if headline else (args.leg_steps, 3)
    combine = None
    if world > 1:
        # which data path carries the combine is decided by measurement: a few steps each way, every rank sees the same
        # max-over-ranks times and therefore picks the same one
        combine = {}
        if cgd.peer_window():
            calib = {}
            for mode in (1, 0):
                cg.set_option("peer_window", mode)
                calib[mode] = env.timed(step, max(5, steps // 2), 3, profile=False)[0]
            best = 1 if calib[1] < 0.98 * calib[0] else 0          # a tie goes to ncclReduce (the peer path must win by 2 %)
            cg.set_option("peer_window", best)
            step()
            combine["calibration_ms_per_step"] = {"peer_window": calib[1], "ncclReduce": calib[0]}
        combine["data_path"] = ("peer window: every rank's packed words mapped into every rank (CUDA IPC); rank s sums slice s over "
                                "NVLink into the root's window; flag barriers in peer memory") if cgd.peer_window() else "ncclReduce"
    ms, clocks, all_launches, nscan, ktotal, last = env.timed(step, steps, warmup)
    ngroups = last[0] if last else 0
    if headline and args.dump_outputs and rank == 0:
        dump_c2_result(args.dump_outputs, partial.fetch())      # the partial still holds the last timed step's result
    value = total_rows / (ms / 1e3)
    if world > 1 and headline:
        # where a step's time goes on this rank (events between the phases; outside the timed loop)
        def phases(reps=10):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            acc = np.zeros(3)
            for _ in range(reps):
                env.barrier()
                ev[0].record()
                partial.reset()
                for s in my_shards:
                    partial.scan_shard(shards[s], want_stats=False)
                ev[1].record()
                cgd.combine_partials(partial, dst=0, local_status=0)
                ev[2].record()
                if rank == 0:
                    partial.export_device(out_keys.data_ptr(), out_nulls.data_ptr(), out_words.data_ptr(), NKEYS + 2)
                ev[3].record()
                torch.cuda.synchronize()
                acc += [ev[i].elapsed_time(ev[i + 1]) for i in range(3)]
            acc /= reps
            return {"reset_and_scans": float(acc[0]), "combine_incl_wait_for_slowest_rank": float(acc[1]),
                    "export_on_root": float(acc[2]), "reset_and_scans_max_over_ranks": env.max_over_ranks(float(acc[0]))}

        chosen = 1 if cgd.peer_window() else 0
        combine["phases_ms_rank0"] = phases()
        combine["phases_ms_rank0"]["note"] = ("every step starts at a barrier here, so waiting for the slowest rank shows up in the "
                                              "combine phase; in the timed loop the ranks run ahead of the root")
        if "calibration_ms_per_step" in combine:         # the other data path, for the record
            cg.set_option("peer_window", 1 - chosen)
            step()
            combine["phases_ms_rank0_other_path"] = phases()
            cg.set_option("peer_window", chosen)
            step()
    avg_bytes = float(np.mean(algo_bytes)) if algo_bytes else 0.0
    kernel = ("cg_jit_scan nullable form (exists bitmap + rank directory; fused decode+filter+partial aggregate)" if nulls else
              "cg_scan_fast_kernel<1,DENSE,1> (fused decode+filter+partial aggregate)")
    roofline = roofline_of(env, avg_bytes, nscan, ktotal, steps, ms, kernel)
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            roofline["traffic"] = json.load(f).get("dram_bytes_per_launch_c2null" if nulls else "dram_bytes_per_launch")
    except Exception:
        pass

    # ---- end to end on host buffers (headline only)
    e2e = None
    if headline and not args.no_e2e:
        t0 = time.time()
        pinned, refused = not args.pageable, None
        if pinned:
            try:
                for s in my_shards:           # pin the page images once
                    rels[s].register()
            except capi.CitusGpuError as e:
                refused = f"rank {rank}: {e}"
            if env.sum_over_ranks([refused is not None])[0]:
                # the OS would not pin every image (an unprivileged process can be refused): every rank times the
                # pageable path instead, and the line says so
                refused = refused or "refused on another rank"
                for s in my_shards:
                    rels[s].unregister()
                pinned = False
                log(f"rank {rank}: page images not pinned ({refused}); e2e uses pageable pages")
        reg_s = time.time() - t0
        if pinned:
            log(f"rank {rank}: registered {len(my_shards)} page images in {reg_s:.1f}s")
        partial.reset()
        h2d = 0
        for s in my_shards:                   # instrumented warm-up pass: bytes moved
            h2d += partial.scan_relation(rels[s], want_stats=True).h2d_bytes
        d2h = [0]

        def e2e_step():
            status = 0
            try:
                partial.reset()
                for s in my_shards:
                    partial.scan_relation(rels[s], want_stats=False)
            except capi.CitusGpuError as e:
                status = e.code
            cgd.combine_partials(partial, dst=0, local_status=status)
            if rank == 0:
                res = partial.fetch(reuse=True)   # device -> host read of the result rows, into caller-owned buffers
                d2h[0] = res["n"] * (9 + 8 * nw)

        ems, _, _, _, _, _ = env.timed(e2e_step, max(args.e2e_steps, 5), 1, profile=False)
        h2d = env.sum_over_ranks([h2d])[0]
        e2e = {"value": total_rows / (ems / 1e3), "unit": "rows/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h[0]), "ms_per_step": ems, "steps": max(args.e2e_steps, 5),
               "host_buffers": "pageable pages -> host de-frame into pinned blocks -> cudaMemcpyAsync" if not pinned else
                               "pinned (cudaHostRegister) page images -> 1-D DMA of whole pages -> GPU drops page headers + realigns",
               "assumption": None if not pinned else
                             f"the page images are pinned ONCE, outside the timed region ({reg_s:.1f} s for this rank's {len(my_shards)} shards "
                             f"here): what registering the shared_buffers segment at postmaster start would do; --pageable times the "
                             f"path that needs no registration",
               "api": "cg_scan_relation + cg_comm_combine + cg_partial_fetch", "numa_node": env.numa_node}
        if refused:
            e2e["pinning_refused"] = refused
        for s in my_shards:
            rels[s].unregister()

    # ---- CPU arm + parity of every group of the combined result, at every N
    cpu, parity = None, None
    cg.numa_unbind()                          # the CPU leg may use every core this rank is allowed
    if not args.no_cpu:
        from oracle import oracle as orc
        attlen = [c[0] for c in columns]
        oaggs = [orc.sum_(2), orc.count_star()]
        nthreads = max(1, min(len(my_shards), max(1, env.ncpu // 2) // world)) if my_shards else 1
        rows, secs, results, sample, use = cpu_scan(rels, attlen, C2_QUALS, C2_GROUP, oaggs, nthreads, full=True) \
            if my_shards else (0, 0.0, {}, "no shard on this rank", 0)
        if world == 1:
            cpu = {"value": rows / secs, "unit": "rows/s", "cores": nthreads, "kind": "port", "sample": sample}
        covered = env.sum_over_ranks([rows])[0]
        if covered == total_rows:             # the oracle covered the whole workload: compare every group after the combine
            S, Cn, Nn = dense_from_oracle(results, NKEYS)
            S, Cn, Nn = reduce_host_arrays([S, Cn, Nn], world)
            n = checked_step()
            if rank == 0:
                f = partial.fetch()
                gS, gC, gN = dense_from_gpu(f, NKEYS)
                same = bool(np.array_equal(S, gS) and np.array_equal(Cn, gC) and np.array_equal(Nn, gN))
                parity = {"groups": int((Cn > 0).sum()), "bit_exact": same, "n_gpus": world,
                          "checked": "sum(v), count(*) and the non-NULL input count of every group of the combined result "
                                     "(after cg_comm_combine) against the oracle over all shards"}
                if not same:
                    log("PARITY FAILURE at full size")
    line = None
    if rank == 0:
        line = {
            "metric": "rows/sec scan+GROUP BY over 1B-row columnar shards", "value": value, "unit": "rows/s",
            "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int64",
            "data": "synthetic", "config": c2_config(args, f"shard s -> GPU s mod {world}", nulls),
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(all_launches), "scan_kernel_launches": int(nscan),
            "roofline": roofline, "cpu_baseline": cpu, "groups": int(ngroups), "resident_bytes_rank0": int(resident),
            "hbm_gbs_whole_step": total_rows * C2_BYTES_PER_ROW / (ms / 1e3) / 1e9 / world,
            "packed_accumulators": not state["unpacked"],
        }
        if combine is not None:
            line["combine"] = combine
        if parity is not None:
            line["parity_full_size"] = parity
    for sh in shards.values():
        sh.free()
    partial.free()
    del rels, shards
    if world > 1:
        cg.set_option("peer_window", 1)          # the next leg measures its own choice
    return line


# ----------------------------------------------------------------------------- leg: C1
def run_c1(env, args):
    """BASELINE configs[0]: 4 shards, 10 M rows x 4 int8, SELECT sum(a) WHERE b < 250000 (25 %), and the same over a
    sorted filter column so that chunk-group skipping fires.  Parity at full size."""
    cg, cgd = env.cg, env.cgd
    rank, world = env.rank, env.world
    nsh, rows = 4, 10_000_000
    per = rows // nsh
    cols = [(8, 0, -(1 << 31), 1 << 31, 0), (8, 0, 0, 1_000_000, 0), (8, 0, 0, 1 << 40, 0), (8, 1, 0, 0, 0)]   # a, b, c, d = row id
    mine = cgd.shards_of_rank(nsh, rank, world)
    rels = generate_shards(env, cols, mine, per, 20260921)
    shards = {s: cg.Shard(rels[s]) for s in mine}
    out = {}
    from oracle import oracle as orc
    for name, quals in (("random_b", [(1, "<", 250_000)]), ("sorted_filter", [(3, "<", rows // 4)])):
        aggs = [cg.sum_(0), cg.count_star()]
        partial, desc = make_partial(env, rels, quals, [], aggs, rows, columns=cols)
        algo = []
        partial.reset()
        skipped = 0
        for s in mine:
            st = partial.scan_shard(shards[s], want_stats=True)
            algo.append(st.bytes_scanned)
            skipped += st.chunk_groups_filtered

        def step():
            partial.reset()
            for s in mine:
                partial.scan_shard(shards[s], want_stats=False)
            cgd.combine_partials(partial, dst=0)
            return partial.ngroups() if rank == 0 else 0

        ms, clocks, launches, nscan, ktotal, _ = env.timed(step, max(args.leg_steps, 10), 3)
        # parity at full size + CPU arm
        attlen = [8, 8, 8, 8]
        oaggs = [orc.sum_(0), orc.count_star()]
        results = {}
        nthreads = max(1, min(len(mine), 4)) if mine else 1

        def work(s):
            results[s] = oracle_attach(orc, rels[s], attlen).scan(quals, [], oaggs)

        secs = run_pinned(work, list(mine), nthreads) if mine else 0.0
        want_sum = sum(r.groups()[0][0]["sum"] for r in results.values() if r.groups())
        want_cnt = sum(r.groups()[0][1]["count"] for r in results.values() if r.groups())
        tot = env.sum_over_ranks([want_sum, want_cnt, sum(r.rows_scanned for r in results.values()), int(secs * 1e6), skipped])
        step()
        ok = None
        if rank == 0:
            g = list(partial.groups().values())[0]
            ok = bool(g[0]["sum"] == tot[0] and g[1]["count"] == tot[1])
        avg = float(np.mean(algo)) if algo else 0.0
        rf = roofline_of(env, avg, nscan, ktotal, max(args.leg_steps, 10), ms, "cg_scan_fast_kernel<1,GLOBAL,1>")
        out[name] = {"rows_per_s": rows / (ms / 1e3), "ms_per_step": ms, "frac": rf["frac"], "achieved_gbs": rf["achieved"],
                     "bytes_per_launch": avg, "avg_launch_ms": rf["avg_launch_ms"], "chunk_groups_skipped": int(tot[4]),
                     "bit_exact": ok, "clocks": clocks, "gpu_launches": launches,
                     "cpu_arm": {"value": tot[2] / max(tot[3] / 1e6 / max(min(world, nsh), 1), 1e-9), "unit": "rows/s", "kind": "port",
                                 "cores": nthreads * min(world, nsh), "sample": f"all {rows} rows, one thread per shard"}}
        partial.free()
    for sh in shards.values():
        sh.free()
    if rank != 0:
        return None
    return {"workload": "C1: 4 shards, 10M rows x 4 int8, SELECT sum(a) WHERE b < 250000 (and a sorted filter column)",
            "n_gpus": world, "note": "16.25 algorithmic B/row; at 10 M rows a launch moves 40 MB, so launch latency, not HBM, bounds it",
            "queries": out}


# ----------------------------------------------------------------------------- leg: C5
LINEITEM = [(8, 0, 100, 5100, 0),          # 0 l_quantity      1.00 .. 50.99   decimal(15,2) as scaled int8
            (8, 0, 90000, 10500000, 0),    # 1 l_extendedprice
            (8, 0, 0, 11, 0),              # 2 l_discount      0.00 .. 0.10
            (8, 0, 0, 9, 0),               # 3 l_tax
            (1, 0, 65, 68, 0),             # 4 l_returnflag
            (1, 0, 70, 72, 0),             # 5 l_linestatus
            (4, 0, -2922, -365, 0),        # 6 l_shipdate      days since 2000-01-01
            (4, 0, 1, 10001, 0)]           # 7 l_suppkey
TPCH_BYTES = {"q6": 28.5, "q1": 38.75}     # SURVEY.md 8(d)


def tpch_queries(cg):
    q6 = dict(quals=[(6, ">=", -2192), (6, "<", -1827), (2, ">=", 5), (2, "<=", 7), (0, "<", 2400)], group=[],
              aggs=[cg.Agg(2, [(1, 0, 1), (2, 0, 1)])])
    q1 = dict(quals=[(6, "<=", -486)], group=[4, 5],
              aggs=[cg.sum_(0), cg.sum_(1), cg.Agg(2, [(1, 0, 1), (2, 100, -1)]),
                    cg.Agg(2, [(1, 0, 1), (2, 100, -1), (3, 100, 1)]), cg.sum_(2), cg.count_star()])
    return {"q6": q6, "q1": q1}


def run_c5(env, args):
    """BASELINE configs[4]: TPC-H Q1 + Q6 on a synthetic lineitem at SF100 (600 M rows, 32 shards)."""
    cg, cgd = env.cg, env.cgd
    rank, world = env.rank, env.world
    rows = 600_000_000
    per = rows // NSHARDS
    mine = cgd.shards_of_rank(NSHARDS, rank, world)
    rels = generate_shards(env, LINEITEM, mine, per, 100)
    shards = {s: cg.Shard(rels[s], [0, 1, 2, 3, 4, 5, 6]) for s in mine}
    from oracle import oracle as orc
    attlen = [c[0] for c in LINEITEM]
    out = {}
    for name, q in tpch_queries(cg).items():
        partial, desc = make_partial(env, rels, q["quals"], q["group"], q["aggs"], per * NSHARDS, expected_groups=16, columns=LINEITEM)
        algo = []
        partial.reset()
        for s in mine:
            algo.append(partial.scan_shard(shards[s], want_stats=True).bytes_scanned)

        def step():
            partial.reset()
            for s in mine:
                partial.scan_shard(shards[s], want_stats=False)
            cgd.combine_partials(partial, dst=0)
            return partial.ngroups() if rank == 0 else 0

        ms, clocks, launches, nscan, ktotal, ng = env.timed(step, args.leg_steps, 3)
        oaggs = [orc.Agg(x.kind, list(x.factors), x.is_float) for x in q["aggs"]]
        ok, ncmp, crow, csec, cth = sample_parity(env, rels, mine, attlen, q["quals"], q["group"], q["aggs"], oaggs, 6, per * NSHARDS)
        count_ok = None
        if rank == 0 and name == "q1":
            g = partial.groups()
            count_ok = sum(v[5]["count"] for v in g.values()) > 0.9 * per * NSHARDS
        avg = float(np.mean(algo)) if algo else 0.0
        rf = roofline_of(env, avg, nscan, ktotal, args.leg_steps, ms, "cg_jit_scan (plan-specialised, NVRTC)")
        out[name] = {"rows_per_s": per * NSHARDS / (ms / 1e3), "ms_per_step": ms, "groups": int(ng or 0), "frac": rf["frac"],
                     "achieved_gbs": rf["achieved"], "bytes_per_row": TPCH_BYTES[name], "avg_launch_ms": rf["avg_launch_ms"],
                     "bit_exact": bool(ok) and (count_ok is not False), "parity": f"first 6 stripes of every shard (= {crow} rows), every group and "
                     f"aggregate of every shard's partial against the oracle ({ncmp} groups)", "clocks": clocks, "gpu_launches": launches,
                     "cpu_arm": {"value": crow / max(csec, 1e-9), "unit": "rows/s", "kind": "port", "cores": cth,
                                 "sample": f"{crow} rows (first 6 stripes of every shard), one pinned thread per shard"}}
        partial.free()
    for sh in shards.values():
        sh.free()
    if rank != 0:
        return None
    return {"workload": "C5: TPC-H Q1 + Q6, synthetic lineitem SF100 (600M rows, decimal(15,2) as scaled int8, dates as int4), 32 shards",
            "n_gpus": world, "queries": out}


# ----------------------------------------------------------------------------- leg: C4
def run_c4(env, args):
    """BASELINE configs[3]: two 256 M-row tables r(k, x), s(k, y) on a non-colocated key: hash repartition into
    P = 32 partitions (partition p -> rank p mod N) with cg_comm_repartition_exchange, then the merge-side join
    SELECT count(*), sum(x + y) FROM r JOIN s USING (k) over the co-located partitions."""
    cg, cgd, torch = env.cg, env.cgd, env.torch
    rank, world = env.rank, env.world
    rows = 256_000_000
    n = rows // world
    P = 32
    g = torch.Generator(device="cuda")
    tables = {}
    sums = {}
    for tname, seed in (("r", 11), ("s", 12)):
        g.manual_seed(seed * 1000 + rank)
        k = torch.randint(0, 1 << 28, (n,), dtype=torch.int64, device="cuda", generator=g)
        pay = torch.randint(-(1 << 40), 1 << 40, (n,), dtype=torch.int64, device="cuda", generator=g)
        tables[tname] = (k, pay)
        sums[tname] = (int(k.sum()), int(pay.sum()))
    torch.cuda.synchronize()

    def shuffle():
        got_r = cgd.repartition_exchange(0, [tables["r"][0].data_ptr(), tables["r"][1].data_ptr()], n, P)
        got_s = cgd.repartition_exchange(1, [tables["s"][0].data_ptr(), tables["s"][1].data_ptr()], n, P)
        cgd.exchange_wait(0)
        cgd.exchange_wait(1)
        return got_r, got_s

    def step():
        got_r, got_s = shuffle()
        r0, r1 = cgd.exchange_result(0, 2), cgd.exchange_result(1, 2)
        joined, jsum = cg.join_count_sum(r0["cols"][0], r0["cols"][1], r0["nrows"], r1["cols"][0], r1["cols"][1], r1["nrows"])
        return joined, jsum, got_r, got_s

    nccl_shuffle_ms = None
    if world > 1 and cgd.peer_window():                  # the same shuffle with NCCL send/recv as the data path
        cg.set_option("peer_window", 0)
        nccl_shuffle_ms = env.timed(shuffle, args.leg_steps, 2, profile=False)[0]
        cg.set_option("peer_window", 1)
    shuffle_ms, sclocks, slaunches, _, _, _ = env.timed(shuffle, args.leg_steps, 2, profile=False)     # the config's metric: the shuffle
    if nccl_shuffle_ms is not None and nccl_shuffle_ms < shuffle_ms:          # measured choice, the same on every rank
        cg.set_option("peer_window", 0)
        shuffle_ms, sclocks, slaunches, _, _, _ = env.timed(shuffle, args.leg_steps, 2, profile=False)
    ms, clocks, launches, _, _, last = env.timed(step, max(args.leg_steps // 2, 2), 1, profile=False)  # shuffle + merge-side join
    joined, jsum, got_r, got_s = last
    r0, r1 = cgd.exchange_result(0, 2, timing=True), cgd.exchange_result(1, 2, timing=True)
    ex_ms = env.max_over_ranks(r0["exchange_ms"] + r1["exchange_ms"])       # the two tables' exchanges run one after the other
    sent = env.sum_over_ranks([r0["sent_bytes"] + r1["sent_bytes"]])[0]
    # ---- checks: conservation, ownership, routing vs the oracle, the join vs an independent computation
    ok = True
    view = {}
    for slot, tname in ((0, "r"), (1, "s")):
        res = cgd.exchange_result(slot, 2)
        kk = cgd_device_view(torch, res["cols"][0], res["nrows"])
        pp = cgd_device_view(torch, res["cols"][1], res["nrows"])
        view[tname] = (kk, pp)
        tot = env.sum_over_ranks([sums[tname][0], sums[tname][1], int(kk.sum()), int(pp.sum()), res["nrows"],
                                  int(res["part_counts"].sum())])
        ok &= tot[0] == tot[2] and tot[1] == tot[3] and tot[4] == n * world and tot[5] == tot[4]
        mins, maxs = cgd.synthetic_intervals(P)
        idx = torch.empty(max(res["nrows"], 1), dtype=torch.int32, device="cuda")
        cnt = torch.empty(P, dtype=torch.int64, device="cuda")
        cg.worker_partition_query_result(res["cols"][0], None, res["nrows"], 8, "hash", mins, maxs, idx.data_ptr(), cnt.data_ptr())
        torch.cuda.synchronize()
        ok &= bool(((idx[: res["nrows"]] % world) == rank).all())
    from oracle import oracle as orc
    cpu = None
    if rank == 0:
        m = min(n, 1_000_000)
        mins, maxs = cgd.synthetic_intervals(P)
        idx = torch.empty(n, dtype=torch.int32, device="cuda")
        cnt = torch.empty(P, dtype=torch.int64, device="cuda")
        cg.worker_partition_query_result(tables["r"][0].data_ptr(), None, n, 8, "hash", mins, maxs, idx.data_ptr(), cnt.data_ptr())
        hk = tables["r"][0][:m].cpu().numpy()
        t0 = time.time()
        want_idx, _ = orc.partition_rows(hk, None, 8, "h", mins, maxs)
        t_route = time.time() - t0
        ok &= bool(np.array_equal(idx[:m].cpu().numpy(), want_idx))
        # the oracle's row-at-a-time join on a sample of this rank's co-located rows; also the CPU arm
        bk, bx = view["r"][0][:m].cpu().numpy(), view["r"][1][:m].cpu().numpy()
        pk, py = view["s"][0][:m].cpu().numpy(), view["s"][1][:m].cpu().numpy()
        t0 = time.time()
        wj, ws = orc.join_count_sum(bk, bx, pk, py)
        t_join = time.time() - t0
        gj, gs = cg.join_count_sum(view["r"][0][:m].data_ptr(), view["r"][1][:m].data_ptr(), m, view["s"][0][:m].data_ptr(),
                                   view["s"][1][:m].data_ptr(), m)
        ok &= (gj, gs) == (wj, ws)
        cpu = {"value": 2 * m / (2 * t_route + t_join), "unit": "rows/s", "kind": "port", "cores": 1,
               "sample": f"{m} rows per table: hashint8 + interval search per row, then the row-at-a-time join"}
    # full size: per-key build counts / payload sums by scatter_add over the 2^28 key domain, one gather per probe row
    (bk, bx), (pk, py) = view["r"], view["s"]
    cnt_r = torch.zeros(1 << 28, dtype=torch.int64, device="cuda").scatter_add_(0, bk, torch.ones_like(bk))
    sum_r = torch.zeros(1 << 28, dtype=torch.int64, device="cuda").scatter_add_(0, bk, bx)
    c = cnt_r[pk]
    term = sum_r[pk] + py * c
    want_joined = int(c.sum())
    want_sum = int((term & 0xFFFFFFFF).sum()) + (int((term >> 32).sum()) << 32)
    ok &= joined == want_joined and jsum == want_sum
    del cnt_r, sum_r, c, term
    lo, mid, hi = jsum & 0xFFFFFFFF, (jsum >> 32) & 0xFFFFFFFF, jsum >> 64
    tj = env.sum_over_ranks([joined, lo, mid, hi, 0 if ok else 1])
    peer_path = world > 1 and cgd.peer_window()
    if world > 1:
        cg.set_option("peer_window", 1)
    if rank != 0:
        return None
    total_sum = tj[1] + (tj[2] << 32) + (tj[3] << 64)
    hbm_bytes = 2 * rows * 32                     # SURVEY 8(d): read 16 + write 16 B/row on the map side
    return {"workload": "C4: hash repartition of r(k,x), s(k,y), 256M rows each, P=32, + merge-side join count(*), sum(x+y)",
            "n_gpus": world, "rows_per_s": 2 * rows / (shuffle_ms / 1e3), "ms_per_step": shuffle_ms, "partitions": P,
            "step": "routing + scatter + all-to-all of both tables (the shuffle); the join is timed on top of it below",
            "shuffle_plus_join": {"rows_per_s": 2 * rows / (ms / 1e3), "ms_per_step": ms, "join_ms": ms - shuffle_ms},
            "data_path": ("peer window: the scatter kernel stores rows into the owners' receive buffers over NVLink (CUDA IPC)"
                          if peer_path else "grouped ncclSend/ncclRecv" if world > 1 else "local"),
            "ms_per_step_with_nccl_sendrecv": nccl_shuffle_ms,
            "exchange_ms": ex_ms, "nvlink_gbs": (sent / 1e9) / (ex_ms / 1e3) if world > 1 and ex_ms > 0 else None,
            "nvlink_bytes": int(sent), "nvlink_peak_note": "900 GB/s per direction and GPU (NVLink 5)",
            "hbm_gbs_map_side": hbm_bytes / 1e9 / (shuffle_ms / 1e3) / world,
            "frac": hbm_bytes / 1e9 / (shuffle_ms / 1e3) / world / env.peak,
            "frac_note": "the whole shuffle step (routing + scatter + exchange of both tables) against SURVEY 8(d)'s 32 B/row of map-side "
                         "HBM traffic per GPU",
            "joined_rows": int(tj[0]), "sum_x_plus_y": str(total_sum), "bit_exact": tj[4] == 0,
            "checks": "key and payload checksums conserved, every received row belongs to a partition this rank owns, routing and the "
                      "join bit-exact against the oracle on 1 M rows, join count and 128-bit sum equal an independent scatter_add/gather "
                      "computation at full size",
            "clocks": sclocks, "gpu_launches": slaunches, "cpu_arm": cpu}


def cgd_device_view(torch, ptr, n):
    class _V:
        def __init__(self, p, n):
            self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i8", "data": (p, False), "version": 2}
    if n == 0:
        return torch.empty(0, dtype=torch.int64, device="cuda")
    return torch.as_tensor(_V(ptr, n), device="cuda")


# ----------------------------------------------------------------------------- driver
LEGS = {"c2null": lambda env, args: run_c2(env, args, nulls=True, headline=False), "c1": run_c1, "c4": run_c4, "c5": run_c5}


def run_ours(args, rank, world, local_rank):
    env = Env(args, rank, world, local_rank)
    try:
        if args.workload != "c2":
            leg = LEGS[args.workload](env, args)
            if rank == 0:
                emit(leg)
            return
        line = run_c2(env, args)
        extra = {}
        if not args.no_extra:
            # The headline is measured; the extra legs must not be able to lose it.  Each leg runs under a deadline: if
            # a rank is still inside the leg when it expires (a collective a peer never entered), rank 0 prints the line
            # with what it has and every rank leaves.  After each leg the ranks agree (gloo) on whether it failed anywhere.
            state = {"name": None, "timer": None}

            def expire():
                log(f"rank {rank}: leg {state['name']} passed its {args.leg_timeout}s deadline; giving up on the extra legs")
                if rank == 0:
                    extra[state["name"]] = {"error": f"deadline of {args.leg_timeout}s passed"}
                    line["extra"] = extra
                    emit(line)
                os._exit(0)

            for name in ("c2null", "c1", "c5", "c4"):
                t0 = time.time()
                state["name"] = name
                state["timer"] = threading.Timer(args.leg_timeout, expire)
                state["timer"].daemon = True
                state["timer"].start()
                failed = 0
                try:
                    leg = LEGS[name](env, args)
                except Exception as e:          # noqa -- a leg must not take the headline down with it
                    import traceback
                    log(f"rank {rank}: leg {name} failed:\n{traceback.format_exc()}")
                    leg = {"error": repr(e)} if rank == 0 else None
                    failed = 1
                if world > 1:                   # a peer stuck in a collective never arrives here: the deadline ends the run
                    t = env.torch.tensor([failed])
                    env.dist.all_reduce(t)
                    if int(t[0]) and not failed and rank == 0:
                        leg = {"error": f"leg failed on {int(t[0])} rank(s)"}
                state["timer"].cancel()
                if rank == 0:
                    if name == "c2null" and leg and "error" not in leg:
                        leg = {k: leg[k] for k in ("value", "unit", "ms_per_step", "steps", "roofline", "clocks", "gpu_launches",
                                                   "groups", "config", "cpu_baseline") if k in leg} | \
                              {"bit_exact": (leg.get("parity_full_size") or {}).get("bit_exact"), "parity": leg.get("parity_full_size")}
                    extra[name] = leg
                    log(f"leg {name}: {time.time() - t0:.1f}s")
        if rank == 0:
            line["extra"] = extra
            emit(line)
    finally:
        env.cgd.destroy()


_REAL_STDOUT = None


def emit(line: dict):
    """the ONE JSON line goes to the real stdout; everything else (NCCL banners, library
    chatter) was redirected to stderr at start-up"""
    data = (json.dumps(line) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            if dist.is_initialized():
                dist.destroy_process_group()


if __name__ == "__main__":
    main()
