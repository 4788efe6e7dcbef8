#!/usr/bin/env python
"""bench.py — benchmarks of the sort / shuffle / aggregate hot path (BASELINE.json configs).

  python bench.py --gpus N --steps K --warmup W                  # this repo's CUDA path, headline = configs[1]
  python bench.py --impl reference --gpus N --steps K ...        # the reference's CPU algorithm on the host cores
  python bench.py --workload composite|pipeline ...              # configs[2] / configs[4] (see below)
  python bench.py ... --dump-outputs DIR                         # also writes a seeded sample of the last timed step's outputs

Workloads (a step = one pass of the hot path over one batch of synthetic input):
  sort      : configs[1]: 10^8 rows x 64 B (uint64 key + 56-byte payload) per GPU, sort by key.
              N = 1: ytgpu_sort_fixed_rows.  N > 1: weak scaling, ytgpu_shuffle_sort (sample -> pivots -> partition ->
              fused NVLink peer scatter -> local sort, all behind the C ABI).  --keys uniform|zipf|sorted selects the key
              distribution (SURVEY §8d C2 variants), the default line carries them as `variants`.
  composite : configs[2]: (k1 uint64 ~U[0,2^16), k2 string[16], payload[40]), sort by (k1, k2).
  pipeline  : configs[4]: (key uint64 ~U[0,10^7), val int64, payload[48]): shuffle-sort by key, then segmented
              SUM(val), COUNT(*) over the sorted rows (ytgpu_reduce_sorted_fixed_rows, no hash table).
`value` is whole-job rows/s with inputs resident in HBM; `e2e` is the same step through the C ABI with HOST (pinned)
buffers, H2D and D2H inside the timed region.  Every N > 1 run VERIFIES its last timed step (per-rank sortedness, rank
boundaries, row count, an order-independent checksum of whole rows, tie stability) and exits non-zero on a mismatch.
One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the (possibly read-only) tree as the build left it

SEED = 0x5954534155525553  # "YTSAURUS" (SURVEY §8d)
ROW_BYTES = 64
METRIC = "rows/s sorted (64B rows, u64 key)"
ALGO_BYTES_PER_ROW_PASS = 24.0   # onesweep pass: read 8 B key + 4 B index, write the same
ALGO_BYTES_PER_ROW_SORT = 332.0  # SURVEY §8(d): 8 + 8*24 + 4 + 2*64
NVLINK_PEER_GBS = 770.0          # measured peer copy per direction per GPU on this pool (B200_PROFILING.md; 900 nominal)
MIN64 = -2**63


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples SM clocks / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        self._nv = self._h = None
        try:  # NVML is initialised BEFORE the timed region so that the first sample lands inside it
            import pynvml as nv
            nv.nvmlInit()
            self._nv, self._h = nv, nv.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self._h, nv.NVML_CLOCK_SM)
        except Exception as e:  # pragma: no cover
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def _sample(self):
        nv, h = self._nv, self._h
        self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
        try:
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        for bit, name in names.items():
            if bit and (r & bit):
                self.reasons.add(name)

    def _run(self):
        if self._nv is None:
            return
        try:
            while not self._stop.is_set():
                self._sample()
                time.sleep(0.004)
        except Exception as e:  # pragma: no cover
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def __enter__(self):
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._thread.join(timeout=2)

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "samples": len(self.samples), "reasons": sorted(self.reasons)}


# ------------------------------------------------------------------------------------------------------------
# synthetic tables (device side, Philox via torch's CUDA generator)
# ------------------------------------------------------------------------------------------------------------
def _mix64(x):
    """splitmix64 finaliser on int64 tensors (wrapping arithmetic; logical shifts emulated)."""
    def lsr(v, s):
        return (v >> s) & ((1 << (64 - s)) - 1)
    x = (x ^ lsr(x, 30)) * -4658895280553007687   # 0xBF58476D1CE4E5B9
    x = (x ^ lsr(x, 27)) * -7723592293110705685   # 0x94D049BB133111EB
    return x ^ lsr(x, 31)


def gen_rows_device(n, device, rank, workload="sort", keys="uniform"):
    """[n, 8] int64 rows.  Word 6 = source rank, word 7 = position (the verifier reads them back: integrity and
    tie stability); everything else follows the workload's schema."""
    import torch
    g = torch.Generator(device=device).manual_seed(SEED + rank)
    rows = torch.empty((n, 8), dtype=torch.int64, device=device)
    chunk = 1 << 24
    for s in range(0, n, chunk):
        e = min(n, s + chunk)
        rows[s:e] = torch.randint(MIN64, 2**63 - 1, (e - s, 8), dtype=torch.int64, device=device, generator=g)
    rows[:, 6] = rank
    rows[:, 7] = torch.arange(n, device=device, dtype=torch.int64)
    if workload == "composite":
        rows[:, 0] &= 0xFFFF                              # k1 ~ U[0, 2^16); k2 = words 1..2 (16 random bytes)
    elif workload == "pipeline":
        rows[:, 0] = torch.remainder(rows[:, 0], 10_000_000)   # key ~ U[0, 10^7); val = word 1
        rows[:, 1] >>= 20                                      # |val| < 2^43: sums stay far from wrapping for checks
    elif keys in ("zipf", "zipf_hashed"):
        # Zipf(1.1) over 10^6 distinct values through the inverse CDF ("maniac" keys): the value's rank is the key, or
        # (zipf_hashed) its 64-bit hash — duplicates spread over the whole key space
        m = 1_000_000
        w = torch.arange(1, m + 1, device=device, dtype=torch.float64).pow(-1.1)
        cdf = torch.cumsum(w, 0)
        cdf /= cdf[-1].clone()
        for s in range(0, n, chunk):
            e = min(n, s + chunk)
            u = torch.rand(e - s, device=device, dtype=torch.float64, generator=g)
            ranks = torch.searchsorted(cdf, u).to(torch.int64) + 1
            rows[s:e, 0] = _mix64(ranks) if keys == "zipf_hashed" else ranks
    elif keys == "sorted":
        k = rows[:, 0] ^ MIN64
        rows[:, 0] = torch.sort(k).values ^ MIN64          # ascending as unsigned
    return rows.view(torch.uint8).reshape(-1)


def key_columns_of(workload):
    from ytsaurus_b200.rowset import EValueType as T
    if workload == "composite":
        return [(0, 0, T.Uint64, 0, 1), (8, 16, T.String, 0, 1)]
    return [(0, 0, T.Uint64, 0, 1)]


# ------------------------------------------------------------------------------------------------------------
# verification of a (distributed) sort result — torch ops only, outside every timed region
# ------------------------------------------------------------------------------------------------------------
def _bswap64(x):
    """Byte swap of int64 words (string key bytes -> big-endian integers) with shifts only."""
    r = None
    for i in range(8):
        b = (x >> (8 * i)) & 0xFF
        t = b << (8 * (7 - i))
        r = t if r is None else (r | t)
    return r


def sortable_key_words(rows2d, key_cols):
    """Key columns -> list of int64 tensors whose SIGNED lexicographic order equals the key order."""
    from ytsaurus_b200.rowset import EValueType as T
    words = []
    for off, width, typ, desc, _req in key_cols:
        if typ == T.String:
            assert off % 8 == 0 and width % 8 == 0
            ws = [_bswap64(rows2d[:, off // 8 + j]) ^ MIN64 for j in range(width // 8)]
        elif typ == T.Uint64:
            ws = [rows2d[:, off // 8] ^ MIN64]
        else:
            ws = [rows2d[:, off // 8].clone()]
        words += [~w for w in ws] if desc else ws
    return words


def _lex_cmp(a, b):
    """-> (less, equal) boolean tensors for lists of int64 word tensors."""
    import torch
    less = torch.zeros_like(a[0], dtype=torch.bool)
    eq = torch.ones_like(a[0], dtype=torch.bool)
    for x, y in zip(a, b):
        less |= eq & (x < y)
        eq &= x == y
    return less, eq


def _row_checksum(rows2d):
    """Order-independent checksum of whole rows: sum over rows of a non-linear mix of all 8 words (wrapping int64)."""
    h = rows2d[:, 0] * -7046029254386353131
    for j in range(1, rows2d.shape[1]):
        h = _mix64(h + rows2d[:, j] * (2 * j + 1))
    return h.sum(), (h * h).sum()


def verify_sort(out_flat, in_flat, row_bytes, key_cols, world=1, rank=0, dist=None, origin=(6, 7)):
    """Checks that `out` (this rank's slice of the result) is the stable sort of the union of all ranks' `in`:
    sorted inside the rank, rank r's last key <= rank r+1's first key (ties across ranks ordered by origin), same row
    count, same multiset of rows (checksums), equal keys keep (source rank, position) order."""
    import torch
    dev = out_flat.device
    o = out_flat.view(torch.int64).view(-1, row_bytes // 8)
    i = in_flat.view(torch.int64).view(-1, row_bytes // 8)
    res = {}
    kw = sortable_key_words(o, key_cols)
    m = o.shape[0]
    if m > 1:
        less, eq = _lex_cmp([w[:-1] for w in kw], [w[1:] for w in kw])
        res["sorted_in_rank"] = bool((less | eq).all())
        org = o[:, origin[0]] * (1 << 40) + o[:, origin[1]]
        res["ties_stable"] = bool((org[1:] > org[:-1])[eq].all())
    else:
        res["sorted_in_rank"] = res["ties_stable"] = True
    cs_out, cs_in = _row_checksum(o), _row_checksum(i)
    tot = torch.stack([torch.tensor(m, device=dev), cs_out[0], cs_out[1], torch.tensor(i.shape[0], device=dev), cs_in[0], cs_in[1]])
    nk = len(kw)
    edge = torch.zeros(2 * nk + 3, dtype=torch.int64, device=dev)  # [first key words][last key words] first_origin last_origin count
    if m:
        edge[:nk] = torch.stack([w[0] for w in kw])
        edge[nk:2 * nk] = torch.stack([w[-1] for w in kw])
        edge[2 * nk] = o[0, origin[0]] * (1 << 40) + o[0, origin[1]]
        edge[2 * nk + 1] = o[-1, origin[0]] * (1 << 40) + o[-1, origin[1]]
    edge[2 * nk + 2] = m
    if world > 1:
        dist.all_reduce(tot)
        edges = [torch.zeros_like(edge) for _ in range(world)]
        dist.all_gather(edges, edge)
        edges = [e.cpu().tolist() for e in edges]
    else:
        edges = [edge.cpu().tolist()]
    tot = tot.cpu().tolist()
    res["row_count"] = tot[0] == tot[3]
    res["checksum"] = tot[1] == tot[4] and tot[2] == tot[5]
    ok_edges = True
    prev = None
    for e in edges:
        if e[2 * nk + 2] == 0:
            continue
        if prev is not None:
            a, b = prev[nk:2 * nk], e[:nk]
            if a > b or (a == b and prev[2 * nk + 1] >= e[2 * nk]):
                ok_edges = False
        prev = e
    res["rank_boundaries"] = ok_edges
    ok = all(res.values())
    return {"ok": ok, "ranks": world, "rows": tot[0], "checks": res,
            "what": "per-rank sortedness, rank r last key <= rank r+1 first key, global row count, order-independent "
                    "checksum of whole rows, equal keys keep (source rank, position) order"}


def dump_outputs(dirname, outputs, world, rank):
    """Writes what the last timed step returned, so that two builds can be compared output for output: for every output
    (name -> (int64 tensor [rows, words], row budget)) a fixed, seeded sample of its rows as <name>.npy, every 64-bit word
    split into its low and high 32-bit halves (exact in float64), and the sampled row indices as <name>_index.npy.
    The budgets over all ranks keep the files under 64 MB."""
    import torch
    os.makedirs(dirname, exist_ok=True)
    prefix = f"rank{rank}_" if world > 1 else ""
    for name, (t, budget) in outputs.items():
        m = t.shape[0]
        k = min(m, budget // world)
        idx = np.sort(np.random.default_rng(SEED).choice(m, k, replace=False))
        s = t[torch.from_numpy(idx).to(t.device)].cpu().numpy()
        np.save(os.path.join(dirname, f"{prefix}{name}.npy"), s.view(np.uint32).reshape(k, -1).astype(np.float64))
        np.save(os.path.join(dirname, f"{prefix}{name}_index.npy"), idx.astype(np.float64))


# ------------------------------------------------------------------------------------------------------------
# GROUP BY (configs[3]) — secondary metric, with its own CPU baselines
# ------------------------------------------------------------------------------------------------------------
def bench_groupby(ctx, args, device, peak, world, rank, dist):
    """SELECT key, SUM(val), COUNT(*) GROUP BY key over a columnar chunk (key uint64, val int64) resident in HBM.
    Algorithmic traffic: 16 B/row in + 24 B/group out (SURVEY §8d).  N > 1: every rank holds its own chunk; partial
    states are hash-partitioned over the ranks and merged (distributed_groupby)."""
    import torch
    from ytsaurus_b200 import Column, capi
    from ytsaurus_b200.rowset import EValueType as T
    from ytsaurus_b200.shuffle import distributed_groupby
    n = args.groupby_rows
    g = torch.Generator(device=device).manual_seed(SEED + 4 + rank)
    vals = torch.randint(-2**40, 2**40, (n,), dtype=torch.int64, device=device, generator=g)
    out = {"unit": "rows/s", "rows_per_gpu": n, "n_gpus": world, "columns": "key uint64, val int64",
           "timing": "median of 7 individually timed calls (CUDA events), max over ranks; kernel_ms = mean group-by kernel launch", "cases": []}

    def timed(fn, steps=7, warm=3):
        """-> (result, MEDIAN ms per step over `steps` individually timed calls, max over ranks; group-by kernel ms).  A call
        is ~0.5-3 ms with three host round trips inside, so a single host hiccup would dominate a mean."""
        for _ in range(warm):
            fn()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ctx.enable_timers(True)
        ctx.reset_timers()
        per = []
        for _ in range(steps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn()
            e1.record()
            torch.cuda.synchronize()
            per.append(e0.elapsed_time(e1))
        ms = torch.tensor([float(np.median(per))], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        kms, kl = ctx.kernel_ms(capi.KC_GROUPBY)
        ctx.enable_timers(False)
        return r, float(ms.item()), kms / max(kl, 1)

    def case(name, kc, vc, groups, pred=None, packed_bytes=None, expect_rows=None):
        hint = groups
        fn = (lambda: distributed_groupby(ctx, kc, vc, pred, group_count_hint=hint)) if world > 1 else \
             (lambda: ctx.scan_filter_groupby(kc, vc, pred, group_count_hint=hint, capacity=min(n, groups) + 2))
        res, ms, kms = timed(fn)
        cnt = res["count"].to(torch.int64).sum()
        if world > 1:
            dist.all_reduce(cnt)
        if expect_rows is not None:
            assert int(cnt) == expect_rows, f"{name}: COUNT(*) sums to {int(cnt)}, expected {expect_rows}"
        algo = (packed_bytes if packed_bytes is not None else 16.0 * n) + 24.0 * min(groups, n)
        out["cases"].append({"name": name, "groups": groups, "value": n * world / (ms / 1e3), "ms_per_step": ms,
                             "kernel_ms": kms, "roofline_frac": algo / (kms / 1e3) / 1e9 / peak, "algorithmic_bytes": algo})

    keys3 = torch.randint(0, 1000, (n,), dtype=torch.int64, device=device, generator=g)
    keys6 = torch.randint(0, 1_000_000, (n,), dtype=torch.int64, device=device, generator=g)
    vcol = Column(T.Int64, values=vals)
    case("direct64, 10^3 groups", Column(T.Uint64, values=keys3), vcol, 1000, expect_rows=n * world)
    case("direct64, 10^6 groups", Column(T.Uint64, values=keys6), vcol, 1_000_000, expect_rows=n * world)
    if not args.quick:
        # SURVEY §8d C4 variants
        ks = torch.sort(keys6).values
        case("direct64, 10^6 groups, sorted keys", Column(T.Uint64, values=ks), vcol, 1_000_000, expect_rows=n * world)
        runs = torch.cat([torch.zeros(1, dtype=torch.int64, device=device), torch.nonzero(ks[1:] != ks[:-1]).flatten() + 1])
        case("RLE keys (sorted), 10^6 groups", Column(T.Uint64, values=ks[runs].contiguous(), rle_indexes=runs, value_count=n), vcol,
             1_000_000, packed_bytes=8.0 * n + 16.0 * runs.numel(), expect_rows=n * world)
        del ks, runs
        dict_vals = torch.arange(1000, dtype=torch.int64, device=device) * 7919
        case("dictionary keys (10^3 values, 32-bit ids)", Column(T.Uint64, values=dict_vals, dictionary_indexes=(keys3 + 1).to(torch.int32),
                                                                value_count=n), vcol, 1000, packed_bytes=12.0 * n, expect_rows=n * world)
        case("direct64, 10^3 groups, filter val > 0 (50 %)", Column(T.Uint64, values=keys3), vcol, 1000, pred=(capi.CMP_GT, 0))
        case("direct64, 10^3 groups, filter val > 0.98*2^40 (1 %)", Column(T.Uint64, values=keys3), vcol, 1000,
             pred=(capi.CMP_GT, int(0.98 * 2**40)))
        nullmask = torch.rand(n, device=device, generator=g) < 0.05
        bm = torch.from_numpy(np.packbits(nullmask.cpu().numpy(), bitorder="little")).to(device)
        case("direct64 keys, 5 % NULL values, 10^3 groups", Column(T.Uint64, values=keys3), Column(T.Int64, values=vals, null_bitmap=bm), 1000,
             packed_bytes=16.125 * n, expect_rows=n * world)
        dv = torch.rand(n, device=device, dtype=torch.float64, generator=g)
        case("SUM(double), 10^3 groups", Column(T.Uint64, values=keys3), Column(T.Double, values=dv.view(torch.int64)), 1000, expect_rows=n * world)
        del dv, bm, nullmask
        if world == 1:
            k8 = torch.randperm(n, device=device, generator=g)
            case("direct64, 10^8 groups (all distinct)", Column(T.Uint64, values=k8), vcol, n, expect_rows=n)
            del k8
    if not args.no_cpu_baseline and rank == 0 and world == 1:
        import oracle
        m = min(n, 20_000_000)
        rng = np.random.Generator(np.random.Philox(SEED + 4))
        hk = rng.integers(0, 1_000_000, m, dtype=np.uint64)
        hv = rng.integers(-2**40, 2**40, m, dtype=np.int64)
        threads = oracle.hardware_threads()
        r1 = oracle.groupby_sum_count(hk, hv, oracle.VAL_INT64, style=oracle.STYLE_QL, threads=1)
        rn = oracle.groupby_sum_count(hk, hv, oracle.VAL_INT64, style=oracle.STYLE_CH_TWO_LEVEL, threads=threads)
        out["cpu_baseline"] = {"groups": 1_000_000, "sample_rows": m, "kind": "port",
                               "ql_row_at_a_time_1_thread": m / r1["seconds"],
                               "clickhouse_two_level": {"value": m / rn["seconds"], "cores": threads,
                                                        "what": "every thread aggregates its slice of the rows into 256 hash-bucketed "
                                                                "tables, buckets are merged in parallel (Aggregator.cpp:1486 two-level)"}}
    return out


# ------------------------------------------------------------------------------------------------------------
# the reference arm: the reference's CPU sort (oracle port) on the host cores
# ------------------------------------------------------------------------------------------------------------
def workload_config(args, world, exchange=None):
    """The `config` object both arms print (identical keys and values for the same command line)."""
    names = {"sort": "configs[1]: 10^8 rows x 64 B, uint64 key, sort by key",
             "composite": "configs[2]: 64 B rows, composite (uint64 ~U[0,2^16), string[16]) key, sort by (k1, k2)",
             "pipeline": "configs[4]: 64 B rows (key uint64 ~U[0,10^7), val int64, payload[48]): sort by key, then SUM(val), COUNT(*) "
                         "GROUP BY key over the sorted rows"}
    return {"workload": names[args.workload], "keys": args.keys, "rows_per_gpu": args.rows, "row_bytes": ROW_BYTES,
            "l2": "inputs (6.4 GB per GPU) larger than L2, no flush",
            "parallelism": f"range-shard x{world}" if world > 1 else "single GPU"}


def run_reference(args):
    """One sort job per host thread over range partitions of the table (oracle port of TPartitionSortReader:
    10k-row bucket std::sort + heap merge) — how YT runs the sort phase on an exec node's CPU slots."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    from ytsaurus_b200.rowset import EValueType as T
    world = args.gpus
    threads = oracle.hardware_threads()
    n = args.ref_rows if args.ref_rows else args.rows   # N = 1: the same 10^8 rows; N > 1: a bounded sample (one GPU's share)
    rng = np.random.Generator(np.random.Philox(SEED))
    rows = rng.integers(0, 256, n * ROW_BYTES, dtype=np.uint8)
    if args.workload == "composite":
        r2 = rows.reshape(n, ROW_BYTES)
        r2[:, 2:8] = 0
        cols = [(0, 8, T.Uint64, 0), (8, 16, T.String, 0)]
    else:
        cols = [(0, 8, T.Uint64, 0)]
    times = []
    for i in range(args.warmup + args.steps):
        _, sec = oracle.sort_fixed_rows(rows, ROW_BYTES, cols, algo=oracle.SORT_PARTITION_READER, threads=threads)
        if i >= args.warmup:
            times.append(sec)
    ms = 1e3 * float(np.mean(times))
    value = n / (ms / 1e3)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": threads, "kind": "port",
                         "sample": f"{n} rows x {ROW_BYTES} B per step"
                                   + ("" if world == 1 else f" (one GPU's share of the {world}x{args.rows}-row table: a bounded sample)")
                                   + f", range-partitioned into {threads} sort jobs (TPartitionSortReader port: 10k-row bucket "
                                     "std::sort + heap merge), one per host thread"},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def pin_to_gpu_numa_node(index: int):
    """Binds this rank's host threads to the CPUs NVML reports as local to its GPU, so that the pinned staging buffers of
    the e2e leg are first-touched on the GPU's own NUMA node (8 ranks x 12.8 GB per step otherwise cross the socket link)."""
    try:
        import pynvml as nv
        import torch
        nv.nvmlInit()
        try:  # the CUDA ordinal is not the NVML index under CUDA_VISIBLE_DEVICES: go through the PCI address
            pr = torch.cuda.get_device_properties(index)
            h = nv.nvmlDeviceGetHandleByPciBusId(f"{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0")
        except Exception:
            h = nv.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = nv.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1]
        cpus = [c for c in cpus if c in os.sched_getaffinity(0)]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"cpus": len(cpus), "first": cpus[0], "last": cpus[-1]}
    except Exception as ex:  # pragma: no cover
        return {"error": f"{type(ex).__name__}: {ex}"}
    return None


# ------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ytgpu", choices=["ytgpu", "reference"])
    ap.add_argument("--workload", default="sort", choices=["sort", "composite", "pipeline"])
    ap.add_argument("--keys", default="uniform", choices=["uniform", "zipf", "zipf_hashed", "sorted"])
    ap.add_argument("--rows", type=int, default=100_000_000, help="rows per GPU per step")
    ap.add_argument("--ref-rows", type=int, default=0, help="rows per step of the reference arm (0 = --rows)")
    ap.add_argument("--cpu-sample-rows", type=int, default=20_000_000, help="bounded sample of the cpu_baseline leg")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--e2e-jobs", type=int, default=2, help="N=1: sort jobs in flight in the e2e leg (1 = serial calls)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-groupby", action="store_true")
    ap.add_argument("--no-variants", action="store_true")
    ap.add_argument("--quick", action="store_true", help="headline + verification only (no variants, two group-by cases)")
    ap.add_argument("--exchange", default="native", choices=["native", "peer", "nccl"],
                    help="N>1: ytgpu_shuffle_sort (default), the round-1 Python-driven peer scatter, or NCCL all_to_all_single")
    ap.add_argument("--groupby-rows", type=int, default=100_000_000)
    ap.add_argument("--dropin-rows", type=int, default=10_000_000, help="rows of the CreateSortingReader end-to-end leg (C++ adapter)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the last timed step's outputs to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)
    if args.quick:
        args.no_variants = True

    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist
    from ytsaurus_b200 import GpuContext, capi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    distributed = world > 1
    numa = pin_to_gpu_numa_node(local_rank) if distributed else None
    if distributed:
        # NCCL prints its version banner to STDOUT when the first communicator is created; stdout must carry exactly one
        # JSON line, so fd 1 points at stderr until the communicator exists.
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=device)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    n = args.rows
    key_cols = key_columns_of(args.workload)

    ctx = GpuContext(local_rank)
    rows = gen_rows_device(n, device, rank, args.workload, args.keys)
    capacity = int(n * 1.25) + 65536
    sorter = None
    out = None
    if distributed:
        from ytsaurus_b200.shuffle import NativeShuffleSorter, PeerMemoryUnavailable, PeerShuffleSorter, ShuffleSorter
        try:
            if args.exchange == "native":
                sorter = NativeShuffleSorter(ctx, capacity_rows=capacity, row_bytes=ROW_BYTES)
            elif args.exchange == "peer":
                sorter = PeerShuffleSorter(ctx, capacity_rows=capacity, row_bytes=ROW_BYTES)
        except PeerMemoryUnavailable as ex:  # raised on every rank together: all switch to NCCL
            if rank == 0:
                print(f"peer memory unavailable ({ex}); using the NCCL exchange", file=sys.stderr)
            args.exchange = "nccl"
        if sorter is None:
            args.exchange = "nccl"
            sorter = ShuffleSorter(ctx)
    else:
        out = torch.empty_like(rows)

    reduce_out = None
    if args.workload == "pipeline":
        gcap = 12_000_000
        reduce_out = dict(keys=torch.empty(gcap, dtype=torch.int64, device=device), sums=torch.empty(gcap, dtype=torch.int64, device=device),
                          counts=torch.empty(gcap, dtype=torch.int64, device=device))

    last = {}

    def step(src=None):
        src = rows if src is None else src
        if distributed:
            o, st = sorter.sort(src, ROW_BYTES, key_cols)
        else:
            ctx.sort_fixed_rows(src, ROW_BYTES, key_cols, want_rows=True, out_rows=out)
            o, st = out, None
        last["out"], last["stats"] = o, st
        if args.workload == "pipeline":
            last["groups"] = ctx.reduce_sorted_fixed_rows(o, ROW_BYTES, 0, 8, capi.TYPE_INT64, reduce_out["keys"], reduce_out["sums"],
                                                          reduce_out["counts"])
        return o

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    def time_steps(steps, fn=step):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        for _ in range(steps):
            fn()
        ev1.record()
        barrier()
        t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=device)
        if distributed:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    ctx.enable_timers(True)
    ctx.reset_timers()
    launches0 = ctx.launch_count()
    with ClockSampler(local_rank) as clocks:
        ms_total_max = time_steps(args.steps)
    launches = ctx.launch_count() - launches0
    KC = capi
    timers = {name: ctx.kernel_ms(cls) for name, cls in
              [("radix_pass", KC.KC_RADIX_PASS), ("pass_skipped", KC.KC_PASS_SKIPPED), ("gather", KC.KC_GATHER), ("extract", KC.KC_EXTRACT),
               ("histogram", KC.KC_HISTOGRAM), ("partition", KC.KC_PARTITION), ("scatter", KC.KC_SCATTER), ("sync", KC.KC_SHUFFLE_SYNC),
               ("reduce", KC.KC_REDUCE)]}
    active_passes = ctx.last_sort_passes()
    ctx.enable_timers(False)
    ms_step = ms_total_max / args.steps
    value = n * world / (ms_step / 1e3)

    # ---- correctness of the last timed step (outside the timed region) ----
    parity = verify_sort(last["out"], rows, ROW_BYTES, key_cols, world, rank, dist if distributed else None)
    if args.workload == "pipeline":
        # the segmented reduce against an independent computation: per-key sums through torch's scatter_add
        gk = reduce_out["keys"][: last["groups"]]
        gs = reduce_out["sums"][: last["groups"]]
        gc = reduce_out["counts"][: last["groups"]]
        r2 = rows.view(torch.int64).view(-1, 8)
        want_s = torch.zeros(10_000_000, dtype=torch.int64, device=device).scatter_add_(0, r2[:, 0], r2[:, 1])
        want_c = torch.zeros(10_000_000, dtype=torch.int64, device=device).scatter_add_(0, r2[:, 0], torch.ones_like(r2[:, 0]))
        got_s = torch.zeros(10_000_000, dtype=torch.int64, device=device).scatter_add_(0, gk, gs)
        got_c = torch.zeros(10_000_000, dtype=torch.int64, device=device).scatter_add_(0, gk, gc)
        if distributed:
            for t in (want_s, want_c, got_s, got_c):
                dist.all_reduce(t)
        parity["checks"]["reduce_sums"] = bool((want_s == got_s).all())
        parity["checks"]["reduce_counts"] = bool((want_c == got_c).all())
        parity["checks"]["reduce_keys_increasing"] = bool((gk[1:] > gk[:-1]).all()) if gk.numel() > 1 else True
        parity["ok"] = all(parity["checks"].values())
        del want_s, want_c, got_s, got_c
    if args.dump_outputs:
        outputs = {"sorted_rows": (last["out"].view(torch.int64).view(-1, ROW_BYTES // 8), 1 << 18)}
        if args.workload == "pipeline":
            g = last["groups"]
            outputs["groups"] = (torch.stack([reduce_out["keys"][:g], reduce_out["sums"][:g], reduce_out["counts"][:g]], 1), 1 << 17)
        dump_outputs(args.dump_outputs, outputs, world, rank)

    # ---- key-distribution variants of the sort (SURVEY §8d C2) ----
    variants = None
    if args.workload == "sort" and not args.no_variants and not distributed:
        variants = []
        for kd in ("zipf", "zipf_hashed", "sorted"):
            vrows = gen_rows_device(n, device, rank, "sort", kd)
            for _ in range(3):
                step(vrows)
            vms = time_steps(5, lambda: step(vrows)) / 5
            vpar = verify_sort(out, vrows, ROW_BYTES, key_cols)
            variants.append({"keys": kd, "value": n / (vms / 1e3), "ms_per_step": vms, "passes_run": ctx.last_sort_passes(),
                             "parity_ok": vpar["ok"], "whole_sort_frac": ALGO_BYTES_PER_ROW_SORT * n / (vms / 1e3) / 1e9 / peaks()[0]})
            del vrows
        ctx.set_option("sort_hybrid", 0)   # full 8-digit LSD on the uniform table, for comparison
        for _ in range(3):
            step()
        vms = time_steps(5) / 5
        variants.append({"keys": "uniform, full LSD (hybrid schedule off)", "value": n / (vms / 1e3), "ms_per_step": vms,
                         "passes_run": ctx.last_sort_passes(), "whole_sort_frac": ALGO_BYTES_PER_ROW_SORT * n / (vms / 1e3) / 1e9 / peaks()[0]})
        ctx.set_option("sort_hybrid", 1)
        step()

    # ---- e2e: host (pinned) buffers through the C ABI, H2D + D2H inside the timed region ----
    e2e = None
    if not args.no_e2e:
        try:
            e2e = bench_e2e(args, ctx, sorter, rows, key_cols, n, world, rank, local_rank, device, distributed, dist, barrier, capacity)
        except Exception as ex:  # pragma: no cover
            e2e = {"value": None, "unit": "rows/s", "error": f"{type(ex).__name__}: {ex}"}

    peak, peak_src = peaks()
    # ---- secondary metric: GROUP BY rows/s (configs[3]) at this N ----
    groupby = None
    if not args.no_groupby and args.workload == "sort":
        del rows
        if out is not None:
            del out
        last.clear()
        torch.cuda.empty_cache()
        groupby = bench_groupby(ctx, args, device, peak, world, rank, dist if distributed else None)

    if rank != 0:
        if distributed:
            dist.barrier()
            if hasattr(sorter, "close"):
                sorter.close()
            dist.destroy_process_group()
        if not parity["ok"]:
            sys.exit(3)
        return

    ms_total = ms_total_max
    steps = args.steps

    def per_launch(name):
        t, c = timers[name]
        return (t / c) if c else None

    def kernel_roofline(name, bytes_per_row, avg_ms, launches_n, traffic_key, note, bound="hbm", rows_per_launch=n, peak_gbs=None):
        pk = peak_gbs or peak
        ach = (bytes_per_row * rows_per_launch / (avg_ms / 1e3) / 1e9) if avg_ms else None
        return {"bound": bound, "kernel": name, "achieved": ach, "peak": pk, "unit": "GB/s", "frac": (ach / pk) if ach else None,
                "peak_source": peak_src if bound == "hbm" else "measured peer copy per direction (B200_PROFILING.md)",
                "traffic": traffic.get(traffic_key), "algorithmic_bytes_per_row": bytes_per_row, "avg_launch_ms": avg_ms,
                "timed_launches": launches_n, "note": note}

    traffic = {}
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        pass
    rows_local = parity["rows"] / world  # rows a rank sorts locally (== n up to the partition imbalance)
    k_pass = kernel_roofline("onesweep_pass_kernel<256,16,3> (one 8-bit digit of (u64 key, u32 index) pairs)",
                             ALGO_BYTES_PER_ROW_PASS, per_launch("radix_pass"), timers["radix_pass"][1], "onesweep_pass_kernel_bytes_per_launch",
                             "traffic == algorithmic bytes; bound by issue slots (8-ballot ranking); 1.65x faster per pass than "
                             "cub::DeviceRadixSort on the same GPU (profiles/r2_microbench.md)", rows_per_launch=rows_local)
    k_gather = kernel_roofline("gather_rows_kernel (out[j] = rows[perm[j]], 64-byte rows)",
                               132.0, per_launch("gather"), timers["gather"][1], "gather_rows_kernel_bytes_per_launch",
                               "B200 DRAM reads 128 B per random 64 B access: real traffic 19.5 GB per launch = 70-77 % of the copy "
                               "peak; grouping the reads by source chunk (random 64 B WRITES instead) measured slower "
                               "(profiles/r2_microbench.md)", rows_per_launch=rows_local)
    kernels = {"radix_pass": k_pass, "row_gather": k_gather}
    if distributed and timers["scatter"][1]:
        off_rank = n * (world - 1) / world  # rows leaving the GPU per launch with balanced partitions
        kernels["peer_scatter"] = kernel_roofline(
            "scatter_stream_kernel (rows read sequentially, written to their slot in the destination GPU's receive buffer)",
            float(ROW_BYTES), per_launch("scatter"), timers["scatter"][1], None,
            "NVLink roofline: bytes that leave the GPU per launch / measured peer-copy bandwidth per direction; the HBM side "
            "(64 B read + 64 B/g local write per row) is far from its bound", bound="nvlink", rows_per_launch=off_rank, peak_gbs=NVLINK_PEER_GBS)
        kernels["partition_count"] = kernel_roofline(
            "partition_count_kernel (+3 scan launches): key -> partition index + per-tile counts, one pass over the rows",
            68.0, per_launch("partition"), timers["partition"][1], None, "reads every 64 B row for its 8 B key")
    if args.workload == "pipeline" and timers["reduce"][1]:
        kernels["sorted_reduce"] = kernel_roofline("reduce_sorted_kernel (segmented SUM/COUNT over sorted rows, decoupled look-back)",
                                                   64.0, per_launch("reduce"), timers["reduce"][1], None,
                                                   "one pass over the sorted rows; 24 B per group written", rows_per_launch=rows_local)
    dominant = max(kernels.values(), key=lambda k: (k["avg_launch_ms"] or 0) * (k["timed_launches"] or 0))
    roofline = dict(dominant)
    passes_per_step = max(1, active_passes)
    roofline.update({
        "kernels": kernels,
        "launches_per_step": {k: timers[k][1] / steps for k in timers},
        "step_share": {k: (timers[k][0] / ms_total if timers[k][0] else 0.0) for k in timers},
        "passes_run": passes_per_step,
        "schedule": ("hybrid: only the most significant active digits are sorted, runs of equal prefixes are fixed up "
                     "(radix_sort.cu)" if passes_per_step < 8 else "full LSD, 8 digits"),
        "whole_sort": {"algorithmic_bytes_per_row": ALGO_BYTES_PER_ROW_SORT,
                       "bytes_per_row_of_the_schedule_run": 16.0 + 24.0 * passes_per_step + 16.0 + 132.0,
                       "achieved_gbs": ALGO_BYTES_PER_ROW_SORT * n * world / (ms_step / 1e3) / 1e9,
                       "frac": ALGO_BYTES_PER_ROW_SORT * n / (ms_step / 1e3) / 1e9 / peak,
                       "floor_128B_frac": 128.0 * n / (ms_step / 1e3) / 1e9 / peak},
    })
    if distributed:
        roofline["note_sync"] = ("step_share.sync is sampling + pivot selection + count exchange + the three peer barriers, i.e. it includes "
                                 "the time a rank WAITS for slower ranks")

    cpu_baseline = None
    if not args.no_cpu_baseline and world == 1 and args.workload == "sort":
        import oracle
        from ytsaurus_b200.rowset import EValueType as TT
        threads = oracle.hardware_threads()
        m = args.cpu_sample_rows
        rng = np.random.Generator(np.random.Philox(SEED))
        sample = rng.integers(0, 256, m * ROW_BYTES, dtype=np.uint8)
        _, sec = oracle.sort_fixed_rows(sample, ROW_BYTES, [(0, 8, TT.Uint64, 0)], algo=oracle.SORT_PARTITION_READER, threads=threads)
        m1 = min(m, 4_000_000)
        _, sec1 = oracle.sort_fixed_rows(sample[: m1 * ROW_BYTES], ROW_BYTES, [(0, 8, TT.Uint64, 0)], algo=oracle.SORT_STD, threads=1)
        cpu_baseline = {"value": m / sec, "unit": "rows/s", "cores": threads, "kind": "port",
                        "sample": f"{m} rows x {ROW_BYTES} B in {threads} range-partitioned sort jobs "
                                  "(TPartitionSortReader port), one per host thread",
                        "single_job": {"value": m1 / sec1, "cores": 1,
                                       "sample": f"{m1} rows, TSortingReader port (std::sort over row pointers)"}}

    # ---- the honest drop-in number: CreateSortingReader over TUnversionedRow handles, end to end (C++ adapter) ----
    dropin = None
    if world == 1 and args.workload == "sort" and not args.no_e2e:
        exe = os.path.join(ROOT, "host", "sorting_reader_bench")
        try:
            import subprocess
            if not os.path.exists(exe):
                subprocess.check_call(["make", "-C", os.path.join(ROOT, "host")], stdout=subprocess.DEVNULL)
            r = subprocess.run([exe, str(args.dropin_rows)], capture_output=True, text=True, timeout=600)
            dropin = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 else {"error": (r.stderr or r.stdout)[-300:]}
        except Exception as ex:  # pragma: no cover
            dropin = {"error": f"{type(ex).__name__}: {ex}"}

    cfg = workload_config(args, world)
    if distributed:
        cfg["numa_binding_rank0"] = numa
        cfg["exchange"] = {"native": "ytgpu_shuffle_sort: peer-memory sample/count exchange + device barriers + fused NVLink scatter",
                           "peer": "round-1 path: Python-driven pivots, fused NVLink scatter", "nccl": "NCCL all_to_all_single"}[args.exchange]
    line = {
        "metric": METRIC if args.workload != "pipeline" else "rows/s sorted then aggregated (64B rows, u64 key)",
        "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic", "config": cfg,
        "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "parity_check": parity, "gpu_launches": launches,
        "clocks": clocks.summary(),
    }
    if variants is not None:
        line["variants"] = variants
    if dropin is not None:
        line["dropin_sorting_reader_e2e"] = dropin
    if groupby is not None:
        line["groupby"] = groupby
        for c in groupby["cases"]:
            if c["name"].startswith("direct64, 10^3"):
                line["groupby_rows_per_s_1e3_groups"] = c["value"]
                line["groupby_roofline_frac_1e3_groups"] = c["roofline_frac"]
            if c["name"] == "direct64, 10^6 groups":
                line["groupby_rows_per_s_1e6_groups"] = c["value"]
                line["groupby_roofline_frac_1e6_groups"] = c["roofline_frac"]
    if args.workload == "pipeline":
        line["pipeline"] = {"groups_on_rank0": last.get("groups")}
    print(json.dumps(line), flush=True)
    if distributed:
        dist.barrier()
        if hasattr(sorter, "close"):
            sorter.close()
        dist.destroy_process_group()
    if not parity["ok"]:
        print(f"PARITY CHECK FAILED: {parity}", file=sys.stderr)
        sys.exit(3)


def bench_e2e(args, ctx, sorter, rows, key_cols, n, world, rank, local_rank, device, distributed, dist, barrier, capacity):
    """The same step with HOST (pinned) buffers: every step copies its 6.4 GB per GPU in and its result out inside the
    timed region.  N = 1: blocking ytgpu_sort_fixed_rows calls with HOST buffers (e2e_jobs of them in flight, as a node
    runs several job slots); N > 1: per rank H2D on a copy stream, shuffle-sort, D2H, double-buffered so that a step's
    D2H overlaps the next step's H2D (PCIe is full duplex)."""
    import torch
    from ytsaurus_b200 import GpuContext
    nb = n * ROW_BYTES
    # N = 1: the job threads and their pinned buffers live on the GPU's own NUMA node for the length of this leg, as a job
    # proxy pins its GPU slot (with the buffers on the other socket both copy directions share the socket link and two jobs
    # in flight gain nothing: 239 vs 158 ms per step on the same kind of box).  N > 1: the ranks were bound at start-up.
    numa_binding, saved_affinity = None, None
    if not distributed and not os.environ.get("YTGPU_BENCH_NO_NUMA"):
        saved_affinity = os.sched_getaffinity(0)
        numa_binding = pin_to_gpu_numa_node(local_rank)
    try:
        return _bench_e2e_bound(args, ctx, sorter, rows, key_cols, n, world, rank, local_rank, device, distributed, dist, barrier, capacity,
                                nb, numa_binding)
    finally:
        if saved_affinity is not None:
            os.sched_setaffinity(0, saved_affinity)  # the CPU legs use every host thread again


def _bench_e2e_bound(args, ctx, sorter, rows, key_cols, n, world, rank, local_rank, device, distributed, dist, barrier, capacity, nb,
                     numa_binding):
    import torch
    from ytsaurus_b200 import GpuContext
    h_in = torch.empty(nb, dtype=torch.uint8).pin_memory()
    h_in.copy_(rows)
    if distributed:
        h_out = torch.empty(capacity * ROW_BYTES, dtype=torch.uint8).pin_memory()
        copy_in, copy_out = torch.cuda.Stream(device), torch.cuda.Stream(device)
        dbuf = [torch.empty_like(rows) for _ in range(2)]
        main = torch.cuda.current_stream(device)
        steps = args.e2e_steps + 1

        def run(k):
            evs = []
            with torch.cuda.stream(copy_in):
                dbuf[0].copy_(h_in, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy_in)
                evs.append(ev)
            for s in range(k):
                main.wait_event(evs[s])
                o, _ = sorter.sort(dbuf[s % 2], ROW_BYTES, key_cols)
                done = torch.cuda.Event()
                done.record(main)
                if s + 1 < k:  # next step's input travels while this step's output leaves
                    with torch.cuda.stream(copy_in):
                        dbuf[(s + 1) % 2].copy_(h_in, non_blocking=True)
                        ev = torch.cuda.Event()
                        ev.record(copy_in)
                        evs.append(ev)
                copy_out.wait_event(done)
                with torch.cuda.stream(copy_out):
                    h_out[: o.numel()].copy_(o, non_blocking=True)
                    fin = torch.cuda.Event()
                    fin.record(copy_out)
                main.wait_event(fin)  # the sorter's output buffer is reused by the next sort
            torch.cuda.synchronize()

        run(1)
        barrier()
        t0 = time.perf_counter()
        run(steps)
        barrier()
        e_ms = torch.tensor([(time.perf_counter() - t0) * 1e3 / steps], dtype=torch.float64, device=device)
        dist.all_reduce(e_ms, op=dist.ReduceOp.MAX)
        ms = float(e_ms.item())
        return {"value": n * world / (ms / 1e3), "unit": "rows/s", "h2d_bytes_per_step": nb * world, "d2h_bytes_per_step": nb * world,
                "ms_per_step": ms, "steps": steps,
                "timer": "host perf_counter, max over ranks; per rank: pinned H2D (copy stream) -> ytgpu_shuffle_sort -> pinned D2H, "
                         "double-buffered (step s+1's H2D overlaps step s's D2H)"}
    h_out = torch.empty(nb, dtype=torch.uint8).pin_memory()
    hin_np, hout_np = h_in.numpy(), h_out.numpy()
    return_numa = numa_binding

    def e2e_step():
        ctx.sort_fixed_rows(hin_np, ROW_BYTES, key_cols, want_rows=True, out_rows=hout_np)

    e2e_step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    serial_ms = (time.perf_counter() - t0) * 1e3 / args.e2e_steps
    e2e = {"value": n / (serial_ms / 1e3), "unit": "rows/s", "h2d_bytes_per_step": nb, "d2h_bytes_per_step": nb,
           "ms_per_step": serial_ms, "steps": args.e2e_steps, "jobs_in_flight": 1,
           "timer": "host perf_counter around the blocking C-ABI call (the call synchronises its stream)"}
    if args.e2e_jobs > 1:
        # The same call from several sort jobs at once (one context + private stream + host thread each, as a node runs
        # several job slots): one job's sorted rows leave while the next job's input arrives.  Measured for 2..e2e_jobs jobs in
        # flight; the best one is the headline.  (On the pool's B200 boxes the PCIe link moves ~54 GB/s one way and ~79 GB/s
        # with both directions busy, so two jobs already sit at the link's duplex limit: 12.8 GB / 79 GB/s = 162 ms per step.)
        ctxs = [GpuContext(local_rank, use_torch_stream=False) for _ in range(args.e2e_jobs)]
        outs = [hout_np] + [torch.empty(nb, dtype=torch.uint8).pin_memory().numpy() for _ in range(args.e2e_jobs - 1)]
        for j in range(args.e2e_jobs):  # warm-up: staging buffers and scratch of every context
            ctxs[j].sort_fixed_rows(hin_np, ROW_BYTES, key_cols, want_rows=True, out_rows=outs[j])
        by_jobs = {}
        for jobs in range(2, args.e2e_jobs + 1):
            per_job = max(2, args.e2e_steps)
            errors = []
            start = threading.Barrier(jobs + 1)

            def job(j):
                try:
                    start.wait()
                    for _ in range(per_job):
                        ctxs[j].sort_fixed_rows(hin_np, ROW_BYTES, key_cols, want_rows=True, out_rows=outs[j])
                except Exception as ex:  # pragma: no cover
                    errors.append(ex)
                    start.abort()

            threads = [threading.Thread(target=job, args=(j,)) for j in range(jobs)]
            for th in threads:
                th.start()
            start.wait()
            t0 = time.perf_counter()
            for th in threads:
                th.join()
            torch.cuda.synchronize()
            piped_ms = (time.perf_counter() - t0) * 1e3 / (per_job * jobs)
            if errors:
                raise errors[0]
            by_jobs[jobs] = {"value": n / (piped_ms / 1e3), "ms_per_step": piped_ms, "steps": per_job * jobs}
        for o in outs:  # every job's last output is the sorted table
            chk = verify_sort(torch.from_numpy(o).to(device), rows, ROW_BYTES, key_cols)
            assert chk["ok"], f"e2e output failed verification: {chk}"
        best = max(by_jobs, key=lambda k: by_jobs[k]["value"])
        e2e.update({"value": by_jobs[best]["value"], "ms_per_step": by_jobs[best]["ms_per_step"], "steps": by_jobs[best]["steps"],
                    "jobs_in_flight": best, "by_jobs_in_flight": {str(k): v for k, v in by_jobs.items()},
                    "single_job": {"value": n / (serial_ms / 1e3), "ms_per_step": serial_ms},
                    "timer": "host perf_counter from the common start of the job threads to the last join; each step is one "
                             "blocking C-ABI call with pinned HOST buffers"})
    e2e["numa_binding"] = return_numa
    return e2e


if __name__ == "__main__":
    main()
