#!/usr/bin/env python
"""bench.py — Sort keys/s (headline) and ReduceByKey records/s of the B200-native Thrill hot path.

  python bench.py --gpus N --steps K --warmup W [--metric sort|reduce]      (N > 1: launched by torch.distributed.run)
  python bench.py --impl reference --gpus N --steps K --warmup W [--metric sort|reduce]
  python bench.py ... --dump-outputs DIR      (also writes what the last timed step computed, see write_outputs)

One "step" = one pass of the hot path over one synthetic batch (SURVEY.md §8d generators, seed 42):
  sort   : DIA<uint64_t>::Sort of 1e8 uniform keys per GPU          (BASELINE.json configs[1]; weak scaling)
  reduce : ReducePair<uint64_t,double>(plus) of 1.25e8 Zipf(s=1, U=2^26) records per GPU (configs[2] per-GPU share)
`value` is the device-resident whole-job throughput (inputs already in HBM); `e2e` is the same operator through the
reference-facing call (host Blocks in pinned memory -> tg_sort_file / tg_reduce_file -> tg_fetch_output, H2D and D2H
inside the timed region).  `roofline` is measured live with CUDA events around every launch of the dominant kernel;
`cpu_baseline` is the UNMODIFIED reference (oracle/_ref/thrill_ref_driver) timed on this box's host cores.
`parity_check` (outside the timed region) proves the measured run produced the right answer on every rank: global
multiset checksum before/after, rank boundaries in order, balance; for reduce key ownership and exact sums of a sample
against a plain numpy group-by.  The oracle / reference are only ever the checker or the baseline here.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 42
SORT_N_PER_GPU = 100000000
REDUCE_N_PER_GPU = 125000000
ZIPF_UNIVERSE = 1 << 26
SORT_PASS_BYTES_PER_KEY = 16.0          # one stable partition pass: read 8 + write 8 (DESIGN.md §5)
SORT_MODEL_BYTES_PER_KEY = {1: 136.0}   # SURVEY.md §8(d): LSB radix sort, p = 1; p > 1: 184
REDUCE_PASS_BYTES_PER_RECORD = 32.0     # one hash-digit partition pass: read 16 + write 16
REDUCE_MODEL_BYTES_PER_RECORD = 25.5    # SURVEY.md §8(d): 16 B/record + 64 B x D_local/N_local for Zipf(1, 2^26), 1.25e8 per GPU
DUMP_ITEMS = 1 << 20                    # --dump-outputs: items written per job (at most 4 float64 arrays of them: 32 MiB)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json (measured)"
    return 6650.0, "B200_PROFILING.md fallback"


def profile_traffic(name):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch from the committed `ncu --set full` summary
    profiles/<name> (first kernel block); None if the file is absent"""
    path = os.path.join(ROOT, "profiles", name)
    if not os.path.exists(path):
        return None, None
    rd = wr = None
    unit = {"Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "byte": 1.0}
    for line in open(path):
        f = line.split()
        if len(f) >= 3 and f[0] == "dram__bytes_read.sum" and rd is None:
            rd = float(f[2]) * unit.get(f[1], 1.0)
        if len(f) >= 3 and f[0] == "dram__bytes_write.sum" and wr is None:
            wr = float(f[2]) * unit.get(f[1], 1.0)
    if rd is None or wr is None:
        return None, None
    return rd + wr, "profiles/%s (ncu --set full, one launch)" % name


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.path = tempfile.mktemp(suffix=".csv")
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.proc.wait()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        # median over the samples taken under load (the upper half of the observed clocks)
        sm_sorted = sorted(sm)
        load = sm_sorted[len(sm_sorted) // 2:] if sm_sorted else []
        return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def max_over_ranks(x, world):
    if world == 1:
        return x
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def gather_objects(obj, world):
    if world == 1:
        return [obj]
    import torch.distributed as dist
    out = [None] * world
    dist.all_gather_object(out, obj)
    return out


# ---------------------------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the unmodified reference, oracle/_ref/thrill_ref_driver (bench.py's only use of oracle/)

def ref_driver_path():
    return os.path.join(ROOT, "oracle", "_ref", "thrill_ref_driver")


_REF_WORKERS = {}


def _run_reference_once(op, n, iters, workers, extra=()):
    env = dict(os.environ, THRILL_NET="mock", THRILL_LOCAL="1", THRILL_WORKERS_PER_HOST=str(workers), THRILL_LOG="")
    args = [ref_driver_path(), "op=%s" % op, "n=%d" % n, "iters=%d" % iters, "seed=%d" % SEED] + list(extra)
    res = subprocess.run(args, env=env, capture_output=True, text=True, timeout=3000)
    if res.returncode != 0:
        raise RuntimeError("thrill_ref_driver failed (%d): %s" % (res.returncode, res.stderr[-1500:]))
    return [float(l.rsplit("time=", 1)[1]) for l in res.stdout.splitlines() if l.startswith("RESULT")]


def reference_workers(op, extra=()):
    """The reference's throughput is not monotone in its worker count (p^2 streams, one thread per worker):
    calibrate on a small sample and keep the best of a few counts up to all host threads."""
    if op in _REF_WORKERS:
        return _REF_WORKERS[op]
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (ncpu, ncpu // 2, ncpu // 4, 32, 16, 8) if 1 <= c <= ncpu}, reverse=True)
    best, best_t = cands[0], None
    for c in cands:
        try:
            t = _run_reference_once(op, 20000000 if op == "sort_u64" else 5000000, 2, c, extra)[-1]
        except Exception:
            continue
        if best_t is None or t < best_t:
            best, best_t = c, t
    _REF_WORKERS[op] = best
    return best


REDUCE_REF_EXTRA = ("gen=zipf", "universe=%d" % ZIPF_UNIVERSE)


def run_oracle_port_sort(n):
    """fallback CPU baseline when the reference binary is absent: the single-threaded C restatement"""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    keys = O.gen_sort_uniform(0, n, SEED)
    t0 = time.time()
    O.lib().to_sort_items(keys.ctypes.data, n, C.byref(O.U64_DESC))
    return time.time() - t0


def cpu_baseline(metric, n_sample):
    op, extra, unit = ("sort_u64", (), "keys/s") if metric == "sort" else ("reduce_f64", REDUCE_REF_EXTRA, "records/s")
    if os.path.exists(ref_driver_path()):
        workers = reference_workers(op, extra)
        times = _run_reference_once(op, n_sample, 3, workers, extra)
        t = statistics.median(times[1:]) if len(times) > 1 else times[0]
        what = ("Generate(splitmix64).Cache -> Sort().Size() of %d u64 keys" % n_sample if metric == "sort" else
                "Generate(Zipf s=1 U=2^26).Cache -> ReducePair(plus<double>).Size() of %d records" % n_sample)
        return {"value": n_sample / t, "unit": unit, "cores": workers, "kind": "reference",
                "sample": "thrill_ref_driver %s, THRILL_WORKERS_PER_HOST=%d (best of a calibration over worker counts up to %d host "
                          "threads), median of iterations 2-3 (%.3f s)" % (what, workers, os.cpu_count() or 1, t)}
    if metric != "sort":
        return None
    t = run_oracle_port_sort(n_sample // 10)
    return {"value": (n_sample // 10) / t, "unit": unit, "cores": 1, "kind": "port",
            "sample": "oracle/thrill_oracle.c to_sort_items on %d keys, 1 thread (%.3f s)" % (n_sample // 10, t)}


def workload_config(metric, n, world):
    """the `config` object: identical in both arms so that the driver compares like with like"""
    if metric == "sort":
        cfg = {"workload": "sort_uniform_u64_1e8_per_gpu", "keys_per_gpu": n, "keys_per_step": n * world,
               "generator": "splitmix64(i+42)"}
    else:
        cfg = {"workload": "reduce_pair_u64_f64_zipf_s1_U2^26_1.25e8_per_gpu", "records_per_gpu": n, "records_per_step": n * world,
               "generator": "key = Zipf(s=1, U=2^26) rank of splitmix64(i+42), val = splitmix64(i+42+2^40) as [0,1) double"}
    cfg["l2"] = "GPU arm: inputs (%.1f GB per GPU) larger than the 126 MB L2, regenerated on the device before every step" % (
        n * (8 if metric == "sort" else 16) / 1e9)
    cfg["exchange"] = "none (1 worker group)" if world == 1 else (
        "GPU arm: the classification / hash-partition pass stores straight into the peers' HBM windows over NVLink (P2P), NCCL "
        "all-gathers carry samples and counts; CPU arm: the reference's own MixStream between its worker threads")
    return cfg


def main_reference(args):
    """the reference's own CPU implementation of the path, all the host threads it can use, on OUR arm's config: the
    whole job's items (n per GPU x N) per step"""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    metric = args.metric
    n = (args.n if metric == "sort" else args.reduce_n) * args.gpus
    op, extra, unit = ("sort_u64", (), "keys/s") if metric == "sort" else ("reduce_f64", REDUCE_REF_EXTRA, "records/s")
    name = "sort_keys_per_s" if metric == "sort" else "reduce_records_per_s"
    if not os.path.exists(ref_driver_path()):
        if metric != "sort":
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/thrill_ref_driver is not built and the C port has no timed reduce leg"}))
            return 0
        times = [run_oracle_port_sort(n // 10) for _ in range(args.warmup + args.steps)][args.warmup:]
        t = sum(times) / len(times)
        value, cores, kind, sample = (n // 10) / t, 1, "port", "oracle C port on %d keys" % (n // 10)
        ms = t * 1e3
    else:
        cores = reference_workers(op, extra)
        times = _run_reference_once(op, n, args.warmup + args.steps, cores, extra)
        timed = times[args.warmup:]
        ms = 1e3 * sum(timed) / len(timed)
        value, kind = n / (ms / 1e3), "reference"
        sample = ("unmodified thrill/thrill %s of %d items per step (the whole job of the %d-GPU arm) on %d host threads "
                  "(mock net, 1 host)" % ("Sort()" if metric == "sort" else "ReducePair(plus<double>)", n, args.gpus, cores))
    line = {"impl": "reference", "metric": name, "value": value, "unit": unit, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64" if metric == "sort" else "u64 keys, f64 sums", "data": "synthetic",
            "config": workload_config(metric, n // args.gpus, args.gpus),
            "cpu_baseline": {"value": value, "unit": unit, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------------------------------
# numpy restatements used by parity_check only (no oracle import on this path)

def hash128to64_np(keys):
    """common/hash.hpp:64-73 with upper = 0 (uint64 arithmetic wraps)"""
    k = np.uint64(0x9DDFEA08EB382D69)
    with np.errstate(over="ignore"):
        a = keys.astype(np.uint64) * k
        a ^= a >> np.uint64(47)
        b = a * k
        b ^= b >> np.uint64(47)
        b *= k
    return b


def zipf_cdf_numpy(universe, s=1.0):
    """cumulative Zipf table, probabilities as common/zipf_distribution.hpp:119-140 (k^-s normalised).
    Sequential accumulation like the oracle (np.cumsum is sequential in float64)."""
    k = np.arange(1, universe + 1, dtype=np.float64)
    prob = 1.0 / np.power(k, s)
    p_sum = float(np.cumsum(prob)[-1])
    return np.cumsum(prob * (1.0 / p_sum))


# ---------------------------------------------------------------------------------------------------------------------
# --dump-outputs: what the last timed step handed to its caller, so that two builds can be compared output for output

def write_outputs(out_dir, prefix, world, rank, keys, vals=None):
    """Writes <prefix>_count (items this rank received) and, at fixed positions of the output in key order, <prefix>_index,
    the u64 keys split into exact halves <prefix>_keys_hi32 / _lo32 and, for a reduce, the f64 sums <prefix>_vals; all
    float64 .npy.  Outputs of more than DUMP_ITEMS / world items are sampled at positions drawn with the fixed seed, so equal
    outputs give equal files.  Ranks of a multi-GPU job write <name>_rank<r>.npy."""
    n = len(keys)
    take = DUMP_ITEMS // world
    idx = np.arange(n) if n <= take else np.sort(np.random.default_rng(SEED).choice(n, take, replace=False))
    k = keys[idx]
    arrays = {"count": [n], "index": idx, "keys_hi32": k >> np.uint64(32), "keys_lo32": k & np.uint64(0xFFFFFFFF)}
    if vals is not None:
        arrays["vals"] = vals[idx]
    os.makedirs(out_dir, exist_ok=True)
    suffix = "" if world == 1 else "_rank%d" % rank
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, "%s_%s%s.npy" % (prefix, name, suffix)), np.asarray(a, dtype=np.float64))


# ---------------------------------------------------------------------------------------------------------------------

def bench_sort(args, ctx, world, rank, hbm_peak, peak_src, zipf=False, d_cdf=None, steps=None, warmup=None, e2e=True, dump=None):
    """device-resident Sort of n u64 keys per GPU (+ the end-to-end form); returns the line's fields.  dump: directory for
    write_outputs of the last timed step"""
    from thrill_b200 import api, capi
    tg = ctx.tg
    L = tg.L
    n = args.n
    K = steps or args.steps
    W = warmup or max(args.warmup, 3)
    desc = capi.u64_desc()
    d_in = tg.alloc(n * 8)

    def gen():
        if zipf:
            tg.ck(L.tg_gen_sort_zipf(tg.h, d_in, rank * n, n, SEED, d_cdf, ZIPF_UNIVERSE))
        else:
            tg.ck(L.tg_gen_sort_uniform(tg.h, d_in, rank * n, n, SEED))

    step_ms = []
    launches = 0                                             # kernels of ours launched inside the timed regions
    fallbacks0 = int(L.tg_prefix_sort_fallbacks(tg.h))
    for it in range(W + K):
        gen()
        if it == W:
            tg.profile_enable(True)
        if it == W + K - 1:
            before = tg.checksum(d_in, n, 8)                 # (outside the timed region)
        tg.barrier()
        l0 = tg.launches()
        tg.timer_start()
        out_p, out_n = C.c_void_p(), C.c_size_t()
        tg.ck(L.tg_sort(tg.h, C.byref(desc), d_in, n, SEED + it, C.byref(out_p), C.byref(out_n)))
        ms = max_over_ranks(tg.timer_stop(), world)
        if it >= W:
            step_ms.append(ms)
            launches += tg.launches() - l0
    prof = {name: tg.profile_get(cls) for name, cls in (("partition", capi.K_PARTITION), ("hist", capi.K_RADIX_HIST),
                                                        ("merge", capi.K_MERGE), ("fixup", capi.K_FIXUP),
                                                        ("segcount", capi.K_SEGCOUNT), ("exchange", capi.K_EXCHANGE))}
    tg.profile_enable(False)
    # ---- parity of the last timed step: sortedness, multiset, rank boundaries, balance
    ok_sorted = tg.is_sorted(desc, out_p.value, out_n.value)
    after = tg.checksum(out_p.value, out_n.value, 8) if out_n.value else (0, 0)
    first = int(tg.download(out_p.value, 8, np.uint64)[0]) if out_n.value else None
    last = int(tg.download(out_p.value + (out_n.value - 1) * 8, 8, np.uint64)[0]) if out_n.value else None
    allv = gather_objects((before, after, int(out_n.value), first, last, bool(ok_sorted)), world)
    m64 = (1 << 64) - 1
    sum_b = sum(v[0][0] for v in allv) & m64
    sum_a = sum(v[1][0] for v in allv) & m64
    xor_b = xor_a = 0
    for v in allv:
        xor_b ^= v[0][1]; xor_a ^= v[1][1]
    total_out = sum(v[2] for v in allv)
    bounds = [(v[3], v[4]) for v in allv if v[2]]
    ordered = all(bounds[i][1] <= bounds[i + 1][0] for i in range(len(bounds) - 1))
    balance = max(v[2] for v in allv) / (float(total_out) / world) if total_out else 1.0
    parity = {"sorted_on_every_rank": all(v[5] for v in allv), "items_out": total_out, "items_in": n * world,
              "multiset_sum_match": sum_b == sum_a, "multiset_xor_match": xor_b == xor_a,
              "rank_boundaries_ordered": ordered, "max_over_mean_items": round(balance, 4)}
    parity["ok"] = bool(parity["sorted_on_every_rank"] and total_out == n * world and parity["multiset_sum_match"]
                        and parity["multiset_xor_match"] and ordered and balance <= 1.5)
    if not parity["ok"]:
        raise SystemExit("bench: sort parity check FAILED: %s" % json.dumps(parity))
    if dump:
        write_outputs(dump, "sort", world, rank, tg.download(out_p.value, out_n.value * 8, np.uint64))

    ms_per_step = sum(step_ms) / len(step_ms)
    value = n * world / (ms_per_step / 1e3)
    part_ms, part_cnt = prof["partition"]
    xchg_ms, xchg_cnt = prof["exchange"]
    # the local partition passes (the exchange pass is timed on its own: NVLink, not HBM, bounds it)
    local_ms, local_cnt = (part_ms - xchg_ms, part_cnt - xchg_cnt) if world > 1 and xchg_cnt else (part_ms, part_cnt)
    pass_launch_ms = local_ms / max(local_cnt, 1)
    # a pass of the local sort moves the items this rank holds after the exchange
    n_pass = float(out_n.value) if world > 1 else float(n)
    achieved = SORT_PASS_BYTES_PER_KEY * n_pass / (pass_launch_ms / 1e3) / 1e9
    traffic, traffic_src = profile_traffic("r2_partition_pass_u64.txt")
    model = 136.0 if world == 1 else 184.0
    roofline = {"bound": "hbm", "kernel": "tgp::partition_kernel<1,256,16,3,RadixDigit,SEG> (one stable 8-bit partition pass: "
                                          "read 8 B + write 8 B per key)",
                "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "peak_source": peak_src,
                "traffic": traffic * (n_pass / 1e8) if traffic else None, "traffic_source": traffic_src,
                "algorithmic_bytes_per_launch": SORT_PASS_BYTES_PER_KEY * n_pass, "launch_ms": pass_launch_ms,
                "launches_timed": local_cnt,
                "operator_model": {"bytes_per_key": model, "what": "SURVEY.md 8(d) Sort total, p %s 1" % ("=" if world == 1 else ">"),
                                   "achieved_GBps": model * n / (ms_per_step / 1e3) / 1e9,
                                   "frac": model * n / (ms_per_step / 1e3) / 1e9 / hbm_peak},
                "step_share": {"partition_ms": local_ms / K, "partition_launches_per_step": local_cnt / K,
                               "count_ms": (prof["hist"][0] + prof["segcount"][0]) / K, "finishing_pass_ms": prof["fixup"][0] / K,
                               "merge_ms": prof["merge"][0] / K, "exchange_pass_ms": xchg_ms / K, "step_ms": ms_per_step},
                "prefix_sort_fallbacks": int(L.tg_prefix_sort_fallbacks(tg.h)) - fallbacks0}
    if world > 1 and xchg_cnt:
        sent = n * 8.0 * (world - 1) / world            # bytes a rank stores into peer windows per step (uniform keys)
        roofline["exchange"] = {"kernel": "tgp::partition_kernel<...,SplitterDigit,SEG,PEER> (classify + scatter + Alltoallv: stores into the "
                                          "peers' windows over NVLink)", "launch_ms": xchg_ms / xchg_cnt,
                                "nvlink_GBps_out_per_gpu": sent / (xchg_ms / xchg_cnt / 1e3) / 1e9, "nvlink_peak_GBps": 770.0,
                                "peak_source": "B200_PROFILING.md measured peer copy, per direction"}
    res = {"value": value, "ms_per_step": ms_per_step, "roofline": roofline, "parity_check": parity, "gpu_launches": int(launches),
           "steps": K, "warmup": W}

    # ---- end to end: host Blocks in pinned memory -> tg_sort_file -> tg_fetch_output
    if e2e:
        host_in = tg.host_alloc(n * 8)
        host_out = tg.host_alloc(n * 8 + (n // 4) * 8)        # a worker may receive more than it sent (eps = 0.1)
        gen()
        tg.ck(L.tg_download(tg.h, host_in.ctypes.data, d_in, n * 8))
        tg.sync()
        dia = api.DIA(ctx, host_in.view(np.uint64))
        e2e_s = []
        for it in range(2 + K):
            tg.barrier()
            t0 = time.perf_counter()
            r = dia.Sort(_pinned_out=host_out)               # tg_sort_file + tg_fetch_output (synchronises)
            dt = max_over_ranks(time.perf_counter() - t0, world)
            if it >= 2:
                e2e_s.append(dt)
        if not bool(np.all(r.items[1:] >= r.items[:-1])):
            raise SystemExit("bench: e2e sort result is not sorted")
        out_total = sum(gather_objects(int(len(r.items)), world))
        res["e2e"] = {"value": n * world / (sum(e2e_s) / len(e2e_s)), "unit": "keys/s", "h2d_bytes_per_step": n * 8 * world,
                      "d2h_bytes_per_step": out_total * 8, "ms_per_step": 1e3 * sum(e2e_s) / len(e2e_s),
                      "call": "thrill_b200.api.DIA.Sort -> tg_sort_file + tg_fetch_output over 1 MiB pinned Blocks"}
        tg.host_free(host_in); tg.host_free(host_out)
    tg.free(d_in)
    return res


def bench_terasort(args, ctx, world, rank, hbm_peak, steps=2, warmup=1):
    """cfg4's per-GPU share: Sort of 100-byte records (10-byte key), device resident; parity = sortedness + multiset + rank
    boundaries on every rank"""
    from thrill_b200 import capi
    tg = ctx.tg
    L = tg.L
    n = args.terasort_n
    desc = capi.record_desc()
    d_in = tg.alloc(n * 100)
    ms_list = []
    for it in range(warmup + steps):
        tg.ck(L.tg_gen_records(tg.h, d_in, rank * n, n, SEED))
        if it == warmup:
            tg.profile_enable(True)
        if it == warmup + steps - 1:
            before = tg.checksum(d_in, n, 100)
        tg.barrier()
        tg.timer_start()
        op, on = C.c_void_p(), C.c_size_t()
        tg.ck(L.tg_sort(tg.h, C.byref(desc), d_in, n, SEED + it, C.byref(op), C.byref(on)))
        ms = max_over_ranks(tg.timer_stop(), world)
        if it >= warmup:
            ms_list.append(ms)
    gather_ms, gather_cnt = tg.profile_get(capi.K_MERGE)
    xchg_ms, xchg_cnt = tg.profile_get(capi.K_EXCHANGE)
    part_ms, part_cnt = tg.profile_get(capi.K_PARTITION)
    tg.profile_enable(False)
    ok_sorted = tg.is_sorted(desc, op.value, on.value)
    after = tg.checksum(op.value, on.value, 100) if on.value else (0, 0)
    first = bytes(tg.download(op.value, 10)) if on.value else None
    last = bytes(tg.download(op.value + (on.value - 1) * 100, 10)) if on.value else None
    allv = gather_objects((before, after, int(on.value), first, last, bool(ok_sorted)), world)
    m64 = (1 << 64) - 1
    xb = xa = 0
    for v in allv:
        xb ^= v[0][1]; xa ^= v[1][1]
    total_out = sum(v[2] for v in allv)
    bounds = [(v[3], v[4]) for v in allv if v[2]]
    parity = {"sorted_on_every_rank": all(v[5] for v in allv), "items_out": total_out, "items_in": n * world,
              "multiset_sum_match": (sum(v[0][0] for v in allv) & m64) == (sum(v[1][0] for v in allv) & m64),
              "multiset_xor_match": xb == xa,
              "rank_boundaries_ordered": all(bounds[i][1] <= bounds[i + 1][0] for i in range(len(bounds) - 1)),
              "max_over_mean_items": round(max(v[2] for v in allv) / (float(total_out) / world), 4) if total_out else 1.0}
    parity["ok"] = bool(parity["sorted_on_every_rank"] and total_out == n * world and parity["multiset_sum_match"]
                        and parity["multiset_xor_match"] and parity["rank_boundaries_ordered"])
    tg.free(d_in)
    step = sum(ms_list) / len(ms_list)
    model = 668.0 if world == 1 else 1270.0
    g_launch = gather_ms / max(gather_cnt, 1)
    return {"records_per_s": n * world / (step / 1e3), "ms_per_step": step, "workload": "terasort_100B_records_10B_key", "records_per_gpu": n,
            "parity_check": parity,
            "operator_model": {"bytes_per_record": model, "what": "SURVEY.md 8(d) TeraSort total, p %s 1" % ("=" if world == 1 else ">"),
                               "achieved_GBps": model * n / (step / 1e3) / 1e9, "frac": model * n / (step / 1e3) / 1e9 / hbm_peak},
            "gather_kernel": {"kernel": "gather_records_kernel (read 16 B tuple + 100 B record, write 100 B)", "launch_ms": g_launch,
                              "achieved_GBps": 216.0 * (float(on.value) if world > 1 else n) / (g_launch / 1e3) / 1e9 if g_launch else None},
            "step_share": {"gather_ms": gather_ms / steps, "tuple_partition_ms": part_ms / steps, "exchange_ms": xchg_ms / steps, "step_ms": step}}


def e2e_in_thrill(n=20000000):
    """The drop-in inside a real Thrill job (tests/host/gpu_nodes_test.cpp, built into oracle/_ref/host: api::Run, 1 worker,
    the unmodified reference library around the GPU nodes): wall time of Generate -> thrill_gpu::Sort -> AllGather against the stock Sort on the same worker
    thread.  BlockPool memory is pageable here: this is the number a Thrill user gets without pinning it."""
    exe = os.path.join(ROOT, "oracle", "_ref", "host", "gpu_nodes_test")
    if not os.path.exists(exe):
        return None
    env = dict(os.environ, THRILL_NET="mock", THRILL_LOCAL="1", THRILL_WORKERS_PER_HOST="1", THRILL_LOG="")
    try:
        res = subprocess.run([exe, str(n)], env=env, capture_output=True, text=True, timeout=600)
    except Exception as e:          # noqa: BLE001
        return {"error": str(e)[:200]}
    out = {"binary": "oracle/_ref/host/gpu_nodes_test %d (THRILL_WORKERS_PER_HOST=1)" % n, "rc": res.returncode, "sections": []}
    for l in res.stdout.splitlines():
        if l.startswith(("PASS", "FAIL")):
            out["sections"].append(l[:160])
    return out


def reduce_parity(ctx, world, rank, d_cdf):
    """exact-mode sample (integer-valued doubles: sums are order independent) through the same operator, every key on the
    worker the reference's ReduceByHash puts it on, sums equal to a numpy group-by of the same records"""
    from thrill_b200 import capi
    tg = ctx.tg
    L = tg.L
    ns = 1 << 20
    KV = np.dtype([("key", "<u8"), ("val", "<f8")])
    d = tg.alloc(ns * 16)
    tg.ck(L.tg_gen_reduce_zipf(tg.h, d, rank * ns, ns, SEED, d_cdf, ZIPF_UNIVERSE, 1))
    inp = tg.download(d, ns * 16, KV)
    rp, rc = C.c_void_p(), C.c_size_t()
    tg.ck(L.tg_reduce_by_key(tg.h, C.byref(capi.KVDesc(16, capi.OP_SUM_F64)), d, ns, C.byref(rp), C.byref(rc)))
    out = tg.download(rp.value, rc.value * 16, KV) if rc.value else np.zeros(0, KV)
    tg.free(d)
    owner_ok = bool(np.all(hash128to64_np(out["key"]) % np.uint64(world) == np.uint64(rank)))
    parts = gather_objects((inp, out, owner_ok), world)
    keys = np.concatenate([p[0]["key"] for p in parts])
    vals = np.concatenate([p[0]["val"] for p in parts])
    uk, inv = np.unique(keys, return_inverse=True)
    sums = np.bincount(inv, weights=vals, minlength=len(uk))
    got = np.sort(np.concatenate([p[1] for p in parts]), order="key")
    same = len(got) == len(uk) and bool(np.array_equal(got["key"], uk)) and bool(np.array_equal(got["val"], sums))
    return {"sample_records": ns * world, "sample_distinct": int(len(uk)), "exact_sums_match_numpy_groupby": same,
            "every_key_on_hash_owner": all(p[2] for p in parts)}


def bench_reduce(args, ctx, world, rank, hbm_peak, peak_src, d_cdf, steps=None, warmup=None, e2e=True, uniform=False, dump=None):
    """device-resident ReducePair of rn records per GPU (+ the end-to-end form); returns the line's fields.  dump: directory
    for write_outputs of the last timed step"""
    from thrill_b200 import api, capi
    tg = ctx.tg
    L = tg.L
    rn = args.reduce_n
    K = steps or args.steps
    W = warmup or max(args.warmup, 3)
    kvd = capi.KVDesc(16, capi.OP_SUM_F64)
    d_rin = tg.alloc(rn * 16)

    def gen():
        if uniform:
            tg.ck(L.tg_gen_reduce_uniform(tg.h, d_rin, rank * rn, rn, SEED, ZIPF_UNIVERSE, 0))
        else:
            tg.ck(L.tg_gen_reduce_zipf(tg.h, d_rin, rank * rn, rn, SEED, d_cdf, ZIPF_UNIVERSE, 0))

    r_ms = []
    launches = 0
    hot0 = 0
    for it in range(W + K):
        gen()
        if it == W:
            tg.profile_enable(True)
            hot0 = int(L.tg_hot_records(tg.h))
        tg.barrier()
        l0 = tg.launches()
        tg.timer_start()
        rp, rcount = C.c_void_p(), C.c_size_t()
        tg.ck(L.tg_reduce_by_key(tg.h, C.byref(kvd), d_rin, rn, C.byref(rp), C.byref(rcount)))
        ms = max_over_ranks(tg.timer_stop(), world)
        if it >= W:
            r_ms.append(ms)
            launches += tg.launches() - l0
    part_list = tg.profile_list(capi.K_PARTITION)
    hot_per_step = (int(L.tg_hot_records(tg.h)) - hot0) / float(K)       # records folded by the counting read, never moved
    prof = {name: tg.profile_get(cls) for name, cls in (("partition", capi.K_PARTITION), ("hist", capi.K_RADIX_HIST),
                                                        ("aggregate", capi.K_AGGREGATE), ("compact", capi.K_COMPACT),
                                                        ("segcount", capi.K_SEGCOUNT), ("exchange", capi.K_EXCHANGE),
                                                        ("preagg", capi.K_PREAGG))}
    tg.profile_enable(False)
    if dump:        # before the parity sample below, whose operator call reuses the output buffer
        out = tg.download(rp.value, rcount.value * 16, np.dtype([("key", "<u8"), ("val", "<f8")]))
        out = out[np.argsort(out["key"], kind="stable")]          # the operator's output order is unspecified
        write_outputs(dump, "reduce", world, rank, out["key"], out["val"])
        del out
    # parity of the measured run: ownership of (a sample of) the output keys, then the exact-mode sample
    nchk = min(int(rcount.value), 1 << 20)
    okeys = tg.download(rp.value, nchk * 16, np.dtype([("key", "<u8"), ("val", "<f8")]))["key"] if nchk else np.zeros(0, np.uint64)
    own = bool(np.all(hash128to64_np(okeys) % np.uint64(world) == np.uint64(rank)))
    distinct = sum(gather_objects(int(rcount.value), world))
    parity = {"measured_run_keys_on_hash_owner": all(gather_objects(own, world)), "distinct_out": distinct}
    if not uniform:
        parity.update(reduce_parity(ctx, world, rank, d_cdf))
        parity["ok"] = bool(parity["measured_run_keys_on_hash_owner"] and parity["exact_sums_match_numpy_groupby"]
                            and parity["every_key_on_hash_owner"])
    else:
        parity["ok"] = bool(parity["measured_run_keys_on_hash_owner"])
    if not parity["ok"]:
        raise SystemExit("bench: reduce parity check FAILED: %s" % json.dumps(parity))
    r_step = sum(r_ms) / len(r_ms)
    value = rn * world / (r_step / 1e3)
    part_ms, part_cnt = prof["partition"]
    xchg_ms, xchg_cnt = prof["exchange"]
    # dominant kernel: the stable hash-digit partition pass over the 16-byte records; the two passes of the pre phase move all rn
    # records (read 16 + write 16 bytes each), later launches of a multi-GPU step move the (few) partial aggregates
    # (a step's launch list: the first two partition launches are the pre-phase passes over all rn records)
    per_step = len(part_list) // K if K else 0
    full = [part_list[i * per_step + j] for i in range(K) for j in range(min(2, per_step))] if per_step else []
    launch_ms = sum(full) / len(full) if full else None
    # algorithmic bytes of the two passes of a step: the first reads every record and writes those that were not folded, the
    # second reads and writes the rest; per launch = half of that
    moved = rn - hot_per_step                # (this rank's counter; at N > 1 it includes the few records folded in the post phase)
    pass_bytes = (16.0 * rn + 16.0 * moved + 32.0 * moved) / 2.0
    ach = pass_bytes / (launch_ms / 1e3) / 1e9 if launch_ms else None
    traffic, traffic_src = profile_traffic("r2_partition_pass_kv16.txt")
    model_ach = REDUCE_MODEL_BYTES_PER_RECORD * rn / (r_step / 1e3) / 1e9
    agg_ms, agg_cnt = prof["aggregate"]
    roofline = {"bound": "hbm", "kernel": "tgp::partition_kernel<2,256,8,3,Hot/HashLevelDigit,SEG,unstable> (the two hash-digit passes of a step, averaged: "
                                          "read 16 B + write 16 B per record that is moved; records of popular keys are only read)",
                "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": (ach / hbm_peak) if ach else None, "peak_source": peak_src,
                "traffic": traffic * (rn / 1.25e8) if traffic else None, "traffic_source": traffic_src,
                "algorithmic_bytes_per_launch": pass_bytes, "launch_ms": launch_ms,
                "launches_timed": len(full), "records_folded_by_the_counting_read_per_step": hot_per_step,
                "operator_model": {"bytes_per_record": REDUCE_MODEL_BYTES_PER_RECORD, "what": "SURVEY.md 8(d) ReduceByKey total, Zipf(1, 2^26)",
                                   "achieved_GBps": model_ach, "frac": model_ach / hbm_peak},
                "step_share": {"partition_ms": (part_ms - xchg_ms) / K, "partition_launches_per_step": (part_cnt - xchg_cnt) / K,
                               "count_ms": (prof["hist"][0] + prof["segcount"][0]) / K, "aggregate_ms": agg_ms / K,
                               "preagg_ms": prof["preagg"][0] / K,
                               "compact_ms": prof["compact"][0] / K, "exchange_pass_ms": xchg_ms / K, "step_ms": r_step}}
    res = {"value": value, "ms_per_step": r_step, "roofline": roofline, "parity_check": parity, "gpu_launches": int(launches),
           "steps": K, "warmup": W}
    if e2e:
        KV = api.KV
        host_in = tg.host_alloc(rn * 16)
        cap = int(rcount.value) * 16 * 2 + (1 << 20)
        host_out = tg.host_alloc(cap)
        gen()
        tg.ck(L.tg_download(tg.h, host_in.ctypes.data, d_rin, rn * 16))
        tg.sync()
        dia = api.DIA(ctx, host_in.view(KV))
        e2e_s = []
        for it in range(2 + K):
            tg.barrier()
            t0 = time.perf_counter()
            r = dia.ReducePair(api.PlusDouble, _pinned_out=host_out)
            dt = max_over_ranks(time.perf_counter() - t0, world)
            if it >= 2:
                e2e_s.append(dt)
        out_total = sum(gather_objects(int(len(r.items)), world))
        res["e2e"] = {"value": rn * world / (sum(e2e_s) / len(e2e_s)), "unit": "records/s", "h2d_bytes_per_step": rn * 16 * world,
                      "d2h_bytes_per_step": out_total * 16, "ms_per_step": 1e3 * sum(e2e_s) / len(e2e_s),
                      "call": "thrill_b200.api.DIA.ReducePair -> tg_reduce_file + tg_fetch_output over 1 MiB pinned Blocks"}
        tg.host_free(host_in); tg.host_free(host_out)
    tg.free(d_rin)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--metric", default="sort", choices=["sort", "reduce"], help="which operator is the line's metric")
    ap.add_argument("--n", type=int, default=SORT_N_PER_GPU, help="sort keys per GPU")
    ap.add_argument("--reduce-n", type=int, default=REDUCE_N_PER_GPU, help="reduce records per GPU")
    ap.add_argument("--terasort-n", type=int, default=125000000, help="TeraSort records per GPU of the extra (0 = skip)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="only the metric itself (no second operator, no Zipf sort)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the output of the metric's last timed step to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the GPU arm's outputs; --impl reference has none to write")
        return main_reference(args)

    from thrill_b200 import api
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("bench.py --gpus %d must be launched with torch.distributed.run --nproc-per-node %d" % (args.gpus, args.gpus))
    ctx = api.Context.from_env(rng_seed=SEED)
    tg = ctx.tg
    hbm_peak, peak_src = measured_peaks()
    sampler = ClockSampler(tg.device)
    sampler.start()
    d_cdf = tg.to_device(zipf_cdf_numpy(ZIPF_UNIVERSE))
    extra = {}
    if args.metric == "sort":
        main_res = bench_sort(args, ctx, world, rank, hbm_peak, peak_src, dump=args.dump_outputs)
        if not args.no_extras:
            try:        # an extra must never cost the headline line
                z = bench_sort(args, ctx, world, rank, hbm_peak, peak_src, zipf=True, d_cdf=d_cdf, steps=3, warmup=2, e2e=False)
                extra["sort_zipf"] = {"keys_per_s": z["value"], "ms_per_step": z["ms_per_step"], "workload": "sort_zipf_s1_U2^26_u64_1e8_per_gpu",
                                      "prefix_sort_fallbacks": z["roofline"]["prefix_sort_fallbacks"], "parity_check": z["parity_check"],
                                      "step_share": z["roofline"]["step_share"]}
            except BaseException as e:          # noqa: BLE001
                extra["sort_zipf"] = {"error": str(e)[:300]}
            try:
                r = bench_reduce(args, ctx, world, rank, hbm_peak, peak_src, d_cdf, steps=3, warmup=2, e2e=False)
                extra["reduce"] = {"records_per_s": r["value"], "ms_per_step": r["ms_per_step"], "parity_check": r["parity_check"],
                                   "operator_model": r["roofline"]["operator_model"], "step_share": r["roofline"]["step_share"],
                                   "note": "full line: bench.py --metric reduce"}
            except BaseException as e:          # noqa: BLE001
                extra["reduce"] = {"error": str(e)[:300]}
            if args.terasort_n:
                try:
                    extra["terasort"] = bench_terasort(args, ctx, world, rank, hbm_peak)
                except BaseException as e:          # noqa: BLE001
                    extra["terasort"] = {"error": str(e)[:300]}
        name, unit, dtype, n_item = "sort_keys_per_s", "keys/s", "u64", args.n
    else:
        main_res = bench_reduce(args, ctx, world, rank, hbm_peak, peak_src, d_cdf, dump=args.dump_outputs)
        if not args.no_extras:
            try:
                u = bench_reduce(args, ctx, world, rank, hbm_peak, peak_src, d_cdf, steps=3, warmup=2, e2e=False, uniform=True)
                extra["reduce_uniform"] = {"records_per_s": u["value"], "ms_per_step": u["ms_per_step"], "workload": "reduce_pair_u64_f64_uniform_U2^26",
                                           "distinct_out": u["parity_check"]["distinct_out"], "step_share": u["roofline"]["step_share"]}
            except BaseException as e:          # noqa: BLE001
                extra["reduce_uniform"] = {"error": str(e)[:300]}
        name, unit, dtype, n_item = "reduce_records_per_s", "records/s", "u64 keys, f64 sums", args.reduce_n
    tg.free(d_cdf)
    clocks = sampler.stop()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # bounded sample: the sort baseline runs the full 1e8 keys (~0.7 s per iteration), the reduce baseline 2.5e7 records
        cpu = cpu_baseline(args.metric, n_item if args.metric == "sort" else min(n_item, 25000000))
        if args.metric == "sort" and isinstance(extra.get("reduce"), dict) and "records_per_s" in extra["reduce"]:
            try:        # the second operator's reference throughput on the same box (bounded sample), so both ratios are in one line
                extra["reduce"]["cpu_baseline"] = cpu_baseline("reduce", min(args.reduce_n, 25000000))
            except BaseException as e:          # noqa: BLE001
                extra["reduce"]["cpu_baseline"] = {"error": str(e)[:200]}

    if rank == 0 and world == 1 and args.metric == "sort" and not args.no_extras and not args.no_cpu_baseline:
        extra["e2e_in_thrill"] = e2e_in_thrill()
    if rank == 0:
        cfg = workload_config(args.metric, n_item, world)
        line = {"metric": name, "value": main_res["value"], "unit": unit, "n_gpus": world, "steps": main_res["steps"],
                "warmup": main_res["warmup"], "ms_per_step": main_res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": dtype, "data": "synthetic", "config": cfg, "roofline": main_res["roofline"],
                "cpu_baseline": cpu, "e2e": main_res.get("e2e"), "gpu_launches": main_res["gpu_launches"],
                "parity_check": main_res["parity_check"], "clocks": clocks, "extra": extra}
        print(json.dumps(line))
    ctx.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
