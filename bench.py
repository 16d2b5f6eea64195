#!/usr/bin/env python
"""bench.py -- shuffled rows/sec of the shuffle hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c2|c3|c4] [--dump-outputs DIR]

A "step" is one pass of the shuffle hot path over one batch of synthetic input: map-side hash-partition ->
exchange (NVLink peer push / NCCL alltoallv when N>1) -> reduce-side merge (reduceByKey) or ordered group
(groupByKey).  Weak scaling: the per-GPU work is fixed.  Configs (BASELINE.json `configs`):

  c2 (default)  reduceByKey(sum) over 1e8 (int64,int64) rows per GPU, uniform keys in [0, 2^31), 8 map splits and
                8 reduce partitions per GPU -- configs[1] at 1 GPU, the one `metric` is quoted on.
  c4            benchmarks/stream_shuffle.py shape: (int32,float32) rows, keys in [0, 2^24) (dup-key shape),
                combine = sum (float64 accumulators like the reference's Python floats), 5e8 rows per GPU
                (4e9 at 8 GPUs).
  c3            groupByKey over Zipf(1.1) int64 keys (support 1e9, permuted), values = global row ids,
                8 partitions per GPU (64 at 8 GPUs), 1.25e8 rows per GPU (1e9 at 8 GPUs).

Before the timed loop EVERY run (any N, any config) compares one full reduce partition per rank with the oracle
(oracle/ C restatement) evaluated on that partition's rows gathered from all ranks' inputs, and aborts on a mismatch
(`parity` in the JSON line).

--dump-outputs DIR writes the result of the last timed step (dump_outputs).  The inputs come from fixed seeds, so two
builds run with the same arguments can be compared output for output.

--impl reference times the reference's own CPU implementation on the host cores: the UNMODIFIED douban/dpark built
into baseline/_ref (oracle/build_reference.py) driven through DparkContext('process') by oracle/ref_runner.py;
if that tree is absent, the oracle's CPython port of the same loops (kind "port").
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "shuffled rows/sec (reduceByKey end-to-end)"
UNIT = "rows/s"

CONFIGS = {
    "c2": dict(kind="reduce", kdt="int64", vdt="int64", rows=100_000_000, parts=8, splits=8,
               text="reduceByKey(sum) over %.0e (int64,int64) rows/GPU, uniform keys in [0,2^31), %d map splits/GPU, "
                    "%d reduce partitions/GPU (BASELINE.json configs[1] at 1 GPU)"),
    "c4": dict(kind="reduce", kdt="int32", vdt="float32", rows=500_000_000, parts=8, splits=8,
               text="benchmarks/stream_shuffle.py shape: reduceByKey(sum) over %.0e (int32,float32) rows/GPU, keys in "
                    "[0,2^24) (dup-key shape), %d map splits/GPU, %d reduce partitions/GPU (BASELINE.json configs[3] at 8 GPUs)"),
    "c3": dict(kind="group", kdt="int64", vdt="int64", rows=125_000_000, parts=8, splits=8,
               text="groupByKey over %.3g rows/GPU, Zipf(1.1) int64 keys (support 1e9, odd-multiplier permutation), values = "
                    "global row ids, %d map splits/GPU, %d partitions/GPU (BASELINE.json configs[2] at 8 GPUs)"),
}


AUTO_PIPELINE = "2x2"     # N > 1 default of --pipeline (profiles/r02_ncu_findings.md, session 2)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--rows-per-gpu", type=int, default=0)
    ap.add_argument("--parts-per-gpu", type=int, default=0)
    ap.add_argument("--map-splits", type=int, default=0)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--e2e-depth", type=int, default=3, help="batches in flight in the e2e leg (1 = serial)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--cpu-sample-rows", type=int, default=4_000_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-run oracle comparison (profiling runs only)")
    ap.add_argument("--map-combine", action="store_true", help="merge each rank's map output before the exchange")
    ap.add_argument("--reduce-impl", type=int, default=2, help="A/B switch of the reduce-side kernel (dpk_set_option)")
    ap.add_argument("--sub-bits", type=int, default=-1, help="override the sub-bucket bits (default: auto)")
    ap.add_argument("--agg-target-rows", type=int, default=0, help="override rows per fine bucket (dpk_set_option)")
    ap.add_argument("--count-mode", type=int, default=1, help="A/B switch of the histogram pass (dpk_set_option)")
    ap.add_argument("--agg-wide", type=int, default=-1, help="A/B: 128-bit slot CAS in the round-1 merge kernel (0|1)")
    ap.add_argument("--scatter-items", type=int, default=0, help="A/B: rows per thread and tile of the round-1 multisplit (8|16)")
    ap.add_argument("--scatter-bulk", type=int, default=-1, help="A/B: TMA bulk-store multisplit kernel (0|1)")
    ap.add_argument("--scatter-threads", type=int, default=0, help="A/B: CTA size of the bulk multisplit (256|512)")
    ap.add_argument("--agg-ctas", type=int, default=0, help="A/B: resident CTAs per SM the merge kernel is compiled for (3|4)")
    ap.add_argument("--agg-cursor", type=int, default=-1, help="A/B: merge kernel output ranges by atomic cursor (1) or chained look-back (0)")
    ap.add_argument("--agg-batched", type=int, default=-1, help="A/B: four rows in flight per thread in the merge kernel's insert phase")
    ap.add_argument("--agg-pipe", type=int, default=-1, help="A/B: register-pipelined merge kernel (0 | 1 | 2 = two CTAs per SM)")
    ap.add_argument("--agg-impl", type=int, default=-1, help="A/B: reduce-side merge kernel (0 = round 1, 1 = row-index tags)")
    ap.add_argument("--overlap-push", type=int, default=1, help="N>1, push exchange: groups of map splits whose push "
                    "overlaps the scatter of the next group (1 = no overlap)")
    ap.add_argument("--pipeline", default="auto", help="N>1, push exchange, reduceByKey configs: GxQ = map splits in G groups "
                    "(push of one overlaps the multisplit of the next) and every block in Q parts (reduce side of a part "
                    "overlaps the push of the next): dpark_b200.peer.shuffle_pipelined; 'off' = one push, then reduce; 'auto' = AUTO_PIPELINE")
    ap.add_argument("--copy-engine", type=int, default=-1, help="N>1, --pipeline: pushes by the copy engines (1) or by dpk_copy_segments on --copy-sms SMs (0)")
    ap.add_argument("--copy-sms", type=int, default=-1, help="N>1, overlapped push: whole SMs the overlapped copy kernel takes")
    ap.add_argument("--exchange", default="push", choices=["push", "fused", "peer", "nccl"],
                    help="N>1: push = local scatter, then one kernel pushing each peer's block over NVLink; "
                         "fused (alias peer) = the scatter kernel stores into peer memory; nccl = alltoallv")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last step returned "
                    "as DIR/<name>.npy (float64, rows in key order, a seeded sample above DUMP_ROWS rows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's results (--impl ours)")
    cfg = CONFIGS[args.config]
    args.rows_per_gpu = args.rows_per_gpu or cfg["rows"]
    args.parts_per_gpu = args.parts_per_gpu or cfg["parts"]
    args.map_splits = args.map_splits or cfg["splits"]
    return args


def _isz(name):
    return {"int64": 8, "int32": 4, "float32": 4, "float64": 8}[name]


def workload_config(args, world):
    cfg = CONFIGS[args.config]
    from dpark_b200 import shuffle
    return {
        "workload": cfg["text"] % (args.rows_per_gpu, args.map_splits, args.parts_per_gpu),
        "config": args.config, "rows_per_gpu": args.rows_per_gpu, "partitions": args.parts_per_gpu * world,
        "map_splits_per_gpu": args.map_splits, "parallelism": "dp%d" % world,
        "exchange": None if world == 1 else args.exchange, "map_combine": bool(args.map_combine),
        "overlap_push_groups": args.overlap_push if world > 1 else None,
        "pipeline": ((AUTO_PIPELINE if args.pipeline == "auto" else args.pipeline) or None) if world > 1 else None,
        "l2_policy": "inputs_larger_than_l2 (%.1f GB of rows per GPU per step vs 126 MB L2)"
                     % (args.rows_per_gpu * (_isz(cfg["kdt"]) + _isz(cfg["vdt"])) / 1e9),
        "sub_buckets_per_partition": 1 << shuffle.choose_sub_bits(args.rows_per_gpu, args.parts_per_gpu * world, world),
    }


# ------------------------------------------------------------------------------
# clocks sampler (nvidia-smi in the background, exact PID killed afterwards)
# ------------------------------------------------------------------------------
class Clocks(object):
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.path = tempfile.mktemp(prefix="dpk_clocks_", suffix=".csv")
        self.proc = None
        try:
            self.fh = open(self.path, "w")
            self.proc = subprocess.Popen(
                ["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(index)], stdout=self.fh, stderr=subprocess.DEVNULL)
            time.sleep(0.3)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            try:
                self.proc.kill()
            except Exception:
                pass
        self.fh.close()
        sm, mx, allc, reasons = [], [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    clk, cmax, pw = float(f[2]), float(f[3]), float(f[4])
                except ValueError:
                    continue
                mx.append(cmax)
                allc.append(clk)
                if pw > 200.0:          # under load
                    sm.append(clk)
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                      "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if not sm:
            sm = allc
        if sm:
            sm.sort()
            out["sm_mhz"] = sm[len(sm) // 2]
        if mx:
            out["sm_max_mhz"] = max(mx)
        out["reasons"] = sorted(reasons)
        out["samples"] = len(sm)
        return out


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------
# CPU arm
# ------------------------------------------------------------------------------
def _cpu_map_task(arg):
    """One ShuffleMapTask (dpark/task.py:209-226) + its dump (marshal, as BucketDumper task.py:332-343 does for
    marshalable rows) -- the oracle's CPython port, used when baseline/_ref is absent."""
    import marshal
    import numpy as np
    from oracle import oracle as orc
    seed, n, P = arg
    rng = np.random.default_rng(seed)
    keys = rng.integers(0, 2 ** 31, n, dtype=np.int64).tolist()
    vals = rng.integers(0, 2 ** 16, n, dtype=np.int64).tolist()
    rows = list(zip(keys, vals))
    t0 = time.perf_counter()
    import operator
    buckets = orc.py_shuffle_map_task(rows, P, lambda x: x, operator.add, None, hash)  # ints: portable_hash == hash()
    blobs = [marshal.dumps(list(b.items())) for b in buckets]
    return blobs, time.perf_counter() - t0


def _cpu_reduce_task(blobs):
    """One reducer: fetch every map's bucket and merge (dpark/shuffle.py:247-289, 600-608)."""
    import marshal
    import operator
    from oracle import oracle as orc
    t0 = time.perf_counter()
    d = orc.py_merge((marshal.loads(b) for b in blobs), operator.add)
    return len(d), time.perf_counter() - t0


def cpu_port_run(rows, P, procs):
    """Throughput of the CPython port on `procs` cores: M=procs map tasks in parallel, then P reduce tasks in
    parallel, like the reference's MultiProcessScheduler (dpark/schedule.py:841-910).  Input generation is not timed."""
    import multiprocessing as mp
    M = max(1, procs)
    per = rows // M
    args = [(1000 + i, per, P) for i in range(M)]
    if procs <= 1:
        outs = [_cpu_map_task(a) for a in args]
        gen_excl = sum(t for _, t in outs)
        blobs = [o for o, _ in outs]
        red = [_cpu_reduce_task([b[r] for b in blobs]) for r in range(P)]
        secs = gen_excl + sum(t for _, t in red)
        return per * M / secs, per * M, secs
    ctx = mp.get_context("fork")
    with ctx.Pool(procs) as pool:
        outs = pool.map(_cpu_map_task, args)
        map_wall = max(t for _, t in outs)           # tasks run concurrently, one per core
        blobs = [o for o, _ in outs]
        t0 = time.perf_counter()
        pool.map(_cpu_reduce_task, [[b[r] for b in blobs] for r in range(P)])
        red_wall = time.perf_counter() - t0
    secs = map_wall + red_wall
    return per * M / secs, per * M, secs


def reference_available():
    import sysconfig
    ext = sysconfig.get_config_var("EXT_SUFFIX")
    return os.path.exists(os.path.join(ROOT, "baseline", "_ref", "dpark", "portable_hash" + ext))


def reference_run(config, rows, splits, parts, procs, master="process", timeout=600):
    """One bounded run of the UNMODIFIED reference in its own process group (killed as a group on timeout).
    Returns the runner's JSON dict or None."""
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "ref_runner.py"), "--config", config, "--rows", str(rows),
           "--splits", str(splits), "--parts", str(parts), "--procs", str(procs), "--master", master]
    out_path = tempfile.mktemp(prefix="dpk_ref_", suffix=".json")
    try:
        with open(out_path, "w") as fo:
            p = subprocess.Popen(cmd, stdout=fo, stderr=subprocess.DEVNULL, stdin=subprocess.DEVNULL,
                                 start_new_session=True, cwd=ROOT)
            try:
                p.wait(timeout=timeout)
            except subprocess.TimeoutExpired:
                try:
                    os.killpg(p.pid, 9)          # the exact process group this call started
                except Exception:
                    pass
                p.wait()
                return None
        for line in open(out_path):
            line = line.strip()
            if line.startswith("{"):
                return json.loads(line)
    except Exception:
        return None
    finally:
        try:
            os.unlink(out_path)
        except Exception:
            pass
    return None


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    P = args.parts_per_gpu * args.gpus
    steps = max(1, min(args.steps, 3))
    warm = min(args.warmup, 1)
    use_ref = reference_available()
    vals, t_all, info = [], 0.0, None
    if use_ref:
        # bounded sample: the reference moves ~0.5-1 M rows/s per map process through pickle + dict loops
        sample = min(args.cpu_sample_rows, 8_000_000)
        splits = max(args.map_splits * args.gpus, min(cores, 128))
        if warm:
            reference_run(args.config, max(sample // 8, 100_000), splits, P, cores, timeout=300)
        for _ in range(steps):
            r = reference_run(args.config, sample, splits, P, cores, timeout=600)
            if r is None:
                use_ref = False
                break
            info = r
            vals.append(r["rows"] / r["shuffle_s"])
            t_all += r["shuffle_s"]
    if not use_ref:
        vals, t_all = [], 0.0
        sample = min(args.cpu_sample_rows * max(1, min(cores, 32)) // 4, 64_000_000)
        for _ in range(warm):
            cpu_port_run(sample // 4, P, cores)
        for _ in range(steps):
            v, nrows, secs = cpu_port_run(sample, P, cores)
            vals.append(v)
            t_all += secs
    value = sum(vals) / len(vals)
    if use_ref:
        cb = {"value": value, "unit": UNIT, "cores": cores, "kind": "reference",
              "sample": "%d rows per step through the UNMODIFIED reference (baseline/_ref, DparkContext('process') -p %d, "
                        "%d map splits, %d reduce partitions, tracker shim of SURVEY Appendix B); shuffle-only time = "
                        "job time - source count() time (SURVEY 8d): last step job %.2f s, source %.2f s"
                        % (info["rows"], cores, info["splits"], P, info["job_s"], info["src_count_s"]),
              "native_so_loaded": info.get("native_so_loaded"), "whole_job_value": info["rows"] / info["job_s"]}
    else:
        cb = {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
              "sample": "baseline/_ref absent: CPython port of task.py:209-226 + shuffle.py:600-608 with marshal dumps, "
                        "M=%d map tasks then P=%d reduce tasks in a fork pool" % (cores, P)}
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": 1e3 * t_all / steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64" if args.config == "c4" else CONFIGS[args.config]["vdt"],
        "data": "synthetic", "config": workload_config(args, args.gpus), "cpu_baseline": cb,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# ------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------
def gen_inputs(args, rank, world, dev):
    """Synthetic columns of this rank (SURVEY.md 8d generators), device tensors."""
    import torch
    n = args.rows_per_gpu
    g = torch.Generator(device=dev)
    if args.config == "c2":
        g.manual_seed(1234 + rank)
        keys = torch.randint(0, 2 ** 31, (n,), dtype=torch.int64, device=dev, generator=g)
        g.manual_seed(1235 + rank)
        vals = torch.randint(0, 2 ** 16, (n,), dtype=torch.int64, device=dev, generator=g)
    elif args.config == "c4":
        g.manual_seed(77 + rank)
        keys = torch.randint(0, 2 ** 24, (n,), dtype=torch.int32, device=dev, generator=g)
        g.manual_seed(78 + rank)
        vals = torch.rand((n,), dtype=torch.float32, device=dev, generator=g)
    else:  # c3: Zipf(1.1) ranks over a support of 1e9 by inverse CDF, permuted by an odd multiplier mod 2^31
        g.manual_seed(2025 + rank)
        s, support = 1.1, 1.0e9
        keys = torch.empty(n, dtype=torch.int64, device=dev)
        chunk = 1 << 24
        for a in range(0, n, chunk):
            b = min(n, a + chunk)
            u = torch.rand((b - a,), dtype=torch.float64, device=dev, generator=g)
            r = torch.pow(1.0 - u * (1.0 - support ** (1.0 - s)), 1.0 / (1.0 - s)).clamp_(1.0, support).to(torch.int64)
            keys[a:b] = (r * 0x9E3779B1) & 0x7FFFFFFF
            del u, r
        vals = torch.arange(rank * n, rank * n + n, dtype=torch.int64, device=dev)
    return keys, vals


def parity_check(args, keys, vals, out, P, world, rank, dev):
    """Oracle comparison inside the bench, at every N: rank r checks the FIRST partition it owns against the oracle
    (C restatement of DiskHashMerger._merge / OrderedGroupByDiskHashMerger) run on that partition's rows, which every
    rank selects from its own input with the oracle's portable_hash / getPartition and sends over.  Returns a dict
    for the JSON line; raises on a mismatch."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from dpark_b200 import shuffle
    from oracle import oracle as orc
    t0 = time.perf_counter()
    blocks = shuffle.owner_blocks(P, world)
    check_parts = [blocks[r] if blocks[r + 1] > blocks[r] else -1 for r in range(world)]
    hk = keys.cpu().numpy()
    hv = vals.cpu().numpy()
    pid = orc.partition_vec(orc.hash_vec(hk), P)
    send_k, send_v, counts = [], [], []
    for r in range(world):
        sel = np.nonzero(pid == check_parts[r])[0] if check_parts[r] >= 0 else np.zeros(0, np.int64)
        send_k.append(hk[sel])
        send_v.append(hv[sel])
        counts.append(len(sel))
    del pid
    if world > 1:
        cnt = torch.tensor(counts, dtype=torch.int64, device=dev)
        rcnt = torch.empty_like(cnt)
        dist.all_to_all_single(rcnt, cnt)
        rc = rcnt.cpu().tolist()
        sk = torch.from_numpy(np.concatenate(send_k)).to(dev)
        sv = torch.from_numpy(np.concatenate(send_v)).to(dev)
        rk = torch.empty(sum(rc), dtype=sk.dtype, device=dev)
        rv = torch.empty(sum(rc), dtype=sv.dtype, device=dev)
        dist.all_to_all_single(rk, sk, rc, counts)
        dist.all_to_all_single(rv, sv, rc, counts)
        gk, gv = rk.cpu().numpy(), rv.cpu().numpy()      # source-rank-major == map order
        del sk, sv, rk, rv
    else:
        gk, gv = send_k[0], send_v[0]
    p = check_parts[rank]
    rows_checked, ok, detail = int(len(gk)), True, ""
    if p >= 0:
        if CONFIGS[args.config]["kind"] == "reduce":
            wk, wv = orc.merge(gk.astype(np.int64), gv, "sum")
            okeys, ovals, po, cnt_h = out
            j = p - blocks[rank]
            a, c = int(po[j]), int(cnt_h[j])
            mk = okeys[a:a + c].cpu().numpy().astype(np.int64)
            mv = ovals[a:a + c].cpu().numpy()
            o1, o2 = np.argsort(mk, kind="stable"), np.argsort(wk, kind="stable")
            ok = len(mk) == len(wk) and np.array_equal(mk[o1], wk[o2])
            if ok:
                if mv.dtype.kind == "f":   # float sums: order differs from the oracle's; tolerance as in DESIGN.md section 7
                    asum = np.zeros(len(wk))
                    np.add.at(asum, np.searchsorted(wk[o2], gk.astype(np.int64)), np.abs(gv.astype(np.float64)))
                    ok = bool(np.all(np.abs(mv[o1] - wv[o2]) <= 1e-9 * asum + 1e-300))
                    detail = "float64 sums within 1e-9 * sum|v| per key"
                else:
                    ok = np.array_equal(mv[o1], wv[o2])
                    detail = "bit-exact"
        else:
            wk, wo, wvals = orc.group(gk, gv)
            gkeys, gstarts, ng, ovals, poff = out
            G = int(ng.item())
            j = p - blocks[rank]
            poff_h = poff.cpu().numpy()
            gs = gstarts[:G + 1].cpu().numpy()
            g0 = int(np.searchsorted(gs[:-1], poff_h[j], side="left"))
            g1 = int(np.searchsorted(gs[:-1], poff_h[j + 1], side="left"))
            mk = gkeys[g0:g1].cpu().numpy()
            mo = gs[g0:g1 + 1]
            mvals = ovals[int(mo[0]):int(mo[-1])].cpu().numpy() if g1 > g0 else np.zeros(0, np.int64)
            o1, o2 = np.argsort(mk, kind="stable"), np.argsort(wk, kind="stable")
            ok = len(mk) == len(wk) and np.array_equal(mk[o1], wk[o2])
            if ok:   # same group sizes and the same value list per key, in (map split, position) order
                ml, wl = (mo[1:] - mo[:-1])[o1], (wo[1:] - wo[:-1])[o2]
                ok = np.array_equal(ml, wl)
                if ok and len(mk):
                    ms, ws = (mo[:-1] - mo[0])[o1], wo[:-1][o2]
                    within = np.arange(int(ml.sum())) - np.repeat(np.cumsum(ml) - ml, ml)
                    ok = np.array_equal(mvals[np.repeat(ms, ml) + within], wvals[np.repeat(ws, wl) + within])
            detail = "groups and per-key value order bit-exact"
    flags = [None] * world
    if world > 1:
        dist.all_gather_object(flags, (bool(ok), rows_checked, p))
    else:
        flags = [(bool(ok), rows_checked, p)]
    if not all(f[0] for f in flags):
        raise SystemExit("PARITY FAILURE against the oracle: %r" % (flags,))
    return {"parity_checked": True, "partitions": [f[2] for f in flags], "rows": sum(f[1] for f in flags),
            "how": "one full partition per rank vs oracle/ C restatement on the gathered input rows; " + detail,
            "seconds": round(time.perf_counter() - t0, 1)}


DUMP_ROWS = 1 << 20     # rows per array kept by dump_outputs over all ranks: at most 4 x 8 MiB of .npy files


def dump_outputs(path, out, group, world, rank, first_part):
    """Writes one step's result as float64 .npy files under `path` (names prefixed rank<r>_ when N > 1).  Rows are
    put in key order, which no run-to-run detail of the kernels changes: keys are unique in a reduce result and name
    one group each in a group result.  Above DUMP_ROWS / N rows a kind is sampled at positions drawn with a fixed seed.
    Integer keys and values are exact in float64 for every config (all below 2^53).

      reduce: keys, values, partition (global id per row), partition_counts (distinct keys per local partition)
      group:  keys, group_sizes, partition (per group), partition_counts (groups per local partition), and values:
              the groups' values concatenated in key order, each group's in the order the step returned them"""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    cap = DUMP_ROWS // world
    rng = np.random.default_rng(20240611)
    prefix = "rank%d_" % rank if world > 1 else ""

    def sample(n, dev):
        if n <= cap:
            return torch.arange(n, device=dev)
        return torch.from_numpy(np.sort(rng.choice(n, cap, replace=False))).to(dev)

    def save(name, t):
        np.save(os.path.join(path, prefix + name + ".npy"), t.cpu().numpy().astype(np.float64))

    if group:
        gkeys, gstarts, ng, vals, poff = out
        G = int(ng.item())
        keys, starts, poff = gkeys[:G], gstarts[:G + 1].to(torch.int64), poff.to(torch.int64)
        dev = keys.device
        part = torch.searchsorted(poff, starts[:-1], right=True) - 1
        order = torch.argsort(keys, stable=True)
        sizes, src = (starts[1:] - starts[:-1])[order], starts[:-1][order]
        sel = order[sample(G, dev)]
        save("keys", keys[sel])
        save("group_sizes", starts[1:][sel] - starts[:-1][sel])
        save("partition", part[sel] + first_part)
        save("partition_counts", torch.bincount(part, minlength=len(poff) - 1))
        ends = torch.cumsum(sizes, 0)
        q = sample(int(ends[-1]) if G else 0, dev)
        g = torch.searchsorted(ends, q, right=True)
        save("values", vals[src[g] + q - (ends[g] - sizes[g])])
    else:
        okeys, ovals, po, cnt = out
        po_h, cnt_h = po.cpu().tolist(), cnt.cpu().tolist()
        dev = okeys.device
        rows = torch.cat([torch.arange(po_h[j], po_h[j] + cnt_h[j], device=dev) for j in range(len(cnt_h))])
        keys, vals = okeys[rows], ovals[rows]
        part = torch.repeat_interleave(torch.arange(len(cnt_h), device=dev), cnt.to(torch.int64))
        sel = torch.argsort(keys, stable=True)[sample(len(rows), dev)]
        save("keys", keys[sel])
        save("values", vals[sel])
        save("partition", part[sel] + first_part)
        save("partition_counts", cnt)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from dpark_b200 import _native as nv
    from dpark_b200 import shuffle

    cfg = CONFIGS[args.config]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (no CPU fallback)")
    numa = shuffle.bind_to_gpu_numa_node(local)
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    n, P, M = args.rows_per_gpu, args.parts_per_gpu * world, args.map_splits
    kdt, vdt = getattr(torch, cfg["kdt"]), getattr(torch, cfg["vdt"])
    KB, VB = _isz(cfg["kdt"]), _isz(cfg["vdt"])
    group = cfg["kind"] == "group"

    keys, vals = gen_inputs(args, rank, world, dev)
    per = (n + M - 1) // M
    kc = [keys[i * per:min(n, (i + 1) * per)] for i in range(M)]
    vc = [vals[i * per:min(n, (i + 1) * per)] for i in range(M)]

    sub_bits = shuffle.choose_sub_bits(n, P, world) if args.sub_bits < 0 else args.sub_bits
    nv.set_option("reduce_impl", args.reduce_impl)
    if args.agg_target_rows > 0:
        nv.set_option("agg_target_rows", args.agg_target_rows)
    nv.set_option("count_mode", args.count_mode)
    if args.scatter_items:
        nv.set_option("scatter_items", args.scatter_items)
    if args.agg_wide >= 0:
        nv.set_option("agg_wide", args.agg_wide)
    if args.scatter_bulk >= 0:
        nv.set_option("scatter_bulk", args.scatter_bulk)
    if args.agg_impl >= 0:
        nv.set_option("agg_impl", args.agg_impl)
    if args.scatter_threads:
        nv.set_option("scatter_threads", args.scatter_threads)
    if args.agg_ctas:
        nv.set_option("agg_ctas", args.agg_ctas)
    if args.agg_cursor >= 0:
        nv.set_option("agg_cursor", args.agg_cursor)
    if args.agg_batched >= 0:
        nv.set_option("agg_batched", args.agg_batched)
    if args.agg_pipe >= 0:
        nv.set_option("agg_pipe", args.agg_pipe)

    ex_events = []
    px = None
    acc_dt = nv.acc_dtype(vdt)
    xv_dt = acc_dt if args.map_combine else vdt     # after a map-side combine the value column is the accumulator type
    recv_factor = 2.6 if args.config == "c3" else 1.25   # c3: the owner of the hottest key receives ~2.2x its share
    if world > 1 and args.exchange != "nccl":
        try:
            from dpark_b200 import peer
            px = peer.PeerExchange(int(n * recv_factor) + (1 << 20), kdt, xv_dt, dev,
                                   mode="push" if args.exchange == "push" else "fused")
            if args.copy_sms >= 0:
                px.copy_sms = args.copy_sms
            if args.copy_engine >= 0:
                px.copy_engine = args.copy_engine
        except Exception as e:  # symmetric memory unavailable on this box/build: say so, use NCCL
            sys.stderr.write("peer exchange unavailable (%s: %s); using NCCL alltoallv\n" % (type(e).__name__, e))
            px = None

    pipe = None
    if args.pipeline == "auto":
        args.pipeline = AUTO_PIPELINE if world > 1 else "off"
    if args.pipeline and args.pipeline != "off" and px is not None and px.mode == "push" and not group and not args.map_combine:
        g_, q_ = args.pipeline.lower().split("x")
        pipe = (int(g_), int(q_))

    def step():
        if pipe is not None:
            return peer.shuffle_pipelined(px, kc, vc, P, "sum", None, sub_bits, pipe[0], pipe[1])
        if px is not None and px.mode == "fused" and not group and not args.map_combine:
            rx = peer.map_side_push(px, kc, vc, P, None, sub_bits)
            return shuffle.reduce_side(rx, "sum", P)
        if px is not None and px.mode == "push" and args.overlap_push > 1 and not group and not args.map_combine:
            rx = peer.map_exchange_overlapped(px, kc, vc, P, None, sub_bits, True, args.overlap_push)
            return shuffle.reduce_side(rx, "sum", P)
        mo = shuffle.map_side(kc, vc, P, None, False, sub_bits, unordered=not group)
        if args.map_combine and not group:
            mo = shuffle.combine_map_output(mo, "sum")
        if px is not None:
            rx = peer.exchange_push(px, mo)
        elif world > 1:    # bracket the one collective (alltoallv) for the NVLink roofline
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            rx = shuffle.exchange(mo)
            b.record()
            ex_events.append((a, b))
        else:
            rx = shuffle.exchange(mo)
        if group:
            return shuffle.group_side(rx, P)
        return shuffle.reduce_side(rx, "sum", P)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        out = step()
    barrier()
    if px is not None:
        px.check()                     # device-side capacity flag of the peer receive buffers
    # ---- parity inside the bench (every N): one full partition per rank against the oracle
    if group:
        gk_, gs_, ng_, ov_, poff_ = out
        distinct_local = int(ng_.item())
        nrecv_local = int(ov_.numel())
        checked = (gk_, gs_, ng_, ov_, poff_)
    else:
        if pipe is not None:
            out = peer.merge_part_results(out)
        ok_, ov_, po_, cnt_ = out
        po_h, cnt_h = po_.cpu().tolist(), cnt_.cpu().tolist()
        if any(c < 0 for c in cnt_h):
            raise SystemExit("reduce side reported a failed partition (table overflow)")
        distinct_local = sum(cnt_h)
        nrecv_local = int(po_h[-1])        # part_offsets[nparts] = rows this rank's reduce side received
        checked = (ok_, ov_, po_h, cnt_h)
    parity = {"parity_checked": False}
    if not args.no_parity:
        parity = parity_check(args, keys, vals, checked, P, world, rank, dev)
    tot = torch.tensor([distinct_local, nrecv_local], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(tot)
    distinct_all, nrecv_all = int(tot[0]), int(tot[1])
    assert nrecv_all == n * world or args.map_combine, "rows were lost in the exchange"
    del out, checked, ov_

    clocks = Clocks(local) if rank == 0 else None
    launches0 = nv.launch_count()
    nv.prof_enable(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    del ex_events[:]
    e0.record()
    for _ in range(args.steps - 1):
        step()
    last = step()
    e1.record()
    barrier()
    nv.prof_enable(False)
    if args.dump_outputs:
        try:
            if pipe is not None:
                last = peer.merge_part_results(last)
            dump_outputs(args.dump_outputs, last, group, world, rank, shuffle.owner_blocks(P, world)[rank])
        except BaseException:      # the clocks sampler is a child process: do not leave it running
            if clocks:
                clocks.stop()
            raise
    del last
    launches = nv.launch_count() - launches0
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_step = float(ms) / args.steps
    value = n * world / (ms_step * 1e-3)

    # per-kernel device times from the library's own CUDA events (same stream)
    prof = nv.prof_collect()
    agg = {}
    for name, t in prof:
        a = agg.setdefault(name, [0.0, 0])
        a[0] += t
        a[1] += 1
    kv = KB + VB
    okv = KB + 8                       # output pairs: key + 8-byte accumulator
    nrecv = nrecv_local                # rows THIS rank's reduce side received
    alg = {  # algorithmic bytes per STEP for each kernel of this rank (SURVEY.md 8d)
        "part_count": KB * n,                         # the two-pass histogram re-read: not credited to the map side
        "part_scatter": 2 * kv * n,                   # read each pair once, write it once
        "tbl_init": 0,
        "tbl_insert": kv * nrecv,
        "tbl_compact": okv * distinct_local,
        "bucket_reduce": kv * nrecv + okv * distinct_local,
        "seg_count": KB * nrecv,                      # second-level split: histogram re-read (not credited)
        "seg_scatter": 2 * kv * nrecv,                # second-level split: read + write every received pair
        "smem_aggregate": kv * nrecv + okv * distinct_local,   # read every pair once, write one pair per distinct key
        "radix_scatter": 2 * kv * nrecv,              # one LSD pass of the group-by sort
        "group_heads": KB * nrecv + (KB + 8) * distinct_local,
    }
    kernels = []
    ktotal = sum(a[0] for a in agg.values()) or 1.0
    for name, (t, c) in sorted(agg.items(), key=lambda x: -x[1][0])[:12]:
        per_step_ms = t / args.steps
        kernels.append({"kernel": name, "n": round(c / args.steps, 2), "ms": round(per_step_ms, 4),
                        "share": round(t / ktotal, 4),
                        "alg_gbs": round(alg.get(name, 0) / (per_step_ms * 1e-3) / 1e9, 1) if per_step_ms > 0 else None})
    peak, peak_src = hbm_peak()
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic_tab = json.load(f).get(args.config, {})
    except Exception:
        traffic_tab = {}
    titles = {"part_scatter": "k_part_scatter (map-side stable multisplit)" if group else
                              "k_part_scatter_bulk (map-side multisplit, TMA bulk stores)",
              "smem_aggregate": "k_smem_aggregate2 (reduce-side merge, row-index tags in shared memory)",
              "seg_scatter": "k_part_scatter_bulk in segmented mode (reduce-side second-level split)",
              "bucket_reduce": "k_bucket_reduce (reduce-side merge, cluster per bucket)",
              "tbl_insert": "k_tbl_insert (reduce-side merge, global tables)",
              "radix_scatter": "k_part_scatter, radix digit mode (stable LSD pass of the group-by sort)"}

    def roofline_of(name):
        t_ms, cnt = agg.get(name, [0.0, 0])
        if not cnt or t_ms <= 0:
            return None
        launch_ms = t_ms / cnt
        bytes_launch = alg.get(name, 0) * args.steps / cnt          # algorithmic bytes of ONE launch
        gbs = bytes_launch / (launch_ms * 1e-3) / 1e9
        tr = traffic_tab.get(name, {})
        return {"bound": "hbm", "kernel": titles.get(name, name), "achieved": gbs, "peak": peak, "unit": "GB/s",
                "frac": gbs / peak, "traffic": tr.get("dram_bytes_per_launch"), "traffic_source": tr.get("source"),
                "peak_source": peak_src, "alg_bytes_per_launch": bytes_launch, "ms_per_launch": launch_ms,
                "share_of_step": t_ms / ktotal}

    cands = [k for k in titles if k in agg]
    dom = max(cands, key=lambda k: agg[k][0]) if cands else "part_scatter"
    roofline = roofline_of(dom)
    roofline_map_scatter = roofline_of("part_scatter")
    map_ms = sum(agg.get(k, [0.0, 0])[0] for k in ("part_count", "part_scan", "part_offsets", "part_scatter")) / args.steps
    roofline_map_side = None
    if map_ms > 0:
        roofline_map_side = {"bound": "hbm", "kernel": "map side, all kernels (histogram + scan + scatter; credited 2*(K+V) per row)",
                             "achieved": alg["part_scatter"] / (map_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": alg["part_scatter"] / (map_ms * 1e-3) / 1e9 / peak, "ms_per_step": map_ms}
    red_names = ("tbl_plan", "side_init", "side_flush", "tbl_init", "tbl_insert", "tbl_compact", "bucket_reduce",
                 "seg_plan", "seg_count", "seg_scan", "seg_scatter", "smem_aggregate", "radix_count", "radix_scatter",
                 "group_heads", "key_or")
    red_ms = sum(agg.get(k, [0.0, 0])[0] for k in red_names) / args.steps
    roofline_reduce = None
    if red_ms > 0:
        red_bytes = (kv * nrecv + VB * nrecv + (KB + 8) * distinct_local) if group else alg["smem_aggregate"]
        roofline_reduce = {"bound": "hbm", "kernel": "reduce side, all kernels (%s)" % (
                               "ordered group-by: LSD passes + CSR heads" if group else
                               "second-level split + shared-memory merge"),
                           "achieved": red_bytes / (red_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                           "frac": red_bytes / (red_ms * 1e-3) / 1e9 / peak, "ms_per_step": red_ms,
                           "alg_bytes_per_step": red_bytes}
    roofline_exchange = None
    xb = KB + (8 if args.map_combine else VB)
    if world > 1 and ex_events:
        ex_ms = torch.tensor([sum(a.elapsed_time(b) for a, b in ex_events) / len(ex_events)],
                             dtype=torch.float64, device=dev)
        dist.all_reduce(ex_ms, op=dist.ReduceOp.MAX)
        sent = xb * n * (world - 1) / world
        gbs = sent / (float(ex_ms) * 1e-3) / 1e9
        roofline_exchange = {"bound": "nvlink", "kernel": "alltoallv (counts all-gather + 2 x all_to_all_single)",
                             "achieved": gbs, "peak": 770.0, "unit": "GB/s per GPU per direction",
                             "frac": gbs / 770.0, "ms_per_step_max_over_ranks": float(ex_ms),
                             "peak_source": "measured peer copy on this pool (B200_PROFILING.md); nominal 900"}
    if world > 1 and px is not None:
        exk = "part_scatter" if px.mode == "fused" else "copy_segments"
        sc_ms = sum(t for name, t in prof if name == exk) / args.steps
        sc = torch.tensor([sc_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(sc, op=dist.ReduceOp.MAX)
        sent = xb * n * (world - 1) / world          # bytes a rank pushes to OTHER ranks per step (uniform keys)
        if float(sc) > 0:
            gbs = sent / (float(sc) * 1e-3) / 1e9
            roofline_exchange = {"bound": "nvlink", "kernel": "k_part_scatter_bulk storing into peer receive buffers (TMA)" if
                                 px.mode == "fused" else "k_copy_segments: one launch pushing every peer's block",
                                 "achieved": gbs, "peak": 770.0, "unit": "GB/s per GPU per direction",
                                 "frac": gbs / 770.0, "ms_per_step_max_over_ranks": float(sc),
                                 "peak_source": "measured peer copy on this pool (B200_PROFILING.md); nominal 900"}
        else:    # pipelined step with copy-engine pushes: no kernel of ours moves the bytes; they cross NVLink under the
            # multisplit and the merge, so what the step pays for the exchange is its time beyond the kernels' sum
            roofline_exchange = {"bound": "nvlink", "kernel": "copy engines (cudaMemcpyAsync on the peers' mapped receive "
                                 "buffers), overlapped with the multisplit and the merge", "achieved": None, "peak": 770.0,
                                 "unit": "GB/s per GPU per direction", "frac": None,
                                 "bytes_pushed_per_gpu_per_step": sent,
                                 "lower_bound_ms": sent / 770e9 * 1e3,
                                 "step_ms_minus_kernel_ms": ms_step - ktotal / args.steps,
                                 "peak_source": "measured peer copy on this pool (B200_PROFILING.md); nominal 900"}

    # ---- e2e: host buffers through the public HostShuffleStream call ---------------------------------------
    e2e = None
    if not args.no_e2e:
        del kc, vc
        e2e = run_e2e(args, keys, vals, kdt, vdt, P, M, sub_bits, world, dev, barrier, group, recv_factor, px)
    clk = clocks.stop() if clocks else None

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline = cpu_baseline_leg(args, P)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64" if args.config == "c4" else cfg["vdt"],
            "data": "synthetic", "kernels": kernels,
            "config": workload_config(args, world), "gpu_launches": launches, "numa_node": numa,
            "distinct_keys": distinct_all, "cpu_baseline": cpu_baseline, "clocks": clk,
            "roofline_reduce": roofline_reduce, "roofline_map_side": roofline_map_side,
            "roofline_map_scatter": roofline_map_scatter, "roofline": roofline,
            "roofline_exchange": roofline_exchange, "parity": parity, "e2e": e2e,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def cpu_baseline_leg(args, P):
    """Reported CPU baseline at N=1: the UNMODIFIED reference on all host cores when baseline/_ref travelled with
    the snapshot, else the CPython port on one core.  Bounded sample."""
    cores = os.cpu_count() or 1
    if reference_available():
        sample = min(args.cpu_sample_rows, 4_000_000)
        splits = max(args.map_splits, min(cores, 128))
        r = reference_run(args.config, sample, splits, P, cores, timeout=420)
        if r is not None:
            return {"value": r["rows"] / r["shuffle_s"], "unit": UNIT, "cores": cores, "kind": "reference",
                    "sample": "%d rows through the UNMODIFIED reference (baseline/_ref, DparkContext('process') -p %d, %d "
                              "map splits, %d reduce partitions); shuffle-only = job %.2f s - source count %.2f s"
                              % (r["rows"], cores, r["splits"], P, r["job_s"], r["src_count_s"]),
                    "whole_job_value": r["rows"] / r["job_s"], "native_so_loaded": r.get("native_so_loaded")}
    v, nrows, secs = cpu_port_run(min(args.cpu_sample_rows, 4_000_000), P, 1)
    return {"value": v, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": "%d rows (same generator), CPython port of task.py:209-226 + shuffle.py:600-608, %.1f s"
                      % (nrows, secs)}


def run_e2e(args, keys, vals, kdt, vdt, P, M, sub_bits, world, dev, barrier, group, recv_factor, px):
    """Same metric through the public host-buffer API: pinned host columns in, pinned host result out, both
    copies inside the timed region every step.  Pipelined (HostShuffleStream, `depth` batches in flight, one
    PeerExchange per slot when N>1) unless --e2e-depth 1."""
    import torch
    import torch.distributed as dist
    from dpark_b200 import shuffle
    n = args.rows_per_gpu
    kind = "group" if group else "reduce"
    h_keys = torch.empty(n, dtype=kdt).pin_memory()
    h_vals = torch.empty(n, dtype=vdt).pin_memory()
    h_keys.copy_(keys)
    h_vals.copy_(vals)
    torch.cuda.synchronize()
    del keys, vals
    if px is not None:
        px.close()
    torch.cuda.empty_cache()
    depth = max(1, args.e2e_depth)
    st = shuffle.HostShuffleStream(n, kdt, vdt, P, "sum", splits=M, sub_bits=sub_bits, depth=depth, kind=kind,
                                   peer_mode=None if (world == 1 or args.exchange == "nccl") else "push",
                                   recv_factor=recv_factor)
    for _ in range(depth):
        st.submit(h_keys, h_vals)
    for _ in range(depth):
        st.collect()
    barrier()
    K2 = max(args.e2e_steps * 4, 12) if depth > 1 else max(args.e2e_steps, 3)
    t0 = time.perf_counter()
    inflight = 0
    for _ in range(K2):
        if inflight == depth:
            st.collect()
            inflight -= 1
        st.submit(h_keys, h_vals)
        inflight += 1
    while inflight:
        st.collect()
        inflight -= 1
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) * 1e3
    t = torch.tensor([wall], dtype=torch.float64, device=dev)
    b = torch.tensor([float(st.h2d_bytes), float(st.d2h_bytes)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(b)
    step_ms = float(t) / K2
    st.close()
    return {"value": n * world / (step_ms * 1e-3), "unit": UNIT, "ms_per_step": step_ms, "steps": K2,
            "h2d_bytes_per_step": int(b[0]), "d2h_bytes_per_step": int(b[1]), "depth": depth,
            "api": "dpark_b200.shuffle.HostShuffleStream.submit/collect on every rank (pinned host in, pinned host "
                   "out, %d batches in flight%s); wall clock over %d batches incl. pipeline fill and drain, max over ranks"
                   % (depth, ", one PeerExchange per slot" if world > 1 else "", K2)}


_REAL_STDOUT = None


def emit(line):
    """The one JSON line goes to the process's real stdout; everything else any library prints
    (NCCL's version banner, warnings) was diverted to stderr in main()."""
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    global _REAL_STDOUT
    args = parse()
    # keep stdout clean: fd 1 -> stderr for the whole run, the JSON line is written to a dup of the original fd 1
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
