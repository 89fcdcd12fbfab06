#!/usr/bin/env python3
"""bench.py - the corpus-scan hot path on N B200s of one node (BASELINE.json metric: source MB/s, files/s,
fraction of the HBM-read roofline).

    python bench.py --gpus N --steps K --warmup W [--config C2|C3|C4|C5]    # this repo's sm_100a path
    python bench.py --impl reference --gpus N --steps K ... [--config ..]   # the CPU restatement on the host cores
    python bench.py ... --dump-outputs DIR     # also write what the last timed step computed, DIR/<name>.npy (float64)

Configs (BASELINE.json `configs`, SURVEY.md section 8d; the default and the headline is C2):
  C2  100 000 synthetic files x 4 KiB per GPU (weak scaling), tokenise + line-hash + classify + aggregate
  C3  1 000 000 files x 4 KiB in total, sharded round-robin over the N GPUs (strong scaling), one allreduce of the counts
  C4  100 000 files per GPU with Zipf sizes 128 B - 1 MiB (weak scaling; load-balance stress)
  C5  50 000 (old, new) revision pairs in total, dealt size-descending round-robin over the N GPUs (strong scaling):
      line records of both sides (k_scan), Myers edit distance, canonical hunks + changed assertion lines

A step = one pass of the hot path over the rank's batch(es), and for N > 1 the single allreduce of the count table
(overlapped with the next step's scan on a side stream; C5: of the churn totals).
`value`  = source MB/s, inputs resident in HBM, CUDA events on the launching stream, max over ranks.
`e2e`    = same metric through the host C-ABI call path (pinned host arena -> H2D -> kernels -> allreduce -> D2H of
           per-file / per-pair results) inside the timed region.
The reference ships no scanner (SURVEY.md section 0), so the reference arm times the repo's own plain-C restatement
(oracle/, kind "port") on the host cores through a pthread pool (oracle/orc_mt.c): one C call per step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "tosem-2021-replication_b200"))

import numpy as np  # noqa: E402

sys.dont_write_bytecode = True         # the benchmark leaves the tree as the build left it (it may be read-only)
FILE_SIZE = 4096
N_GROUPS = 9
MAX_BATCH_FILES_4K = 500000            # 500 000 x 4 KiB = 2.048e9 B: the largest 4 KiB batch an int32-indexed arena holds
METRIC = "source MB/s scanned (tokenise + line-hash + classify + aggregate)"
CONFIGS = {
    "C2": {"kind": "scan", "law": 0, "per_gpu": 100000, "seed": 0x7053454D0002, "scaling": "weak",
           "what": "100 000 synthetic files x 4 096 B per GPU"},
    "C3": {"kind": "scan", "law": 0, "total": 1000000, "seed": 0x7053454D0003, "scaling": "strong",
           "what": "1 000 000 synthetic files x 4 096 B in total, sharded round-robin over the GPUs"},
    "C4": {"kind": "scan", "law": 1, "per_gpu": 100000, "seed": 0x7053454D0004, "scaling": "weak",
           "what": "100 000 synthetic files per GPU, Zipf sizes 128 B - 1 MiB (pdf ~ x^-1.5)"},
    "C5": {"kind": "diff", "total": 50000, "seed": 0x7053454D0005, "scaling": "strong",
           "what": "50 000 (old, new) revision pairs in total (old ~ Zipf law clamped to 64 KiB, new = old with Poisson(6) line edits), "
                   "dealt size-descending round-robin over the GPUs"},
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="C2", choices=sorted(CONFIGS))
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the workload (smoke runs); 1.0 = the named config")
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = min(steps, 10)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of the last timed step to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    return args


DUMP_MAX_ROWS = 800000                 # per-file / per-pair rows --dump-outputs keeps: <= 8 float64 columns, < 52 MB


def dump_outputs(out_dir, rows, tables):
    """--dump-outputs: every array as out_dir/<name>.npy in float64, which holds these integers exactly (64-bit digests
    come split into 32-bit halves).  rows: per-file or per-pair columns; past DUMP_MAX_ROWS rows a fixed seeded sample of
    them, whose row numbers go to row_index.npy.  tables: arrays written whole."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(next(iter(rows.values())))
    if n > DUMP_MAX_ROWS:
        keep = np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_ROWS, replace=False))
        rows = dict({k: v[keep] for k, v in rows.items()}, row_index=keep)
    for name, a in list(rows.items()) + list(tables.items()):
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a).astype(np.float64))


def config_json(args, n, extra):
    c = CONFIGS[args.config]
    out = {"workload": "%s: %s (seed 0x%X, SURVEY.md section 8d)" % (args.config, c["what"], c["seed"]),
           "sharding": "round-robin by file index, no data-path collective" if c["kind"] == "scan"
           else "pairs sorted by size, dealt to the ranks in alternating direction (equal byte totals), no data-path collective",
           "collective": ("one allreduce(SUM) of the int64 [n_groups+1][128]+4 count table per step, overlapped with the next step's scan"
                          if c["kind"] == "scan" else "one allreduce(SUM) of the 7 churn totals per step") if n > 1 else "none",
           "l2": "input per GPU exceeds the 126 MB L2, no explicit flush"}
    if args.scale != 1.0:
        out["scale"] = args.scale
    out.update(extra)
    return out


# --------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def bind_to_gpu_numa_node(local):
    """Run this rank (and first-touch its pinned arenas) on the host NUMA node its GPU hangs off."""
    try:
        import torch
        p = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        before = os.sched_getaffinity(0)
        cpus &= before
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"node": node, "cpus": len(cpus), "before": sorted(before)}
    except (OSError, ValueError, AttributeError, RuntimeError):
        pass
    return None


# --------------------------------------------------------------------------------------- workloads
def scan_batches(ts, args, rank, n):
    """This rank's batches of the scan configs: list of Corpus."""
    c = CONFIGS[args.config]
    if "per_gpu" in c:
        nf = max(1, int(c["per_gpu"] * args.scale))
        return [ts.gen_corpus(c["seed"], nf, c["law"], FILE_SIZE, first_index=rank, index_stride=n, n_groups=N_GROUPS, pinned=True)], nf * n
    total = max(n, int(c["total"] * args.scale))
    mine = (total - rank + n - 1) // n                     # logical files rank, rank + n, ...
    out, done = [], 0
    while done < mine:
        k = min(MAX_BATCH_FILES_4K, mine - done)
        out.append(ts.gen_corpus(c["seed"], k, c["law"], FILE_SIZE, first_index=rank + done * n, index_stride=n,
                                 n_groups=N_GROUPS, pinned=True))
        done += k
    return out, total


def diff_shard(ts, args, rank, n, pinned=True):
    """This rank's share of the C5 pairs: all pairs sorted by size (descending), dealt round-robin."""
    c = CONFIGS[args.config]
    total = max(n, int(c["total"] * args.scale))
    lo, ln, ext = ts.gen_pair_sizes(c["seed"], total)
    order = np.argsort(-(lo.astype(np.int64) + ln), kind="stable")
    pos = np.arange(total)
    lane = pos % n
    owner = np.where((pos // n) % 2 == 0, lane, n - 1 - lane)      # dealt in alternating direction: equal byte totals per rank
    mine = np.sort(order[owner == rank]).astype(np.int32)
    a, b = ts.gen_pairs(c["seed"], 0, index=mine, sizes=(lo[mine], ln[mine], ext[mine]), pinned=pinned)
    return a, b, total, int(lo.astype(np.int64).sum() + ln.astype(np.int64).sum())


# --------------------------------------------------------------------------------------- CPU arm
def cpu_pool(max_groups=16, numa=None):
    if numa and numa.get("before"):                       # the CPU baseline may use every host core again
        os.sched_setaffinity(0, set(numa["before"]))
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import orc  # the one place bench.py executes oracle/: as the measured CPU baseline
    return orc, orc.MtScanner(0, max_groups=max_groups)


def cpu_rate_scan(mt, corpus, passes):
    t0 = time.perf_counter()
    for _ in range(passes):
        res = mt.scan(corpus.arena, corpus.off, corpus.len, corpus.ext, corpus.grp, corpus.n_groups)
    dt = time.perf_counter() - t0
    return corpus.source_bytes * passes / dt / 1e6, corpus.n_files * passes / dt, dt, int(res["global_counts"].sum())


def cpu_rate_diff(mt, a, b, passes):
    t0 = time.perf_counter()
    for _ in range(passes):
        add, rem, det = mt.diff((a.arena, a.off, a.len, a.ext), (b.arena, b.off, b.len, b.ext))
    dt = time.perf_counter() - t0
    return (a.source_bytes + b.source_bytes) * passes / dt / 1e6, a.n_files * passes / dt, dt, int(add.sum() + rem.sum())


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import tosemscan as ts
    orc, mt = cpu_pool()
    c = CONFIGS[args.config]
    if c["kind"] == "scan":
        # bounded sample of rank 0's shard: at most 100 000 files / ~1.2 GB per step (2 - 6 CPU-seconds)
        batches, total = scan_batches(ts, argparse.Namespace(**{**vars(args), "scale": args.scale * (0.1 if args.config == "C3" else 1.0)}), 0, args.gpus)
        corpus = batches[0]
        unit_bytes, unit_n = corpus.source_bytes, corpus.n_files
        step = lambda: cpu_rate_scan(mt, corpus, 1)
        sample = "%d files, %.1f MB per step (rank 0's shard%s), %d host threads (sched_getaffinity), arena in RAM" % (
            unit_n, unit_bytes / 1e6, ", first 100 000 files" if args.config == "C3" else "", mt.threads)
    else:
        a, b, total, _ = diff_shard(ts, argparse.Namespace(**{**vars(args), "scale": args.scale * 0.2}), 0, 1, pinned=False)
        unit_bytes, unit_n = a.source_bytes + b.source_bytes, a.n_files
        step = lambda: cpu_rate_diff(mt, a, b, 1)
        sample = "%d of 50 000 pairs, %.1f MB of revision text per step, %d host threads (sched_getaffinity)" % (unit_n, unit_bytes / 1e6, mt.threads)
    for _ in range(max(1, min(args.warmup, 2))):
        step()
    dts = [step()[2] for _ in range(args.steps)]
    v = unit_bytes * len(dts) / sum(dts) / 1e6
    threads = mt.threads
    mt.close()
    one = cpu_rate_one_thread(orc, args, ts)
    out = {"impl": "reference", "metric": METRIC, "value": v, "unit": "MB/s", "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": 1e3 * sum(dts) / len(dts), "higher_is_better": True, "scaling": c["scaling"],
           "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config_json(args, args.gpus, {}),
           "files_per_s" if c["kind"] == "scan" else "pairs_per_s": unit_n * len(dts) / sum(dts),
           "cpu_baseline": {"value": v, "unit": "MB/s", "cores": threads, "kind": "port", "sample": sample,
                            "one_thread_MBps": one, "scaling_vs_one_thread": v / one if one else None},
           "e2e": {"value": v, "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "note": "the reference package ships no scanner; this is the repo's plain-C restatement (oracle/) on a pthread pool"}
    print(json.dumps(out))


def cpu_rate_one_thread(orc, args, ts):
    """Single-thread rate of the same oracle on a small slice (what the pool's scaling is judged against)."""
    c = CONFIGS[args.config]
    one = orc.MtScanner(1)
    try:
        if c["kind"] == "scan":
            small = ts.gen_corpus(c["seed"], 4000 if c["law"] == 0 else 1500, c["law"], FILE_SIZE, n_groups=N_GROUPS, pinned=False)
            return cpu_rate_scan(one, small, 2)[0]
        a, b = ts.gen_pairs(c["seed"], 400, pinned=False)
        return cpu_rate_diff(one, a, b, 1)[0]
    finally:
        one.close()


# --------------------------------------------------------------------------------------- GPU arm
def init_dist(n, local):
    import torch
    import torch.distributed as dist
    # keep stdout to the one JSON line: with NCCL_DEBUG=VERSION/INFO set by the caller NCCL prints there,
    # so stdout is pointed at stderr while the communicator comes up (NCCL_DEBUG itself is left alone)
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist.barrier()
        torch.cuda.synchronize()
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)
    return dist


class _Arr:   # __cuda_array_interface__ view of a device buffer of the library, no copy
    def __init__(self, p, m):
        self.__cuda_array_interface__ = {"shape": (m,), "typestr": "<i8", "data": (p, False), "version": 3}


def run_b200(args):
    import torch
    import tosemscan as ts
    n = args.gpus
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != n:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d (launch with torch.distributed.run for N > 1)" % (n, world))
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    numa = bind_to_gpu_numa_node(local)                    # before the pinned arenas are allocated
    dist = init_dist(n, local) if n > 1 else None
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "6650 GB/s (of fallback)"
    env = {"n": n, "rank": rank, "local": local, "dist": dist, "peak": peak, "peak_src": peak_src, "numa": numa}
    if CONFIGS[args.config]["kind"] == "scan":
        bench_scan(args, ts, torch, env)
    else:
        bench_diff(args, ts, torch, env)
    if dist:
        dist.destroy_process_group()


def max_over_ranks(torch, dist, x):
    t = torch.tensor([x], dtype=torch.float64, device="cuda")
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def bench_scan(args, ts, torch, env):
    n, rank, local, dist = env["n"], env["rank"], env["local"], env["dist"]
    batches, total_files = scan_batches(ts, args, rank, n)
    scs = [ts.Scanner(device=local, max_arena_bytes=int(c.off[-1]) + 4096, max_files=c.n_files, max_groups=16) for c in batches]
    stream = torch.cuda.current_stream()
    side = torch.cuda.Stream()
    sp = stream.cuda_stream
    views = []
    for sc, c in zip(scs, batches):
        sc.upload(c, sp)
        sc.scan_resident(0, sp)
        ptr, n64 = sc.device_counts()
        views.append(torch.as_tensor(_Arr(ptr, n64), device=torch.device("cuda", local)))
    stage = [torch.zeros_like(views[0]) for _ in range(2)]   # the table that is allreduced: double-buffered so that the
    done = [torch.cuda.Event() for _ in range(2)]            # allreduce of step i overlaps the scan of step i + 1
    ready = torch.cuda.Event()
    it = [0]

    def step():
        for sc in scs:
            sc.scan_resident(0, sp)
        if n > 1 or len(scs) > 1:
            k = it[0] & 1
            stream.wait_event(done[k])                      # the allreduce that last used this buffer is over
            stage[k].copy_(views[0])
            for v in views[1:]:
                stage[k].add_(v)
            if n > 1:
                ready.record(stream)
                with torch.cuda.stream(side):
                    side.wait_event(ready)
                    dist.all_reduce(stage[k])
                    done[k].record(side)
        it[0] += 1

    def fence():
        stream.wait_stream(side)
        torch.cuda.synchronize()
        if n > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    fence()
    for sc in scs:
        sc.kernel_ms_stats(reset=True)
    sampler = ClockSampler(local) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fence()
    e0.record(stream)
    for _ in range(args.steps):
        step()
    stream.wait_stream(side)                                # the last allreduce belongs to the timed region
    e1.record(stream)
    fence()
    ms = max_over_ranks(torch, dist, e0.elapsed_time(e1))
    stats = [sc.kernel_ms_stats(reset=True) for sc in scs]
    clocks = sampler.stop() if sampler else None
    launches = sum(sc.last_launch_count() for sc in scs) * args.steps
    # sanity: the resident result is the corpus' own (guards against timing a no-op)
    res = [sc.download(0, sp) for sc in scs]
    glob_assert = sum(int(r["global_counts"].sum()) for r in res)
    lines = sum(int(r["totals"][0]) for r in res)
    assert lines > 0 and glob_assert > 0
    if n > 1:                                               # the allreduced table is the sum over the ranks
        k = (it[0] - 1) & 1
        mine = torch.tensor([glob_assert], dtype=torch.int64, device="cuda")
        dist.all_reduce(mine)
        assert int(stage[k][N_GROUPS * 128:(N_GROUPS + 1) * 128].sum().item()) == int(mine.item()), "allreduced counts"
    if args.dump_outputs and rank == 0:                     # this rank's files in batch order, its tables summed over batches
        st = np.concatenate([r["stats"] for r in res])
        tables = {k: sum(r[k] for r in res) for k in ("group_counts", "global_counts", "totals")}
        if n > 1:
            tables["counts_all_ranks"] = stage[(it[0] - 1) & 1].cpu().numpy()
        dump_outputs(args.dump_outputs, {"n_lines": st["n_lines"], "n_assert": st["n_assert"], "n_headers": st["n_headers"],
                                         "n_fixture": st["n_fixture"], "digest_lo": st["digest"] & np.uint64(0xFFFFFFFF),
                                         "digest_hi": st["digest"] >> np.uint64(32)}, tables)
    # ---- e2e through the host C-ABI path
    ke = args.e2e_steps or min(args.steps, 10)
    nf_rank = sum(c.n_files for c in batches)
    h2d = sum(int(c.off[-1]) + 4 * (c.n_files + 1) + 4 * c.n_files + c.n_files + 2 * c.n_files for c in batches)
    d2h = 24 * nf_rank + len(batches) * (8 * (N_GROUPS + 1) * 128 + 64)

    def e2e_step():
        # tsm_scan: index H2D, arena H2D in 32 MiB slabs overlapped with the scan of earlier slabs,
        # classify/aggregate, D2H of the per-file records and count tables; then the allreduce
        outs = [sc.scan(c, 0, sp, reuse=True) for sc, c in zip(scs, batches)]
        if n > 1:
            stage[0].copy_(views[0])
            for v in views[1:]:
                stage[0].add_(v)
            dist.all_reduce(stage[0])
            outs[0]["global_counts_all_ranks"] = stage[0].cpu()
        return outs
    e2e_step()
    fence()
    t0 = time.perf_counter()
    for _ in range(ke):
        e2e_step()
    fence()
    e2e_s = max_over_ranks(torch, dist, time.perf_counter() - t0)
    # what the link gives: the same arena + index as ONE plain copy per batch, no kernels (the ceiling of e2e)
    fence()
    t0 = time.perf_counter()
    for _ in range(3):
        for sc, c in zip(scs, batches):
            sc.upload(c, sp)
    fence()
    h2d_plain_s = (time.perf_counter() - t0) / 3
    if rank != 0:
        for sc in scs:
            sc.close()
        return
    src_rank = sum(c.source_bytes for c in batches)
    src_all = src_rank * n if "per_gpu" in CONFIGS[args.config] else total_files * FILE_SIZE
    alg = [c.algorithmic_bytes for c in batches]
    scan_ms = sum(s[0][1] for s in stats) / max(sum(s[1] for s in stats), 1)          # average k_scan launch
    achieved = (sum(alg) / len(alg)) / (scan_ms * 1e-3) / 1e9 if scan_ms > 0 else 0.0
    traffic, traffic_src = None, None
    try:   # one `ncu --set full` capture of this kernel on this workload (tools/ncu_summary.py --traffic)
        tj = json.load(open(os.path.join(ROOT, "profiles", "k_scan_traffic.json")))
        tj = tj.get(args.config) or (tj if args.config == "C2" and "k_scan" in tj else {})
        if args.scale == 1.0 and tj:
            traffic, traffic_src = tj["k_scan"]["dram_bytes_read"] + tj["k_scan"]["dram_bytes_write"], tj["k_scan"]["source"]
    except (OSError, KeyError, ValueError, TypeError):
        pass
    nscan = max(sum(s[1] for s in stats), 1)
    out = {"metric": METRIC, "value": src_all * args.steps / (ms * 1e-3) / 1e6, "unit": "MB/s", "n_gpus": n,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
           "scaling": CONFIGS[args.config]["scaling"], "vs_baseline": None, "dtype": "u8", "data": "synthetic",
           "config": config_json(args, n, {"files_per_gpu": nf_rank, "global_files": total_files, "file_bytes": FILE_SIZE if CONFIGS[args.config]["law"] == 0 else "zipf",
                                           "n_groups": N_GROUPS, "batches_per_gpu": len(batches),
                                           "numa": {k: v for k, v in env["numa"].items() if k != "before"} if env["numa"] else None}),
           "files_per_s": total_files * args.steps / (ms * 1e-3),
           "roofline": {"bound": "hbm", "kernel": "k_scan", "achieved": achieved, "peak": env["peak"], "unit": "GB/s",
                        "frac": achieved / env["peak"], "traffic": traffic, "traffic_source": traffic_src,
                        "peak_source": env["peak_src"], "algorithmic_bytes_per_launch": sum(alg) / len(alg),
                        "kernel_ms": {"k_plan": sum(s[0][0] for s in stats) / nscan, "k_scan": scan_ms,
                                      "k_classify": sum(s[0][2] for s in stats) / nscan},
                        "scans_timed": nscan},
           "e2e": {"value": src_all * ke / e2e_s / 1e6, "unit": "MB/s", "h2d_bytes_per_step": h2d,
                   "d2h_bytes_per_step": d2h, "steps": ke, "ms_per_step": 1e3 * e2e_s / ke,
                   "path": "tsm_scan(pinned host arena): slab-pipelined H2D + kernels + D2H, then the allreduce",
                   "plain_h2d_copy_of_the_same_bytes_MBps_this_gpu": h2d / h2d_plain_s / 1e6,
                   "fraction_of_plain_copy_rate": (h2d * ke / e2e_s) / (h2d / h2d_plain_s)},
           "gpu_launches": launches, "clocks": clocks,
           "check": {"lines": lines, "assertion_lines": sum(int(r["totals"][1]) for r in res), "classified": glob_assert}}
    if n == 1 and not args.no_cpu_baseline:
        orc, mt = cpu_pool(numa=env["numa"])
        c0 = batches[0]
        passes = max(1, int(round(2.5e9 / max(c0.source_bytes, 1))))      # ~ 10 - 15 CPU-seconds of oracle work
        mb, fps, dt, tot = cpu_rate_scan(mt, c0, passes)
        out["cpu_baseline"] = {"value": mb, "unit": "MB/s", "cores": mt.threads, "kind": "port", "files_per_s": fps,
                               "sample": "%d files (%.0f MB) x %d passes (%.2f s wall), oracle/liborc.so -O2 on a pool of %d threads, arena in RAM"
                                         % (c0.n_files, c0.source_bytes / 1e6, passes, dt, mt.threads)}
        mt.close()
        out["cpu_baseline"]["one_thread_MBps"] = cpu_rate_one_thread(orc, args, ts)
    print(json.dumps(out))
    for sc in scs:
        sc.close()


def bench_diff(args, ts, torch, env):
    n, rank, local, dist = env["n"], env["rank"], env["local"], env["dist"]
    a, b, total_pairs, total_bytes = diff_shard(ts, args, rank, n)
    sc = ts.Scanner(device=local, max_arena_bytes=1 << 20, max_files=16, max_groups=1)
    stream = torch.cuda.current_stream()
    sp = stream.cuda_stream
    sc.diff_upload(a, b, sp)
    tot = torch.zeros(7, dtype=torch.int64, device="cuda")
    ms_acc = np.zeros(3)

    def totals(add, rem, det):
        return np.array([add.sum(), rem.sum()] + [det[f].sum() for f in det.dtype.names], np.int64)

    def step(timed=False):
        add, rem, det = sc.diff_resident(True, sp)
        if timed:
            ms_acc[:] += sc.diff_last_ms()
        if n > 1:
            tot.copy_(torch.from_numpy(totals(add, rem, det)))
            dist.all_reduce(tot)
        return add, rem, det

    def fence():
        torch.cuda.synchronize()
        if n > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    fence()
    sampler = ClockSampler(local) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fence()
    e0.record(stream)
    for _ in range(args.steps):
        add, rem, det = step(True)
    e1.record(stream)
    fence()
    ms = max_over_ranks(torch, dist, e0.elapsed_time(e1))
    clocks = sampler.stop() if sampler else None
    launches = sc.last_launch_count() * args.steps
    # checks: added - removed = change in line count (from the scan's own line records), identical pairs have no churn
    la = sc.line_hashes(a)[0]
    lb = sc.line_hashes(b)[0]
    assert np.array_equal(add - rem, np.diff(lb) - np.diff(la)), "added - removed must equal the change in line count"
    assert int(add.sum() + rem.sum()) > 0
    if args.dump_outputs and rank == 0:                     # this rank's pairs in ascending logical order
        dump_outputs(args.dump_outputs, dict({"added": add, "removed": rem}, **{f: det[f] for f in det.dtype.names}),
                     {"churn_totals_all_ranks": tot.cpu().numpy()} if n > 1 else {})
    ke = args.e2e_steps or min(args.steps, 10)

    def e2e_step():
        out = sc.diff_pairs(a, b, sp, detail=True)          # H2D of both sides + kernels + D2H of the per-pair results
        if n > 1:
            tot.copy_(torch.from_numpy(totals(*out)))
            dist.all_reduce(tot)
            return out, tot.cpu()
        return out
    e2e_step()
    fence()
    t0 = time.perf_counter()
    for _ in range(ke):
        e2e_step()
    fence()
    e2e_s = max_over_ranks(torch, dist, time.perf_counter() - t0)
    if rank != 0:
        sc.close()
        return
    src_rank = a.source_bytes + b.source_bytes
    alg = src_rank + 4 * (a.n_files + 1) * 2
    scan_ms = ms_acc[0] / args.steps                        # both sides: two k_scan launches per step
    achieved = alg / (scan_ms * 1e-3) / 1e9 if scan_ms > 0 else 0.0
    kern_ms = ms_acc / args.steps
    out = {"metric": METRIC, "value": total_bytes * args.steps / (ms * 1e-3) / 1e6, "unit": "MB/s", "n_gpus": n,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
           "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
           "config": config_json(args, n, {"pairs_per_gpu": a.n_files, "global_pairs": total_pairs, "bytes_per_gpu": src_rank,
                                           "global_bytes": total_bytes,
                                           "numa": {k: v for k, v in env["numa"].items() if k != "before"} if env["numa"] else None}),
           "pairs_per_s": total_pairs * args.steps / (ms * 1e-3),
           "roofline": {"bound": "hbm", "kernel": "k_scan (line records of both sides)", "achieved": achieved, "peak": env["peak"],
                        "unit": "GB/s", "frac": achieved / env["peak"], "traffic": None, "peak_source": env["peak_src"],
                        "algorithmic_bytes_per_launch": alg / 2,
                        "kernel_ms": {"k_scan_both_sides": float(kern_ms[0]), "k_diff_small": float(kern_ms[1]), "k_myers_and_trace_of_the_left_over_pairs": float(kern_ms[2])},
                        "lcs_phase": {"note": "compute / latency bound on 8-byte line hashes, reported in pairs/s (SURVEY.md section 8d)",
                                      "pairs_per_s_kernels_only_this_gpu": a.n_files / (float(kern_ms.sum()) * 1e-3) if kern_ms.sum() > 0 else None}},
           "e2e": {"value": total_bytes * ke / e2e_s / 1e6, "unit": "MB/s", "h2d_bytes_per_step": int(a.off[-1]) + int(b.off[-1]) + 18 * a.n_files + 16,
                   "d2h_bytes_per_step": 56 * a.n_files + 16 * (a.n_files + 1), "steps": ke, "ms_per_step": 1e3 * e2e_s / ke,
                   "pairs_per_s": total_pairs * ke / e2e_s,
                   "path": "tsm_diff_pairs_detail(pinned host arenas): H2D of both sides + k_scan x 2 + k_diff_small (+ k_myers, k_myers_trace for the pairs it leaves over) + D2H"},
           "gpu_launches": launches, "clocks": clocks,
           "check": {"added": int(add.sum()), "removed": int(rem.sum()), "hunks": int(det["hunks_add"].sum() + det["hunks_del"].sum() + det["hunks_mod"].sum()),
                     "added_assert": int(det["added_assert"].sum()), "removed_assert": int(det["removed_assert"].sum())}}
    if n == 1 and not args.no_cpu_baseline:
        orc, mt = cpu_pool(numa=env["numa"])
        k = min(a.n_files, 10000)
        sa = ts.pack([a.file_bytes(i) for i in range(k)], a.ext[:k])
        sb = ts.pack([b.file_bytes(i) for i in range(k)], b.ext[:k])
        mb, pps, dt, chk = cpu_rate_diff(mt, sa, sb, 1)
        wadd, wrem, wdet = mt.diff((sa.arena, sa.off, sa.len, sa.ext), (sb.arena, sb.off, sb.len, sb.ext))
        assert np.array_equal(add[:k], wadd) and np.array_equal(rem[:k], wrem) and np.array_equal(det[:k], wdet), "GPU diff differs from the oracle"
        out["check"]["pairs_compared_with_the_oracle"] = k
        out["cpu_baseline"] = {"value": mb, "unit": "MB/s", "cores": mt.threads, "kind": "port", "pairs_per_s": pps,
                               "sample": "first %d pairs of the shard (%.0f MB), oracle diff with hunks on a pool of %d threads (%.2f s wall)"
                                         % (k, (sa.source_bytes + sb.source_bytes) / 1e6, mt.threads, dt)}
        mt.close()
        out["cpu_baseline"]["one_thread_MBps"] = cpu_rate_one_thread(orc, args, ts)
    print(json.dumps(out))
    sc.close()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
