#!/usr/bin/env python
"""bench.py -- split-read DP throughput (GCUPS, tasks/s) of the B200 path, with the reference's
CPU implementation timed beside it.

  python bench.py --gpus N --steps K --warmup W            # our arm (torchrun launches N ranks)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU aligner on host cores

Workload (BASELINE.json configs[2], the split-read metric's own config, per GPU):
dosplitalign-shaped batch of 20 000 candidate clusters x 100 candidate reads = 2.0 M
SplitReadAligner tasks, 100-bp reads against ~340-bp breakpoint window pairs, scoring 2/-1/-2,
minSplitScore 8, minScore = floor(1.8 L).  Weak scaling: every rank aligns its own shard of that
size (work is partitioned by cluster, no collective on the data path).

A "step" = one pass of the hot path over the batch.  `value` times the step with the batch resident
in HBM (first sweep + probe sweep kernels); `e2e` times the C-ABI call with pinned HOST buffers
(H2D copy, pack, both sweeps, D2H, host assembly of the winning rows).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "split_read_dp_gcups"
UNIT = "GCUPS"


def workload_params(args):
    return dict(n_clusters=args.clusters, tasks_per_cluster=args.tasks_per_cluster, L=100, R_lo=320, R_hi=360)


def config_dict(args, n_gpus):
    return {
        "workload": "BASELINE.json configs[2]: dosplitalign split-read DP shard, %d clusters x %d candidate reads "
                    "= %d SplitReadAligner tasks per GPU, L=100, R1,R2 in [320,360], scoring 2/-1/-2, "
                    "minSplitScore 8, minScore floor(1.8L); planted junctions, 1%% substitutions, 0.1%% N"
                    % (args.clusters, args.tasks_per_cluster, args.clusters * args.tasks_per_cluster),
        "tasks_per_gpu": args.clusters * args.tasks_per_cluster,
        "partitioning": "by cluster, %d shard(s), no collective" % n_gpus,
        "l2_policy": "inputs larger than L2 (packed pool + job list + outputs ~ 0.6 GB per step vs 126 MB L2)",
        "seed": args.seed,
    }


# --------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------

class ClockSampler:
    """nvidia-smi sampled every 200 ms during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return out
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            top = sorted(sm)[len(sm) // 2:]  # samples under load = upper half
            out.update(sm_mhz=float(np.median(top)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


# --------------------------------------------------------------------------------------------
# CPU arm: the reference's own aligner (oracle/_ref, compiled from /root/reference) or the C port
# --------------------------------------------------------------------------------------------

def cpu_split_throughput(w, n_tasks, threads):
    """Times SplitReadAligner::Align + GetAlignments on `n_tasks` tasks of the workload with `threads`
    host threads (one aligner object per thread, like one dosplitalign process per core).
    Returns (gcups, tasks_per_s, seconds, kind)."""
    import oracle  # cpu_baseline leg: the one place bench.py may execute oracle/
    kind = "reference" if oracle.have_ref() else "port"
    impl = "ref" if kind == "reference" else "port"
    n_tasks = min(n_tasks, w["n_tasks"])
    bounds = np.linspace(0, n_tasks, threads + 1).astype(int)
    cells = int((w["L"] * ((w["ref_off"][2 * w["task_cluster"][:n_tasks].astype(np.int64) + 2]
                            - w["ref_off"][2 * w["task_cluster"][:n_tasks].astype(np.int64)]))).sum())

    def run(k):
        a, b = bounds[k], bounds[k + 1]
        if b > a:
            oracle.split_align_batch(w["ref_bytes"], w["ref_off"], w["read_bytes"], w["read_off"],
                                     w["task_cluster"][a:b], w["task_read"][a:b], w["min_score"][a:b], impl=impl)

    oracle._lib(impl)
    ths = [threading.Thread(target=run, args=(k,)) for k in range(threads)]
    t0 = time.perf_counter()
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    dt = time.perf_counter() - t0
    return cells / dt / 1e9, n_tasks / dt, dt, kind


def run_reference_arm(args):
    import synth
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = os.cpu_count() or 1
    per_step = args.ref_tasks_per_core * threads
    n_clusters = max(1, min(args.clusters, (per_step * (args.steps + args.warmup)) // args.tasks_per_cluster + 1))
    w = synth.split_workload(args.seed, n_clusters, args.tasks_per_cluster, 100, 320, 360)
    sub = dict(w)
    times, gc, tps, kind = [], [], [], "port"
    for s in range(args.warmup + args.steps):
        a = (s * per_step) % max(1, w["n_tasks"] - per_step + 1)
        for key in ("task_cluster", "task_read", "min_score"):
            sub[key] = w[key][a:a + per_step]
        sub["n_tasks"] = len(sub["task_cluster"])
        g, t, dt, kind = cpu_split_throughput(sub, per_step, threads)
        if s >= args.warmup:
            times.append(dt)
            gc.append(g)
            tps.append(t)
    value = float(np.mean(gc))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": float(np.mean(times) * 1e3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": config_dict(args, args.gpus), "tasks_per_s": float(np.mean(tps)),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind,
                         "sample": "%d tasks per step (%d per host thread) of the same workload" % (per_step, args.ref_tasks_per_core)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    args.out.write(json.dumps(line) + "\n")
    args.out.flush()
    return 0


# --------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------

def exception_words(seq_bytes, seq_off, reverse=False):
    """16-base words of a CSR byte table that hold a byte other than A, C, G, T (the pack kernel writes a 16-byte raw
    copy only for those).  `reverse`: words of the reversed copies."""
    off = np.asarray(seq_off, dtype=np.int64)
    lens = off[1:] - off[:-1]
    if lens.size == 0 or int(lens.max()) == 0:
        return 0
    bad = ~np.isin(np.asarray(seq_bytes), np.frombuffer(b"ACGT", dtype=np.uint8))
    if not bad.any():
        return 0
    idx = np.nonzero(bad)[0]
    seq = np.searchsorted(off, idx, side="right") - 1
    pos = idx - off[seq]
    if reverse:
        pos = lens[seq] - 1 - pos
    words_before = np.concatenate([[0], np.cumsum((lens + 15) // 16)])
    return int(np.unique(words_before[seq] + pos // 16).size)


def pinned(arr):
    import torch
    t = torch.empty(arr.shape, dtype=getattr(torch, str(arr.dtype)), pin_memory=True)
    out = t.numpy()
    out[...] = arr
    return out, t


def measure_stress(ctx, stream, args):
    """BASELINE.json configs[4] as SURVEY 8(d) writes it (synth.STRESS): 250-bp reads, 8 % substitutions, 2 % indels,
    1 % N, 5 % poly-A-tail reads, lowercase runs in 1 % of the windows, cluster sizes Zipf(1.2) (the heaviest clusters
    hold most candidates), windows 700-860 bp.  A sample of the tasks is compared with the oracle (checker only)."""
    import torch
    import defuse_b200 as d
    import synth
    w = synth.split_workload(5, 4000, 50, **synth.STRESS)
    refs = d.SeqTable(w["ref_bytes"], w["ref_off"])
    reads = d.SeqTable(w["read_bytes"], w["read_off"])
    al = d.SplitReadAligner(2, -1, -2, False, 8, ctx=ctx)
    plan = al.plan(refs, reads, w["task_cluster"], w["task_read"], w["min_score"])
    plan.set_timing(True)
    for _ in range(3):
        plan.run()
    plan.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps = 5
    torch.cuda.synchronize()
    e0.record(stream)
    for _ in range(steps):
        plan.run()
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    plan.sync()
    st = plan.stats()
    res = plan.fetch(copy=False)
    n_hit = int((res.best > 0).sum())
    # sampled parity (the oracle is the checker here, never the thing measured): every 500th task plus the tasks with
    # the most winning rows, i.e. the tie-heavy ones
    import oracle
    rows_per_task = np.bincount(res.rows["task"], minlength=w["n_tasks"]) if len(res.rows) else np.zeros(w["n_tasks"], int)
    pick = np.unique(np.concatenate([np.arange(0, w["n_tasks"], 500), np.argsort(rows_per_task)[-40:]])).astype(np.int64)
    cnt, want = oracle.split_align_batch(w["ref_bytes"], w["ref_off"], w["read_bytes"], w["read_off"], w["task_cluster"][pick],
                                         w["task_read"][pick], w["min_score"][pick])
    pos = np.concatenate([[0], np.cumsum(cnt)])
    for k, t in enumerate(pick):
        got = res.alignments(int(t))
        assert got.shape == (cnt[k], 7) and (got == want[pos[k]:pos[k + 1]]).all(), "stress task %d differs from the oracle" % t
    plan.close()
    return {"workload": "%d SplitReadAligner tasks, L=250, R 700-860, Zipf(1.2) cluster sizes, 8%% sub, 2%% indels, 1%% N, "
                        "5%% poly-A tails, lowercase runs, poly-A window ends" % w["n_tasks"],
            "gcups": w["cells"] / (ms * 1e-3) / 1e9, "ms_per_step": ms, "sweep_ms": st["ms_sweep"], "probe_ms": st["ms_probe"],
            "tasks_with_split": n_hit, "tasks_per_s": w["n_tasks"] / (ms * 1e-3), "events": int(st["events"]),
            "parity_sample": {"tasks": int(len(pick)), "alignments": int(cnt.sum()), "max_alignments_of_a_task": int(cnt.max()),
                              "checker": "oracle port", "mismatches": 0}}


def measure_local(ctx, stream, args, R=2001, L=100, n_refs=10000, n_tasks=None, own_window=False):
    """BASELINE.json configs[1]: localalign, 1 M 100-bp reads against 10 k references of 2001 bp, 10/-5/-5; and
    configs[3]: matealign-shaped, 150-bp reads against searchlength+1 = 1001-bp windows (reported beside the
    headline; same timing rules)."""
    import torch
    import defuse_b200 as d
    import synth
    w = synth.local_workload(2, n_refs, n_tasks or args.local_tasks, R, L, own_window=own_window)
    refs = d.SeqTable(w["ref_bytes"], w["ref_off"])
    seqs = d.SeqTable(w["seq_bytes"], w["seq_off"])
    al = d.SimpleAligner(10, -5, -5, ctx=ctx)
    plan = al.plan(refs, seqs, w["task_ref"], w["task_seq"])
    for _ in range(3):
        plan.run()
    plan.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps = 5
    torch.cuda.synchronize()
    e0.record(stream)
    for _ in range(steps):
        plan.run()
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    st = plan.stats()
    plan.close()
    # end to end through dfb_simple_align_batch (chunks pipelined: upload + pack of chunk k+1 under the sweep of chunk k),
    # from pageable host arrays as a tool would hand them over, and from pinned ones
    def e2e(refs_t, seqs_t, tr, ts):
        best = None
        first = None
        for _ in range(3):
            t0 = time.perf_counter()
            got = al.align_batch(refs_t, seqs_t, tr, ts)
            dt = (time.perf_counter() - t0) * 1e3
            first = dt if first is None else first
            best = dt if best is None else min(best, dt)
        return best, first, got
    e2e_ms, first_ms, got_pageable = e2e(refs, seqs, w["task_ref"], w["task_seq"])
    keep, hp = [], {}
    for k in ("ref_bytes", "ref_off", "seq_bytes", "seq_off", "task_ref", "task_seq"):
        hp[k], t = pinned(w[k])
        keep.append(t)
    pin_ms, _, got_pinned = e2e(d.SeqTable(hp["ref_bytes"], hp["ref_off"]), d.SeqTable(hp["seq_bytes"], hp["seq_off"]), hp["task_ref"], hp["task_seq"])
    assert np.array_equal(got_pageable, got_pinned)
    return {"workload": "%d SimpleAligner tasks, R=%d, L=%d, 10/-5/-5%s" % (
                w["n_tasks"], R, L, ", one window per task in task order (what matealign submits)" if own_window else
                ", %d references named in any order" % n_refs), "gcups": w["cells"] / (ms * 1e-3) / 1e9,
            "ms_per_step": ms, "reads_per_s": w["n_tasks"] / (ms * 1e-3), "e2e_gcups": w["cells"] / (e2e_ms * 1e-3) / 1e9,
            "e2e_ms": e2e_ms, "e2e_pinned_gcups": w["cells"] / (pin_ms * 1e-3) / 1e9, "e2e_pinned_ms": pin_ms,
            "first_call_ms": first_ms, "kernel_launches": int(st["kernel_launches"]),
            "h2d_bytes": int(w["ref_bytes"].nbytes + w["seq_bytes"].nbytes + w["task_ref"].nbytes + w["task_seq"].nbytes)}


def measure_sharded(aligner, args, rank, world, barrier):
    """The path as the north star partitions it: ONE fixed batch (strong scaling), its tasks dealt to the ranks by
    candidate cluster (defuse_b200.sharding, LPT on DP cells, window table replicated), every rank aligns its shard
    through the C ABI from pinned host buffers, rank 0 gathers and merges the rows back into the batch's task order --
    the reference's emission order (SplitAlignment.cpp:271-301; fan-out + ordered merge: defuse_run.pl:518-533).
    The digest of the merged result does not depend on the number of shards: compare it across the N of a scaling run."""
    import hashlib
    import torch
    import torch.distributed as dist
    import defuse_b200 as d
    import synth
    from defuse_b200 import sharding
    n_clusters, per = args.shard_clusters, args.tasks_per_cluster
    w = synth.split_workload(args.seed + 77, n_clusters, per, 100, 320, 360)   # the same batch on every rank
    n, L = w["n_tasks"], w["L"]
    tc64 = w["task_cluster"].astype(np.int64)
    cost = L * (w["ref_off"][2 * tc64 + 2] - w["ref_off"][2 * tc64])
    shards, _ = sharding.shard_tasks(w["task_cluster"], cost, n_clusters, world)
    mine = shards[rank]
    reads2d = w["read_bytes"].reshape(n, L)
    keep, host = [], {}
    for k, a in (("ref_bytes", w["ref_bytes"]), ("ref_off", w["ref_off"]),
                 ("read_bytes", np.ascontiguousarray(reads2d[mine]).reshape(-1)),
                 ("read_off", np.arange(len(mine) + 1, dtype=np.int64) * L),
                 ("task_cluster", w["task_cluster"][mine]), ("task_read", np.arange(len(mine), dtype=np.int32)),
                 ("min_score", w["min_score"][mine])):
        host[k], t = pinned(a)
        keep.append(t)
    refs = d.SeqTable(host["ref_bytes"], host["ref_off"])
    reads = d.SeqTable(host["read_bytes"], host["read_off"])
    times = []
    res = None
    for rep in range(3):   # first one warms the pools up
        barrier()
        t0 = time.perf_counter()
        res = aligner.align_batch(refs, reads, host["task_cluster"], host["task_read"], host["min_score"], copy=False)
        torch.cuda.synchronize()
        times.append((time.perf_counter() - t0) * 1e3)
    align_ms = min(times[1:])
    # gather on rank 0: best per task, rows (task renumbered to the batch's numbering), columns
    if world > 1:
        # (the first collective of a process sets the communicator's channels up: not part of the merge)
        warm = torch.zeros(1, dtype=torch.uint8, device="cuda")
        dist.gather(warm, [torch.empty_like(warm) for _ in range(world)] if rank == 0 else None, dst=0)
        dist.all_gather([torch.zeros(1, dtype=torch.int64, device="cuda") for _ in range(world)], torch.zeros(1, dtype=torch.int64, device="cuda"))
        torch.cuda.synchronize()
        barrier()
    t0 = time.perf_counter()
    rows = np.array(res.rows, copy=True)
    rows["task"] = mine[rows["task"]]
    cols = np.asarray(res.cols)
    parts = {"idx": mine.astype(np.int64), "best": np.asarray(res.best, dtype=np.int32), "rows": rows.view(np.uint8).reshape(-1), "cols": cols.astype(np.int32)}
    gathered = {}
    for key, a in parts.items():
        a = np.ascontiguousarray(a)
        if world == 1:
            gathered[key] = [a]
            continue
        size = torch.tensor([a.nbytes], dtype=torch.int64, device="cuda")
        sizes = [torch.zeros(1, dtype=torch.int64, device="cuda") for _ in range(world)]
        dist.all_gather(sizes, size)
        sizes = [int(x.item()) for x in sizes]
        buf = torch.zeros(max(max(sizes), 1), dtype=torch.uint8, device="cuda")
        buf[:a.nbytes] = torch.from_numpy(a.view(np.uint8).reshape(-1)).cuda()
        out = [torch.empty_like(buf) for _ in range(world)] if rank == 0 else None
        dist.gather(buf, out, dst=0)
        if rank == 0:
            gathered[key] = [out[r][:sizes[r]].cpu().numpy().view(a.dtype) for r in range(world)]
    result = None
    if rank == 0:
        best = sharding.merge_by_task(n, zip(gathered["idx"], gathered["best"]))
        all_rows = [g.view(rows.dtype) for g in gathered["rows"]]
        col_base = np.concatenate([[0], np.cumsum([len(c) for c in gathered["cols"]])])
        for r, g in enumerate(all_rows):
            g["col_begin"] += col_base[r]
        all_cols = np.concatenate(gathered["cols"])
        merged = sharding.merge_rows_by_task(n, all_rows)   # counting placement; rows of a task stay in their (ascending split row) order
        merge_ms = (time.perf_counter() - t0) * 1e3   # gather + merge into task order; the digest below is bookkeeping
        h = hashlib.sha1()
        h.update(best.tobytes())
        for f in ("task", "read_split", "score1", "score2", "n1", "n2"):
            h.update(np.ascontiguousarray(merged[f]).tobytes())
        # columns in merged row order
        width = merged["n1"].astype(np.int64) + merged["n2"]
        starts = np.repeat(merged["col_begin"].astype(np.int64), width)
        within = np.arange(int(width.sum())) - np.repeat(np.concatenate([[0], np.cumsum(width)[:-1]]), width)
        h.update(np.ascontiguousarray(all_cols[starts + within]).tobytes())
        loads = np.array([cost[g].sum() for g in gathered["idx"]], dtype=np.float64)
        result = {"digest": h.hexdigest(), "merge_ms": merge_ms, "rows": int(len(merged)), "tasks": int(n),
                  "load_imbalance": float(loads.max() / loads.mean())}
    t = torch.tensor([align_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        result.update({"workload": "one batch of %d clusters x %d candidate reads = %d tasks in total, dealt to %d rank(s) by cluster"
                                   % (n_clusters, per, n, world),
                       "scaling": "strong", "align_ms_max_over_ranks": float(t[0]),
                       "e2e_gcups": w["cells"] / (float(t[0]) * 1e-3) / 1e9,
                       "e2e_gcups_incl_merge": w["cells"] / ((float(t[0]) + result["merge_ms"]) * 1e-3) / 1e9})
    return result


def measure_tool(args):
    """BASELINE's second unit, input read pairs per second of process wall time (SURVEY 8d (ii)): the dosplitalign drop-in on
    generated files of one (scaled-down) fastq split, and the compiled reference tool on a stated sample of the same
    generator; outputs compared byte for byte on the sample."""
    from synth import files
    import oracle  # baseline leg: the compiled reference tool
    bin_dir = os.path.join(ROOT, "defuse_b200", "bin")
    ours = os.path.join(bin_dir, "dosplitalign")
    if not os.path.exists(ours):
        return {"unavailable": "defuse_b200/bin/dosplitalign not built"}
    out = {"read_pairs": args.tool_clusters * 100, "clusters": args.tool_clusters}
    with tempfile.TemporaryDirectory() as d:
        a = files.make_split_dataset(os.path.join(d, "s"), seed=3, n_clusters=args.tool_clusters, pairs_per_cluster=100,
                                     n_chrom=8, genes_per_chrom=40)
        res = os.path.join(d, "s", "ours.tmp")
        runs = []
        for _ in range(2):
            t0 = time.perf_counter()
            p = subprocess.run([ours] + a + ["-a", res], capture_output=True)
            runs.append(time.perf_counter() - t0)
            if p.returncode != 0:
                return {"unavailable": "dosplitalign failed: " + p.stderr.decode()[-300:]}
        out.update({"seconds": min(runs), "runs_s": runs, "read_pairs_per_s": out["read_pairs"] / min(runs),
                    "records": sum(1 for _ in open(res))})
        ref = oracle.ref_tool("ref_dosplitalign")
        if ref:
            sub_c = max(20, args.tool_clusters // 50)
            sa = files.make_split_dataset(os.path.join(d, "r"), seed=3, n_clusters=sub_c, pairs_per_cluster=100, n_chrom=8,
                                          genes_per_chrom=40)
            rres, ores = os.path.join(d, "r", "ref.tmp"), os.path.join(d, "r", "ours.tmp")
            t0 = time.perf_counter()
            subprocess.run([ref] + sa + ["-a", rres], check=True, capture_output=True)
            ref_s = time.perf_counter() - t0
            subprocess.run([ours] + sa + ["-a", ores], check=True, capture_output=True)
            out["reference_tool"] = {"read_pairs": sub_c * 100, "seconds": ref_s, "read_pairs_per_s": sub_c * 100 / ref_s,
                                     "cores": 1, "identical_output": open(rres, "rb").read() == open(ores, "rb").read(),
                                     "sample": "%d of the %d clusters of the same generator" % (sub_c, args.tool_clusters)}
    return out


DUMP_TASKS = 1 << 19
DUMP_MAX_BYTES = 60 << 20   # (the .npy headers and the 64 MB limit stay clear of it)


def dump_outputs(out_dir, res, seed):
    """Writes what the resident plan's last step returned as out_dir/<name>.npy, so that two builds can be compared
    output for output on the same inputs.  For a fixed, seeded sample of up to DUMP_TASKS tasks (all of them in a
    smaller batch): the best total per task and the task's winning rows, with each row's column list in row order (the
    library may lay its column pool out differently from build to build).  The sample is the longest prefix of a seeded
    permutation of the tasks that fits in DUMP_MAX_BYTES.  Values are integers, written as float32 when every one of
    them is below 2**24 (exact there), else as float64."""
    n = len(res.best)
    rows, cols = res.rows, res.cols
    width = rows["n1"].astype(np.int64) + rows["n2"]
    fields = ("task", "read_split", "score1", "score2", "n1", "n2")
    big = max([n] + [int(np.abs(a).max(initial=0)) for a in [res.best, cols] + [rows[f] for f in fields]])
    dtype = np.float32 if big < 1 << 24 else np.float64
    per_task = 2 + len(fields) * np.bincount(rows["task"], minlength=n) + np.bincount(rows["task"], weights=width, minlength=n)
    order = np.random.default_rng(seed).permutation(n)[:DUMP_TASKS]
    k = int(np.searchsorted(np.cumsum(per_task[order] * np.dtype(dtype).itemsize), DUMP_MAX_BYTES, side="right"))
    tasks = np.sort(order[:k])
    picked = np.zeros(n, dtype=bool)
    picked[tasks] = True
    sel = picked[rows["task"]]
    rows, width = rows[sel], width[sel]
    first = np.cumsum(width) - width
    out = {"tasks": tasks, "best": res.best[tasks],
           "row_cols": cols[np.repeat(rows["col_begin"], width) + np.arange(int(width.sum())) - np.repeat(first, width)]}
    for f in fields:
        out["row_" + f] = rows[f]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=dtype))


def run_ours(args):
    import torch
    import torch.distributed as dist
    import defuse_b200 as d
    import synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the DP path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    if world > 1:
        # one process per GPU on one host: the ranks share its cores (the context's worker pool defaults to 16 threads)
        local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
        # (measured on 8 GPUs / 32 host threads: 4 workers per rank 79.9 ms per e2e step, 8 -> 67.3, 12 -> 63.6)
        os.environ.setdefault("DFB_HOST_THREADS", str(max(4, min(16, 3 * (os.cpu_count() or 16) // max(1, local_world)))))
    ctx = d.Context(local_rank)
    # a side stream: the legacy default stream has handle 0, which the C ABI reads as "use your own"
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    info = ctx.device_info()

    # every rank owns a different shard of clusters (seed offset), same size: weak scaling
    w = synth.split_workload(args.seed + 1000 * rank, **workload_params(args))
    keep = []
    host = {}
    for k in ("ref_bytes", "ref_off", "read_bytes", "read_off", "task_cluster", "task_read", "min_score"):
        host[k], t = pinned(w[k])
        keep.append(t)
    refs = d.SeqTable(host["ref_bytes"], host["ref_off"])
    reads = d.SeqTable(host["read_bytes"], host["read_off"])
    aligner = d.SplitReadAligner(2, -1, -2, False, 8, ctx=ctx)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- resident: inputs already packed in HBM ----
    # (a small plan first: the first launch of a kernel pays for loading it, which would be charged to the pack timing)
    warm = aligner.plan(refs, reads, host["task_cluster"][:1024], host["task_read"][:1024], host["min_score"][:1024])
    warm.run()
    warm.sync()
    del warm
    plan = aligner.plan(refs, reads, host["task_cluster"], host["task_read"], host["min_score"])
    plan.set_timing(True)
    for _ in range(max(args.warmup, 3)):
        plan.run()
    plan.sync()
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sweep_ms, probe_ms = [], []
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        plan.run()
    e1.record(stream)
    barrier()
    ms_total = e0.elapsed_time(e1)
    plan.sync()
    st = plan.stats()
    sweep_ms.append(st["ms_sweep"])
    probe_ms.append(st["ms_probe"])
    res = plan.fetch(copy=False)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, args.seed)
    st = plan.stats()
    n_hit = int((res.best > 0).sum())
    n_rows = len(res.rows)
    best_resident = res.best.copy()
    del res
    plan.close()   # the end-to-end part below runs without the resident batch: its device memory is its own

    # ---- end to end through the C ABI with host buffers ----
    e2e_ms = []
    e2e_steps = max(1, min(args.steps, args.e2e_steps or args.steps))
    import resource
    cpu_ms = []
    E2E_WARM = 2   # (the first calls grow the device pool and the pinned result buffers)
    for s in range(E2E_WARM + e2e_steps):
        if s == E2E_WARM:
            ctx.memory_info(reset=True)
        barrier()
        ru0 = resource.getrusage(resource.RUSAGE_SELF)
        t0 = time.perf_counter()
        r2 = aligner.align_batch(refs, reads, host["task_cluster"], host["task_read"], host["min_score"], copy=False)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) * 1e3
        ru1 = resource.getrusage(resource.RUSAGE_SELF)
        if s >= E2E_WARM:
            e2e_ms.append(dt)
            cpu_ms.append(((ru1.ru_utime - ru0.ru_utime) + (ru1.ru_stime - ru0.ru_stime)) * 1e3)  # all threads of this rank
    assert (r2.best == best_resident).all() and len(r2.rows) == n_rows
    e2e_mem = ctx.memory_info()
    e2e_st = ctx.split_result_stats()   # what the one-call path itself copied (every window once per batch)
    clocks = sampler.stop() if rank == 0 else None
    sharded = None if args.no_sharded else measure_sharded(aligner, args, rank, world, barrier)

    t = torch.tensor([ms_total, float(np.mean(e2e_ms))], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, e2e_mean = float(t[0]), float(t[1])
    cells_rank = st["cells"]
    tc = torch.tensor([float(cells_rank), float(st["n_tasks"])], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tc, op=dist.ReduceOp.SUM)
    cells_all, tasks_all = float(tc[0]), float(tc[1])
    ms_step = ms_total / args.steps

    if rank == 0:
        value = cells_all / (ms_step * 1e-3) / 1e9
        # roofline of the dominant kernel (first sweep, dp_fast_kernel<8,13,SPLIT>): integer/DPX issue bound.
        rate, _ = ctx.microbench_issue_rate(0, 2000)   # VIADDMNMX.S16x2 warp-instructions/s, measured now
        p_int_lane = rate * 32.0
        peak_gcups = p_int_lane * 2.0 / 6.0 / 1e9      # SURVEY 8(d): 6 INT issues per s16x2 vector of 2 cells
        k_ms = float(np.mean(sweep_ms))
        achieved = cells_rank / (k_ms * 1e-3) / 1e9
        traffic, ncu = None, {}
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tpath):
            try:
                ncu = json.load(open(tpath))
                per_task = ncu.get("dp_fast_kernel_split_dram_bytes_per_task")
                traffic = per_task * st["n_tasks"] if per_task else None  # ncu capture scaled to this launch's task count
            except Exception:
                traffic = None
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        # what the pack kernels move: every raw byte read once per stored copy (window 2 of a cluster reversed, reads
        # forward and reversed), 8 B {codes, mask} written per 16-base word, 16 B raw copy only for words with an exception
        n_exc = (exception_words(w["ref_bytes"], w["ref_off"]) + exception_words(w["read_bytes"], w["read_off"])
                 + exception_words(w["read_bytes"], w["read_off"], reverse=True))
        pack_bytes = st["raw_bytes"] + st["packed_bytes"] + 16 * n_exc
        pack_gbs = pack_bytes / (st["ms_pack"] * 1e-3) / 1e9 if st["ms_pack"] > 0 else None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "s16x2 (int16 pairs, DPX)", "data": "synthetic", "config": config_dict(args, world),
            "tasks_per_s": tasks_all / (ms_step * 1e-3),
            "e2e": {"value": cells_all / (e2e_mean * 1e-3) / 1e9, "unit": UNIT,
                    "tasks_per_s": tasks_all / (e2e_mean * 1e-3), "ms_per_step": e2e_mean,
                    "ms_per_step_min_rank0": float(np.min(e2e_ms)), "ms_per_step_median_rank0": float(np.median(e2e_ms)),
                    "h2d_bytes_per_step": int(e2e_st["h2d_bytes"]),
                    "d2h_bytes_per_step": int(e2e_st["d2h_bytes"]), "steps": e2e_steps,
                    "host_cpu_ms_per_step": float(np.mean(cpu_ms)),   # user+sys of all threads of rank 0 during the call
                    "host_cpus": os.cpu_count(), "host_threads_cap": os.environ.get("DFB_HOST_THREADS"),
                    "device_pool_used_high_bytes": e2e_mem[2], "device_pool_reserved_bytes": e2e_mem[0],
                    "device_pool_note": "high-water mark of the bytes in use during the timed e2e steps (chunk buffers are recycled inside a batch)"},
            "gpu_launches": int(st["kernel_launches"]) * args.steps,
            "roofline": {"bound": "int_issue", "kernel": "dp_fast_kernel<8,13,SPLIT> (first sweep)",
                         "achieved": achieved, "peak": peak_gcups, "unit": UNIT, "frac": achieved / peak_gcups,
                         "traffic": traffic,
                         "peak_source": "measured now: VIADDMNMX.S16x2 issue rate %.1f Gwarp-instr/s x 32 lanes x 2 cells / 6 issues"
                                        % (rate / 1e9),
                         "kernel_ms": k_ms, "probe_sweep_ms": float(np.mean(probe_ms)),
                         "step_frac_incl_probe": value / world / peak_gcups,
                         # the survey's 6-issue definition is generous: the steady-state loop needs 3.5 ALU-pipe issues per
                         # register pair of cells (indicator, two maxima, half a three-input sink), so this is the fraction
                         # of the kernel's own floor -- the number that says how much is left
                         "frac_own_minimum": achieved / (p_int_lane * 2.0 / 3.5 / 1e9),
                         "own_minimum_gcups": p_int_lane * 2.0 / 3.5 / 1e9,
                         "ncu_alu_pipe_pct": ncu.get("dp_fast_kernel_split_alu_pipe_pct"),
                         "ncu_capture": ncu.get("capture")},
            "roofline_staging": {"bound": "hbm", "kernel": "pack_kernel", "achieved": pack_gbs, "peak": hbm_peak,
                                 "unit": "GB/s", "frac": (pack_gbs / hbm_peak) if pack_gbs else None,
                                 "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s",
                                 "bytes": pack_bytes, "ms": st["ms_pack"], "exception_words": n_exc,
                                 "bytes_are": "raw bytes read once per stored copy + 8 B per 16-base word + 16 B per exception word"},
            "clocks": clocks,
            "results": {"tasks_with_split": n_hit, "winning_rows": n_rows, "probe_jobs": int(st["probe_jobs"]),
                        "events": int(st["events"])},
            "device": info["name"],
        }
        if sharded:
            line["sharded_merge"] = sharded
        if world == 1 and not args.no_secondary:
            line["tool_dosplitalign"] = measure_tool(args)
        if world == 1 and not args.no_secondary:
            line["secondary"] = {"localalign_config2": measure_local(ctx, stream, args),
                                 "matealign_config4": measure_local(ctx, stream, args, R=1001, L=150, own_window=True,
                                                                    n_tasks=args.local_tasks // 2),
                                 "stress_config5": measure_stress(ctx, stream, args)}
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            n = args.cpu_baseline_tasks_per_core * threads   # ~10 s of CPU work on the box's host cores
            g, tps, dt, kind = cpu_split_throughput(w, n, threads)
            line["cpu_baseline"] = {"value": g, "unit": UNIT, "cores": threads, "kind": kind, "tasks_per_s": tps,
                                    "seconds": dt,
                                    "sample": "first %d tasks of the same workload (%d per host thread)" % (min(n, w["n_tasks"]), args.cpu_baseline_tasks_per_core)}
            # BASELINE.md 3: also one process on one core (the reference tools are single-threaded)
            g1, tps1, dt1, _ = cpu_split_throughput(w, max(1, args.cpu_baseline_tasks_per_core // 3), 1)
            line["cpu_baseline"]["one_core"] = {"value": g1, "unit": UNIT, "cores": 1, "tasks_per_s": tps1, "seconds": dt1,
                                                "sample": "first %d tasks of the same workload" % max(1, args.cpu_baseline_tasks_per_core // 3)}
        args.out.write(json.dumps(line) + "\n")
        args.out.flush()
    if world > 1:
        dist.destroy_process_group()
    return 0


def _claim_stdout():
    """Everything libraries print to fd 1 (e.g. NCCL's version banner) goes to stderr; the one JSON line is written
    to the real stdout through the returned file object."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--clusters", type=int, default=20000)
    ap.add_argument("--tasks-per-cluster", type=int, default=100)
    ap.add_argument("--seed", type=int, default=3)
    ap.add_argument("--e2e-steps", type=int, default=0)                        # 0: as many as --steps
    ap.add_argument("--ref-tasks-per-core", type=int, default=2000)            # reference arm: tasks per thread per step
    ap.add_argument("--cpu-baseline-tasks-per-core", type=int, default=14000)  # cpu_baseline leg of our arm (one sample)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--local-tasks", type=int, default=1000000)
    ap.add_argument("--no-sharded", action="store_true")
    ap.add_argument("--shard-clusters", type=int, default=8000)                # sharded_merge leg: clusters of the ONE batch all ranks share
    ap.add_argument("--tool-clusters", type=int, default=2000)                 # tool leg: clusters (x 100 read pairs) of the generated split
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step (a seeded sample of rank 0's tasks) to DIR/<name>.npy, 64 MB at most")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.out = _claim_stdout()
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
