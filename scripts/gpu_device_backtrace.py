"""DeviceSplitResult.backtrace() (dfb_split_backtrace_device) per workload: records, runs (consecutive records of one
task), pieces, filled box cells against the cells of both full matrices, pairs out, the time of the backtrace
call next to align_device and records() of the same batch, peak pool memory of the backtrace call, a sweep of the run
cap, and what a caller had before it -- to_host() plus SplitReadAligner.backtrace_batch on host arrays -- timed once.

    python scripts/gpu_device_backtrace.py --out profiles/<tag>_device_backtrace.json [--runs 7] [--skip-before]

Workloads: the bench split shape (synth.split_workload(1, 20000, 100), 2 M tasks) and STRESS (synth.STRESS, 4 000
clusters x 50 = 200 k tasks) with all their records, and the poly-A batch (24 x a 200-base poly-A read against
700-base poly-A windows, min score 360) with every 64th of its 11.2 M records, which keeps runs of 7 300 records.
Times are CUDA events on torch's current stream around one call each, after one warm-up call.  Peak pool memory is the
pool's used high-water mark during the backtrace calls above what was in use before them, with no backtrace result held
at that point (every call frees the previous one on entry, so each call's peak is the same).  The run-cap sweep sets
DFB_BT_RUN_CAP and times three calls per value."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SMEM_BYTES = 96 << 10   # DFB_BT_SMEM_BYTES


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def workloads():
    import synth
    w = synth.split_workload(1, 20000, 100)
    yield "bench_2m", w["ref_bytes"], w["ref_off"], w["read_bytes"], w["read_off"], w["task_cluster"], w["task_read"], w["min_score"], 1
    w = synth.split_workload(5, 4000, 50, **synth.STRESS)
    yield "stress_200k", w["ref_bytes"], w["ref_off"], w["read_bytes"], w["read_off"], w["task_cluster"], w["task_read"], w["min_score"], 1
    polyA = np.frombuffer(b"A" * 700, np.uint8)
    read = np.frombuffer(b"A" * 200, np.uint8)
    yield ("poly_a_every_64th", np.concatenate([polyA, polyA]), np.array([0, 700, 1400], np.int64), np.tile(read, 24),
           np.arange(25, dtype=np.int64) * 200, np.zeros(24, np.int32), np.arange(24, dtype=np.int32), np.full(24, 360, np.int32), 64)


def timed(fn, runs):
    import torch
    out, ms = None, []
    for _ in range(runs):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return out, ms


def geometry(rec, refs, reads, tc, tr, cap):
    """runs, pieces at run cap `cap`, the cells the pieces' boxes fill, the full-matrix cells, and the pieces whose
    boxes exceed shared memory -- the rule of bt_records_kernel / bt_box_kernel restated"""
    n = len(rec)
    task = rec[:, 0].astype(np.int64)
    c, q = tc[task].astype(np.int64), tr[task].astype(np.int64)
    L = reads.off[q + 1] - reads.off[q]
    R1 = refs.off[2 * c + 1] - refs.off[2 * c]
    R2 = refs.off[2 * c + 2] - refs.off[2 * c + 1]
    a, i1, i2 = rec[:, 3].astype(np.int64), rec[:, 1].astype(np.int64), R2 - rec[:, 2] - 1
    k = np.arange(n)
    run_head = np.ones(n, bool)
    run_head[1:] = task[1:] != task[:-1]
    head = run_head | (k % cap == 0)
    starts = np.nonzero(head)[0]
    J1, I1 = np.maximum.reduceat(a, starts), np.maximum.reduceat(i1, starts)
    J2, I2 = np.maximum.reduceat(L - a, starts), np.maximum.reduceat(i2, starts)
    words = J1 * ((I1 + 16) >> 4) + J2 * ((I2 + 16) >> 4) + I1 + I2 + 2
    return {"runs": int(run_head.sum()), "records_per_run": n / max(int(run_head.sum()), 1), "pieces": int(len(starts)),
            "filled_cells": int((J1 * I1 + J2 * I2).sum()), "full_matrix_cells": int((L * (R1 + R2)).sum()),
            "pieces_on_global_arena": int((words * 4 > SMEM_BYTES).sum()), "largest_piece_bytes": int(words.max(initial=0) * 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--runs", type=int, default=7)
    ap.add_argument("--caps", default="64,256,1024")
    ap.add_argument("--skip-before", action="store_true")
    args = ap.parse_args()
    import torch
    import defuse_b200 as d
    ctx = d.default_context(0)
    result = {"card": card(), "device": ctx.device_info(), "runs": args.runs, "workloads": {}}
    print(result["card"], flush=True)
    for name, rb, ro, sb, so, tc, tr, ms, every in workloads():
        refs, reads = d.SeqTable(rb, ro), d.SeqTable(sb, so)
        dr, dq = d.DeviceSeqTable.from_host(refs, "cuda:0"), d.DeviceSeqTable.from_host(reads, "cuda:0")
        tct, trt, mst = (torch.from_numpy(np.ascontiguousarray(x, np.int32)).cuda() for x in (tc, tr, ms))
        al = d.SplitReadAligner(ctx=ctx)
        al.align_device(dr, dq, tct, trt, mst)  # warm-up
        res, align_ms = timed(lambda: al.align_device(dr, dq, tct, trt, mst), args.runs)
        res.records()  # warm-up
        rec_all, records_ms = timed(res.records, args.runs)
        rec = rec_all[::every].contiguous()
        del rec_all
        res.backtrace(rec)  # warm-up
        # the base holds no backtrace result: an empty call releases the warm-up's (each call frees the last on entry)
        res.backtrace(rec[:0])
        ctx.memory_info(reset=True)
        pool_base = ctx.memory_info()[2]
        (off, pairs), bt_ms = timed(lambda: res.backtrace(rec), args.runs)
        pool_high = ctx.memory_info()[2]
        rec_h = rec.cpu().numpy()
        entry = {"tasks": int(len(tc)), "records": int(len(rec_h)), "record_stride": every, "pairs_out": int(pairs.shape[0]),
                 "backtrace_ms": bt_ms, "align_device_ms": align_ms, "records_ms": records_ms,
                 "backtrace_ms_min_max": [min(bt_ms), max(bt_ms)], "align_device_ms_min_max": [min(align_ms), max(align_ms)],
                 "records_ms_min_max": [min(records_ms), max(records_ms)],
                 "pool_used_before_bytes": int(pool_base), "backtrace_pool_peak_bytes": int(pool_high - pool_base)}
        entry.update(geometry(rec_h, refs, reads, np.asarray(tc), np.asarray(tr), 256))
        sweep = {}
        for cap in [int(x) for x in args.caps.split(",") if x]:
            os.environ["DFB_BT_RUN_CAP"] = str(cap)
            res.backtrace(rec)
            _, ms_cap = timed(lambda: res.backtrace(rec), 3)
            g = geometry(rec_h, refs, reads, np.asarray(tc), np.asarray(tr), cap)
            sweep[str(cap)] = {"ms": ms_cap, "pieces": g["pieces"], "filled_cells": g["filled_cells"]}
        os.environ.pop("DFB_BT_RUN_CAP", None)
        entry["run_cap_sweep"] = sweep
        if not args.skip_before:
            off_h, pairs_h = off.cpu().numpy(), pairs.cpu().numpy()
            del off, pairs
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            host = res.to_host()
            r = rec.cpu().numpy()
            tch, trh = np.asarray(tc, np.int32), np.asarray(tr, np.int32)
            w_off, w_pairs = al.backtrace_batch(refs, reads, tch[r[:, 0]], trh[r[:, 0]], r[:, 1], r[:, 2], r[:, 3])
            entry["before_to_host_plus_backtrace_batch_ms"] = (time.perf_counter() - t0) * 1e3
            entry["outputs_equal_backtrace_batch"] = bool(off_h.tobytes() == w_off.tobytes() and pairs_h.tobytes() == w_pairs.tobytes())
            del host, w_off, w_pairs
        result["workloads"][name] = entry
        print(name, json.dumps({k: v for k, v in entry.items() if not isinstance(v, list)}), flush=True)
        del res, rec
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
