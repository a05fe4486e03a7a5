"""DeviceSplitResult.records() (dfb_split_records_device) per workload: rows, raw pairs, records, the share of rows in
multi-row tasks, the time of the records call next to align_device of the same batch, peak pool memory of the records
call, and what a caller had before it -- to_host() plus the numpy rule of tests/test_device_records.py -- timed once.

    python scripts/gpu_device_records.py --out profiles/<tag>_device_records.json [--runs 7] [--skip-before]

Workloads: the bench split shape (synth.split_workload(.., 20000, 100), 2 M tasks), STRESS (synth.STRESS, 4 000
clusters x 50) and the poly-A batch (24 x a 200-base poly-A read against 700-base poly-A windows, min score 360).
Peak pool memory is the pool's used high-water mark during the records calls above what was in use before them.
Times are CUDA events on torch's current stream around one call each, after one warm-up call; records are checked
byte for byte against the numpy rule."""
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


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def workloads():
    import synth
    w = synth.split_workload(1, 20000, 100)
    yield "bench_2m", w["ref_bytes"], w["ref_off"], w["read_bytes"], w["read_off"], w["task_cluster"], w["task_read"], w["min_score"]
    w = synth.split_workload(5, 4000, 50, **synth.STRESS)
    yield "stress", w["ref_bytes"], w["ref_off"], w["read_bytes"], w["read_off"], w["task_cluster"], w["task_read"], w["min_score"]
    polyA = np.frombuffer(b"A" * 700, np.uint8)
    read = np.frombuffer(b"A" * 200, np.uint8)
    yield ("poly_a", np.concatenate([polyA, polyA]), np.array([0, 700, 1400], np.int64), np.tile(read, 24),
           np.arange(25, dtype=np.int64) * 200, np.zeros(24, np.int32), np.arange(24, dtype=np.int32), np.full(24, 360, np.int32))


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--runs", type=int, default=7)
    ap.add_argument("--skip-before", action="store_true")
    args = ap.parse_args()
    import torch
    import defuse_b200 as d
    from test_device_records import rule_records
    ctx = d.default_context(0)
    result = {"card": card(), "device": ctx.device_info(), "runs": args.runs, "workloads": {}}
    for name, rb, ro, sb, so, tc, tr, ms in workloads():
        refs, reads = d.SeqTable(rb, ro), d.SeqTable(sb, so)
        dr, dq = d.DeviceSeqTable.from_host(refs, "cuda:0"), d.DeviceSeqTable.from_host(reads, "cuda:0")
        tct, trt, mst = (torch.from_numpy(np.ascontiguousarray(x, np.int32)).cuda() for x in (tc, tr, ms))
        al = d.SplitReadAligner(ctx=ctx)
        al.align_device(dr, dq, tct, trt, mst)  # warm-up
        res, align_ms = timed(lambda: al.align_device(dr, dq, tct, trt, mst), args.runs)
        res.records()  # warm-up
        # the pool's used high-water mark restarts from what is in use now (the context's last split result, ...)
        ctx.memory_info(reset=True)
        pool_base = ctx.memory_info()[2]
        rec, rec_ms = timed(res.records, args.runs)
        pool_high = ctx.memory_info()[2]
        task = res.task.cpu().numpy()
        n1, n2 = res.n1.cpu().numpy().astype(np.int64), res.n2.cpu().numpy().astype(np.int64)
        rows_per_task = np.bincount(task, minlength=len(tc)) if len(task) else np.zeros(len(tc), np.int64)
        multi_rows = int(rows_per_task[rows_per_task > 1].sum())
        entry = {
            "tasks": int(len(tc)), "rows": int(len(task)), "cols": int(res.cols.numel()), "raw_pairs": int((n1 * n2).sum()),
            "records": int(rec.shape[0]), "rows_in_multi_row_tasks": multi_rows,
            "share_rows_in_multi_row_tasks": multi_rows / max(len(task), 1), "max_rows_per_task": int(rows_per_task.max(initial=0)),
            "records_ms": rec_ms, "align_device_ms": align_ms,
            "records_ms_median": float(np.median(rec_ms)), "align_device_ms_median": float(np.median(align_ms)),
            "pool_used_before_bytes": int(pool_base), "records_pool_peak_bytes": int(pool_high - pool_base),
        }
        if not args.skip_before:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            want = rule_records(res.to_host())
            entry["before_to_host_plus_numpy_rule_ms"] = (time.perf_counter() - t0) * 1e3
            entry["records_equal_numpy_rule"] = bool(rec.cpu().numpy().tobytes() == want.tobytes())
        result["workloads"][name] = entry
        print(name, json.dumps({k: v for k, v in entry.items() if not isinstance(v, list)}), flush=True)
        del res, rec
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
