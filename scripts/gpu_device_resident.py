"""Host one-call form from pinned arrays against the device-resident form from CUDA tensors, per shape: time per call,
PCIe bytes, peak pool memory; plus bench.py's e2e of a parent build (DFB_PARENT_LIB) against this build, alternating.

    python scripts/gpu_device_resident.py --tag r05a [--runs 5] [--parent-lib build/parent/libdefuse_b200.so]

Writes profiles/<tag>_device_resident.json.  Shapes: the bench split shape (20 000 clusters x 100 reads), the
localalign shape (BASELINE config 2: 1 M 100-bp reads, 10 k references of 2001 bp), the matealign shape (config 4:
150-bp reads, one 1001-bp window per task) and the stress shape (synth.STRESS, 4 000 clusters x 50).  The arms
alternate inside every shape after one warm-up call each; both results are compared byte for byte."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def pinned(arr):
    import torch
    t = torch.empty(arr.shape, dtype=getattr(torch, str(arr.dtype)), pin_memory=True)
    out = t.numpy()
    out[...] = arr
    return out, t


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def measure(ctx, kind, w, runs):
    import torch
    import defuse_b200 as d
    keep, h = [], {}
    for k, v in w.items():
        if isinstance(v, np.ndarray):
            h[k], t = pinned(v)
            keep.append(t)
    ta, tb = ("ref_bytes", "ref_off"), ("read_bytes", "read_off") if kind == "split" else ("seq_bytes", "seq_off")
    refs, seqs = d.SeqTable(h[ta[0]], h[ta[1]]), d.SeqTable(h[tb[0]], h[tb[1]])
    drefs, dseqs = d.DeviceSeqTable.from_host(refs, "cuda:0"), d.DeviceSeqTable.from_host(seqs, "cuda:0")
    names = ("task_cluster", "task_read", "min_score") if kind == "split" else ("task_ref", "task_seq")
    host_tasks = [h[n] for n in names]
    dev_tasks = [torch.from_numpy(np.ascontiguousarray(w[n], np.int32)).cuda() for n in names]
    if kind == "split":
        al = d.SplitReadAligner(ctx=ctx)
        host_call = lambda: al.align_batch(refs, seqs, *host_tasks)   # (copies: the device call that follows frees the views)
        dev_call = lambda: al.align_device(drefs, dseqs, *dev_tasks)
    else:
        al = d.SimpleAligner(10, -5, -5, ctx=ctx)
        out_host = np.empty(len(host_tasks[0]), np.int32)
        host_call = lambda: al.align_batch(refs, seqs, *host_tasks, out=out_host)
        dev_call = lambda: al.align_device(drefs, dseqs, *dev_tasks)
    arms = {"host_pinned": host_call, "device": dev_call}
    res = {a: {"ms": [], "pool_used_high_bytes": 0} for a in arms}
    last = {}
    for a, fn in arms.items():  # warm-up
        last[a] = fn()
    torch.cuda.synchronize()
    for _ in range(runs):
        for a, fn in arms.items():
            ctx.memory_info(reset=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            last[a] = fn()
            torch.cuda.synchronize()
            res[a]["ms"].append((time.perf_counter() - t0) * 1e3)
            res[a]["pool_used_high_bytes"] = max(res[a]["pool_used_high_bytes"], ctx.memory_info()[2])
            if kind == "split":
                st = ctx.split_result_stats()
                res[a]["h2d_bytes"], res[a]["d2h_bytes"] = int(st["h2d_bytes"]), int(st["d2h_bytes"])
    if kind == "split":
        hr, dr = last["host_pinned"], last["device"].to_host()
        same = np.array_equal(hr.best, dr.best) and hr.rows.tobytes() == dr.rows.tobytes() and np.array_equal(hr.cols, dr.cols)
    else:
        same = np.array_equal(last["host_pinned"], last["device"].cpu().numpy())
        # the simple one-call forms keep no statistics (the library has no accessor for them): the host arm's figure is
        # what it must move at least (tables and task arrays up, scores down), the device arm's is not counted
        n = len(host_tasks[0])
        res["host_pinned"]["h2d_bytes_lower_bound"] = int(sum(h[k].nbytes for k in (ta + tb)) + 8 * n)
        res["host_pinned"]["d2h_bytes_lower_bound"] = 4 * n
        res["device"]["pcie_bytes"] = None
        res["pcie_note"] = "not counted for the simple form: no statistics accessor; bounds computed from array sizes"
    for a in arms:
        ms = res[a]["ms"]
        res[a].update({"min_ms": min(ms), "median_ms": float(np.median(ms))})
    res["identical_results"] = bool(same)
    res["n_tasks"] = int(len(host_tasks[0]))
    return res


def bench_ab(parent_lib, runs):
    out = {"parent": [], "this": []}
    for _ in range(runs):
        for arm in ("parent", "this"):
            env = dict(os.environ)
            if arm == "parent":
                env["DFB_LIB_PATH"] = parent_lib
            p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "5", "--warmup", "2",
                                "--no-secondary", "--no-sharded", "--no-cpu-baseline"], capture_output=True, text=True, env=env, cwd=ROOT)
            line = [l for l in p.stdout.splitlines() if l.startswith("{")]
            if p.returncode or not line:
                out[arm].append({"error": p.stderr[-2000:]})
                continue
            r = json.loads(line[-1])
            out[arm].append({"value": r["value"], "e2e_ms_per_step": r["e2e"]["ms_per_step"],
                             "e2e_ms_min": r["e2e"]["ms_per_step_min_rank0"], "e2e_gcups": r["e2e"]["value"]})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tag", required=True)
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--bench-runs", type=int, default=3)
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    args = ap.parse_args()
    import defuse_b200 as d
    import synth
    ctx = d.default_context(0)
    result = {"card_before": card(), "device": ctx.device_info(), "runs_per_arm": args.runs, "shapes": {}}
    shapes = {
        "split_bench_20000x100": ("split", lambda: synth.split_workload(3, 20000, 100)),
        "localalign_config2": ("simple", lambda: synth.local_workload(2, 10000, 1000000, 2001, 100)),
        "matealign_config4": ("simple", lambda: synth.local_workload(2, 10000, 1000000, 1001, 150, own_window=True)),
        "stress_config5": ("split", lambda: synth.split_workload(5, 4000, 50, **synth.STRESS)),
    }
    for name, (kind, make) in shapes.items():
        result["shapes"][name] = measure(ctx, kind, make(), args.runs)
        print(name, json.dumps({a: result["shapes"][name][a]["median_ms"] for a in ("host_pinned", "device")}), flush=True)
    if args.parent_lib:
        result["bench_e2e_ab"] = bench_ab(args.parent_lib, args.bench_runs)
    result["card_after"] = card()
    os.makedirs(args.out_dir, exist_ok=True)
    path = os.path.join(args.out_dir, "%s_device_resident.json" % args.tag)
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
