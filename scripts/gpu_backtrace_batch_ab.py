"""SplitReadAligner.backtrace_batch (dfb_split_backtrace_batch) of a parent build against this build: time per call on
the workloads below, the splitseq tool's wall clock, byte equality of every output between the two, and the peak pool
memory of the backtrace calls.

    python scripts/gpu_backtrace_batch_ab.py --parent-lib build/parent/libdefuse_b200.so --out profiles/<tag>.json [--rounds 3]

Each round runs one process per build, the two in alternating order; a process loads its build (DFB_LIB_PATH for the
parent), reads the card's name, power limit and SM clock, warms every workload up with one call, then times `calls`
calls of each with a host clock (the call ends in a stream synchronise) and the splitseq tool three times.  Workloads:
  splitseq_20k / splitseq_200  the shape splitseq passes: synth.split_workload (100-base reads, 320-360-base windows),
                               the first alignment of each task that has one (what a predalign record names), 20 000 of
                               them and 200 (where per-call latency dominates)
  generic_scoring              the same shape under (1, -1, 1, False, 3)
  stress                       synth.STRESS (250-base reads), the first alignment of each task
  bench_200k_all_records       every record of a 200 k-task batch of the bench shape
The splitseq tool runs on a files.make_split_dataset chain (dosplitalign -> sort -> evalsplitalign, built once with this
build) at 6x the size of test_splitseq_vs_reference_tool's first case, over both the predicted and the full sorted
alignments; each build's splitseq binary runs beside a copy of that build's library."""
import argparse
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
THIS_LIB = os.path.join(ROOT, "defuse_b200", "libdefuse_b200.so")
BIN = os.path.join(ROOT, "defuse_b200", "bin")
DATASET = dict(seed=61, n_clusters=360, pairs_per_cluster=50)   # 6x test_splitseq_vs_reference_tool's first case


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def workloads():
    import synth
    s = synth.split_workload(21, 1200, 40)
    yield "splitseq_20k", s, (2, -1, -2, False, 8), True, 20000, 20
    yield "splitseq_200", s, (2, -1, -2, False, 8), True, 200, 200
    yield "generic_scoring", synth.split_workload(22, 1200, 40, match=1), (1, -1, 1, False, 3), True, 20000, 20
    yield "stress", synth.split_workload(5, 1000, 50, **synth.STRESS), (2, -1, -2, False, 8), True, None, 10
    yield "bench_200k_all_records", synth.split_workload(9, 2000, 100), (2, -1, -2, False, 8), False, None, 5


def alignments(ctx, w, params, first_only, limit):
    """the alignments a workload backtraces, as backtrace_batch's arguments: GetAlignments' records of the batch, or the
    first of each task"""
    import torch
    import defuse_b200 as d
    refs, reads = d.SeqTable(w["ref_bytes"], w["ref_off"]), d.SeqTable(w["read_bytes"], w["read_off"])
    al = d.SplitReadAligner(*params, ctx=ctx)
    tc, tr = np.asarray(w["task_cluster"], np.int32), np.asarray(w["task_read"], np.int32)
    dev = [torch.from_numpy(np.ascontiguousarray(x, np.int32)).cuda() for x in (tc, tr, w["min_score"])]
    rec = al.align_device(d.DeviceSeqTable.from_host(refs, "cuda:0"), d.DeviceSeqTable.from_host(reads, "cuda:0"), *dev).records()
    rec = rec.cpu().numpy()
    if first_only:
        rec = rec[np.unique(rec[:, 0], return_index=True)[1]]
    rec = rec[:limit]
    t = rec[:, 0]
    return al, (refs, reads, tc[t], tr[t], rec[:, 1], rec[:, 2], rec[:, 3])


def splitseq_runs(tooldir, data, runs=3):
    out = {}
    common = json.load(open(os.path.join(data, "common.json")))
    for name in ("ours.predalign", "sorted.alignments"):
        cmd = [os.path.join(tooldir, "bin", "splitseq")] + common + ["-a", os.path.join(data, name)]
        ms, digest = [], None
        for _ in range(runs):
            t0 = time.perf_counter()
            p = subprocess.run(cmd, capture_output=True, check=True)
            ms.append((time.perf_counter() - t0) * 1e3)
            digest = hashlib.sha256(p.stdout).hexdigest()
        out[name] = {"ms": ms, "stdout_sha256": digest, "stdout_bytes": len(p.stdout)}
    return out


def worker(arm, data):
    import defuse_b200 as d
    ctx = d.default_context(0)
    result = {"arm": arm, "lib": d.LIB_PATH, "card": card(), "workloads": {}}
    for name, w, params, first_only, limit, calls in workloads():
        al, args = alignments(ctx, w, params, first_only, limit)
        off, pairs = al.backtrace_batch(*args)   # warm-up
        ctx.memory_info(reset=True)
        ms = []
        for _ in range(calls):
            t0 = time.perf_counter()
            off, pairs = al.backtrace_batch(*args)
            ms.append((time.perf_counter() - t0) * 1e3)
        result["workloads"][name] = {
            "alignments": int(len(args[2])), "pairs": int(len(pairs)), "ms": ms, "median_ms": float(np.median(ms)),
            "min_ms": float(min(ms)), "pool_used_high_bytes": int(ctx.memory_info()[2]),
            "output_sha256": hashlib.sha256(off.tobytes() + pairs.tobytes()).hexdigest()}
    result["splitseq_tool"] = splitseq_runs(os.path.join(data, "tools", arm), data)
    result["card_after"] = card()
    print(json.dumps(result))


def make_data(data, parent_lib):
    """the splitseq chain's files (made with this build's tools), and one tool directory per build: splitseq finds the
    library beside its bin/ directory"""
    from synth import files
    args = files.make_split_dataset(data, **DATASET)
    raw, srt = os.path.join(data, "raw.alignments"), os.path.join(data, "sorted.alignments")
    subprocess.run([os.path.join(BIN, "dosplitalign")] + args + ["-a", raw], check=True, capture_output=True)
    files.sort_alignments(raw, srt)
    common, ev = files.downstream_args(args, data)
    names = {k: os.path.join(data, "ours.%s" % k) for k in ("seq", "break", "predalign")}
    subprocess.run([os.path.join(BIN, "evalsplitalign")] + ev + ["-q", names["seq"], "-b", names["break"], "-p", names["predalign"]],
                   check=True, capture_output=True)
    json.dump(common + ["-p", files.write_read_index(data)], open(os.path.join(data, "common.json"), "w"))
    for arm, lib in (("parent", parent_lib), ("this", THIS_LIB)):
        os.makedirs(os.path.join(data, "tools", arm, "bin"))
        shutil.copy(os.path.join(BIN, "splitseq"), os.path.join(data, "tools", arm, "bin", "splitseq"))
        shutil.copy(lib, os.path.join(data, "tools", arm, "libdefuse_b200.so"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", required=True)
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--worker", choices=("parent", "this"))
    ap.add_argument("--data")
    args = ap.parse_args()
    if args.worker:
        return worker(args.worker, args.data)
    parent_lib = os.path.abspath(args.parent_lib)
    runs = {"parent": [], "this": []}
    with tempfile.TemporaryDirectory() as data:
        make_data(data, parent_lib)
        for r in range(args.rounds):
            for arm in (("parent", "this") if r % 2 == 0 else ("this", "parent")):
                env = dict(os.environ)
                env.pop("DFB_LIB_PATH", None)
                if arm == "parent":
                    env["DFB_LIB_PATH"] = parent_lib
                p = subprocess.run([sys.executable, os.path.abspath(__file__), "--parent-lib", parent_lib, "--out", args.out,
                                    "--worker", arm, "--data", data], capture_output=True, text=True, env=env, cwd=ROOT)
                if p.returncode:
                    sys.exit("%s worker failed:\n%s" % (arm, p.stderr[-4000:]))
                runs[arm].append(json.loads(p.stdout.strip().splitlines()[-1]))
                print("round", r, arm, json.dumps({k: v["median_ms"] for k, v in runs[arm][-1]["workloads"].items()}), flush=True)
    summary = {}
    for name in runs["this"][0]["workloads"]:
        row = {}
        for arm in ("parent", "this"):
            med = [x["workloads"][name]["median_ms"] for x in runs[arm]]
            row[arm] = {"median_ms_per_round": med, "median_ms": float(np.median(med)), "spread_ms": max(med) - min(med),
                        "pool_used_high_bytes": max(x["workloads"][name]["pool_used_high_bytes"] for x in runs[arm])}
        row["alignments"] = runs["this"][0]["workloads"][name]["alignments"]
        row["pairs"] = runs["this"][0]["workloads"][name]["pairs"]
        row["outputs_equal"] = len({x["workloads"][name]["output_sha256"] for a in runs for x in runs[a]}) == 1
        summary[name] = row
    for name in runs["this"][0]["splitseq_tool"]:
        row = {}
        for arm in ("parent", "this"):
            med = [float(np.median(x["splitseq_tool"][name]["ms"])) for x in runs[arm]]
            row[arm] = {"median_ms_per_round": med, "median_ms": float(np.median(med)), "spread_ms": max(med) - min(med)}
        row["stdout_equal"] = len({x["splitseq_tool"][name]["stdout_sha256"] for a in runs for x in runs[a]}) == 1
        row["stdout_bytes"] = runs["this"][0]["splitseq_tool"][name]["stdout_bytes"]
        summary["splitseq_tool:" + name] = row
    result = {"card": runs["this"][0]["card"], "dataset": DATASET, "rounds": args.rounds, "summary": summary, "runs": runs}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: {a: v[a]["median_ms"] for a in ("parent", "this")} for k, v in summary.items()}, indent=1))


if __name__ == "__main__":
    main()
