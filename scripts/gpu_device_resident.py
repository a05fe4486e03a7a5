"""Host one-call form from pinned arrays against the device-resident form from CUDA tensors, per shape: time per call,
PCIe bytes, peak pool memory; plus bench.py's e2e of a parent build (DFB_PARENT_LIB) against this build, alternating.

    python scripts/gpu_device_resident.py --tag r05a [--runs 5] [--parent-lib build/parent/libdefuse_b200.so]

Writes profiles/<tag>_device_resident.json.  Shapes: the bench split shape (20 000 clusters x 100 reads), the
localalign shape (BASELINE config 2: 1 M 100-bp reads, 10 k references of 2001 bp), the matealign shape (config 4:
150-bp reads, one 1001-bp window per task) and the stress shape (synth.STRESS, 4 000 clusters x 50).  The arms
alternate inside every shape after one warm-up call each; both results are compared byte for byte.

    python scripts/gpu_device_resident.py --tag r06 --host-ab --parent-lib build/parent/libdefuse_b200.so [--rounds 3]

Writes profiles/<tag>_host_form_ab.json instead: the host one-call form (SplitReadAligner.align_batch, pinned arrays) of
the parent build against this build, one process per build in alternating order per round.  A process reads the card's
name, power limit and SM clock, warms every workload up with one call and times `calls` calls of each with a host clock
(the call ends in a synchronise); it hashes best, rows and columns, which must be equal across both builds, and reads
the peak pool memory.  Workloads: the bench e2e batch (2 M tasks) with DFB_HOST_BUILD=1 and with DFB_DEVICE_BUILD=1,
the 200 k-task bench shape, STRESS, the poly-A batch of tests/test_device_resident.py (one call form and pipelined) and
a 20 k-task batch below DFB_PIPELINE_MIN_TASKS; the device-resident form (align_device + to_host) on the bench e2e batch,
which shares the chunk loop and the collection; then the dosplitalign tool, each build's binary beside its library: one
warm-up run and six timed ones of the whole process, whose wall clock includes CUDA start-up (1-4 s on these boxes,
DESIGN.md section 7), so that leg only shows a difference larger than the start-up's spread."""
import argparse
import hashlib
import json
import shutil
import tempfile
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


TOOL_DATASET = dict(seed=62, n_clusters=2000, pairs_per_cluster=50)


def host_workloads():
    """(name, workload, env, calls)"""
    import synth
    e2e = synth.split_workload(3, 20000, 100)
    yield "e2e_2M_host_build", e2e, {"DFB_HOST_BUILD": "1"}, 5
    yield "e2e_2M_device_build", e2e, {"DFB_DEVICE_BUILD": "1"}, 5
    yield "bench_200k", synth.split_workload(9, 2000, 100), {}, 10
    yield "stress", synth.split_workload(5, 4000, 50, **synth.STRESS), {}, 10
    poly = {"ref_bytes": np.frombuffer(b"A" * 1400, np.uint8), "ref_off": np.array([0, 700, 1400], np.int64),
            "read_bytes": np.frombuffer(b"A" * 200 * 24, np.uint8), "read_off": np.arange(25, dtype=np.int64) * 200,
            "task_cluster": np.zeros(24, np.int32), "task_read": np.arange(24, dtype=np.int32), "min_score": np.full(24, 360, np.int32)}
    yield "poly_a", poly, {}, 5
    yield "poly_a_pipelined", poly, {"DFB_PIPELINE_MIN_TASKS": "16"}, 5
    yield "small_20k", synth.split_workload(4, 200, 100), {}, 20
    yield "device_form_e2e_2M", e2e, {}, 5


def host_worker(arm, data):
    import defuse_b200 as d
    ctx = d.default_context(0)
    out = {"arm": arm, "lib": os.path.relpath(d.LIB_PATH, ROOT), "card": card(), "workloads": {}}
    for name, w, env, calls in host_workloads():
        h, keep = {}, []
        for k, v in w.items():
            h[k], t = pinned(np.ascontiguousarray(v))
            keep.append(t)
        refs, reads = d.SeqTable(h["ref_bytes"], h["ref_off"]), d.SeqTable(h["read_bytes"], h["read_off"])
        al = d.SplitReadAligner(ctx=ctx)
        os.environ.update(env)
        call = lambda: al.align_batch(refs, reads, h["task_cluster"], h["task_read"], h["min_score"])
        if name.startswith("device_form"):
            import torch
            drefs, dreads = d.DeviceSeqTable.from_host(refs, "cuda:0"), d.DeviceSeqTable.from_host(reads, "cuda:0")
            dt = [torch.from_numpy(h[k]).cuda() for k in ("task_cluster", "task_read", "min_score")]

            def call():
                r = al.align_device(drefs, dreads, *dt)
                torch.cuda.synchronize()
                return r
        r = call()  # warm-up
        ctx.memory_info(reset=True)
        ms = []
        for _ in range(calls):
            t0 = time.perf_counter()
            r = call()
            ms.append((time.perf_counter() - t0) * 1e3)
        for k in env:
            del os.environ[k]
        st = ctx.split_result_stats()
        if name.startswith("device_form"):
            r = r.to_host()
        out["workloads"][name] = {
            "n_tasks": int(len(h["task_read"])), "rows": int(len(r.rows)), "cols": int(len(r.cols)), "ms": ms,
            "median_ms": float(np.median(ms)), "min_ms": float(min(ms)), "max_ms": float(max(ms)),
            "pool_used_high_bytes": int(ctx.memory_info()[2]), "d2h_bytes": int(st["d2h_bytes"]), "h2d_bytes": int(st["h2d_bytes"]),
            "output_sha256": hashlib.sha256(r.best.tobytes() + r.rows.tobytes() + r.cols.tobytes()).hexdigest()}
    common = json.load(open(os.path.join(data, "args.json")))
    ms, digest = [], None
    for run in range(7):  # (the first is the warm-up)
        outp = os.path.join(data, "out_%s.alignments" % arm)
        t0 = time.perf_counter()
        subprocess.run([os.path.join(data, "tools", arm, "bin", "dosplitalign")] + common + ["-a", outp], check=True, capture_output=True)
        if run:
            ms.append((time.perf_counter() - t0) * 1e3)
        digest = hashlib.sha256(open(outp, "rb").read()).hexdigest()
    out["workloads"]["dosplitalign_tool"] = {"ms": ms, "median_ms": float(np.median(ms)), "min_ms": float(min(ms)), "max_ms": float(max(ms)),
                                             "output_sha256": digest}
    out["card_after"] = card()
    print(json.dumps(out))


def host_ab(parent_lib, rounds, out_path):
    from synth import files
    this_lib = os.path.join(ROOT, "defuse_b200", "libdefuse_b200.so")
    bin_dir = os.path.join(ROOT, "defuse_b200", "bin")
    runs = {"parent": [], "this": []}
    with tempfile.TemporaryDirectory() as data:
        json.dump(files.make_split_dataset(data, **TOOL_DATASET), open(os.path.join(data, "args.json"), "w"))
        for arm, lib in (("parent", parent_lib), ("this", this_lib)):
            os.makedirs(os.path.join(data, "tools", arm, "bin"))
            shutil.copy(os.path.join(bin_dir, "dosplitalign"), os.path.join(data, "tools", arm, "bin", "dosplitalign"))
            shutil.copy(lib, os.path.join(data, "tools", arm, "libdefuse_b200.so"))
        for r in range(rounds):
            for arm in (("parent", "this") if r % 2 == 0 else ("this", "parent")):
                env = dict(os.environ)
                env.pop("DFB_LIB_PATH", None)
                if arm == "parent":
                    env["DFB_LIB_PATH"] = parent_lib
                p = subprocess.run([sys.executable, os.path.abspath(__file__), "--tag", "worker", "--host-worker", arm, "--data", data],
                                   capture_output=True, text=True, env=env, cwd=ROOT)
                if p.returncode:
                    sys.exit("%s worker failed:\n%s" % (arm, p.stderr[-4000:]))
                runs[arm].append(json.loads(p.stdout.strip().splitlines()[-1]))
                print("round", r, arm, json.dumps({k: v["median_ms"] for k, v in runs[arm][-1]["workloads"].items()}), flush=True)
    summary = {}
    for name in runs["this"][0]["workloads"]:
        row = {}
        for arm in ("parent", "this"):
            ws = [x["workloads"][name] for x in runs[arm]]
            med = [x["median_ms"] for x in ws]
            row[arm] = {"median_ms_per_round": med, "median_ms": float(np.median(med)),
                        "range_ms": [min(x["min_ms"] for x in ws), max(x["max_ms"] for x in ws)]}
            for k in ("pool_used_high_bytes", "d2h_bytes", "h2d_bytes"):
                if k in ws[0]:
                    row[arm][k] = max(x[k] for x in ws)
        row["outputs_equal"] = len({x["workloads"][name]["output_sha256"] for a in runs for x in runs[a]}) == 1
        summary[name] = row
    result = {"card": runs["this"][0]["card"], "card_after": runs["this"][-1]["card_after"], "rounds": rounds,
              "tool_dataset": TOOL_DATASET, "summary": summary, "runs": runs}
    with open(out_path, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: {a: v[a]["median_ms"] for a in ("parent", "this")} for k, v in summary.items()}, indent=1))
    print("wrote", out_path)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tag", required=True)
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--bench-runs", type=int, default=3)
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--host-ab", action="store_true")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--host-worker", choices=("parent", "this"))
    ap.add_argument("--data")
    args = ap.parse_args()
    if args.host_worker:
        return host_worker(args.host_worker, args.data)
    if args.host_ab:
        os.makedirs(args.out_dir, exist_ok=True)
        return host_ab(os.path.abspath(args.parent_lib), args.rounds, os.path.join(args.out_dir, "%s_host_form_ab.json" % args.tag))
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
