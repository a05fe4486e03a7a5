#!/usr/bin/env python
"""Every fastq split of a run: the stock dosplitalign once per split against dosplitalign_multi in one process.

Seeded input (default 8 splits x 1 M read pairs over 10 000 clusters, one make_split_dataset cut with cut_splits, so
every split sees every cluster).  Arms, all in one call:
  a        the stock tool once per split, one after another (DFB_DEVICE=0)
  b<N>     the stock tool N processes at a time, split k on device k mod N (defuse_run.pl -p N, a device per process)
  c<N>     dosplitalign_multi with DFB_DEVICES=0..N-1
for every N in 1/2/4/8 up to the visible GPUs (b1 is a).  Each arm runs --reps times, the arms alternating.  Also the
A/B of dosplitalign_multi's overlap of split k+1's ingest with split k's alignment (DFB_SPLIT_OVERLAP=1 against 0,
N=1, alternating) and one DFB_TRACE=1 run of c1 with its per-split laps.
Reported per arm: wall seconds, input read pairs per second, host CPU seconds (user + system of the tool processes);
identical_output: the SHA-256 of every split's output is the same in every arm.  GPU name, power limit and host core
count are read in the same call.
Usage (on a B200 machine): python scripts/gpu_tool_splits.py [--splits 8] [--pairs-per-split 1000000] [--clusters 10000]
                        [--reps 2] > tool_splits.json"""
import argparse
import hashlib
import json
import os
import resource
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from synth import files  # noqa: E402

BIN = os.path.join(ROOT, "defuse_b200", "bin")


def gpu_facts():
    p = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    rows = [l.strip() for l in p.stdout.splitlines() if l.strip()]
    if p.returncode != 0 or not rows:
        sys.exit("no GPU visible: this measurement runs on the B200")
    return rows


def child_cpu_s():
    r = resource.getrusage(resource.RUSAGE_CHILDREN)
    return r.ru_utime + r.ru_stime


def env_for(**kw):
    e = dict(os.environ)
    for k in ("DFB_DEVICE", "DFB_DEVICES", "DFB_TRACE", "DFB_SPLIT_OVERLAP"):
        e.pop(k, None)
    e.update({k: str(v) for k, v in kw.items()})
    return e


def run_stock(shared, splits, outs, n_lanes):
    """Lane d runs the splits k with k mod n_lanes == d one after another on device d; the lanes run side by side."""
    errors = []

    def lane(d):
        for k in range(d, len(splits), n_lanes):
            s1, s2, sam = splits[k]
            p = subprocess.run([os.path.join(BIN, "dosplitalign")] + shared + ["-i", sam, "-1", s1, "-2", s2, "-a", outs[k]],
                               capture_output=True, env=env_for(DFB_DEVICE=d))
            if p.returncode != 0:
                errors.append(p.stderr.decode()[-2000:])

    th = [threading.Thread(target=lane, args=(d,)) for d in range(n_lanes)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errors, errors[0]
    return ""


def run_multi(shared, splits, outs, n_gpus, overlap=None, trace=False):
    manifest = outs[0] + ".manifest.tsv"
    with open(manifest, "w") as f:
        for (s1, s2, sam), out in zip(splits, outs):
            f.write("\t".join([s1, s2, sam, out]) + "\n")
    kw = {"DFB_DEVICES": ",".join(str(d) for d in range(n_gpus))}
    if overlap is not None:
        kw["DFB_SPLIT_OVERLAP"] = overlap
    if trace:
        kw["DFB_TRACE"] = 1
    p = subprocess.run([os.path.join(BIN, "dosplitalign_multi")] + shared + ["-l", manifest], capture_output=True,
                       env=env_for(**kw))
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    return p.stderr.decode()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--splits", type=int, default=8)
    ap.add_argument("--pairs-per-split", type=int, default=1000000)
    ap.add_argument("--clusters", type=int, default=10000)
    ap.add_argument("--reps", type=int, default=2)
    a = ap.parse_args()
    gpus = gpu_facts()
    n_visible = len(gpus)
    ns = [n for n in (1, 2, 4, 8) if n <= n_visible]
    pairs = a.splits * a.pairs_per_split
    out = {"gpus": gpus, "host_cpus": os.cpu_count(), "splits": a.splits, "read_pairs": pairs, "clusters": a.clusters,
           "not_measured": ["N=%d (the box has %d GPU%s)" % (n, n_visible, "" if n_visible == 1 else "s")
                            for n in (2, 4, 8) if n > n_visible]}
    with tempfile.TemporaryDirectory() as d:
        t0 = time.perf_counter()
        data = os.path.join(d, "data")
        args = files.make_split_dataset(data, seed=3, n_clusters=a.clusters, pairs_per_cluster=max(1, pairs // a.clusters),
                                        n_chrom=8, genes_per_chrom=40)
        splits = files.cut_splits(data, a.splits)
        shared = []
        for k in range(0, len(args), 2):
            if args[k] not in ("-i", "-1", "-2"):
                shared += args[k:k + 2]
        for name in ("reads.1.fastq", "reads.2.fastq", "improper.sam"):
            os.remove(os.path.join(data, name))
        out["generate_s"] = time.perf_counter() - t0

        arms = {"a": lambda o: run_stock(shared, splits, o, 1)}
        for n in ns:
            if n > 1:
                arms["b%d" % n] = (lambda n: lambda o: run_stock(shared, splits, o, n))(n)
            arms["c%d" % n] = (lambda n: lambda o: run_multi(shared, splits, o, n))(n)
        arms["c1_overlap"] = lambda o: run_multi(shared, splits, o, 1, overlap="1")
        arms["c1_sequential"] = lambda o: run_multi(shared, splits, o, 1, overlap="0")
        # warm the page cache and the .fai once, outside the timed runs
        run_stock(shared, splits[:1], [os.path.join(d, "warm")], 1)
        results = {name: {"wall_s": [], "cpu_s": []} for name in arms}
        digests = {}
        for rep in range(a.reps):
            for name, fn in arms.items():
                o = [os.path.join(d, "%s.%d.alignments" % (name, k)) for k in range(a.splits)]
                c0, t0 = child_cpu_s(), time.perf_counter()
                fn(o)
                results[name]["wall_s"].append(time.perf_counter() - t0)
                results[name]["cpu_s"].append(child_cpu_s() - c0)
                h = []
                for path in o:
                    h.append(hashlib.sha256(open(path, "rb").read()).hexdigest())
                    os.remove(path)
                digests.setdefault(name, h)
                assert digests[name] == h, name
                sys.stderr.write("%s rep %d: %.3f s\n" % (name, rep, results[name]["wall_s"][-1]))
        for name, r in results.items():
            best = min(r["wall_s"])
            r["best_wall_s"] = best
            r["read_pairs_per_s"] = pairs / best
            r["cpu_s_at_best"] = r["cpu_s"][r["wall_s"].index(best)]
        out["arms"] = results
        ref = digests["a"]
        out["identical_output"] = all(h == ref for h in digests.values())
        out["split_output_sha256"] = ref
        out["speedup_c1_over_a"] = results["a"]["best_wall_s"] / results["c1"]["best_wall_s"]
        out["overlap_ab"] = {"overlap_best_s": results["c1_overlap"]["best_wall_s"],
                             "sequential_best_s": results["c1_sequential"]["best_wall_s"],
                             "overlap_faster": results["c1_overlap"]["best_wall_s"] < results["c1_sequential"]["best_wall_s"]}
        o = [os.path.join(d, "trace.%d.alignments" % k) for k in range(a.splits)]
        trace = run_multi(shared, splits, o, 1, trace=True)
        out["trace_c1"] = [l for l in trace.splitlines() if l.startswith("[tool]")]
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
