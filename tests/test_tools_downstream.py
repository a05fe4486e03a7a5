"""evalsplitalign (host-only, runs without a GPU) and splitseq (GPU: alignment + backtrace) against the committed
golden outputs of the compiled reference tools, and on fresh files against the stored digests of those tools' outputs
(tests/golden/reference_digests.json; where oracle/_ref exists, the reference tools run as well).  The tools are unchanged
since they last ran beside the compiled reference tools on these inputs and gave the same bytes; the digests are of those
outputs."""
import json
import os
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
BIN = os.path.join(ROOT, "defuse_b200", "bin")
sys.path.insert(0, ROOT)

import util  # noqa: E402


def _tool(name):
    p = os.path.join(BIN, name)
    if not os.path.exists(p):
        pytest.skip("tools not built")
    return p


def _run(cmd, **kw):
    p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=300, **kw)
    assert p.returncode == 0, (cmd[0], p.returncode, p.stderr.decode()[-2000:])
    return p.stdout


def _golden_dataset(tmp_path):
    from synth import files
    g = json.load(open(os.path.join(HERE, "golden", "tools_downstream.json")))
    d = str(tmp_path / "g")
    args = files.make_split_dataset(d, **g["kw"])
    open(os.path.join(d, "sorted.alignments"), "w").write(g["sorted"])
    common, ev = files.downstream_args(args, d)
    return g, d, common, ev


def _eval(tool, ev, d, tag):
    names = {k: os.path.join(d, "%s.%s" % (tag, k)) for k in ("seq", "break", "predalign")}
    _run([tool] + ev + ["-q", names["seq"], "-b", names["break"], "-p", names["predalign"]])
    return {k: open(v).read() for k, v in names.items()}


def _eval_bytes(outs):
    return tuple(outs[k].encode() for k in ("seq", "break", "predalign"))


def _output_file(cmd, path, env=None):
    _run(cmd, env=env)
    return (open(path, "rb").read(),)


def test_evalsplitalign_golden(tmp_path):
    g, d, common, ev = _golden_dataset(tmp_path)
    got = _eval(_tool("evalsplitalign"), ev, d, "ours")
    for k in ("seq", "break", "predalign"):
        assert got[k] == g[k], k


@pytest.mark.parametrize("kw", [dict(seed=51, n_clusters=80, pairs_per_cluster=50),
                                dict(seed=52, n_clusters=40, pairs_per_cluster=40, read_len_jitter=20, lower_frac=0.02, n_rate=0.01)])
def test_evalsplitalign_vs_reference_tool(oracle_mod, tmp_path, kw, device_double):
    """The reference dosplitalign's records, sorted, through our evalsplitalign and the reference's.  Without oracle/_ref
    the records come from our dosplitalign over the device double, checked against the reference's digest first."""
    from synth import files
    d = str(tmp_path / "d")
    args = files.make_split_dataset(d, **kw)
    raw = os.path.join(d, "raw.alignments")
    want_raw = util.reference_tool_digest(oracle_mod, "dosplitalign_tool/%(seed)d" % kw, "ref_dosplitalign",
                                          lambda ref: _output_file([ref] + args + ["-a", raw], raw))
    if not oracle_mod.ref_tool("ref_dosplitalign"):
        _run([_tool("dosplitalign")] + args + ["-a", raw], env=dict(os.environ, LD_PRELOAD=device_double))
    assert util.digest(open(raw, "rb").read()) == want_raw
    files.sort_alignments(raw, os.path.join(d, "sorted.alignments"))
    common, ev = files.downstream_args(args, d)
    ours = _eval(_tool("evalsplitalign"), ev, d, "ours")
    theirs = util.reference_tool_digest(oracle_mod, "evalsplitalign_tool/%(seed)d" % kw, "ref_evalsplitalign",
                                        lambda ref: _eval_bytes(_eval(ref, ev, d, "ref")))
    assert len(ours["seq"].splitlines()) > 10
    assert util.digest(*_eval_bytes(ours)) == theirs


def test_evalsplitalign_errors(tmp_path):
    g, d, common, ev = _golden_dataset(tmp_path)
    tool = _tool("evalsplitalign")
    outs = ["-q", os.path.join(d, "q"), "-b", os.path.join(d, "b"), "-p", os.path.join(d, "p")]
    open(os.path.join(d, "bad.alignments"), "w").write("0\t1\t0\t1\t5\n")
    p = subprocess.run([tool] + common + ["-a", os.path.join(d, "bad.alignments")] + outs, capture_output=True)
    assert p.returncode == 1 and b"Error: Format error for candidate reads line:" in p.stderr
    p = subprocess.run([tool] + common + ["-a", os.path.join(d, "missing.alignments")] + outs, capture_output=True)
    assert p.returncode == 1 and b"Error: Unable to open" in p.stderr
    p = subprocess.run([tool] + common + outs, capture_output=True)
    assert p.returncode == 1 and b"PARSE ERROR" in p.stderr


@pytest.mark.gpu
def test_splitseq_golden(tmp_path):
    from synth import files
    g, d, common, ev = _golden_dataset(tmp_path)
    open(os.path.join(d, "ref.predalign"), "w").write(g["predalign"])
    prefix = files.write_read_index(d)
    base = [_tool("splitseq")] + common + ["-p", prefix, "-a", os.path.join(d, "ref.predalign")]
    assert _run(base).decode() == g["splitseq"]
    for fid, want in g["splitseq_id"].items():
        assert _run(base + ["-i", fid]).decode() == want
    p = subprocess.run(base + ["-i", "99999"], capture_output=True)
    assert p.returncode == 1 and b"Error: Unable to find fusion 99999" in p.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(seed=61, n_clusters=60, pairs_per_cluster=50),
                                dict(seed=62, n_clusters=30, pairs_per_cluster=40, read_len_jitter=20, lower_frac=0.02, n_rate=0.01)])
def test_splitseq_vs_reference_tool(oracle_mod, tmp_path, kw):
    """Whole chain on fresh files: our dosplitalign -> sort -> our evalsplitalign -> our splitseq, against the compiled
    reference tools fed the same files.  splitseq is run on the full sorted alignments too (every record re-aligned and
    back-traced), not only on the predicted ones."""
    from synth import files
    d = str(tmp_path / "d")
    args = files.make_split_dataset(d, **kw)
    _run([_tool("dosplitalign")] + args + ["-a", os.path.join(d, "raw.alignments")])
    files.sort_alignments(os.path.join(d, "raw.alignments"), os.path.join(d, "sorted.alignments"))
    common, ev = files.downstream_args(args, d)
    ours = _eval(_tool("evalsplitalign"), ev, d, "ours")
    theirs = util.reference_tool_digest(oracle_mod, "evalsplitalign_tool/%(seed)d" % kw, "ref_evalsplitalign",
                                        lambda ref: _eval_bytes(_eval(ref, ev, d, "ref")))
    assert util.digest(*_eval_bytes(ours)) == theirs
    prefix = files.write_read_index(d)
    for name in ("ours.predalign", "sorted.alignments"):   # (ours.predalign has the reference's bytes: checked above)
        tail = common + ["-p", prefix, "-a", os.path.join(d, name)]
        a = _run([_tool("splitseq")] + tail)
        b = util.reference_tool_digest(oracle_mod, "splitseq_tool/%d/%s" % (kw["seed"], name.split(".")[1]), "ref_splitseq",
                                       lambda ref: (_run([ref] + tail),))
        assert len(a) > 1000
        assert util.digest(a) == b, name


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(seed=71, n_clusters=70, pairs_per_cluster=50),
                                dict(seed=72, n_clusters=30, pairs_per_cluster=40, read_len_jitter=20, lower_frac=0.02, n_rate=0.01)])
def test_fused_align_evaluate_vs_reference_pipeline(oracle_mod, tmp_path, kw):
    """dosplitalign_eval (align -> evaluate without the alignments file, the sort and the second parse in between) against
    the reference pipeline on the same files: ref dosplitalign | sort -n -k 1 (C locale) | ref evalsplitalign.  The three
    outputs must be byte-identical; with -a the alignments file is still written and equals the reference's; several
    small GPU batches and small evaluation regions give the same bytes."""
    from synth import files
    d = str(tmp_path / "d")
    args = files.make_split_dataset(d, **kw)
    common, ev = files.downstream_args(args, d)

    def reference_pipeline(ref_split):
        _run([ref_split] + args + ["-a", os.path.join(d, "raw.alignments")])
        p = subprocess.run("LC_ALL=C sort -n -k 1 %s > %s" % (os.path.join(d, "raw.alignments"), os.path.join(d, "sorted.alignments")),
                           shell=True)
        assert p.returncode == 0
        return _eval_bytes(_eval(oracle_mod.ref_tool("ref_evalsplitalign"), ev, d, "ref"))

    theirs = util.reference_tool_digest(oracle_mod, "evalsplitalign_pipeline/%(seed)d" % kw, "ref_dosplitalign", reference_pipeline)
    want_raw = util.reference_tool_digest(oracle_mod, "dosplitalign_tool/%(seed)d" % kw, "ref_dosplitalign",
                                          lambda ref: (open(os.path.join(d, "raw.alignments"), "rb").read(),))

    def fused(tag, extra=(), env=None):
        names = {k: os.path.join(d, "%s.%s" % (tag, k)) for k in ("seq", "break", "predalign")}
        _run([_tool("dosplitalign_eval")] + args + list(extra) + ["-q", names["seq"], "-b", names["break"], "-p", names["predalign"]],
             env=dict(os.environ, **env) if env else None)
        return {k: open(v).read() for k, v in names.items()}

    got = fused("fused")
    assert len(got["seq"].splitlines()) > 10
    assert util.digest(*_eval_bytes(got)) == theirs
    assert util.digest(*_eval_bytes(fused("fused_a", ["-a", os.path.join(d, "fused.alignments")]))) == theirs
    assert util.digest(open(os.path.join(d, "fused.alignments"), "rb").read()) == want_raw
    assert util.digest(*_eval_bytes(fused("fused_small", env={"DFB_TOOL_BATCH": "700", "DFB_TOOL_CHUNK_MIN": "400"}))) == theirs


def test_evalsplitalign_score_ties_follow_the_reference_container_order(oracle_mod, tmp_path):
    """Evaluate picks the first split with the highest summed score in the ITERATION order of an
    unordered_map<pair<int,int>,int> (tools/SplitAlignment.cpp:505-528).  Engineered records: many distinct refSplits
    per fusion, summed scores tied on purpose, enough keys to force rehashes.  Host-only, so it runs without a GPU."""
    import numpy as np
    from synth import files
    d = str(tmp_path / "d")
    args = files.make_split_dataset(d, seed=71, n_clusters=40, pairs_per_cluster=2)
    common, ev = files.downstream_args(args, d)
    rng = np.random.default_rng(72)
    lines = []
    for fusion in range(40):
        n_splits = int(rng.choice([1, 2, 3, 8, 20, 60, 200]))
        splits = {(int(rng.integers(0, 120)), int(rng.integers(-1, 100))) for _ in range(n_splits)}
        tie_score = int(rng.integers(20, 60))
        for (s1, s2) in splits:
            # every split reaches the same total through a different number of records (some fall short, some tie)
            parts = int(rng.integers(1, 4))
            total = tie_score if rng.random() < 0.7 else int(rng.integers(1, tie_score))
            cuts = sorted(rng.integers(0, total + 1, parts - 1).tolist())
            scores = [b - a for a, b in zip([0] + cuts, cuts + [total])]
            for sc in scores:
                a = int(rng.integers(4, 97))
                lines.append((fusion, "%d\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t\n" % (
                    fusion, int(rng.integers(0, 10 ** 6)), int(rng.integers(0, 2)), int(rng.integers(0, 2)), s1, s2, a, 100 - a, sc)))
    # records of a fusion stay together, their order inside the fusion is shuffled (insertion order matters too)
    order = rng.permutation(len(lines))
    text = "".join(l for _, l in sorted((lines[k] for k in order), key=lambda x: x[0]))
    open(os.path.join(d, "sorted.alignments"), "w").write(text)
    ours = _eval(_tool("evalsplitalign"), ev, d, "ours")
    theirs = util.reference_tool_digest(oracle_mod, "evalsplitalign_tool/score_ties", "ref_evalsplitalign",
                                        lambda ref: _eval_bytes(_eval(ref, ev, d, "ref")))
    assert len(ours["seq"].splitlines()) == 40
    assert util.digest(*_eval_bytes(ours)) == theirs


def _eval_rc(tool, ev, d, tag, env=None):
    names = {k: os.path.join(d, "%s.%s" % (tag, k)) for k in ("seq", "break", "predalign")}
    p = subprocess.run([tool] + ev + ["-q", names["seq"], "-b", names["break"], "-p", names["predalign"]],
                       capture_output=True, timeout=300, env=dict(os.environ, **(env or {})))
    return p, {k: open(v).read() for k, v in names.items()}


@pytest.mark.parametrize("env", [dict(DFB_TOOL_THREADS="1"), dict(DFB_TOOL_THREADS="3", DFB_TOOL_CHUNK_MIN="64"),
                                 dict(DFB_TOOL_THREADS="7", DFB_TOOL_CHUNK_MIN="700"), dict(DFB_TOOL_THREADS="16", DFB_TOOL_CHUNK_MIN="5000")])
def test_evalsplitalign_regions_and_blocks_reproduce_the_serial_reader(tmp_path, env):
    """The records file is cut into blocks and per-thread regions where the fusion id changes: any cut gives the
    golden bytes (regions of a few lines, several blocks, more threads than runs)."""
    g, d, common, ev = _golden_dataset(tmp_path)
    p, got = _eval_rc(_tool("evalsplitalign"), ev, d, "ours", env)
    assert p.returncode == 0, p.stderr
    for k in ("seq", "break", "predalign"):
        assert got[k] == g[k], k


def test_evalsplitalign_dies_where_the_reference_dies(oracle_mod, tmp_path):
    """A line with too few fields ends the run of the reference at that line (tools/SplitAlignment.cpp:331-335): the
    fusions in front of it are written, and -- because the reader looks at the first line of the NEXT fusion before it
    evaluates the current one -- a bad first line of a fusion also drops the fusion in front of it.  Same sequence and
    break files as the compiled tool for every cut of the file (prediction records are buffered by the reference and
    lost at exit, so they are not compared)."""
    g, d, common, ev = _golden_dataset(tmp_path)
    lines = g["sorted"].splitlines(keepends=True)
    ids = [l.split("\t")[0] for l in lines]
    starts = [k for k in range(1, len(lines)) if ids[k] != ids[k - 1]]
    inside = [k for k in range(1, len(lines) - 1) if ids[k] == ids[k - 1] == ids[k + 1]]
    assert len(starts) > 6 and len(inside) > 6
    cases = {"first line of a fusion": starts[len(starts) // 2], "inside a fusion": inside[len(inside) // 2],
             "first line of the file": 0, "last line of the file": len(lines)}
    for name, at in cases.items():
        bad = lines[:at] + ["12\t3\t0\n"] + lines[at:]
        open(os.path.join(d, "sorted.alignments"), "w").write("".join(bad))

        def reference(ref_eval):
            pr, theirs = _eval_rc(ref_eval, ev, d, "ref")
            assert pr.returncode == 1 and b"Format error" in pr.stderr, name
            stderr = b"".join(l for l in pr.stderr.splitlines(keepends=True) if not l.startswith(b"[fai_load]"))  # samtools' notice
            return stderr.replace(d.encode(), b"<dir>"), theirs["seq"].encode(), theirs["break"].encode()

        want = util.reference_tool_digest(oracle_mod, "evalsplitalign_tool/dies/" + name, "ref_evalsplitalign", reference)
        for env in (dict(DFB_TOOL_THREADS="1"), dict(DFB_TOOL_THREADS="4", DFB_TOOL_CHUNK_MIN="100"),
                    dict(DFB_TOOL_THREADS="8", DFB_TOOL_CHUNK_MIN="1500")):
            po, ours = _eval_rc(_tool("evalsplitalign"), ev, d, "ours", env)
            assert po.returncode == 1 and b"Format error" in po.stderr, (name, env)
            assert util.digest(po.stderr.replace(d.encode(), b"<dir>"), ours["seq"].encode(), ours["break"].encode()) == want, \
                (name, env, po.stderr)
