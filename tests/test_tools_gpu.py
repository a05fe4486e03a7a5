"""Drop-in tools (defuse_b200/bin/*) against (a) the committed golden outputs of the compiled reference tools and
(b) the compiled reference tools' outputs on fresh, larger synthetic files: byte-identical.  For (b) the SHA-256 digests
of the reference's outputs are stored in tests/golden/reference_digests.json; where oracle/_ref/ref_* are built, the
reference tools run as well.  (The tools are unchanged since they last ran beside the compiled reference tools on these
inputs and gave the same bytes; the digests are of those outputs.)"""
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

pytestmark = pytest.mark.gpu


def _run(cmd, stdin=None, env=None):
    p = subprocess.run(cmd, input=stdin, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=300,
                       env=dict(os.environ, **env) if env else None)
    assert p.returncode == 0, (cmd[0], p.returncode, p.stderr.decode()[-2000:])
    return p.stdout


def test_localalign_golden():
    g = json.load(open(os.path.join(HERE, "golden", "localalign_tool.json")))
    for run in g["runs"].values():
        out = _run([os.path.join(BIN, "localalign")] + run["args"], g["stdin"].encode())
        assert out.decode() == run["stdout"]


def test_dosplitalign_and_matealign_golden(tmp_path):
    from synth import files
    g = json.load(open(os.path.join(HERE, "golden", "tools.json")))
    for name in ("split_small", "split_jitter_lower"):
        sub = str(tmp_path / name)
        args = files.make_split_dataset(sub, **g[name]["kw"])
        res = os.path.join(sub, "ours.alignments")
        _run([os.path.join(BIN, "dosplitalign")] + args + ["-a", res])
        assert open(res).read() == g[name]["output"], name
    args, sam = files.make_matealign_dataset(str(tmp_path / "mate"), **g["mate_small"]["kw"])
    assert _run([os.path.join(BIN, "matealign")] + args, sam).decode() == g["mate_small"]["output"]


@pytest.mark.parametrize("scoring", [["-m", "10", "-x", "-5", "-g", "-5", "-t", "0.8"], ["-m", "2", "-x", "-1", "-g", "-2"],
                                     ["-m", "1", "-x", "-1", "-g", "1", "-t", "0.2"]])
def test_localalign_vs_reference_tool(oracle_mod, scoring):
    from synth import files
    text = files.make_localalign_input(seed=11, n_refs=30, n_lines=3000)
    text += b"empty\tACGT\t\n" + b"extra\tACGTACGT\tCGTA\tjunk\n"
    want = util.reference_tool_digest(oracle_mod, "localalign_tool/" + " ".join(scoring), "ref_localalign", lambda ref: (_run([ref] + scoring, text),))
    assert util.digest(_run([os.path.join(BIN, "localalign")] + scoring, text)) == want


def test_localalign_errors_like_reference(oracle_mod):
    args = ["-m", "10", "-x", "-5", "-g", "-5"]
    for k, text in enumerate((b"a\tACGT\tACG\n\nb\tACGT\tACG\n", b"a\tACGT\tACG\nbad line\n")):
        ours = subprocess.run([os.path.join(BIN, "localalign")] + args, input=text, capture_output=True)
        theirs = util.reference_tool_digest(oracle_mod, "localalign_tool_errors/%d" % k, "ref_localalign",
                            lambda ref: _exit_1(subprocess.run([ref] + args, input=text, capture_output=True)))
        assert ours.returncode == 1
        assert util.digest(ours.stdout, ours.stderr) == theirs  # the lines before the bad one are still printed


def test_matealign_vs_reference_tool(oracle_mod, tmp_path):
    from synth import files
    args, sam = files.make_matealign_dataset(str(tmp_path / "m"), seed=21, n_pairs=1500)
    want = util.reference_tool_digest(oracle_mod, "matealign_tool", "ref_matealign", lambda ref: (_run([ref] + args, sam),))
    assert util.digest(_run([os.path.join(BIN, "matealign")] + args, sam)) == want


@pytest.mark.parametrize("kw", [dict(seed=31, n_clusters=120, pairs_per_cluster=60),
                                dict(seed=32, n_clusters=60, pairs_per_cluster=60, read_len_jitter=25, lower_frac=0.02, n_rate=0.01),
                                dict(seed=33, n_clusters=40, pairs_per_cluster=50, L=150, frag_mean=400)])
def test_dosplitalign_vs_reference_tool(oracle_mod, tmp_path, kw):
    from synth import files
    d = str(tmp_path / "d")
    args = files.make_split_dataset(d, **kw)
    ours, theirs = os.path.join(d, "ours.tmp"), os.path.join(d, "ref.tmp")   # cmdrunner hands tools *.tmp outputs
    want = util.reference_tool_digest(oracle_mod, "dosplitalign_tool/%(seed)d" % kw, "ref_dosplitalign",
                      lambda ref: _output_file([ref] + args + ["-a", theirs], theirs))
    _run([os.path.join(BIN, "dosplitalign")] + args + ["-a", ours])
    a = open(ours, "rb").read()
    assert len(a.splitlines()) > 100
    assert util.digest(a) == want


@pytest.mark.parametrize("devices", ["0,0", "0,0,0,0"])
def test_dosplitalign_sharded_over_contexts(oracle_mod, tmp_path, devices):
    """Multi-GPU path of the tool (one context per entry of DFB_DEVICES, candidates dealt out by cluster, merged in
    candidate order), exercised on one GPU by naming it several times: the output must not change."""
    from synth import files
    g = json.load(open(os.path.join(HERE, "golden", "tools.json")))
    sub = str(tmp_path / "s")
    args = files.make_split_dataset(sub, **g["split_small"]["kw"])
    res = os.path.join(sub, "ours.alignments")
    _run([os.path.join(BIN, "dosplitalign")] + args + ["-a", res], env={"DFB_DEVICES": devices})
    assert open(res).read() == g["split_small"]["output"]
    d = str(tmp_path / "big")
    args = files.make_split_dataset(d, seed=41, n_clusters=150, pairs_per_cluster=80)
    ours, theirs = os.path.join(d, "ours.tmp"), os.path.join(d, "ref.tmp")
    want = util.reference_tool_digest(oracle_mod, "dosplitalign_tool/41", "ref_dosplitalign",
                      lambda ref: _output_file([ref] + args + ["-a", theirs], theirs))
    _run([os.path.join(BIN, "dosplitalign")] + args + ["-a", ours], env={"DFB_DEVICES": devices})
    assert util.digest(open(ours, "rb").read()) == want


def _output_file(cmd, path):
    _run(cmd)
    return (open(path, "rb").read(),)


def _exit_1(p):
    assert p.returncode == 1
    return p.stdout, p.stderr


def _n_gpus():
    import defuse_b200
    return max(0, defuse_b200.load_library().dfb_device_count())


@pytest.mark.parametrize("devices", ["0,1", "all"])
def test_dosplitalign_sharded_over_distinct_gpus(oracle_mod, tmp_path, devices):
    """The partition-by-cluster + host-merge path on MORE THAN ONE physical GPU (needs `gpurun --gpus 2` or more; skipped
    on a one-GPU box): a fastq split large enough for every device to get work, its output compared byte for byte with
    the one-GPU run and, on a sample of the same generator, with the compiled reference tool
    (fan-out + ordered merge: scripts/defuse_run.pl:518-533; emission order: tools/SplitAlignment.cpp:271-301)."""
    from synth import files
    n = _n_gpus()
    if n < 2:
        pytest.skip("one GPU visible: the distinct-ordinal path needs at least two")
    d = str(tmp_path / "big")
    args = files.make_split_dataset(d, seed=51, n_clusters=1500, pairs_per_cluster=100, n_chrom=8, genes_per_chrom=40)
    one, many = os.path.join(d, "one.tmp"), os.path.join(d, "many.tmp")
    _run([os.path.join(BIN, "dosplitalign")] + args + ["-a", one], env={"DFB_DEVICES": "0"})
    p = subprocess.run([os.path.join(BIN, "dosplitalign")] + args + ["-a", many], env=dict(os.environ, DFB_DEVICES=devices, DFB_TRACE="1"),
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=300)
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    a, b = open(one, "rb").read(), open(many, "rb").read()
    assert a.count(b"\n") > 20000
    assert a == b
    # one context per named device (the library's trace reports every context it creates), and every one of them ran batches
    trace = p.stderr.decode()
    want = 2 if devices == "0,1" else n
    assert trace.count("ctx: context, streams, pools") == want, trace[-1500:]
    ref = oracle_mod.ref_tool("ref_dosplitalign")
    if ref:
        s = str(tmp_path / "sample")
        sargs = files.make_split_dataset(s, seed=52, n_clusters=200, pairs_per_cluster=80, n_chrom=8, genes_per_chrom=40)
        ours, theirs = os.path.join(s, "ours.tmp"), os.path.join(s, "ref.tmp")
        _run([os.path.join(BIN, "dosplitalign")] + sargs + ["-a", ours], env={"DFB_DEVICES": devices})
        _run([ref] + sargs + ["-a", theirs])
        assert open(ours, "rb").read() == open(theirs, "rb").read()


def test_tools_with_many_small_batches(oracle_mod, tmp_path):
    """The tools flush work to the GPU in batches (1 M tasks by default); DFB_TOOL_BATCH forces many small batches on
    small inputs.  Output bytes must not depend on the batch size."""
    from synth import files
    g = json.load(open(os.path.join(HERE, "golden", "tools.json")))
    sub = str(tmp_path / "s")
    args = files.make_split_dataset(sub, **g["split_small"]["kw"])
    res = os.path.join(sub, "ours.alignments")
    for batch, devices in (("37", "0"), ("64", "0,0")):
        _run([os.path.join(BIN, "dosplitalign")] + args + ["-a", res], env={"DFB_TOOL_BATCH": batch, "DFB_DEVICES": devices})
        assert open(res).read() == g["split_small"]["output"]
    margs, sam = files.make_matealign_dataset(str(tmp_path / "mate"), **g["mate_small"]["kw"])
    assert _run([os.path.join(BIN, "matealign")] + margs, sam, env={"DFB_TOOL_BATCH": "29"}).decode() == g["mate_small"]["output"]
    gl = json.load(open(os.path.join(HERE, "golden", "localalign_tool.json")))
    for run in gl["runs"].values():
        out = _run([os.path.join(BIN, "localalign")] + run["args"], gl["stdin"].encode(), env={"DFB_TOOL_BATCH": "7"})
        assert out.decode() == run["stdout"]


def test_localalign_blocks_pipe_and_mapped_file(oracle_mod, tmp_path):
    """stdin is consumed in blocks of whole lines: read ahead from a pipe, or mapped when it is a file.  Block and
    chunk boundaries anywhere, output bytes unchanged; a bad line still ends the run where the reference ends it."""
    from synth import files
    sc = ["-m", "10", "-x", "-5", "-g", "-5", "-t", "0.3"]
    text = files.make_localalign_input(seed=17, n_refs=12, n_lines=900)
    want = util.reference_tool_digest(oracle_mod, "localalign_tool_blocks", "ref_localalign", lambda ref: (_run([ref] + sc, text),))
    path = str(tmp_path / "in.txt")
    open(path, "wb").write(text)
    for block, chunk in (("5000", "1"), ("70000", "3000"), ("1", "1"), ("300000000", "65536")):
        env = {"DFB_TOOL_BLOCK": block, "DFB_TOOL_CHUNK_MIN": chunk}
        assert util.digest(_run([os.path.join(BIN, "localalign")] + sc, text, env=env)) == want, ("pipe", block, chunk)
        with open(path, "rb") as f:
            p = subprocess.run([os.path.join(BIN, "localalign")] + sc, stdin=f, capture_output=True, env=dict(os.environ, **env))
        assert p.returncode == 0 and util.digest(p.stdout) == want, ("file", block, chunk)
    bad = text + b"oops no tabs\n" + text[:5000]
    theirs = util.reference_tool_digest(oracle_mod, "localalign_tool_blocks_bad_line", "ref_localalign",
                        lambda ref: _exit_1(subprocess.run([ref] + sc, input=bad, capture_output=True)))
    for block in ("4000", "300000000"):
        ours = subprocess.run([os.path.join(BIN, "localalign")] + sc, input=bad, capture_output=True,
                              env=dict(os.environ, DFB_TOOL_BLOCK=block, DFB_TOOL_CHUNK_MIN="500"))
        assert ours.returncode == 1
        assert util.digest(ours.stdout, ours.stderr) == theirs


def test_matealign_chunked_ingest(oracle_mod, tmp_path):
    from synth import files
    args, sam = files.make_matealign_dataset(str(tmp_path / "m"), seed=23, n_pairs=700)
    want = util.reference_tool_digest(oracle_mod, "matealign_tool_chunked", "ref_matealign", lambda ref: (_run([ref] + args, sam),))
    for chunk, threads, batch in (("1", "16", "50"), ("900", "3", "100000")):
        got = _run([os.path.join(BIN, "matealign")] + args, sam,
                   env={"DFB_TOOL_CHUNK_MIN": chunk, "DFB_TOOL_THREADS": threads, "DFB_TOOL_BATCH": batch})
        assert util.digest(got) == want


def _compact_localalign_input(data):
    """The input form of localalign_dedup: '=' where a line's reference equals the one on the line before."""
    out, prev = [], None
    for line in data.split(b"\n"):
        f = line.split(b"\t")
        if len(f) >= 3 and f[1] == prev:
            f[1] = b"="
        elif len(f) >= 3:
            prev = f[1]
        out.append(b"\t".join(f))
    return b"\n".join(out)


@pytest.mark.parametrize("env", [None, {"DFB_TOOL_BATCH": "37", "DFB_TOOL_BLOCK": "30000", "DFB_TOOL_THREADS": "5"}])
def test_localalign_dedup_input_form(oracle_mod, env):
    """localalign_dedup reads the input form that carries every reference once (SURVEY 8f rank 4): same output bytes as the
    reference tool on the expanded input, with blocks and chunks cut in the middle of runs of '=' lines, too."""
    from synth import files
    lines = files.make_localalign_input(seed=9, n_refs=25, n_lines=900).splitlines()
    lines.sort(key=lambda l: l.split(b"\t")[1])   # the pipeline lists the reads of a cluster together: runs of one reference
    data = b"\n".join(lines) + b"\n"
    compact = _compact_localalign_input(data)
    assert len(compact) < len(data) // 8
    sc = ["-m", "10", "-x", "-5", "-g", "-5", "-t", "0.8"]
    want = util.reference_tool_digest(oracle_mod, "localalign_tool_dedup", "ref_localalign", lambda ref: (_run([ref] + sc, data),))
    assert util.digest(_run([os.path.join(BIN, "localalign_dedup")] + sc, compact, env)) == want
    assert util.digest(_run([os.path.join(BIN, "localalign_dedup")] + sc, data, env)) == want      # the stock form is still understood
    # a leading '=' has no reference to stand for
    p = subprocess.run([os.path.join(BIN, "localalign_dedup")] + sc, input=b"a\t=\tACGT\n", stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                       env=dict(os.environ, **env) if env else None)
    assert p.returncode == 1 and b"Format error for line 1" in p.stderr
