"""dosplitalign_multi: every fastq split of a run in one process.

Its whole contract is that it looks like the stock dosplitalign run once per manifest line, in order, stopping after
the first run that fails: the same output files with the same bytes, stdout and stderr the concatenations of those
runs' streams, exit code 0 or 1.  Every test here runs both and compares them.  Without a GPU the tools run over
tests/device_double (LD_PRELOAD), as in test_tools_host_logic.py; the tests marked gpu run the same bodies on the B200."""
import json
import os
import subprocess

import pytest

import util

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
BIN = os.path.join(ROOT, "defuse_b200", "bin")
STOCK = os.path.join(BIN, "dosplitalign")
MULTI = os.path.join(BIN, "dosplitalign_multi")

# many batches, SAM chunks of a few lines, the bucketed de-duplication on every thread
SMALL_BATCHES = {"DFB_TOOL_BATCH": "53", "DFB_TOOL_CHUNK_MIN": "300", "DFB_TOOL_THREADS": "5"}


def _need_tools():
    if not (os.path.exists(STOCK) and os.path.exists(MULTI)):
        pytest.skip("tools not built")


def _shared_args(split_args):
    """make_split_dataset's argument list without the per-split flags (-i, -1, -2)."""
    out = []
    for k in range(0, len(split_args), 2):
        if split_args[k] not in ("-i", "-1", "-2"):
            out += split_args[k:k + 2]
    return out


def _collect(rows):
    """Bytes of every row's output (None where it does not exist), then remove them for the next arm."""
    got = []
    for row in rows:
        path = row[3]
        got.append(open(path, "rb").read() if os.path.exists(path) else None)
        if os.path.exists(path):
            os.remove(path)
    return tuple(got)


def _env(env):
    e = dict(os.environ)
    e.pop("DFB_DEVICE", None)
    e.update(env)
    return e


def stock_sequence(shared, rows, env):
    """The stock tool once per row, in order, stopping after the first run that fails."""
    code, out, err = 0, b"", b""
    for seq1, seq2, sam, align in rows:
        p = subprocess.run([STOCK] + shared + ["-i", sam, "-1", seq1, "-2", seq2, "-a", align], capture_output=True,
                           env=_env(env), timeout=600)
        out += p.stdout
        err += p.stderr
        if p.returncode != 0:
            code = 1
            break
    return code, out, err, _collect(rows)


def multi(shared, rows, env, manifest=None):
    """dosplitalign_multi over a manifest of `rows` (or the given manifest file)."""
    if manifest is None:
        manifest = os.path.join(os.path.dirname(rows[0][3]), "splits.tsv")
        with open(manifest, "w") as f:
            f.write("".join("\t".join(r) + "\n" for r in rows))
    p = subprocess.run([MULTI] + shared + ["-l", manifest], capture_output=True, env=_env(env), timeout=600)
    return p.returncode, p.stdout, p.stderr, _collect(rows)


def _dataset(tmp_path, name, n_splits=3):
    """A golden dataset of tests/golden/tools.json cut into n_splits splits; returns (shared args, split paths, dir)."""
    from synth import files
    g = json.load(open(os.path.join(HERE, "golden", "tools.json")))
    d = str(tmp_path / name)
    args = files.make_split_dataset(d, **g[name]["kw"])
    return _shared_args(args), files.cut_splits(d, n_splits), d


def _unmapped_only_sam(d):
    """A SAM of the dataset in `d` that holds only its unmapped records: the split has no candidate."""
    lines = open(os.path.join(d, "improper.sam"), "rb").read().splitlines(keepends=True)
    path = os.path.join(d, "unmapped_only.sam")
    with open(path, "wb") as f:
        f.write(b"".join(l for l in lines if l.startswith(b"@") or l.split(b"\t")[1] == b"4"))
    return path


def equality_body(tmp_path, devices):
    """Both golden datasets cut into 3 splits, plus the first split listed again (another output) and a split whose SAM
    holds only unmapped records; with and without many small batches; the multi form with and without the overlap of
    one split's ingest with the previous split's alignment."""
    for name in ("split_small", "split_jitter_lower"):
        shared, cut, d = _dataset(tmp_path, name)
        splits = cut + [cut[0], [cut[1][0], cut[1][1], _unmapped_only_sam(d)]]
        rows = [s + [os.path.join(d, "out.%d.alignments" % k)] for k, s in enumerate(splits)]
        for knobs in ({}, SMALL_BATCHES):
            env = dict(knobs, DFB_DEVICES=devices)
            want = stock_sequence(shared, rows, env)
            assert want[0] == 0, want[2].decode()[-2000:]
            files_ = want[3]
            assert all(len(b) > 0 for b in files_[:4]) and files_[3] == files_[0] and files_[4] == b""
            for overlap in ("1", "0"):
                got = multi(shared, rows, dict(env, DFB_SPLIT_OVERLAP=overlap))
                assert got == want, (name, knobs, overlap, got[0], got[2].decode()[-2000:])


@pytest.fixture
def double(device_double, monkeypatch):
    _need_tools()
    monkeypatch.setenv("LD_PRELOAD", device_double)
    return device_double


@pytest.mark.parametrize("devices", ["0", "0,1,2,3"])
def test_multi_equals_stock_runs(devices, double, tmp_path):
    equality_body(tmp_path, devices)


def test_cut_splits_partitions_the_reads(tmp_path):
    """Fragment f goes to split f % n in file order; every SAM keeps the header; nothing is lost or repeated."""
    from synth import files
    d = str(tmp_path / "s")
    files.make_split_dataset(d, seed=2, n_clusters=6, pairs_per_cluster=7)
    cut = files.cut_splits(d, 4)
    assert len(cut) == 4
    for col, name in enumerate(("reads.1.fastq", "reads.2.fastq")):
        whole = open(os.path.join(d, name), "rb").read().splitlines(keepends=True)
        records = [whole[k:k + 4] for k in range(0, len(whole), 4)]
        for k, paths in enumerate(cut):
            part = open(paths[col], "rb").read().splitlines(keepends=True)
            want = [r for r in records if int(r[0][1:].split(b"/")[0]) % 4 == k]
            assert part == [l for r in want for l in r]
    sam = open(os.path.join(d, "improper.sam"), "rb").read().splitlines(keepends=True)
    header = [l for l in sam if l.startswith(b"@")]
    body = [l for l in sam if not l.startswith(b"@")]
    for k, paths in enumerate(cut):
        part = open(paths[2], "rb").read().splitlines(keepends=True)
        assert part == header + [l for l in body if int(l.split(b"/")[0]) % 4 == k]


def test_first_failure_stops_the_run_malformed_sam(double, tmp_path):
    """Split 2 of 3 has a malformed SAM line: split 1 is written, split 2's message ends the run, split 3 is not
    touched."""
    shared, cut, d = _dataset(tmp_path, "split_small")
    bad = os.path.join(d, "bad.sam")
    lines = open(cut[1][2], "rb").read().splitlines(keepends=True)
    with open(bad, "wb") as f:
        f.write(b"".join(lines[:len(lines) // 2] + [b"not\ta\tsam\tline\n"] + lines[len(lines) // 2:]))
    rows = [cut[0] + [os.path.join(d, "o1")], [cut[1][0], cut[1][1], bad, os.path.join(d, "o2")],
            cut[2] + [os.path.join(d, "o3")]]
    for knobs in ({}, SMALL_BATCHES):
        want = stock_sequence(shared, rows, knobs)
        assert want[0] == 1 and b"Format error" in want[2] and want[3][0] and want[3][1:] == (None, None)
        for overlap in ("1", "0"):
            assert multi(shared, rows, dict(knobs, DFB_SPLIT_OVERLAP=overlap)) == want


def test_first_failure_stops_the_run_missing_fastq_read_ahead(double, tmp_path):
    """Split 3 names a missing fastq while split 2 (the whole dataset, many small batches) is still being aligned: the
    failure read ahead is held until split 2 is finished, then said, and split 3's output is never created."""
    shared, cut, d = _dataset(tmp_path, "split_small")
    whole = [os.path.join(d, n) for n in ("reads.1.fastq", "reads.2.fastq", "improper.sam")]
    rows = [cut[0] + [os.path.join(d, "o1")], whole + [os.path.join(d, "o2")],
            [os.path.join(d, "missing.1.fastq"), cut[2][1], cut[2][2], os.path.join(d, "o3")]]
    want = stock_sequence(shared, rows, SMALL_BATCHES)
    assert want[0] == 1 and b"unable to read sequences" in want[1] and want[3][0] and want[3][1] and want[3][2] is None
    assert multi(shared, rows, dict(SMALL_BATCHES, DFB_SPLIT_OVERLAP="1")) == want


def test_setup_error_said_once(double, tmp_path):
    """The set-up every split shares is read once: an error there is said once, as the first stock run says it, and no
    output is created."""
    shared, cut, d = _dataset(tmp_path, "split_small")
    rows = [s + [os.path.join(d, "o%d" % k)] for k, s in enumerate(cut)]
    for flag, bad in (("-e", "no_such.regions"), ("-f", "no_such.fa")):
        broken = list(shared)
        broken[broken.index(flag) + 1] = os.path.join(d, bad)
        want = stock_sequence(broken, rows, {})
        assert want[0] == 1 and want[3] == (None, None, None)
        assert multi(broken, rows, {}) == want


@pytest.mark.parametrize("case", ["missing", "empty", "three_fields", "empty_field", "stdin", "same_output"])
def test_manifest_errors(case, double, tmp_path):
    """A malformed manifest is rejected before any split is read or any output is created."""
    shared, cut, d = _dataset(tmp_path, "split_small", 2)
    rows = [cut[0] + [os.path.join(d, "o1")], cut[1] + [os.path.join(d, "o2")]]
    manifest = os.path.join(d, "splits.tsv")
    lines = ["\t".join(r) for r in rows]
    if case == "empty":
        lines = []
    elif case == "three_fields":
        lines[1] = "\t".join(rows[1][:3])
    elif case == "empty_field":
        lines[1] = "\t".join([rows[1][0], "", rows[1][2], rows[1][3]])
    elif case == "stdin":
        lines[1] = "\t".join([rows[1][0], rows[1][1], "-", rows[1][3]])
    elif case == "same_output":
        lines[1] = "\t".join(rows[1][:3] + [rows[0][3]])
    if case != "missing":
        with open(manifest, "w") as f:
            f.write("".join(l + "\n" for l in lines))
    code, out, err, outputs = multi(shared, rows, {}, manifest=manifest)
    assert code == 1 and err.startswith(b"Error:") and out == b"" and outputs == (None, None), (case, err)


def baseline_config_0_body(tmp_path):
    """A manifest whose first split is BASELINE.json configs[0] (the inputs of test_dosplitalign_baseline_config_0):
    its output is the unmodified reference tool's (stored digest); a second split matches the stock tool."""
    from synth import files
    d = str(tmp_path / "c0")
    args = files.make_split_dataset(d, seed=1, n_clusters=200, pairs_per_cluster=10, L=100, n_chrom=4, genes_per_chrom=10)
    cut = files.cut_splits(d, 2)
    whole = [os.path.join(d, n) for n in ("reads.1.fastq", "reads.2.fastq", "improper.sam")]
    rows = [whole + [os.path.join(d, "o1")], cut[1] + [os.path.join(d, "o2")]]
    shared = _shared_args(args)
    got = multi(shared, rows, {})
    assert got[0] == 0, got[2].decode()[-2000:]
    assert len(got[3][0].splitlines()) > 200
    assert util.digest(got[3][0]) == util.reference_digest("dosplitalign_tool/baseline_config_0")
    assert got == stock_sequence(shared, rows, {})


def test_baseline_config_0_first_split(double, tmp_path):
    baseline_config_0_body(tmp_path)


# ---- on the B200 ----

def _n_gpus():
    import defuse_b200
    return max(0, defuse_b200.load_library().dfb_device_count())


@pytest.mark.gpu
@pytest.mark.parametrize("devices", ["0", "0,0"])
def test_multi_equals_stock_runs_gpu(devices, tmp_path):
    _need_tools()
    equality_body(tmp_path, devices)


@pytest.mark.gpu
def test_multi_equals_stock_runs_distinct_gpus(tmp_path):
    _need_tools()
    n = _n_gpus()
    if n < 2:
        pytest.skip("needs two or more GPUs")
    equality_body(tmp_path, ",".join(str(k) for k in range(min(n, 4))))


@pytest.mark.gpu
def test_baseline_config_0_first_split_gpu(tmp_path):
    _need_tools()
    baseline_config_0_body(tmp_path)
