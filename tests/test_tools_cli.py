"""Command-line grammar and no-GPU behaviour of the drop-in tools (CPU only)."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "defuse_b200", "bin")


def _tool(name):
    p = os.path.join(BIN, name)
    if not os.path.exists(p):
        pytest.skip("tools not built")
    return p


@pytest.mark.parametrize("tool,args", [("localalign", ["-m", "10"]), ("matealign", ["-m", "1", "-x", "-1", "-g", "-1"]),
                                       ("dosplitalign", ["-f", "x.fa"])])
def test_missing_required_arguments(tool, args):
    p = subprocess.run([_tool(tool)] + args, capture_output=True, input=b"")
    assert p.returncode == 1
    assert b"PARSE ERROR" in p.stderr and b"required" in p.stderr.lower()
    assert p.stdout == b""


def test_unknown_flag_and_bad_value():
    p = subprocess.run([_tool("localalign"), "-m", "10", "-x", "-5", "-g", "-5", "-q", "1"], capture_output=True, input=b"")
    assert p.returncode == 1 and b"PARSE ERROR" in p.stderr
    p = subprocess.run([_tool("localalign"), "-m", "ten", "-x", "-5", "-g", "-5"], capture_output=True, input=b"")
    assert p.returncode == 1 and b"PARSE ERROR" in p.stderr


def test_help_lists_the_reference_flags():
    p = subprocess.run([_tool("dosplitalign"), "--help"], capture_output=True)
    assert p.returncode == 0
    for flag in ("--fasta", "--exons", "--ufrag", "--sfrag", "--minread", "--maxread", "--regions", "--improper", "--seq1",
                 "--seq2", "--align"):
        assert flag.encode() in p.stdout
    p = subprocess.run([_tool("matealign"), "-h"], capture_output=True)
    for flag in ("--match", "--mismatch", "--gap", "--threshold", "--searchlength", "--reference", "--seq1", "--seq2"):
        assert flag.encode() in p.stdout


def test_no_gpu_means_failure_not_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    p = subprocess.run([_tool("localalign"), "-m", "10", "-x", "-5", "-g", "-5"], capture_output=True, input=b"a\tACGT\tACG\n")
    assert p.returncode == 1
    assert p.stdout == b"" and b"Error:" in p.stderr and b"no CPU fallback" in p.stderr


def test_dosplitalign_input_errors_like_the_reference(tmp_path):
    """Errors that come before any alignment (so no GPU is needed): same exit code, stdout and stderr as the compiled
    reference tool for unreadable inputs and malformed region tables (its outputs stored as digests, with the dataset's
    directory written as <dir>; where oracle/_ref is built the tool runs as well)."""
    import sys
    sys.path.insert(0, ROOT)
    import oracle
    import util
    from synth import files
    d = str(tmp_path / "s")
    args = files.make_split_dataset(d, seed=3, n_clusters=6, pairs_per_cluster=10)

    def swap(flag, val):
        a = list(args)
        a[a.index(flag) + 1] = val
        return a + ["-a", os.path.join(d, "o.tmp")]

    open(os.path.join(d, "bad2.regions"), "w").write("0\t0\tchr1\t?\t100\t200\n0\t1\tchr1\t+\t100\t200\n")
    open(os.path.join(d, "bad3.regions"), "w").write("0\t0\tnochrom\t+\t100\t200\n0\t1\tchr1\t+\t100\t200\n")
    open(os.path.join(d, "reads.1.txt"), "w").write(open(os.path.join(d, "reads.1.fastq")).read())
    cases = [swap("-e", d + "/nope"), swap("-r", d + "/nope"), swap("-r", d + "/bad2.regions"), swap("-r", d + "/bad3.regions"),
             swap("-1", d + "/reads.1.txt"), swap("-2", d + "/nope.fastq"), swap("-i", d + "/nope.sam")]
    strip = lambda b: b.replace(b"[fai_load] build FASTA index.\n", b"")   # printed when the .fai does not exist yet
    for k, a in enumerate(cases):
        ours = subprocess.run([_tool("dosplitalign")] + a, capture_output=True)
        theirs = util.reference_tool_digest(oracle, "dosplitalign_tool_errors/%d" % k, "ref_dosplitalign",
                                            lambda ref: _exit_1([ref] + a, d, strip))
        assert ours.returncode == 1, a
        assert util.digest(ours.stdout.replace(d.encode(), b"<dir>"), strip(ours.stderr).replace(d.encode(), b"<dir>")) == theirs, a


def test_matealign_input_errors_like_the_reference(tmp_path):
    """matealign's SAM checks and unreadable inputs: they come before any alignment (no GPU needed) and must give the
    compiled reference tool's exit code, stdout and stderr -- with the SAM parsed by chunks on several threads (the
    reference's outputs stored as digests, as above)."""
    import sys
    sys.path.insert(0, ROOT)
    import oracle
    import util
    from synth import files
    d = str(tmp_path / "m")
    args, sam = files.make_matealign_dataset(d, seed=4, n_pairs=50)
    lines = sam.split(b"\n")

    def swap(flag, val):
        a = list(args)
        a[a.index(flag) + 1] = val
        return a

    open(os.path.join(d, "reads.1.txt"), "w").write(open(os.path.join(d, "reads.1.fastq")).read())
    hit = b"\ttr1 some description\t100\t255\t50M\t*\t0\t0\tACGT\tIIII"
    cases = [(swap("-r", d + "/nope.fa"), sam), (swap("-1", d + "/reads.1.txt"), sam), (swap("-2", d + "/nope.fastq"), sam),
             (args, b"\n".join(lines[:10] + [b""] + lines[10:])), (args, b"\n".join(lines[:7] + [b"a\tb\tc"] + lines[7:])),
             (args, b"\n".join(lines[:5] + [b"7/3\t0" + hit] + lines[5:])), (args, b"\n".join(lines[:5] + [b"73\t0" + hit] + lines[5:]))]
    for k, (a, text) in enumerate(cases):
        theirs = util.reference_tool_digest(oracle, "matealign_tool_errors/%d" % k, "ref_matealign",
                                            lambda ref: _exit_1([ref] + a, d, input=text))
        for chunk in ("1", "65536"):
            ours = subprocess.run([_tool("matealign")] + a, input=text, capture_output=True,
                                  env=dict(os.environ, DFB_TOOL_CHUNK_MIN=chunk, DFB_TOOL_THREADS="8"))
            assert ours.returncode == 1, a
            assert util.digest(ours.stdout.replace(d.encode(), b"<dir>"), ours.stderr.replace(d.encode(), b"<dir>")) == theirs, \
                (a, ours.stderr)


def _exit_1(cmd, d, strip=lambda b: b, input=None):
    """stdout and stderr of a run that must exit 1, with the dataset directory `d` written as <dir>."""
    p = subprocess.run(cmd, input=input, capture_output=True)
    assert p.returncode == 1, cmd
    return p.stdout.replace(d.encode(), b"<dir>"), strip(p.stderr).replace(d.encode(), b"<dir>")
