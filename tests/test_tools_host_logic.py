"""Host logic of the drop-in tools without a GPU.

The tools are host code around eight C-ABI calls.  Here the real tool binaries run with tests/device_double (those
eight entry points answered by the parity oracle, preloaded with LD_PRELOAD) in place of the GPU library, and go
through the very test bodies of tests/test_tools_gpu.py and the splitseq tests of tests/test_tools_downstream.py:
golden outputs and byte-for-byte comparison with the compiled reference tools.  What this covers is everything around
the DP -- command line, mapped/chunked ingest, candidate enumeration, task tables, batching, sharding over contexts,
formatting, error exits; the DP itself is covered by the `-m gpu` runs of the same bodies on the B200.
The double is test infrastructure: built into a temporary directory, never next to the tools, and the tools fail
without it on a machine that has no GPU (tests/test_tools_cli.py::test_no_gpu_means_failure_not_fallback)."""
import inspect
import os
import subprocess

import pytest

import test_tools_downstream as td
import test_tools_gpu as tg
import util

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


# the compiled reference tool needs half a minute for this one; the two smaller parameter sets stay
_TOO_SLOW_ON_CPU = {("test_dosplitalign_vs_reference_tool", 0)}


def _cases():
    bodies = [(tg, n) for n in ("test_localalign_golden", "test_dosplitalign_and_matealign_golden",
                                "test_localalign_vs_reference_tool", "test_localalign_errors_like_reference",
                                "test_matealign_vs_reference_tool", "test_dosplitalign_vs_reference_tool",
                                "test_tools_with_many_small_batches",
                                "test_localalign_blocks_pipe_and_mapped_file", "test_matealign_chunked_ingest",
                                "test_localalign_dedup_input_form")]
    bodies += [(td, n) for n in ("test_splitseq_golden", "test_splitseq_vs_reference_tool",
                                 "test_fused_align_evaluate_vs_reference_pipeline")]
    for mod, name in bodies:
        fn = getattr(mod, name)
        marks = [m for m in getattr(fn, "pytestmark", []) if m.name == "parametrize"]
        if not marks:
            yield pytest.param(fn, {}, id=name)
        for m in marks:
            for k, value in enumerate(m.args[1]):
                if (name, k) in _TOO_SLOW_ON_CPU:
                    continue
                yield pytest.param(fn, {m.args[0]: value}, id="%s-%d" % (name, k))


@pytest.mark.parametrize("body,kwargs", list(_cases()))
def test_tool_host_logic(body, kwargs, device_double, oracle_mod, tmp_path, monkeypatch):
    if not os.path.exists(os.path.join(tg.BIN, "dosplitalign")):
        pytest.skip("tools not built")
    monkeypatch.setenv("LD_PRELOAD", device_double)
    monkeypatch.delenv("DFB_DEVICE", raising=False)
    available = {"oracle_mod": oracle_mod, "tmp_path": tmp_path, "device_double": device_double}
    args = {k: available[k] for k in inspect.signature(body).parameters if k in available}
    body(**args, **kwargs)


@pytest.mark.parametrize("devices", ["0,0", "0,1,2,3", "3,1", "all"])
def test_dosplitalign_sharded_over_contexts(devices, device_double, tmp_path, monkeypatch):
    """One context per entry of DFB_DEVICES, candidates dealt out by cluster, results merged in candidate order: the
    output does not depend on the device list.  (The double reports four devices, so distinct ordinals and "all" can
    be exercised here; the GPU run of this test has one device and names it several times.)"""
    import json
    from synth import files
    if not os.path.exists(os.path.join(tg.BIN, "dosplitalign")):
        pytest.skip("tools not built")
    monkeypatch.setenv("LD_PRELOAD", device_double)
    g = json.load(open(os.path.join(HERE, "golden", "tools.json")))
    for name, batch in (("split_small", None), ("split_jitter_lower", "53")):
        sub = str(tmp_path / name)
        args = files.make_split_dataset(sub, **g[name]["kw"])
        res = os.path.join(sub, "ours.alignments")
        env = {"DFB_DEVICES": devices}
        if batch:
            # several batches; SAM chunks of a few lines and the bucketed de-duplication on every thread
            env.update(DFB_TOOL_BATCH=batch, DFB_TOOL_CHUNK_MIN="300", DFB_TOOL_THREADS="5")
        tg._run([os.path.join(tg.BIN, "dosplitalign")] + args + ["-a", res], env=env)
        assert open(res).read() == g[name]["output"], (name, devices)


def test_missing_device_is_an_error(device_double, tmp_path, monkeypatch):
    """A device ordinal the library does not have: the tool reports the library's message and exits 1."""
    import json
    from synth import files
    monkeypatch.setenv("LD_PRELOAD", device_double)
    g = json.load(open(os.path.join(HERE, "golden", "tools.json")))
    args = files.make_split_dataset(str(tmp_path / "s"), **g["split_small"]["kw"])
    p = subprocess.run([os.path.join(tg.BIN, "dosplitalign")] + args + ["-a", str(tmp_path / "out")], capture_output=True,
                       env=dict(os.environ, DFB_DEVICES="0,7"))
    assert p.returncode == 1 and b"Error:" in p.stderr


@pytest.mark.parametrize("tool", ["dosplitalign", "matealign", "localalign", "evalsplitalign", "splitseq"])
def test_input_fuzz_agrees_with_the_reference_tool(tool, oracle_mod):
    """scripts/cpu_fuzz_tools.py, a fixed number of rounds: perturbed inputs (odd but legal records and malformed ones),
    our tool over the device double against the compiled reference tool -- exit codes, outputs, messages."""
    import json
    import sys
    if not os.path.exists(os.path.join(tg.BIN, tool)):
        pytest.skip("tools not built")
    if not oracle_mod.ref_tool("ref_" + tool):
        # (the reference's outcomes on malformed inputs -- signals, its own DebugCheck messages -- are not ours to derive)
        pytest.skip("needs the compiled reference tools (oracle/_ref)")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "cpu_fuzz_tools.py"), tool, "5", "120", "60"],
                       capture_output=True, timeout=600)
    report = json.loads(p.stdout.decode())
    assert report["rounds"] == 60 and not report["disagreements"], report["disagreements"][:2]
    assert report["reference_exit_0"] > 5 and report["reference_exit_1"] > 5  # both kinds of outcome were exercised


def test_dosplitalign_baseline_config_0(device_double, oracle_mod, tmp_path, monkeypatch):
    """BASELINE.json configs[0] ("dosplitalign on synthetic 2k read pairs x 200 planted-fusion breakpoint clusters, 100 bp
    reads"): the whole tool against the compiled reference tool, byte for byte, raw and after the pipeline's sort."""
    from synth import files
    if not os.path.exists(os.path.join(tg.BIN, "dosplitalign")):
        pytest.skip("tools not built")
    monkeypatch.setenv("LD_PRELOAD", device_double)
    d = str(tmp_path / "c0")
    args = files.make_split_dataset(d, seed=1, n_clusters=200, pairs_per_cluster=10, L=100, n_chrom=4, genes_per_chrom=10)
    ours, theirs = os.path.join(d, "ours.tmp"), os.path.join(d, "ref.tmp")
    want = util.reference_tool_digest(oracle_mod, "dosplitalign_tool/baseline_config_0", "ref_dosplitalign",
                         lambda ref: tg._output_file([ref] + args + ["-a", theirs], theirs))
    tg._run([os.path.join(tg.BIN, "dosplitalign")] + args + ["-a", ours])
    a = open(ours, "rb").read()
    assert len(a.splitlines()) > 200 and util.digest(a) == want


def test_dosplitalign_stress_shape(device_double, oracle_mod, tmp_path, monkeypatch):
    """BASELINE.json configs[4] shape at file level: 250-bp reads (-n 230 -x 270 with jitter), 600-bp fragments, N and
    lower-case runs in the reference -- windows, candidates and records against the compiled reference tool."""
    from synth import files
    if not os.path.exists(os.path.join(tg.BIN, "dosplitalign")):
        pytest.skip("tools not built")
    monkeypatch.setenv("LD_PRELOAD", device_double)
    d = str(tmp_path / "c4")
    args = files.make_split_dataset(d, seed=5, n_clusters=30, pairs_per_cluster=16, L=250, frag_mean=600, read_len_jitter=20,
                                    lower_frac=0.01, n_rate=0.01)
    ours, theirs = os.path.join(d, "ours.tmp"), os.path.join(d, "ref.tmp")
    want = util.reference_tool_digest(oracle_mod, "dosplitalign_tool/stress_shape", "ref_dosplitalign",
                         lambda ref: tg._output_file([ref] + args + ["-a", theirs], theirs))
    tg._run([os.path.join(tg.BIN, "dosplitalign")] + args + ["-a", ours])
    a = open(ours, "rb").read()
    assert len(a.splitlines()) > 50 and util.digest(a) == want
