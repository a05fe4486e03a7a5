"""The four-lane class <4,25>: reads of 81-100 bases run in groups of 4 lanes x 25 rows, with 32-step checkpoint blocks
(not 4G = 16) and 64-column ring blocks decoded 16 columns per lane.  Bit-exact against the oracle at the class boundary,
at the edges of the checkpoint interval, with exceptions and ties, on every path that runs the class."""
import numpy as np
import pytest

import util
from test_gpu_parity import _check_simple, _check_split, _tables

pytestmark = pytest.mark.gpu


def _ms(reads, trd):
    import defuse_b200 as d
    return np.array([d.split_min_score(len(reads[r])) for r in trd], np.int32)


def _split(rng, n_clusters, per_cluster, L, r_lo, r_hi, **kw):
    kw.setdefault("indel", 0.0)  # (indels change a read's length: the lengths here are the point)
    return util.split_batch(rng, n_clusters, per_cluster, L, r_lo, r_hi, **kw)


def _kernels_run(fn):
    """names of the CUDA kernels fn launches"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events()}


@pytest.mark.parametrize("L", [81, 88, 99, 100, 101, 104])
def test_read_lengths_at_the_class_boundary(oracle_mod, gpu_ctx, L):
    rng = np.random.default_rng(500 + L)
    refs, reads, tc, trd = _split(rng, 24, 12, L, 150, 420)
    assert {len(r) for r in reads} == {L}
    _check_split(oracle_mod, gpu_ctx, refs, reads, tc, trd, _ms(reads, trd))


@pytest.mark.parametrize("L,four_lane", [(81, True), (100, True), (101, False)])
def test_which_class_serves_the_reads(gpu_ctx, L, four_lane):
    """81-100 bases run on dp_fast_kernel<4, 25, ...> (and its probe sweep), 101 on <8, 13>."""
    import defuse_b200 as d
    rng = np.random.default_rng(600 + L)
    refs, reads, tc, trd = _split(rng, 40, 25, L, 250, 400)
    rt, st = _tables(refs, reads)
    al = d.SplitReadAligner(ctx=gpu_ctx)
    names = _kernels_run(lambda: al.align_batch(rt, st, tc, trd, _ms(reads, trd)))
    fast = {n for n in names if "dp_fast_kernel" in n or "dp_probe_kernel" in n}
    four = {n for n in fast if "<4, 25" in n}
    eight = {n for n in fast if "<8, 13" in n}
    assert fast, names
    if four_lane:
        assert four and not eight, fast
        assert any("dp_probe_kernel" in n for n in four), fast
    else:
        assert eight and not four, fast
    names = _kernels_run(lambda: d.SimpleAligner(10, -5, -5, ctx=gpu_ctx).align_batch(rt, st, tc * 2, trd))
    assert any("<4, 25" in n for n in names) == four_lane, names


@pytest.mark.parametrize("windows", [(1, 31), (31, 34), (62, 67), (94, 99), (126, 131), (190, 194)])
def test_windows_at_the_checkpoint_interval(oracle_mod, gpu_ctx, windows):
    """windows shorter than one 32-step block, and k*32, k*32 +- 1 (wavefront R + 3 steps)"""
    rng = np.random.default_rng(700 + windows[0])
    refs, reads, tc, trd = _split(rng, 40, 10, (81, 100), *windows)
    _check_split(oracle_mod, gpu_ctx, refs, reads, tc, trd, _ms(reads, trd))


def test_window_pairs_differing_by_up_to_40(oracle_mod, gpu_ctx):
    """the two windows of a cluster end at different steps: tail steps of the shorter half"""
    rng = np.random.default_rng(81)
    refs, reads, tc, trd = _split(rng, 30, 10, 100, 200, 240)
    _check_split(oracle_mod, gpu_ctx, refs, reads, tc, trd, _ms(reads, trd))


def test_long_windows_with_coarse_granules(oracle_mod, gpu_ctx):
    """windows of 500-1200 columns: more than 15 checkpoint blocks, so a probe granule spans 2 or 4 of them"""
    rng = np.random.default_rng(82)
    refs, reads, tc, trd = _split(rng, 16, 10, (85, 100), 500, 1200)
    _check_split(oracle_mod, gpu_ctx, refs, reads, tc, trd, _ms(reads, trd))


def test_exceptions_and_lowercase(oracle_mod, gpu_ctx):
    rng = np.random.default_rng(83)
    refs, reads, tc, trd = _split(rng, 30, 10, (81, 100), 100, 400, n_rate=0.03)
    refs = [r.lower() if k % 3 == 0 else r for k, r in enumerate(refs)]
    reads = [r[:20].lower() + r[20:] if k % 4 == 0 else r for k, r in enumerate(reads)]
    _check_split(oracle_mod, gpu_ctx, refs, reads, tc, trd, _ms(reads, trd))


def test_poly_a_ties_and_many_rounds(oracle_mod, gpu_ctx):
    """poly-A reads against poly-A-rich windows: many tied columns (past the 16-entry regions) and rows that reach
    their maxima in several granules (multi-round probes), in the same warps as one-round jobs"""
    rng = np.random.default_rng(84)
    refs, reads, tc, trd = _split(rng, 20, 12, (90, 100), 200, 600)
    for c in range(0, 20, 2):
        for h in (0, 1):
            r = bytearray(refs[2 * c + h])
            for s in range(0, len(r) - 40, 90):
                r[s:s + 40] = b"A" * 40
            refs[2 * c + h] = bytes(r)
    for k in range(0, len(reads), 3):
        reads[k] = b"A" * len(reads[k])
    _check_split(oracle_mod, gpu_ctx, refs, reads, tc, trd, _ms(reads, trd))


@pytest.mark.parametrize("build", ["DFB_DEVICE_BUILD", "DFB_HOST_BUILD"])
def test_job_list_builds_and_paths(oracle_mod, gpu_ctx, monkeypatch, build):
    """device- and host-built job lists, the pipelined one-call path, the resident plan and the device-resident form"""
    import defuse_b200 as d
    monkeypatch.setenv(build, "1")
    monkeypatch.setenv("DFB_PIPELINE_MIN_TASKS", "16")
    rng = np.random.default_rng(85)
    refs, reads, tc, trd = _split(rng, 40, 20, (81, 100), 60, 500, n_rate=0.01)
    ms = _ms(reads, trd)
    piped = _check_split(oracle_mod, gpu_ctx, refs, reads, tc, trd, ms)
    rt, st = _tables(refs, reads)
    al = d.SplitReadAligner(ctx=gpu_ctx)
    plan = al.plan(rt, st, tc, trd, ms)
    plan.run()
    whole = plan.fetch()
    plan.close()
    assert np.array_equal(piped.best, whole.best)
    for f in ("task", "read_split", "score1", "score2", "n1", "n2"):
        assert np.array_equal(piped.rows[f], whole.rows[f]), f
    import torch
    dev = al.align_device(d.DeviceSeqTable.from_host(rt, "cuda:0"), d.DeviceSeqTable.from_host(st, "cuda:0"),
                          *(torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).cuda() for a in (tc, trd, ms)))
    got = dev.to_host()
    assert np.array_equal(got.best, piped.best)
    assert got.rows.tobytes() == piped.rows.tobytes()


def test_simple_aligner_at_100(oracle_mod, gpu_ctx):
    """localalign's shape (10/-5/-5, L = 100): the four-lane class serves SimpleAligner too"""
    rng = np.random.default_rng(86)
    refs, seqs, tr, ts = util.simple_batch(rng, 8, 400, (60, 2001), (81, 100), indel=0.0)
    _check_simple(oracle_mod, gpu_ctx, refs, seqs, tr, ts, 10, -5, -5)
    _check_simple(oracle_mod, gpu_ctx, refs, seqs, tr, ts, 2, -1, -2)
