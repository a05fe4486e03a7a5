"""Parity tests proper: the CUDA path (through the C ABI) against the oracle on the same seeded inputs.
Bit-exact: scores, split positions, column sets, emission order."""
import numpy as np
import pytest

import util

pytestmark = pytest.mark.gpu


def _tables(refs, seqs):
    import defuse_b200 as d
    return d.SeqTable.from_list(refs), d.SeqTable.from_list(seqs)


def _check_simple(oracle, ctx, refs, seqs, task_ref, task_seq, m, x, g):
    import defuse_b200 as d
    rt, st = _tables(refs, seqs)
    got = d.SimpleAligner(m, x, g, ctx=ctx).align_batch(rt, st, task_ref, task_seq)
    want = oracle.simple_align_batch(m, x, g, rt.data, rt.off, st.data, st.off, task_ref, task_seq)
    bad = np.nonzero(got != want)[0]
    assert bad.size == 0, "first mismatch task %d: got %d want %d (R=%d L=%d)" % (
        bad[0], got[bad[0]], want[bad[0]], len(refs[task_ref[bad[0]]]), len(seqs[task_seq[bad[0]]]))
    # the compiled reference class itself as the checker (oracle/_ref travels to the GPU box), on a bounded sample
    if oracle.have_ref():
        pick = _ref_sample(len(task_ref), lambda t: len(refs[task_ref[t]]) * len(seqs[task_seq[t]]))
        ref = oracle.simple_align_batch(m, x, g, rt.data, rt.off, st.data, st.off, np.asarray(task_ref)[pick],
                                        np.asarray(task_seq)[pick], impl="ref")
        assert (got[pick] == ref).all(), "CUDA path differs from the compiled reference SimpleAligner"


def _ref_sample(n, cells_of, budget=4.0e8):
    """Tasks the unmodified reference classes re-check directly: evenly spread, about `budget` DP cells in total
    (a few seconds at the reference's rate)."""
    if n == 0:
        return np.zeros(0, np.int64)
    step = 1
    total = sum(cells_of(t) for t in range(0, n, max(1, n // 64))) * max(1, n // 64)
    if total > budget:
        step = int(np.ceil(total / budget))
    return np.arange(0, n, step, dtype=np.int64)


def _check_split(oracle, ctx, refs, reads, task_cluster, task_read, min_score, params=(2, -1, -2, False, 8)):
    import defuse_b200 as d
    rt, st = _tables(refs, reads)
    m, x, g, eg, ms = params
    res = d.SplitReadAligner(m, x, g, eg, ms, ctx=ctx).align_batch(rt, st, task_cluster, task_read, min_score)
    cnt, want = oracle.split_align_batch(rt.data, rt.off, st.data, st.off, task_cluster, task_read, min_score,
                                         m, x, g, eg, ms)
    pos = np.concatenate([[0], np.cumsum(cnt)])
    for t in range(len(task_cluster)):
        w = want[pos[t]:pos[t + 1]]
        a = res.alignments(t)
        assert a.shape == w.shape and (a == w).all(), "task %d: got\n%s\nwant\n%s" % (t, a[:8], w[:8])
        assert res.best[t] == (w[0, 4] if len(w) else res.best[t])
        rec = res.records(t)
        wrec = oracle.split_dedupe(w)
        assert rec.shape == wrec.shape and (rec == wrec).all()
    # the compiled reference class itself as the checker, on a bounded sample of the tasks
    if oracle.have_ref():
        tc, tr, mn = np.asarray(task_cluster), np.asarray(task_read), np.asarray(min_score)
        pick = _ref_sample(len(tc), lambda t: len(reads[tr[t]]) * (len(refs[2 * tc[t]]) + len(refs[2 * tc[t] + 1])))
        pick = pick[cnt[pick] <= 20000]  # (tie-heavy tasks: millions of tuples through the reference's vectors)
        rcnt, rwant = oracle.split_align_batch(rt.data, rt.off, st.data, st.off, tc[pick], tr[pick], mn[pick],
                                               m, x, g, eg, ms, impl="ref")
        rpos = np.concatenate([[0], np.cumsum(rcnt)])
        for k, t in enumerate(pick):
            w = rwant[rpos[k]:rpos[k + 1]]
            a = res.alignments(int(t))
            assert a.shape == w.shape and (a == w).all(), "task %d differs from the compiled reference SplitReadAligner" % t
    return res


@pytest.mark.parametrize("scoring", [(10, -5, -5), (2, -1, -2), (1, 0, 0), (5, -3, -2), (3, 0, -1)])
def test_simple_random(oracle_mod, gpu_ctx, scoring):
    rng = np.random.default_rng(11)
    refs, seqs, tr, ts = util.simple_batch(rng, 40, 600, (1, 700), (1, 260))
    _check_simple(oracle_mod, gpu_ctx, refs, seqs, tr, ts, *scoring)


def test_simple_localalign_shape(oracle_mod, gpu_ctx):
    rng = np.random.default_rng(12)
    refs, seqs, tr, ts = util.simple_batch(rng, 8, 300, 2001, (90, 110))
    _check_simple(oracle_mod, gpu_ctx, refs, seqs, tr, ts, 10, -5, -5)


def test_simple_long_reads(oracle_mod, gpu_ctx):
    rng = np.random.default_rng(13)
    refs, seqs, tr, ts = util.simple_batch(rng, 6, 60, (800, 1500), (250, 1024))
    _check_simple(oracle_mod, gpu_ctx, refs, seqs, tr, ts, 2, -1, -2)


def test_simple_edge_cases(oracle_mod, gpu_ctx):
    refs = [b"", b"A", b"ACGTN", b"ACGT", b"acgtacgtNNNNacgt", b"A" * 300, bytes(range(1, 200)), b"GATTACA" * 30]
    seqs = [b"", b"A", b"GTN", b"acgt", b"NNNN", b"A" * 120, bytes(range(50, 120)), b"TACAGATT", b"N" * 17, b"ACGT" * 70]
    tr, ts = np.meshgrid(np.arange(len(refs)), np.arange(len(seqs)))
    for sc in [(10, -5, -5), (2, -1, -2)]:
        _check_simple(oracle_mod, gpu_ctx, refs, seqs, tr.ravel().astype(np.int32), ts.ravel().astype(np.int32), *sc)


@pytest.mark.parametrize("scoring", [(1, -1, 1), (0, 0, 0), (-1, -2, -3), (2, 1, -1), (300, -200, -250), (2, -1, 0),
                                     (3, 3, 3)])
def test_simple_generic_scoring(oracle_mod, gpu_ctx, scoring):
    rng = np.random.default_rng(14)
    refs, seqs, tr, ts = util.simple_batch(rng, 10, 120, (1, 300), (1, 300))
    _check_simple(oracle_mod, gpu_ctx, refs, seqs, tr, ts, *scoring)


def test_simple_generic_very_long(oracle_mod, gpu_ctx):
    rng = np.random.default_rng(15)
    refs, seqs, tr, ts = util.simple_batch(rng, 3, 8, (1500, 3000), (1025, 2100))
    _check_simple(oracle_mod, gpu_ctx, refs, seqs, tr, ts, 10, -5, -5)


def test_split_planted(oracle_mod, gpu_ctx):
    import defuse_b200 as d
    rng = np.random.default_rng(21)
    refs, reads, tc, trd = util.split_batch(rng, 30, 12, 100, 280, 420)
    ms = np.array([d.split_min_score(len(reads[r])) for r in trd], np.int32)
    res = _check_split(oracle_mod, gpu_ctx, refs, reads, tc, trd, ms)
    assert (res.best > 0).sum() > 50  # the planted junctions are found


def test_split_varied_lengths(oracle_mod, gpu_ctx):
    import defuse_b200 as d
    rng = np.random.default_rng(22)
    refs, reads, tc, trd = util.split_batch(rng, 25, 10, (20, 260), 60, 700, sub=0.03, indel=0.01, n_rate=0.01)
    ms = np.array([d.split_min_score(len(reads[r])) for r in trd], np.int32)
    _check_split(oracle_mod, gpu_ctx, refs, reads, tc, trd, ms)


def test_split_zero_threshold_ties(oracle_mod, gpu_ctx):
    rng = np.random.default_rng(23)
    refs, reads, tc, trd = util.split_batch(rng, 12, 6, (8, 60), 10, 90, sub=0.05)
    _check_split(oracle_mod, gpu_ctx, refs, reads, tc, trd, np.zeros(len(tc), np.int32))


def test_split_edge_cases(oracle_mod, gpu_ctx):
    import defuse_b200 as d
    polyA = b"A" * 120
    refs = [polyA, polyA,                       # poly-A vs poly-A windows: huge tie sets
            b"ACGT" * 40, b"TTGCA" * 30,        # tandem repeats
            b"", b"ACGTACGTAC",                 # empty reference 1
            b"ACGTTGCANNNNACGT" * 10, b"acgtNNNNACGTTTGA" * 9,  # N and lowercase
            b"GATTACAGATTACA", b"CATCATCAT"]    # windows shorter than the read
    reads = [b"A" * 60, b"ACGT" * 10 + b"TTGCA" * 8, b"", b"ACGTNNNNACGTacgtNNNNACGT", b"GATTACA" * 5, b"N" * 30,
             b"ACGTACGTACGTAAAAAAAAAAAAAAAAAAAA", b"T"]
    tc, trd = np.meshgrid(np.arange(len(refs) // 2), np.arange(len(reads)))
    tc, trd = tc.ravel().astype(np.int32), trd.ravel().astype(np.int32)
    for ms in (np.zeros(len(tc), np.int32), np.array([d.split_min_score(len(reads[r])) for r in trd], np.int32)):
        _check_split(oracle_mod, gpu_ctx, refs, reads, tc, trd, ms)


@pytest.mark.parametrize("params", [(2, -1, -2, True, 8), (2, -1, -2, False, 0), (2, -1, -2, False, -3),
                                    (1, -1, 1, False, 4), (3, 1, -2, True, 0), (300, -200, -250, False, 1200),
                                    (0, 0, 0, False, 0)])
def test_split_generic_params(oracle_mod, gpu_ctx, params):
    rng = np.random.default_rng(24)
    refs, reads, tc, trd = util.split_batch(rng, 6, 5, (5, 40), 8, 70, sub=0.05)
    m = params[0]
    ms = np.array([int(0.9 * m * len(reads[r])) for r in trd], np.int32)
    _check_split(oracle_mod, gpu_ctx, refs, reads, tc, trd, ms, params)
    _check_split(oracle_mod, gpu_ctx, refs, reads, tc, trd, np.zeros(len(tc), np.int32), params)


def test_split_generic_long_read(oracle_mod, gpu_ctx):
    import defuse_b200 as d
    rng = np.random.default_rng(25)
    refs, reads, tc, trd = util.split_batch(rng, 2, 2, (1030, 1200), 1300, 1500)
    ms = np.array([d.split_min_score(len(reads[r])) for r in trd], np.int32)
    _check_split(oracle_mod, gpu_ctx, refs, reads, tc, trd, ms)


def test_staged_plan_matches_one_call(oracle_mod, gpu_ctx):
    import defuse_b200 as d
    rng = np.random.default_rng(26)
    refs, seqs, tr, ts = util.simple_batch(rng, 10, 500, (300, 600), (80, 120))
    rt, st = _tables(refs, seqs)
    al = d.SimpleAligner(10, -5, -5, ctx=gpu_ctx)
    plan = al.plan(rt, st, tr, ts)
    for _ in range(3):  # re-running a resident plan overwrites its outputs
        plan.run()
    got = plan.fetch()
    want = oracle_mod.simple_align_batch(10, -5, -5, rt.data, rt.off, st.data, st.off, tr, ts)
    assert (got == want).all()
    st_ = plan.stats()
    assert st_["cells"] == sum(len(refs[a]) * len(seqs[b]) for a, b in zip(tr, ts))
    assert st_["kernel_launches"] >= 1 and st_["fast_jobs"] > 0
    plan.close()


@pytest.mark.parametrize("pipelined", [False, True])
def test_event_buffer_overflow_is_recovered(oracle_mod, gpu_ctx, monkeypatch, pipelined):
    """poly-A windows give ~R arg-max columns per row and ~L tie rows: far more than the default
    event buffer share; the fetch must notice, re-size and re-sweep.  A chunk of a pipelined batch has given its
    checkpoints back by then and runs both sweeps again."""
    if pipelined:
        monkeypatch.setenv("DFB_PIPELINE_MIN_TASKS", "16")
        monkeypatch.setenv("DFB_DEVICE_BUILD", "1")
    polyA = b"A" * 700
    refs = [polyA, polyA]
    reads = [b"A" * 200] * 24
    tc = np.zeros(len(reads), np.int32)
    trd = np.arange(len(reads), dtype=np.int32)
    import defuse_b200 as d
    rt, st = _tables(refs, reads)
    res = d.SplitReadAligner(ctx=gpu_ctx).align_batch(rt, st, tc, trd, np.full(len(reads), 360, np.int32))
    n_want, best_want = oracle_mod.split_align_count(reads[0], refs[0], refs[1], 360)
    # compare the factorised form (the expansion is ~R*R*L tuples)
    for t in (0, len(reads) - 1):
        rows = res.rows[res.rows["task"] == t]
        assert res.best[t] == best_want
        assert sum(int(r["n1"]) * int(r["n2"]) for r in rows) == n_want
    assert len(res.cols) > (1 << 20)  # more events than the initial buffer held


def test_large_batch_properties_and_sampled_parity(oracle_mod, gpu_ctx):
    """A bench-sized shard (200 k tasks, the shape of BASELINE.json configs[2]): size-independent properties on every
    task, full oracle parity on a random sample, and identical results from the resident plan and the one-call API."""
    import defuse_b200 as d
    import synth
    w = synth.split_workload(9, 2000, 100)
    refs, reads = d.SeqTable(w["ref_bytes"], w["ref_off"]), d.SeqTable(w["read_bytes"], w["read_off"])
    al = d.SplitReadAligner(ctx=gpu_ctx)
    res = al.align_batch(refs, reads, w["task_cluster"], w["task_read"], w["min_score"])
    n, L = w["n_tasks"], w["L"]
    rows = res.rows
    assert np.all(np.diff(rows["task"]) >= 0)                                    # task order
    assert np.all(rows["score1"] + rows["score2"] == res.best[rows["task"]])      # every winning row attains the best total
    assert np.all((res.best == 0) | ((res.best >= w["min_score"]) & (res.best <= 2 * L)))
    assert np.all((rows["read_split"] >= 1) & (rows["read_split"] <= L - 1))
    assert np.all((rows["score1"] >= 8) & (rows["score2"] >= 8))                  # minSplitScore floor on both sides
    assert np.all((rows["n1"] >= 1) & (rows["n2"] >= 1))
    assert np.all(res.best[np.setdiff1d(np.arange(n), rows["task"])] >= 0)
    same = rows["task"][1:] == rows["task"][:-1]
    assert np.all(rows["read_split"][1:][same] > rows["read_split"][:-1][same])   # ascending tie rows inside a task
    ref_len = w["ref_off"][1:] - w["ref_off"][:-1]
    r1 = ref_len[2 * w["task_cluster"].astype(np.int64)][rows["task"]]
    first_col = res.cols[rows["col_begin"]]
    assert np.all((first_col >= 1) & (first_col <= r1))
    # the resident plan gives the same answer, run after run
    plan = al.plan(refs, reads, w["task_cluster"], w["task_read"], w["min_score"])
    for _ in range(2):
        plan.run()
        r2 = plan.fetch()
        assert np.array_equal(r2.best, res.best) and np.array_equal(r2.rows, rows) and np.array_equal(r2.cols, res.cols)
    plan.close()
    # sampled full parity
    rng = np.random.default_rng(0)
    sample = np.sort(rng.choice(n, 400, replace=False)).astype(np.int32)
    cnt, want = oracle_mod.split_align_batch(w["ref_bytes"], w["ref_off"], w["read_bytes"], w["read_off"],
                                             w["task_cluster"][sample], w["task_read"][sample], w["min_score"][sample])
    pos = np.concatenate([[0], np.cumsum(cnt)])
    for k, t in enumerate(sample):
        a = res.alignments(int(t))
        b = want[pos[k]:pos[k + 1]]
        assert a.shape == b.shape and (a == b).all(), t


def test_split_stress_config_as_specified(oracle_mod, gpu_ctx):
    """SURVEY 8(d) config 5 as written (synth.STRESS): 250-bp reads, 8 % substitutions, 2 % indels, 1 % N, 5 % poly-A
    tails, lowercase runs in the windows, poly-A window ends, Zipf(1.2) cluster sizes.  Every task against the oracle,
    a sample against the compiled reference class; the exception plane (N, lowercase) and the tie-heavy overflow path
    (poly-A read tail against a poly-A window end) must both occur."""
    import defuse_b200 as d
    import synth
    w = synth.split_workload(5, 150, 40, **synth.STRESS)
    n = w["n_tasks"]
    refs, reads = d.SeqTable(w["ref_bytes"], w["ref_off"]), d.SeqTable(w["read_bytes"], w["read_off"])
    res = d.SplitReadAligner(ctx=gpu_ctx).align_batch(refs, reads, w["task_cluster"], w["task_read"], w["min_score"])
    cnt, want = oracle_mod.split_align_batch(w["ref_bytes"], w["ref_off"], w["read_bytes"], w["read_off"],
                                             w["task_cluster"], w["task_read"], w["min_score"])
    pos = np.concatenate([[0], np.cumsum(cnt)])
    for t in range(n):
        a = res.alignments(t)
        b = want[pos[t]:pos[t + 1]]
        assert a.shape == b.shape and (a == b).all(), t
    assert (cnt > 0).sum() > n // 50                      # junctions are still found at this error rate
    assert cnt.max() > 64                                  # a tie-heavy task went through the overflow list
    assert (w["ref_bytes"] >= 97).any() and (w["read_bytes"] == ord("N")).any()
    if oracle_mod.have_ref():
        pick = np.unique(np.concatenate([np.arange(0, n, 40), np.argsort(cnt)[-5:]])).astype(np.int32)
        rcnt, rwant = oracle_mod.split_align_batch(w["ref_bytes"], w["ref_off"], w["read_bytes"], w["read_off"],
                                                   w["task_cluster"][pick], w["task_read"][pick], w["min_score"][pick], impl="ref")
        rpos = np.concatenate([[0], np.cumsum(rcnt)])
        for k, t in enumerate(pick):
            a = res.alignments(int(t))
            b = rwant[rpos[k]:rpos[k + 1]]
            assert a.shape == b.shape and (a == b).all(), t


def _expand_cols(res):
    """Per row, its column list as a fixed-width array (padded with -1): layout-independent comparison of results."""
    rows, cols = res.rows, res.cols
    width = int((rows["n1"] + rows["n2"]).max()) if len(rows) else 0
    out = np.full((len(rows), width), -1, dtype=np.int64)
    for k in range(width):
        m = (rows["n1"] + rows["n2"]) > k
        out[m, k] = cols[rows["col_begin"][m] + k]
    return out


@pytest.mark.parametrize("build", ["device", "host"])
def test_full_size_batch_pipelined_equals_resident(oracle_mod, gpu_ctx, monkeypatch, build):
    """BASELINE.json configs[2] at the size bench.py runs (2 M tasks): the one-call path cuts it into eight tapered chunks
    whose rows go straight into the batch's result arrays -- job lists built on the device or on the host --; the resident
    plan assembles the same batch in one piece.  Same rows, same column lists, task by task; size-independent properties
    on every row; sampled oracle parity."""
    import defuse_b200 as d
    import synth
    monkeypatch.setenv("DFB_DEVICE_BUILD" if build == "device" else "DFB_HOST_BUILD", "1")
    w = synth.split_workload(21, 20000, 100)
    refs, reads = d.SeqTable(w["ref_bytes"], w["ref_off"]), d.SeqTable(w["read_bytes"], w["read_off"])
    al = d.SplitReadAligner(ctx=gpu_ctx)
    piped = al.align_batch(refs, reads, w["task_cluster"], w["task_read"], w["min_score"])
    plan = al.plan(refs, reads, w["task_cluster"], w["task_read"], w["min_score"])
    plan.run()
    whole = plan.fetch()
    plan.close()
    assert np.array_equal(piped.best, whole.best)
    assert len(piped.rows) == len(whole.rows) > 10 ** 6
    for f in ("task", "read_split", "score1", "score2", "n1", "n2"):
        assert np.array_equal(piped.rows[f], whole.rows[f]), f
    assert np.array_equal(_expand_cols(piped), _expand_cols(whole))
    rows, L = piped.rows, w["L"]
    assert np.all(np.diff(rows["task"]) >= 0)
    assert np.all(rows["score1"] + rows["score2"] == piped.best[rows["task"]])
    assert np.all((piped.best == 0) | ((piped.best >= w["min_score"]) & (piped.best <= 2 * L)))
    assert np.all((rows["n1"] >= 1) & (rows["n2"] >= 1) & (rows["col_begin"] >= 0))
    assert int((rows["col_begin"] + rows["n1"] + rows["n2"]).max()) <= len(piped.cols)
    sample = np.sort(np.random.default_rng(2).choice(w["n_tasks"], 300, replace=False)).astype(np.int32)
    cnt, want = oracle_mod.split_align_batch(w["ref_bytes"], w["ref_off"], w["read_bytes"], w["read_off"],
                                             w["task_cluster"][sample], w["task_read"][sample], w["min_score"][sample])
    pos = np.concatenate([[0], np.cumsum(cnt)])
    for k, t in enumerate(sample):
        a = piped.alignments(int(t))
        b = want[pos[k]:pos[k + 1]]
        assert a.shape == b.shape and (a == b).all(), t


def test_large_simple_batch_sampled_parity(oracle_mod, gpu_ctx):
    import defuse_b200 as d
    import synth
    w = synth.local_workload(12, 500, 60000, 2001, 100)
    refs, seqs = d.SeqTable(w["ref_bytes"], w["ref_off"]), d.SeqTable(w["seq_bytes"], w["seq_off"])
    got = d.SimpleAligner(10, -5, -5, ctx=gpu_ctx).align_batch(refs, seqs, w["task_ref"], w["task_seq"])
    assert np.all((got >= 0) & (got <= 1000))
    sample = np.sort(np.random.default_rng(1).choice(w["n_tasks"], 300, replace=False)).astype(np.int32)
    want = oracle_mod.simple_align_batch(10, -5, -5, w["ref_bytes"], w["ref_off"], w["seq_bytes"], w["seq_off"],
                                         w["task_ref"][sample], w["task_seq"][sample])
    assert np.array_equal(got[sample], want)


def test_pipelined_simple_batch(oracle_mod, gpu_ctx, monkeypatch):
    """dfb_simple_align_batch cuts large batches (non-decreasing task_seq) into chunks: forced here on small batches,
    with references named in any order (localalign: the whole table per chunk), references in task order (matealign:
    a view per chunk), empty sequences and the generic (s32) kernels.  Same scores as the single plan and the oracle."""
    import defuse_b200 as d
    rng = np.random.default_rng(41)
    refs, seqs, tr, ts = util.simple_batch(rng, 30, 700, (1, 600), (0, 260))
    for scoring in [(10, -5, -5), (2, 1, -1)]:
        monkeypatch.delenv("DFB_PIPELINE_MIN_TASKS", raising=False)
        rt, st = _tables(refs, seqs)
        al = d.SimpleAligner(*scoring, ctx=gpu_ctx)
        single = al.align_batch(rt, st, tr, ts)
        monkeypatch.setenv("DFB_PIPELINE_MIN_TASKS", "16")
        assert np.array_equal(al.align_batch(rt, st, tr, ts), single)
        _check_simple(oracle_mod, gpu_ctx, refs, seqs, tr, ts, *scoring)
        # one reference per task, in task order
        refs2 = [refs[r] for r in tr]
        tr2 = np.arange(len(tr), dtype=np.int32)
        _check_simple(oracle_mod, gpu_ctx, refs2, seqs, tr2, ts, *scoring)
        # decreasing task_seq: single plan
        assert np.array_equal(al.align_batch(rt, st, tr[::-1].copy(), ts[::-1].copy()), single[::-1])


def test_pipelined_one_call_path(oracle_mod, gpu_ctx, monkeypatch):
    """dfb_split_align_batch cuts large batches (non-decreasing task_read) into chunks that overlap host and GPU work;
    forced here on a small batch.  Results must equal the single-plan path and the oracle, including shared reads
    across a chunk boundary, empty reads and the generic (s32) path."""
    import defuse_b200 as d
    rng = np.random.default_rng(31)
    refs, reads, tc, trd = util.split_batch(rng, 40, 25, (0, 120), 60, 400, sub=0.02, indel=0.005, n_rate=0.01)
    # clusters and reads both non-decreasing (dosplitalign's order): every chunk gets a view of the window table too,
    # chunk boundaries fall inside clusters; both job-list builds, and a batch that starts at a later cluster
    assert np.all(np.diff(tc) >= 0) and np.all(np.diff(trd) >= 0)
    ms0 = np.array([d.split_min_score(len(reads[r])) for r in trd], np.int32)
    for knob in ("DFB_DEVICE_BUILD", "DFB_HOST_BUILD"):
        monkeypatch.setenv("DFB_PIPELINE_MIN_TASKS", "16")
        monkeypatch.setenv(knob, "1")
        _check_split(oracle_mod, gpu_ctx, refs, reads, tc, trd, ms0)
        _check_split(oracle_mod, gpu_ctx, refs, reads, tc[333:], trd[333:], ms0[333:])
        monkeypatch.delenv(knob)
        monkeypatch.delenv("DFB_PIPELINE_MIN_TASKS")
    # several tasks per read (same read against neighbouring clusters), still non-decreasing
    tc = np.concatenate([tc, (tc + 1) % 40]).astype(np.int32)
    trd = np.concatenate([trd, trd]).astype(np.int32)
    order = np.argsort(trd, kind="stable")
    tc, trd = tc[order], trd[order]
    ms = np.array([d.split_min_score(len(reads[r])) for r in trd], np.int32)
    rt, st = _tables(refs, reads)
    al = d.SplitReadAligner(ctx=gpu_ctx)
    single = al.align_batch(rt, st, tc, trd, ms)
    monkeypatch.setenv("DFB_PIPELINE_MIN_TASKS", "16")
    # job lists built on the device (forced: a context with 16 host threads of its own builds them on the host) ...
    monkeypatch.setenv("DFB_DEVICE_BUILD", "1")
    piped = al.align_batch(rt, st, tc, trd, ms)
    # ... and on the host
    monkeypatch.delenv("DFB_DEVICE_BUILD")
    monkeypatch.setenv("DFB_HOST_BUILD", "1")
    piped_host = al.align_batch(rt, st, tc, trd, ms)
    monkeypatch.delenv("DFB_HOST_BUILD")
    monkeypatch.setenv("DFB_DEVICE_BUILD", "1")
    assert np.array_equal(piped_host.best, single.best) and np.array_equal(piped_host.rows["task"], single.rows["task"])
    assert np.array_equal(piped.best, single.best)
    # the column pool may be laid out differently (col_begin is explicit); rows and their column lists must agree
    assert len(piped.rows) == len(single.rows)
    for f in ("task", "read_split", "score1", "score2", "n1", "n2"):
        assert np.array_equal(piped.rows[f], single.rows[f]), f
    for a, b in zip(piped.rows, single.rows):
        assert np.array_equal(piped.cols[a["col_begin"]:a["col_begin"] + a["n1"] + a["n2"]],
                              single.cols[b["col_begin"]:b["col_begin"] + b["n1"] + b["n2"]])
    _check_split(oracle_mod, gpu_ctx, refs, reads, tc, trd, ms)                       # pipelined vs oracle
    _check_split(oracle_mod, gpu_ctx, refs, reads, tc, trd, ms, (2, -1, -2, True, 0))   # generic kernels, pipelined
    # a batch whose task_read decreases somewhere falls back to the single plan
    back = al.align_batch(rt, st, tc[::-1].copy(), trd[::-1].copy(), ms[::-1].copy())
    assert np.array_equal(back.best, single.best[::-1])


# ---------------------------------------------------------------------------------------------
# backtrace: GetAlignments(..., backtrace=true) -- dfb_split_backtrace_batch against the oracle
# ---------------------------------------------------------------------------------------------

def _backtrace_vs_oracle(oracle, al, refs, reads, tc, trd, s1, s2, a):
    """backtrace_batch of the alignments against the oracle's backtrace of each"""
    rt, st = _tables(refs, reads)
    m, x, g, eg = al.params.match, al.params.mismatch, al.params.gap, bool(al.params.end_gaps)
    off, pairs = al.backtrace_batch(rt, st, tc, trd, s1, s2, a)
    assert off[0] == 0 and off[-1] == len(pairs) and (np.diff(off) >= 0).all()
    for k in range(len(tc)):
        w1, w2 = oracle.split_backtrace(reads[trd[k]], refs[2 * tc[k]], refs[2 * tc[k] + 1], (s1[k], s2[k]), a[k], m, x, g, eg)
        g1, g2 = pairs[off[2 * k]:off[2 * k + 1]], pairs[off[2 * k + 1]:off[2 * k + 2]]
        assert g1.shape == w1.shape and (g1 == w1).all(), "alignment %d matches1: got\n%s\nwant\n%s" % (k, g1[:6], w1[:6])
        assert g2.shape == w2.shape and (g2 == w2).all(), "alignment %d matches2: got\n%s\nwant\n%s" % (k, g2[:6], w2[:6])
    return off, pairs


def _check_backtrace(oracle, ctx, refs, reads, task_cluster, task_read, min_score, params=(2, -1, -2, False, 8), per_task=4):
    import defuse_b200 as d
    rt, st = _tables(refs, reads)
    al = d.SplitReadAligner(*params, ctx=ctx)
    res = al.align_batch(rt, st, task_cluster, task_read, min_score)
    tc, trd, s1, s2, a = [], [], [], [], []
    for t in range(len(task_cluster)):
        for row in res.alignments(t)[:per_task]:
            tc.append(task_cluster[t]); trd.append(task_read[t]); s1.append(row[0]); s2.append(row[1]); a.append(row[2])
    _backtrace_vs_oracle(oracle, al, refs, reads, tc, trd, s1, s2, a)
    return len(tc)


def test_backtrace_dosplitalign_shape(oracle_mod, gpu_ctx):
    import defuse_b200 as d
    rng = np.random.default_rng(41)
    refs, reads, tc, trd = util.split_batch(rng, 12, 10, 100, 300, 380, sub=0.02, indel=0.01)
    ms = np.array([d.split_min_score(len(reads[r])) for r in trd], np.int32)
    assert _check_backtrace(oracle_mod, gpu_ctx, refs, reads, tc, trd, ms) > 40


@pytest.mark.parametrize("params", [(2, -1, -2, True, 8), (1, -1, 1, False, 3), (5, -4, -3, False, -2), (3, -2, 0, False, 1)])
def test_backtrace_generic_scoring(oracle_mod, gpu_ctx, params):
    rng = np.random.default_rng(42)
    refs, reads, tc, trd = util.split_batch(rng, 8, 6, (1, 90), 1, 200, sub=0.04, indel=0.02, n_rate=0.01)
    ms = np.array([int(0.5 * params[0] * len(reads[r])) for r in trd], np.int32)
    assert _check_backtrace(oracle_mod, gpu_ctx, refs, reads, tc, trd, ms, params) > 5


def test_backtrace_long_reads_and_ties(oracle_mod, gpu_ctx):
    """Reads longer than one 32-row tile, repeats (many equal-score paths), non-ACGT bytes."""
    rng = np.random.default_rng(43)
    refs, reads, tc, trd = [], [], [], []
    for c in range(6):
        unit = util.rand_seq(rng, int(rng.integers(2, 7)))
        r1 = (unit * 80)[:int(rng.integers(150, 420))]
        r2 = util.rand_seq(rng, 30) + (unit * 80)[:int(rng.integers(150, 400))]
        refs += [r1, r2]
        for _ in range(4):
            L = int(rng.integers(33, 300))
            read = util.mutate(rng, (r1[-L // 2:] + r2[:L - L // 2]), 0.03, 0.01, 0.02)
            tc.append(c); trd.append(len(reads)); reads.append(read)
    ms = np.array([int(1.2 * len(reads[r])) for r in trd], np.int32)
    assert _check_backtrace(oracle_mod, gpu_ctx, refs, reads, np.array(tc, np.int32), np.array(trd, np.int32), ms, per_task=6) > 10


@pytest.mark.parametrize("end_gaps", [False, True])
def test_backtrace_edge_start_cells(oracle_mod, gpu_ctx, end_gaps):
    """start cells on the corners and edges of both matrices -- i1 in {0, R1}, i2 in {0, R2}, a in {0, L} -- and inner
    points, whether or not an alignment exists there; the last task's read is empty"""
    import defuse_b200 as d
    rng = np.random.default_rng(44)
    refs, reads, tc, trd = util.split_batch(rng, 3, 2, 100, 280, 420)
    reads.append(b"")
    tc, trd = np.append(tc, 1).astype(np.int32), np.append(trd, len(reads) - 1).astype(np.int32)
    k_tc, k_trd, s1, s2, a = [], [], [], [], []
    for t in range(len(tc)):
        R1, R2, L = len(refs[2 * tc[t]]), len(refs[2 * tc[t] + 1]), len(reads[trd[t]])
        for i1 in (0, R1 // 2, R1):
            for rs2 in (-1, R2 // 3, R2 - 1):      # i2 = R2, ..., 0
                for split in sorted({0, min(1, L), L // 2, L}):
                    k_tc.append(tc[t]); k_trd.append(trd[t]); s1.append(i1); s2.append(rs2); a.append(split)
    al = d.SplitReadAligner(2, -1, -2, end_gaps, 8, ctx=gpu_ctx)
    off, pairs = _backtrace_vs_oracle(oracle_mod, al, refs, reads, k_tc, k_trd, s1, s2, a)
    assert len(pairs) > 0


def test_backtrace_reads_longer_than_1024(oracle_mod, gpu_ctx):
    """reads over 1024 bases against 1300-1500-base windows: boxes too large for shared memory (the global arena)"""
    import defuse_b200 as d
    rng = np.random.default_rng(25)
    refs, reads, tc, trd = util.split_batch(rng, 2, 2, (1030, 1200), 1300, 1500)
    ms = np.array([d.split_min_score(len(reads[r])) for r in trd], np.int32)
    assert _check_backtrace(oracle_mod, gpu_ctx, refs, reads, tc, trd, ms, per_task=3) > 0


def test_backtrace_size_only_and_short_buffer(gpu_ctx):
    """matches = NULL sizes the output; a matches_cap below the total is refused after match_off and n_pairs are
    written, and matches is left as it was"""
    import ctypes
    import defuse_b200 as d
    rng = np.random.default_rng(46)
    refs, reads, tc, trd = util.split_batch(rng, 4, 3, 100, 280, 420)
    rt, st = _tables(refs, reads)
    s1 = np.array([len(refs[2 * c]) // 2 for c in tc], np.int32)
    s2 = np.array([len(refs[2 * c + 1]) // 2 for c in tc], np.int32)
    a = np.array([len(reads[r]) // 2 for r in trd], np.int32)
    al = d.SplitReadAligner(ctx=gpu_ctx)
    want_off, want = al.backtrace_batch(rt, st, tc, trd, s1, s2, a)
    assert len(want) > 1
    lib, n = gpu_ctx._lib, len(tc)
    rts, sts = rt.c_struct(), st.c_struct()
    arrays = [np.ascontiguousarray(x, np.int32) for x in (tc, trd, s1, s2, a)]

    def call(matches, cap):
        off, total = np.full(2 * n + 1, -1, np.int64), ctypes.c_int64(-1)
        rc = lib.dfb_split_backtrace_batch(gpu_ctx._h, ctypes.byref(al.params), ctypes.byref(rts), ctypes.byref(sts),
                                           *[x.ctypes.data for x in arrays], n, off.ctypes.data, matches, cap, ctypes.byref(total))
        return rc, off, total.value

    rc, off, total = call(None, 0)
    assert rc == 0 and off.tobytes() == want_off.tobytes() and total == len(want)
    short = np.full((len(want) - 1, 2), -7, np.int32)
    rc, off, total = call(short.ctypes.data, len(want) - 1)
    assert rc == 2
    assert b"matches buffer holds %d pairs, %d needed" % (len(want) - 1, len(want)) in lib.dfb_last_error(gpu_ctx._h)
    assert off.tobytes() == want_off.tobytes() and total == len(want)
    assert (short == -7).all()


def test_device_backtrace_survives_a_host_backtrace(gpu_ctx):
    """a dfb_split_backtrace_device result stays on the context across a dfb_split_backtrace_batch call and is still
    what dfb_split_backtrace_copy_device copies out"""
    import ctypes
    import torch
    import defuse_b200 as d
    rng = np.random.default_rng(47)
    refs, reads, tc, trd = util.split_batch(rng, 10, 5, 100, 280, 420)
    rt, st = _tables(refs, reads)
    ms = np.array([d.split_min_score(len(reads[r])) for r in trd], np.int32)
    al = d.SplitReadAligner(ctx=gpu_ctx)
    dev = [torch.from_numpy(x).cuda() for x in (tc, trd, ms)]
    res = al.align_device(d.DeviceSeqTable.from_host(rt, "cuda:0"), d.DeviceSeqTable.from_host(st, "cuda:0"), *dev)
    rec = res.records()
    r = rec.cpu().numpy()
    assert len(r) > 10
    want_off, want = al.backtrace_batch(rt, st, tc[r[:, 0]], trd[r[:, 0]], r[:, 1], r[:, 2], r[:, 3])
    lib, n = gpu_ctx._lib, ctypes.c_int64()
    rts, sts = res.refs.c_struct(), res.reads.c_struct()
    assert lib.dfb_split_backtrace_device(gpu_ctx._h, ctypes.byref(res.params), ctypes.byref(rts), ctypes.byref(sts),
                                          res.task_cluster.data_ptr(), res.task_read.data_ptr(), res.task_cluster.numel(),
                                          rec.data_ptr(), rec.shape[0], ctypes.byref(n)) == 0
    assert n.value == len(want)
    other_off, _ = al.backtrace_batch(rt, st, tc[r[::3, 0]], trd[r[::3, 0]], r[::3, 1], r[::3, 2], r[::3, 3])
    assert len(other_off) != len(want_off)
    off = torch.empty(2 * len(r) + 1, dtype=torch.int64, device="cuda:0")
    pairs = torch.empty((n.value, 2), dtype=torch.int32, device="cuda:0")
    assert lib.dfb_split_backtrace_copy_device(gpu_ctx._h, off.data_ptr(), pairs.data_ptr()) == 0
    assert off.cpu().numpy().tobytes() == want_off.tobytes()
    assert pairs.cpu().numpy().tobytes() == want.tobytes()


def test_backtrace_argument_errors(gpu_ctx):
    import defuse_b200 as d
    rt, st = _tables([b"ACGTACGT", b"TTTTACGT"], [b"ACGTTTTT"])
    al = d.SplitReadAligner(ctx=gpu_ctx)
    with pytest.raises(d.DefuseB200Error):
        al.backtrace_batch(rt, st, [0], [0], [9], [0], [4])   # i1 beyond reference 1
    with pytest.raises(d.DefuseB200Error):
        al.backtrace_batch(rt, st, [0], [0], [4], [0], [9])   # read split beyond the read
    off, pairs = al.backtrace_batch(rt, st, [], [], [], [], [])
    assert len(off) == 1 and len(pairs) == 0


def test_random_parameters(oracle_mod, gpu_ctx):
    """Random scoring triples (positive gaps, negative matches, zeros: both the s16x2 and the s32 kernels get picked),
    endGaps either way, minSplitScore and minScore either side of zero, alphabets from one letter to mixed case with N,
    empty strings; lengths that land in several (G,S) classes (util.random_parameter_round, the generator of the
    oracle-vs-reference loop with longer sequences every fourth round).  scripts/gpu_fuzz.py runs the same loop by the
    clock."""
    rng = np.random.default_rng(41)
    for rnd in range(48):
        util.check_random_parameter_round(rng, rnd, oracle_mod, gpu_ctx, _check_split, _check_simple)
