"""Records of device-resident split results (dfb_split_records_device, dfb_split_records_copy_device and
DeviceSplitResult.records()): byte-equal to SplitResult.records of the host form on the same batch, right against the
oracle run through the de-duplication rule, the argument checks on the rows, and ordering behind torch's current
stream."""
import ctypes

import numpy as np
import pytest

import util


# ---- the rule, restated in numpy (independent of the kernels' mask method) -------------------------------------------

def rule_records_task(rows, cols, L, R2, task):
    """Records of one task from its rows (SPLIT_ROW_DTYPE, in order): walk the rows, new = outer(B1[r], B2[r]) & ~seen,
    emit np.nonzero(new) (row-major: i1, then i2, ascending), seen |= new.  (k, 6) int32 with the task prepended."""
    lists = [(cols[r["col_begin"]:r["col_begin"] + r["n1"]], cols[r["col_begin"] + r["n1"]:r["col_begin"] + r["n1"] + r["n2"]])
             for r in rows]
    out = [np.zeros((0, 6), np.int32)]
    if not lists:
        return out[0]
    u1 = np.unique(np.concatenate([c1 for c1, _ in lists] + [np.zeros(0, np.int32)]))
    u2 = np.unique(np.concatenate([c2 for _, c2 in lists] + [np.zeros(0, np.int32)]))
    seen = np.zeros((len(u1), len(u2)), bool)
    for r, (c1, c2) in zip(rows, lists):
        new = np.outer(np.isin(u1, c1), np.isin(u2, c2)) & ~seen
        i, j = np.nonzero(new)
        a = int(r["read_split"])
        rec = np.empty((len(i), 6), np.int32)
        rec[:, 0] = task
        rec[:, 1] = u1[i]
        rec[:, 2] = R2 - u2[j] - 1
        rec[:, 3] = a
        rec[:, 4] = L - a
        rec[:, 5] = min(int(r["score1"]), int(r["score2"]))
        out.append(rec)
        seen |= new
    return np.concatenate(out)


def rule_records(res, tasks=None):
    """Records of a host SplitResult for `tasks` (all by default), concatenated in task order.  One-row tasks (which
    hold no duplicates: a row's lists are strictly ascending) are expanded vectorised, the others task by task."""
    n_tasks = len(res.best)
    tasks = np.arange(n_tasks) if tasks is None else np.asarray(tasks)
    rs = res._row_start
    n_rows_of = rs[tasks + 1] - rs[tasks]
    L_all, R2_all = res._read_len, res._ref2_len
    parts, keys = [], []
    single = tasks[n_rows_of == 1]
    if len(single):
        rows = res.rows[rs[single]]
        n1, n2 = rows["n1"].astype(np.int64), rows["n2"].astype(np.int64)
        cnt = n1 * n2
        rep = np.repeat(np.arange(len(rows)), cnt)
        off = np.arange(int(cnt.sum())) - np.repeat(np.cumsum(cnt) - cnt, cnt)
        a, b = off // n2[rep], off % n2[rep]
        cb = rows["col_begin"][rep]
        t = single[rep]
        rec = np.empty((len(rep), 6), np.int32)
        rec[:, 0] = t
        rec[:, 1] = res.cols[cb + a]
        rec[:, 2] = R2_all[t] - res.cols[cb + n1[rep] + b] - 1
        rec[:, 3] = rows["read_split"][rep]
        rec[:, 4] = L_all[t] - rows["read_split"][rep]
        rec[:, 5] = np.minimum(rows["score1"], rows["score2"])[rep]
        parts.append(rec)
        keys.append(t)
    for t in tasks[n_rows_of > 1]:
        rec = rule_records_task(res.rows[rs[t]:rs[t + 1]], res.cols, int(L_all[t]), int(R2_all[t]), int(t))
        parts.append(rec)
        keys.append(np.full(len(rec), t))
    if not parts:
        return np.zeros((0, 6), np.int32)
    allrec, allkey = np.concatenate(parts), np.concatenate(keys)
    return np.ascontiguousarray(allrec[np.argsort(allkey, kind="stable")])


def records_of(res, tasks):
    """SplitResult.records(t) with the task prepended, concatenated (the per-task host path)"""
    parts = [np.zeros((0, 6), np.int32)]
    for t in tasks:
        r = res.records(int(t))
        parts.append(np.hstack([np.full((len(r), 1), t, np.int32), r]))
    return np.concatenate(parts)


# ---- CPU ---------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def ctx():
    import defuse_b200
    return defuse_b200.default_context(0)


@pytest.fixture(scope="module")
def orc():
    import os
    import oracle
    if not os.path.exists(oracle.PORT_LIB):
        oracle.build()
    return oracle


def test_record_symbols_are_exported():
    import defuse_b200 as d
    lib = d.load_library()
    for name in ("dfb_split_records_device", "dfb_split_records_copy_device"):
        assert hasattr(lib, name) and name in d.ABI_SYMBOLS
    assert d.SPLIT_RECORD_DTYPE.itemsize == 24


def test_null_context_is_rejected_without_cuda():
    import defuse_b200 as d
    lib = d.load_library()
    t = d._DeviceSeqTable(0, 0, 0, 0)
    n = ctypes.c_int64()
    assert lib.dfb_split_records_device(None, ctypes.byref(t), ctypes.byref(t), None, None, 0, None, 0, None, 0, ctypes.byref(n)) == 2
    assert lib.dfb_split_records_copy_device(None, None) == 2


def _hand_result(spec, read_len, ref2_len):
    """SplitResult from per-row (task, read_split, score1, score2, cols1, cols2)"""
    import defuse_b200 as d
    rows = np.zeros(len(spec), d.SPLIT_ROW_DTYPE)
    cols = []
    for k, (task, a, s1, s2, c1, c2) in enumerate(spec):
        rows[k] = (task, a, s1, s2, len(cols), len(c1), len(c2))
        cols += list(c1) + list(c2)
    n_tasks = len(read_len)
    lens = (np.asarray(read_len, np.int32), np.asarray(ref2_len, np.int32))
    return d.SplitResult(np.zeros(n_tasks, np.int32), rows, np.asarray(cols, np.int32), lambda: lens)


def test_rule_matches_split_result_records():
    spec = [
        (0, 10, 20, 30, [3, 5, 9], [1, 2]),
        (0, 11, 25, 22, [5, 9, 12], [2, 4]),        # (5,2), (9,2) seen in row 0
        (0, 12, 21, 21, [], [1, 2]),                # empty side 1: nothing
        (0, 13, 24, 26, [3, 12], [1, 2, 4]),         # (3,1), (3,2), (12,2), (12,4) seen
        (2, 40, 50, 60, [0, 7], [0, 8]),             # task 1 has no rows
        (3, 0, 9, 9, [4], []),                       # empty side 2
        (3, 1, 8, 7, [4], [5]),
        (3, 2, 8, 7, [4], [5]),                      # all seen
        (4, 5, 10, 10, [1, 2, 3], [3, 6, 9]),
    ]
    read_len, ref2_len = [40, 50, 90, 20, 60], [30, 31, 32, 33, 40]
    res = _hand_result(spec, read_len, ref2_len)
    want = records_of(res, range(5))
    got = rule_records(res)
    assert got.dtype == np.int32 and got.shape == want.shape
    assert got.tobytes() == want.tobytes()
    for t in range(5):
        assert np.array_equal(rule_records(res, [t]), records_of(res, [t]))
    # a wide multi-row task against the host path
    rng = np.random.default_rng(3)
    spec = []
    for k in range(70):
        c1 = np.sort(rng.choice(40, rng.integers(0, 6), replace=False))
        c2 = np.sort(rng.choice(40, rng.integers(0, 6), replace=False))
        spec.append((0, k, int(rng.integers(1, 9)), int(rng.integers(1, 9)), c1, c2))
    res = _hand_result(spec, [100], [50])
    assert rule_records(res).tobytes() == records_of(res, [0]).tobytes()


# ---- GPU -----------------------------------------------------------------------------------------------------------

def _dev(table):
    import defuse_b200 as d
    return d.DeviceSeqTable.from_host(table, "cuda:0")


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).cuda()


def _tables(refs, seqs):
    import defuse_b200 as d
    return d.SeqTable.from_list(refs), d.SeqTable.from_list(seqs)


def _records_both(ctx, refs, reads, tc, tr, ms, params=(2, -1, -2, False, 8), per_task=False):
    """device records of the device result against the rule on the host result of the same batch, byte for byte"""
    import defuse_b200 as d
    al = d.SplitReadAligner(*params, ctx=ctx)
    host = al.align_batch(refs, reads, tc, tr, ms)
    dev = al.align_device(_dev(refs), _dev(reads), _t(tc), _t(tr), _t(ms))
    got = dev.records().cpu().numpy()
    assert got.dtype == np.int32 and got.ndim == 2 and got.shape[1] == 6
    want = records_of(host, range(len(host.best))) if per_task else rule_records(host)
    assert got.shape == want.shape
    assert got.tobytes() == want.tobytes()
    return host, got


def _check_oracle(orc, refs, reads, tc, tr, ms, got, sample=None, params=(2, -1, -2, False, 8)):
    tc, tr, ms = np.asarray(tc), np.asarray(tr), np.asarray(ms)
    pick = np.arange(len(tc)) if sample is None else np.asarray(sample)
    cnt, want = orc.split_align_batch(refs.data, refs.off, reads.data, reads.off, tc[pick], tr[pick], ms[pick], *params)
    pos = np.concatenate([[0], np.cumsum(cnt)])
    at = np.searchsorted(got[:, 0], np.arange(len(tc) + 1)) if len(got) else np.zeros(len(tc) + 1, np.int64)
    for k, t in enumerate(pick):
        w = orc.split_dedupe(want[pos[k]:pos[k + 1]]) if cnt[k] else np.zeros((0, 5), np.int32)
        g = got[at[t]:at[t + 1], 1:]
        assert g.shape == w.shape and (g == w).all(), "task %d" % t


@pytest.mark.gpu
def test_bench_shape_200k_spans_chunks(ctx, orc, monkeypatch):
    import defuse_b200 as d
    import synth
    monkeypatch.setenv("DFB_PIPELINE_MIN_TASKS", "16")
    w = synth.split_workload(9, 2000, 100)
    refs, reads = d.SeqTable(w["ref_bytes"], w["ref_off"]), d.SeqTable(w["read_bytes"], w["read_off"])
    host, got = _records_both(ctx, refs, reads, w["task_cluster"], w["task_read"], w["min_score"])
    assert len(got) > 0
    rng = np.random.default_rng(0)
    sample = np.sort(rng.choice(w["n_tasks"], 300, replace=False))
    _check_oracle(orc, refs, reads, w["task_cluster"], w["task_read"], w["min_score"], got, sample)
    # multi-row tasks are checked task by task on the host path too
    rs = host._row_start
    multi = np.nonzero(rs[1:] - rs[:-1] > 1)[0][:200]
    at = np.searchsorted(got[:, 0], np.arange(len(host.best) + 1))
    for t in multi:
        assert np.array_equal(got[at[t]:at[t + 1]], records_of(host, [t])), "task %d" % t


@pytest.mark.gpu
@pytest.mark.parametrize("chunked", [False, True])
def test_stress(ctx, orc, monkeypatch, chunked):
    import defuse_b200 as d
    import synth
    if chunked:
        monkeypatch.setenv("DFB_PIPELINE_MIN_TASKS", "16")
    w = synth.split_workload(5, 150, 40, **synth.STRESS)
    refs, reads = d.SeqTable(w["ref_bytes"], w["ref_off"]), d.SeqTable(w["read_bytes"], w["read_off"])
    _, got = _records_both(ctx, refs, reads, w["task_cluster"], w["task_read"], w["min_score"])
    _check_oracle(orc, refs, reads, w["task_cluster"], w["task_read"], w["min_score"], got)


@pytest.mark.gpu
def test_poly_a_multi_word_masks(ctx, orc):
    """193 rows per task: masks of up to four words; ~6.9e7 raw pairs per task collapse to a few 10^5 records"""
    import defuse_b200 as d
    polyA = b"A" * 700
    refs, reads = _tables([polyA, polyA], [b"A" * 200] * 24)
    tc, tr, ms = np.zeros(24, np.int32), np.arange(24, dtype=np.int32), np.full(24, 360, np.int32)
    al = d.SplitReadAligner(ctx=ctx)
    host = al.align_batch(refs, reads, tc, tr, ms)
    got = al.align_device(_dev(refs), _dev(reads), _t(tc), _t(tr), _t(ms)).records().cpu().numpy()
    rs = host._row_start
    assert (rs[1:] - rs[:-1]).max() > 128
    want0 = rule_records(host, [0])
    counts = np.bincount(got[:, 0], minlength=24)
    assert (counts == len(want0)).all()       # the 24 tasks are the same alignment
    at = np.concatenate([[0], np.cumsum(counts)])
    assert np.array_equal(got[at[0]:at[1]], want0)
    assert np.array_equal(got[at[23]:at[24]], rule_records(host, [23]))
    n_want, _ = orc.split_align_count(b"A" * 200, polyA, polyA, 360)
    assert sum(int(r["n1"]) * int(r["n2"]) for r in host.rows[rs[0]:rs[1]]) == n_want
    # the oracle's alignments through the rule, on a poly-A task small enough to materialise (~10^5 alignments)
    refs, reads = _tables([b"A" * 90, b"A" * 90], [b"A" * 60])
    _, got = _records_both(ctx, refs, reads, [0], [0], [100])
    al = orc.split_align(b"A" * 60, b"A" * 90, b"A" * 90, 100)
    assert len(al) > 10000 and len(got) < len(al)
    key = (al[:, 0].astype(np.int64) << 32) | (al[:, 1].astype(np.int64) & 0xffffffff)
    first = np.sort(np.unique(key, return_index=True)[1])
    want = np.column_stack([al[first, :4], np.minimum(al[first, 5], al[first, 6])])
    assert np.array_equal(got[:, 1:], want)


@pytest.mark.gpu
@pytest.mark.parametrize("params", [(2, -1, -2, True, 8), (300, -200, -250, False, 1200), (1, -1, 1, False, 4)])
def test_s32_only_scoring(ctx, orc, params):
    rng = np.random.default_rng(24)
    refs, reads, tc, tr = util.split_batch(rng, 6, 5, (5, 40), 8, 70, sub=0.05)
    refs, reads = _tables(refs, reads)
    ms = np.array([int(0.9 * params[0] * reads.length(r)) for r in tr], np.int32)
    _, got = _records_both(ctx, refs, reads, tc, tr, ms, params, per_task=True)
    _check_oracle(orc, refs, reads, tc, tr, ms, got, params=params)


@pytest.mark.gpu
def test_reads_longer_than_1024(ctx, orc):
    import defuse_b200 as d
    rng = np.random.default_rng(25)
    refs, reads, tc, tr = util.split_batch(rng, 2, 2, (1030, 1200), 1300, 1500)
    refs, reads = _tables(refs, reads)
    ms = np.array([d.split_min_score(reads.length(r)) for r in tr], np.int32)
    _, got = _records_both(ctx, refs, reads, tc, tr, ms, per_task=True)
    _check_oracle(orc, refs, reads, tc, tr, ms, got)


@pytest.mark.gpu
def test_long_tie_rows_over_64_per_task(ctx, orc):
    """reads over 1024 bases on repeats: more than 64 rows per task on the s32 path (multi-word masks there)"""
    import defuse_b200 as d
    rep = b"AC" * 600
    refs, reads = _tables([rep, rep], [b"AC" * 520, b"CA" * 530])
    tc, tr = np.zeros(2, np.int32), np.arange(2, dtype=np.int32)
    ms = np.array([d.split_min_score(reads.length(r)) for r in tr], np.int32)
    host, got = _records_both(ctx, refs, reads, tc, tr, ms)
    rs = host._row_start
    assert (rs[1:] - rs[:-1]).max() > 64
    assert ctx.split_result_stats()["generic_jobs"] > 0
    for t in range(2):
        n, _ = orc.split_align_count(reads.get(t), rep, rep, int(ms[t]))
        rows = host.rows[rs[t]:rs[t + 1]]
        assert sum(int(r["n1"]) * int(r["n2"]) for r in rows) == n


@pytest.mark.gpu
def test_non_monotone_task_order(ctx, orc, monkeypatch):
    monkeypatch.setenv("DFB_PIPELINE_MIN_TASKS", "16")
    import defuse_b200 as d
    rng = np.random.default_rng(31)
    refs, reads, tc, tr = util.split_batch(rng, 30, 12, 100, 280, 420)
    perm = rng.permutation(len(tc))
    tc, tr = np.asarray(tc)[perm], np.asarray(tr)[perm]
    refs, reads = _tables(refs, reads)
    ms = np.array([d.split_min_score(reads.length(r)) for r in tr], np.int32)
    _, got = _records_both(ctx, refs, reads, tc, tr, ms, per_task=True)
    _check_oracle(orc, refs, reads, tc, tr, ms, got)


@pytest.mark.gpu
def test_empty_and_one_task(ctx, orc):
    refs, reads = _tables([b"ACGTACGTAAAA" * 10, b"TTTTGGGGCCCC" * 10], [b"ACGTACGTAAAATTTTGGGGCCCC"])
    z = np.zeros(0, np.int32)
    _, got = _records_both(ctx, refs, reads, z, z, z)
    assert got.shape == (0, 6)
    _, got = _records_both(ctx, refs, reads, [0], [0], [0], per_task=True)
    assert len(got) > 0
    _check_oracle(orc, refs, reads, [0], [0], [0], got)


@pytest.mark.gpu
def test_result_kept_across_a_later_split_call(ctx):
    import defuse_b200 as d
    rng = np.random.default_rng(5)
    al = d.SplitReadAligner(ctx=ctx)
    batches = []
    for _ in range(2):
        refs, reads, tc, tr = util.split_batch(rng, 20, 10, 100, 280, 420)
        refs, reads = _tables(refs, reads)
        ms = np.array([d.split_min_score(reads.length(r)) for r in tr], np.int32)
        batches.append((refs, reads, tc, tr, ms))
    first = al.align_device(*[_dev(x) for x in batches[0][:2]], *[_t(x) for x in batches[0][2:]])
    second = al.align_device(*[_dev(x) for x in batches[1][:2]], *[_t(x) for x in batches[1][2:]])
    got1 = first.records().cpu().numpy()
    got2 = second.records().cpu().numpy()
    assert got1.tobytes() == records_of(al.align_batch(*batches[0]), range(len(batches[0][2]))).tobytes()
    assert got2.tobytes() == records_of(al.align_batch(*batches[1]), range(len(batches[1][2]))).tobytes()


def _err(fn):
    import defuse_b200 as d
    with pytest.raises(d.DefuseB200Error) as e:
        fn()
    return e.value.status, str(e.value)


@pytest.mark.gpu
def test_malformed_rows_and_memory_are_refused(ctx):
    import defuse_b200 as d
    import torch
    lib = d.load_library()
    fresh = d.Context(0)
    assert fresh._lib.dfb_split_records_copy_device(fresh._h, None) == 5   # nothing to copy yet
    fresh.close()
    rng = np.random.default_rng(8)
    refs, reads, tc, tr = util.split_batch(rng, 6, 6, 100, 280, 420)
    refs, reads = _tables(refs, reads)
    ms = np.array([d.split_min_score(reads.length(r)) for r in tr], np.int32)
    res = d.SplitReadAligner(ctx=ctx).align_device(_dev(refs), _dev(reads), _t(tc), _t(tr), _t(ms))
    rows0, cols0 = res.rows.clone(), res.cols.clone()
    assert rows0.shape[0] >= 3 and cols0.numel() >= 4
    n_cols = cols0.numel()

    def run(rows, cols):
        res.rows, res.cols = rows, cols
        return _err(res.records)

    cases = []
    r = rows0.clone(); r[1, 0] = len(tc); cases.append((r, cols0, "task out of range"))
    r = rows0.clone(); r[2, 0] = -1; cases.append((r, cols0, "task out of range"))
    r = rows0.clone(); r[1, 0] = len(tc) - 1; r[2, 0] = 0; cases.append((r, cols0, "tasks decrease"))
    r = rows0.clone(); r[0, 7] = n_cols; cases.append((r, cols0, "columns outside the column pool"))
    r = rows0.clone(); r[0, 1] = 100000; cases.append((r, cols0, "read_split outside"))
    c = cols0.clone(); c[int(rows0[0, 4])] = 100000; cases.append((rows0, c, "outside its window"))
    c = cols0.clone(); first = int(rows0[0, 4]); n1 = int(rows0[0, 6])
    if n1 >= 2:
        c[first], c[first + 1] = c[first + 1].clone(), c[first].clone()
    else:
        c[first + n1] = -1
    cases.append((rows0, c, "not ascending" if n1 >= 2 else "outside its window"))
    for rows, cols, msg in cases:
        status, text = run(rows, cols)
        assert status == 2 and msg in text, text
    res.rows, res.cols = rows0, cols0
    assert res.records().shape[1] == 6
    # host memory for the rows: refused before any work
    pinned = torch.zeros(rows0.shape, dtype=torch.int32).pin_memory()
    host = np.zeros(rows0.shape, np.int32)
    rt, st = res.refs.c_struct(), res.reads.c_struct()
    n = ctypes.c_int64()
    for p in (pinned.data_ptr(), host.ctypes.data):
        rc = lib.dfb_split_records_device(ctx._h, ctypes.byref(rt), ctypes.byref(st), res.task_cluster.data_ptr(), res.task_read.data_ptr(),
                                          len(tc), p, rows0.shape[0], cols0.data_ptr(), n_cols, ctypes.byref(n))
        assert rc == 2 and b"rows is not device memory" in lib.dfb_last_error(ctx._h)
    assert lib.dfb_split_records_copy_device(ctx._h, None) == 5            # the failed call left nothing to copy


@pytest.mark.gpu
def test_rows_written_on_the_current_stream_are_seen(ctx):
    """a torch kernel on a busy side stream writes the rows right before records(): the call must wait for it"""
    import defuse_b200 as d
    import torch
    rng = np.random.default_rng(41)
    refs, reads, tc, tr = util.split_batch(rng, 40, 20, 100, 280, 420)
    refs, reads = _tables(refs, reads)
    ms = np.array([d.split_min_score(reads.length(r)) for r in tr], np.int32)
    al = d.SplitReadAligner(ctx=ctx)
    want = records_of(al.align_batch(refs, reads, tc, tr, ms), range(len(tc)))
    res = al.align_device(_dev(refs), _dev(reads), _t(tc), _t(tr), _t(ms))
    src = res.rows.clone()
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(20_000_000)
        res.rows = torch.zeros_like(src)
        res.rows.copy_(src)
        got = res.records()
    s.synchronize()
    assert got.cpu().numpy().tobytes() == want.tobytes()
