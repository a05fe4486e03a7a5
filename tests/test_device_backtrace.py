"""Backtrace of device-resident split records (dfb_split_backtrace_device, dfb_split_backtrace_copy_device and
DeviceSplitResult.backtrace()): byte-equal to SplitReadAligner.backtrace_batch on the same alignments, samples right
against the oracle's backtrace, the argument checks on the records, and ordering behind torch's current stream."""
import ctypes

import numpy as np
import pytest

import util


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


def test_backtrace_symbols_are_exported():
    import defuse_b200 as d
    lib = d.load_library()
    for name in ("dfb_split_backtrace_device", "dfb_split_backtrace_copy_device"):
        assert hasattr(lib, name) and name in d.ABI_SYMBOLS


def test_null_context_is_rejected_without_cuda():
    import defuse_b200 as d
    lib = d.load_library()
    t = d._DeviceSeqTable(0, 0, 0, 0)
    p = d._SplitParams(2, -1, -2, 0, 8)
    n = ctypes.c_int64()
    assert lib.dfb_split_backtrace_device(None, ctypes.byref(p), ctypes.byref(t), ctypes.byref(t), None, None, 0, None, 0,
                                          ctypes.byref(n)) == 2
    assert lib.dfb_split_backtrace_copy_device(None, None, None) == 2


def test_record_tensor_errors_need_no_gpu():
    import defuse_b200 as d
    import torch
    res = d.DeviceSplitResult(None, torch.zeros((0, 8), dtype=torch.int32), None, None, None, None, None, None,
                              d._SplitParams(2, -1, -2, 0, 8))
    with pytest.raises(TypeError):
        res.backtrace(np.zeros((3, 6), np.int32))
    with pytest.raises(TypeError):
        res.backtrace(torch.zeros((3, 6), dtype=torch.int64))
    with pytest.raises(ValueError, match="CUDA"):
        res.backtrace(torch.zeros((3, 6), dtype=torch.int32))


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


def _align(ctx, refs, reads, tc, tr, ms, params=(2, -1, -2, False, 8)):
    import defuse_b200 as d
    al = d.SplitReadAligner(*params, ctx=ctx)
    return al, al.align_device(_dev(refs), _dev(reads), _t(tc), _t(tr), _t(ms))


def _backtrace_both(al, res, refs, reads, tc, tr, rec):
    """device backtrace of the records against backtrace_batch on the same alignments, byte for byte"""
    rec = np.ascontiguousarray(rec, dtype=np.int32).reshape(-1, 6)
    off, pairs = res.backtrace(_t(rec))
    off, pairs = off.cpu().numpy(), pairs.cpu().numpy()
    assert off.dtype == np.int64 and off.shape == (2 * len(rec) + 1,)
    assert pairs.dtype == np.int32 and pairs.ndim == 2 and pairs.shape[1] == 2
    t = rec[:, 0]
    tc, tr = np.asarray(tc, np.int32), np.asarray(tr, np.int32)
    w_off, w_pairs = al.backtrace_batch(refs, reads, tc[t], tr[t], rec[:, 1], rec[:, 2], rec[:, 3])
    assert off.tobytes() == w_off.tobytes()
    assert pairs.tobytes() == w_pairs.tobytes()
    return off, pairs


def _piece_bytes(rec, refs, reads, tc, tr, cap=256):
    """footprint of every piece (runs of one task cut where k % cap == 0): both boxes' pointer words and tile-edge rows,
    the rule of bt_box_kernel restated"""
    task = rec[:, 0].astype(np.int64)
    c, q = np.asarray(tc, np.int64)[task], np.asarray(tr, np.int64)[task]
    L = reads.off[q + 1] - reads.off[q]
    R2 = refs.off[2 * c + 2] - refs.off[2 * c + 1]
    a, i1, i2 = rec[:, 3].astype(np.int64), rec[:, 1].astype(np.int64), R2 - rec[:, 2] - 1
    k = np.arange(len(rec))
    head = (k % cap == 0) | np.concatenate([[True], task[1:] != task[:-1]])
    st = np.nonzero(head)[0]
    J1, I1 = np.maximum.reduceat(a, st), np.maximum.reduceat(i1, st)
    J2, I2 = np.maximum.reduceat(L - a, st), np.maximum.reduceat(i2, st)
    return 4 * (J1 * ((I1 + 16) >> 4) + J2 * ((I2 + 16) >> 4) + I1 + I2 + 2)


SMEM_BYTES = 96 << 10   # DFB_BT_SMEM_BYTES: larger pieces take the global arena


def _check_oracle(orc, refs, reads, tc, tr, rec, off, pairs, sample, params=(2, -1, -2, False, 8)):
    for k in sample:
        t = int(rec[k, 0])
        c, q = int(tc[t]), int(tr[t])
        m1, m2 = orc.split_backtrace(reads.get(q), refs.get(2 * c), refs.get(2 * c + 1), (int(rec[k, 1]), int(rec[k, 2])),
                                     int(rec[k, 3]), *params[:4])
        assert np.array_equal(pairs[off[2 * k]:off[2 * k + 1]], m1), "record %d" % k
        assert np.array_equal(pairs[off[2 * k + 1]:off[2 * k + 2]], m2), "record %d" % k


@pytest.mark.gpu
def test_bench_shape_200k_chunked_all_records(ctx, orc, monkeypatch):
    import defuse_b200 as d
    import synth
    monkeypatch.setenv("DFB_PIPELINE_MIN_TASKS", "16")
    w = synth.split_workload(9, 2000, 100)
    refs, reads = d.SeqTable(w["ref_bytes"], w["ref_off"]), d.SeqTable(w["read_bytes"], w["read_off"])
    al, res = _align(ctx, refs, reads, w["task_cluster"], w["task_read"], w["min_score"])
    rec = res.records().cpu().numpy()
    assert len(rec) > 100000
    off, pairs = _backtrace_both(al, res, refs, reads, w["task_cluster"], w["task_read"], rec)
    rng = np.random.default_rng(0)
    _check_oracle(orc, refs, reads, w["task_cluster"], w["task_read"], rec, off, pairs, rng.choice(len(rec), 200, replace=False))


@pytest.mark.gpu
def test_stress_walks_with_gaps(ctx, orc):
    import defuse_b200 as d
    import synth
    w = synth.split_workload(5, 150, 40, **synth.STRESS)
    refs, reads = d.SeqTable(w["ref_bytes"], w["ref_off"]), d.SeqTable(w["read_bytes"], w["read_off"])
    al, res = _align(ctx, refs, reads, w["task_cluster"], w["task_read"], w["min_score"])
    rec = res.records().cpu().numpy()
    off, pairs = _backtrace_both(al, res, refs, reads, w["task_cluster"], w["task_read"], rec)
    # gaps: some walk takes a non-diagonal step between two matches
    d1 = np.diff(pairs, axis=0)
    assert ((d1[:, 0] != 1) | (d1[:, 1] != 1)).any()
    rng = np.random.default_rng(1)
    _check_oracle(orc, refs, reads, w["task_cluster"], w["task_read"], rec, off, pairs, rng.choice(len(rec), 100, replace=False))


@pytest.mark.gpu
def test_poly_a_subset_and_small_task(ctx, orc):
    """24 x 467 k tie-heavy records: a fixed subset, including a contiguous stretch longer than a piece of one task
    (run splitting); then every record of a 60 x 90 poly-A task"""
    polyA = b"A" * 700
    refs, reads = _tables([polyA, polyA], [b"A" * 200] * 24)
    tc, tr, ms = np.zeros(24, np.int32), np.arange(24, dtype=np.int32), np.full(24, 360, np.int32)
    al, res = _align(ctx, refs, reads, tc, tr, ms)
    rec = res.records().cpu().numpy()
    assert len(rec) > 24 * 400000
    first5 = int(np.searchsorted(rec[:, 0], 5))
    sub = np.concatenate([rec[::4999], rec[first5 + 1000:first5 + 1700], rec[-3:]])
    off, pairs = _backtrace_both(al, res, refs, reads, tc, tr, sub)
    _check_oracle(orc, refs, reads, tc, tr, sub, off, pairs, np.arange(0, len(sub), 37))
    refs, reads = _tables([b"A" * 90, b"A" * 90], [b"A" * 60])
    al, res = _align(ctx, refs, reads, [0], [0], [100])
    rec = res.records().cpu().numpy()
    assert len(rec) > 1000
    off, pairs = _backtrace_both(al, res, refs, reads, [0], [0], rec)
    _check_oracle(orc, refs, reads, [0], [0], rec, off, pairs, np.arange(0, len(rec), 97))


@pytest.mark.gpu
@pytest.mark.parametrize("params", [(2, -1, -2, True, 8), (300, -200, -250, False, 1200), (1, -1, 1, False, 4)])
def test_s32_only_scoring(ctx, orc, params):
    rng = np.random.default_rng(24)
    refs, reads, tc, tr = util.split_batch(rng, 6, 5, (5, 40), 8, 70, sub=0.05)
    refs, reads = _tables(refs, reads)
    ms = np.array([int(0.9 * params[0] * reads.length(r)) for r in tr], np.int32)
    al, res = _align(ctx, refs, reads, tc, tr, ms, params)
    rec = res.records().cpu().numpy()
    assert len(rec) > 0
    off, pairs = _backtrace_both(al, res, refs, reads, tc, tr, rec)
    _check_oracle(orc, refs, reads, tc, tr, rec, off, pairs, range(len(rec)), params)


@pytest.mark.gpu
def test_reads_longer_than_1024_global_arena(ctx, orc):
    import defuse_b200 as d
    rng = np.random.default_rng(25)
    refs, reads, tc, tr = util.split_batch(rng, 2, 2, (1030, 1200), 1300, 1500)
    refs, reads = _tables(refs, reads)
    ms = np.array([d.split_min_score(reads.length(r)) for r in tr], np.int32)
    al, res = _align(ctx, refs, reads, tc, tr, ms)
    rec = res.records().cpu().numpy()
    assert len(rec) > 0
    size = _piece_bytes(rec, refs, reads, tc, tr)
    assert (size > SMEM_BYTES).any()   # pieces on the global arena (bt_fill_walk_kernel<false>)
    off, pairs = _backtrace_both(al, res, refs, reads, tc, tr, rec)
    _check_oracle(orc, refs, reads, tc, tr, rec, off, pairs, range(0, len(rec), max(1, len(rec) // 20)))


@pytest.mark.gpu
def test_output_spanning_several_waves(ctx):
    """records whose capacity slots (len(read) each) exceed one wave of 2^27 pairs: the output comes in one block per
    wave and is copied out in order.  The first records of one long-read task, repeated: every record's lists are known,
    and the run is long, so pieces fill once per 256 records"""
    rng = np.random.default_rng(26)
    refs, reads, tc, tr = util.split_batch(rng, 1, 2, (1100, 1100), 1300, 1400)
    refs, reads = _tables(refs, reads)
    al, res = _align(ctx, refs, reads, tc, tr, np.zeros(2, np.int32))
    rec = res.records().cpu().numpy()
    base = rec[rec[:, 0] == rec[0, 0]][:2]
    m = len(base)
    w_off, w_pairs = al.backtrace_batch(refs, reads, np.asarray(tc)[base[:, 0]], np.asarray(tr)[base[:, 0]], base[:, 1], base[:, 2], base[:, 3])
    slots = int((base[:, 3] + base[:, 4]).sum())   # len(read) capacity slots per record
    reps = (1 << 27) // slots + 2000000 // slots   # about 2 M slots over one wave
    off, pairs = res.backtrace(_t(np.tile(base, (reps, 1))))
    off, pairs = off.cpu().numpy(), pairs.cpu().numpy()
    n_pair = int(w_off[-1])
    assert off.shape == (2 * m * reps + 1,) and pairs.shape == (reps * n_pair, 2)
    assert np.array_equal(off[:-1].reshape(reps, 2 * m) - off[:-1:2 * m, None], np.tile(w_off[:-1], (reps, 1)))
    assert pairs.reshape(reps, n_pair, 2).tobytes() == np.tile(w_pairs, (reps, 1)).tobytes()


@pytest.mark.gpu
def test_subsets_orders_and_repeats(ctx, orc):
    import defuse_b200 as d
    rng = np.random.default_rng(31)
    refs, reads, tc, tr = util.split_batch(rng, 30, 12, 100, 280, 420)
    refs, reads = _tables(refs, reads)
    ms = np.array([d.split_min_score(reads.length(r)) for r in tr], np.int32)
    al, res = _align(ctx, refs, reads, tc, tr, ms)
    rec = res.records().cpu().numpy()
    assert len(np.unique(rec[:, 0])) > 10
    base_off, base_pairs = _backtrace_both(al, res, refs, reads, tc, tr, rec)
    _backtrace_both(al, res, refs, reads, tc, tr, rec[::7])
    rev_off, rev_pairs = _backtrace_both(al, res, refs, reads, tc, tr, rec[::-1])
    n = len(rec)
    for k in range(0, n, max(1, n // 25)):   # record k of the reversed order is record n - 1 - k
        j = n - 1 - k
        assert np.array_equal(rev_pairs[rev_off[2 * k]:rev_off[2 * k + 2]], base_pairs[base_off[2 * j]:base_off[2 * j + 2]])
    _backtrace_both(al, res, refs, reads, tc, tr, np.repeat(rec[:5], 3, axis=0))
    _backtrace_both(al, res, refs, reads, tc, tr, rec[[0, 5, 0, 5, 0]])
    tasks = np.unique(rec[:, 0])
    a, b = rec[rec[:, 0] == tasks[0]], rec[rec[:, 0] == tasks[1]]
    m = min(len(a), len(b))
    _backtrace_both(al, res, refs, reads, tc, tr, np.stack([a[:m], b[:m]], axis=1).reshape(-1, 6))


@pytest.mark.gpu
def test_hand_built_edge_start_cells(ctx, orc):
    rng = np.random.default_rng(12)
    refs, reads, tc, tr = util.split_batch(rng, 3, 2, 100, 280, 420)
    refs, reads = _tables(refs, reads)
    ms = np.zeros(len(tc), np.int32)
    al, res = _align(ctx, refs, reads, tc, tr, ms)
    rec = []
    for t in range(len(tc)):
        c, q = int(tc[t]), int(tr[t])
        R1, R2, L = refs.length(2 * c), refs.length(2 * c + 1), reads.length(q)
        for i1 in (0, R1 // 2, R1):
            for rs2 in (-1, R2 // 3, R2 - 1):      # i2 = R2, ..., 0
                for a in (0, 1, L // 2, L):
                    rec.append((t, i1, rs2, a, L - a, 0))
    rec = np.array(rec, np.int32)
    off, pairs = _backtrace_both(al, res, refs, reads, tc, tr, rec)
    _check_oracle(orc, refs, reads, tc, tr, rec, off, pairs, range(0, len(rec), 5))


@pytest.mark.gpu
def test_zero_and_one_record(ctx, orc):
    import torch
    refs, reads = _tables([b"ACGTACGTAAAA" * 10, b"TTTTGGGGCCCC" * 10], [b"ACGTACGTAAAATTTTGGGGCCCC"])
    al, res = _align(ctx, refs, reads, [0], [0], [0])
    off, pairs = res.backtrace(torch.zeros((0, 6), dtype=torch.int32, device="cuda:0"))
    assert off.cpu().tolist() == [0] and tuple(pairs.shape) == (0, 2)
    rec = res.records().cpu().numpy()[:1]
    assert len(rec) == 1
    off, pairs = _backtrace_both(al, res, refs, reads, [0], [0], rec)
    assert len(pairs) > 0
    _check_oracle(orc, refs, reads, [0], [0], rec, off, pairs, [0])


def _err(fn):
    import defuse_b200 as d
    with pytest.raises(d.DefuseB200Error) as e:
        fn()
    return e.value.status, str(e.value)


@pytest.mark.gpu
def test_malformed_records_tables_and_memory_are_refused(ctx):
    import defuse_b200 as d
    import torch
    lib = d.load_library()
    fresh = d.Context(0)
    assert fresh._lib.dfb_split_backtrace_copy_device(fresh._h, None, None) == 5   # nothing to copy yet
    fresh.close()
    rng = np.random.default_rng(8)
    refs, reads, tc, tr = util.split_batch(rng, 6, 6, 100, 280, 420)
    refs, reads = _tables(refs, reads)
    ms = np.array([d.split_min_score(reads.length(r)) for r in tr], np.int32)
    _, res = _align(ctx, refs, reads, tc, tr, ms)
    rec0 = res.records()
    assert rec0.shape[0] >= 4
    t1 = int(rec0[1, 0])
    L = reads.length(int(tr[t1]))
    R1, R2 = refs.length(2 * int(tc[t1])), refs.length(2 * int(tc[t1]) + 1)
    cases = []
    r = rec0.clone(); r[1, 0] = len(tc); cases.append((r, "record 1: task out of range"))
    r = rec0.clone(); r[1, 0] = -1; cases.append((r, "record 1: task out of range"))
    r = rec0.clone(); r[1, 3] = L + 1; r[1, 4] = -1; cases.append((r, "record 1: start cell outside the matrices"))
    r = rec0.clone(); r[1, 3] = -1; r[1, 4] = L + 1; cases.append((r, "record 1: start cell outside the matrices"))
    r = rec0.clone(); r[1, 1] = R1 + 1; cases.append((r, "record 1: start cell outside the matrices"))
    r = rec0.clone(); r[1, 1] = -1; cases.append((r, "record 1: start cell outside the matrices"))
    r = rec0.clone(); r[1, 2] = R2; cases.append((r, "record 1: start cell outside the matrices"))        # i2 = -1
    r = rec0.clone(); r[1, 2] = -2; cases.append((r, "record 1: start cell outside the matrices"))        # i2 = R2 + 1
    r = rec0.clone(); r[1, 4] += 1; cases.append((r, "record 1: read_split2 != len(read) - read_split1"))
    r = rec0.clone(); r[3, 0] = -1; r[2, 4] += 1; cases.append((r, "record 2: read_split2"))                # the lowest bad record
    for rec, msg in cases:
        status, text = _err(lambda: res.backtrace(rec))
        assert status == 2 and msg in text, text
        assert lib.dfb_split_backtrace_copy_device(ctx._h, None, None) == 5   # a failed call leaves nothing to copy
    off, _ = res.backtrace(rec0)
    assert off.shape[0] == 2 * rec0.shape[0] + 1
    # table and task errors: align_device's messages
    tcl = res.task_cluster
    res.task_cluster = tcl.clone()
    res.task_cluster[2] = 1000
    status, text = _err(lambda: res.backtrace(rec0))
    assert status == 2 and "task 2: table index out of range" in text, text
    res.task_cluster = tcl
    refs_odd = d.DeviceSeqTable(res.refs.data, res.refs.off[:-1].contiguous())
    good_refs, res.refs = res.refs, refs_odd
    status, text = _err(lambda: res.backtrace(rec0))
    assert status == 2 and "refs must hold two windows per cluster" in text, text
    res.refs = good_refs
    # host memory for the records: refused before any work
    pinned = torch.zeros(rec0.shape, dtype=torch.int32).pin_memory()
    host = np.zeros(tuple(rec0.shape), np.int32)
    rt, st = res.refs.c_struct(), res.reads.c_struct()
    n = ctypes.c_int64()
    for p in (pinned.data_ptr(), host.ctypes.data):
        rc = lib.dfb_split_backtrace_device(ctx._h, ctypes.byref(res.params), ctypes.byref(rt), ctypes.byref(st),
                                            res.task_cluster.data_ptr(), res.task_read.data_ptr(), len(tc), p, rec0.shape[0],
                                            ctypes.byref(n))
        assert rc == 2 and b"records is not device memory" in lib.dfb_last_error(ctx._h)
        assert lib.dfb_split_backtrace_copy_device(ctx._h, None, None) == 5
    # Python-side errors need no library call
    with pytest.raises(ValueError):
        res.backtrace(rec0[:, :5])
    with pytest.raises(ValueError):
        res.backtrace(rec0.t().contiguous().t())


@pytest.mark.gpu
def test_records_written_on_the_current_stream_are_seen(ctx):
    """a torch kernel on a busy side stream writes the records right before backtrace(): the call must wait for it"""
    import defuse_b200 as d
    import torch
    rng = np.random.default_rng(41)
    refs, reads, tc, tr = util.split_batch(rng, 40, 20, 100, 280, 420)
    refs, reads = _tables(refs, reads)
    ms = np.array([d.split_min_score(reads.length(r)) for r in tr], np.int32)
    _, res = _align(ctx, refs, reads, tc, tr, ms)
    src = res.records()
    want_off, want_pairs = (x.cpu().numpy() for x in res.backtrace(src))
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(20_000_000)
        rec = torch.zeros_like(src)
        rec.copy_(src)
        off, pairs = res.backtrace(rec)
    s.synchronize()
    assert off.cpu().numpy().tobytes() == want_off.tobytes()
    assert pairs.cpu().numpy().tobytes() == want_pairs.tobytes()


@pytest.mark.gpu
def test_result_survives_a_later_align_and_records_call(ctx):
    import defuse_b200 as d
    rng = np.random.default_rng(5)
    batches = []
    for _ in range(2):
        refs, reads, tc, tr = util.split_batch(rng, 20, 10, 100, 280, 420)
        refs, reads = _tables(refs, reads)
        ms = np.array([d.split_min_score(reads.length(r)) for r in tr], np.int32)
        batches.append((refs, reads, tc, tr, ms))
    al, first = _align(ctx, *batches[0])
    rec1 = first.records()
    lib = ctx._lib
    n = ctypes.c_int64()
    rt, st = first.refs.c_struct(), first.reads.c_struct()
    assert lib.dfb_split_backtrace_device(ctx._h, ctypes.byref(first.params), ctypes.byref(rt), ctypes.byref(st),
                                          first.task_cluster.data_ptr(), first.task_read.data_ptr(), first.task_cluster.numel(),
                                          rec1.data_ptr(), rec1.shape[0], ctypes.byref(n)) == 0
    _, second = _align(ctx, *batches[1])
    assert second.records().shape[0] > 0
    import torch
    off = torch.empty(2 * rec1.shape[0] + 1, dtype=torch.int64, device="cuda:0")
    pairs = torch.empty((n.value, 2), dtype=torch.int32, device="cuda:0")
    assert lib.dfb_split_backtrace_copy_device(ctx._h, off.data_ptr(), pairs.data_ptr()) == 0
    refs, reads, tc, tr, _ = batches[0]
    r = rec1.cpu().numpy()
    w_off, w_pairs = al.backtrace_batch(refs, reads, np.asarray(tc)[r[:, 0]], np.asarray(tr)[r[:, 0]], r[:, 1], r[:, 2], r[:, 3])
    assert off.cpu().numpy().tobytes() == w_off.tobytes()
    assert pairs.cpu().numpy().tobytes() == w_pairs.tobytes()
