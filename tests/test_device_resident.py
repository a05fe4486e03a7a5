"""The device-resident forms (dfb_simple_align_device, dfb_split_align_device, dfb_split_result_copy_device and their
torch face): results byte-equal to the host one-call forms on the same data and right against the oracle, the same
errors, inputs and outputs that never cross PCIe, and ordering behind torch's current stream."""
import ctypes

import numpy as np
import pytest

import util


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


# ---- CPU: the ABI surface ------------------------------------------------------------------------------------------

def test_device_symbols_are_exported():
    import defuse_b200 as d
    lib = d.load_library()
    for name in ("dfb_simple_align_device", "dfb_split_align_device", "dfb_split_result_copy_device"):
        assert hasattr(lib, name) and name in d.ABI_SYMBOLS
    assert ctypes.sizeof(d._DeviceSeqTable) == 32
    assert ctypes.sizeof(d._SeqTable) == 24


def test_null_context_is_rejected_without_cuda():
    import defuse_b200 as d
    lib = d.load_library()
    t = d._DeviceSeqTable(0, 0, 0, 0)
    i64 = ctypes.c_int64()
    assert lib.dfb_simple_align_device(None, ctypes.byref(d._SimpleParams(10, -5, -5)), ctypes.byref(t), ctypes.byref(t),
                                       None, None, 0, None) == 2
    assert lib.dfb_split_align_device(None, ctypes.byref(d._SplitParams(2, -1, -2, 0, 8)), ctypes.byref(t), ctypes.byref(t),
                                      None, None, None, 0, None, ctypes.byref(i64), ctypes.byref(i64)) == 2
    assert lib.dfb_split_result_copy_device(None, None, None) == 2


def test_device_table_rejects_wrong_tensors_before_any_call():
    torch = pytest.importorskip("torch")
    import defuse_b200 as d
    with pytest.raises(TypeError):
        d.DeviceSeqTable(np.zeros(3, np.uint8), np.zeros(1, np.int64))
    with pytest.raises(TypeError):
        d.DeviceSeqTable(torch.zeros(3, dtype=torch.int32), torch.zeros(1, dtype=torch.int64))
    with pytest.raises(ValueError):
        d.DeviceSeqTable(torch.zeros(3, dtype=torch.uint8), torch.zeros(1, dtype=torch.int64))  # CPU tensors


# ---- GPU -----------------------------------------------------------------------------------------------------------

def _dev(table):
    import defuse_b200 as d
    return d.DeviceSeqTable.from_host(table, "cuda:0")


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).cuda()


def _split_both(ctx, refs, reads, tc, tr, ms, params=(2, -1, -2, False, 8)):
    """host one-call result and device result of the same batch; asserts byte equality"""
    import defuse_b200 as d
    al = d.SplitReadAligner(*params, ctx=ctx)
    host = al.align_batch(refs, reads, tc, tr, ms)
    dev = al.align_device(_dev(refs), _dev(reads), _t(tc), _t(tr), _t(ms))
    got = dev.to_host()
    assert np.array_equal(got.best, host.best)
    assert got.rows.tobytes() == host.rows.tobytes()
    assert np.array_equal(got.cols, host.cols)
    return host, got


def _check_oracle(orc, refs, reads, tc, tr, ms, res, sample=None, params=(2, -1, -2, False, 8)):
    tc, tr, ms = np.asarray(tc), np.asarray(tr), np.asarray(ms)
    pick = np.arange(len(tc)) if sample is None else sample
    cnt, want = orc.split_align_batch(refs.data, refs.off, reads.data, reads.off, tc[pick], tr[pick], ms[pick], *params)
    pos = np.concatenate([[0], np.cumsum(cnt)])
    for k, t in enumerate(pick):
        w = want[pos[k]:pos[k + 1]]
        a = res.alignments(int(t))
        assert a.shape == w.shape and (a == w).all(), "task %d" % t


def _tables(refs, seqs):
    import defuse_b200 as d
    return d.SeqTable.from_list(refs), d.SeqTable.from_list(seqs)


@pytest.mark.gpu
def test_bench_shape_200k_spans_chunks(ctx, orc, monkeypatch):
    import defuse_b200 as d
    import synth
    monkeypatch.setenv("DFB_PIPELINE_MIN_TASKS", "16")   # 200 k tasks: cut into chunks like a full batch
    w = synth.split_workload(9, 2000, 100)
    refs, reads = d.SeqTable(w["ref_bytes"], w["ref_off"]), d.SeqTable(w["read_bytes"], w["read_off"])
    _, res = _split_both(ctx, refs, reads, w["task_cluster"], w["task_read"], w["min_score"])
    rng = np.random.default_rng(0)
    _check_oracle(orc, refs, reads, w["task_cluster"], w["task_read"], w["min_score"], res,
                  np.sort(rng.choice(w["n_tasks"], 300, replace=False)))


@pytest.mark.gpu
def test_bench_shape_1m_three_chunks(ctx, orc):
    """10 000 clusters x 100 reads: a batch the host form cuts into three chunks, so the result arrays grow and the
    batch's totals advance over more than two chunks"""
    import defuse_b200 as d
    import synth
    w = synth.split_workload(3, 10000, 100)
    refs, reads = d.SeqTable(w["ref_bytes"], w["ref_off"]), d.SeqTable(w["read_bytes"], w["read_off"])
    _, res = _split_both(ctx, refs, reads, w["task_cluster"], w["task_read"], w["min_score"])
    rng = np.random.default_rng(1)
    _check_oracle(orc, refs, reads, w["task_cluster"], w["task_read"], w["min_score"], res,
                  np.sort(rng.choice(w["n_tasks"], 200, replace=False)))


@pytest.mark.gpu
def test_chunked_with_small_pipeline_threshold(ctx, orc, monkeypatch):
    """Several chunks, cluster views, and the overflow list in each of them."""
    import defuse_b200 as d
    import synth
    monkeypatch.setenv("DFB_PIPELINE_MIN_TASKS", "16")
    w = synth.split_workload(5, 150, 40, **synth.STRESS)
    refs, reads = d.SeqTable(w["ref_bytes"], w["ref_off"]), d.SeqTable(w["read_bytes"], w["read_off"])
    _, res = _split_both(ctx, refs, reads, w["task_cluster"], w["task_read"], w["min_score"])
    _check_oracle(orc, refs, reads, w["task_cluster"], w["task_read"], w["min_score"], res)


@pytest.mark.gpu
def test_stress(ctx, orc):
    import defuse_b200 as d
    import synth
    w = synth.split_workload(5, 150, 40, **synth.STRESS)
    refs, reads = d.SeqTable(w["ref_bytes"], w["ref_off"]), d.SeqTable(w["read_bytes"], w["read_off"])
    _, res = _split_both(ctx, refs, reads, w["task_cluster"], w["task_read"], w["min_score"])
    _check_oracle(orc, refs, reads, w["task_cluster"], w["task_read"], w["min_score"], res)


@pytest.mark.gpu
@pytest.mark.parametrize("pipelined", [False, True])
def test_poly_a_overflow_retry(ctx, orc, monkeypatch, pipelined):
    """more than 2^20 overflow columns: the list is resized and the probe sweep run again; one task holds ~10^5 events"""
    if pipelined:
        monkeypatch.setenv("DFB_PIPELINE_MIN_TASKS", "16")
    polyA = b"A" * 700
    refs, reads = _tables([polyA, polyA], [b"A" * 200] * 24)
    tc = np.zeros(24, np.int32)
    tr = np.arange(24, dtype=np.int32)
    host, res = _split_both(ctx, refs, reads, tc, tr, np.full(24, 360, np.int32))
    assert len(res.cols) > (1 << 20)
    n_want, best_want = orc.split_align_count(b"A" * 200, polyA, polyA, 360)
    for t in (0, 23):
        rows = res.rows[res.rows["task"] == t]
        assert res.best[t] == best_want
        assert sum(int(r["n1"]) * int(r["n2"]) for r in rows) == n_want
    assert ctx.split_result_stats()["events"] == len(res.cols)


@pytest.mark.gpu
@pytest.mark.parametrize("params", [(2, -1, -2, True, 8), (300, -200, -250, False, 1200), (1, -1, 1, False, 4)])
def test_s32_only_scoring(ctx, orc, params):
    rng = np.random.default_rng(24)
    refs, reads, tc, tr = util.split_batch(rng, 6, 5, (5, 40), 8, 70, sub=0.05)
    refs, reads = _tables(refs, reads)
    ms = np.array([int(0.9 * params[0] * reads.length(r)) for r in tr], np.int32)
    _, res = _split_both(ctx, refs, reads, tc, tr, ms, params)
    _check_oracle(orc, refs, reads, tc, tr, ms, res, params=params)
    st = ctx.split_result_stats()
    assert st["generic_jobs"] > 0


@pytest.mark.gpu
def test_reads_longer_than_1024(ctx, orc):
    rng = np.random.default_rng(25)
    refs, reads, tc, tr = util.split_batch(rng, 2, 2, (1030, 1200), 1300, 1500)
    refs, reads = _tables(refs, reads)
    import defuse_b200 as d
    ms = np.array([d.split_min_score(reads.length(r)) for r in tr], np.int32)
    _, res = _split_both(ctx, refs, reads, tc, tr, ms)
    _check_oracle(orc, refs, reads, tc, tr, ms, res)


@pytest.mark.gpu
def test_empty_and_one_task(ctx, orc):
    import defuse_b200 as d
    refs, reads = _tables([b"ACGTACGTAAAA" * 10, b"TTTTGGGGCCCC" * 10], [b"ACGTACGTAAAATTTTGGGGCCCC"])
    z = np.zeros(0, np.int32)
    _split_both(ctx, refs, reads, z, z, z)
    _split_both(ctx, refs, reads, [0], [0], [0])
    al = d.SimpleAligner(10, -5, -5, ctx=ctx)
    assert al.align_device(_dev(refs), _dev(reads), _t(z), _t(z)).numel() == 0
    got = al.align_device(_dev(refs), _dev(reads), _t([1]), _t([0])).cpu().numpy()
    assert np.array_equal(got, al.align_batch(refs, reads, [1], [0]))


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
    _, res = _split_both(ctx, refs, reads, tc, tr, ms)
    _check_oracle(orc, refs, reads, tc, tr, ms, res)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["localalign", "matealign"])
def test_simple_shapes(ctx, orc, shape):
    import defuse_b200 as d
    import synth
    if shape == "localalign":
        w = synth.local_workload(2, 200, 60000, 2001, 100)
    else:
        w = synth.local_workload(2, 200, 60000, 1001, 150, own_window=True)
    refs, seqs = d.SeqTable(w["ref_bytes"], w["ref_off"]), d.SeqTable(w["seq_bytes"], w["seq_off"])
    al = d.SimpleAligner(10, -5, -5, ctx=ctx)
    host = al.align_batch(refs, seqs, w["task_ref"], w["task_seq"])
    dev = al.align_device(_dev(refs), _dev(seqs), _t(w["task_ref"]), _t(w["task_seq"])).cpu().numpy()
    assert np.array_equal(dev, host)
    pick = np.arange(0, w["n_tasks"], 97)
    want = orc.simple_align_batch(10, -5, -5, refs.data, refs.off, seqs.data, seqs.off, w["task_ref"][pick], w["task_seq"][pick])
    assert np.array_equal(dev[pick], want)


@pytest.mark.gpu
@pytest.mark.parametrize("scoring", [(10, -5, -5), (1, -1, 1), (3, 3, 3)])
def test_simple_random_and_s32(ctx, orc, scoring):
    import defuse_b200 as d
    rng = np.random.default_rng(14)
    refs, seqs, tr, ts = util.simple_batch(rng, 10, 300, (1, 300), (1, 300))
    refs, seqs = _tables(refs, seqs)
    al = d.SimpleAligner(*scoring, ctx=ctx)
    dev = al.align_device(_dev(refs), _dev(seqs), _t(tr), _t(ts)).cpu().numpy()
    assert np.array_equal(dev, al.align_batch(refs, seqs, tr, ts))
    assert np.array_equal(dev, orc.simple_align_batch(*scoring, refs.data, refs.off, seqs.data, seqs.off, tr, ts))


def _err(fn):
    import defuse_b200 as d
    with pytest.raises(d.DefuseB200Error) as e:
        fn()
    return e.value.status, str(e.value)


@pytest.mark.gpu
def test_errors_match_the_host_form(ctx):
    import defuse_b200 as d
    import torch
    al = d.SplitReadAligner(ctx=ctx)
    refs, reads = _tables([b"ACGT" * 20, b"GGCC" * 20], [b"ACGTGGCC" * 4, b"ACGT" * 8])
    tc, tr, ms = np.zeros(2, np.int32), np.array([0, 1], np.int32), np.zeros(2, np.int32)
    cases = []
    bad_off = d.SeqTable(reads.data, np.array([0, 40, 20], np.int64))             # offsets decrease at 1
    cases.append((refs, bad_off, tc, tr))
    cases.append((d.SeqTable(refs.data, np.array([4, 80, 160], np.int64)), reads, tc, tr))  # off[0] != 0
    cases.append((d.SeqTable(refs.data, refs.off[:2]), reads, tc, tr))            # odd refs->n
    cases.append((refs, reads, np.array([0, 1], np.int32), tr))                   # cluster out of range
    cases.append((refs, reads, tc, np.array([0, 5], np.int32)))                   # read out of range
    for rt, st, c, r in cases:
        want = _err(lambda: al.align_batch(rt, st, c, r, ms))
        got = _err(lambda: al.align_device(_dev(rt), _dev(st), _t(c), _t(r), _t(ms)))
        assert got == want
    # off[n] beyond the allocation
    short = d.DeviceSeqTable(torch.zeros(10, dtype=torch.uint8, device="cuda:0"), torch.tensor([0, 12], dtype=torch.int64, device="cuda:0"))
    status, msg = _err(lambda: al.align_device(_dev(refs), short, _t([0]), _t([0]), _t([0])))
    assert status == 2 and "exceeds n_bytes" in msg
    sal = d.SimpleAligner(10, -5, -5, ctx=ctx)
    want = _err(lambda: sal.align_batch(refs, bad_off, [0], [1]))
    assert _err(lambda: sal.align_device(_dev(refs), _dev(bad_off), _t([0]), _t([1]))) == want


@pytest.mark.gpu
def test_host_and_other_device_memory_is_refused(ctx):
    import defuse_b200 as d
    import torch
    lib = d.load_library()
    refs, reads = _tables([b"ACGT" * 20, b"GGCC" * 20], [b"ACGTGGCC" * 4])
    dr, dq = _dev(refs), _dev(reads)
    one = _t([0])
    host_task = np.zeros(1, np.int32)
    out = torch.empty(1, dtype=torch.int32, device="cuda:0")
    n_rows, n_cols = ctypes.c_int64(), ctypes.c_int64()
    sp = d._SplitParams(2, -1, -2, 0, 8)
    rt, st = dr.c_struct(), dq.c_struct()
    rc = lib.dfb_split_align_device(ctx._h, ctypes.byref(sp), ctypes.byref(rt), ctypes.byref(st), host_task.ctypes.data,
                                    one.data_ptr(), one.data_ptr(), 1, out.data_ptr(), ctypes.byref(n_rows), ctypes.byref(n_cols))
    assert rc == 2 and b"not device memory" in lib.dfb_last_error(ctx._h)
    pinned = torch.zeros(1, dtype=torch.int32).pin_memory()
    rc = lib.dfb_split_align_device(ctx._h, ctypes.byref(sp), ctypes.byref(rt), ctypes.byref(st), one.data_ptr(), one.data_ptr(),
                                    one.data_ptr(), 1, pinned.data_ptr(), ctypes.byref(n_rows), ctypes.byref(n_cols))
    assert rc == 2
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU visible: no other device's memory to refuse")
    other = torch.zeros(1, dtype=torch.int32, device="cuda:1")
    rc = lib.dfb_split_align_device(ctx._h, ctypes.byref(sp), ctypes.byref(rt), ctypes.byref(st), other.data_ptr(), one.data_ptr(),
                                    one.data_ptr(), 1, out.data_ptr(), ctypes.byref(n_rows), ctypes.byref(n_cols))
    assert rc == 2


@pytest.mark.gpu
@pytest.mark.parametrize("side_stream", [True, False])
def test_inputs_written_on_the_current_stream_are_seen(ctx, orc, side_stream):
    """a torch kernel on the current stream (a side stream, or torch's default stream) writes an input right before the
    call, behind a long sleep: the call must wait for it"""
    import contextlib
    import defuse_b200 as d
    import torch
    rng = np.random.default_rng(41)
    refs, reads, tc, tr = util.split_batch(rng, 40, 20, 100, 280, 420)
    refs, reads = _tables(refs, reads)
    ms = np.array([d.split_min_score(reads.length(r)) for r in tr], np.int32)
    al = d.SplitReadAligner(ctx=ctx)
    want = al.align_batch(refs, reads, tc, tr, ms)
    torch.cuda.synchronize()
    s = torch.cuda.Stream() if side_stream else torch.cuda.current_stream()
    with torch.cuda.stream(s) if side_stream else contextlib.nullcontext():
        dr, dq = _dev(refs), _dev(reads)
        src = _t(tr)
        torch.cuda._sleep(20_000_000)                    # keeps the stream busy: the kernels below are late
        task_read = torch.zeros_like(src)
        task_read.copy_(src)                             # written by a kernel right before the call
        got = al.align_device(dr, dq, _t(tc), task_read, _t(ms)).to_host()
    s.synchronize()
    assert np.array_equal(got.best, want.best) and got.rows.tobytes() == want.rows.tobytes()
    assert np.array_equal(got.cols, want.cols)
    # the simple form too
    sal = d.SimpleAligner(10, -5, -5, ctx=ctx)
    want_s = sal.align_batch(refs, reads, tc, tr)
    with torch.cuda.stream(s) if side_stream else contextlib.nullcontext():
        torch.cuda._sleep(20_000_000)
        seq_idx = torch.zeros_like(src)
        seq_idx.copy_(src)
        got_s = sal.align_device(dr, dq, _t(tc), seq_idx)
    s.synchronize()
    assert np.array_equal(got_s.cpu().numpy(), want_s)


@pytest.mark.gpu
def test_only_counters_cross_pcie(ctx):
    import defuse_b200 as d
    import synth
    sizes = []
    for n_clusters in (300, 3000):
        w = synth.split_workload(3, n_clusters, 100)
        refs, reads = d.SeqTable(w["ref_bytes"], w["ref_off"]), d.SeqTable(w["read_bytes"], w["read_off"])
        d.SplitReadAligner(ctx=ctx).align_device(_dev(refs), _dev(reads), _t(w["task_cluster"]), _t(w["task_read"]),
                                                 _t(w["min_score"]))
        st = ctx.split_result_stats()
        assert st["generic_jobs"] == 0
        sizes.append((st["h2d_bytes"], st["d2h_bytes"]))
    for h2d, d2h in sizes:
        assert h2d < 16384 and d2h < 16384        # a few KB per chunk
    assert sizes[0] == sizes[1] or max(sizes[1]) < 16384
    with pytest.raises(d.DefuseB200Error):
        ctx._check(ctx._lib.dfb_split_result_size(ctx._h, None, None))  # the result is in device memory
