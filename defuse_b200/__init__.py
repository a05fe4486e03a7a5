"""defuse_b200 -- B200-native (sm_100a) DP alignment hot path of deFuse.

Python face of the C ABI in include/defuse_b200.h (ctypes; no torch types cross the
boundary).  The classes mirror the reference's two aligner classes:

  SimpleAligner(match, mismatch, gap).Align(reference, sequence)      tools/SimpleAligner.h:20-22
  SplitReadAligner(match, mismatch, gap, endGaps, minSplitScore)
      .Align(read, reference1, reference2); .GetAlignments(minScore, ...)   tools/SplitReadAligner.h:35-38

plus their batch forms, which is what the GPU wants.  There is NO CPU implementation in this
package: importing works anywhere (so that CPU-only tests can check the ABI surface), but
creating a Context without the built library or without a B200 raises.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# (DFB_LIB_PATH: another build of the same CUDA library, for A/B runs of kernel variants; never a fallback)
LIB_PATH = os.environ.get("DFB_LIB_PATH") or os.path.join(_HERE, "libdefuse_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "defuse_b200.h")

DFB_OK = 0
STATUS_NAMES = {0: "DFB_OK", 1: "DFB_ERR_CUDA", 2: "DFB_ERR_ARG", 3: "DFB_ERR_NOMEM", 4: "DFB_ERR_NODEVICE",
                5: "DFB_ERR_STATE"}

MICROBENCH_KINDS = {
    0: "VIADDMNMX.S16x2", 1: "VIMNMX.U16x2", 2: "VIMNMX3.S16x2", 3: "LOP3", 4: "IMAD", 5: "IADD3", 6: "PRMT",
    7: "dp_cell_body_s16x2", 8: "SHFL.UP", 9: "VIADDMNMX.S32",
}


class DefuseB200Error(RuntimeError):
    def __init__(self, status, message):
        super().__init__("%s: %s" % (STATUS_NAMES.get(status, status), message))
        self.status = status


class _SeqTable(ctypes.Structure):
    _fields_ = [("bytes", ctypes.c_void_p), ("off", ctypes.c_void_p), ("n", ctypes.c_int64)]


class _DeviceSeqTable(ctypes.Structure):
    _fields_ = [("bytes", ctypes.c_void_p), ("off", ctypes.c_void_p), ("n", ctypes.c_int64), ("n_bytes", ctypes.c_int64)]


class _SimpleParams(ctypes.Structure):
    _fields_ = [("match", ctypes.c_int32), ("mismatch", ctypes.c_int32), ("gap", ctypes.c_int32)]


class _SplitParams(ctypes.Structure):
    _fields_ = [("match", ctypes.c_int32), ("mismatch", ctypes.c_int32), ("gap", ctypes.c_int32),
                ("end_gaps", ctypes.c_int32), ("min_split_score", ctypes.c_int32)]


class _PlanStats(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int64) for n in
                ("n_tasks", "cells", "fast_jobs", "generic_jobs", "probe_jobs", "events", "kernel_launches",
                 "h2d_bytes", "d2h_bytes", "packed_bytes", "raw_bytes")] + \
               [(n, ctypes.c_double) for n in ("ms_pack", "ms_sweep", "ms_probe")]


class _DeviceInfo(ctypes.Structure):
    _fields_ = [("name", ctypes.c_char * 128), ("ordinal", ctypes.c_int32), ("sm_count", ctypes.c_int32),
                ("cc_major", ctypes.c_int32), ("cc_minor", ctypes.c_int32), ("clock_khz", ctypes.c_int32),
                ("total_mem", ctypes.c_int64)]


SPLIT_ROW_DTYPE = np.dtype([("task", "<i4"), ("read_split", "<i4"), ("score1", "<i4"), ("score2", "<i4"),
                            ("col_begin", "<i8"), ("n1", "<i4"), ("n2", "<i4")])
assert SPLIT_ROW_DTYPE.itemsize == 32

# dfb_split_record: what SplitAlignmentTask::Align keeps per distinct refSplit (DeviceSplitResult.records())
SPLIT_RECORD_DTYPE = np.dtype([("task", "<i4"), ("ref_split1", "<i4"), ("ref_split2", "<i4"), ("read_split1", "<i4"),
                               ("read_split2", "<i4"), ("score", "<i4")])
assert SPLIT_RECORD_DTYPE.itemsize == 24

_lib = None


def build(verbose=False):
    """Compile libdefuse_b200.so for sm_100a (nvcc cross-compiles without a GPU)."""
    out = None if verbose else subprocess.DEVNULL
    subprocess.run(["make", "-C", os.path.join(_HERE, "csrc"), "all"], check=True, stdout=out)
    if os.path.exists(os.path.join(_HERE, "host", "Makefile")):
        subprocess.run(["make", "-C", os.path.join(_HERE, "host"), "all"], check=True, stdout=out)


def load_library():
    """Load the C ABI.  Raises if the CUDA extension has not been built -- there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DefuseB200Error(4, "CUDA extension %s is missing; run __graft_entry__.build() (no CPU fallback exists)"
                              % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    vp, i32, i64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64
    P = ctypes.POINTER
    sig = {
        "dfb_abi_version": ([], ctypes.c_int),
        "dfb_device_count": ([], ctypes.c_int),
        "dfb_ctx_create": ([ctypes.c_int, P(vp)], ctypes.c_int),
        "dfb_ctx_destroy": ([vp], None),
        "dfb_last_error": ([vp], ctypes.c_char_p),
        "dfb_ctx_set_stream": ([vp, vp], ctypes.c_int),
        "dfb_ctx_device_info": ([vp, P(_DeviceInfo)], ctypes.c_int),
        "dfb_simple_align_batch": ([vp, P(_SimpleParams), P(_SeqTable), P(_SeqTable), vp, vp, i64, vp], ctypes.c_int),
        "dfb_split_align_batch": ([vp, P(_SplitParams), P(_SeqTable), P(_SeqTable), vp, vp, vp, i64, vp], ctypes.c_int),
        "dfb_split_result_size": ([vp, P(i64), P(i64)], ctypes.c_int),
        "dfb_split_result_copy": ([vp, vp, vp], ctypes.c_int),
        "dfb_split_result_view": ([vp, P(vp), P(i64), P(vp), P(i64)], ctypes.c_int),
        "dfb_split_plan_view": ([vp, P(vp), P(i64), P(vp), P(i64)], ctypes.c_int),
        "dfb_simple_plan_create": ([vp, P(_SimpleParams), P(_SeqTable), P(_SeqTable), vp, vp, i64, P(vp)], ctypes.c_int),
        "dfb_split_plan_create": ([vp, P(_SplitParams), P(_SeqTable), P(_SeqTable), vp, vp, vp, i64, P(vp)], ctypes.c_int),
        "dfb_plan_run": ([vp], ctypes.c_int),
        "dfb_plan_sync": ([vp], ctypes.c_int),
        "dfb_plan_set_timing": ([vp, ctypes.c_int], ctypes.c_int),
        "dfb_simple_plan_fetch": ([vp, vp], ctypes.c_int),
        "dfb_split_plan_fetch": ([vp, vp, P(i64), P(i64)], ctypes.c_int),
        "dfb_split_plan_copy": ([vp, vp, vp], ctypes.c_int),
        "dfb_plan_get_stats": ([vp, P(_PlanStats)], ctypes.c_int),
        "dfb_split_result_stats": ([vp, P(_PlanStats)], ctypes.c_int),
        "dfb_plan_destroy": ([vp], None),
        "dfb_microbench_issue_rate": ([vp, ctypes.c_int, ctypes.c_int, P(ctypes.c_double), P(ctypes.c_double)], ctypes.c_int),
        "dfb_ctx_memory_info": ([vp, ctypes.c_int, P(i64), P(i64), P(i64)], ctypes.c_int),
        "dfb_simple_align_device": ([vp, P(_SimpleParams), P(_DeviceSeqTable), P(_DeviceSeqTable), vp, vp, i64, vp], ctypes.c_int),
        "dfb_split_align_device": ([vp, P(_SplitParams), P(_DeviceSeqTable), P(_DeviceSeqTable), vp, vp, vp, i64, vp, P(i64), P(i64)],
                                   ctypes.c_int),
        "dfb_split_result_copy_device": ([vp, vp, vp], ctypes.c_int),
        "dfb_split_records_device": ([vp, P(_DeviceSeqTable), P(_DeviceSeqTable), vp, vp, i64, vp, i64, vp, i64, P(i64)], ctypes.c_int),
        "dfb_split_records_copy_device": ([vp, vp], ctypes.c_int),
        "dfb_split_backtrace_batch": ([vp, P(_SplitParams), P(_SeqTable), P(_SeqTable), vp, vp, vp, vp, vp, i64, vp, vp, i64,
                                       P(i64)], ctypes.c_int),
        "dfb_split_backtrace_device": ([vp, P(_SplitParams), P(_DeviceSeqTable), P(_DeviceSeqTable), vp, vp, i64, vp, i64, P(i64)],
                                       ctypes.c_int),
        "dfb_split_backtrace_copy_device": ([vp, vp, vp], ctypes.c_int),
    }
    for name, (args, res) in sig.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = res
    _lib = lib
    return lib


ABI_SYMBOLS = (
    "dfb_abi_version", "dfb_device_count", "dfb_ctx_create", "dfb_ctx_destroy", "dfb_last_error", "dfb_ctx_set_stream",
    "dfb_ctx_device_info", "dfb_simple_align_batch", "dfb_split_align_batch", "dfb_split_result_size",
    "dfb_split_result_copy", "dfb_split_result_view", "dfb_split_plan_view", "dfb_simple_plan_create", "dfb_split_plan_create", "dfb_plan_run", "dfb_plan_sync",
    "dfb_plan_set_timing",
    "dfb_simple_plan_fetch", "dfb_split_plan_fetch", "dfb_split_plan_copy", "dfb_plan_get_stats", "dfb_plan_destroy",
    "dfb_microbench_issue_rate", "dfb_split_backtrace_batch", "dfb_ctx_memory_info",
    "dfb_split_result_stats", "dfb_simple_align_device", "dfb_split_align_device", "dfb_split_result_copy_device",
    "dfb_split_records_device", "dfb_split_records_copy_device", "dfb_split_backtrace_device", "dfb_split_backtrace_copy_device",
)


# ------------------------------------------------------------------------------------------------
# tables
# ------------------------------------------------------------------------------------------------

class SeqTable:
    """CSR table of byte strings (the batch form of `const string&`)."""

    def __init__(self, data, off):
        self.data = np.ascontiguousarray(data, dtype=np.uint8)
        self.off = np.ascontiguousarray(off, dtype=np.int64)
        assert self.off.ndim == 1 and self.off.size >= 1
        self._keep = self.data if self.data.size else np.zeros(1, dtype=np.uint8)

    @classmethod
    def from_list(cls, seqs):
        seqs = [bytes(s) for s in seqs]
        off = np.zeros(len(seqs) + 1, dtype=np.int64)
        if seqs:
            off[1:] = np.cumsum([len(s) for s in seqs])
        data = np.frombuffer(b"".join(seqs), dtype=np.uint8) if seqs else np.zeros(0, dtype=np.uint8)
        return cls(data, off)

    def __len__(self):
        return self.off.size - 1

    def length(self, k):
        return int(self.off[k + 1] - self.off[k])

    def get(self, k):
        return self.data[self.off[k]:self.off[k + 1]].tobytes()

    def c_struct(self):
        return _SeqTable(self._keep.ctypes.data, self.off.ctypes.data, len(self))


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _check_tensor(name, t, dtype, device=None):
    """A contiguous 1-D CUDA tensor of `dtype` (on `device` when given); TypeError / ValueError otherwise."""
    import torch
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor, got %s" % (name, type(t).__name__))
    if t.dtype != dtype:
        raise TypeError("%s must be %s, got %s" % (name, dtype, t.dtype))
    if not t.is_cuda:
        raise ValueError("%s must be a CUDA tensor, got one on %s" % (name, t.device))
    if device is not None and t.device != device:
        raise ValueError("%s is on %s, expected %s" % (name, t.device, device))
    if t.dim() != 1 or not t.is_contiguous():
        raise ValueError("%s must be a contiguous 1-D tensor" % name)
    return t


def _dptr(t):
    """Device address of a tensor; a placeholder for an empty one (the library reads nothing through it)."""
    return t.data_ptr() if t.numel() else 0


class DeviceSeqTable:
    """CSR table of byte strings in GPU memory: `data` (torch.uint8) and `off` (torch.int64, n + 1 entries), contiguous
    CUDA tensors on one device.  The device-resident aligner calls read them where they are."""

    def __init__(self, data, off):
        import torch
        _check_tensor("data", data, torch.uint8)
        _check_tensor("off", off, torch.int64, data.device)
        if off.numel() < 1:
            raise ValueError("off must hold n + 1 >= 1 entries")
        self.data = data
        self.off = off
        self.device = data.device

    @classmethod
    def from_host(cls, table, device):
        """The device copy of a SeqTable."""
        import torch
        data = table.data if table.data.flags.writeable else table.data.copy()   # (torch refuses read-only arrays)
        return cls(torch.from_numpy(data).to(device), torch.from_numpy(table.off).to(device))

    def __len__(self):
        return self.off.numel() - 1

    def c_struct(self):
        return _DeviceSeqTable(_dptr(self.data), _dptr(self.off), len(self), self.data.numel())


# ------------------------------------------------------------------------------------------------
# context and plans
# ------------------------------------------------------------------------------------------------

class Context:
    """One per GPU (dfb_ctx)."""

    def __init__(self, device=0):
        self._lib = load_library()
        h = ctypes.c_void_p()
        rc = self._lib.dfb_ctx_create(int(device), ctypes.byref(h))
        if rc != DFB_OK:
            raise DefuseB200Error(rc, self._lib.dfb_last_error(None).decode())
        self._h = h
        self.device = int(device)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.dfb_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != DFB_OK:
            raise DefuseB200Error(rc, self._lib.dfb_last_error(self._h).decode())

    def set_stream(self, cuda_stream_ptr):
        """Run on a caller's cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream); None resets."""
        self._check(self._lib.dfb_ctx_set_stream(self._h, ctypes.c_void_p(cuda_stream_ptr or 0)))
        self._stream = cuda_stream_ptr or None

    def _on_torch_stream(self, fn):
        """fn() with the context on torch's current stream of its device; the context's stream is restored after."""
        import torch
        prev = getattr(self, "_stream", None)
        # torch's default stream is the legacy NULL stream (handle 0); the library takes NULL to mean its own non-blocking
        # stream, which would not wait for torch's work, so it gets cudaStreamLegacy ((cudaStream_t)1) instead
        self.set_stream(torch.cuda.current_stream(self.device).cuda_stream or 1)
        try:
            return fn()
        finally:
            self.set_stream(prev)

    def device_info(self):
        info = _DeviceInfo()
        self._check(self._lib.dfb_ctx_device_info(self._h, ctypes.byref(info)))
        return {"name": info.name.decode(), "ordinal": info.ordinal, "sm_count": info.sm_count,
                "cc": (info.cc_major, info.cc_minor), "clock_khz": info.clock_khz, "total_mem": info.total_mem}

    def split_result_stats(self):
        """Accounting of the last one-call split batch on this context (what the call itself copied and launched)."""
        st = _PlanStats()
        self._check(self._lib.dfb_split_result_stats(self._h, ctypes.byref(st)))
        return {n: getattr(st, n) for n, _ in _PlanStats._fields_}

    def memory_info(self, reset=False):
        """Device memory of the context's pool: (reserved now, reserved high-water mark, used high-water mark) in bytes."""
        a, b, c = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64()
        self._check(self._lib.dfb_ctx_memory_info(self._h, int(bool(reset)), ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)))
        return a.value, b.value, c.value

    def microbench_issue_rate(self, kind, iters=2000):
        rate = ctypes.c_double()
        ms = ctypes.c_double()
        self._check(self._lib.dfb_microbench_issue_rate(self._h, int(kind), int(iters), ctypes.byref(rate), ctypes.byref(ms)))
        return rate.value, ms.value


_default_ctx = {}


def default_context(device=0):
    if device not in _default_ctx:
        _default_ctx[device] = Context(device)
    return _default_ctx[device]


class _Plan:
    def __init__(self, ctx, handle, n_tasks):
        self.ctx = ctx
        self._h = handle
        self.n_tasks = n_tasks

    def run(self):
        """Enqueue every DP kernel of the batch on the context's stream (no synchronisation)."""
        self.ctx._check(self.ctx._lib.dfb_plan_run(self._h))

    def sync(self):
        self.ctx._check(self.ctx._lib.dfb_plan_sync(self._h))

    def set_timing(self, enable=True):
        """Bracket the kernel groups of run() with CUDA events (stats: ms_sweep, ms_probe)."""
        self.ctx._check(self.ctx._lib.dfb_plan_set_timing(self._h, int(bool(enable))))

    def stats(self):
        st = _PlanStats()
        self.ctx._check(self.ctx._lib.dfb_plan_get_stats(self._h, ctypes.byref(st)))
        return {n: getattr(st, n) for n, _ in _PlanStats._fields_}

    def close(self):
        if self._h:
            self.ctx._lib.dfb_plan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class SimplePlan(_Plan):
    def fetch(self, out=None):
        if out is None:
            out = np.zeros(self.n_tasks, dtype=np.int32)
        self.ctx._check(self.ctx._lib.dfb_simple_plan_fetch(self._h, out.ctypes.data))
        return out


class SplitResult:
    """Winning split rows of a batch, in task order (dfb_split_row + column pool)."""

    def __init__(self, best, rows, cols, lens):
        self.best = best
        self.rows = rows
        self.cols = cols
        self._lens = lens  # callable -> (read_len[task], ref2_len[task]); evaluated on first use
        self._lens_cache = None
        self._row_start_cache = None

    @property
    def _read_len(self):
        if self._lens_cache is None:
            self._lens_cache = self._lens()
        return self._lens_cache[0]

    @property
    def _ref2_len(self):
        if self._lens_cache is None:
            self._lens_cache = self._lens()
        return self._lens_cache[1]

    @property
    def _row_start(self):
        if self._row_start_cache is None:
            if len(self.rows):
                self._row_start_cache = np.searchsorted(np.ascontiguousarray(self.rows["task"]), np.arange(len(self.best) + 1))
            else:
                self._row_start_cache = np.zeros(len(self.best) + 1, dtype=np.int64)
        return self._row_start_cache

    def alignments(self, task):
        """What GetAlignments appends for this task (tools/SplitReadAligner.cpp:272-297), as an (n,7) int32
        array: refSplit.first, refSplit.second, readSplit.first, readSplit.second, score, score1, score2."""
        out = []
        L = int(self._read_len[task])
        R2 = int(self._ref2_len[task])
        for r in self.rows[self._row_start[task]:self._row_start[task + 1]]:
            c1 = self.cols[r["col_begin"]:r["col_begin"] + r["n1"]]
            c2 = self.cols[r["col_begin"] + r["n1"]:r["col_begin"] + r["n1"] + r["n2"]]
            a = int(r["read_split"])
            for i1 in c1:
                for i2 in c2:
                    out.append((int(i1), R2 - int(i2) - 1, a, L - a, int(r["score1"]) + int(r["score2"]),
                                int(r["score1"]), int(r["score2"])))
        return np.array(out, dtype=np.int32).reshape(-1, 7)

    def records(self, task):
        """The records SplitAlignmentTask::Align keeps (tools/SplitAlignment.cpp:381-400): first alignment per
        distinct refSplit, score = min(score1, score2): (k,5) refSplit.first, refSplit.second, readSplit.first,
        readSplit.second, score."""
        seen = set()
        out = []
        for a in self.alignments(task):
            key = (int(a[0]), int(a[1]))
            if key in seen:
                continue
            seen.add(key)
            out.append((a[0], a[1], a[2], a[3], min(a[5], a[6])))
        return np.array(out, dtype=np.int32).reshape(-1, 5)


class DeviceSplitResult:
    """Result of SplitReadAligner.align_device, in GPU memory: `best` (int32, per task), `rows` (the 32-byte
    dfb_split_row records as an (n, 8) int32 tensor; the field accessors below read it) and `cols` (int32 column pool).
    It keeps the context, the tables and the task tensors of the batch it was computed from, and the aligner's scoring
    (`params`), which backtrace() uses."""

    def __init__(self, best, rows, cols, ctx, refs, reads, task_cluster, task_read, params=None):
        self.best = best
        self.rows = rows
        self.cols = cols
        self.ctx = ctx
        self.refs = refs
        self.reads = reads
        self.task_cluster = task_cluster
        self.task_read = task_read
        self.params = params

    def _lens(self):
        tc, tr = self.task_cluster.cpu().numpy(), self.task_read.cpu().numpy()
        return SplitReadAligner._lens(SeqTable(np.zeros(0, np.uint8), self.refs.off.cpu().numpy()),
                                      SeqTable(np.zeros(0, np.uint8), self.reads.off.cpu().numpy()), tc, tr)

    # fields of the records (SPLIT_ROW_DTYPE): task, read_split, score1, score2, col_begin (int64), n1, n2
    @property
    def task(self):
        return self.rows[:, 0]

    @property
    def read_split(self):
        return self.rows[:, 1]

    @property
    def score1(self):
        return self.rows[:, 2]

    @property
    def score2(self):
        return self.rows[:, 3]

    @property
    def col_begin(self):
        import torch
        return self.rows[:, 4:6].contiguous().view(torch.int64).reshape(-1)

    @property
    def n1(self):
        return self.rows[:, 6]

    @property
    def n2(self):
        return self.rows[:, 7]

    def to_host(self):
        """The same result as a SplitResult (host arrays), so that alignments() / records() work.  The read and window
        lengths it needs are read from the batch's tables and task tensors now: call it before reusing them."""
        rows = np.ascontiguousarray(self.rows.cpu().numpy()).view(SPLIT_ROW_DTYPE).reshape(-1)
        lens = self._lens()
        return SplitResult(self.best.cpu().numpy(), rows, self.cols.cpu().numpy(), lambda: lens)

    def records(self):
        """The records SplitAlignmentTask::Align keeps for every task (tools/SplitAlignment.cpp:381-400), expanded and
        de-duplicated on the GPU through dfb_split_records_device: an (n, 6) int32 CUDA tensor with the columns of
        SPLIT_RECORD_DTYPE (task, ref_split1, ref_split2, read_split1, read_split2, score), in task order and, within
        a task, in GetAlignments' order -- np.concatenate of SplitResult.records(t) with the task prepended.  Runs on
        torch's current stream.  The read and window lengths come from the batch's tables and task tensors: they must
        not have been reused since the align_device call."""
        import torch
        ctx, lib = self.ctx, self.ctx._lib
        _check_tensor("cols", self.cols, torch.int32, self.rows.device)
        if self.rows.dtype != torch.int32 or self.rows.dim() != 2 or self.rows.shape[1] != 8 or not self.rows.is_contiguous():
            raise ValueError("rows must be a contiguous (n, 8) int32 tensor of dfb_split_row records")
        rt, st = self.refs.c_struct(), self.reads.c_struct()
        n = ctypes.c_int64()

        def run():
            ctx._check(lib.dfb_split_records_device(ctx._h, ctypes.byref(rt), ctypes.byref(st), _dptr(self.task_cluster),
                                                    _dptr(self.task_read), self.task_cluster.numel(), _dptr(self.rows),
                                                    self.rows.shape[0], _dptr(self.cols), self.cols.numel(), ctypes.byref(n)))
            out = torch.empty((n.value, 6), dtype=torch.int32, device=self.rows.device)
            ctx._check(lib.dfb_split_records_copy_device(ctx._h, _dptr(out)))
            return out
        return ctx._on_torch_stream(run)

    def backtrace(self, records):
        """matches1 / matches2 of chosen alignments (GetAlignments(..., backtrace=True)) through
        dfb_split_backtrace_device, with the scoring of the align_device call: the device twin of
        SplitReadAligner.backtrace_batch.  `records` is an (n, 6) int32 CUDA tensor of SPLIT_RECORD_DTYPE rows -- the
        output of records() or any rows of it, in any order; record k names the alignment of task records[k, 0] with
        refSplit (records[k, 1], records[k, 2]) and readSplit records[k, 3:5].  Returns (match_off, pairs): an int64
        CUDA tensor of 2n + 1 entries and an (n_pairs, 2) int32 CUDA tensor of (refPos, readPos) rows, with
        pairs[match_off[2k]:match_off[2k+1]] = matches1 of record k and pairs[match_off[2k+1]:match_off[2k+2]] its
        matches2.  Runs on torch's current stream.  The tables and task tensors must not have been reused since the
        align_device call."""
        import torch
        if not isinstance(records, torch.Tensor):
            raise TypeError("records must be a torch.Tensor, got %s" % type(records).__name__)
        if records.dtype != torch.int32:
            raise TypeError("records must be torch.int32, got %s" % records.dtype)
        if not records.is_cuda:
            raise ValueError("records must be a CUDA tensor, got one on %s" % records.device)
        if records.device != self.rows.device:
            raise ValueError("records is on %s, the result on %s" % (records.device, self.rows.device))
        if records.dim() != 2 or records.shape[1] != 6 or not records.is_contiguous():
            raise ValueError("records must be a contiguous (n, 6) int32 tensor of dfb_split_record rows")
        if self.params is None:
            raise ValueError("this result carries no scoring: it was not made by SplitReadAligner.align_device")
        ctx, lib = self.ctx, self.ctx._lib
        rt, st = self.refs.c_struct(), self.reads.c_struct()
        n = records.shape[0]
        total = ctypes.c_int64()

        def run():
            ctx._check(lib.dfb_split_backtrace_device(ctx._h, ctypes.byref(self.params), ctypes.byref(rt), ctypes.byref(st),
                                                      _dptr(self.task_cluster), _dptr(self.task_read), self.task_cluster.numel(),
                                                      _dptr(records), n, ctypes.byref(total)))
            off = torch.empty(2 * n + 1, dtype=torch.int64, device=records.device)
            pairs = torch.empty((total.value, 2), dtype=torch.int32, device=records.device)
            ctx._check(lib.dfb_split_backtrace_copy_device(ctx._h, _dptr(off), _dptr(pairs)))
            return off, pairs
        return ctx._on_torch_stream(run)


def _view_arrays(rows_p, n_rows, cols_p, n_cols, copy):
    """numpy arrays over (or copied from) the library-owned result buffers."""
    if n_rows:
        rows = np.frombuffer((ctypes.c_char * (n_rows * SPLIT_ROW_DTYPE.itemsize)).from_address(rows_p), dtype=SPLIT_ROW_DTYPE)
    else:
        rows = np.zeros(0, dtype=SPLIT_ROW_DTYPE)
    if n_cols:
        cols = np.frombuffer((ctypes.c_char * (n_cols * 4)).from_address(cols_p), dtype=np.int32)
    else:
        cols = np.zeros(0, dtype=np.int32)
    if copy:
        rows, cols = rows.copy(), cols.copy()
    return rows, cols


class SplitPlan(_Plan):
    def __init__(self, ctx, handle, n_tasks, lens):
        super().__init__(ctx, handle, n_tasks)
        self._lens = lens

    def fetch(self, copy=True):
        """Results of the last run.  copy=False returns views into library memory that stay valid until the
        next fetch on this plan."""
        best = np.zeros(self.n_tasks, dtype=np.int32)
        n_rows = ctypes.c_int64()
        n_cols = ctypes.c_int64()
        lib = self.ctx._lib
        self.ctx._check(lib.dfb_split_plan_fetch(self._h, best.ctypes.data, ctypes.byref(n_rows), ctypes.byref(n_cols)))
        rp, cp = ctypes.c_void_p(), ctypes.c_void_p()
        self.ctx._check(lib.dfb_split_plan_view(self._h, ctypes.byref(rp), ctypes.byref(n_rows), ctypes.byref(cp), ctypes.byref(n_cols)))
        rows, cols = _view_arrays(rp.value, n_rows.value, cp.value, n_cols.value, copy)
        return SplitResult(best, rows, cols, self._lens)


# ------------------------------------------------------------------------------------------------
# the reference's operator interface
# ------------------------------------------------------------------------------------------------

class SimpleAligner:
    """SimpleAligner(matchScore, misMatchScore, gapScore) -- tools/SimpleAligner.h:20."""

    def __init__(self, match, mismatch, gap, ctx=None):
        self.params = _SimpleParams(int(match), int(mismatch), int(gap))
        self.ctx = ctx or default_context()

    def plan(self, refs, seqs, task_ref, task_seq):
        task_ref, task_seq = _i32(task_ref), _i32(task_seq)
        assert task_ref.shape == task_seq.shape
        h = ctypes.c_void_p()
        rt, st = refs.c_struct(), seqs.c_struct()
        self.ctx._check(self.ctx._lib.dfb_simple_plan_create(self.ctx._h, ctypes.byref(self.params), ctypes.byref(rt),
                                                             ctypes.byref(st), task_ref.ctypes.data, task_seq.ctypes.data,
                                                             task_ref.size, ctypes.byref(h)))
        return SimplePlan(self.ctx, h, task_ref.size)

    def align_batch(self, refs, seqs, task_ref, task_seq, out=None):
        """out[t] = Align(refs[task_ref[t]], seqs[task_seq[t]]) through dfb_simple_align_batch (host buffers in,
        host buffer out)."""
        task_ref, task_seq = _i32(task_ref), _i32(task_seq)
        if out is None:
            out = np.empty(task_ref.size, dtype=np.int32)   # (the call writes every entry)
        rt, st = refs.c_struct(), seqs.c_struct()
        self.ctx._check(self.ctx._lib.dfb_simple_align_batch(self.ctx._h, ctypes.byref(self.params), ctypes.byref(rt),
                                                             ctypes.byref(st), task_ref.ctypes.data, task_seq.ctypes.data,
                                                             task_ref.size, out.ctypes.data))
        return out

    def align_device(self, refs, seqs, task_ref, task_seq, out=None):
        """align_batch for a batch in GPU memory (DeviceSeqTable, int32 CUDA tensors) through dfb_simple_align_device:
        nothing but counters crosses PCIe.  Returns `out` (int32 CUDA tensor), written on torch's current stream."""
        import torch
        dev = _device_args(self.ctx, refs, seqs)
        _check_tensor("task_ref", task_ref, torch.int32, dev)
        _check_tensor("task_seq", task_seq, torch.int32, dev)
        if task_ref.numel() != task_seq.numel():
            raise ValueError("task_ref and task_seq differ in length")
        n = task_ref.numel()
        if out is None:
            out = torch.empty(n, dtype=torch.int32, device=dev)
        _check_tensor("out", out, torch.int32, dev)
        if out.numel() < n:
            raise ValueError("out holds fewer than n_tasks entries")
        rt, st = refs.c_struct(), seqs.c_struct()
        lib = self.ctx._lib
        self.ctx._on_torch_stream(lambda: self.ctx._check(lib.dfb_simple_align_device(
            self.ctx._h, ctypes.byref(self.params), ctypes.byref(rt), ctypes.byref(st), _dptr(task_ref), _dptr(task_seq), n,
            _dptr(out))))
        return out

    def Align(self, reference, sequence):
        """int SimpleAligner::Align(const string& reference, const string& sequence)."""
        return int(self.align_batch(SeqTable.from_list([reference]), SeqTable.from_list([sequence]), [0], [0])[0])


class SplitReadAligner:
    """SplitReadAligner(matchScore, misMatchScore, gapScore, endGaps, minSplitScore) -- tools/SplitReadAligner.h:35."""

    def __init__(self, match=2, mismatch=-1, gap=-2, end_gaps=False, min_split_score=8, ctx=None):
        self.params = _SplitParams(int(match), int(mismatch), int(gap), int(bool(end_gaps)), int(min_split_score))
        self.ctx = ctx or default_context()
        self._last = None
        self._best_buf = None

    @staticmethod
    def _lens(refs, reads, task_cluster, task_read):
        read_len = (reads.off[1:] - reads.off[:-1])[task_read].astype(np.int32) if len(task_read) else np.zeros(0, np.int32)
        ref_len = refs.off[1:] - refs.off[:-1]
        ref2_len = ref_len[2 * task_cluster.astype(np.int64) + 1].astype(np.int32) if len(task_cluster) else np.zeros(0, np.int32)
        return read_len, ref2_len

    def plan(self, refs, reads, task_cluster, task_read, task_min_score):
        task_cluster, task_read, task_min_score = _i32(task_cluster), _i32(task_read), _i32(task_min_score)
        h = ctypes.c_void_p()
        rt, st = refs.c_struct(), reads.c_struct()
        self.ctx._check(self.ctx._lib.dfb_split_plan_create(self.ctx._h, ctypes.byref(self.params), ctypes.byref(rt),
                                                            ctypes.byref(st), task_cluster.ctypes.data, task_read.ctypes.data,
                                                            task_min_score.ctypes.data, task_cluster.size, ctypes.byref(h)))
        return SplitPlan(self.ctx, h, task_cluster.size, lambda: self._lens(refs, reads, task_cluster, task_read))

    def align_batch(self, refs, reads, task_cluster, task_read, task_min_score, copy=True):
        """Batch of Align + GetAlignments(minScore, forceSplits=True, firstOnly=False) through
        dfb_split_align_batch; cluster c uses refs[2c] / refs[2c+1].  copy=False returns views into
        library memory (and, for `best`, into a buffer of this aligner) that stay valid until the next split call."""
        task_cluster, task_read, task_min_score = _i32(task_cluster), _i32(task_read), _i32(task_min_score)
        n = task_cluster.size
        if copy:
            best = np.empty(n, dtype=np.int32)   # (the call writes every entry)
        else:
            # views all round: `best` too lives in a buffer of this aligner that the next call reuses -- a fresh 4 n-byte
            # array per call is 2 000 page faults per 2 M tasks under the library's copies
            if self._best_buf is None or self._best_buf.size < n:
                self._best_buf = np.empty(max(n, 1), dtype=np.int32)
            best = self._best_buf[:n]
        rt, st = refs.c_struct(), reads.c_struct()
        lib = self.ctx._lib
        self.ctx._check(lib.dfb_split_align_batch(self.ctx._h, ctypes.byref(self.params), ctypes.byref(rt), ctypes.byref(st),
                                                  task_cluster.ctypes.data, task_read.ctypes.data, task_min_score.ctypes.data,
                                                  task_cluster.size, best.ctypes.data))
        n_rows, n_cols = ctypes.c_int64(), ctypes.c_int64()
        rp, cp = ctypes.c_void_p(), ctypes.c_void_p()
        self.ctx._check(lib.dfb_split_result_view(self.ctx._h, ctypes.byref(rp), ctypes.byref(n_rows), ctypes.byref(cp),
                                                  ctypes.byref(n_cols)))
        rows, cols = _view_arrays(rp.value, n_rows.value, cp.value, n_cols.value, copy)
        return SplitResult(best, rows, cols, lambda: self._lens(refs, reads, task_cluster, task_read))

    def align_device(self, refs, reads, task_cluster, task_read, task_min_score, out=None):
        """align_batch for a batch in GPU memory (DeviceSeqTable, int32 CUDA tensors) through dfb_split_align_device.
        Returns a DeviceSplitResult whose best / rows / cols are CUDA tensors equal to align_batch's arrays; the work
        runs on torch's current stream and nothing but counters crosses PCIe."""
        import torch
        dev = _device_args(self.ctx, refs, reads)
        for name, t in (("task_cluster", task_cluster), ("task_read", task_read), ("task_min_score", task_min_score)):
            _check_tensor(name, t, torch.int32, dev)
        n = task_cluster.numel()
        if task_read.numel() != n or task_min_score.numel() != n:
            raise ValueError("task arrays differ in length")
        if out is None:
            out = torch.empty(n, dtype=torch.int32, device=dev)
        _check_tensor("out", out, torch.int32, dev)
        if out.numel() < n:
            raise ValueError("out holds fewer than n_tasks entries")
        rt, st = refs.c_struct(), reads.c_struct()
        lib, h = self.ctx._lib, self.ctx._h
        n_rows, n_cols = ctypes.c_int64(), ctypes.c_int64()

        def run():
            self.ctx._check(lib.dfb_split_align_device(h, ctypes.byref(self.params), ctypes.byref(rt), ctypes.byref(st),
                                                       _dptr(task_cluster), _dptr(task_read), _dptr(task_min_score), n,
                                                       _dptr(out), ctypes.byref(n_rows), ctypes.byref(n_cols)))
            rows = torch.empty((n_rows.value, 8), dtype=torch.int32, device=dev)
            cols = torch.empty(n_cols.value, dtype=torch.int32, device=dev)
            self.ctx._check(lib.dfb_split_result_copy_device(h, _dptr(rows), _dptr(cols)))
            return rows, cols

        rows, cols = self.ctx._on_torch_stream(run)
        return DeviceSplitResult(out[:n], rows, cols, self.ctx, refs, reads, task_cluster, task_read, self.params)

    def backtrace_batch(self, refs, reads, task_cluster, task_read, ref_split1, ref_split2, read_split):
        """matches1 / matches2 of chosen alignments (GetAlignments(..., backtrace=True), tools/SplitReadAligner.cpp:
        124-154,287-292) through dfb_split_backtrace_batch.  Task t names the alignment of reads[task_read[t]] against
        cluster task_cluster[t] with refSplit (ref_split1[t], ref_split2[t]) and readSplit.first read_split[t].
        Returns (match_off[2n+1], pairs[(total,2)]): pairs[match_off[2t]:match_off[2t+1]] = matches1 of task t,
        pairs[match_off[2t+1]:match_off[2t+2]] = matches2, each row (refPos, readPos)."""
        task_cluster, task_read = _i32(task_cluster), _i32(task_read)
        a1, a2, a3 = _i32(ref_split1), _i32(ref_split2), _i32(read_split)
        n = task_cluster.size
        cap = int((reads.off[1:] - reads.off[:-1])[task_read].sum()) if n else 0
        off = np.zeros(2 * n + 1, dtype=np.int64)
        pairs = np.zeros((max(cap, 1), 2), dtype=np.int32)
        total = ctypes.c_int64()
        rt, st = refs.c_struct(), reads.c_struct()
        self.ctx._check(self.ctx._lib.dfb_split_backtrace_batch(
            self.ctx._h, ctypes.byref(self.params), ctypes.byref(rt), ctypes.byref(st), task_cluster.ctypes.data,
            task_read.ctypes.data, a1.ctypes.data, a2.ctypes.data, a3.ctypes.data, n, off.ctypes.data, pairs.ctypes.data,
            cap, ctypes.byref(total)))
        return off, pairs[:total.value].copy()

    # single-task mirror of the reference's two-call protocol
    def Align(self, read, reference1, reference2):
        self._last = (bytes(read), bytes(reference1), bytes(reference2))

    def GetAlignments(self, min_score, force_splits=True, first_only=False, backtrace=False):
        """(n,7) array as the reference emits it; with backtrace=True a list of (row, matches1, matches2)."""
        if not force_splits or first_only:
            raise NotImplementedError("only forceSplits=true, firstOnly=false is on the hot path "
                                      "(tools/SplitAlignment.cpp:379)")
        read, r1, r2 = self._last
        refs, reads = SeqTable.from_list([r1, r2]), SeqTable.from_list([read])
        res = self.align_batch(refs, reads, [0], [0], [min_score])
        al = res.alignments(0)
        if not backtrace:
            return al
        n = len(al)
        off, pairs = self.backtrace_batch(refs, reads, np.zeros(n, np.int32), np.zeros(n, np.int32), al[:, 0], al[:, 1], al[:, 2])
        return [(al[k], pairs[off[2 * k]:off[2 * k + 1]], pairs[off[2 * k + 1]:off[2 * k + 2]]) for k in range(n)]


def _device_args(ctx, *tables):
    """The CUDA device of the context, which every DeviceSeqTable must be on."""
    import torch
    dev = torch.device("cuda", ctx.device)
    for t in tables:
        if not isinstance(t, DeviceSeqTable):
            raise TypeError("tables must be DeviceSeqTable, got %s" % type(t).__name__)
        if t.device != dev:
            raise ValueError("table is on %s, the context on %s" % (t.device, dev))
    return dev


def split_min_score(read_len, match=2):
    """(int)((float)readSeq.length() * (float)matchScore * 0.90) -- tools/SplitAlignment.cpp:379, evaluated in the
    same float/double steps."""
    return int(np.float64(np.float32(np.float32(read_len) * np.float32(match))) * np.float64(0.90))
