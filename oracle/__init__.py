"""TEST INFRASTRUCTURE ONLY -- ctypes loader for the parity oracle.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
may import this package.  The product (defuse_b200/) never does.

Two implementations of the same per-task interface:
  impl="port"  oracle/_build/libdp_oracle.so  -- plain-C restatement (oracle/dp_oracle.c)
  impl="ref"   oracle/_ref/libref_aligners.so -- the UNMODIFIED reference classes
               (tools/SplitReadAligner.cpp, tools/SimpleAligner.cpp) behind oracle/ref_harness.cpp
"""
import ctypes
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
PORT_LIB = os.path.join(_HERE, "_build", "libdp_oracle.so")
REF_LIB = os.path.join(_HERE, "_ref", "libref_aligners.so")
REF_DIR = os.path.join(_HERE, "_ref")

_c_u8p = ctypes.POINTER(ctypes.c_uint8)
_c_i32p = ctypes.POINTER(ctypes.c_int32)
_c_i64p = ctypes.POINTER(ctypes.c_int64)


def build(quiet=True):
    """Compile the C restatement and, when /root/reference is present, the reference."""
    out = subprocess.DEVNULL if quiet else None
    subprocess.run(["make", "-C", _HERE, "all"], check=True, stdout=out)


def have_ref():
    return os.path.exists(REF_LIB)


def ref_tool(name):
    """Path of a compiled reference tool (ref_localalign, ref_dosplitalign, ...) or None."""
    p = os.path.join(REF_DIR, name)
    return p if os.path.exists(p) else None


_libs = {}


def _lib(impl):
    if impl in _libs:
        return _libs[impl]
    if impl == "port":
        if not os.path.exists(PORT_LIB):
            build()
        lib = ctypes.CDLL(PORT_LIB)
        lib.dpo_fill_matrix.argtypes = [_c_u8p, ctypes.c_int, _c_u8p, ctypes.c_int] + [ctypes.c_int] * 4 + [_c_i32p]
        lib.dpo_fill_matrix.restype = None
        lib.dpo_simple_align.argtypes = [_c_u8p, ctypes.c_int, _c_u8p, ctypes.c_int] + [ctypes.c_int] * 3
        lib.dpo_simple_align.restype = ctypes.c_int
        lib.dpo_split_align.argtypes = ([_c_u8p, ctypes.c_int] * 3 + [ctypes.c_int] * 6 +
                                        [_c_i32p, ctypes.c_int64, _c_i32p, _c_i32p])
        lib.dpo_split_align.restype = ctypes.c_int64
        lib.dpo_split_min_score.argtypes = [ctypes.c_int, ctypes.c_int]
        lib.dpo_split_min_score.restype = ctypes.c_int
        lib.dpo_split_dedupe.argtypes = [_c_i32p, ctypes.c_int64, _c_i32p]
        lib.dpo_split_dedupe.restype = ctypes.c_int64
        lib.dpo_reverse_complement.argtypes = [_c_u8p, ctypes.c_int]
        lib.dpo_reverse_complement.restype = None
        lib.dpo_simple_align_batch.argtypes = ([ctypes.c_int] * 3 + [_c_u8p, _c_i64p, _c_u8p, _c_i64p, _c_i32p, _c_i32p,
                                                                    ctypes.c_int64, _c_i32p])
        lib.dpo_simple_align_batch.restype = ctypes.c_int64
        lib.dpo_split_align_batch.argtypes = ([ctypes.c_int] * 5 + [_c_u8p, _c_i64p, _c_u8p, _c_i64p, _c_i32p, _c_i32p,
                                                                   _c_i32p, ctypes.c_int64, _c_i32p, _c_i32p, ctypes.c_int64])
        lib.dpo_split_align_batch.restype = ctypes.c_int64
        lib.dpo_split_backtrace.argtypes = ([_c_u8p, ctypes.c_int] * 3 + [ctypes.c_int] * 7 + [_c_i32p] * 4)
        lib.dpo_split_backtrace.restype = None
        lib.dpo_split_backtrace_batch.argtypes = ([ctypes.c_int] * 4 + [_c_u8p, _c_i64p, _c_u8p, _c_i64p] + [_c_i32p] * 5 +
                                                  [ctypes.c_int64] * 2 + [_c_i64p, _c_i32p])
        lib.dpo_split_backtrace_batch.restype = ctypes.c_int64
    elif impl == "ref":
        if not os.path.exists(REF_LIB):
            raise FileNotFoundError("oracle/_ref/libref_aligners.so not built (run `make -C oracle ref` where /root/reference exists)")
        lib = ctypes.CDLL(REF_LIB)
        lib.ref_simple_align.argtypes = [ctypes.c_int] * 3 + [ctypes.c_char_p, ctypes.c_int, ctypes.c_char_p, ctypes.c_int]
        lib.ref_simple_align.restype = ctypes.c_int
        lib.ref_split_align.argtypes = ([ctypes.c_int] * 5 + [ctypes.c_char_p, ctypes.c_int] * 3 +
                                        [ctypes.c_int, _c_i32p, ctypes.c_int64])
        lib.ref_split_align.restype = ctypes.c_int64
        lib.ref_simple_align_batch.argtypes = ([ctypes.c_int] * 3 + [_c_u8p, _c_i64p, _c_u8p, _c_i64p, _c_i32p, _c_i32p,
                                                                    ctypes.c_int64, _c_i32p])
        lib.ref_simple_align_batch.restype = ctypes.c_int64
        lib.ref_split_align_batch.argtypes = ([ctypes.c_int] * 5 + [_c_u8p, _c_i64p, _c_u8p, _c_i64p, _c_i32p, _c_i32p,
                                                                   _c_i32p, ctypes.c_int64, _c_i32p, _c_i32p, ctypes.c_int64])
        lib.ref_split_align_batch.restype = ctypes.c_int64
        lib.ref_split_backtrace.argtypes = ([ctypes.c_int] * 5 + [ctypes.c_char_p, ctypes.c_int] * 3 +
                                            [ctypes.c_int, ctypes.c_int64] + [_c_i32p] * 5)
        lib.ref_split_backtrace.restype = ctypes.c_int64
        lib.ref_reverse_complement.argtypes = [ctypes.c_char_p, ctypes.c_int]
        lib.ref_reverse_complement.restype = None
    else:
        raise ValueError(impl)
    _libs[impl] = lib
    return lib


def _u8(b):
    a = np.frombuffer(bytes(b), dtype=np.uint8) if not isinstance(b, np.ndarray) else np.ascontiguousarray(b, dtype=np.uint8)
    if a.size == 0:
        a = np.zeros(1, dtype=np.uint8)[:0]
    return a


def _p(a, t):
    return a.ctypes.data_as(t)


# --------------------------------------------------------------------------------------
# per-task interface
# --------------------------------------------------------------------------------------

def simple_align(ref, seq, match, mismatch, gap, impl="port"):
    """SimpleAligner(match,mismatch,gap).Align(ref, seq) -- tools/SimpleAligner.cpp:23-63."""
    ref, seq = bytes(ref), bytes(seq)
    lib = _lib(impl)
    if impl == "ref":
        return int(lib.ref_simple_align(match, mismatch, gap, ref, len(ref), seq, len(seq)))
    r, s = _u8(ref), _u8(seq)
    return int(lib.dpo_simple_align(_p(r, _c_u8p), len(ref), _p(s, _c_u8p), len(seq), match, mismatch, gap))


def split_align(read, ref1, ref2, min_score, match=2, mismatch=-1, gap=-2, end_gaps=False, min_split_score=8,
                impl="port", cap=1 << 16):
    """SplitReadAligner(...).Align(read, ref1, ref2); GetAlignments(min_score, True, False, False).

    Returns an (n, 7) int32 array: refSplit.first, refSplit.second, readSplit.first,
    readSplit.second, score, score1, score2 -- in the reference's emission order."""
    read, ref1, ref2 = bytes(read), bytes(ref1), bytes(ref2)
    lib = _lib(impl)
    while True:
        out = np.zeros((max(cap, 1), 7), dtype=np.int32)
        if impl == "ref":
            n = lib.ref_split_align(match, mismatch, gap, int(end_gaps), min_split_score,
                                    read, len(read), ref1, len(ref1), ref2, len(ref2),
                                    min_score, _p(out, _c_i32p), cap)
        else:
            a, b, c = _u8(read), _u8(ref1), _u8(ref2)
            n = lib.dpo_split_align(_p(a, _c_u8p), len(read), _p(b, _c_u8p), len(ref1), _p(c, _c_u8p), len(ref2),
                                    match, mismatch, gap, int(end_gaps), min_split_score, min_score,
                                    _p(out, _c_i32p), cap, None, None)
        if n <= cap:
            return out[:n].copy()
        cap = int(n)


def split_align_count(read, ref1, ref2, min_score, match=2, mismatch=-1, gap=-2, end_gaps=False, min_split_score=8,
                      impl="port"):
    """Number of alignments GetAlignments would emit and the winning total (0 if none), without
    materialising them (tie-heavy inputs emit millions)."""
    read, ref1, ref2 = bytes(read), bytes(ref1), bytes(ref2)
    lib = _lib(impl)
    out = np.zeros((1, 7), dtype=np.int32)
    if impl == "ref":
        n = lib.ref_split_align(match, mismatch, gap, int(end_gaps), min_split_score,
                                read, len(read), ref1, len(ref1), ref2, len(ref2), min_score, _p(out, _c_i32p), 1)
    else:
        a, b, c = _u8(read), _u8(ref1), _u8(ref2)
        n = lib.dpo_split_align(_p(a, _c_u8p), len(read), _p(b, _c_u8p), len(ref1), _p(c, _c_u8p), len(ref2),
                                match, mismatch, gap, int(end_gaps), min_split_score, min_score,
                                _p(out, _c_i32p), 1, None, None)
    return int(n), (int(out[0, 4]) if n else 0)


def split_alignment(read, ref1, ref2, min_score, which, match=2, mismatch=-1, gap=-2, end_gaps=False, min_split_score=8):
    """Number of alignments GetAlignments would emit and alignment number `which` in emission order (None when
    there are not that many), without materialising the others (port only)."""
    read, ref1, ref2 = bytes(read), bytes(ref1), bytes(ref2)
    out = np.zeros((which + 1, 7), dtype=np.int32)
    a, b, c = _u8(read), _u8(ref1), _u8(ref2)
    n = _lib("port").dpo_split_align(_p(a, _c_u8p), len(read), _p(b, _c_u8p), len(ref1), _p(c, _c_u8p), len(ref2),
                                     match, mismatch, gap, int(end_gaps), min_split_score, min_score,
                                     _p(out, _c_i32p), which + 1, None, None)
    return int(n), (out[which].copy() if which < n else None)


def split_rowmax(read, ref1, ref2, match=2, mismatch=-1, gap=-2, end_gaps=False, min_split_score=8):
    """FindMaxRowEntry of every row of both matrices (port only): two (L+1,) int32 arrays."""
    read, ref1, ref2 = bytes(read), bytes(ref1), bytes(ref2)
    lib = _lib("port")
    L = len(read)
    rm1 = np.zeros(L + 1, dtype=np.int32)
    rm2 = np.zeros(L + 1, dtype=np.int32)
    out = np.zeros((1, 7), dtype=np.int32)
    a, b, c = _u8(read), _u8(ref1), _u8(ref2)
    lib.dpo_split_align(_p(a, _c_u8p), L, _p(b, _c_u8p), len(ref1), _p(c, _c_u8p), len(ref2),
                        match, mismatch, gap, int(end_gaps), min_split_score, 1 << 30,
                        _p(out, _c_i32p), 0, _p(rm1, _c_i32p), _p(rm2, _c_i32p))
    return rm1, rm2


def fill_matrix(ref, read, match, mismatch, gap, end_gaps=False):
    """FillMatrix (tools/SplitReadAligner.cpp:24-75) as an (L+1, R+1) int32 array [j, i] (port only)."""
    ref, read = bytes(ref), bytes(read)
    H = np.zeros((len(read) + 1, len(ref) + 1), dtype=np.int32)
    a, b = _u8(ref), _u8(read)
    _lib("port").dpo_fill_matrix(_p(a, _c_u8p), len(ref), _p(b, _c_u8p), len(read), match, mismatch, gap,
                                 int(end_gaps), _p(H, _c_i32p))
    return H


def split_backtrace(read, ref1, ref2, ref_split, read_split, match=2, mismatch=-1, gap=-2, end_gaps=False):
    """matches1, matches2 of the alignment with this refSplit / readSplit.first -- GetAlignments(backtrace=True),
    tools/SplitReadAligner.cpp:124-154,287-292 (port).  Two (n,2) int32 arrays of (refPos, readPos)."""
    read, ref1, ref2 = bytes(read), bytes(ref1), bytes(ref2)
    L = len(read)
    m1 = np.zeros((L + 1, 2), dtype=np.int32)
    m2 = np.zeros((L + 1, 2), dtype=np.int32)
    n1 = np.zeros(1, dtype=np.int32)
    n2 = np.zeros(1, dtype=np.int32)
    a, b, c = _u8(read), _u8(ref1), _u8(ref2)
    _lib("port").dpo_split_backtrace(_p(a, _c_u8p), L, _p(b, _c_u8p), len(ref1), _p(c, _c_u8p), len(ref2),
                                     match, mismatch, gap, int(end_gaps), int(ref_split[0]), int(ref_split[1]),
                                     int(read_split), _p(m1, _c_i32p), _p(n1, _c_i32p), _p(m2, _c_i32p), _p(n2, _c_i32p))
    return m1[:n1[0]].copy(), m2[:n2[0]].copy()


def ref_split_backtrace(read, ref1, ref2, min_score, which, match=2, mismatch=-1, gap=-2, end_gaps=False,
                        min_split_score=8):
    """The compiled reference's GetAlignments(backtrace=True): alignment number `which` in emission order.
    Returns (n_alignments, header[7], matches1, matches2) or (n_alignments, None, None, None)."""
    read, ref1, ref2 = bytes(read), bytes(ref1), bytes(ref2)
    L = len(read)
    hdr = np.zeros(7, dtype=np.int32)
    m1 = np.zeros((L + 1, 2), dtype=np.int32)
    m2 = np.zeros((L + 1, 2), dtype=np.int32)
    n1 = np.zeros(1, dtype=np.int32)
    n2 = np.zeros(1, dtype=np.int32)
    n = _lib("ref").ref_split_backtrace(match, mismatch, gap, int(end_gaps), min_split_score, read, L, ref1, len(ref1),
                                        ref2, len(ref2), min_score, which, _p(hdr, _c_i32p), _p(m1, _c_i32p),
                                        _p(n1, _c_i32p), _p(m2, _c_i32p), _p(n2, _c_i32p))
    if n < 0:
        return 0, None, None, None
    return int(n), hdr, m1[:n1[0]].copy(), m2[:n2[0]].copy()


def split_min_score(read_len, match=2):
    """(int)((float)L * (float)match * 0.90) -- tools/SplitAlignment.cpp:379."""
    return int(_lib("port").dpo_split_min_score(read_len, match))


def split_dedupe(alignments):
    """tools/SplitAlignment.cpp:381-400: first alignment per refSplit, score=min(score1,score2).
    (n,7) -> (k,5) {refSplit.first, refSplit.second, readSplit.first, readSplit.second, score}."""
    a = np.ascontiguousarray(alignments, dtype=np.int32).reshape(-1, 7)
    out = np.zeros((max(len(a), 1), 5), dtype=np.int32)
    n = _lib("port").dpo_split_dedupe(_p(a, _c_i32p), len(a), _p(out, _c_i32p))
    return out[:n].copy()


def reverse_complement(seq, impl="port"):
    """tools/Common.cpp:32-54."""
    seq = bytes(seq)
    if impl == "ref":
        buf = ctypes.create_string_buffer(seq, len(seq))
        _lib("ref").ref_reverse_complement(buf, len(seq))
        return buf.raw[:len(seq)]
    a = _u8(seq).copy()
    _lib("port").dpo_reverse_complement(_p(a, _c_u8p), len(seq))
    return a.tobytes()


# --------------------------------------------------------------------------------------
# batch interface (CSR byte tables, same layout as include/defuse_b200.h)
# --------------------------------------------------------------------------------------

def simple_align_batch(match, mismatch, gap, ref_bytes, ref_off, seq_bytes, seq_off, task_ref, task_seq, impl="port"):
    lib = _lib(impl)
    fn = lib.ref_simple_align_batch if impl == "ref" else lib.dpo_simple_align_batch
    rb, sb = _u8(ref_bytes), _u8(seq_bytes)
    ro = np.ascontiguousarray(ref_off, dtype=np.int64)
    so = np.ascontiguousarray(seq_off, dtype=np.int64)
    tr = np.ascontiguousarray(task_ref, dtype=np.int32)
    ts = np.ascontiguousarray(task_seq, dtype=np.int32)
    out = np.zeros(len(tr), dtype=np.int32)
    fn(match, mismatch, gap, _p(rb, _c_u8p), _p(ro, _c_i64p), _p(sb, _c_u8p), _p(so, _c_i64p),
       _p(tr, _c_i32p), _p(ts, _c_i32p), len(tr), _p(out, _c_i32p))
    return out


def split_align_batch(ref_bytes, ref_off, read_bytes, read_off, task_cluster, task_read, task_min_score,
                      match=2, mismatch=-1, gap=-2, end_gaps=False, min_split_score=8, impl="port", cap=None):
    """Returns (count[n_tasks], alignments[(total,7)]) in task order."""
    lib = _lib(impl)
    fn = lib.ref_split_align_batch if impl == "ref" else lib.dpo_split_align_batch
    rb, sb = _u8(ref_bytes), _u8(read_bytes)
    ro = np.ascontiguousarray(ref_off, dtype=np.int64)
    so = np.ascontiguousarray(read_off, dtype=np.int64)
    tc = np.ascontiguousarray(task_cluster, dtype=np.int32)
    tr = np.ascontiguousarray(task_read, dtype=np.int32)
    tm = np.ascontiguousarray(task_min_score, dtype=np.int32)
    n = len(tc)
    if cap is None:
        cap = max(16 * n, 1024)
    while True:
        cnt = np.zeros(n, dtype=np.int32)
        out = np.zeros((cap, 7), dtype=np.int32)
        total = fn(match, mismatch, gap, int(end_gaps), min_split_score,
                   _p(rb, _c_u8p), _p(ro, _c_i64p), _p(sb, _c_u8p), _p(so, _c_i64p),
                   _p(tc, _c_i32p), _p(tr, _c_i32p), _p(tm, _c_i32p), n, _p(cnt, _c_i32p), _p(out, _c_i32p), cap)
        if total <= cap:
            return cnt, out[:total].copy()
        cap = int(total)


def split_backtrace_batch(refs, reads, task_cluster, task_read, ref_split1, ref_split2, read_split, params=(2, -1, -2, False),
                          threads=None):
    """split_backtrace for every alignment of a batch, in the layout of dfb_split_backtrace_batch (port).  refs / reads
    are CSR tables (`.data` bytes, `.off` n+1 offsets; cluster c owns windows 2c and 2c+1); alignment t is
    reads[task_read[t]] against cluster task_cluster[t] with refSplit (ref_split1[t], ref_split2[t]) and readSplit.first
    read_split[t]; params starts with (match, mismatch, gap, end_gaps).  Returns (match_off[2n+1] int64, pairs[(total,2)]
    int32).  The alignments are spread over threads (ctypes releases the GIL)."""
    m, x, g, eg = params[:4]
    lib = _lib("port")
    rb, sb = _u8(refs.data), _u8(reads.data)
    ro = np.ascontiguousarray(refs.off, dtype=np.int64)
    so = np.ascontiguousarray(reads.off, dtype=np.int64)
    arrs = [np.ascontiguousarray(a, dtype=np.int32) for a in (task_cluster, task_read, ref_split1, ref_split2, read_split)]
    n = len(arrs[0])
    assert all(len(a) == n for a in arrs)
    off = np.zeros(2 * n + 1, dtype=np.int64)
    threads = threads or min(32, os.cpu_count() or 1)
    bounds = np.linspace(0, n, min(threads, max(n, 1)) + 1).astype(np.int64)
    lengths = (so[1:] - so[:-1])[arrs[1]] if n else np.zeros(0, np.int64)

    def run(k):
        t0, t1 = int(bounds[k]), int(bounds[k + 1])
        pairs = np.zeros((max(int(lengths[t0:t1].sum()), 1), 2), dtype=np.int32)
        got = lib.dpo_split_backtrace_batch(m, x, g, int(eg), _p(rb, _c_u8p), _p(ro, _c_i64p), _p(sb, _c_u8p), _p(so, _c_i64p),
                                            *[_p(a, _c_i32p) for a in arrs], t0, t1, _p(off, _c_i64p), _p(pairs, _c_i32p))
        return pairs[:got]

    with ThreadPoolExecutor(len(bounds) - 1) as ex:
        parts = list(ex.map(run, range(len(bounds) - 1)))
    base = 0
    for k, part in enumerate(parts):   # ranges count from their own start
        off[2 * bounds[k] + 1:2 * bounds[k + 1] + 1] += base
        base += len(part)
    return off, np.concatenate(parts)
