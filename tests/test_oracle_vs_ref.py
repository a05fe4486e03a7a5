"""The C restatement against the unmodified reference.  Every case is checked against the SHA-256 digest of the
reference's output stored in tests/golden/reference_digests.json, so the comparison runs on any machine; where
oracle/_ref/libref_aligners.so is built (oracle/Makefile), the compiled reference runs beside the restatement too.

The restatement is unchanged since these cases last ran against the compiled reference and agreed on every one of them
(commit "Oracle pinning: backtrace match lists under random parameters against the compiled reference"); the digests are
of those outputs.  With the reference built, DFB_RECORD_DIGESTS=1 rewrites them from the reference itself."""
import numpy as np
import pytest

import util


@pytest.fixture(scope="module")
def ref(oracle_mod):
    return oracle_mod


class _Outputs:
    """The restatement's outputs of one test case, in order: each compared with the compiled reference's where that is
    built, all of them together with the stored digest of the reference's outputs."""

    def __init__(self, oracle_mod, key):
        self.oracle, self.key, self.arrays = oracle_mod, key, []

    def agree(self, ours, theirs):
        """`ours`: a tuple of arrays; `theirs`: a callable computing the same with the compiled reference."""
        if self.oracle.have_ref():
            want = theirs()
            assert len(want) == len(ours) and all(np.array_equal(a, b) for a, b in zip(ours, want)), self.key
        self.arrays += ours

    def check(self):
        # (with the reference built, every output was compared one by one above: its digest is the reference's)
        ours = util.digest(*self.arrays)
        want = util.reference_digest(self.key, (lambda: ours) if self.oracle.have_ref() else None)
        assert ours == want, "%s: outputs differ from the reference's" % self.key


def test_simple_random_vs_ref(ref):
    rng = np.random.default_rng(5)
    out = _Outputs(ref, "simple_random")
    for scoring in [(10, -5, -5), (2, -1, -2), (1, -1, 1), (0, 0, 0), (-2, -3, -1), (7, 2, -3)]:
        refs, seqs, tr, ts = util.simple_batch(rng, 8, 60, (0, 200), (0, 120))
        import defuse_b200 as d
        rt, st = d.SeqTable.from_list(refs), d.SeqTable.from_list(seqs)
        a = ref.simple_align_batch(*scoring, rt.data, rt.off, st.data, st.off, tr, ts, impl="port")
        out.agree((a,), lambda: (ref.simple_align_batch(*scoring, rt.data, rt.off, st.data, st.off, tr, ts, impl="ref"),))
    out.check()


@pytest.mark.parametrize("params", [(2, -1, -2, False, 8), (2, -1, -2, True, 8), (2, -1, -2, False, 0), (1, -1, 1, False, 3),
                                    (5, -4, -3, False, -2), (0, 0, 0, False, 0)])
def test_split_random_vs_ref(ref, params):
    import defuse_b200 as d
    rng = np.random.default_rng(6)
    refs, reads, tc, trd = util.split_batch(rng, 10, 6, (0, 90), 0, 200, sub=0.03, indel=0.01, n_rate=0.01)
    rt, st = d.SeqTable.from_list(refs), d.SeqTable.from_list(reads)
    m, x, g, eg, ms = params
    out = _Outputs(ref, "split_random/%d,%d,%d,%d,%d" % params)
    for thr in (np.zeros(len(tc), np.int32), np.array([int(0.9 * m * len(reads[r])) for r in trd], np.int32)):
        ours = ref.split_align_batch(rt.data, rt.off, st.data, st.off, tc, trd, thr, m, x, g, eg, ms, impl="port")
        out.agree(ours, lambda: ref.split_align_batch(rt.data, rt.off, st.data, st.off, tc, trd, thr, m, x, g, eg, ms, impl="ref"))
    out.check()


def test_reverse_complement_vs_ref(ref):
    rng = np.random.default_rng(7)
    out = _Outputs(ref, "reverse_complement")
    for _ in range(50):
        s = bytes(rng.integers(32, 127, int(rng.integers(0, 60))).astype(np.uint8))
        out.agree((np.frombuffer(ref.reverse_complement(s, impl="port"), np.uint8),),
                  lambda: (np.frombuffer(ref.reverse_complement(s, impl="ref"), np.uint8),))
    out.check()


def _backtrace(ref, out, read, ref1, ref2, thr, which, m, x, g, eg, mss):
    """Alignment number `which` of GetAlignments(backtrace=True) and its match lists, restatement against reference.
    Returns the number of alignments."""
    n, hdr = ref.split_alignment(read, ref1, ref2, thr, which, m, x, g, eg, mss)
    ours = (np.array([n], np.int64),)
    if hdr is not None:
        ours += (hdr,) + ref.split_backtrace(read, ref1, ref2, (hdr[0], hdr[1]), hdr[2], m, x, g, eg)

    def theirs():
        rn, rhdr, m1, m2 = ref.ref_split_backtrace(read, ref1, ref2, thr, which, m, x, g, eg, mss)
        return (np.array([rn], np.int64),) + ((rhdr, m1, m2) if which < rn else ())

    out.agree(ours, theirs)
    return n


@pytest.mark.parametrize("params", [(2, -1, -2, False, 8), (2, -1, -2, True, 8), (1, -1, 1, False, 3), (5, -4, -3, False, -2),
                                    (3, -2, 0, False, 1)])
def test_backtrace_vs_ref(ref, params):
    """GetAlignments(backtrace=True): match lists of every alignment (up to a cap per task), port vs reference."""
    rng = np.random.default_rng(8)
    refs, reads, tc, trd = util.split_batch(rng, 6, 5, (0, 70), 0, 150, sub=0.04, indel=0.02, n_rate=0.01)
    m, x, g, eg, ms = params
    out = _Outputs(ref, "backtrace/%d,%d,%d,%d,%d" % params)
    checked = 0
    for c, r in zip(tc, trd):
        read, ref1, ref2 = reads[r], refs[2 * c], refs[2 * c + 1]
        thr = int(0.6 * m * len(read))
        for which in range(6):
            if which >= _backtrace(ref, out, read, ref1, ref2, thr, which, m, x, g, eg, ms):
                break
            checked += 1
    out.check()
    assert checked > 10


def test_random_parameters_vs_ref(ref):
    """Random scoring triples (positive gaps, negative matches, zeros), endGaps either way, minSplitScore and minScore
    below and above zero, alphabets from one letter to mixed case with N, empty strings: restatement == compiled
    reference for the split tuples and the simple score.  (The same loop ran for 21 000 rounds / 630 000 tasks while the
    oracle was being pinned; 150 rounds stay in the suite.)"""
    import defuse_b200 as d
    rng = np.random.default_rng(9)
    alphabets = [util.ACGT] + [np.frombuffer(a, np.uint8) for a in (b"ACGTN", b"AC", b"ACGTacgtN", b"A")]
    out = _Outputs(ref, "random_parameters")
    for _ in range(150):
        m, x, g = int(rng.integers(-2, 12)), int(rng.integers(-8, 3)), int(rng.integers(-8, 3))
        eg, mss = bool(rng.integers(0, 2)), int(rng.integers(-5, 20))
        alpha = alphabets[int(rng.integers(0, len(alphabets)))]
        refs, reads, tc, trd = [], [], [], []
        for c in range(6):
            refs += [util.rand_seq(rng, int(rng.integers(0, 120)), alpha), util.rand_seq(rng, int(rng.integers(0, 120)), alpha)]
            for _k in range(5):
                L = int(rng.integers(0, 70))
                joined = refs[-2] + refs[-1]
                if rng.random() < 0.6 and 0 < L <= len(joined):
                    s = int(rng.integers(0, len(joined) - L + 1))
                    read = util.mutate(rng, joined[s:s + L], 0.05, 0.02, 0.01)
                else:
                    read = util.rand_seq(rng, L, alpha)
                tc.append(c)
                trd.append(len(reads))
                reads.append(read)
        tc, trd = np.array(tc, np.int32), np.array(trd, np.int32)
        rt, st = d.SeqTable.from_list(refs), d.SeqTable.from_list(reads)
        thr = np.array([int(rng.integers(-5, max(1, m) * len(reads[r]) + 2)) for r in trd], np.int32)
        ours = ref.split_align_batch(rt.data, rt.off, st.data, st.off, tc, trd, thr, m, x, g, eg, mss, impl="port")
        out.agree(ours, lambda: ref.split_align_batch(rt.data, rt.off, st.data, st.off, tc, trd, thr, m, x, g, eg, mss, impl="ref"))
        tr = rng.integers(0, len(refs), len(reads)).astype(np.int32)
        sa = ref.simple_align_batch(m, x, g, rt.data, rt.off, st.data, st.off, tr, trd, impl="port")
        out.agree((sa,), lambda: (ref.simple_align_batch(m, x, g, rt.data, rt.off, st.data, st.off, tr, trd, impl="ref"),))
    out.check()


def test_backtrace_random_parameters_vs_ref(ref):
    """Match lists of GetAlignments(backtrace=True) under random scoring triples / endGaps / thresholds and odd
    alphabets (the generator of test_random_parameters_vs_ref): restatement == compiled reference."""
    rng = np.random.default_rng(10)
    out = _Outputs(ref, "backtrace_random_parameters")
    checked = 0
    for rnd in range(20):
        params, refs, reads, tc, trd, thr = util.random_parameter_round(rng, rnd if rnd % 4 != 3 else rnd + 1)  # short sequences only
        m, x, g, eg, mss = params
        for c, r, th in zip(tc, trd, thr):
            read, ref1, ref2 = reads[r], refs[2 * c], refs[2 * c + 1]
            for which in range(3):
                if which >= _backtrace(ref, out, read, ref1, ref2, int(th), which, m, x, g, eg, mss):
                    break
                checked += 1
    out.check()
    assert checked > 100
