"""Seeded synthetic tasks shared by the parity tests (no reference code involved), and the stored digests of the
reference's outputs."""
import hashlib
import json
import os

import numpy as np

REFERENCE_DIGESTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_digests.json")

ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


def rand_seq(rng, n, alphabet=ACGT):
    if n == 0:
        return b""
    return alphabet[rng.integers(0, len(alphabet), n)].tobytes()


def mutate(rng, seq, sub=0.02, indel=0.005, n_rate=0.0):
    out = bytearray()
    for c in seq:
        r = rng.random()
        if r < indel / 2:
            continue  # deletion
        if r < indel:
            out.append(int(ACGT[rng.integers(0, 4)]))  # insertion before
        if rng.random() < sub:
            c = int(ACGT[rng.integers(0, 4)])
        if n_rate and rng.random() < n_rate:
            c = ord("N")
        out.append(c)
    return bytes(out)


def planted_split_cluster(rng, R1, R2):
    """Two windows and a function that draws reads spanning (or not) the planted junction."""
    ref1 = rand_seq(rng, R1)
    ref2 = rand_seq(rng, R2)
    bp1 = int(rng.integers(R1 // 3, R1 - 5)) if R1 > 20 else R1
    bp2 = int(rng.integers(5, 2 * R2 // 3)) if R2 > 20 else 0
    fusion = ref1[:bp1] + ref2[bp2:]

    def draw(L, kind):
        if kind == "span" and len(fusion) > L:
            lo = max(0, bp1 - L + 4)
            hi = min(bp1 - 4, len(fusion) - L)
            if hi < lo:
                lo, hi = 0, max(0, len(fusion) - L)
            s = int(rng.integers(lo, hi + 1))
            return fusion[s:s + L]
        if kind == "left" and R1 >= L:
            s = int(rng.integers(0, R1 - L + 1))
            return ref1[s:s + L]
        if kind == "right" and R2 >= L:
            s = int(rng.integers(0, R2 - L + 1))
            return ref2[s:s + L]
        return rand_seq(rng, L)

    return ref1, ref2, draw


def split_batch(rng, n_clusters, reads_per_cluster, L, R_lo, R_hi, sub=0.01, indel=0.002, n_rate=0.002,
                kinds=("span", "span", "left", "right", "random")):
    refs, reads, task_cluster, task_read = [], [], [], []
    for c in range(n_clusters):
        R1 = int(rng.integers(R_lo, R_hi + 1))
        R2 = int(rng.integers(R_lo, R_hi + 1))
        ref1, ref2, draw = planted_split_cluster(rng, R1, R2)
        refs += [ref1, ref2]
        for _ in range(reads_per_cluster):
            Lr = L if isinstance(L, int) else int(rng.integers(L[0], L[1] + 1))
            read = mutate(rng, draw(Lr, kinds[int(rng.integers(0, len(kinds)))]), sub, indel, n_rate)
            task_cluster.append(c)
            task_read.append(len(reads))
            reads.append(read)
    return refs, reads, np.array(task_cluster, np.int32), np.array(task_read, np.int32)


def simple_batch(rng, n_refs, n_tasks, R, L, related=0.8, sub=0.02, indel=0.002):
    refs = [rand_seq(rng, R if isinstance(R, int) else int(rng.integers(R[0], R[1] + 1))) for _ in range(n_refs)]
    seqs, task_ref, task_seq = [], [], []
    for t in range(n_tasks):
        r = int(rng.integers(0, n_refs))
        Lr = L if isinstance(L, int) else int(rng.integers(L[0], L[1] + 1))
        ref = refs[r]
        if rng.random() < related and len(ref) >= Lr:
            s = int(rng.integers(0, len(ref) - Lr + 1))
            seq = mutate(rng, ref[s:s + Lr], sub, indel)
        else:
            seq = rand_seq(rng, Lr)
        task_ref.append(r)
        task_seq.append(len(seqs))
        seqs.append(seq)
    return refs, seqs, np.array(task_ref, np.int32), np.array(task_seq, np.int32)


def random_parameter_round(rng, rnd):
    """One round of the random-parameter parity loops: (params, refs, reads, task_cluster, task_read, min_score) with
    params = (match, mismatch, gap, endGaps, minSplitScore).  Every third round stays inside the s16x2 kernels'
    parameter range, every fourth one uses sequences long enough for several (G,S) classes."""
    alphabets = [ACGT] + [np.frombuffer(a, np.uint8) for a in (b"ACGTN", b"AC", b"ACGTacgtN", b"A")]
    big = rnd % 4 == 3
    m, x, g = int(rng.integers(-2, 12)), int(rng.integers(-8, 3)), int(rng.integers(-8, 3))
    if rnd % 3 == 0:
        m, x, g = int(rng.integers(1, 12)), int(rng.integers(-8, 1)), int(rng.integers(-8, 1))
    eg, mss = bool(rng.integers(0, 2)) and rnd % 3 != 0, int(rng.integers(-5, 20))
    alpha = alphabets[int(rng.integers(0, len(alphabets)))]
    r_hi, l_hi = (700, 300) if big else (120, 70)
    refs, reads, tc, trd = [], [], [], []
    for c in range(5):
        refs += [rand_seq(rng, int(rng.integers(0, r_hi)), alpha), rand_seq(rng, int(rng.integers(0, r_hi)), alpha)]
        for _k in range(4):
            L = int(rng.integers(0, l_hi))
            joined = refs[-2] + refs[-1]
            if rng.random() < 0.6 and 0 < L <= len(joined):
                s = int(rng.integers(0, len(joined) - L + 1))
                read = mutate(rng, joined[s:s + L], 0.05, 0.02, 0.01)
            else:
                read = rand_seq(rng, L, alpha)
            tc.append(c)
            trd.append(len(reads))
            reads.append(read)
    tc, trd = np.array(tc, np.int32), np.array(trd, np.int32)
    thr = np.array([int(rng.integers(-5, max(1, m) * len(reads[r]) + 2)) for r in trd], np.int32)
    return (m, x, g, eg, mss), refs, reads, tc, trd, thr


def check_random_parameter_round(rng, rnd, oracle, ctx, check_split, check_simple):
    """CUDA path against the oracle on one random_parameter_round; returns the number of tasks compared."""
    import defuse_b200 as d
    params, refs, reads, tc, trd, thr = random_parameter_round(rng, rnd)
    m, x, g, eg, mss = params
    # (one-letter alphabets with free gaps tie everywhere: tasks with more than 20 000 tuples are left to
    # test_split_edge_cases, expanding millions of tuples in Python is not what this loop is for)
    rt, st = d.SeqTable.from_list(refs), d.SeqTable.from_list(reads)
    cnt, _ = oracle.split_align_batch(rt.data, rt.off, st.data, st.off, tc, trd, thr, m, x, g, eg, mss)
    keep = cnt <= 20000
    check_split(oracle, ctx, refs, reads, tc[keep], trd[keep], thr[keep], params)
    tr = rng.integers(0, len(refs), len(reads)).astype(np.int32)
    check_simple(oracle, ctx, refs, reads, tr, trd, m, x, g)
    return int(keep.sum()) + len(trd)


def digest(*parts):
    """SHA-256 over byte strings and arrays (with their dtype and shape), in order."""
    h = hashlib.sha256()
    for p in parts:
        if isinstance(p, (bytes, bytearray)):
            p = np.frombuffer(bytes(p), np.uint8)
        p = np.ascontiguousarray(p)
        h.update(("%s%s" % (p.dtype.str, p.shape)).encode())
        h.update(p.tobytes())
    return h.hexdigest()


def reference_digest(key, compute=None):
    """The stored digest of the unmodified reference's output for case `key` (tests/golden/reference_digests.json).
    Where the compiled reference is built (oracle/_ref), `compute` returns the digest of its output now: it must equal
    the stored one, or replaces it when DFB_RECORD_DIGESTS=1.

    How the file was made: digests of the outputs of the C restatement (oracle/dp_oracle.c) and of the tools
    (defuse_b200/host, over tests/device_double) at commit f0d5442, where oracle/, synth/, defuse_b200/ and this module
    were as in the last runs that compared them byte for byte with the compiled reference, and they agreed."""
    with open(REFERENCE_DIGESTS) as f:
        stored = json.load(f)
    if compute is None:
        return stored[key]
    d = compute()
    if os.environ.get("DFB_RECORD_DIGESTS") == "1":
        stored[key] = d
        with open(REFERENCE_DIGESTS, "w") as f:
            json.dump(dict(sorted(stored.items())), f, indent=0)
    else:
        assert stored.get(key) == d, "%s: the compiled reference's output differs from its stored digest" % key
    return d


def reference_tool_digest(oracle_mod, key, name, run):
    """reference_digest() of what the compiled reference tool `name` gives in case `key`: where oracle/_ref has the tool,
    `run(path)` runs it and returns the byte strings compared (stdout, output files, ...)."""
    path = oracle_mod.ref_tool(name)
    return reference_digest(key, (lambda: digest(*run(path))) if path else None)
