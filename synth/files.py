"""Synthetic input FILES for the three tools (formats of SURVEY.md appendix B): a small genome with
multi-exon genes on both strands, its cDNA, fusion clusters, read pairs, improper-pair SAM.
Seeded; meant for differential tests (our tool vs the compiled reference on the same files), so the
geometry only has to produce plenty of overlaps and alignments, not be biologically exact."""
import os

import numpy as np

ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
_COMP = bytes.maketrans(b"ACGTacgt", b"TGCAtgca")


def revcomp(s):
    return s.translate(_COMP)[::-1]


def rand_seq(rng, n):
    return ACGT[rng.integers(0, 4, n)].tobytes()


def mutate(rng, s, sub=0.01, n_rate=0.002, lower=0.0):
    a = np.frombuffer(s, dtype=np.uint8).copy()
    m = rng.random(a.size) < sub
    a[m] = ACGT[rng.integers(0, 4, int(m.sum()))]
    m = rng.random(a.size) < n_rate
    a[m] = ord("N")
    if lower:
        m = rng.random(a.size) < lower
        a[m] = np.frombuffer(bytes(a[m]).lower(), dtype=np.uint8)
    return a.tobytes()


def write_fasta(path, entries, width=60):
    with open(path, "wb") as f:
        for name, seq in entries:
            f.write(b">" + name.encode() + b"\n")
            for k in range(0, len(seq), width):
                f.write(seq[k:k + width] + b"\n")


def make_genome(rng, n_chrom=3, genes_per_chrom=6, lower_frac=0.0):
    """chromosomes, genes (1-3 exons, either strand), cDNA sequences named gene|transcript."""
    chroms, genes = [], []
    for c in range(n_chrom):
        pos = 500
        exon_lists = []
        for g in range(genes_per_chrom):
            n_ex = int(rng.integers(1, 4))
            exons = []
            for _ in range(n_ex):
                ln = int(rng.integers(300, 900))
                exons.append((pos, pos + ln - 1))
                pos += ln + int(rng.integers(100, 400))
            pos += int(rng.integers(500, 1500))
            exon_lists.append(exons)
        seq = rand_seq(rng, pos + 500)
        if lower_frac:
            seq = mutate(rng, seq, 0.0, 0.0, lower_frac)
        name = "chr%d" % (c + 1)
        chroms.append((name, seq))
        for g, exons in enumerate(exon_lists):
            strand = "+" if rng.random() < 0.5 else "-"
            gene, tr = "G%d_%d" % (c + 1, g), "T%d_%d" % (c + 1, g)
            cdna = b"".join(seq[s - 1:e] for s, e in exons)
            if strand == "-":
                cdna = revcomp(cdna)
            genes.append(dict(gene=gene, transcript=tr, chrom=name, strand=strand, exons=exons, cdna=cdna,
                              id="%s|%s" % (gene, tr)))
    return chroms, genes


def make_split_dataset(outdir, seed=1, n_clusters=40, pairs_per_cluster=30, L=100, n_chrom=3, genes_per_chrom=6,
                       frag_mean=250, lower_frac=0.0, n_rate=0.002, read_len_jitter=0):
    """Files for dosplitalign: reference.fa, exons.regions, clusters.regions, reads.{1,2}.fastq, improper.sam.
    Returns the argument list (without the program name and the -a output)."""
    rng = np.random.default_rng(seed)
    os.makedirs(outdir, exist_ok=True)
    chroms, genes = make_genome(rng, n_chrom, genes_per_chrom, lower_frac)
    write_fasta(os.path.join(outdir, "reference.fa"), chroms + [(g["id"], g["cdna"]) for g in genes])
    with open(os.path.join(outdir, "exons.regions"), "w") as f:
        for g in genes:
            f.write("\t".join([g["gene"], g["transcript"], g["chrom"], g["strand"]] +
                              [str(v) for e in g["exons"] for v in e]) + "\n")
    refs = dict(chroms)
    refs.update({g["id"]: g["cdna"] for g in genes})

    regions, sam, fq1, fq2 = [], [], [], []
    frag = 0
    for c in range(n_clusters):
        ga, gb = rng.choice(len(genes), 2, replace=False)
        ends = []
        for end, gi in enumerate((ga, gb)):
            g = genes[gi]
            on_transcript = rng.random() < 0.7
            name = g["id"] if on_transcript else g["chrom"]
            seq = refs[name]
            if on_transcript:
                lo, hi = 1, len(seq)
            else:
                lo, hi = g["exons"][0][0], g["exons"][-1][1]
            span = int(rng.integers(60, 200))
            start = int(rng.integers(lo, max(lo + 1, hi - span)))
            strand = "+" if rng.random() < 0.5 else "-"
            ends.append(dict(name=name, seq=seq, start=start, end=min(len(seq), start + span), strand=strand))
            regions.append("%d\t%d\t%s\t%s\t%d\t%d" % (c, end, name, strand, start, ends[-1]["end"]))
        for p in range(pairs_per_cluster):
            Lr = L + (int(rng.integers(-read_len_jitter, read_len_jitter + 1)) if read_len_jitter else 0)
            # the anchored end: somewhere around one of the two cluster regions, on either strand
            e = ends[int(rng.integers(0, 2))]
            off = int(rng.integers(-400, 400))
            apos = max(1, min(len(e["seq"]) - 50, (e["start"] if rng.random() < 0.5 else e["end"]) + off))
            aseq = e["seq"][apos - 1:apos - 1 + 50]
            flag = 0 if rng.random() < 0.5 else 16
            # the candidate end: a chimera of sequence near both regions (either orientation), or plain sequence
            a, b = ends[0], ends[1]
            pa = max(0, min(len(a["seq"]) - Lr, a["end"] - int(rng.integers(0, 2 * Lr))))
            pb = max(0, min(len(b["seq"]) - Lr, b["start"] - int(rng.integers(0, Lr))))
            sa, sb = a["seq"][pa:pa + Lr], b["seq"][pb:pb + Lr]
            if rng.random() < 0.5:
                sa = revcomp(sa)
            if rng.random() < 0.5:
                sb = revcomp(sb)
            kind = rng.random()
            if kind < 0.6:
                cut = int(rng.integers(10, Lr - 10))
                cand = sa[:cut] + sb[len(sb) - (Lr - cut):]
            elif kind < 0.8:
                cand = sa
            elif kind < 0.95:
                cand = sb
            else:
                cand = rand_seq(rng, Lr)
            cand = mutate(rng, cand[:Lr], 0.01, n_rate)
            anchor_end = 1 if rng.random() < 0.5 else 2
            r1, r2 = (aseq + rand_seq(rng, Lr - 50), cand) if anchor_end == 1 else (cand, aseq + rand_seq(rng, Lr - 50))
            fq1.append("@%d/1\n%s\n+\n%s\n" % (frag, r1.decode(), "I" * len(r1)))
            fq2.append("@%d/2\n%s\n+\n%s\n" % (frag, r2.decode(), "I" * len(r2)))
            sam.append("%d/%d\t%d\t%s\t%d\t255\t50M\t*\t0\t0\t%s\t%s" % (frag, anchor_end, flag, e["name"], apos, aseq.decode(), "I" * 50))
            if rng.random() < 0.05:  # unmapped records are skipped by the tools
                sam.append("%d/%d\t4\t*\t0\t0\t*\t*\t0\t0\t%s\t%s" % (frag, 3 - anchor_end, cand.decode(), "I" * len(cand)))
            frag += 1
    with open(os.path.join(outdir, "clusters.regions"), "w") as f:
        f.write("\n".join(regions) + "\n")
    with open(os.path.join(outdir, "improper.sam"), "w") as f:
        f.write("@HD\tVN:1.0\n" + "\n".join(sam) + "\n")
    open(os.path.join(outdir, "reads.1.fastq"), "w").write("".join(fq1))
    open(os.path.join(outdir, "reads.2.fastq"), "w").write("".join(fq2))
    return ["-f", os.path.join(outdir, "reference.fa"), "-e", os.path.join(outdir, "exons.regions"), "-u", str(frag_mean),
            "-s", "30", "-n", str(L - read_len_jitter), "-x", str(L + read_len_jitter), "-r", os.path.join(outdir, "clusters.regions"),
            "-i", os.path.join(outdir, "improper.sam"), "-1", os.path.join(outdir, "reads.1.fastq"),
            "-2", os.path.join(outdir, "reads.2.fastq")]


def cut_splits(outdir, n_splits):
    """Cut the reads of a make_split_dataset directory into n_splits fastq splits, as split_fastq.pl does with real
    reads: fragment f goes to split f % n_splits, file order is kept, every split's SAM starts with the header.  Writes
    split.K.1.fastq, split.K.2.fastq and split.K.improper.sam (K = 0 .. n_splits-1) and returns, per split, the list
    [seq1, seq2, improper sam].  Every split sees every cluster."""
    def fragment(name):  # "@12/1" (fastq) or "12/1" (SAM qname)
        return int(name.lstrip(b"@").split(b"/", 1)[0])

    fq = []
    for end in (1, 2):
        lines = open(os.path.join(outdir, "reads.%d.fastq" % end), "rb").read().splitlines(keepends=True)
        parts = [[] for _ in range(n_splits)]
        for k in range(0, len(lines), 4):
            parts[fragment(lines[k]) % n_splits] += lines[k:k + 4]
        fq.append(parts)
    header, sam = [], [[] for _ in range(n_splits)]
    for line in open(os.path.join(outdir, "improper.sam"), "rb").read().splitlines(keepends=True):
        if line.startswith(b"@"):
            header.append(line)
        else:
            sam[fragment(line.split(b"\t", 1)[0]) % n_splits].append(line)
    out = []
    for k in range(n_splits):
        paths = [os.path.join(outdir, "split.%d.%s" % (k, name)) for name in ("1.fastq", "2.fastq", "improper.sam")]
        for path, data in zip(paths, (fq[0][k], fq[1][k], header + sam[k])):
            with open(path, "wb") as f:
                f.write(b"".join(data))
        out.append(paths)
    return out


def write_read_index(outdir):
    """<outdir>/reads.fqi for reads.{1,2}.fastq: little-endian int64 offsets of the '@' lines, entry 2*fragment+end
    (tools/ReadIndex.cpp:67-77; writer scripts/index_paired_fastq.pl:56-60).  Returns the reads prefix."""
    offs = {}
    n = 0
    for end in (0, 1):
        pos = 0
        with open(os.path.join(outdir, "reads.%d.fastq" % (end + 1)), "rb") as f:
            for k, line in enumerate(f):
                if k % 4 == 0:
                    frag = int(line[1:line.index(b"/")])
                    offs[(frag, end)] = pos
                    n = max(n, frag + 1)
                pos += len(line)
    idx = np.zeros(2 * n, dtype="<i8")
    for (frag, end), pos in offs.items():
        idx[2 * frag + end] = pos
    idx.tofile(os.path.join(outdir, "reads.fqi"))
    return os.path.join(outdir, "reads")


def sort_alignments(src, dst):
    """What the pipeline does between dosplitalign and evalsplitalign (scripts/defuse_run.pl:528, `sort -n -k 1`):
    records grouped by fusion id; ties ordered bytewise so that the result does not depend on the locale."""
    lines = open(src, "rb").read().splitlines(keepends=True)
    lines.sort(key=lambda l: (int(l.split(b"\t", 1)[0]), l))
    open(dst, "wb").write(b"".join(lines))


def downstream_args(split_args, outdir):
    """Argument lists of evalsplitalign / splitseq from a make_split_dataset argument list."""
    common, k = [], 0
    while k < len(split_args):
        if split_args[k] not in ("-i", "-1", "-2"):
            common += split_args[k:k + 2]
        k += 2
    ev = common + ["-a", os.path.join(outdir, "sorted.alignments")]
    return common, ev


def make_localalign_input(seed=2, n_refs=20, n_lines=400, R=2001, L=(60, 140)):
    """stdin of localalign: id \\t reference \\t sequence."""
    rng = np.random.default_rng(seed)
    refs = [rand_seq(rng, R) for _ in range(n_refs)]
    lines = []
    for k in range(n_lines):
        r = refs[int(rng.integers(0, n_refs))]
        ln = int(rng.integers(L[0], L[1] + 1))
        if rng.random() < 0.8:
            s = int(rng.integers(0, R - ln))
            seq = mutate(rng, r[s:s + ln], 0.03, 0.003)
        else:
            seq = rand_seq(rng, ln)
        lines.append(b"c%d\t%s\t%s" % (k, r, seq))
    return b"\n".join(lines) + b"\n"


def make_matealign_dataset(outdir, seed=4, n_pairs=300, L=150, search=1000):
    """Files for matealign: transcripts.fa, reads.{1,2}.fastq and the SAM for stdin.  Returns (args, sam_bytes)."""
    rng = np.random.default_rng(seed)
    os.makedirs(outdir, exist_ok=True)
    trs = [("tr%d some description" % k, rand_seq(rng, int(rng.integers(600, 3000)))) for k in range(12)]
    write_fasta(os.path.join(outdir, "transcripts.fa"), trs)
    sam, fq1, fq2 = ["@SQ\tSN:x\tLN:1"], [], []
    for frag in range(n_pairs):
        name, seq = trs[int(rng.integers(0, len(trs)))]
        strand = 0 if rng.random() < 0.5 else 16
        pos = int(rng.integers(1, max(2, len(seq) - L)))
        aligned = seq[pos - 1:pos - 1 + L]
        # the mate lies downstream on the mate strand for most pairs
        if rng.random() < 0.7:
            if strand == 0:
                mpos = min(len(seq) - L, pos + int(rng.integers(0, search - L)))
                mate = revcomp(seq[max(0, mpos):max(0, mpos) + L])
            else:
                mpos = max(0, pos + L - 1 - int(rng.integers(L, search)))
                mate = seq[mpos:mpos + L]
        else:
            mate = rand_seq(rng, L)
        mate = mutate(rng, mate.ljust(L, b"A")[:L], 0.02, 0.002)
        end = 1 if rng.random() < 0.5 else 2
        r1, r2 = (aligned, mate) if end == 1 else (mate, aligned)
        fq1.append("@%d/1\n%s\n+\n%s\n" % (frag, r1.decode(), "I" * len(r1)))
        fq2.append("@%d/2\n%s\n+\n%s\n" % (frag, r2.decode(), "I" * len(r2)))
        n_hits = 1 if rng.random() < 0.8 else 2
        for _ in range(n_hits):
            sam.append("%d/%d\t%d\t%s\t%d\t255\t%dM\t*\t0\t0\t%s\t*" % (frag, end, strand, name, pos, L, aligned.decode()))
            pos = int(rng.integers(1, max(2, len(seq) - L)))
    open(os.path.join(outdir, "reads.1.fastq"), "w").write("".join(fq1))
    open(os.path.join(outdir, "reads.2.fastq"), "w").write("".join(fq2))
    args = ["-m", "10", "-x", "-5", "-g", "-5", "-t", "0.5", "-s", str(search), "-r", os.path.join(outdir, "transcripts.fa"),
            "-1", os.path.join(outdir, "reads.1.fastq"), "-2", os.path.join(outdir, "reads.2.fastq")]
    return args, ("\n".join(sam) + "\n").encode()
