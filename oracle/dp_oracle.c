/*
 * TEST INFRASTRUCTURE ONLY -- the parity oracle.  Never imported, linked or executed by
 * the product path (defuse_b200/), only by tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline leg.
 *
 * Plain-C restatement of the reference's DP alignment hot path (SURVEY.md section 8a).
 * Every function cites the reference file:line it follows.  PARITY IS PINNED: this file
 * is checked cell-for-cell / tuple-for-tuple against the unmodified reference compiled
 * from /root/reference (oracle/_ref/libref_aligners.so, oracle/Makefile) by
 * tests/test_oracle_vs_ref.py, and against the committed golden vectors the reference
 * produced (tests/golden/, generator tests/golden/make_golden.py) by tests/test_oracle_golden.py.
 * The reference itself ships no tests or golden vectors for this path (SURVEY.md section 4).
 *
 * Conventions: `ref` has R bytes, `read` has L bytes; matrix H has (R+1) x (L+1) entries
 * addressed H[j*(R+1)+i] with i over the reference and j over the read, which is the
 * storage order of tools/Matrix.h:63-66.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define DPO_API __attribute__((visibility("default")))

static inline int imax(int a, int b) { return a > b ? a : b; }

/* tools/SplitReadAligner.cpp:24-75 (FillMatrix) and tools/SimpleAligner.cpp:23-63 share this
 * recurrence: H(i,0)=0; H(0,j)=H(0,j-1)+(endGaps?0:gap); otherwise the max of the diagonal
 * (byte equality -> match / mismatch), the cell above in i plus gap, the cell before in j
 * plus gap.  No clamp at zero. */
DPO_API void dpo_fill_matrix(const uint8_t* ref, int R, const uint8_t* read, int L,
                             int match, int mismatch, int gap, int end_gaps, int32_t* H)
{
	const size_t W = (size_t)R + 1;
	for (int i = 0; i <= R; i++)
	{
		H[i] = 0; /* j == 0: matrix(i,0) = 0   (SplitReadAligner.cpp:40-43) */
	}
	for (int j = 1; j <= L; j++)
	{
		/* i == 0: matrix(0,j) = matrix(0,j-1) + (endGaps ? 0 : gap)   (:44-48) */
		H[j * W] = H[(j - 1) * W] + (end_gaps ? 0 : gap);
	}
	for (int i = 1; i <= R; i++)
	{
		const uint8_t a = ref[i - 1];
		for (int j = 1; j <= L; j++)
		{
			int diag = H[(j - 1) * W + (i - 1)] + (a == read[j - 1] ? match : mismatch); /* :51 */
			int gap_ref = H[j * W + (i - 1)] + gap;                                     /* :52 */
			int gap_read = H[(j - 1) * W + i] + gap;                                    /* :53 */
			H[j * W + i] = imax(diag, imax(gap_ref, gap_read));                         /* :54,71 */
		}
	}
}

/* tools/SimpleAligner.cpp:23-63: best interior cell (i>=1, j>=1), floor 0. */
DPO_API int dpo_simple_align(const uint8_t* ref, int R, const uint8_t* seq, int L,
                             int match, int mismatch, int gap)
{
	/* rolling storage over i: col[j] = H(i,j) */
	int32_t* col = (int32_t*)malloc(sizeof(int32_t) * (size_t)(L + 1));
	int best = 0; /* overallMaxScore starts at 0 (:30) */
	col[0] = 0;
	for (int j = 1; j <= L; j++)
	{
		col[j] = col[j - 1] + gap; /* row i == 0 (:44-47); not a candidate for the max */
	}
	for (int i = 1; i <= R; i++)
	{
		const uint8_t a = ref[i - 1];
		int diag_src = col[0]; /* H(i-1, j-1) */
		col[0] = 0;            /* H(i,0) = 0 (:40-43) */
		for (int j = 1; j <= L; j++)
		{
			int up = col[j]; /* H(i-1, j) */
			int v = imax(diag_src + (a == seq[j - 1] ? match : mismatch), imax(up + gap, col[j - 1] + gap));
			best = imax(best, v); /* :55 */
			col[j] = v;
			diag_src = up;
		}
	}
	free(col);
	return best;
}

/* tools/SplitReadAligner.cpp:91-122 (FindMaxRowEntry): over i = 0..R, the largest H(i,j)
 * that is >= min_accepted and > 0, else 0; `cols` (optional) = every i attaining it, ascending;
 * empty when the max stays 0. */
static int row_max(const int32_t* H, int R, int j, int min_accepted, int* cols, int* n_cols)
{
	const int32_t* row = H + (size_t)j * (R + 1);
	int best = 0;
	int n = 0;
	for (int i = 0; i <= R; i++)
	{
		int v = row[i];
		if (v >= min_accepted && v > best)
		{
			best = v;
			n = 0;
			if (cols) cols[n] = i;
			n++;
		}
		else if (v >= min_accepted && v == best)
		{
			if (cols) cols[n] = i;
			n++;
		}
	}
	if (n_cols) *n_cols = n;
	return best;
}

static void reverse_copy(uint8_t* dst, const uint8_t* src, int n)
{
	for (int k = 0; k < n; k++) dst[k] = src[n - 1 - k];
}

/* tools/SplitReadAligner.cpp:77-89 (Align) + :156-298 (GetAlignments with forceSplit=true,
 * firstOnly=false, backTrace=false -- the only combination any caller uses,
 * tools/SplitAlignment.cpp:379).
 * Output: 7 ints per alignment {refSplit.first, refSplit.second, readSplit.first,
 * readSplit.second, score, score1, score2}, in the reference's emission order.
 * Returns the number of alignments (may exceed cap; only `cap` are written).
 * rowmax1/rowmax2 (optional, L+1 ints each) receive FindMaxRowEntry of each matrix row. */
DPO_API int64_t dpo_split_align(const uint8_t* read, int L,
                                const uint8_t* ref1, int R1, const uint8_t* ref2, int R2,
                                int match, int mismatch, int gap, int end_gaps, int min_split_score,
                                int min_score, int32_t* out, int64_t cap,
                                int32_t* rowmax1, int32_t* rowmax2)
{
	uint8_t* ref2r = (uint8_t*)malloc((size_t)R2 + 1);
	uint8_t* readr = (uint8_t*)malloc((size_t)L + 1);
	reverse_copy(ref2r, ref2, R2); /* :80-81 */
	reverse_copy(readr, read, L);  /* :84-85 */
	int32_t* H1 = (int32_t*)malloc(sizeof(int32_t) * (size_t)(R1 + 1) * (size_t)(L + 1));
	int32_t* H2 = (int32_t*)malloc(sizeof(int32_t) * (size_t)(R2 + 1) * (size_t)(L + 1));
	dpo_fill_matrix(ref1, R1, read, L, match, mismatch, gap, end_gaps, H1);   /* :87 */
	dpo_fill_matrix(ref2r, R2, readr, L, match, mismatch, gap, end_gaps, H2); /* :88 */

	/* :194-222 -- best split total over a = alignedToRef1 = 0..L, ties kept ascending */
	int best = 0;
	int* ties = (int*)malloc(sizeof(int) * (size_t)(L + 1));
	int n_ties = 0;
	for (int a = 0; a <= L; a++)
	{
		int b = L - a;
		int m1 = row_max(H1, R1, a, min_split_score, NULL, NULL);
		int m2 = row_max(H2, R2, b, min_split_score, NULL, NULL);
		if (rowmax1) rowmax1[a] = m1;
		if (rowmax2) rowmax2[b] = m2;
		int tot = m1 + m2;
		if (tot >= min_score && tot > best)
		{
			best = tot;
			n_ties = 0;
			ties[n_ties++] = a;
		}
		else if (tot >= min_score && tot == best)
		{
			ties[n_ties++] = a;
		}
	}

	int64_t n_out = 0;
	if (best != 0) /* :224-227 */
	{
		int* c1 = (int*)malloc(sizeof(int) * (size_t)(R1 + 1));
		int* c2 = (int*)malloc(sizeof(int) * (size_t)(R2 + 1));
		for (int t = 0; t < n_ties; t++) /* :233-269 */
		{
			int a = ties[t];
			int b = L - a;
			int n1 = 0, n2 = 0;
			row_max(H1, R1, a, min_split_score, c1, &n1);
			row_max(H2, R2, b, min_split_score, c2, &n2);
			for (int p = 0; p < n1; p++)
			{
				for (int q = 0; q < n2; q++)
				{
					if (n_out < cap) /* :272-297 */
					{
						int32_t* o = out + 7 * n_out;
						o[0] = c1[p];
						o[1] = R2 - c2[q] - 1;
						o[2] = a;
						o[3] = b;
						o[4] = best;
						o[5] = H1[(size_t)a * (R1 + 1) + c1[p]];
						o[6] = H2[(size_t)b * (R2 + 1) + c2[q]];
					}
					n_out++;
				}
			}
		}
		free(c1);
		free(c2);
	}
	free(ties);
	free(H1);
	free(H2);
	free(ref2r);
	free(readr);
	return n_out;
}

/* tools/SplitAlignment.cpp:379 -- the threshold handed to GetAlignments. */
DPO_API int dpo_split_min_score(int read_len, int match)
{
	return (int)((float)read_len * (float)match * 0.90);
}

/* tools/SplitAlignment.cpp:381-400 -- keep the first alignment of each distinct refSplit,
 * record score = min(score1, score2).  in: 7 ints per alignment; out: 5 ints per record
 * {refSplit.first, refSplit.second, readSplit.first, readSplit.second, score}.
 * Quadratic scan on purpose (small inputs; no hashing to get wrong). */
DPO_API int64_t dpo_split_dedupe(const int32_t* in, int64_t n_in, int32_t* out)
{
	int64_t n_out = 0;
	for (int64_t k = 0; k < n_in; k++)
	{
		const int32_t* a = in + 7 * k;
		int seen = 0;
		for (int64_t r = 0; r < n_out; r++)
		{
			if (out[5 * r] == a[0] && out[5 * r + 1] == a[1])
			{
				seen = 1;
				break;
			}
		}
		if (seen) continue;
		int32_t* o = out + 5 * n_out++;
		o[0] = a[0];
		o[1] = a[1];
		o[2] = a[2];
		o[3] = a[3];
		o[4] = a[5] < a[6] ? a[5] : a[6];
	}
	return n_out;
}

/* tools/Common.cpp:32-54 -- reverse, then complement ACGTacgt only. */
DPO_API void dpo_reverse_complement(uint8_t* seq, int n)
{
	for (int lo = 0, hi = n - 1; lo < hi; lo++, hi--)
	{
		uint8_t t = seq[lo];
		seq[lo] = seq[hi];
		seq[hi] = t;
	}
	for (int k = 0; k < n; k++)
	{
		switch (seq[k])
		{
			case 'A': seq[k] = 'T'; break;
			case 'C': seq[k] = 'G'; break;
			case 'T': seq[k] = 'A'; break;
			case 'G': seq[k] = 'C'; break;
			case 'a': seq[k] = 't'; break;
			case 'c': seq[k] = 'g'; break;
			case 't': seq[k] = 'a'; break;
			case 'g': seq[k] = 'c'; break;
			default: break;
		}
	}
}

/* Batch drivers over CSR byte tables (same table layout as include/defuse_b200.h). */

DPO_API int64_t dpo_simple_align_batch(int match, int mismatch, int gap,
                                       const uint8_t* ref_bytes, const int64_t* ref_off,
                                       const uint8_t* seq_bytes, const int64_t* seq_off,
                                       const int32_t* task_ref, const int32_t* task_seq,
                                       int64_t n_tasks, int32_t* out_score)
{
	for (int64_t t = 0; t < n_tasks; t++)
	{
		int r = task_ref[t], s = task_seq[t];
		out_score[t] = dpo_simple_align(ref_bytes + ref_off[r], (int)(ref_off[r + 1] - ref_off[r]),
		                                seq_bytes + seq_off[s], (int)(seq_off[s + 1] - seq_off[s]),
		                                match, mismatch, gap);
	}
	return n_tasks;
}

/* cluster c owns ref windows 2c (ref1) and 2c+1 (ref2). */
DPO_API int64_t dpo_split_align_batch(int match, int mismatch, int gap, int end_gaps, int min_split_score,
                                      const uint8_t* ref_bytes, const int64_t* ref_off,
                                      const uint8_t* read_bytes, const int64_t* read_off,
                                      const int32_t* task_cluster, const int32_t* task_read,
                                      const int32_t* task_min_score, int64_t n_tasks,
                                      int32_t* out_count, int32_t* out, int64_t cap)
{
	int64_t total = 0;
	for (int64_t t = 0; t < n_tasks; t++)
	{
		int c = task_cluster[t], r = task_read[t];
		int64_t room = cap > total ? cap - total : 0;
		int64_t n = dpo_split_align(read_bytes + read_off[r], (int)(read_off[r + 1] - read_off[r]),
		                            ref_bytes + ref_off[2 * c], (int)(ref_off[2 * c + 1] - ref_off[2 * c]),
		                            ref_bytes + ref_off[2 * c + 1], (int)(ref_off[2 * c + 2] - ref_off[2 * c + 1]),
		                            match, mismatch, gap, end_gaps, min_split_score, task_min_score[t],
		                            out + 7 * (total < cap ? total : cap), room, NULL, NULL);
		out_count[t] = (int32_t)n;
		total += n;
	}
	return total;
}

/* tools/SplitReadAligner.cpp:124-143 (BackTracePath) over the pointers FillMatrix leaves (:56-69):
 * at (i,j) the pointer is (i-1,j-1) when the diagonal attains the cell's score, overwritten by
 * (i-1,j) when that one does, overwritten by (i,j-1) when that one does; row i == 0 points to
 * (0,j-1) (:46-47).  The walk starts at (start_i,start_j), stops at j == 0 and collects
 * (refPos,readPos) = (i-1,j-1) of every diagonal step; the list is reversed at the end (:142).
 * The pointers are recomputed from H here instead of being stored.  Returns the number of pairs. */
static int backtrace_path(const int32_t* H, const uint8_t* ref, int R, const uint8_t* read,
                          int match, int mismatch, int gap, int start_i, int start_j, int32_t* pairs)
{
	const size_t W = (size_t)R + 1;
	int i = start_i, j = start_j, n = 0;
	while (j > 0)
	{
		int dir;
		if (i == 0)
		{
			dir = 2;
		}
		else
		{
			int v = H[j * W + i];
			int diag = H[(j - 1) * W + (i - 1)] + (ref[i - 1] == read[j - 1] ? match : mismatch);
			int gap_ref = H[j * W + (i - 1)] + gap;
			int gap_read = H[(j - 1) * W + i] + gap;
			dir = -1;
			if (diag == v) dir = 0;     /* :56-59 */
			if (gap_ref == v) dir = 1;  /* :61-64 */
			if (gap_read == v) dir = 2; /* :66-69 */
		}
		if (dir == 0)
		{
			pairs[2 * n] = i - 1;
			pairs[2 * n + 1] = j - 1;
			n++;
			i--;
			j--;
		}
		else if (dir == 1)
		{
			i--;
		}
		else
		{
			j--;
		}
	}
	for (int a = 0, b = n - 1; a < b; a++, b--)
	{
		int32_t t0 = pairs[2 * a], t1 = pairs[2 * a + 1];
		pairs[2 * a] = pairs[2 * b];
		pairs[2 * a + 1] = pairs[2 * b + 1];
		pairs[2 * b] = t0;
		pairs[2 * b + 1] = t1;
	}
	return n;
}

/* GetAlignments(..., backTrace=true) for ONE alignment named by its refSplit and readSplit.first
 * (tools/SplitReadAligner.cpp:271-292): start cells (ref_split1, read_split) in matrix 1 and
 * (R2 - ref_split2 - 1, L - read_split) in matrix 2; matches2 goes through ReverseMatches
 * (:145-154: coordinates mapped back to the unreversed sequences, list reversed again).
 * matches1/matches2 hold up to L pairs each; n1/n2 receive the counts. */
DPO_API void dpo_split_backtrace(const uint8_t* read, int L, const uint8_t* ref1, int R1,
                                 const uint8_t* ref2, int R2, int match, int mismatch, int gap,
                                 int end_gaps, int ref_split1, int ref_split2, int read_split,
                                 int32_t* matches1, int32_t* n1, int32_t* matches2, int32_t* n2)
{
	uint8_t* ref2r = (uint8_t*)malloc((size_t)R2 + 1);
	uint8_t* readr = (uint8_t*)malloc((size_t)L + 1);
	reverse_copy(ref2r, ref2, R2);
	reverse_copy(readr, read, L);
	int32_t* H1 = (int32_t*)malloc(sizeof(int32_t) * (size_t)(R1 + 1) * (size_t)(L + 1));
	int32_t* H2 = (int32_t*)malloc(sizeof(int32_t) * (size_t)(R2 + 1) * (size_t)(L + 1));
	dpo_fill_matrix(ref1, R1, read, L, match, mismatch, gap, end_gaps, H1);
	dpo_fill_matrix(ref2r, R2, readr, L, match, mismatch, gap, end_gaps, H2);
	*n1 = backtrace_path(H1, ref1, R1, read, match, mismatch, gap, ref_split1, read_split, matches1);
	int m = backtrace_path(H2, ref2r, R2, readr, match, mismatch, gap, R2 - ref_split2 - 1, L - read_split, matches2);
	for (int k = 0; k < m; k++) /* :147-151 */
	{
		matches2[2 * k] = R2 - matches2[2 * k] - 1;
		matches2[2 * k + 1] = L - matches2[2 * k + 1] - 1;
	}
	for (int a = 0, b = m - 1; a < b; a++, b--) /* :153 */
	{
		int32_t t0 = matches2[2 * a], t1 = matches2[2 * a + 1];
		matches2[2 * a] = matches2[2 * b];
		matches2[2 * a + 1] = matches2[2 * b + 1];
		matches2[2 * b] = t0;
		matches2[2 * b + 1] = t1;
	}
	*n2 = m;
	free(H1);
	free(H2);
	free(ref2r);
	free(readr);
}

/* dpo_split_backtrace over alignments [t0, t1) of a batch, in the layout of dfb_split_backtrace_batch: alignment t
 * of reads[task_read[t]] against cluster task_cluster[t] (windows 2c and 2c+1).  match_off[2t+1] and match_off[2t+2]
 * receive the ends of its matches1 and matches2, counted from pairs of the range, which holds 2 * sum(len(read)) ints;
 * match_off[2 * t0] is left to the caller.  Returns the number of pairs written. */
DPO_API int64_t dpo_split_backtrace_batch(int match, int mismatch, int gap, int end_gaps,
                                          const uint8_t* ref_bytes, const int64_t* ref_off,
                                          const uint8_t* read_bytes, const int64_t* read_off,
                                          const int32_t* task_cluster, const int32_t* task_read,
                                          const int32_t* ref_split1, const int32_t* ref_split2,
                                          const int32_t* read_split, int64_t t0, int64_t t1,
                                          int64_t* match_off, int32_t* pairs)
{
	int64_t total = 0;
	for (int64_t t = t0; t < t1; t++)
	{
		int c = task_cluster[t], r = task_read[t];
		int L = (int)(read_off[r + 1] - read_off[r]);
		int32_t* m2 = (int32_t*)malloc(sizeof(int32_t) * 2 * ((size_t)L + 1));
		int32_t n1 = 0, n2 = 0;
		dpo_split_backtrace(read_bytes + read_off[r], L, ref_bytes + ref_off[2 * c], (int)(ref_off[2 * c + 1] - ref_off[2 * c]),
		                    ref_bytes + ref_off[2 * c + 1], (int)(ref_off[2 * c + 2] - ref_off[2 * c + 1]), match, mismatch,
		                    gap, end_gaps, ref_split1[t], ref_split2[t], read_split[t], pairs + 2 * total, &n1, m2, &n2);
		memcpy(pairs + 2 * (total + n1), m2, sizeof(int32_t) * 2 * (size_t)n2);
		free(m2);
		match_off[2 * t + 1] = total + n1;
		match_off[2 * t + 2] = total + n1 + n2;
		total += n1 + n2;
	}
	return total;
}
