/*
 * defuse_b200.h -- C ABI of the B200-native (sm_100a) replacement for deFuse's
 * dynamic-programming alignment hot path.
 *
 * The reference (amcpherson/defuse) has no plugin/FFI seam for this path; the seam is two
 * C++ classes that its tools call one task at a time:
 *
 *   SimpleAligner(int match, int mismatch, int gap)                 tools/SimpleAligner.h:20
 *   int  SimpleAligner::Align(const string& reference,
 *                             const string& sequence)                tools/SimpleAligner.h:22
 *        callers: tools/localalign.cpp:79, tools/matealign.cpp:209
 *
 *   SplitReadAligner(int match, int mismatch, int gap,
 *                    bool endGaps, int minSplitScore)                tools/SplitReadAligner.h:35
 *   void SplitReadAligner::Align(read, reference1, reference2)       tools/SplitReadAligner.h:37
 *   void SplitReadAligner::GetAlignments(SplitReadAlignVec&, int minScore,
 *        bool forceSplits, bool firstOnly, bool backtrace)           tools/SplitReadAligner.h:38
 *        caller: tools/SplitAlignment.cpp:376-379 (forceSplits=true, firstOnly=false)
 *
 * This header is the batch form of those entry points: many (reference, sequence) tasks per
 * call, plain pointers and sizes, no C++ or torch types.  Host buffers are owned by the
 * caller and only read during the call; device memory, streams and staging buffers are
 * owned by the library inside dfb_ctx / dfb_plan.  Every function returns an int status
 * (DFB_OK == 0); nothing throws or exits.  There is no CPU fallback: without a usable
 * sm_100 GPU dfb_ctx_create fails.  A ctx is not re-entrant (one host thread at a time).
 *
 * Results are bit-exact with the reference classes for every byte value (equality is on
 * raw bytes: case-sensitive, 'N' == 'N'), every scoring triple and every length; see
 * DESIGN.md for which kernel variant serves which parameter range.
 */
#ifndef DEFUSE_B200_H_
#define DEFUSE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DFB_ABI_VERSION 1

/* every entry point below is exported; everything else in the library is hidden */
#if defined(__GNUC__)
#define DFB_API __attribute__((visibility("default")))
#else
#define DFB_API
#endif

enum dfb_status
{
	DFB_OK = 0,
	DFB_ERR_CUDA = 1,     /* a CUDA runtime call or kernel failed; see dfb_last_error */
	DFB_ERR_ARG = 2,      /* invalid argument (null pointer, index out of range, ...) */
	DFB_ERR_NOMEM = 3,    /* host or device allocation failed */
	DFB_ERR_NODEVICE = 4, /* no usable sm_100 device (there is no CPU fallback) */
	DFB_ERR_STATE = 5     /* call made in the wrong order (e.g. fetch before run) */
};

typedef struct dfb_ctx dfb_ctx;   /* one per GPU; owns the stream and scratch buffers */
typedef struct dfb_plan dfb_plan; /* one batch resident in HBM: packed sequences + jobs + outputs */

/* A table of byte strings in CSR form: string k is bytes[off[k] .. off[k+1]), k in [0, n).
 * This is the batch equivalent of the `const string&` arguments of the reference classes. */
typedef struct dfb_seq_table
{
	const uint8_t* bytes;
	const int64_t* off; /* n + 1 entries, off[0] == 0, non-decreasing */
	int64_t n;
} dfb_seq_table;

/* SimpleAligner constructor arguments (tools/SimpleAligner.cpp:18-21). */
typedef struct dfb_simple_params
{
	int32_t match;
	int32_t mismatch;
	int32_t gap;
} dfb_simple_params;

/* SplitReadAligner constructor arguments (tools/SplitReadAligner.cpp:19-22).
 * dosplitalign uses {2, -1, -2, 0, 8} (tools/SplitAlignment.cpp:25-29,231-234). */
typedef struct dfb_split_params
{
	int32_t match;
	int32_t mismatch;
	int32_t gap;
	int32_t end_gaps;
	int32_t min_split_score;
} dfb_split_params;

/* One winning split row of one task: the factorised form of what
 * SplitReadAligner::GetAlignments emits (tools/SplitReadAligner.cpp:229-297).  For a task the
 * rows come in ascending read_split; GetAlignments' output for the task is, in order,
 *   for row in rows(task): for i1 in cols[col_begin .. +n1): for i2 in cols[col_begin+n1 .. +n2):
 *     refSplit  = (i1, len(reference2) - i2 - 1)      readSplit = (read_split, len(read) - read_split)
 *     score = score1 + score2,  score1,  score2
 * Rows whose column set is empty on either side emit nothing in the reference and are omitted. */
typedef struct dfb_split_row
{
	int32_t task;       /* index into the batch */
	int32_t read_split; /* alignedToRef1 (tools/SplitReadAligner.cpp:196) */
	int32_t score1;     /* row maximum of matrix 1 at read_split */
	int32_t score2;     /* row maximum of matrix 2 at len(read) - read_split */
	int64_t col_begin;  /* into the column pool: n1 ascending matrix-1 columns i1, then n2 ascending
	                       matrix-2 columns i2 (columns of the REVERSED reference2) */
	int32_t n1;
	int32_t n2;
} dfb_split_row;

/* Work/launch accounting of the last dfb_plan_run (for bench.py and the tools' --stats). */
typedef struct dfb_plan_stats
{
	int64_t n_tasks;
	int64_t cells;            /* interior DP cells: sum L*R (simple) or L*(R1+R2) (split) */
	int64_t fast_jobs;        /* s16x2 job pairs (two DPs per 32-bit lane word) */
	int64_t generic_jobs;     /* s32 jobs (parameters or lengths outside the s16x2 range) */
	int64_t probe_jobs;       /* split tasks re-swept to enumerate arg-max columns */
	int64_t events;           /* arg-max columns found */
	int64_t kernel_launches;  /* kernels launched by the last dfb_plan_run */
	int64_t h2d_bytes;        /* bytes copied host->device by plan creation */
	int64_t d2h_bytes;        /* bytes copied device->host by the last fetch */
	int64_t packed_bytes;     /* bytes of packed sequence data resident in HBM */
	int64_t raw_bytes;        /* bytes of raw sequence data the pack kernel read */
	/* CUDA-event timings on the context's stream, in ms; valid after dfb_plan_sync when
	 * dfb_plan_set_timing(plan, 1) was called, else 0 */
	double ms_pack;           /* the pack kernel at plan creation (always measured) */
	double ms_sweep;          /* first-sweep DP kernels of the last run (all classes) */
	double ms_probe;          /* probe-sweep kernels of the last run */
} dfb_plan_stats;

typedef struct dfb_device_info
{
	char name[128];
	int32_t ordinal;
	int32_t sm_count;
	int32_t cc_major;
	int32_t cc_minor;
	int32_t clock_khz; /* max SM clock */
	int64_t total_mem;
} dfb_device_info;

/* ---- context -------------------------------------------------------------------------- */

DFB_API int dfb_abi_version(void);
/* Number of visible CUDA devices, or a negative dfb_status. */
DFB_API int dfb_device_count(void);
/* Creates a context on CUDA device `device_ordinal`.  Fails with DFB_ERR_NODEVICE when the
 * device is absent or is not compute capability 10.x. */
DFB_API int dfb_ctx_create(int device_ordinal, dfb_ctx** ctx);
DFB_API void dfb_ctx_destroy(dfb_ctx* ctx);
/* Message of the last failure on `ctx`; with ctx == NULL, of the last failed dfb_ctx_create
 * on this thread.  Never NULL. */
DFB_API const char* dfb_last_error(const dfb_ctx* ctx);
/* Run on a caller-provided cudaStream_t (e.g. torch's current stream) instead of the
 * context's own; pass NULL to go back.  (NULL does not name the legacy default stream here: the context's own stream
 * does not wait for it.  Pass cudaStreamLegacy, (void*)1, to run behind work on the legacy default stream.) */
DFB_API int dfb_ctx_set_stream(dfb_ctx* ctx, void* cuda_stream);
DFB_API int dfb_ctx_device_info(const dfb_ctx* ctx, dfb_device_info* info);

/* ---- SimpleAligner::Align, batched (replaces tools/localalign.cpp:79, matealign.cpp:209) -- */

/* out_score[t] = SimpleAligner(params).Align(refs[task_ref[t]], seqs[task_seq[t]]).
 * One call = copy in, pack, align, copy out. */
DFB_API int dfb_simple_align_batch(dfb_ctx* ctx, const dfb_simple_params* params,
                           const dfb_seq_table* refs, const dfb_seq_table* seqs,
                           const int32_t* task_ref, const int32_t* task_seq, int64_t n_tasks,
                           int32_t* out_score);

/* ---- SplitReadAligner::Align + GetAlignments, batched (replaces SplitAlignment.cpp:376-379) -- */

/* Task t aligns reads[task_read[t]] against the window pair of cluster c = task_cluster[t]:
 * reference1 = refs[2c], reference2 = refs[2c+1] (refs->n must be even), with
 * minScore = task_min_score[t], forceSplits=true, firstOnly=false, backtrace=false.
 * out_best[t] = the winning split total (GetAlignments' maxScore), 0 when there is none.
 * The winning rows stay in the context until the next call on it; size them with
 * dfb_split_result_size and copy them out with dfb_split_result_copy. */
DFB_API int dfb_split_align_batch(dfb_ctx* ctx, const dfb_split_params* params,
                          const dfb_seq_table* refs, const dfb_seq_table* reads,
                          const int32_t* task_cluster, const int32_t* task_read,
                          const int32_t* task_min_score, int64_t n_tasks,
                          int32_t* out_best);
DFB_API int dfb_split_result_size(const dfb_ctx* ctx, int64_t* n_rows, int64_t* n_cols);
DFB_API int dfb_split_result_copy(const dfb_ctx* ctx, dfb_split_row* rows, int32_t* cols);
/* Zero-copy alternative: pointers into library-owned host memory, valid until the next split
 * call on this context (or its destruction). */
DFB_API int dfb_split_result_view(const dfb_ctx* ctx, const dfb_split_row** rows, int64_t* n_rows,
                                  const int32_t** cols, int64_t* n_cols);
/* Accounting of the last dfb_split_align_batch on this context (bytes copied each way, arg-max columns, probe jobs):
 * what the call itself moved -- a batch cut into chunks uploads every window once, a resident plan's statistics
 * (dfb_plan_get_stats) do not describe it.  Timings are 0. */
DFB_API int dfb_split_result_stats(const dfb_ctx* ctx, dfb_plan_stats* stats);

/* ---- device-resident forms: batches already in GPU memory, results left there ----------------- */

/* A table of byte strings in device memory (e.g. torch tensors): the CSR form of dfb_seq_table with `bytes` and `off`
 * on the GPU.  `n` and `n_bytes` are host values; n_bytes is the size of the `bytes` allocation, and off[n] may not
 * exceed it. */
typedef struct dfb_device_seq_table
{
	const uint8_t* bytes; /* device memory */
	const int64_t* off;   /* device memory, n + 1 entries, off[0] == 0, non-decreasing */
	int64_t n;            /* host value */
	int64_t n_bytes;      /* host value: size of the `bytes` allocation */
} dfb_device_seq_table;

/* The device-resident forms of dfb_simple_align_batch and dfb_split_align_batch.  Every array -- both tables, the task
 * arrays and the outputs -- is device memory of the context's device; host memory (pinned or pageable), managed memory
 * and memory of another device are refused with DFB_ERR_ARG before any work is queued.  The work is ordered behind what
 * was queued on the context's stream (dfb_ctx_set_stream) before the call, and the call returns once the outputs are
 * written.  Results are those of the host forms on the same data, byte for byte and in the same order; malformed
 * tables and task indices fail with the same status and message (plus "off[n] exceeds n_bytes"), except that an index
 * out of range is always reported at the lowest bad task of the batch (the host form cuts a large batch with
 * non-decreasing reads into chunks first and may name a chunk's first task).  Sequence bytes,
 * offsets, task arrays and results stay on the GPU: what crosses PCIe is fixed-size counters (the argument-check record,
 * class counts, overflow and row/column totals; dfb_split_result_stats counts them), except for chunks holding tasks
 * only the s32 kernels take (scoring triples or lengths outside the s16x2 range), whose offsets and task arrays -- never
 * their bytes -- are read back to build their job lists on the host. */
DFB_API int dfb_simple_align_device(dfb_ctx* ctx, const dfb_simple_params* params,
                                    const dfb_device_seq_table* refs, const dfb_device_seq_table* seqs,
                                    const int32_t* d_task_ref, const int32_t* d_task_seq, int64_t n_tasks,
                                    int32_t* d_out_score);
/* out_best as for dfb_split_align_batch; *n_rows / *n_cols receive the result's size.  The rows and columns stay in
 * device memory owned by the context until the next split call on it: copy them with dfb_split_result_copy_device.
 * (dfb_split_result_size / _copy / _view refuse a device-resident result with DFB_ERR_STATE.) */
DFB_API int dfb_split_align_device(dfb_ctx* ctx, const dfb_split_params* params,
                                   const dfb_device_seq_table* refs, const dfb_device_seq_table* reads,
                                   const int32_t* d_task_cluster, const int32_t* d_task_read,
                                   const int32_t* d_task_min_score, int64_t n_tasks,
                                   int32_t* d_out_best, int64_t* n_rows, int64_t* n_cols);
/* Copies the last dfb_split_align_device result into device buffers of n_rows / n_cols entries. */
DFB_API int dfb_split_result_copy_device(dfb_ctx* ctx, dfb_split_row* d_rows, int32_t* d_cols);

/* One record SplitAlignmentTask::Align keeps (tools/SplitAlignment.cpp:381-400): the first alignment of a task with
 * a given refSplit, scored min(score1, score2).  This is what dosplitalign writes per task. */
typedef struct dfb_split_record
{
	int32_t task;
	int32_t ref_split1;  /* refSplit.first  = i1 */
	int32_t ref_split2;  /* refSplit.second = len(reference2) - i2 - 1 */
	int32_t read_split1; /* readSplit.first  = read_split */
	int32_t read_split2; /* readSplit.second = len(read) - read_split */
	int32_t score;       /* min(score1, score2) */
} dfb_split_record;

/* The records of a device-resident split result, expanded and de-duplicated on the GPU.  rows / cols are a result in
 * the form dfb_split_result_copy_device writes (any device buffers holding one: the call keeps no state of the last
 * split call), refs / reads / d_task_cluster / d_task_read the batch it was computed from; len(read) and
 * len(reference2) are read from them.  Order, which is the order GetAlignments emits (tools/SplitReadAligner.cpp:
 * 272-297) and dosplitalign keeps: tasks ascending; within a task, rows in the order given, then i1 ascending, then
 * i2 ascending; of the alignments with the same (i1, i2) only the first in this order is kept.  Rows with n1 == 0 or
 * n2 == 0 and tasks without rows give nothing.  Every array is device memory of the context's device (else
 * DFB_ERR_ARG before any work is queued).  The argument checks run on the GPU: those of dfb_split_align_device on the
 * tables and task arrays (same statuses and messages), and on the rows -- task in [0, n_tasks) and non-decreasing,
 * col_begin >= 0, n1, n2 >= 0, col_begin + n1 + n2 <= n_cols, 0 <= read_split <= len(read), every column in
 * [0, len(window)] on its side and strictly ascending within its list -- which also catch tables that do not belong to
 * the rows.  The work is ordered behind the context's stream and the call returns once the records are written; what
 * crosses PCIe is the check record and the totals.  *n_records receives the number of records, which stay in device
 * memory owned by the context until the next dfb_split_records_device call on it (or dfb_ctx_destroy). */
DFB_API int dfb_split_records_device(dfb_ctx* ctx, const dfb_device_seq_table* refs, const dfb_device_seq_table* reads,
                                     const int32_t* d_task_cluster, const int32_t* d_task_read, int64_t n_tasks,
                                     const dfb_split_row* d_rows, int64_t n_rows, const int32_t* d_cols, int64_t n_cols,
                                     int64_t* n_records);
/* Copies the records of the last successful dfb_split_records_device call into a device buffer of n_records entries;
 * DFB_ERR_STATE when there are none. */
DFB_API int dfb_split_records_copy_device(dfb_ctx* ctx, dfb_split_record* d_records);

/* ---- backtrace of chosen split alignments (GetAlignments(..., backtrace=true)) ------------- */

/* The matches1 / matches2 lists of SplitReadAlignment (tools/SplitReadAligner.h:21-30) for alignments the caller
 * picked from a dfb_split_align_batch result -- what SplitAlignmentTask::ReAlign needs (tools/SplitAlignment.cpp:
 * 443-464, caller tools/splitseq.cpp:122).  Task t names one alignment of reads[task_read[t]] against cluster
 * task_cluster[t] by its refSplit = (task_ref_split1[t], task_ref_split2[t]) and readSplit.first =
 * task_read_split[t]; the start cells are (refSplit.first, readSplit.first) in matrix 1 and
 * (len(reference2) - refSplit.second - 1, len(read) - readSplit.first) in matrix 2 (SplitReadAligner.cpp:271-292).
 * Pointers follow the reference's rule -- (i,j-1) over (i-1,j) over the diagonal when scores tie (:56-69) -- and
 * every diagonal step on the way to read position 0 is a match pair (refPos, readPos) (:124-143); matrix 2's pairs
 * are mapped back to the unreversed sequences (:145-154).  Both lists come out ascending.
 *   match_off : 2*n_tasks + 1 entries; pairs [match_off[2t], match_off[2t+1]) are matches1 of task t,
 *               [match_off[2t+1], match_off[2t+2]) its matches2
 *   matches   : interleaved (refPos, readPos); at most sum(len(read)) pairs are produced, so a buffer of
 *               2 * sum(len(read)) int32 always suffices (matches_cap counts pairs); NULL only sizes; a matches_cap
 *               below the total is DFB_ERR_ARG, with match_off and n_pairs written and matches untouched
 *   n_pairs   : total number of pairs
 * The arguments are checked on the host; the tables, task arrays and one dfb_split_record per alignment are then
 * uploaded and the kernels of dfb_split_backtrace_device run on them.  Nothing stays allocated after the call, and the
 * context's dfb_split_backtrace_device result is left as it was.  At most 0x7fffff00 alignments per call (records
 * carry an int32 task index); more is DFB_ERR_ARG "too many tasks in one batch". */
DFB_API int dfb_split_backtrace_batch(dfb_ctx* ctx, const dfb_split_params* params,
                          const dfb_seq_table* refs, const dfb_seq_table* reads,
                          const int32_t* task_cluster, const int32_t* task_read,
                          const int32_t* task_ref_split1, const int32_t* task_ref_split2,
                          const int32_t* task_read_split, int64_t n_tasks,
                          int64_t* match_off, int32_t* matches, int64_t matches_cap, int64_t* n_pairs);

/* The device-resident form of dfb_split_backtrace_batch, for records of a device-resident split result.  Record k
 * names one alignment of task t = d_records[k].task: reads[d_task_read[t]] against cluster d_task_cluster[t], with
 * refSplit (ref_split1, ref_split2) and readSplit.first = read_split1; the start cells are those of
 * dfb_split_backtrace_batch, and score is not read.  The records may be any rows of a dfb_split_records_device output
 * or records built by hand, in any order and with repeats.  The output has the layout of dfb_split_backtrace_batch --
 * 2 * n_records + 1 int64 offsets, interleaved int32 (refPos, readPos) pairs, both lists ascending -- and is byte-equal
 * to it called per record with (task_cluster[t], task_read[t], ref_split1, ref_split2, read_split1); it is exact-size
 * and *n_pairs receives the total.  Every array is device memory of the context's device (else DFB_ERR_ARG before any
 * work is queued).  The argument checks run on the GPU: those of dfb_split_align_device on the tables and task arrays
 * (same statuses and messages), and per record -- task in [0, n_tasks), both start cells inside their matrices,
 * read_split2 == len(read) - read_split1 (which also catches tables that do not belong to the records) -- reported at
 * the lowest bad record.  The work is ordered behind the context's stream and the call returns once the output is
 * written; what crosses PCIe is the check record and the totals.  The output stays in device memory owned by the
 * context until the next dfb_split_backtrace_device call on it (or dfb_ctx_destroy). */
DFB_API int dfb_split_backtrace_device(dfb_ctx* ctx, const dfb_split_params* params,
                                       const dfb_device_seq_table* refs, const dfb_device_seq_table* reads,
                                       const int32_t* d_task_cluster, const int32_t* d_task_read, int64_t n_tasks,
                                       const dfb_split_record* d_records, int64_t n_records, int64_t* n_pairs);
/* Copies the output of the last successful dfb_split_backtrace_device call into device buffers of 2 * n_records + 1
 * offsets and 2 * n_pairs int32; DFB_ERR_STATE when there is none. */
DFB_API int dfb_split_backtrace_copy_device(dfb_ctx* ctx, int64_t* d_match_off, int32_t* d_matches);

/* ---- staged form: the same work with the batch resident in HBM -------------------------- */

/* Copies the tables to the device, packs them (2-bit codes + exception plane) and builds
 * the length-bucketed job lists.  The host buffers are not referenced afterwards. */
DFB_API int dfb_simple_plan_create(dfb_ctx* ctx, const dfb_simple_params* params,
                           const dfb_seq_table* refs, const dfb_seq_table* seqs,
                           const int32_t* task_ref, const int32_t* task_seq, int64_t n_tasks,
                           dfb_plan** plan);
DFB_API int dfb_split_plan_create(dfb_ctx* ctx, const dfb_split_params* params,
                          const dfb_seq_table* refs, const dfb_seq_table* reads,
                          const int32_t* task_cluster, const int32_t* task_read,
                          const int32_t* task_min_score, int64_t n_tasks,
                          dfb_plan** plan);
/* Enqueues every DP kernel of the plan on the context's stream and returns without
 * synchronising.  May be called repeatedly (outputs are overwritten). */
DFB_API int dfb_plan_run(dfb_plan* plan);
/* With enable != 0, dfb_plan_run brackets its kernel groups with CUDA events (ms_sweep, ms_probe). */
DFB_API int dfb_plan_set_timing(dfb_plan* plan, int enable);
/* Waits for the stream and reports any kernel failure. */
DFB_API int dfb_plan_sync(dfb_plan* plan);
DFB_API int dfb_simple_plan_fetch(dfb_plan* plan, int32_t* out_score);
/* Copies the split outputs to the host and assembles the rows (re-running the probe sweep
 * with a larger event buffer if it overflowed).  Then use dfb_split_plan_copy. */
DFB_API int dfb_split_plan_fetch(dfb_plan* plan, int32_t* out_best, int64_t* n_rows, int64_t* n_cols);
DFB_API int dfb_split_plan_copy(const dfb_plan* plan, dfb_split_row* rows, int32_t* cols);
/* Zero-copy alternative, valid until the next fetch on this plan (or its destruction). */
DFB_API int dfb_split_plan_view(const dfb_plan* plan, const dfb_split_row** rows, int64_t* n_rows,
                                const int32_t** cols, int64_t* n_cols);
DFB_API int dfb_plan_get_stats(const dfb_plan* plan, dfb_plan_stats* stats);
DFB_API void dfb_plan_destroy(dfb_plan* plan);

/* ---- measurement support --------------------------------------------------------------- */

/* Device memory of the context's stream-ordered pool: bytes reserved from the driver now, and the
 * high-water marks of reserved and used bytes since the context was created (or since the last
 * call with reset != 0).  What a batch holds on the GPU at most (DESIGN.md 3). */
DFB_API int dfb_ctx_memory_info(dfb_ctx* ctx, int reset, int64_t* reserved_now, int64_t* reserved_high,
                                int64_t* used_high);

/* Integer/DPX issue-rate microbenchmark (the denominator of the DP roofline, SURVEY.md 8d).
 * Runs dependent-free streams of one instruction kind on every SM and returns
 * warp-instructions issued per second (whole chip).  `kind`:
 *   0 VIADDMNMX.S16x2   1 VIMNMX.U16x2   2 VIMNMX3.S16x2   3 LOP3   4 IMAD   5 IADD3
 *   6 PRMT              7 the 6-instruction s16x2 DP cell body (per body, not per instruction)
 *   8 SHFL.UP           9 VIADDMNMX (s32)
 *   10 HMNMX2   11 HADD2   12 HFMA2   13 HSET2 (fp16x2: candidates for the fma pipe)
 *   14 / 15 / 16  VIADDMNMX.S16x2 interleaved 1:1 with HMNMX2 / HFMA2 / HADD2 (do the two pipes issue side by side?)
 * *elapsed_ms receives the kernel time. */
DFB_API int dfb_microbench_issue_rate(dfb_ctx* ctx, int kind, int iters, double* warp_instr_per_s,
                              double* elapsed_ms);

#ifdef __cplusplus
}
#endif

#endif /* DEFUSE_B200_H_ */
