// Records of a device-resident split result: what SplitAlignmentTask::Align keeps of GetAlignments' output
// (tools/SplitAlignment.cpp:381-400, tools/SplitReadAligner.cpp:272-297) -- the first alignment of every distinct
// refSplit of a task, scored min(score1, score2) -- expanded from the factorised rows + column pool on the GPU.
//
// Included at the end of dfb_api.cu (it needs dfb_ctx).  A task's alignments are the raw pairs (i1, i2) of
// cols1 x cols2 of each of its rows, in row order.  A pair of row r is a duplicate iff an earlier row of the same task
// holds i1 on side 1 and i2 on side 2, so the first row of a task (and every row of a one-row task) is all fresh.
// For the other rows, every column entry gets a bitmask of the earlier rows of its task whose list on that side holds
// the column (one binary search per earlier row); a pair is fresh iff mask(i1) & mask(i2) == 0, ceil(k / 64) words for
// the row's index k within its task.  The raw-pair space (int64) is never materialised: blocks take contiguous ranges
// of it, count their fresh pairs, and after a scan of the block counts write them in raw order.
//
//   rec_rows_kernel        per row: argument checks, n1 * n2, index within the task, mask words, lengths
//   rec_cols_kernel        one warp per row: columns inside their window and strictly ascending
//   rec_mask_kernel        one thread per mask word (64 earlier rows of one column entry)
//   rec_count_kernel       fresh pairs per block of DFB_REC_SPAN raw pairs
//   rec_write_kernel       the same pairs again, compacted in raw order (block prefix of the fresh flags)
#pragma once

namespace dfb
{

#define DFB_REC_BLOCK 256
#define DFB_REC_ITEMS 16
#define DFB_REC_SPAN (DFB_REC_BLOCK * DFB_REC_ITEMS)

enum RecBad
{
	REC_BAD_TASK,  // task out of [0, n_tasks)
	REC_BAD_ORDER, // tasks decrease
	REC_BAD_POOL,  // col_begin / n1 / n2 outside the column pool
	REC_BAD_SPLIT, // read_split outside [0, len(read)]
	REC_BAD_COLS,  // a column outside its window, or a list not strictly ascending
	REC_NUM_BAD
};

struct RecCheck
{
	DeviceCheck dc;                       // the tables and task arrays, as for dfb_split_align_device
	unsigned long long bad[REC_NUM_BAD];  // lowest row with each fault (~0: none)
	unsigned long long raw_pairs, mask_words, n_records;
};

struct RecRow
{
	int32_t k;  // index of the row within its task
	int32_t L;  // len(read)
	int32_t R2; // len(reference2)
	int32_t pad;
};

struct RecTables
{
	const int64_t* ref_off;
	const int64_t* read_off;
	const int32_t* task_cluster;
	const int32_t* task_read;
	long long n_clusters, n_reads, n_tasks, n_cols;
};

__global__ void rec_check_init_kernel(RecCheck* c)
{
	for (int k = 0; k < REC_NUM_BAD; k++) c->bad[k] = ~0ull;
	c->raw_pairs = c->mask_words = c->n_records = 0;
}

// the row's lengths, when its task, its pool range and the task's table indices are in range (nothing else is read)
__device__ __forceinline__ bool rec_row_lengths(const RecTables& t, const dfb_split_row& w, int* L, int* R1, int* R2)
{
	if (w.task < 0 || w.task >= t.n_tasks) return false;
	if (w.col_begin < 0 || w.n1 < 0 || w.n2 < 0 || w.col_begin > t.n_cols - (long long)w.n1 - (long long)w.n2) return false;
	const int c = t.task_cluster[w.task], q = t.task_read[w.task];
	if (c < 0 || c >= t.n_clusters || q < 0 || q >= t.n_reads) return false;
	*L = (int)(t.read_off[q + 1] - t.read_off[q]);
	*R1 = (int)(t.ref_off[2 * c + 1] - t.ref_off[2 * c]);
	*R2 = (int)(t.ref_off[2 * c + 2] - t.ref_off[2 * c + 1]);
	return true;
}

__global__ void __launch_bounds__(DFB_BUILD_BLOCK) rec_rows_kernel(const dfb_split_row* __restrict__ rows, long long n_rows, RecTables t,
                                                                    RecCheck* chk, unsigned long long* pairs, unsigned long long* mwords,
                                                                    RecRow* info)
{
	const long long stride = (long long)gridDim.x * DFB_BUILD_BLOCK;
	for (long long r = (long long)blockIdx.x * DFB_BUILD_BLOCK + threadIdx.x; r < n_rows; r += stride)
	{
		const dfb_split_row w = rows[r];
		if (w.task < 0 || w.task >= t.n_tasks) atomicMin(&chk->bad[REC_BAD_TASK], (unsigned long long)r);
		if (r > 0 && w.task < rows[r - 1].task) atomicMin(&chk->bad[REC_BAD_ORDER], (unsigned long long)r);
		if (w.col_begin < 0 || w.n1 < 0 || w.n2 < 0 || w.col_begin > t.n_cols - (long long)w.n1 - (long long)w.n2)
			atomicMin(&chk->bad[REC_BAD_POOL], (unsigned long long)r);
		int L = 0, R1 = 0, R2 = 0;
		const bool ok = rec_row_lengths(t, w, &L, &R1, &R2);
		if (ok && (w.read_split < 0 || w.read_split > L)) atomicMin(&chk->bad[REC_BAD_SPLIT], (unsigned long long)r);
		// first row of the task: rows are in task order (checked above; a batch that is not is refused before use)
		long long lo = 0, hi = r;
		while (lo < hi)
		{
			const long long m = (lo + hi) >> 1;
			if (rows[m].task < w.task) lo = m + 1;
			else hi = m;
		}
		const long long k = r - lo;
		const bool live = ok && w.n1 > 0 && w.n2 > 0;
		pairs[r] = live ? (unsigned long long)w.n1 * (unsigned long long)w.n2 : 0ull;
		mwords[r] = live && k > 0 ? (unsigned long long)(w.n1 + w.n2) * (unsigned long long)((k + 63) >> 6) : 0ull;
		info[r] = RecRow{(int32_t)min(k, (long long)INT32_MAX), L, R2, 0};
	}
}

__global__ void __launch_bounds__(DFB_BUILD_BLOCK) rec_cols_kernel(const dfb_split_row* __restrict__ rows, long long n_rows,
                                                                    const int32_t* __restrict__ cols, RecTables t, RecCheck* chk)
{
	const int lane = threadIdx.x & 31;
	const long long warps = (long long)gridDim.x * (DFB_BUILD_BLOCK / 32);
	for (long long r = ((long long)blockIdx.x * DFB_BUILD_BLOCK + threadIdx.x) >> 5; r < n_rows; r += warps)
	{
		const dfb_split_row w = rows[r];
		int L, R1, R2;
		if (!rec_row_lengths(t, w, &L, &R1, &R2)) continue;
		const int n = w.n1 + w.n2;
		int bad = 0;
		for (int e = lane; e < n; e += 32)
		{
			const int32_t c = cols[w.col_begin + e];
			const int lim = e < w.n1 ? R1 : R2; // a matrix has len(window) + 1 columns
			bad |= c < 0 || c > lim || (e != 0 && e != w.n1 && cols[w.col_begin + e - 1] >= c);
		}
		if (__any_sync(0xffffffffu, bad) && lane == 0) atomicMin(&chk->bad[REC_BAD_COLS], (unsigned long long)r);
	}
}

// largest r in [lo, hi) with scan[r] <= x (scan: exclusive prefix sums; the row that holds item x)
__device__ __forceinline__ long long rec_find(const unsigned long long* __restrict__ scan, long long lo, long long hi, unsigned long long x)
{
	while (hi - lo > 1)
	{
		const long long m = (lo + hi) >> 1;
		if (scan[m] <= x) lo = m;
		else hi = m;
	}
	return lo;
}

struct RecParams
{
	const dfb_split_row* rows;
	const int32_t* cols;
	long long n_rows;
	const unsigned long long* pstart; // first raw pair of each row
	const unsigned long long* moff;   // first mask word of each row
	const RecRow* info;
	unsigned long long* masks;
	unsigned long long raw, n_mask_words;
	unsigned long long* counts; // fresh pairs per block; scanned: first record of each block
	dfb_split_record* out;
};

__device__ __forceinline__ bool rec_holds(const int32_t* __restrict__ list, int n, int32_t c)
{
	int lo = 0, hi = n;
	while (lo < hi)
	{
		const int m = (lo + hi) >> 1;
		if (list[m] < c) lo = m + 1;
		else hi = m;
	}
	return lo < n && list[lo] == c;
}

// mask word g: bits j - 64 w of the earlier rows j in [64 w, min(64 w + 64, k)) of the task whose list on the entry's
// side holds the entry's column
__global__ void __launch_bounds__(DFB_BUILD_BLOCK) rec_mask_kernel(RecParams p)
{
	const unsigned long long stride = (unsigned long long)gridDim.x * DFB_BUILD_BLOCK;
	for (unsigned long long g = (unsigned long long)blockIdx.x * DFB_BUILD_BLOCK + threadIdx.x; g < p.n_mask_words; g += stride)
	{
		const long long r = rec_find(p.moff, 0, p.n_rows, g);
		const dfb_split_row w = p.rows[r];
		const int k = p.info[r].k;
		const unsigned W = (unsigned)((k + 63) >> 6);
		const unsigned long long local = g - p.moff[r];
		const long long e = (long long)(local / W);
		const int word = (int)(local % W);
		const int32_t c = p.cols[w.col_begin + e];
		const bool side2 = e >= w.n1;
		const long long first = r - k;
		unsigned long long bits = 0;
		const int j_end = min(64 * word + 64, k);
		for (int j = 64 * word; j < j_end; j++)
		{
			const dfb_split_row o = p.rows[first + j];
			const bool has = side2 ? rec_holds(p.cols + o.col_begin + o.n1, o.n2, c) : rec_holds(p.cols + o.col_begin, o.n1, c);
			bits |= (unsigned long long)has << (j - 64 * word);
		}
		p.masks[g] = bits;
	}
}

// raw pair idx -> row r, i1 index a, i2 index b; fresh iff no earlier row of the task holds both columns
struct RecPair
{
	long long r;
	int a, b;
	bool fresh;
};

__device__ __forceinline__ RecPair rec_pair(const RecParams& p, long long r_lo, long long r_hi, unsigned long long idx)
{
	RecPair q;
	q.r = rec_find(p.pstart, r_lo, r_hi, idx);
	const unsigned long long off = idx - p.pstart[q.r];
	const unsigned n2 = (unsigned)p.rows[q.r].n2;
	if (off < (1ull << 32))
	{
		q.a = (int)((unsigned)off / n2);
		q.b = (int)((unsigned)off - (unsigned)q.a * n2);
	}
	else
	{
		q.a = (int)(off / n2);
		q.b = (int)(off - (unsigned long long)q.a * n2);
	}
	q.fresh = true;
	const int k = p.info[q.r].k;
	if (k > 0)
	{
		const unsigned W = (unsigned)((k + 63) >> 6);
		const unsigned long long* m1 = p.masks + p.moff[q.r] + (unsigned long long)q.a * W;
		const unsigned long long* m2 = p.masks + p.moff[q.r] + (unsigned long long)(p.rows[q.r].n1 + q.b) * W;
		for (unsigned v = 0; v < W && q.fresh; v++) q.fresh = (m1[v] & m2[v]) == 0;
	}
	return q;
}

// rows holding the raw pairs [start, end) of this block
__device__ __forceinline__ void rec_block_rows(const RecParams& p, unsigned long long start, unsigned long long end, long long* r_lo, long long* r_hi)
{
	__shared__ long long s_r[2];
	if (threadIdx.x == 0)
	{
		s_r[0] = rec_find(p.pstart, 0, p.n_rows, start);
		s_r[1] = rec_find(p.pstart, s_r[0], p.n_rows, end - 1) + 1;
	}
	__syncthreads();
	*r_lo = s_r[0];
	*r_hi = s_r[1];
}

__global__ void __launch_bounds__(DFB_REC_BLOCK) rec_count_kernel(RecParams p)
{
	const unsigned long long start = (unsigned long long)blockIdx.x * DFB_REC_SPAN;
	const unsigned long long end = min(start + DFB_REC_SPAN, p.raw);
	long long r_lo, r_hi;
	rec_block_rows(p, start, end, &r_lo, &r_hi);
	unsigned long long n = 0;
#pragma unroll 4
	for (int it = 0; it < DFB_REC_ITEMS; it++)
	{
		const unsigned long long idx = start + (unsigned long long)it * DFB_REC_BLOCK + threadIdx.x;
		if (idx < end) n += rec_pair(p, r_lo, r_hi, idx).fresh;
	}
	unsigned long long all = 0;
	block_exclusive_scan(n, &all);
	if (threadIdx.x == 0) p.counts[blockIdx.x] = all;
}

__global__ void __launch_bounds__(DFB_REC_BLOCK) rec_write_kernel(RecParams p)
{
	const unsigned long long start = (unsigned long long)blockIdx.x * DFB_REC_SPAN;
	const unsigned long long end = min(start + DFB_REC_SPAN, p.raw);
	long long r_lo, r_hi;
	rec_block_rows(p, start, end, &r_lo, &r_hi);
	unsigned long long at = p.counts[blockIdx.x];
	for (int it = 0; it < DFB_REC_ITEMS; it++)
	{
		const unsigned long long idx = start + (unsigned long long)it * DFB_REC_BLOCK + threadIdx.x;
		RecPair q{0, 0, 0, false};
		if (idx < end) q = rec_pair(p, r_lo, r_hi, idx);
		unsigned long long all = 0;
		const unsigned long long pos = at + block_exclusive_scan(q.fresh ? 1ull : 0ull, &all);
		if (q.fresh)
		{
			const dfb_split_row w = p.rows[q.r];
			const RecRow inf = p.info[q.r];
			dfb_split_record o;
			o.task = w.task;
			o.ref_split1 = p.cols[w.col_begin + q.a];
			o.ref_split2 = inf.R2 - p.cols[w.col_begin + w.n1 + q.b] - 1;
			o.read_split1 = w.read_split;
			o.read_split2 = inf.L - w.read_split;
			o.score = min(w.score1, w.score2);
			p.out[pos] = o;
		}
		at += all;
	}
}

}  // namespace dfb

// ---- dfb_split_records_device ---------------------------------------------------------------------------------------

static int dfb_split_records_device_body(dfb_ctx* ctx, const dfb_device_seq_table* refs, const dfb_device_seq_table* reads,
                                         const int32_t* task_cluster, const int32_t* task_read, int64_t n_tasks,
                                         const dfb_split_row* rows, int64_t n_rows, const int32_t* cols, int64_t n_cols, int64_t* n_records)
{
	if (!ctx) return DFB_ERR_ARG;
	ctx->has_records = false;
	ctx->n_records = 0;
	dfree(ctx, ctx->d_records);
	if (!n_records || n_tasks < 0 || n_rows < 0 || n_cols < 0 || (n_tasks > 0 && (!task_cluster || !task_read)) || (n_rows > 0 && !rows) ||
	    (n_cols > 0 && !cols))
		return set_err(ctx, DFB_ERR_ARG, "dfb_split_records_device: null argument");
	const char* names[2] = {"refs", "reads"};
	const dfb_device_seq_table* tabs[2] = {refs, reads};
	for (int k = 0; k < 2; k++)
		if (!tabs[k] || !tabs[k]->off || tabs[k]->n < 0 || tabs[k]->n_bytes < 0) return set_err(ctx, DFB_ERR_ARG, "%s: null table", names[k]);
	CK(ctx, cudaSetDevice(ctx->device));
	const void* ptrs[8] = {refs->bytes, refs->off, reads->bytes, reads->off, task_cluster, task_read, rows, cols};
	const char* what[8] = {"refs->bytes", "refs->off", "reads->bytes", "reads->off", "task_cluster", "task_read", "rows", "cols"};
	for (int k = 0; k < 8; k++)
		if (!is_ctx_device_memory(ctx, ptrs[k]))
			return set_err(ctx, DFB_ERR_ARG, "%s is not device memory of device %d", what[k], ctx->device);
	if (n_tasks > 0x7fffff00LL) return set_err(ctx, DFB_ERR_ARG, "too many tasks in one batch");

	cudaStream_t s = ctx->stream;
	RecCheck* d_chk = nullptr;
	unsigned long long *pairs = nullptr, *mwords = nullptr, *sums = nullptr, *masks = nullptr, *counts = nullptr;
	RecRow* info = nullptr;
	auto cleanup = [&]() {
		dfree(ctx, d_chk);
		dfree(ctx, pairs);
		dfree(ctx, mwords);
		dfree(ctx, sums);
		dfree(ctx, masks);
		dfree(ctx, counts);
		dfree(ctx, info);
	};
	auto fail = [&](int code) {
		cleanup();
		cudaStreamSynchronize(s);
		return code;
	};
	auto scan_sums = [](long long n) { return (size_t)(n / (DFB_BUILD_BLOCK * DFB_BUILD_ITEMS) + 2) * sizeof(unsigned long long); };
	cudaError_t e = dalloc(ctx, (void**)&d_chk, sizeof(RecCheck));
	if (e == cudaSuccess) e = dalloc(ctx, (void**)&pairs, (size_t)n_rows * 8);
	if (e == cudaSuccess) e = dalloc(ctx, (void**)&mwords, (size_t)n_rows * 8);
	if (e == cudaSuccess) e = dalloc(ctx, (void**)&info, (size_t)n_rows * sizeof(RecRow));
	if (e == cudaSuccess) e = dalloc(ctx, (void**)&sums, scan_sums(n_rows));
	if (e == cudaSuccess) e = ctx->h_out.ensure(sizeof(RecCheck));
	if (e != cudaSuccess) return fail(set_err(ctx, DFB_ERR_NOMEM, "records: %s", cudaGetErrorString(e)));
	RecCheck* h_chk = (RecCheck*)ctx->h_out.p;

	// 1. checks, per-row counts and their scans; one read-back
	const RecTables t{refs->off, reads->off, task_cluster, task_read, refs->n / 2, reads->n, n_tasks, n_cols};
	const long long max_grid = (long long)ctx->prop.multiProcessorCount * 8;
	auto grid = [&](long long n) { return (unsigned)std::max<long long>(1, std::min<long long>((n + DFB_BUILD_BLOCK - 1) / DFB_BUILD_BLOCK, max_grid)); };
	enqueue_device_checks(ctx, false, refs, reads, task_cluster, task_read, n_tasks, &d_chk->dc);
	rec_check_init_kernel<<<1, 1, 0, s>>>(d_chk);
	if (n_rows)
	{
		rec_rows_kernel<<<grid(n_rows), DFB_BUILD_BLOCK, 0, s>>>(rows, n_rows, t, d_chk, pairs, mwords, info);
		rec_cols_kernel<<<grid(32 * n_rows), DFB_BUILD_BLOCK, 0, s>>>(rows, n_rows, cols, t, d_chk);
		int rc = scan_u64(ctx, pairs, n_rows, sums, &d_chk->raw_pairs);
		if (!rc) rc = scan_u64(ctx, mwords, n_rows, sums, &d_chk->mask_words);
		if (rc) return fail(rc);
	}
	e = cudaGetLastError();
	if (e == cudaSuccess) e = cudaMemcpyAsync(h_chk, d_chk, sizeof(RecCheck), cudaMemcpyDeviceToHost, s);
	if (e == cudaSuccess) e = cudaStreamSynchronize(s);
	if (e != cudaSuccess) return fail(set_err(ctx, DFB_ERR_CUDA, "records checks: %s", cudaGetErrorString(e)));
	const RecCheck chk = *h_chk;
	if (int rc = device_check_status(ctx, false, refs, reads, n_tasks, chk.dc)) return fail(rc);
	static const char* const bad_msg[REC_NUM_BAD] = {"task out of range", "tasks decrease", "columns outside the column pool",
	                                                  "read_split outside [0, len(read)]", "a column outside its window or not ascending"};
	for (int k = 0; k < REC_NUM_BAD; k++)
		if (chk.bad[k] != ~0ull) return fail(set_err(ctx, DFB_ERR_ARG, "row %lld: %s", (long long)chk.bad[k], bad_msg[k]));

	// 2. masks, fresh pairs per block, their scan; the total comes back to size the output
	const unsigned long long raw = chk.raw_pairs;
	const unsigned long long n_blocks = (raw + DFB_REC_SPAN - 1) / DFB_REC_SPAN;
	if (n_blocks > 0x7fffffffull) return fail(set_err(ctx, DFB_ERR_ARG, "%llu alignments before de-duplication: too many for one call", raw));
	RecParams p;
	p.rows = rows;
	p.cols = cols;
	p.n_rows = n_rows;
	p.pstart = pairs;
	p.moff = mwords;
	p.info = info;
	p.masks = nullptr;
	p.raw = raw;
	p.n_mask_words = chk.mask_words;
	p.counts = nullptr;
	p.out = nullptr;
	unsigned long long n_out = 0;
	if (raw)
	{
		dfree(ctx, sums);
		e = dalloc(ctx, (void**)&masks, (size_t)chk.mask_words * 8);
		if (e == cudaSuccess) e = dalloc(ctx, (void**)&counts, (size_t)n_blocks * 8);
		if (e == cudaSuccess) e = dalloc(ctx, (void**)&sums, scan_sums((long long)n_blocks));
		if (e != cudaSuccess) return fail(set_err(ctx, DFB_ERR_NOMEM, "records scratch (%llu mask words): %s", chk.mask_words, cudaGetErrorString(e)));
		p.masks = masks;
		p.counts = counts;
		if (chk.mask_words)
			rec_mask_kernel<<<(unsigned)std::min<unsigned long long>((chk.mask_words + DFB_BUILD_BLOCK - 1) / DFB_BUILD_BLOCK, (unsigned long long)max_grid * 4),
			                  DFB_BUILD_BLOCK, 0, s>>>(p);
		rec_count_kernel<<<(unsigned)n_blocks, DFB_REC_BLOCK, 0, s>>>(p);
		if (int rc = scan_u64(ctx, counts, (long long)n_blocks, sums, &d_chk->n_records)) return fail(rc);
		e = cudaMemcpyAsync(h_chk, d_chk, sizeof(RecCheck), cudaMemcpyDeviceToHost, s);
		if (e == cudaSuccess) e = cudaStreamSynchronize(s);
		if (e != cudaSuccess) return fail(set_err(ctx, DFB_ERR_CUDA, "records count: %s", cudaGetErrorString(e)));
		n_out = h_chk->n_records;
	}
	// 3. the records
	if (n_out)
	{
		e = dalloc(ctx, (void**)&ctx->d_records, (size_t)n_out * sizeof(dfb_split_record));
		if (e != cudaSuccess) return fail(set_err(ctx, DFB_ERR_NOMEM, "%llu records: %s", n_out, cudaGetErrorString(e)));
		p.out = ctx->d_records;
		rec_write_kernel<<<(unsigned)n_blocks, DFB_REC_BLOCK, 0, s>>>(p);
		e = cudaGetLastError();
		if (e != cudaSuccess)
		{
			dfree(ctx, ctx->d_records);
			return fail(set_err(ctx, DFB_ERR_CUDA, "records write: %s", cudaGetErrorString(e)));
		}
	}
	cleanup();
	e = cudaStreamSynchronize(s);
	if (e != cudaSuccess)
	{
		dfree(ctx, ctx->d_records);
		return set_err(ctx, DFB_ERR_CUDA, "records: %s", cudaGetErrorString(e));
	}
	if (int rc = bounds_check_status(ctx)) return rc;
	ctx->n_records = (int64_t)n_out;
	ctx->has_records = true;
	*n_records = (int64_t)n_out;
	return DFB_OK;
}

extern "C" int dfb_split_records_device(dfb_ctx* ctx, const dfb_device_seq_table* refs, const dfb_device_seq_table* reads,
                                        const int32_t* task_cluster, const int32_t* task_read, int64_t n_tasks, const dfb_split_row* rows,
                                        int64_t n_rows, const int32_t* cols, int64_t n_cols, int64_t* n_records)
{
	return guarded(ctx, [&] {
		return dfb_split_records_device_body(ctx, refs, reads, task_cluster, task_read, n_tasks, rows, n_rows, cols, n_cols, n_records);
	});
}

extern "C" int dfb_split_records_copy_device(dfb_ctx* ctx, dfb_split_record* records)
{
	return guarded(ctx, [&]() -> int {
		if (!ctx) return DFB_ERR_ARG;
		if (!ctx->has_records) return set_err(ctx, DFB_ERR_STATE, "no records on this context: call dfb_split_records_device first");
		if (ctx->n_records && !records) return set_err(ctx, DFB_ERR_ARG, "dfb_split_records_copy_device: null argument");
		CK(ctx, cudaSetDevice(ctx->device));
		if (!is_ctx_device_memory(ctx, records)) return set_err(ctx, DFB_ERR_ARG, "records is not device memory of device %d", ctx->device);
		if (ctx->n_records)
			CK(ctx, cudaMemcpyAsync(records, ctx->d_records, (size_t)ctx->n_records * sizeof(dfb_split_record), cudaMemcpyDeviceToDevice, ctx->stream));
		CK(ctx, cudaStreamSynchronize(ctx->stream));
		return DFB_OK;
	});
}
