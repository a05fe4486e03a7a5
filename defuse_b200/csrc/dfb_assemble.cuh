// Result assembly on the GPU: the second half of SplitReadAligner::GetAlignments (tools/SplitReadAligner.cpp:229-285)
// for the common task -- at most DFB_SLOT_EVENTS arg-max columns, all of them in the task's fixed 128-byte region
// left by the probe sweep.  The kernels order those columns the way GetAlignments walks them (matrix, row, column),
// pair every winning row a of matrix 1 with row L-a of matrix 2 and write the dfb_split_row records and their column
// lists in TASK ORDER into two dense arrays, so that the host only copies them back.  Tasks whose columns spilled into
// the overflow list (tie-heavy ones; a fraction of a percent of a dosplitalign batch) are left to the host: their region entries
// are appended to that list here, which makes the list self-contained.
//
//   asm_count_kernel   rows / columns per task -> sums per block of 256 tasks
//   asm_scan_kernel    exclusive scan of the block sums (one block), totals
//   asm_write_kernel   per-task offsets by an in-block scan, records written
// HBM-bound and tiny next to the sweeps: 128 B read and <= 320 B written per winning task.
#pragma once

namespace dfb
{
#define DFB_ASM_MAX_CLASSES 16
#define DFB_ASM_BLOCK 256

struct AsmParams
{
	long long n_tasks;
	const int32_t* task_slot; // global slot per task, -1: none
	int n_classes;
	long long job_base[DFB_ASM_MAX_CLASSES + 1]; // first global slot of every class (slots are numbered in job space)
	const int* slot_n[DFB_ASM_MAX_CLASSES];
	const uint2* slot_ev[DFB_ASM_MAX_CLASSES];
	const int* hitq[DFB_ASM_MAX_CLASSES];
	const JobPair* jobs[DFB_ASM_MAX_CLASSES];
	unsigned long long* block_sums; // [n_blocks][2] rows, cols; scanned in place into exclusive offsets
	unsigned long long* totals;     // [2]
	dfb_split_row* rows;
	int32_t* cols;
	Event* events; // overflow list (append)
	unsigned long long* ev_count;
	unsigned long long ev_cap;
	unsigned long long rows_cap, cols_cap; // entries allocated (bounds-check builds)
};

// the task's region entries ordered by key (matrix << 27 | row << 16 | column); returns their number, -1 for a task
// that has none to assemble here (no slot, or spilled)
__device__ __forceinline__ int asm_load(const AsmParams& p, long long t, uint2 (&e)[DFB_SLOT_EVENTS], int& L, int& cls, long long& local)
{
	const int32_t s = p.task_slot[t];
	if (s < 0) return -1;
	int c = 0;
	while (c + 1 < p.n_classes && (long long)s >= p.job_base[c + 1]) c++;
	cls = c;
	local = (long long)s - p.job_base[c];
	const int n = p.slot_n[c][local];
	if (n > DFB_SLOT_EVENTS) return -2;
	L = p.jobs[c][p.hitq[c][local]].L[0];
	const uint2* src = p.slot_ev[c] + local * DFB_SLOT_EVENTS;
	for (int k = 0; k < n; k++)
	{
		const uint2 v = src[k];
		int b = k - 1;
		while (b >= 0 && e[b].x > v.x)
		{
			e[b + 1] = e[b];
			b--;
		}
		e[b + 1] = v;
	}
	return n;
}

// walks the rows of one task; F(a, i, i_end, j, j_end) is called for every emitted row
template <class F>
__device__ __forceinline__ void asm_rows(const uint2 (&e)[DFB_SLOT_EVENTS], int n, int L, F emit)
{
	int n0 = 0;
	while (n0 < n && !(e[n0].x >> 27)) n0++;
	int i = 0;
	while (i < n0)
	{
		const uint32_t a = (e[i].x >> 16) & 0x7ff;
		int i_end = i + 1;
		while (i_end < n0 && ((e[i_end].x >> 16) & 0x7ff) == a) i_end++;
		const uint32_t want = (uint32_t)L - a;
		int j = n0;
		while (j < n && ((e[j].x >> 16) & 0x7ff) != want) j++;
		if (j < n)
		{
			int j_end = j + 1;
			while (j_end < n && ((e[j_end].x >> 16) & 0x7ff) == want) j_end++;
			emit((int)a, i, i_end, j, j_end);
		}
		i = i_end;
	}
}

__global__ void __launch_bounds__(DFB_ASM_BLOCK) asm_count_kernel(AsmParams p)
{
	__shared__ unsigned int s_rows, s_cols;
	if (threadIdx.x == 0) s_rows = s_cols = 0;
	__syncthreads();
	const long long t = (long long)blockIdx.x * DFB_ASM_BLOCK + threadIdx.x;
	unsigned nr = 0, nc = 0;
	if (t < p.n_tasks)
	{
		uint2 e[DFB_SLOT_EVENTS];
		int L = 0, cls = 0;
		long long local = 0;
		const int n = asm_load(p, t, e, L, cls, local);
		if (n == -2)
		{
			// spilled: hand the region's entries to the overflow list, the host assembles the task from that list alone
			const uint2* src = p.slot_ev[cls] + local * DFB_SLOT_EVENTS;
			for (int k = 0; k < DFB_SLOT_EVENTS; k++)
			{
				const unsigned long long idx = atomicAdd(p.ev_count, 1ull);
				if (idx < p.ev_cap)
				{
					const uint2 v = src[k];
					Event ev;
					ev.task = (int32_t)t;
					ev.half_row = (int32_t)(((v.x >> 27) << 30) | ((v.x >> 16) & 0x7ff));
					ev.col = (int32_t)(v.x & 0xffff);
					ev.score = (int32_t)v.y;
					p.events[idx] = ev;
				}
			}
		}
		else if (n > 0)
		{
			asm_rows(e, n, L, [&](int, int i, int i_end, int j, int j_end) {
				nr++;
				nc += (unsigned)((i_end - i) + (j_end - j));
			});
		}
	}
	// block sums (warp reduce, then one atomic per warp)
	for (int o = 16; o > 0; o >>= 1)
	{
		nr += __shfl_down_sync(0xffffffffu, nr, o);
		nc += __shfl_down_sync(0xffffffffu, nc, o);
	}
	if ((threadIdx.x & 31) == 0)
	{
		atomicAdd(&s_rows, nr);
		atomicAdd(&s_cols, nc);
	}
	__syncthreads();
	if (threadIdx.x == 0)
	{
		p.block_sums[2 * (size_t)blockIdx.x] = s_rows;
		p.block_sums[2 * (size_t)blockIdx.x + 1] = s_cols;
	}
}

// one block: exclusive scan of the per-block sums, in place
__global__ void __launch_bounds__(1024) asm_scan_kernel(unsigned long long* sums, long long n_blocks, unsigned long long* totals)
{
	__shared__ unsigned long long warp_r[32], warp_c[32];
	__shared__ unsigned long long carry_r, carry_c;
	if (threadIdx.x == 0) carry_r = carry_c = 0;
	__syncthreads();
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	for (long long base = 0; base < n_blocks; base += 1024)
	{
		const long long k = base + threadIdx.x;
		unsigned long long r = k < n_blocks ? sums[2 * k] : 0, c = k < n_blocks ? sums[2 * k + 1] : 0;
		const unsigned long long r0 = r, c0 = c;
		for (int o = 1; o < 32; o <<= 1)
		{
			const unsigned long long ur = __shfl_up_sync(0xffffffffu, r, o), uc = __shfl_up_sync(0xffffffffu, c, o);
			if (lane >= o)
			{
				r += ur;
				c += uc;
			}
		}
		if (lane == 31)
		{
			warp_r[warp] = r;
			warp_c[warp] = c;
		}
		__syncthreads();
		if (warp == 0)
		{
			unsigned long long wr = warp_r[lane], wc = warp_c[lane];
			for (int o = 1; o < 32; o <<= 1)
			{
				const unsigned long long ur = __shfl_up_sync(0xffffffffu, wr, o), uc = __shfl_up_sync(0xffffffffu, wc, o);
				if (lane >= o)
				{
					wr += ur;
					wc += uc;
				}
			}
			warp_r[lane] = wr; // inclusive over warps
			warp_c[lane] = wc;
		}
		__syncthreads();
		const unsigned long long before_r = carry_r + (warp ? warp_r[warp - 1] : 0), before_c = carry_c + (warp ? warp_c[warp - 1] : 0);
		if (k < n_blocks)
		{
			sums[2 * k] = before_r + r - r0;
			sums[2 * k + 1] = before_c + c - c0;
		}
		__syncthreads();
		if (threadIdx.x == 0)
		{
			carry_r += warp_r[31];
			carry_c += warp_c[31];
		}
		__syncthreads();
	}
	if (threadIdx.x == 0)
	{
		totals[0] = carry_r;
		totals[1] = carry_c;
	}
}

__global__ void __launch_bounds__(DFB_ASM_BLOCK) asm_write_kernel(AsmParams p)
{
	__shared__ unsigned int w_rows[DFB_ASM_BLOCK / 32], w_cols[DFB_ASM_BLOCK / 32];
	const long long t = (long long)blockIdx.x * DFB_ASM_BLOCK + threadIdx.x;
	uint2 e[DFB_SLOT_EVENTS];
	int L = 0, cls = 0, n = -1;
	long long local = 0;
	unsigned nr = 0, nc = 0;
	if (t < p.n_tasks)
	{
		n = asm_load(p, t, e, L, cls, local);
		if (n > 0)
			asm_rows(e, n, L, [&](int, int i, int i_end, int j, int j_end) {
				nr++;
				nc += (unsigned)((i_end - i) + (j_end - j));
			});
	}
	// exclusive offsets inside the block
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	unsigned ir = nr, ic = nc;
	for (int o = 1; o < 32; o <<= 1)
	{
		const unsigned ur = __shfl_up_sync(0xffffffffu, ir, o), uc = __shfl_up_sync(0xffffffffu, ic, o);
		if (lane >= o)
		{
			ir += ur;
			ic += uc;
		}
	}
	if (lane == 31)
	{
		w_rows[warp] = ir;
		w_cols[warp] = ic;
	}
	__syncthreads();
	unsigned long long row_at = p.block_sums[2 * (size_t)blockIdx.x] + (ir - nr);
	unsigned long long col_at = p.block_sums[2 * (size_t)blockIdx.x + 1] + (ic - nc);
	for (int w = 0; w < warp; w++)
	{
		row_at += w_rows[w];
		col_at += w_cols[w];
	}
	if (n > 0 && nr)
	{
		asm_rows(e, n, L, [&](int a, int i, int i_end, int j, int j_end) {
			dfb_split_row row;
			row.task = (int32_t)t;
			row.read_split = a;
			row.score1 = (int32_t)e[i].y;
			row.score2 = (int32_t)e[j].y;
			row.col_begin = (int64_t)col_at;
			row.n1 = i_end - i;
			row.n2 = j_end - j;
			DFB_BC(row_at < p.rows_cap && col_at + (unsigned)(row.n1 + row.n2) <= p.cols_cap, 501);
			p.rows[row_at++] = row;
			for (int k = i; k < i_end; k++) p.cols[col_at++] = (int32_t)(e[k].x & 0xffff);
			for (int k = j; k < j_end; k++) p.cols[col_at++] = (int32_t)(e[k].x & 0xffff);
		});
	}
}

// ---- overflow list assembled on the device (the device-resident entry points) ----------------------------------
// The same rows the host makes of the overflow list (emit_task_rows in dfb_api.cu), in the same order:
//   1. an LSD radix sort of the events, 8 bits per pass, stable: first over the (matrix, row, column) key, then over
//      the task -- ov_hist_kernel + a scan of the digit-major histogram + ov_scatter_kernel per pass.  Any number of
//      events per task and per batch; the passes needed follow from the longest read, window and the chunk's tasks.
//   2. groups = runs of equal (task, matrix, row): ov_head_kernel flags their first events, a scan numbers them.
//   3. ov_match_kernel pairs every matrix-1 group (row a) with the matrix-2 group of its task at row L - a (binary
//      search over the sorted groups); a matched pair is one dfb_split_row with n1 + n2 columns.  Two scans number the
//      rows and place their columns.
//   4. ov_rows_kernel / ov_cols_kernel write the rows and the columns (one thread per event: a row of 10^5 tied
//      columns is spread over the grid).
//   5. ov_place_kernel merges these rows with the region-assembled rows of the chunk by task (the two never share a
//      task) into the batch's row array, behind the chunks before it; columns: the region part first, then this part.
#define DFB_OV_BLOCK 256

struct OvKey
{
	int sub_passes; // passes over the (matrix, row, column) key; the task's passes follow
	int rb, cb;     // bits of a row and of a column
};

__device__ __forceinline__ unsigned ov_digit(const Event& e, int pass, const OvKey& k)
{
	if (pass < k.sub_passes)
	{
		const unsigned long long row = (unsigned)e.half_row & 0x3fffffffu, half = (unsigned)e.half_row >> 30;
		const unsigned long long sub = (half << (k.rb + k.cb)) | (row << k.cb) | (unsigned long long)(unsigned)e.col;
		return (unsigned)(sub >> (8 * pass)) & 0xffu;
	}
	return ((unsigned)e.task >> (8 * (pass - k.sub_passes))) & 0xffu;
}

// block b's count of digit d at hist[d * n_blocks + b]: the exclusive scan of that order is every element's first slot
__global__ void __launch_bounds__(DFB_OV_BLOCK) ov_hist_kernel(const Event* __restrict__ in, long long n, int pass, OvKey key,
                                                               unsigned long long* hist, long long n_blocks)
{
	__shared__ unsigned int s[256];
	s[threadIdx.x] = 0;
	__syncthreads();
	const long long i = (long long)blockIdx.x * DFB_OV_BLOCK + threadIdx.x;
	if (i < n) atomicAdd(&s[ov_digit(in[i], pass, key)], 1u);
	__syncthreads();
	hist[(size_t)threadIdx.x * n_blocks + blockIdx.x] = s[threadIdx.x];
}

__global__ void __launch_bounds__(DFB_OV_BLOCK) ov_scatter_kernel(const Event* __restrict__ in, Event* __restrict__ out, long long n, int pass,
                                                                  OvKey key, const unsigned long long* __restrict__ hist, long long n_blocks)
{
	__shared__ unsigned int s_wc[DFB_OV_BLOCK / 32][257]; // [warp][digit]: elements of the digit in the warp
	for (int k = threadIdx.x; k < (DFB_OV_BLOCK / 32) * 257; k += DFB_OV_BLOCK) (&s_wc[0][0])[k] = 0;
	__syncthreads();
	const long long i = (long long)blockIdx.x * DFB_OV_BLOCK + threadIdx.x;
	Event e;
	unsigned d = 256; // (past the end: a digit of its own)
	if (i < n)
	{
		e = in[i];
		d = ov_digit(e, pass, key);
	}
	const unsigned peers = __match_any_sync(0xffffffffu, d);
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	if (lane == __ffs(peers) - 1) s_wc[warp][d] = (unsigned)__popc(peers);
	__syncthreads();
	if (i < n)
	{
		unsigned long long at = hist[(size_t)d * n_blocks + blockIdx.x] + (unsigned)__popc(peers & ((1u << lane) - 1u));
		for (int w = 0; w < warp; w++) at += s_wc[w][d];
		out[at] = e;
	}
}

__device__ __forceinline__ unsigned long long ov_group_key(const Event& e)
{
	return ((unsigned long long)(unsigned)e.task << 32) | (unsigned)e.half_row;
}

struct OvAsmParams
{
	const Event* ev;            // sorted
	long long n;                // events
	unsigned long long* head;   // [n]: 1 at the first event of a group -> scanned: groups before
	unsigned long long* scal;   // [0] groups, [1] rows, [2] columns (scan totals)
	long long* g_first;         // [n + 1] first event of every group, then n
	int32_t* g_match;           // [n] matrix-2 group paired with a matrix-1 group, -1
	int32_t* g_matched_by;      // [n] the reverse, -1
	unsigned long long* g_rows; // [n] 1 for a paired matrix-1 group -> scanned: its row
	unsigned long long* g_cols; // [n] n1 + n2 -> scanned: its first column
	// read length of chunk task t: read_off[r + 1] - read_off[r], r = task_read[task_base + t]
	const int64_t* read_off;
	const int32_t* task_read;
	long long task_base;
	dfb_split_row* x_rows;      // the rows, in order; col_begin relative to the chunk's columns
	long long asm_cols;         // columns of the region assembly of the chunk (in front of these)
	int32_t* cols;              // the batch's column array
	const unsigned long long* base; // [0] rows, [1] columns of the batch before this chunk
};

__device__ __forceinline__ bool ov_is_head(const Event* ev, long long i)
{
	return i == 0 || ov_group_key(ev[i]) != ov_group_key(ev[i - 1]);
}

__global__ void __launch_bounds__(DFB_OV_BLOCK) ov_head_kernel(OvAsmParams p)
{
	const long long i = (long long)blockIdx.x * DFB_OV_BLOCK + threadIdx.x;
	if (i < p.n) p.head[i] = ov_is_head(p.ev, i) ? 1ull : 0ull;
}

__global__ void __launch_bounds__(DFB_OV_BLOCK) ov_group_kernel(OvAsmParams p)
{
	const long long i = (long long)blockIdx.x * DFB_OV_BLOCK + threadIdx.x;
	if (i >= p.n) return;
	if (ov_is_head(p.ev, i)) p.g_first[p.head[i]] = i;
	if (i == 0) p.g_first[p.scal[0]] = p.n;
}

__global__ void __launch_bounds__(DFB_OV_BLOCK) ov_match_kernel(OvAsmParams p)
{
	const long long g = (long long)blockIdx.x * DFB_OV_BLOCK + threadIdx.x;
	if (g >= p.n) return;
	const long long n_groups = (long long)p.scal[0];
	unsigned long long rows = 0, cols = 0;
	int32_t match = -1;
	if (g < n_groups)
	{
		const Event e = p.ev[p.g_first[g]];
		if (((unsigned)e.half_row >> 30) == 0)
		{
			const long long r = p.task_read[p.task_base + e.task];
			const long long want = (p.read_off[r + 1] - p.read_off[r]) - (long long)(e.half_row & 0x3fffffff);
			if (want >= 0 && want <= 0x3fffffff)
			{
				const unsigned long long k = ((unsigned long long)(unsigned)e.task << 32) | (1u << 30) | (unsigned)want;
				long long lo = g + 1, hi = n_groups; // (matrix 2 sorts behind matrix 1 in the task)
				while (lo < hi)
				{
					const long long mid = (lo + hi) >> 1;
					if (ov_group_key(p.ev[p.g_first[mid]]) < k) lo = mid + 1;
					else hi = mid;
				}
				if (lo < n_groups && ov_group_key(p.ev[p.g_first[lo]]) == k)
				{
					match = (int32_t)lo;
					p.g_matched_by[lo] = (int32_t)g;
					rows = 1;
					cols = (unsigned long long)(p.g_first[g + 1] - p.g_first[g] + p.g_first[lo + 1] - p.g_first[lo]);
				}
			}
		}
	}
	p.g_match[g] = match;
	p.g_rows[g] = rows;
	p.g_cols[g] = cols;
}

__global__ void __launch_bounds__(DFB_OV_BLOCK) ov_rows_kernel(OvAsmParams p)
{
	const long long g = (long long)blockIdx.x * DFB_OV_BLOCK + threadIdx.x;
	if (g >= p.n || g >= (long long)p.scal[0]) return;
	const int32_t j = p.g_match[g];
	if (j < 0) return;
	const Event e1 = p.ev[p.g_first[g]], e2 = p.ev[p.g_first[j]];
	dfb_split_row row;
	row.task = e1.task;
	row.read_split = e1.half_row & 0x3fffffff;
	row.score1 = e1.score;
	row.score2 = e2.score;
	row.col_begin = p.asm_cols + (long long)p.g_cols[g];
	row.n1 = (int32_t)(p.g_first[g + 1] - p.g_first[g]);
	row.n2 = (int32_t)(p.g_first[j + 1] - p.g_first[j]);
	p.x_rows[p.g_rows[g]] = row;
}

__global__ void __launch_bounds__(DFB_OV_BLOCK) ov_cols_kernel(OvAsmParams p)
{
	const long long i = (long long)blockIdx.x * DFB_OV_BLOCK + threadIdx.x;
	if (i >= p.n) return;
	const long long g = (long long)p.head[i] + (ov_is_head(p.ev, i) ? 1 : 0) - 1;
	long long at;
	if (p.g_match[g] >= 0) at = (long long)p.g_cols[g] + (i - p.g_first[g]);
	else if (p.g_matched_by[g] >= 0)
	{
		const long long g1 = p.g_matched_by[g];
		at = (long long)p.g_cols[g1] + (p.g_first[g1 + 1] - p.g_first[g1]) + (i - p.g_first[g]);
	}
	else return;
	p.cols[(long long)p.base[1] + p.asm_cols + at] = p.ev[i].col;
}

// items [0, n_asm): region rows; [n_asm, n_asm + n_x_bound): overflow rows (as many as scal[1]); then the region columns
__global__ void __launch_bounds__(DFB_OV_BLOCK) ov_place_kernel(const dfb_split_row* __restrict__ asm_rows, long long n_asm,
                                                                const int32_t* __restrict__ asm_cols, long long n_asm_cols,
                                                                const dfb_split_row* __restrict__ x_rows, long long n_x_bound,
                                                                const unsigned long long* __restrict__ scal, int32_t task_shift,
                                                                const unsigned long long* __restrict__ base, dfb_split_row* out_rows,
                                                                int32_t* out_cols)
{
	const long long i = (long long)blockIdx.x * DFB_OV_BLOCK + threadIdx.x;
	const long long n_x = scal ? (long long)scal[1] : 0;
	auto below = [](const dfb_split_row* r, long long n, int32_t task) { // rows with a smaller task
		long long lo = 0, hi = n;
		while (lo < hi)
		{
			const long long mid = (lo + hi) >> 1;
			if (r[mid].task < task) lo = mid + 1;
			else hi = mid;
		}
		return lo;
	};
	dfb_split_row row;
	long long at;
	if (i < n_asm)
	{
		row = asm_rows[i];
		at = i + below(x_rows, n_x, row.task);
	}
	else if (i < n_asm + n_x_bound)
	{
		const long long q = i - n_asm;
		if (q >= n_x) return;
		row = x_rows[q];
		at = q + below(asm_rows, n_asm, row.task);
	}
	else
	{
		const long long c = i - n_asm - n_x_bound;
		if (c < n_asm_cols) out_cols[(long long)base[1] + c] = asm_cols[c];
		return;
	}
	row.task += task_shift;
	row.col_begin += (long long)base[1];
	out_rows[(long long)base[0] + at] = row;
}

// the batch's totals behind the chunk
__global__ void ov_advance_kernel(unsigned long long* base, long long n_asm, long long n_asm_cols, const unsigned long long* scal)
{
	base[0] += (unsigned long long)n_asm + (scal ? scal[1] : 0ull);
	base[1] += (unsigned long long)n_asm_cols + (scal ? scal[2] : 0ull);
}
}  // namespace dfb
