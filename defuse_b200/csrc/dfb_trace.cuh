// Backtrace of chosen split alignments: SplitReadAligner::GetAlignments(..., backtrace=true)
// (tools/SplitReadAligner.cpp:56-69 pointer rule, :124-143 BackTracePath, :145-154 ReverseMatches, :287-292).
//
// Included at the end of dfb_api.cu (it needs dfb_ctx).  The workload is small by construction -- splitseq
// re-aligns only the reads that support one predicted break (tools/splitseq.cpp:100-125) -- so this path is
// built for exactness over every parameter set (s32 arithmetic, raw byte equality, any length), not for TCUPS:
//
//   trace_fill_kernel   one warp per matrix (a task has two: read x ref1, rev(read) x rev(ref2)).  Lane l owns
//                       read row j = tile + l + 1 and sweeps the reference as a skewed wavefront, exactly the
//                       geometry of the s32 DP kernel; what is new is the pointer of every cell, 2 bits, packed
//                       16 columns per word by the lane that owns the row:
//                         0 diagonal, 1 (i-1,j), 2 (i,j-1); later writers win, so 2 > 1 > 0 (:56-69)
//   trace_walk_kernel   one thread per matrix walks the pointers from the start cell until j == 0 and records
//                       the diagonal steps in walk order (descending positions).
// The host reverses matrix 1's list and maps matrix 2's coordinates back to the unreversed sequences (whose
// double reversal is the walk order itself).
#pragma once

namespace dfb
{
struct TraceJob
{
	long long ref_off;  // first byte of the reference in the raw pool
	long long read_off; // first byte of the read in the raw pool
	int R, L;
	int reversed;       // 1: both sequences are consumed back to front (matrix 2)
	int start_i, start_j;
	long long bits_off;    // words; (L+1) rows of W = (R+16)/16 words
	long long scratch_off; // ints; R+1 row-boundary values
	long long match_off;   // pairs; capacity L
};

__device__ __forceinline__ int trace_ref_byte(const unsigned char* raw, const TraceJob& jb, int i) // i = 1..R
{
	return raw[jb.ref_off + (jb.reversed ? jb.R - i : i - 1)];
}
__device__ __forceinline__ int trace_read_byte(const unsigned char* raw, const TraceJob& jb, int j) // j = 1..L
{
	return raw[jb.read_off + (jb.reversed ? jb.L - j : j - 1)];
}

__global__ void __launch_bounds__(128) trace_fill_kernel(const unsigned char* __restrict__ raw, const TraceJob* __restrict__ jobs,
                                                         int n_jobs, int match, int mismatch, int gap, int end_gaps,
                                                         unsigned* __restrict__ bits, int* __restrict__ scratch)
{
	const int lane = threadIdx.x & 31;
	const int warps = (gridDim.x * blockDim.x) >> 5;
	for (int job = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; job < n_jobs; job += warps)
	{
		const TraceJob jb = jobs[job];
		const int R = jb.R, L = jb.L;
		const int W = (R + 16) >> 4;
		unsigned* const my_bits = bits + jb.bits_off;
		int* const edge = scratch + jb.scratch_off;
		const int row0 = end_gaps ? 0 : gap; // H(0,j) = j * row0 (:44-48)
		for (int tile = 0; tile < L; tile += 32)
		{
			const int j = tile + lane + 1;
			const bool live = j <= L;
			const int rc = live ? trace_read_byte(raw, jb, j) : -1;
			int own = j * row0;        // H(i-1, j), starts at column 0
			int diag = (j - 1) * row0; // H(i-1, j-1)
			int cur = 0;               // H(i, j) just computed: what the lane below sees as H(i, j-1)
			unsigned word = 0;
			unsigned* const row_bits = my_bits + (long long)j * W;
			const bool last_lane = lane == 31 && tile + 32 < L;
			for (int s = 1; s <= R + 31; s++)
			{
				const int i = s - lane;
				int above = __shfl_up_sync(0xffffffffu, cur, 1);
				if (live && i >= 1 && i <= R)
				{
					if (lane == 0) above = tile == 0 ? 0 : edge[i]; // H(i, tile): row 0 is all zero (:40-43)
					const int m = diag + (trace_ref_byte(raw, jb, i) == rc ? match : mismatch);
					const int gr = own + gap;   // from (i-1, j)
					const int gd = above + gap; // from (i, j-1)
					const int mx = max(m, max(gr, gd));
					const unsigned dir = gd == mx ? 2u : (gr == mx ? 1u : 0u);
					word |= dir << (2 * (i & 15));
					if ((i & 15) == 15 || i == R)
					{
						row_bits[i >> 4] = word;
						word = 0;
					}
					diag = above;
					own = mx;
					cur = mx;
					if (last_lane) edge[i] = mx;
				}
			}
			__syncwarp();
		}
	}
}

__global__ void trace_walk_kernel(const TraceJob* __restrict__ jobs, int n_jobs, const unsigned* __restrict__ bits,
                                  int2* __restrict__ matches, int* __restrict__ n_matches)
{
	const int job = blockIdx.x * blockDim.x + threadIdx.x;
	if (job >= n_jobs) return;
	const TraceJob jb = jobs[job];
	const int W = (jb.R + 16) >> 4;
	const unsigned* const my_bits = bits + jb.bits_off;
	int2* out = matches + jb.match_off;
	int i = jb.start_i, j = jb.start_j, n = 0;
	while (j > 0)
	{
		// row i == 0 points along the read (:46-47)
		const unsigned dir = i == 0 ? 2u : (my_bits[(long long)j * W + (i >> 4)] >> (2 * (i & 15))) & 3u;
		if (dir == 0)
		{
			out[n++] = make_int2(i - 1, j - 1); // (refPos, readPos) of a diagonal step (:133-139)
			i--;
			j--;
		}
		else if (dir == 1)
			i--;
		else
			j--;
	}
	n_matches[job] = n;
}
}  // namespace dfb

// ------------------------------------------------------------------------------------------
// host entry
// ------------------------------------------------------------------------------------------

extern "C" int dfb_split_backtrace_batch(dfb_ctx* ctx, const dfb_split_params* params, const dfb_seq_table* refs,
                                         const dfb_seq_table* reads, const int32_t* task_cluster, const int32_t* task_read,
                                         const int32_t* task_ref_split1, const int32_t* task_ref_split2,
                                         const int32_t* task_read_split, int64_t n_tasks, int64_t* match_off,
                                         int32_t* matches, int64_t matches_cap, int64_t* n_pairs_out)
{
	if (!ctx) return DFB_ERR_ARG;
	if (!params || n_tasks < 0 || !match_off || !n_pairs_out ||
	    (n_tasks > 0 && (!task_cluster || !task_read || !task_ref_split1 || !task_ref_split2 || !task_read_split)))
		return set_err(ctx, DFB_ERR_ARG, "dfb_split_backtrace_batch: null argument");
	int rc = check_table(ctx, refs, "refs");
	if (rc) return rc;
	rc = check_table(ctx, reads, "reads");
	if (rc) return rc;
	if (refs->n % 2) return set_err(ctx, DFB_ERR_ARG, "refs must hold two windows per cluster");
	CK(ctx, cudaSetDevice(ctx->device));

	// validate and size: the start cells of task t are (i1, a) in matrix 1 and (R2 - refSplit2 - 1, L - a) in matrix 2
	match_off[0] = 0;
	for (int64_t t = 0; t < n_tasks; t++)
	{
		const int64_t c = task_cluster[t], r = task_read[t];
		if (c < 0 || 2 * c + 1 >= refs->n || r < 0 || r >= reads->n)
			return set_err(ctx, DFB_ERR_ARG, "task %lld: index out of range", (long long)t);
		const int64_t R1 = refs->off[2 * c + 1] - refs->off[2 * c], R2 = refs->off[2 * c + 2] - refs->off[2 * c + 1];
		const int64_t L = reads->off[r + 1] - reads->off[r];
		const int64_t a = task_read_split[t], i1 = task_ref_split1[t], i2 = R2 - (int64_t)task_ref_split2[t] - 1;
		if (a < 0 || a > L || i1 < 0 || i1 > R1 || i2 < 0 || i2 > R2)
			return set_err(ctx, DFB_ERR_ARG, "task %lld: start cell outside the matrices", (long long)t);
		match_off[2 * t + 1] = match_off[2 * t] + a;       // a diagonal step consumes one read base
		match_off[2 * t + 2] = match_off[2 * t + 1] + (L - a);
	}
	// (match_off holds capacities for now; it is compacted to the real counts below)
	const int64_t cap_pairs = match_off[2 * n_tasks];
	std::vector<int64_t> cap_off(match_off, match_off + 2 * n_tasks + 1);

	// chunks bounded by pointer-matrix memory
	const size_t kMaxBitsWords = (size_t)1 << 28; // 1 GiB of pointer words per chunk
	std::vector<TraceJob> jobs;
	std::vector<int2> h_pairs;
	std::vector<int> h_cnt;
	std::vector<int64_t> counts((size_t)(2 * n_tasks), 0);
	std::vector<int2> all_pairs((size_t)cap_pairs);
	const int64_t raw_ref = refs->off[refs->n], raw_read = reads->off[reads->n];
	unsigned char* d_raw = nullptr;
	cudaStream_t st = ctx->stream;
	CK(ctx, cudaMallocAsync((void**)&d_raw, (size_t)(raw_ref + raw_read + 16), st));
	auto fail = [&](int code) {
		cudaStreamSynchronize(st);
		cudaFreeAsync(d_raw, st);
		return code;
	};
	cudaError_t e = cudaSuccess;
	if (raw_ref) e = cudaMemcpyAsync(d_raw, refs->bytes, (size_t)raw_ref, cudaMemcpyHostToDevice, st);
	if (e == cudaSuccess && raw_read) e = cudaMemcpyAsync(d_raw + raw_ref, reads->bytes, (size_t)raw_read, cudaMemcpyHostToDevice, st);
	if (e != cudaSuccess) return fail(set_err(ctx, DFB_ERR_CUDA, "upload failed: %s", cudaGetErrorString(e)));

	for (int64_t first = 0; first < n_tasks;)
	{
		jobs.clear();
		size_t words = 0, scratch = 0, pairs = 0;
		int64_t last = first;
		for (; last < n_tasks; last++)
		{
			const int64_t c = task_cluster[last], r = task_read[last];
			const int64_t R1 = refs->off[2 * c + 1] - refs->off[2 * c], R2 = refs->off[2 * c + 2] - refs->off[2 * c + 1];
			const int64_t L = reads->off[r + 1] - reads->off[r];
			const size_t w1 = (size_t)(L + 1) * (size_t)((R1 + 16) >> 4), w2 = (size_t)(L + 1) * (size_t)((R2 + 16) >> 4);
			if (!jobs.empty() && words + w1 + w2 > kMaxBitsWords) break;
			const int a = task_read_split[last];
			TraceJob j1{refs->off[2 * c], raw_ref + reads->off[r], (int)R1, (int)L, 0, task_ref_split1[last], a,
			            (long long)words, (long long)scratch, (long long)pairs};
			words += w1;
			scratch += (size_t)R1 + 1;
			pairs += (size_t)a;
			TraceJob j2{refs->off[2 * c + 1], raw_ref + reads->off[r], (int)R2, (int)L, 1,
			            (int)(R2 - task_ref_split2[last] - 1), (int)(L - a), (long long)words, (long long)scratch, (long long)pairs};
			words += w2;
			scratch += (size_t)R2 + 1;
			pairs += (size_t)(L - a);
			jobs.push_back(j1);
			jobs.push_back(j2);
		}
		const int n_jobs = (int)jobs.size();
		TraceJob* d_jobs = nullptr;
		unsigned* d_bits = nullptr;
		int* d_scratch = nullptr;
		int2* d_pairs = nullptr;
		int* d_cnt = nullptr;
		if ((e = cudaMallocAsync((void**)&d_jobs, sizeof(TraceJob) * (size_t)n_jobs, st)) != cudaSuccess ||
		    (e = cudaMallocAsync((void**)&d_bits, sizeof(unsigned) * (words + 1), st)) != cudaSuccess ||
		    (e = cudaMallocAsync((void**)&d_scratch, sizeof(int) * (scratch + 1), st)) != cudaSuccess ||
		    (e = cudaMallocAsync((void**)&d_pairs, sizeof(int2) * (pairs + 1), st)) != cudaSuccess ||
		    (e = cudaMallocAsync((void**)&d_cnt, sizeof(int) * (size_t)n_jobs, st)) != cudaSuccess)
		{
			// (blocks already taken go back to the pool with the stream)
			if (d_jobs) cudaFreeAsync(d_jobs, st);
			if (d_bits) cudaFreeAsync(d_bits, st);
			if (d_scratch) cudaFreeAsync(d_scratch, st);
			if (d_pairs) cudaFreeAsync(d_pairs, st);
			return fail(set_err(ctx, DFB_ERR_NOMEM, "device allocation failed: %s", cudaGetErrorString(e)));
		}
		h_pairs.resize(pairs + 1);
		h_cnt.resize((size_t)n_jobs);
		e = cudaMemcpyAsync(d_jobs, jobs.data(), sizeof(TraceJob) * (size_t)n_jobs, cudaMemcpyHostToDevice, st);
		if (e == cudaSuccess)
		{
			const int warps_per_block = 4;
			const int grid = std::max(1, std::min((n_jobs + warps_per_block - 1) / warps_per_block, ctx->prop.multiProcessorCount * 8));
			trace_fill_kernel<<<grid, 32 * warps_per_block, 0, st>>>(d_raw, d_jobs, n_jobs, params->match, params->mismatch,
			                                                         params->gap, params->end_gaps, d_bits, d_scratch);
			trace_walk_kernel<<<(n_jobs + 63) / 64, 64, 0, st>>>(d_jobs, n_jobs, d_bits, d_pairs, d_cnt);
			e = cudaGetLastError();
		}
		if (e == cudaSuccess) e = cudaMemcpyAsync(h_pairs.data(), d_pairs, sizeof(int2) * pairs, cudaMemcpyDeviceToHost, st);
		if (e == cudaSuccess) e = cudaMemcpyAsync(h_cnt.data(), d_cnt, sizeof(int) * (size_t)n_jobs, cudaMemcpyDeviceToHost, st);
		if (e == cudaSuccess) e = cudaStreamSynchronize(st);
		cudaFreeAsync(d_jobs, st);
		cudaFreeAsync(d_bits, st);
		cudaFreeAsync(d_scratch, st);
		cudaFreeAsync(d_pairs, st);
		cudaFreeAsync(d_cnt, st);
		if (e != cudaSuccess) return fail(set_err(ctx, DFB_ERR_CUDA, "backtrace kernels failed: %s", cudaGetErrorString(e)));
		for (int k = 0; k < n_jobs; k++)
		{
			const int64_t t = first + k / 2;
			const int half = k & 1;
			const TraceJob& jb = jobs[(size_t)k];
			const int n = h_cnt[(size_t)k];
			counts[(size_t)(2 * t + half)] = n;
			int2* dst = all_pairs.data() + cap_off[(size_t)(2 * t + half)];
			const int2* src = h_pairs.data() + jb.match_off;
			if (!half)
				for (int q = 0; q < n; q++) dst[q] = src[n - 1 - q]; // BackTracePath's reverse (:142)
			else
				for (int q = 0; q < n; q++) dst[q] = make_int2(jb.R - src[q].x - 1, jb.L - src[q].y - 1); // ReverseMatches (:145-154)
		}
		first = last;
	}
	cudaFreeAsync(d_raw, st);

	// compact: real counts instead of capacities
	int64_t total = 0;
	for (int64_t k = 0; k < 2 * n_tasks; k++)
	{
		match_off[k] = total;
		total += counts[(size_t)k];
	}
	match_off[2 * n_tasks] = total;
	*n_pairs_out = total;
	if (matches)
	{
		if (matches_cap < total) return set_err(ctx, DFB_ERR_ARG, "matches buffer holds %lld pairs, %lld needed", (long long)matches_cap, (long long)total);
		for (int64_t k = 0; k < 2 * n_tasks; k++)
		{
			const int2* src = all_pairs.data() + cap_off[(size_t)k];
			int32_t* dst = matches + 2 * match_off[k];
			for (int64_t q = 0; q < counts[(size_t)k]; q++)
			{
				dst[2 * q] = src[q].x;
				dst[2 * q + 1] = src[q].y;
			}
		}
	}
	return DFB_OK;
}

// ------------------------------------------------------------------------------------------
// device-resident form: dfb_split_backtrace_device
// ------------------------------------------------------------------------------------------
//
// Record k names one alignment of task t = records[k].task: start cell (ref_split1, read_split1) in matrix 1 and
// (len(ref2) - ref_split2 - 1, len(read) - read_split1) in matrix 2.  Cell (i, j) depends only on cells up and to the
// left, so the pointers every record of a group of same-task records needs are those of the bounding box of its start
// cells -- rows 0..max j, columns 0..max i of each matrix -- filled with trace_fill_kernel's arithmetic and pointer rule.
//
//   bt_records_kernel   per record: argument checks, piece heads, capacity len(read)
//   bt_pieces_kernel    per record: the first record of each piece
//   bt_box_kernel       per piece: the two boxes, their footprint, the piece's wave
//   bt_fill_walk_kernel per piece: warp 0 fills matrix 1's box, warp 1 matrix 2's, then every thread walks records
//                       of the piece from their start cells into capacity slots (matrix 1 reversed into place, matrix 2
//                       mapped back to the unreversed sequences); templated on where the pointer bits live
//   bt_compact_kernel   per (record, matrix): the walked pairs of a wave, compacted by the scan of their counts
//
// A piece is a run of consecutive records of one task, also cut where k is a multiple of the run cap, so that one
// heavy task (poly-A: 467 k records) spreads over many blocks; each piece fills its boxes once.
#define DFB_BT_THREADS 128
#define DFB_BT_RUN_CAP 256                      // records per piece at most (DESIGN.md 4.5b: the measurement)
#define DFB_BT_SMEM_BYTES (96 << 10)            // pieces whose boxes fit take the shared-memory kernel
#define DFB_BT_WAVE_PAIRS (1ull << 27)          // capacity slots per wave: 1 GiB of int2 ...
#define DFB_BT_ARENA_BYTES ((size_t)256 << 20)  // ... plus the global arena of the pieces too large for shared memory

namespace dfb
{
enum BtBad
{
	BT_BAD_TASK,   // task outside [0, n_tasks)
	BT_BAD_CELL,   // a start cell outside its matrix
	BT_BAD_SPLIT2, // read_split2 != len(read) - read_split1
};

struct BtCheck
{
	DeviceCheck dc;                      // the tables and task arrays, as for dfb_split_align_device
	unsigned long long bad;              // min over bad records of 4 * record + BtBad (~0: none)
	unsigned long long n_pieces, cap_total;
	unsigned long long smem_words, glob_words; // largest footprint (32-bit words) of a piece on each path
	unsigned long long n_glob;           // pieces on the global-arena path
	unsigned long long wave_pairs;       // pairs walked in the current wave (its count scan)
};

struct BtTables
{
	const unsigned char* ref_bytes;
	const unsigned char* read_bytes;
	const int64_t* ref_off;
	const int64_t* read_off;
	const int32_t* task_cluster;
	const int32_t* task_read;
	long long n_clusters, n_reads, n_tasks;
};

struct BtPiece
{
	long long k0, k1;        // records [k0, k1)
	long long ref1, ref2, read; // first bytes of the sequences
	int L, R2;
	int I1, J1, I2, J2;      // boxes: columns 0..I, rows 0..J
	int glob;                // 1: the boxes live in a global arena slot
};

struct BtWave
{
	unsigned long long p_lo, p_hi, k_lo, k_hi, c_lo, c_hi; // pieces, records, capacity slots
};

__device__ __forceinline__ long long bt_words(int I, int J) { return (long long)J * ((I + 16) >> 4); } // rows 1..J of a box

// footprint of a piece: both boxes' pointer words, then both tile-edge rows
__device__ __forceinline__ unsigned long long bt_footprint(const BtPiece& pc)
{
	return (unsigned long long)(bt_words(pc.I1, pc.J1) + bt_words(pc.I2, pc.J2) + (pc.I1 + 1) + (pc.I2 + 1));
}

__global__ void bt_check_init_kernel(BtCheck* c)
{
	c->bad = ~0ull;
	c->n_pieces = c->cap_total = c->smem_words = c->glob_words = c->n_glob = c->wave_pairs = 0;
}

__global__ void bt_wave_init_kernel(BtWave* waves, long long n_waves)
{
	const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
	if (k < n_waves) waves[k] = BtWave{~0ull, 0ull, ~0ull, 0ull, ~0ull, 0ull};
}

__device__ __forceinline__ bool bt_head(const dfb_split_record* rec, long long k, int cap)
{
	return k == 0 || k % cap == 0 || rec[k].task != rec[k - 1].task;
}

__global__ void __launch_bounds__(DFB_BUILD_BLOCK) bt_records_kernel(const dfb_split_record* __restrict__ rec, long long n, BtTables t, int cap,
                                                                      BtCheck* chk, unsigned long long* head, unsigned long long* capv)
{
	const long long stride = (long long)gridDim.x * DFB_BUILD_BLOCK;
	for (long long k = (long long)blockIdx.x * DFB_BUILD_BLOCK + threadIdx.x; k < n; k += stride)
	{
		const dfb_split_record r = rec[k];
		int bad = -1;
		long long L = 0;
		if (r.task < 0 || r.task >= t.n_tasks) bad = BT_BAD_TASK;
		else
		{
			const long long c = t.task_cluster[r.task], q = t.task_read[r.task];
			if (c >= 0 && c < t.n_clusters && q >= 0 && q < t.n_reads) // (else the task check reports it)
			{
				L = t.read_off[q + 1] - t.read_off[q];
				const long long R1 = t.ref_off[2 * c + 1] - t.ref_off[2 * c], R2 = t.ref_off[2 * c + 2] - t.ref_off[2 * c + 1];
				const long long a = r.read_split1, i1 = r.ref_split1, i2 = R2 - (long long)r.ref_split2 - 1;
				if (a < 0 || a > L || i1 < 0 || i1 > R1 || i2 < 0 || i2 > R2) bad = BT_BAD_CELL;
				else if ((long long)r.read_split2 != L - a) bad = BT_BAD_SPLIT2;
			}
			else L = -1;
		}
		if (bad >= 0) atomicMin(&chk->bad, 4ull * (unsigned long long)k + (unsigned long long)bad);
		head[k] = bt_head(rec, k, cap) ? 1ull : 0ull;
		capv[k] = bad < 0 && L > 0 ? (unsigned long long)L : 0ull;
	}
}

// head: the exclusive scan of the head flags (the piece of each head)
__global__ void __launch_bounds__(DFB_BUILD_BLOCK) bt_pieces_kernel(const dfb_split_record* __restrict__ rec, long long n, int cap,
                                                                     const unsigned long long* __restrict__ head, long long* piece_start)
{
	const long long stride = (long long)gridDim.x * DFB_BUILD_BLOCK;
	for (long long k = (long long)blockIdx.x * DFB_BUILD_BLOCK + threadIdx.x; k < n; k += stride)
		if (bt_head(rec, k, cap)) piece_start[head[k]] = k;
}

__global__ void __launch_bounds__(DFB_BUILD_BLOCK) bt_box_kernel(const dfb_split_record* __restrict__ rec, long long n, BtTables t,
                                                                  const long long* __restrict__ piece_start, long long n_pieces,
                                                                  const unsigned long long* __restrict__ cap_off, BtCheck* chk,
                                                                  BtPiece* pieces, BtWave* waves)
{
	const long long stride = (long long)gridDim.x * DFB_BUILD_BLOCK;
	for (long long p = (long long)blockIdx.x * DFB_BUILD_BLOCK + threadIdx.x; p < n_pieces; p += stride)
	{
		BtPiece pc;
		pc.k0 = piece_start[p];
		pc.k1 = p + 1 < n_pieces ? piece_start[p + 1] : n;
		const int task = rec[pc.k0].task;
		const long long c = t.task_cluster[task], q = t.task_read[task];
		pc.ref1 = t.ref_off[2 * c];
		pc.ref2 = t.ref_off[2 * c + 1];
		pc.read = t.read_off[q];
		pc.L = (int)(t.read_off[q + 1] - pc.read);
		pc.R2 = (int)(t.ref_off[2 * c + 2] - pc.ref2);
		pc.I1 = pc.J1 = pc.I2 = pc.J2 = 0;
		for (long long k = pc.k0; k < pc.k1; k++)
		{
			const dfb_split_record r = rec[k];
			pc.I1 = max(pc.I1, r.ref_split1);
			pc.J1 = max(pc.J1, r.read_split1);
			pc.I2 = max(pc.I2, pc.R2 - r.ref_split2 - 1);
			pc.J2 = max(pc.J2, pc.L - r.read_split1);
		}
		const unsigned long long words = bt_footprint(pc);
		pc.glob = words * 4 > DFB_BT_SMEM_BYTES;
		pieces[p] = pc;
		atomicMax(pc.glob ? &chk->glob_words : &chk->smem_words, words);
		if (pc.glob) atomicAdd(&chk->n_glob, 1ull);
		// the wave of a piece: where its capacity slots start, in units of the wave budget (waves are contiguous)
		const unsigned long long c0 = cap_off[pc.k0], c1 = pc.k1 < n ? cap_off[pc.k1] : chk->cap_total;
		BtWave* w = waves + c0 / DFB_BT_WAVE_PAIRS;
		atomicMin(&w->p_lo, (unsigned long long)p);
		atomicMax(&w->p_hi, (unsigned long long)p + 1);
		atomicMin(&w->k_lo, (unsigned long long)pc.k0);
		atomicMax(&w->k_hi, (unsigned long long)pc.k1);
		atomicMin(&w->c_lo, c0);
		atomicMax(&w->c_hi, c1);
	}
}

// H over rows 1..J (read) and columns 1..I (reference) of one matrix, by one warp: trace_fill_kernel's wavefront, s32
// arithmetic and pointer rule on the top-left corner of the matrix; the pointer of (i, j) goes to bits[(j - 1) W + i / 16]
__device__ __forceinline__ void bt_fill(const unsigned char* __restrict__ ref, const unsigned char* __restrict__ read, int R, int L,
                                        bool reversed, int I, int J, unsigned* bits, int* edge, int match, int mismatch, int gap, int row0)
{
	const int lane = threadIdx.x & 31;
	const int W = (I + 16) >> 4;
	for (int tile = 0; tile < J; tile += 32)
	{
		const int j = tile + lane + 1;
		const bool live = j <= J;
		const int rc = live ? read[reversed ? L - j : j - 1] : -1;
		int own = j * row0;        // H(i-1, j), starts at column 0
		int diag = (j - 1) * row0; // H(i-1, j-1)
		int cur = 0;
		unsigned word = 0;
		unsigned* const row_bits = bits + (long long)(j - 1) * W;
		const bool last_lane = lane == 31 && tile + 32 < J;
		for (int s = 1; s <= I + 31; s++)
		{
			const int i = s - lane;
			int above = __shfl_up_sync(0xffffffffu, cur, 1);
			if (live && i >= 1 && i <= I)
			{
				if (lane == 0) above = tile == 0 ? 0 : edge[i]; // H(i, tile): row 0 is all zero
				const int m = diag + (ref[reversed ? R - i : i - 1] == rc ? match : mismatch);
				const int gr = own + gap;
				const int gd = above + gap;
				const int mx = max(m, max(gr, gd));
				const unsigned dir = gd == mx ? 2u : (gr == mx ? 1u : 0u);
				word |= dir << (2 * (i & 15));
				if ((i & 15) == 15 || i == I)
				{
					row_bits[i >> 4] = word;
					word = 0;
				}
				diag = above;
				own = mx;
				cur = mx;
				if (last_lane) edge[i] = mx;
			}
		}
		__syncwarp();
	}
}

struct BtWalk
{
	const dfb_split_record* rec;
	const BtPiece* pieces;
	const unsigned long long* cap_off; // first capacity slot of each record (len(read) slots: a for matrix 1, then L - a)
	unsigned long long c_lo;           // first slot of the wave
	int2* cap;
	unsigned long long* cnt;           // pairs per (record, matrix)
	unsigned long long* wcnt;          // the same, scanned per wave
	int match, mismatch, gap, row0;
};

template <bool kShared>
__global__ void __launch_bounds__(DFB_BT_THREADS) bt_fill_walk_kernel(BtTables t, BtWalk p, long long p_lo, long long p_hi, unsigned* arena,
                                                                       unsigned long long slot_words)
{
	extern __shared__ unsigned bt_smem[];
	unsigned* const base = kShared ? bt_smem : arena + (unsigned long long)blockIdx.x * slot_words;
	for (long long q = p_lo + blockIdx.x; q < p_hi; q += gridDim.x)
	{
		const BtPiece pc = p.pieces[q];
		if (pc.glob == (int)kShared) continue;
		const int W1 = (pc.I1 + 16) >> 4, W2 = (pc.I2 + 16) >> 4;
		unsigned* const bits1 = base;
		unsigned* const bits2 = bits1 + bt_words(pc.I1, pc.J1);
		int* const edge1 = (int*)(bits2 + bt_words(pc.I2, pc.J2));
		int* const edge2 = edge1 + pc.I1 + 1;
		const int warp = threadIdx.x >> 5;
		if (warp < 2)
		{
			const bool m2 = warp == 1;
			bt_fill(t.ref_bytes + (m2 ? pc.ref2 : pc.ref1), t.read_bytes + pc.read, m2 ? pc.R2 : (int)(pc.ref2 - pc.ref1), pc.L, m2,
			        m2 ? pc.I2 : pc.I1, m2 ? pc.J2 : pc.J1, m2 ? bits2 : bits1, m2 ? edge2 : edge1, p.match, p.mismatch, p.gap, p.row0);
		}
		__syncthreads();
		for (long long w = threadIdx.x; w < 2 * (pc.k1 - pc.k0); w += DFB_BT_THREADS)
		{
			const long long k = pc.k0 + (w >> 1);
			const int half = (int)(w & 1);
			const dfb_split_record r = p.rec[k];
			const int a = r.read_split1;
			const unsigned* const bits = half ? bits2 : bits1;
			const int W = half ? W2 : W1;
			int i = half ? pc.R2 - r.ref_split2 - 1 : r.ref_split1, j = half ? pc.L - a : a, n = 0;
			int2* const out = p.cap + (p.cap_off[k] - p.c_lo) + (half ? a : 0);
			while (j > 0)
			{
				const unsigned dir = i == 0 ? 2u : (bits[(long long)(j - 1) * W + (i >> 4)] >> (2 * (i & 15))) & 3u; // row i == 0 points along the read
				if (dir == 0)
				{
					// walk order is descending: matrix 1 fills its slots from the top (BackTracePath's reverse), matrix 2
					// maps (i - 1, j - 1) of the reversed sequences back (ReverseMatches)
					if (half) out[n] = make_int2(pc.R2 - i, pc.L - j);
					else out[a - 1 - n] = make_int2(i - 1, j - 1);
					n++;
					i--;
					j--;
				}
				else if (dir == 1)
					i--;
				else
					j--;
			}
			p.cnt[2 * k + half] = (unsigned long long)n;
			p.wcnt[2 * k + half] = (unsigned long long)n;
		}
		__syncthreads();
	}
}

// one warp per (record, matrix) of the wave: its walked pairs from their capacity slots to the wave's output
__global__ void __launch_bounds__(DFB_BUILD_BLOCK) bt_compact_kernel(BtWalk p, long long s_lo, long long s_hi, int2* out)
{
	const int lane = threadIdx.x & 31;
	const long long warps = (long long)gridDim.x * (DFB_BUILD_BLOCK / 32);
	for (long long s = s_lo + (((long long)blockIdx.x * DFB_BUILD_BLOCK + threadIdx.x) >> 5); s < s_hi; s += warps)
	{
		const long long k = s >> 1;
		const int a = p.rec[k].read_split1;
		const long long n = (long long)p.cnt[s];
		const int2* src = p.cap + (p.cap_off[k] - p.c_lo) + ((s & 1) ? a : a - n);
		int2* dst = out + p.wcnt[s];
		for (long long e = lane; e < n; e += 32) dst[e] = src[e];
	}
}
}  // namespace dfb

static int dfb_split_backtrace_device_body(dfb_ctx* ctx, const dfb_split_params* params, const dfb_device_seq_table* refs,
                                           const dfb_device_seq_table* reads, const int32_t* task_cluster, const int32_t* task_read,
                                           int64_t n_tasks, const dfb_split_record* records, int64_t n_records, int64_t* n_pairs)
{
	using namespace dfb;
	if (!ctx) return DFB_ERR_ARG;
	ctx->has_bt = false;
	ctx->n_bt_records = ctx->n_bt_pairs = 0;
	dfree(ctx, ctx->d_bt_off);
	for (auto& c : ctx->bt_chunks) dfree(ctx, c.first);
	ctx->bt_chunks.clear();
	if (!params || !n_pairs || n_tasks < 0 || n_records < 0 || (n_tasks > 0 && (!task_cluster || !task_read)) || (n_records > 0 && !records))
		return set_err(ctx, DFB_ERR_ARG, "dfb_split_backtrace_device: null argument");
	const char* names[2] = {"refs", "reads"};
	const dfb_device_seq_table* tabs[2] = {refs, reads};
	for (int k = 0; k < 2; k++)
		if (!tabs[k] || !tabs[k]->off || tabs[k]->n < 0 || tabs[k]->n_bytes < 0) return set_err(ctx, DFB_ERR_ARG, "%s: null table", names[k]);
	CK(ctx, cudaSetDevice(ctx->device));
	const void* ptrs[7] = {refs->bytes, refs->off, reads->bytes, reads->off, task_cluster, task_read, records};
	const char* what[7] = {"refs->bytes", "refs->off", "reads->bytes", "reads->off", "task_cluster", "task_read", "records"};
	for (int k = 0; k < 7; k++)
		if (!is_ctx_device_memory(ctx, ptrs[k]))
			return set_err(ctx, DFB_ERR_ARG, "%s is not device memory of device %d", what[k], ctx->device);
	if (n_tasks > 0x7fffff00LL) return set_err(ctx, DFB_ERR_ARG, "too many tasks in one batch");
	int run_cap = DFB_BT_RUN_CAP;
	if (const char* e = getenv("DFB_BT_RUN_CAP")) // (measurement: DESIGN.md 4.5b)
		if (atoi(e) > 0) run_cap = atoi(e);

	cudaStream_t s = ctx->stream;
	const long long n = n_records;
	BtCheck* d_chk = nullptr;
	BtWave* d_waves = nullptr;
	BtPiece* pieces = nullptr;
	long long* piece_start = nullptr;
	unsigned long long *head = nullptr, *cap_off = nullptr, *cnt = nullptr, *wcnt = nullptr, *sums = nullptr;
	unsigned* arena = nullptr;
	int2* cap = nullptr;
	std::vector<std::pair<int2*, int64_t>> chunks; // the output: one exact-size block of pairs per wave
	auto cleanup = [&]() {
		dfree(ctx, d_chk);
		dfree(ctx, d_waves);
		dfree(ctx, pieces);
		dfree(ctx, piece_start);
		dfree(ctx, head);
		dfree(ctx, cap_off);
		dfree(ctx, cnt);
		dfree(ctx, wcnt);
		dfree(ctx, sums);
		dfree(ctx, arena);
		dfree(ctx, cap);
		for (auto& c : chunks) dfree(ctx, c.first);
		chunks.clear();
	};
	auto fail = [&](int code) {
		cleanup();
		cudaStreamSynchronize(s);
		return code;
	};
	cudaError_t e = dalloc(ctx, (void**)&d_chk, sizeof(BtCheck));
	if (e == cudaSuccess) e = dalloc(ctx, (void**)&head, (size_t)n * 8);
	if (e == cudaSuccess) e = dalloc(ctx, (void**)&cap_off, (size_t)n * 8);
	if (e == cudaSuccess) e = dalloc(ctx, (void**)&cnt, (size_t)(2 * n + 1) * 8);
	if (e == cudaSuccess) e = dalloc(ctx, (void**)&sums, (size_t)(2 * n / (DFB_BUILD_BLOCK * DFB_BUILD_ITEMS) + 2) * 8);
	if (e == cudaSuccess) e = ctx->h_out.ensure(sizeof(BtCheck));
	if (e != cudaSuccess) return fail(set_err(ctx, DFB_ERR_NOMEM, "backtrace: %s", cudaGetErrorString(e)));
	BtCheck* h_chk = (BtCheck*)ctx->h_out.p;

	// 1. checks, piece heads and capacities, their scans; one read-back
	const BtTables t{refs->bytes, reads->bytes, refs->off, reads->off, task_cluster, task_read, refs->n / 2, reads->n, n_tasks};
	const long long max_grid = (long long)ctx->prop.multiProcessorCount * 8;
	auto grid = [&](long long m) { return (unsigned)std::max<long long>(1, std::min<long long>((m + DFB_BUILD_BLOCK - 1) / DFB_BUILD_BLOCK, max_grid)); };
	enqueue_device_checks(ctx, false, refs, reads, task_cluster, task_read, n_tasks, &d_chk->dc);
	bt_check_init_kernel<<<1, 1, 0, s>>>(d_chk);
	if (n)
	{
		bt_records_kernel<<<grid(n), DFB_BUILD_BLOCK, 0, s>>>(records, n, t, run_cap, d_chk, head, cap_off);
		int rc = scan_u64(ctx, head, n, sums, &d_chk->n_pieces);
		if (!rc) rc = scan_u64(ctx, cap_off, n, sums, &d_chk->cap_total);
		if (rc) return fail(rc);
	}
	e = cudaGetLastError();
	if (e == cudaSuccess) e = cudaMemcpyAsync(h_chk, d_chk, sizeof(BtCheck), cudaMemcpyDeviceToHost, s);
	if (e == cudaSuccess) e = cudaStreamSynchronize(s);
	if (e != cudaSuccess) return fail(set_err(ctx, DFB_ERR_CUDA, "backtrace checks: %s", cudaGetErrorString(e)));
	if (int rc = device_check_status(ctx, false, refs, reads, n_tasks, h_chk->dc)) return fail(rc);
	if (h_chk->bad != ~0ull)
	{
		static const char* const bad_msg[3] = {"task out of range", "start cell outside the matrices", "read_split2 != len(read) - read_split1"};
		return fail(set_err(ctx, DFB_ERR_ARG, "record %lld: %s", (long long)(h_chk->bad >> 2), bad_msg[h_chk->bad & 3]));
	}
	const long long n_pieces = (long long)h_chk->n_pieces;
	// a wave takes the pieces whose capacity slots start in one DFB_BT_WAVE_PAIRS span of the records' slots
	const long long n_waves = n ? (long long)(h_chk->cap_total / DFB_BT_WAVE_PAIRS) + 1 : 0;
	std::vector<BtWave> waves((size_t)n_waves);

	// 2. pieces, their boxes and waves; the footprints come back to size the launches
	if (n)
	{
		e = dalloc(ctx, (void**)&d_waves, sizeof(BtWave) * (size_t)n_waves);
		if (e == cudaSuccess) e = dalloc(ctx, (void**)&piece_start, (size_t)n_pieces * 8);
		if (e == cudaSuccess) e = dalloc(ctx, (void**)&pieces, (size_t)n_pieces * sizeof(BtPiece));
		if (e == cudaSuccess) e = dalloc(ctx, (void**)&wcnt, (size_t)(2 * n) * 8);
		if (e != cudaSuccess) return fail(set_err(ctx, DFB_ERR_NOMEM, "backtrace pieces: %s", cudaGetErrorString(e)));
		bt_wave_init_kernel<<<(unsigned)((n_waves + 255) / 256), 256, 0, s>>>(d_waves, n_waves);
		bt_pieces_kernel<<<grid(n), DFB_BUILD_BLOCK, 0, s>>>(records, n, run_cap, head, piece_start);
		bt_box_kernel<<<grid(n_pieces), DFB_BUILD_BLOCK, 0, s>>>(records, n, t, piece_start, n_pieces, cap_off, d_chk, pieces, d_waves);
		e = cudaGetLastError();
		if (e == cudaSuccess) e = cudaMemcpyAsync(h_chk, d_chk, sizeof(BtCheck), cudaMemcpyDeviceToHost, s);
		if (e == cudaSuccess) e = cudaMemcpyAsync(waves.data(), d_waves, sizeof(BtWave) * (size_t)n_waves, cudaMemcpyDeviceToHost, s);
		if (e == cudaSuccess) e = cudaStreamSynchronize(s);
		if (e != cudaSuccess) return fail(set_err(ctx, DFB_ERR_CUDA, "backtrace pieces: %s", cudaGetErrorString(e)));
	}
	dfree(ctx, head);
	const BtCheck chk = *h_chk;

	// 3. per wave: fill and walk into capacity slots, count scan, compaction
	unsigned long long cap_pairs = 0;
	for (const BtWave& w : waves)
		if (w.p_lo < w.p_hi) cap_pairs = std::max(cap_pairs, w.c_hi - w.c_lo);
	const size_t smem_bytes = (size_t)chk.smem_words * 4;
	const unsigned long long slot_words = chk.glob_words;
	unsigned glob_grid = 0;
	if (chk.n_glob)
	{
		glob_grid = (unsigned)std::max<unsigned long long>(1, std::min<unsigned long long>(
			{chk.n_glob, (unsigned long long)ctx->prop.multiProcessorCount * 8, (unsigned long long)(DFB_BT_ARENA_BYTES / 4 / slot_words)}));
		e = dalloc(ctx, (void**)&arena, (size_t)glob_grid * slot_words * 4);
		if (e != cudaSuccess) return fail(set_err(ctx, DFB_ERR_NOMEM, "backtrace arena: %s", cudaGetErrorString(e)));
	}
	if (cap_pairs)
	{
		e = dalloc(ctx, (void**)&cap, (size_t)cap_pairs * sizeof(int2));
		if (e != cudaSuccess) return fail(set_err(ctx, DFB_ERR_NOMEM, "backtrace capacity (%llu pairs): %s", cap_pairs, cudaGetErrorString(e)));
	}
	if (smem_bytes > 48u << 10 &&
	    (e = cudaFuncSetAttribute(bt_fill_walk_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes)) != cudaSuccess)
		return fail(set_err(ctx, DFB_ERR_CUDA, "backtrace shared memory: %s", cudaGetErrorString(e)));
	BtWalk p{records, pieces, cap_off, 0, cap, cnt, wcnt, params->match, params->mismatch, params->gap, params->end_gaps ? 0 : params->gap};
	for (const BtWave& w : waves)
	{
		if (w.p_lo >= w.p_hi) continue;
		p.c_lo = w.c_lo;
		const long long wp = (long long)(w.p_hi - w.p_lo);
		if (smem_bytes)
			bt_fill_walk_kernel<true><<<(unsigned)std::min<long long>(wp, 1ll << 30), DFB_BT_THREADS, smem_bytes, s>>>(
				t, p, (long long)w.p_lo, (long long)w.p_hi, nullptr, 0);
		if (glob_grid)
			bt_fill_walk_kernel<false><<<glob_grid, DFB_BT_THREADS, 0, s>>>(t, p, (long long)w.p_lo, (long long)w.p_hi, arena, slot_words);
		const long long s_lo = 2 * (long long)w.k_lo, s_hi = 2 * (long long)w.k_hi;
		int rc = scan_u64(ctx, wcnt + s_lo, s_hi - s_lo, sums, &d_chk->wave_pairs);
		if (rc) return fail(rc);
		e = cudaGetLastError();
		if (e == cudaSuccess) e = cudaMemcpyAsync(h_chk, d_chk, sizeof(BtCheck), cudaMemcpyDeviceToHost, s);
		if (e == cudaSuccess) e = cudaStreamSynchronize(s);
		if (e != cudaSuccess) return fail(set_err(ctx, DFB_ERR_CUDA, "backtrace kernels: %s", cudaGetErrorString(e)));
		const unsigned long long got = h_chk->wave_pairs;
		if (!got) continue;
		int2* out = nullptr;
		e = dalloc(ctx, (void**)&out, (size_t)got * sizeof(int2));
		if (e != cudaSuccess) return fail(set_err(ctx, DFB_ERR_NOMEM, "%llu match pairs: %s", got, cudaGetErrorString(e)));
		chunks.push_back({out, (int64_t)got});
		bt_compact_kernel<<<grid(32 * (s_hi - s_lo)), DFB_BUILD_BLOCK, 0, s>>>(p, s_lo, s_hi, out);
	}

	// 4. match_off: the scan of all counts.  The waves' blocks stay as they are (copied out one after another): joining
	// them here would hold the whole output twice.
	int64_t total = 0;
	for (auto& c : chunks) total += c.second;
	if (n)
	{
		if (int rc = scan_u64(ctx, cnt, 2 * n, sums, cnt + 2 * n)) return fail(rc);
	}
	else if ((e = cudaMemsetAsync(cnt, 0, 8, s)) != cudaSuccess)
		return fail(set_err(ctx, DFB_ERR_CUDA, "backtrace: %s", cudaGetErrorString(e)));
	e = cudaGetLastError();
	if (e == cudaSuccess) e = cudaStreamSynchronize(s);
	if (e != cudaSuccess) return fail(set_err(ctx, DFB_ERR_CUDA, "backtrace: %s", cudaGetErrorString(e)));
	if (int rc = bounds_check_status(ctx)) return fail(rc);
	ctx->d_bt_off = (int64_t*)cnt;
	cnt = nullptr;
	ctx->bt_chunks.swap(chunks);
	cleanup();
	ctx->n_bt_records = n;
	ctx->n_bt_pairs = total;
	ctx->has_bt = true;
	*n_pairs = (int64_t)total;
	return DFB_OK;
}

extern "C" int dfb_split_backtrace_device(dfb_ctx* ctx, const dfb_split_params* params, const dfb_device_seq_table* refs,
                                          const dfb_device_seq_table* reads, const int32_t* task_cluster, const int32_t* task_read,
                                          int64_t n_tasks, const dfb_split_record* records, int64_t n_records, int64_t* n_pairs)
{
	return guarded(ctx, [&] {
		return dfb_split_backtrace_device_body(ctx, params, refs, reads, task_cluster, task_read, n_tasks, records, n_records, n_pairs);
	});
}

extern "C" int dfb_split_backtrace_copy_device(dfb_ctx* ctx, int64_t* match_off, int32_t* matches)
{
	return guarded(ctx, [&]() -> int {
		if (!ctx) return DFB_ERR_ARG;
		if (!ctx->has_bt) return set_err(ctx, DFB_ERR_STATE, "no backtrace on this context: call dfb_split_backtrace_device first");
		if (!match_off || (ctx->n_bt_pairs && !matches)) return set_err(ctx, DFB_ERR_ARG, "dfb_split_backtrace_copy_device: null argument");
		CK(ctx, cudaSetDevice(ctx->device));
		if (!is_ctx_device_memory(ctx, match_off)) return set_err(ctx, DFB_ERR_ARG, "match_off is not device memory of device %d", ctx->device);
		if (!is_ctx_device_memory(ctx, matches)) return set_err(ctx, DFB_ERR_ARG, "matches is not device memory of device %d", ctx->device);
		CK(ctx, cudaMemcpyAsync(match_off, ctx->d_bt_off, (size_t)(2 * ctx->n_bt_records + 1) * 8, cudaMemcpyDeviceToDevice, ctx->stream));
		int64_t at = 0;
		for (const auto& c : ctx->bt_chunks)
		{
			CK(ctx, cudaMemcpyAsync(matches + 2 * at, c.first, (size_t)c.second * sizeof(int2), cudaMemcpyDeviceToDevice, ctx->stream));
			at += c.second;
		}
		CK(ctx, cudaStreamSynchronize(ctx->stream));
		return DFB_OK;
	});
}
