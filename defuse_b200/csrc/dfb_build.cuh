// Job lists built on the GPU.  What SplitAlignmentTask::Align / SplitReadRealigner::DoAlignment hand to the aligner one
// task at a time (tools/SplitAlignment.cpp:266-303, 371-379: two windows of a cluster and one read) arrives here as
// the caller's raw task arrays; the batch form needs them grouped by kernel class and reference length.  The host
// used to classify the tasks, lay out the packed pool and write a 32-byte job record per task (about half of the CPU
// time of a batch); these kernels do it on the device from the uploaded offsets and task arrays:
//
//   desc_count / desc_scan / desc_write   sequence descriptors {source byte, length, first pool word} of a CSR table
//   split_classify_kernel                 class + reference-length bin per task, bin histogram, work statistics
//   bin_scan_kernel                       histogram -> first job of every bin, jobs per class
//   split_scatter_kernel                  one JobPair per task into its bin (warp-aggregated slots, task order kept
//                                         inside a warp)
// HBM-bound and small next to the sweeps (about 60 B read and 52 B written per task).
#pragma once

namespace dfb
{

#define DFB_BUILD_BLOCK 256
#define DFB_BUILD_ITEMS 4
#define DFB_BUILD_RBINS 1024
#define DFB_BUILD_MAX_CLASSES 16

__device__ __forceinline__ unsigned long long desc_words(const int64_t* __restrict__ off, long long i, long long n, int copies, int* bad)
{
	if (i >= n) return 0;
	const long long len = off[i + 1] - off[i];
	if (len < 0 || len > 0x7fffff00LL)
	{
		*bad = 1;
		return 0;
	}
	unsigned long long w = (unsigned long long)((len + 15) >> 4) * (unsigned)copies;
	return w + (w & 1); // every sequence starts on an even word (16-byte cp.async)
}

// block-wide sum / exclusive scan of one value per thread (DFB_BUILD_BLOCK threads)
__device__ __forceinline__ unsigned long long block_exclusive_scan(unsigned long long v, unsigned long long* total)
{
	__shared__ unsigned long long s_warp[DFB_BUILD_BLOCK / 32];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	unsigned long long x = v;
#pragma unroll
	for (int o = 1; o < 32; o <<= 1)
	{
		const unsigned long long y = __shfl_up_sync(0xffffffffu, x, o);
		if (lane >= o) x += y;
	}
	if (lane == 31) s_warp[warp] = x;
	__syncthreads();
	unsigned long long before = 0, all = 0;
#pragma unroll
	for (int k = 0; k < DFB_BUILD_BLOCK / 32; k++)
	{
		const unsigned long long w = s_warp[k];
		if (k < warp) before += w;
		all += w;
	}
	__syncthreads();
	if (total) *total = all;
	return before + x - v;
}

struct DescParams
{
	const int64_t* off; // device copy of the table's offsets, off[0 .. n]
	long long n;
	int copies;          // stored copies per sequence: 1, or 2 (forward + reversed reads of the split aligner)
	long long src_base;  // byte of off[0] in the raw upload
	SeqDesc* desc;
	unsigned long long* block_sums;       // [blocks]
	const unsigned long long* word_base;  // device scalar: first word of this table (null: 0)
	unsigned long long* total;            // device scalar: word_base + words of this table
	int* bad;                             // set when a length is negative or too long
};

__global__ void __launch_bounds__(DFB_BUILD_BLOCK) desc_count_kernel(DescParams p)
{
	const long long i0 = ((long long)blockIdx.x * DFB_BUILD_BLOCK + threadIdx.x) * DFB_BUILD_ITEMS;
	unsigned long long sum = 0;
#pragma unroll
	for (int k = 0; k < DFB_BUILD_ITEMS; k++) sum += desc_words(p.off, i0 + k, p.n, p.copies, p.bad);
	unsigned long long all = 0;
	block_exclusive_scan(sum, &all);
	if (threadIdx.x == 0) p.block_sums[blockIdx.x] = all;
}

// one block: exclusive scan of the block sums in place, starting at *word_base
__global__ void __launch_bounds__(DFB_BUILD_BLOCK) desc_scan_kernel(unsigned long long* sums, long long n_blocks, const unsigned long long* word_base,
                                                                     unsigned long long* total)
{
	unsigned long long carry = word_base ? *word_base : 0ull;
	for (long long base = 0; base < n_blocks; base += DFB_BUILD_BLOCK)
	{
		const long long i = base + threadIdx.x;
		const unsigned long long v = i < n_blocks ? sums[i] : 0ull;
		unsigned long long all = 0;
		const unsigned long long ex = block_exclusive_scan(v, &all);
		if (i < n_blocks) sums[i] = carry + ex;
		carry += all;
	}
	if (threadIdx.x == 0) *total = carry;
}

__global__ void __launch_bounds__(DFB_BUILD_BLOCK) desc_write_kernel(DescParams p)
{
	const long long i0 = ((long long)blockIdx.x * DFB_BUILD_BLOCK + threadIdx.x) * DFB_BUILD_ITEMS;
	unsigned long long w[DFB_BUILD_ITEMS], sum = 0;
	int bad = 0;
#pragma unroll
	for (int k = 0; k < DFB_BUILD_ITEMS; k++)
	{
		w[k] = desc_words(p.off, i0 + k, p.n, p.copies, &bad);
		sum += w[k];
	}
	unsigned long long at = p.block_sums[blockIdx.x] + block_exclusive_scan(sum, nullptr);
	const long long o0 = p.off[0];
#pragma unroll
	for (int k = 0; k < DFB_BUILD_ITEMS; k++)
	{
		const long long i = i0 + k;
		if (i < p.n)
		{
			SeqDesc d;
			d.src = 16 + p.src_base + (p.off[i] - o0);
			const long long len = p.off[i + 1] - p.off[i];
			d.len = (uint32_t)(len < 0 ? 0LL : (len > 0x7fffff00LL ? 0x7fffff00LL : len));
			d.word = (uint32_t)at;
			p.desc[i] = d;
		}
		at += w[k];
	}
}

// what the host needs back before it can size the per-class buffers and launch the sweeps
struct BuildStats
{
	unsigned long long cells;
	unsigned long long bad_task;   // lowest task index with a table index out of range (~0: none)
	unsigned long long total_words;
	unsigned int n_gen;            // tasks only the s32 kernels can take
	unsigned int gen_max_R;
	int bad_table;
	int pad;
	unsigned int cls_jobs[DFB_BUILD_MAX_CLASSES];
	unsigned int cls_max_R[DFB_BUILD_MAX_CLASSES];
};

struct SplitBuildParams
{
	const SeqDesc* desc_a; // two windows per cluster
	long long n_clusters;
	const SeqDesc* desc_b;
	long long n_reads;
	const int32_t* task_cluster;
	const int32_t* task_read;
	const int32_t* task_min_score;
	long long n_tasks;
	int32_t read_base;        // first entry of table b in the caller's numbering (a chunk sees a view of it)
	int32_t ref_base;         // simple batches: the same for table a
	int simple;               // 0: split tasks (cluster, read, minScore); 1: SimpleAligner tasks (reference, sequence), two per job
	unsigned int cls_first_task[DFB_BUILD_MAX_CLASSES]; // simple scatter: first task position / first job of every class
	unsigned int cls_first_job[DFB_BUILD_MAX_CLASSES];
	int32_t* bin_of;          // [n_tasks]: class * RBINS + bin, -1: no work (empty read), -2: generic path
	unsigned int* bin_count;  // [classes * RBINS], zeroed; the scan turns it into the first job of every bin
	unsigned int* bin_fill;   // [classes * RBINS], zeroed
	int n_classes;
	int cls_rows[DFB_BUILD_MAX_CLASSES]; // read rows a class holds (ascending)
	int cls_ok[DFB_BUILD_MAX_CLASSES];   // the s16x2 kernels are exact for this class with the batch's scoring
	int max_fast_rows;
	BuildStats* stats;
	JobPair* jobs;
};

__global__ void __launch_bounds__(DFB_BUILD_BLOCK) split_classify_kernel(SplitBuildParams p)
{
	const long long t = (long long)blockIdx.x * DFB_BUILD_BLOCK + threadIdx.x;
	int bin = -1;
	unsigned int fast_R = 0;
	unsigned long long cells = 0;
	if (t < p.n_tasks)
	{
		const long long c0 = (long long)p.task_cluster[t] - p.ref_base, rd = (long long)p.task_read[t] - p.read_base;
		if (c0 < 0 || c0 >= p.n_clusters || rd < 0 || rd >= p.n_reads)
		{
			atomicMin(&p.stats->bad_task, (unsigned long long)t);
		}
		else
		{
			// split: the two windows of cluster c0; simple: reference c0 alone
			const long long R1 = p.simple ? p.desc_a[c0].len : p.desc_a[2 * c0].len;
			const long long R2 = p.simple ? 0 : p.desc_a[2 * c0 + 1].len, L = p.desc_b[rd].len;
			cells = (unsigned long long)((R1 + R2) * L);
			// an empty read has no split (SplitReadAligner.cpp:224-227); no interior cell: score 0 (SimpleAligner.cpp:30)
			if (L > 0 && (!p.simple || R1 > 0))
			{
				const long long Rm = max(R1, R2);
				int c = -1;
				if (L <= p.max_fast_rows && Rm <= 65535)
				{
					c = 0;
					while (c < p.n_classes && p.cls_rows[c] < L) c++;
					if (c >= p.n_classes || !p.cls_ok[c]) c = -1;
				}
				if (c < 0)
				{
					bin = -2;
					atomicAdd(&p.stats->n_gen, 1u); // (rare: these tasks send the chunk to the host path)
					atomicMax(&p.stats->gen_max_R, (unsigned int)(Rm > 0xffffffffLL ? 0xffffffffLL : Rm));
				}
				else
				{
					const long long rb = Rm >> 4;
					bin = c * DFB_BUILD_RBINS + (DFB_BUILD_RBINS - 1 - (int)(rb < DFB_BUILD_RBINS - 1 ? rb : DFB_BUILD_RBINS - 1));
					fast_R = (unsigned int)Rm;
				}
			}
		}
		p.bin_of[t] = bin;
	}
	// histogram and longest reference per class: the tasks of a cluster are neighbours and share a bin, one atomic per
	// group of equal bins in a warp (every task on its own would serialise on a handful of addresses)
	const unsigned active = __ballot_sync(0xffffffffu, bin >= 0);
	if (bin >= 0)
	{
		const unsigned same = __match_any_sync(active, bin);
		const unsigned int group_R = __reduce_max_sync(same, fast_R);
		if ((int)(threadIdx.x & 31) == __ffs(same) - 1)
		{
			atomicAdd(&p.bin_count[bin], (unsigned)__popc(same));
			const int c = bin / DFB_BUILD_RBINS;
			if (group_R > p.stats->cls_max_R[c]) atomicMax(&p.stats->cls_max_R[c], group_R);
		}
	}
	// cells: block sum, one atomic per block
	unsigned long long all = 0;
	block_exclusive_scan(cells, &all);
	if (threadIdx.x == 0 && all) atomicAdd(&p.stats->cells, all);
}

// one block of 896 threads, 16 consecutive bins per thread (a class is 64 threads): histogram -> exclusive prefix
__global__ void __launch_bounds__(1024) bin_scan_kernel(unsigned int* bin_count, int n_classes, BuildStats* stats)
{
	__shared__ unsigned int s_tot[1024];
	const int tid = threadIdx.x;
	const int n_bins = n_classes * DFB_BUILD_RBINS;
	unsigned int v[16], sum = 0;
#pragma unroll
	for (int k = 0; k < 16; k++)
	{
		const int b = tid * 16 + k;
		v[k] = b < n_bins ? bin_count[b] : 0u;
		sum += v[k];
	}
	s_tot[tid] = sum;
	__syncthreads();
	// (a serial prefix over <= 1024 partial sums by every thread would be 1024^2 reads; two levels instead)
	__shared__ unsigned int s_cls[DFB_BUILD_MAX_CLASSES + 1];
	if (tid <= n_classes && tid <= DFB_BUILD_MAX_CLASSES)
	{
		unsigned int before = 0;
		for (int k = 0; k < tid * 64 && k < 1024; k++) before += s_tot[k];
		s_cls[tid] = before;
	}
	__syncthreads();
	const int cls = tid / 64;
	unsigned int at = cls <= DFB_BUILD_MAX_CLASSES ? s_cls[min(cls, n_classes)] : 0u;
	for (int k = cls * 64; k < tid; k++) at += s_tot[k];
#pragma unroll
	for (int k = 0; k < 16; k++)
	{
		const int b = tid * 16 + k;
		if (b < n_bins) bin_count[b] = at;
		at += v[k];
	}
	if (tid < n_classes) stats->cls_jobs[tid] = s_cls[tid + 1] - s_cls[tid];
}

// The statistics go to the host through a store into pinned host memory, not through a copy: the copy engine may be
// busy for a millisecond or two with a previous chunk's result rows, and the host is waiting for these 200 bytes to
// launch the next chunk.
__global__ void stats_to_host_kernel(const BuildStats* __restrict__ d_stats, BuildStats* __restrict__ h_stats)
{
	const unsigned int* src = reinterpret_cast<const unsigned int*>(d_stats);
	unsigned int* dst = reinterpret_cast<unsigned int*>(h_stats);
	for (unsigned k = threadIdx.x; k < sizeof(BuildStats) / sizeof(unsigned int); k += blockDim.x) dst[k] = src[k];
	__threadfence_system();
}

__global__ void __launch_bounds__(DFB_BUILD_BLOCK) split_scatter_kernel(SplitBuildParams p)
{
	const long long t = (long long)blockIdx.x * DFB_BUILD_BLOCK + threadIdx.x;
	const int bin = t < p.n_tasks ? p.bin_of[t] : -1;
	const unsigned active = __ballot_sync(0xffffffffu, bin >= 0);
	if (bin < 0) return;
	const unsigned same = __match_any_sync(active, bin);
	const int lane = threadIdx.x & 31, leader = __ffs(same) - 1;
	unsigned int base = 0;
	if (lane == leader) base = atomicAdd(&p.bin_fill[bin], (unsigned)__popc(same));
	base = __shfl_sync(same, base, leader);
	const unsigned int pos = p.bin_count[bin] + base + (unsigned)__popc(same & ((1u << lane) - 1u));
	const long long c2 = 2 * ((long long)p.task_cluster[t] - p.ref_base);
	const SeqDesc r1 = p.desc_a[c2], r2 = p.desc_a[c2 + 1], rdd = p.desc_b[(long long)p.task_read[t] - p.read_base];
	JobPair jp;
	jp.ref_w[0] = r1.word;
	jp.ref_w[1] = r2.word;
	jp.read_w[0] = rdd.word;
	jp.read_w[1] = rdd.word + ((rdd.len + 15) >> 4); // the reversed copy sits right behind the forward one
	jp.R[0] = (uint16_t)r1.len;
	jp.R[1] = (uint16_t)r2.len;
	jp.L[0] = jp.L[1] = (uint16_t)rdd.len;
	jp.out0 = (int32_t)t;
	jp.out1 = p.task_min_score[t];
	DFB_BC((long long)pos < p.n_tasks && bin < p.n_classes * DFB_BUILD_RBINS, 401);
	p.jobs[pos] = jp;
}

// SimpleAligner batches: two tasks share a job (low / high half of the registers); the task at position q inside its
// class goes to job q/2, half q%2.  The last job of a class with an odd number of tasks keeps an empty half.
__global__ void __launch_bounds__(DFB_BUILD_BLOCK) jobs_init_kernel(JobPair* jobs, long long n_jobs)
{
	const long long j = (long long)blockIdx.x * DFB_BUILD_BLOCK + threadIdx.x;
	if (j >= n_jobs) return;
	JobPair jp;
	jp.ref_w[0] = jp.ref_w[1] = jp.read_w[0] = jp.read_w[1] = 0;
	jp.R[0] = jp.R[1] = jp.L[0] = jp.L[1] = 0;
	jp.out0 = jp.out1 = -1;
	jobs[j] = jp;
}

__global__ void __launch_bounds__(DFB_BUILD_BLOCK) simple_scatter_kernel(SplitBuildParams p)
{
	const long long t = (long long)blockIdx.x * DFB_BUILD_BLOCK + threadIdx.x;
	const int bin = t < p.n_tasks ? p.bin_of[t] : -1;
	const unsigned active = __ballot_sync(0xffffffffu, bin >= 0);
	if (bin < 0) return;
	const unsigned same = __match_any_sync(active, bin);
	const int lane = threadIdx.x & 31, leader = __ffs(same) - 1;
	unsigned int base = 0;
	if (lane == leader) base = atomicAdd(&p.bin_fill[bin], (unsigned)__popc(same));
	base = __shfl_sync(same, base, leader);
	const unsigned int pos = p.bin_count[bin] + base + (unsigned)__popc(same & ((1u << lane) - 1u)); // among all fast tasks
	const int c = bin / DFB_BUILD_RBINS;
	const unsigned int q = pos - p.cls_first_task[c];
	const SeqDesc r = p.desc_a[(long long)p.task_cluster[t] - p.ref_base], sq = p.desc_b[(long long)p.task_read[t] - p.read_base];
	JobPair* jp = p.jobs + p.cls_first_job[c] + (q >> 1);
	DFB_BC((long long)(p.cls_first_job[c] + (q >> 1)) < (p.n_tasks + DFB_BUILD_MAX_CLASSES) / 2 + DFB_BUILD_MAX_CLASSES, 402);
	const int h = (int)(q & 1u);
	jp->ref_w[h] = r.word;
	jp->read_w[h] = sq.word;
	jp->R[h] = (uint16_t)r.len;
	jp->L[h] = (uint16_t)sq.len;
	if (h == 0) jp->out0 = (int32_t)t;
	else jp->out1 = (int32_t)t;
}

// ---- argument checks of the device-resident entry points ------------------------------------------------------
// What check_table and the host builder's task pass find, computed where the caller's arrays live; only this record
// goes to the host, which words the same messages from it.
struct TableCheck
{
	unsigned long long first_bad; // 2k: offsets decrease at k; 2k + 1: sequence k too long (~0: none)
	unsigned long long max_len;
	long long off0, off_n;
};

struct DeviceCheck
{
	TableCheck tab[2];            // table A (references / windows), table B (sequences / reads)
	unsigned long long bad_task;  // lowest task with an index out of range (~0: none)
	int a_decreases, b_decreases; // the task arrays decrease somewhere
};

__global__ void device_check_init_kernel(DeviceCheck* c)
{
	c->tab[0].first_bad = c->tab[1].first_bad = ~0ull;
	c->tab[0].max_len = c->tab[1].max_len = 0;
	c->bad_task = ~0ull;
	c->a_decreases = c->b_decreases = 0;
}

__global__ void __launch_bounds__(DFB_BUILD_BLOCK) table_check_kernel(const int64_t* __restrict__ off, long long n, TableCheck* out)
{
	const long long k0 = (long long)blockIdx.x * DFB_BUILD_BLOCK + threadIdx.x, stride = (long long)gridDim.x * DFB_BUILD_BLOCK;
	if (k0 == 0)
	{
		out->off0 = off[0];
		out->off_n = off[n];
	}
	unsigned long long mx = 0;
	for (long long k = k0; k < n; k += stride)
	{
		const long long len = off[k + 1] - off[k];
		if (len < 0) atomicMin(&out->first_bad, 2ull * (unsigned long long)k);
		else if (len > 0x7fffff00LL) atomicMin(&out->first_bad, 2ull * (unsigned long long)k + 1);
		else mx = max(mx, (unsigned long long)len);
	}
	for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_down_sync(0xffffffffu, mx, o));
	if ((threadIdx.x & 31) == 0 && mx) atomicMax(&out->max_len, mx);
}

// a_lim / b_lim: entries task_a / task_b may name (split: clusters, reads; simple: references, sequences)
__global__ void __launch_bounds__(DFB_BUILD_BLOCK) task_check_kernel(const int32_t* __restrict__ ta, const int32_t* __restrict__ tb, long long n,
                                                                      long long a_lim, long long b_lim, DeviceCheck* out)
{
	const long long t0 = (long long)blockIdx.x * DFB_BUILD_BLOCK + threadIdx.x, stride = (long long)gridDim.x * DFB_BUILD_BLOCK;
	int a_dec = 0, b_dec = 0;
	for (long long t = t0; t < n; t += stride)
	{
		const int32_t a = ta[t], b = tb[t];
		if (a < 0 || a >= a_lim || b < 0 || b >= b_lim) atomicMin(&out->bad_task, (unsigned long long)t);
		if (t > 0)
		{
			a_dec |= a < ta[t - 1];
			b_dec |= b < tb[t - 1];
		}
	}
	if (__any_sync(0xffffffffu, a_dec) && (threadIdx.x & 31) == 0) out->a_decreases = 1;
	if (__any_sync(0xffffffffu, b_dec) && (threadIdx.x & 31) == 0) out->b_decreases = 1;
}

// Where the chunks of a device-resident batch sit in the tables: for chunk k over tasks [t0[k], t0[k+1]),
// b_lo = task_b[t0[k]], b_hi = task_b[t0[k+1] - 1] + 1 and, with a_monotone, the same for task_a (else a covers the
// whole table); then the byte offsets of those views.  out[k]: a_lo, a_hi, b_lo, b_hi, off_a[per a_lo],
// off_a[per a_hi], off_b[b_lo], off_b[b_hi].
#define DFB_MAX_CHUNKS 8
struct ChunkStarts
{
	long long t[DFB_MAX_CHUNKS + 1];
};

__global__ void chunk_bounds_kernel(const int64_t* __restrict__ off_a, long long n_a_items, int per, const int64_t* __restrict__ off_b,
                                    const int32_t* __restrict__ ta, const int32_t* __restrict__ tb, ChunkStarts t0, int K, int a_monotone,
                                    long long* out)
{
	const int k = threadIdx.x;
	if (k >= K) return;
	const long long lo = t0.t[k], hi = t0.t[k + 1];
	long long a_lo = 0, a_hi = n_a_items;
	if (a_monotone)
	{
		a_lo = ta[lo];
		a_hi = (long long)ta[hi - 1] + 1;
	}
	const long long b_lo = tb[lo], b_hi = (long long)tb[hi - 1] + 1;
	long long* o = out + 8 * k;
	o[0] = a_lo;
	o[1] = a_hi;
	o[2] = b_lo;
	o[3] = b_hi;
	o[4] = off_a[per * a_lo];
	o[5] = off_a[per * a_hi];
	o[6] = off_b[b_lo];
	o[7] = off_b[b_hi];
}

// ---- exclusive scan of a u64 array in place (the desc_count / desc_scan / desc_write pattern) -------------------
__global__ void __launch_bounds__(DFB_BUILD_BLOCK) u64_scan_sums_kernel(const unsigned long long* __restrict__ v, long long n,
                                                                         unsigned long long* block_sums)
{
	const long long i0 = ((long long)blockIdx.x * DFB_BUILD_BLOCK + threadIdx.x) * DFB_BUILD_ITEMS;
	unsigned long long sum = 0;
#pragma unroll
	for (int k = 0; k < DFB_BUILD_ITEMS; k++)
		if (i0 + k < n) sum += v[i0 + k];
	unsigned long long all = 0;
	block_exclusive_scan(sum, &all);
	if (threadIdx.x == 0) block_sums[blockIdx.x] = all;
}

__global__ void __launch_bounds__(DFB_BUILD_BLOCK) u64_scan_write_kernel(unsigned long long* v, long long n,
                                                                          const unsigned long long* __restrict__ block_sums)
{
	const long long i0 = ((long long)blockIdx.x * DFB_BUILD_BLOCK + threadIdx.x) * DFB_BUILD_ITEMS;
	unsigned long long x[DFB_BUILD_ITEMS], sum = 0;
#pragma unroll
	for (int k = 0; k < DFB_BUILD_ITEMS; k++)
	{
		x[k] = i0 + k < n ? v[i0 + k] : 0ull;
		sum += x[k];
	}
	unsigned long long at = block_sums[blockIdx.x] + block_exclusive_scan(sum, nullptr);
#pragma unroll
	for (int k = 0; k < DFB_BUILD_ITEMS; k++)
		if (i0 + k < n)
		{
			v[i0 + k] = at;
			at += x[k];
		}
}

}  // namespace dfb
