// Host side of the C ABI in include/defuse_b200.h: context, plan building (packing,
// length-bucketed job lists), kernel dispatch and result assembly.  No CPU implementation
// of the DP exists in this library: without a GPU every entry point fails.
//
// Host-path design (it bounds the end-to-end number once the kernels run at TCUPS rates):
//  * device memory comes from the stream-ordered pool (cudaMallocAsync, nothing released
//    back to the driver between batches); host-built arrays are written straight into a
//    grow-only pinned staging buffer, results land in another one;
//  * jobs are ordered by one counting sort (kernel class, reference length), O(n);
//  * the probe sweep leaves its arg-max columns in fixed 128-byte regions per winning task,
//    so the host only has to order a handful of entries per task; that assembly is
//    spread over host threads.
#include "../../include/defuse_b200.h"
#include "dfb_kernels.cuh"
#include "dfb_build.cuh"
#include "dfb_assemble.cuh"

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <atomic>
#include <condition_variable>
#include <cstring>
#include <functional>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>
#include <time.h>

using namespace dfb;

// ------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------

struct PinnedBuf
{
	void* p = nullptr;
	size_t cap = 0;
	cudaError_t ensure(size_t n)
	{
		if (n <= cap) return cudaSuccess;
		if (p) cudaFreeHost(p);
		p = nullptr;
		cap = 0;
		size_t want = n + n / 4 + 4096;
		cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocPortable | cudaHostAllocMapped); // (kernels store the build statistics into it)
		if (e == cudaSuccess) cap = want;
		return e;
	}
	void release()
	{
		if (p) cudaFreeHost(p);
		p = nullptr;
		cap = 0;
	}
};

// malloc-backed array without value-initialisation (result arrays of ~10^8 bytes: no memset, and the
// pages of a recycled buffer are already mapped)
template <class T>
struct HostArr
{
	T* p = nullptr;
	size_t n = 0, cap = 0;
	bool ensure(size_t want)
	{
		if (want > cap)
		{
			free(p);
			cap = want + want / 8 + 64;
			p = (T*)malloc(cap * sizeof(T));
			if (!p) { cap = 0; n = 0; return false; }
		}
		n = want;
		return true;
	}
	// grows without losing the first `keep` elements
	bool ensure_keep(size_t want, size_t keep)
	{
		if (want > cap)
		{
			const size_t ncap = want + want / 4 + 64;
			T* q = (T*)malloc(ncap * sizeof(T));
			if (!q) return false;
			if (keep) memcpy(q, p, keep * sizeof(T));
			free(p);
			p = q;
			cap = ncap;
		}
		n = want;
		return true;
	}
	void release() { free(p); p = nullptr; n = cap = 0; }
	void swap(HostArr& o) { std::swap(p, o.p); std::swap(n, o.n); std::swap(cap, o.cap); }
	size_t size() const { return n; }
	bool empty() const { return n == 0; }
	T* data() { return p; }
	const T* data() const { return p; }
};

// Persistent host workers of a context: the batch path runs a dozen short parallel loops per call, and
// spawning threads for each of them costs more than the loops.
class HostPool
{
public:
	explicit HostPool(int n_threads)
	{
		for (int k = 1; k < n_threads; k++) mWorkers.emplace_back([this, k] { Work(k); });
	}
	~HostPool()
	{
		{
			std::lock_guard<std::mutex> lk(mMutex);
			mStop = true;
			mGeneration++;
		}
		mStart.notify_all();
		for (auto& t : mWorkers) t.join();
	}
	int Size() const { return (int)mWorkers.size() + 1; }
	// runs fn(0..T-1) on T threads (the caller is thread 0) and waits for all of them
	void Run(int T, const std::function<void(int)>& fn)
	{
		T = std::max(1, std::min(T, Size()));
		if (T == 1) { fn(0); return; }
		{
			std::lock_guard<std::mutex> lk(mMutex);
			mFn = &fn;
			mActive = T;
			mPending = T - 1;
			mGeneration++;
		}
		mStart.notify_all();
		fn(0);
		std::unique_lock<std::mutex> lk(mMutex);
		mDone.wait(lk, [this] { return mPending == 0; });
		mFn = nullptr;
	}

private:
	void Work(int k)
	{
		long long seen = 0;
		for (;;)
		{
			const std::function<void(int)>* fn = nullptr;
			{
				std::unique_lock<std::mutex> lk(mMutex);
				mStart.wait(lk, [&] { return mGeneration != seen; });
				seen = mGeneration;
				if (mStop) return;
				if (k < mActive) fn = mFn;
			}
			if (fn)
			{
				(*fn)(k);
				std::lock_guard<std::mutex> lk(mMutex);
				if (--mPending == 0) mDone.notify_one();
			}
		}
	}
	std::vector<std::thread> mWorkers;
	std::mutex mMutex;
	std::condition_variable mStart, mDone;
	const std::function<void(int)>* mFn = nullptr;
	long long mGeneration = 0;
	int mActive = 0, mPending = 0;
	bool mStop = false;
};

template <class F>
static void parallel_for(HostPool* pool, int T, F fn)
{
	if (T <= 1) { fn(0); return; }
	if (pool && T <= pool->Size())
	{
		const std::function<void(int)> f = fn;
		pool->Run(T, f);
		return;
	}
	std::vector<std::thread> th;
	th.reserve((size_t)T - 1);
	for (int k = 1; k < T; k++) th.emplace_back(fn, k);
	fn(0);
	for (auto& x : th) x.join();
}

// Match lists of a backtrace in device memory of the stream-ordered pool: 2 n + 1 offsets and the (refPos, readPos)
// pairs, one exact-size block per wave of the call, in order
struct BtResult
{
	int64_t* d_off = nullptr;
	std::vector<std::pair<int2*, int64_t>> chunks;
	int64_t n_records = 0, n_pairs = 0;
};

struct dfb_ctx
{
	int device = 0;
	cudaStream_t own_stream = nullptr;
	cudaStream_t stream = nullptr;
	cudaDeviceProp prop;
	mutable std::string err;
	mutable std::mutex err_mu; // the two lanes of a pipelined batch may both report
	static const int kStageSlots = 8;
	PinnedBuf h_in[kStageSlots]; // host-built descriptors and job lists, on their way to the device (one per batch chunk in flight)
	PinnedBuf h_out;             // results on their way back
	cudaStream_t copy_stream = nullptr; // device->host result copies, ordered after a plan's kernels by an event
	cudaStream_t upload_stream = nullptr; // uploads + packing of the next chunk of a pipelined batch
	cudaStream_t upload_stream2 = nullptr; // host-built chunks alternate between the two: chunk k+1's uploads do not hold up chunk k's packing
	// first-sweep state (checkpoints, probe targets, read symbols) of the chunk of a pipelined batch that is on the GPU:
	// ONE buffer for all chunks and batches -- chunk k+1's first sweep is queued behind chunk k's probe sweep on the compute
	// stream, so they never overlap --, grown when a chunk needs more.  (Allocated per chunk, a chunk slightly larger than
	// the one before it grew the pool by gigabytes in the middle of a batch: 8 ms of idle GPU, profiles/r04f.)
	uint8_t* sweep_arena = nullptr;
	size_t sweep_arena_cap = 0;
	cudaEvent_t copied_ev = nullptr;      // blocking-sync event behind the result copies of a fetch
	// pageable caller buffers are staged through a small ring of pinned blocks by the context's workers (the driver's own
	// staging copies with one thread and blocks the caller for the whole transfer)
	static const int kRingSlots = 4;
	static const size_t kRingBlock = (size_t)8 << 20;
	PinnedBuf h_ring;
	cudaEvent_t ring_ev[kRingSlots] = {nullptr, nullptr, nullptr, nullptr};
	unsigned long long ring_next = 0;
	HostPool* pool = nullptr;       // plan building (and everything else on the caller's thread)
	HostPool* pool_fetch = nullptr; // result assembly when it runs on the pipelining helper thread
	dfb_plan* last_split = nullptr; // result holder of dfb_split_align_batch
	// records of the last dfb_split_records_device call (device memory of the stream-ordered pool)
	dfb_split_record* d_records = nullptr;
	int64_t n_records = 0;
	bool has_records = false;
	BtResult bt; // match lists of the last dfb_split_backtrace_device call (none: bt.d_off == nullptr)
	int host_threads = 1;
	// recycled host memory of the result assembly (kept mapped between batches)
	HostArr<dfb_split_row> spare_rows;
	HostArr<int32_t> spare_cols;
};

static thread_local std::string g_create_err;

// DFB_TRACE=1: phase timings of the host path on stderr
#include <chrono>
static bool trace_on()
{
	static int on = -1;
	if (on < 0) { const char* e = getenv("DFB_TRACE"); on = (e && *e && *e != '0') ? 1 : 0; }
	return on == 1;
}
struct Trace
{
	std::chrono::steady_clock::time_point t0;
	Trace() : t0(std::chrono::steady_clock::now()) {}
	void lap(const char* what)
	{
		if (!trace_on()) return;
		auto t1 = std::chrono::steady_clock::now();
		static const auto origin = t1;
		fprintf(stderr, "[dfb] %-28s %8.3f ms   (at %9.3f)\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count(),
		        std::chrono::duration<double, std::milli>(t1 - origin).count());
		t0 = t1;
	}
};

// Waiting for an event on a pipeline's critical path.  A blocking-sync wait sleeps until the driver's interrupt wakes the
// thread: 0.4-0.9 ms late on the VMs this was measured on (DFB_TRACE device timeline against the host laps), three or four
// times per batch where nothing else covers it.  So: poll, sleeping 30 us between queries (a few per cent of one core,
// which matters when eight ranks share a host).  DFB_WAIT=block restores the blocking wait.
static cudaError_t wait_event(cudaEvent_t ev)
{
	static int mode = -1;
	if (mode < 0)
	{
		const char* e = getenv("DFB_WAIT");
		mode = (e && !strcmp(e, "block")) ? 1 : 0;
	}
	if (mode == 1) return cudaEventSynchronize(ev);
	for (int spins = 0;; spins++)
	{
		const cudaError_t q = cudaEventQuery(ev);
		if (q != cudaErrorNotReady)
		{
			// ("not ready" is an answer, not a failure: it must not be what a later cudaGetLastError() of this thread finds)
			if (spins && q == cudaSuccess) (void)cudaGetLastError();
			return q;
		}
		if (spins < 8) continue;
		struct timespec ts = {0, 30000};
		nanosleep(&ts, nullptr);
	}
}

static void presize_pool(dfb_ctx* ctx, size_t want);

static int set_err(const dfb_ctx* ctx, int code, const char* fmt, ...)
{
	char buf[512];
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(buf, sizeof(buf), fmt, ap);
	va_end(ap);
	if (ctx)
	{
		std::lock_guard<std::mutex> lk(ctx->err_mu);
		ctx->err = buf;
	}
	else g_create_err = buf;
	return code;
}

#define CK(ctx, call)                                                                                  \
	do                                                                                                 \
	{                                                                                                  \
		cudaError_t e__ = (call);                                                                      \
		if (e__ != cudaSuccess)                                                                        \
			return set_err(ctx, DFB_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), \
			               __FILE__, __LINE__);                                                        \
	} while (0)

// Nothing may unwind through the C ABI: allocation failures of the batch-sized host arrays (std::vector, std::thread)
// become DFB_ERR_NOMEM / DFB_ERR_STATE like every other failure.
template <class F>
static int guarded(dfb_ctx* ctx, F f)
{
	try
	{
		return f();
	}
	catch (const std::bad_alloc&)
	{
		return set_err(ctx, DFB_ERR_NOMEM, "out of host memory");
	}
	catch (const std::exception& e)
	{
		return set_err(ctx, DFB_ERR_STATE, "%s", e.what());
	}
	catch (...)
	{
		return set_err(ctx, DFB_ERR_STATE, "unexpected exception");
	}
}

extern "C" int dfb_abi_version(void) { return DFB_ABI_VERSION; }

extern "C" int dfb_device_count(void)
{
	int n = 0;
	cudaError_t e = cudaGetDeviceCount(&n);
	if (e != cudaSuccess)
	{
		set_err(nullptr, DFB_ERR_NODEVICE, "cudaGetDeviceCount failed: %s", cudaGetErrorString(e));
		return -DFB_ERR_NODEVICE;
	}
	return n;
}

extern "C" int dfb_ctx_create(int device_ordinal, dfb_ctx** out)
{
	if (!out) return set_err(nullptr, DFB_ERR_ARG, "dfb_ctx_create: null output pointer");
	*out = nullptr;
	Trace tr;
	int n = 0;
	cudaError_t e = cudaGetDeviceCount(&n);
	tr.lap("ctx: cudaGetDeviceCount");
	if (e != cudaSuccess || n <= 0)
	{
		return set_err(nullptr, DFB_ERR_NODEVICE, "no CUDA device available (%s); this library has no CPU fallback",
		               e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
	}
	if (device_ordinal < 0 || device_ordinal >= n)
	{
		return set_err(nullptr, DFB_ERR_NODEVICE, "device ordinal %d out of range (0..%d)", device_ordinal, n - 1);
	}
	dfb_ctx* ctx = new (std::nothrow) dfb_ctx();
	if (!ctx) return set_err(nullptr, DFB_ERR_NOMEM, "out of host memory");
	ctx->device = device_ordinal;
	e = cudaGetDeviceProperties(&ctx->prop, device_ordinal);
	if (e != cudaSuccess)
	{
		delete ctx;
		return set_err(nullptr, DFB_ERR_CUDA, "cudaGetDeviceProperties failed: %s", cudaGetErrorString(e));
	}
	if (ctx->prop.major != 10)
	{
		int major = ctx->prop.major, minor = ctx->prop.minor;
		delete ctx;
		return set_err(nullptr, DFB_ERR_NODEVICE,
		               "device %d is compute capability %d.%d; the kernels are built for sm_100a only", device_ordinal,
		               major, minor);
	}
	if ((e = cudaSetDevice(device_ordinal)) != cudaSuccess ||
	    (e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking)) != cudaSuccess)
	{
		delete ctx;
		return set_err(nullptr, DFB_ERR_CUDA, "stream creation failed: %s", cudaGetErrorString(e));
	}
	ctx->stream = ctx->own_stream;
	// the upload streams outrank the compute stream: their small kernels (packing, job build) take the first SM slots
	// that a persistent sweep kernel gives back, instead of queueing behind the next sweep's whole grid
	int prio_lo = 0, prio_hi = 0;
	cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
	if ((e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking)) != cudaSuccess ||
	    (e = cudaStreamCreateWithPriority(&ctx->upload_stream, cudaStreamNonBlocking, prio_hi)) != cudaSuccess ||
	    (e = cudaStreamCreateWithPriority(&ctx->upload_stream2, cudaStreamNonBlocking, prio_hi)) != cudaSuccess)
	{
		cudaStreamDestroy(ctx->own_stream);
		delete ctx;
		return set_err(nullptr, DFB_ERR_CUDA, "stream creation failed: %s", cudaGetErrorString(e));
	}
	cudaEventCreateWithFlags(&ctx->copied_ev, cudaEventDisableTiming | cudaEventBlockingSync);
	// keep freed blocks in the stream-ordered pool: a batch re-uses the previous batch's memory
	cudaMemPool_t pool;
	if (cudaDeviceGetDefaultMemPool(&pool, device_ordinal) == cudaSuccess)
	{
		unsigned long long keep = ~0ull;
		cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
	}
	unsigned hc = std::thread::hardware_concurrency();
	ctx->host_threads = (int)std::max(1u, std::min(hc ? hc : 1u, 16u));
	// several contexts share one host (one process per GPU): DFB_HOST_THREADS caps the workers of each
	if (const char* e = getenv("DFB_HOST_THREADS"))
		if (atoi(e) > 0) ctx->host_threads = std::min(atoi(e), 64);
	ctx->pool = new (std::nothrow) HostPool(ctx->host_threads);
	ctx->pool_fetch = new (std::nothrow) HostPool(std::max(2, ctx->host_threads / 2));
	if (const char* e = getenv("DFB_POOL_PRESIZE_MB"))
		if (atoll(e) > 0) presize_pool(ctx, (size_t)atoll(e) << 20);
	tr.lap("ctx: context, streams, pools");
	*out = ctx;
	return DFB_OK;
}

extern "C" void dfb_ctx_destroy(dfb_ctx* ctx)
{
	if (!ctx) return;
	cudaSetDevice(ctx->device);
	if (ctx->last_split) dfb_plan_destroy(ctx->last_split);
	if (ctx->d_records) cudaFreeAsync(ctx->d_records, ctx->stream);
	if (ctx->bt.d_off) cudaFreeAsync(ctx->bt.d_off, ctx->stream);
	for (auto& c : ctx->bt.chunks) cudaFreeAsync(c.first, ctx->stream);
	cudaStreamSynchronize(ctx->stream);
	for (auto& b : ctx->h_in) b.release();
	ctx->h_ring.release();
	for (auto& ev : ctx->ring_ev)
		if (ev) cudaEventDestroy(ev);
	ctx->h_out.release();
	if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
	if (ctx->sweep_arena) cudaFree(ctx->sweep_arena);
	if (ctx->upload_stream) cudaStreamDestroy(ctx->upload_stream);
	if (ctx->upload_stream2) cudaStreamDestroy(ctx->upload_stream2);
	if (ctx->copied_ev) cudaEventDestroy(ctx->copied_ev);
	delete ctx->pool;
	delete ctx->pool_fetch;
	ctx->spare_rows.release();
	ctx->spare_cols.release();
	if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
	delete ctx;
}

extern "C" const char* dfb_last_error(const dfb_ctx* ctx)
{
	return ctx ? ctx->err.c_str() : g_create_err.c_str();
}

extern "C" int dfb_ctx_set_stream(dfb_ctx* ctx, void* cuda_stream)
{
	if (!ctx) return DFB_ERR_ARG;
	ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
	return DFB_OK;
}

extern "C" int dfb_ctx_device_info(const dfb_ctx* ctx, dfb_device_info* info)
{
	if (!ctx || !info) return DFB_ERR_ARG;
	memset(info, 0, sizeof(*info));
	snprintf(info->name, sizeof(info->name), "%s", ctx->prop.name);
	info->ordinal = ctx->device;
	info->sm_count = ctx->prop.multiProcessorCount;
	info->cc_major = ctx->prop.major;
	info->cc_minor = ctx->prop.minor;
	int khz = 0;
	cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, ctx->device);
	info->clock_khz = khz;
	info->total_mem = (int64_t)ctx->prop.totalGlobalMem;
	return DFB_OK;
}

extern "C" int dfb_ctx_memory_info(dfb_ctx* ctx, int reset, int64_t* reserved_now, int64_t* reserved_high, int64_t* used_high)
{
	if (!ctx) return DFB_ERR_ARG;
	cudaMemPool_t pool;
	CK(ctx, cudaDeviceGetDefaultMemPool(&pool, ctx->device));
	unsigned long long now = 0, rhigh = 0, uhigh = 0;
	CK(ctx, cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &now));
	CK(ctx, cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemHigh, &rhigh));
	CK(ctx, cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemHigh, &uhigh));
	if (reserved_now) *reserved_now = (int64_t)now;
	if (reserved_high) *reserved_high = (int64_t)rhigh;
	if (used_high) *used_high = (int64_t)uhigh;
	if (reset)
	{
		unsigned long long zero = 0;
		CK(ctx, cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReservedMemHigh, &zero));
		CK(ctx, cudaMemPoolSetAttribute(pool, cudaMemPoolAttrUsedMemHigh, &zero));
	}
	return DFB_OK;
}

// ------------------------------------------------------------------------------------------
// kernel classes: (lanes per job pair, rows per lane); capacity G*S read rows
// ------------------------------------------------------------------------------------------

// Reads of 81-100 bases go to four-lane groups of 25 rows: exactly 100 rows (eight-lane groups of 13 sweep 104) and half
// the wavefront skew (3 head and tail steps instead of 7), with the per-step fixed cost shared by 25 rows instead of 13.
// -DDFB_NARROW_GROUPS=0 takes the class out (build-time knob for A/B runs; those reads then run at <8,13>).
#ifndef DFB_NARROW_GROUPS
#define DFB_NARROW_GROUPS 1
#endif
#if DFB_NARROW_GROUPS
#define DFB_NARROW_CLASS(X) X(4, 25)
#else
#define DFB_NARROW_CLASS(X)
#endif
#define DFB_CLASSES(X) \
	X(8, 4) X(8, 7) X(8, 10) DFB_NARROW_CLASS(X) X(8, 13) X(8, 16) X(8, 19) X(8, 22) X(8, 25) X(8, 32) \
	X(16, 20) X(16, 25) X(16, 32) X(32, 24) X(32, 32)

struct ClassDef
{
	int G, S;
};
#define X(g, s) {g, s},
static const ClassDef kClasses[] = {DFB_CLASSES(X)};
#undef X
static const int kNumClasses = (int)(sizeof(kClasses) / sizeof(kClasses[0]));
static const int kMaxFastRows = 1024;
static const int kRBins = 1024; // job order inside a class: reference length / 16, longest first

// persistent grid: one CTA per resident slot of every SM (or fewer when the work is less), warps pull job pairs from a queue
template <class K>
static cudaError_t launch_persistent(K kernel, int& occ, int G, const FastParams& p, int sm_count, cudaStream_t stream, int n_items_bound)
{
	if (occ == 0)
	{
		int o = 0;
		cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, kernel, 128, 0);
		if (e != cudaSuccess) return e;
		occ = o > 0 ? o : 1;
	}
	const int per_block = 4 * (32 / G);
	long long want = ((long long)n_items_bound + per_block - 1) / per_block;
	long long cap = (long long)sm_count * occ;
	int grid = (int)std::max(1LL, std::min(want, cap));
	kernel<<<grid, 128, 0, stream>>>(p);
	return cudaGetLastError();
}

template <int G, int S, int MODE>
static cudaError_t launch_fast_t(const FastParams& p, int sm_count, cudaStream_t stream, int n_items_bound)
{
	static int occ = 0;
	return launch_persistent(dp_fast_kernel<G, S, MODE>, occ, G, p, sm_count, stream, n_items_bound);
}

template <int G, int S>
static cudaError_t launch_probe_t(const FastParams& p, int sm_count, cudaStream_t stream, int n_items_bound)
{
	static int occ = 0;
	return launch_persistent(dp_probe_kernel<G, S>, occ, G, p, sm_count, stream, n_items_bound);
}

static cudaError_t launch_fast(int cls, int mode, const FastParams& p, int sm_count, cudaStream_t stream, int bound)
{
	int idx = 0;
#define X(g, s)                                                                                   \
	if (idx++ == cls)                                                                             \
	{                                                                                             \
		if (mode == MODE_SIMPLE) return launch_fast_t<g, s, MODE_SIMPLE>(p, sm_count, stream, bound); \
		if (mode == MODE_SPLIT) return launch_fast_t<g, s, MODE_SPLIT>(p, sm_count, stream, bound);   \
		return launch_probe_t<g, s>(p, sm_count, stream, bound);                                      \
	}
	DFB_CLASSES(X)
#undef X
	return cudaErrorInvalidValue;
}

// ------------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------------

struct ClassWork
{
	int64_t n_jobs = 0;
	JobPair* d_jobs = nullptr; // inside the plan's staged upload
	int* d_ctrl = nullptr;     // [0] cursor, [1] short-window hits, [2] probe cursor, [3] long-window hits (inside plan->d_ctrl)
	int* d_hitq = nullptr;
	int32_t* d_slot_task = nullptr;
	int* d_slot_n = nullptr;
	uint2* d_slot_ev = nullptr;
	uint32_t* d_ntg = nullptr;
	uint32_t* d_rdq = nullptr;
	uint32_t* d_ckpt = nullptr;    // wavefront checkpoints of the first sweep (probe windows resume from them)
	uint32_t* d_slot_rng = nullptr;
	int ckpt_blocks = 0;
	unsigned long long ckpt_words = 0;
	uint32_t max_R = 0;            // longest reference in the class
	FastParams fp;
};

struct dfb_plan
{
	dfb_ctx* ctx = nullptr;
	bool split = false;
	dfb_split_params sp{};
	int64_t n_tasks = 0;
	bool fast_ok[kNumClasses];
	uint32_t bias[kNumClasses];

	// device
	uint8_t* d_raw = nullptr;
	uint8_t* d_stage = nullptr; // descriptors + fast jobs + generic jobs (one upload)
	unsigned long long pool_words = 0, raw_bytes = 0; // allocated sizes of d_pool / d_obytes (entries) and d_raw (bytes)
	uint8_t* d_build = nullptr; // job build on the device: offsets, task arrays, descriptors, bins, jobs (one arena)
	// (device-built plans look a task's read length up in the caller's arrays, which outlive the one-call batch)
	const int64_t* h_read_off = nullptr;
	const int32_t* h_task_read = nullptr;
	int32_t h_read_base = 0;
	// between the two halves of a device build (enqueue: uploads + descriptor / classify kernels; finish: allocations,
	// packing, job scatter once the class counts are back)
	struct BuildPending
	{
		bool active = false;
		SplitBuildParams bp;
		DescParams da, db;
		const SeqDesc* d_desc_a = nullptr;
		const SeqDesc* d_desc_b = nullptr;
		int64_t na = 0, nb = 0, raw_a = 0, raw_b = 0, blocks_a = 0, blocks_b = 0;
		BuildStats* d_stats = nullptr;
		unsigned long long* d_words_a_end = nullptr;
		BuildStats* h_stats = nullptr;
		cudaEvent_t uploaded = nullptr; // behind the chunk's uploads (upload stream)
		cudaEvent_t ready = nullptr;    // behind the read-back of the statistics (blocking-sync: the waiting thread sleeps)
	} pending;
	uint2* d_pool = nullptr;
	uint8_t* d_obytes = nullptr;
	int32_t* d_out = nullptr; // score / best per task
	int32_t* d_task_slot = nullptr; // split: result slot of every task (-1: none), written by the first sweep
	int64_t job_base[kNumClasses] = {0}; // first global slot number of every class
	int* d_ctrl = nullptr;    // all classes' control words
	Event* d_events = nullptr;
	unsigned long long* d_ev_count = nullptr;
	unsigned long long ev_cap = 0;
	// chunks of a pipelined batch hand the first sweep's state (checkpoints, probe targets, read symbols: 6.5 KB per task
	// at dosplitalign's shape) back to the pool right behind their probe sweep, so that the next chunk's allocation reuses it
	bool early_release = false;
	bool sweep_state_released = false;
	bool sweep_in_arena = false; // the three buffers live in ctx->sweep_arena (chunk of a pipelined batch): nothing to free
	ClassWork cls[kNumClasses];
	// generic path
	int64_t n_gen_jobs = 0;
	GenJob* d_gen_jobs = nullptr;
	int* d_gen_ctrl = nullptr; // [0] cursor pass 1, [1] cursor probe
	int32_t* d_gen_rowmax = nullptr;
	uint8_t* d_gen_row_en = nullptr;
	int32_t* d_gen_bnd = nullptr;
	int64_t gen_bnd_stride = 0;
	int gen_grid = 0;
	int* d_gen_probe_flag = nullptr;
	int32_t* d_task_min_score = nullptr;
	int64_t gen_rows_total = 0;
	// result assembly on the device (split): rows / columns of the tasks whose arg-max columns fit their region
	dfb_split_row* d_asm_rows = nullptr;
	int32_t* d_asm_cols = nullptr;
	unsigned long long* d_asm_sums = nullptr; // [blocks][2] + totals[2] behind them
	int64_t asm_blocks = 0;
	int64_t n_fast_tasks = 0;
	bool dev_inputs = false; // tables (and, for a device build, offsets and tasks) are the caller's device memory
	// result holder of dfb_split_align_device: the batch's rows and columns in device memory
	dfb_split_row* d_res_rows = nullptr;
	int32_t* d_res_cols = nullptr;
	int64_t d_res_n_rows = 0, d_res_n_cols = 0;
	bool device_result = false;

	// host
	std::vector<int32_t> task_L; // read length per task (split)
	HostArr<dfb_split_row> rows;
	HostArr<int32_t> cols;
	bool ran = false, fetched = false;
	bool timing = false;
	bool pack_timed = false;
	bool run_timed = false;
	cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
	cudaEvent_t done_ev = nullptr; // recorded behind the last kernel of dfb_plan_run
	cudaStream_t up = nullptr;     // stream of the upload + pack work (the compute stream unless pipelined)
	cudaEvent_t packed_ev = nullptr; // recorded behind the pack kernels when `up` is not the compute stream
	dfb_plan_stats stats{};
};

// -DDFB_BOUNDS_CHECK builds: a range violation recorded by a kernel becomes an error of the call that waits for it
static int bounds_check_status(dfb_ctx* ctx)
{
#ifdef DFB_BOUNDS_CHECK
	int code = 0;
	if (cudaMemcpyFromSymbol(&code, dfb::g_dfb_bounds_err, sizeof(int)) == cudaSuccess && code != 0)
		return set_err(ctx, DFB_ERR_STATE, "device bounds check %d failed", code);
#else
	(void)ctx;
#endif
	return DFB_OK;
}

// Grows the context's stream-ordered pool to `want` reserved bytes in one step (an allocation of the difference, freed at
// once: the release threshold keeps it).  Opt-in (DFB_POOL_PRESIZE_MB, read when the context is created -- the tools
// create theirs on a background thread while they parse their inputs): what a first batch pays for device memory is
// per byte and depends on the box's state -- 5 GB cost 30 ms in one process and 1.1 s in the next on the same box
// (profiles/r04f_first_batch_pool_presize.txt) --, so sizing the pool inside the first call only moves the cost.
static void presize_pool(dfb_ctx* ctx, size_t want)
{
	cudaMemPool_t pool;
	unsigned long long now = 0;
	size_t free_b = 0, total_b = 0;
	if (cudaDeviceGetDefaultMemPool(&pool, ctx->device) != cudaSuccess ||
	    cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &now) != cudaSuccess || cudaMemGetInfo(&free_b, &total_b) != cudaSuccess)
	{
		cudaGetLastError();
		return;
	}
	want = std::min<size_t>(want, (size_t)now + free_b / 2);
	if (want <= (size_t)now + ((size_t)64 << 20)) return;
	Trace tr;
	void* p = nullptr;
	if (cudaMallocAsync(&p, want - (size_t)now, ctx->stream) == cudaSuccess) cudaFreeAsync(p, ctx->stream);
	else cudaGetLastError();
	tr.lap("pool presized");
}

static cudaError_t dalloc(dfb_ctx* ctx, void** p, size_t bytes)
{
	return cudaMallocAsync(p, std::max<size_t>(bytes, 256), ctx->stream);
}
#define DALLOC(ctx, ptr, bytes) CK(ctx, dalloc(ctx, (void**)&(ptr), (bytes)))

template <class T>
static void dfree(dfb_ctx* ctx, T*& p)
{
	if (p) cudaFreeAsync(p, ctx->stream);
	p = nullptr;
}

static void release_device(dfb_plan* plan)
{
	dfb_ctx* ctx = plan->ctx;
	// blocks filled on the plan's upload stream go back to the pool on the compute stream: nothing of this plan may
	// still be in flight there (a plan that failed half way through its creation, for one)
	if (plan->up) cudaStreamSynchronize(plan->up);
	dfree(ctx, plan->d_raw);
	dfree(ctx, plan->d_stage);
	dfree(ctx, plan->d_build);
	dfree(ctx, plan->d_pool);
	dfree(ctx, plan->d_obytes);
	dfree(ctx, plan->d_out);
	dfree(ctx, plan->d_task_slot);
	dfree(ctx, plan->d_ctrl);
	dfree(ctx, plan->d_events);
	dfree(ctx, plan->d_ev_count);
	for (int c = 0; c < kNumClasses; c++)
	{
		ClassWork& cw = plan->cls[c];
		cw.d_jobs = nullptr;
		cw.d_ctrl = nullptr;
		dfree(ctx, cw.d_hitq);
		dfree(ctx, cw.d_slot_task);
		dfree(ctx, cw.d_slot_n);
		dfree(ctx, cw.d_slot_ev);
		if (plan->sweep_in_arena) cw.d_ntg = cw.d_rdq = cw.d_ckpt = nullptr;
		dfree(ctx, cw.d_ntg);
		dfree(ctx, cw.d_rdq);
		dfree(ctx, cw.d_ckpt);
		dfree(ctx, cw.d_slot_rng);
	}
	plan->d_gen_jobs = nullptr;
	dfree(ctx, plan->d_gen_ctrl);
	dfree(ctx, plan->d_gen_rowmax);
	dfree(ctx, plan->d_gen_row_en);
	dfree(ctx, plan->d_gen_bnd);
	dfree(ctx, plan->d_gen_probe_flag);
	dfree(ctx, plan->d_task_min_score);
	dfree(ctx, plan->d_asm_rows);
	dfree(ctx, plan->d_asm_cols);
	dfree(ctx, plan->d_asm_sums);
	dfree(ctx, plan->d_res_rows);
	dfree(ctx, plan->d_res_cols);
}

extern "C" void dfb_plan_destroy(dfb_plan* plan)
{
	if (!plan) return;
	if (plan->ctx)
	{
		cudaSetDevice(plan->ctx->device);
		if (plan->ctx->last_split == plan) plan->ctx->last_split = nullptr;
		release_device(plan);
		// hand the result arrays back for the next batch
		if (plan->rows.cap > plan->ctx->spare_rows.cap) plan->rows.swap(plan->ctx->spare_rows);
		if (plan->cols.cap > plan->ctx->spare_cols.cap) plan->cols.swap(plan->ctx->spare_cols);
	}
	if (plan->pending.ready) cudaEventDestroy(plan->pending.ready);
	if (plan->pending.uploaded) cudaEventDestroy(plan->pending.uploaded);
	if (plan->done_ev) cudaEventDestroy(plan->done_ev);
	if (plan->packed_ev) cudaEventDestroy(plan->packed_ev);
	plan->rows.release();
	plan->cols.release();
	for (int k = 0; k < 3; k++)
		if (plan->ev[k]) cudaEventDestroy(plan->ev[k]);
	delete plan;
}

static int check_table(const dfb_ctx* ctx, const dfb_seq_table* t, const char* what)
{
	if (!t || !t->off || t->n < 0 || (t->n > 0 && !t->bytes && t->off[t->n] > 0))
		return set_err(ctx, DFB_ERR_ARG, "%s: null table", what);
	if (t->off[0] != 0) return set_err(ctx, DFB_ERR_ARG, "%s: off[0] must be 0", what);
	// (internally, views with off[0] != 0 are used for chunks of a table; every size below is off[k] - off[0])
	for (int64_t k = 0; k < t->n; k++)
	{
		const int64_t len = t->off[k + 1] - t->off[k];
		if (len < 0) return set_err(ctx, DFB_ERR_ARG, "%s: offsets decrease at %lld", what, (long long)k);
		if (len > 0x7fffff00LL) return set_err(ctx, DFB_ERR_ARG, "%s: sequence %lld too long", what, (long long)k);
	}
	return DFB_OK;
}

// the same checks over a table of millions of sequences, spread over the context's workers
static int check_table_parallel(const dfb_ctx* ctx, const dfb_seq_table* t, const char* what)
{
	if (!t || !t->off || t->n < (1 << 18)) return check_table(ctx, t, what);
	if (t->n > 0 && !t->bytes && t->off[t->n] > 0) return set_err(ctx, DFB_ERR_ARG, "%s: null table", what);
	if (t->off[0] != 0) return set_err(ctx, DFB_ERR_ARG, "%s: off[0] must be 0", what);
	const int T = (int)std::max<int64_t>(1, std::min<int64_t>(ctx->host_threads, t->n / 262144 + 1));
	std::vector<int64_t> bad((size_t)T, -1);
	parallel_for(ctx->pool, T, [&](int tid) {
		for (int64_t k = t->n * tid / T; k < t->n * (tid + 1) / T; k++)
		{
			const int64_t len = t->off[k + 1] - t->off[k];
			if (len < 0 || len > 0x7fffff00LL)
			{
				bad[(size_t)tid] = k;
				return;
			}
		}
	});
	for (int64_t k : bad)
		if (k >= 0) return check_table(ctx, t, what); // (the sequential pass words the message)
	return DFB_OK;
}

// Scoring triples the s16x2 kernels are exact for (DESIGN.md "number range"):
//   match >= 1, mismatch <= 0, gap <= 0  =>  j*gap <= H(i,j) <= j*match  for every cell,
// so H - match*j fits 16 bits for the class' row capacity.  Everything else goes to s32.
static void classify_params(dfb_plan* pl, int m, int x, int g, bool extra_ok)
{
	for (int c = 0; c < kNumClasses; c++)
	{
		const int rows = kClasses[c].G * kClasses[c].S;
		bool ok = extra_ok && m >= 1 && x <= 0 && g <= 0;
		long long range = (long long)rows * ((long long)m - g) + ((long long)m - x);
		long long B = range + 8;
		if (B > 32000 || B + (long long)m * kClasses[c].S > 32767 || (long long)m * rows > 32767) ok = false;
		pl->fast_ok[c] = ok;
		pl->bias[c] = ok ? (uint32_t)B : 0;
	}
}

static int class_for_rows(int L)
{
	for (int c = 0; c < kNumClasses; c++)
		if (kClasses[c].G * kClasses[c].S >= L) return c;
	return -1;
}

static uint32_t pack2(int v) { return ((uint32_t)v & 0xFFFFu) | ((uint32_t)v << 16); }

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Everything the host builds for one batch, laid out in the pinned staging buffer and
// uploaded with a single copy: [table A descs][table B descs][fast jobs, class by class][generic jobs]
struct Staging
{
	size_t off_desc_a = 0, off_desc_b = 0, off_jobs = 0, off_gen = 0, total = 0;
	void* host = nullptr;
	SeqDesc* desc_a = nullptr;
	SeqDesc* desc_b = nullptr;
	JobPair* jobs = nullptr;
	GenJob* gen = nullptr;
};

static cudaError_t stage_layout(dfb_ctx* ctx, int stage_slot, Staging& st, int64_t na, int64_t nb, int64_t n_fast, int64_t n_gen)
{
	PinnedBuf& hin = ctx->h_in[stage_slot];
	st.off_desc_a = 0;
	st.off_desc_b = align_up(st.off_desc_a + (size_t)na * sizeof(SeqDesc), 256);
	st.off_jobs = align_up(st.off_desc_b + (size_t)nb * sizeof(SeqDesc), 256);
	st.off_gen = align_up(st.off_jobs + (size_t)n_fast * sizeof(JobPair), 256);
	st.total = align_up(st.off_gen + (size_t)n_gen * sizeof(GenJob), 256) + 256;
	cudaError_t e = hin.ensure(st.total);
	if (e != cudaSuccess) return e;
	uint8_t* base = (uint8_t*)hin.p;
	st.host = hin.p;
	st.desc_a = (SeqDesc*)(base + st.off_desc_a);
	st.desc_b = (SeqDesc*)(base + st.off_desc_b);
	st.jobs = (JobPair*)(base + st.off_jobs);
	st.gen = (GenJob*)(base + st.off_gen);
	return cudaSuccess;
}

// word layout of the two tables; returns total words.  Every sequence starts on an even word: the sweep copies
// reference words into shared memory 16 bytes at a time (cp.async)
static uint32_t layout_words(dfb_ctx* ctx, const dfb_seq_table* a, int mode_a, const dfb_seq_table* b, int mode_b, SeqDesc* da,
                             SeqDesc* db, uint32_t* words_a_end, bool* overflow)
{
	// one table: words per range of sequences on every worker, a prefix over the ranges, then the descriptors
	auto one = [&](const dfb_seq_table* t, int mode, SeqDesc* d, int64_t src_base, uint64_t w0) -> uint64_t {
		const int copies = mode == PACK_BOTH ? 2 : 1;
		const int64_t o0 = t->off[0];
		auto words_of = [copies](uint32_t len) -> uint64_t {
			const uint64_t w = (uint64_t)((len + 15) / 16) * (unsigned)copies;
			return w + (w & 1);
		};
		const int T = (int)std::max<int64_t>(1, std::min<int64_t>(ctx->host_threads, t->n / 65536 + 1));
		std::vector<uint64_t> before((size_t)T + 1, 0);
		parallel_for(ctx->pool, T, [&](int tid) {
			uint64_t w = 0;
			for (int64_t k = t->n * tid / T; k < t->n * (tid + 1) / T; k++) w += words_of((uint32_t)(t->off[k + 1] - t->off[k]));
			before[(size_t)tid + 1] = w;
		});
		before[0] = w0;
		for (int k = 0; k < T; k++) before[(size_t)k + 1] += before[(size_t)k];
		parallel_for(ctx->pool, T, [&](int tid) {
			uint64_t w = before[(size_t)tid];
			for (int64_t k = t->n * tid / T; k < t->n * (tid + 1) / T; k++)
			{
				const uint32_t len = (uint32_t)(t->off[k + 1] - t->off[k]);
				d[k].src = 16 + src_base + (t->off[k] - o0);
				d[k].len = len;
				d[k].word = (uint32_t)w;
				w += words_of(len);
			}
		});
		return before[(size_t)T];
	};
	const uint64_t wa = one(a, mode_a, da, 0, 0);
	*words_a_end = (uint32_t)wa;
	const uint64_t w = one(b, mode_b, db, a->off[a->n] - a->off[0], wa);
	*overflow = w >= 0xFFFFFFF0ull;
	return (uint32_t)w;
}

// Host -> device copy of a caller buffer on stream `up`.  Pinned (or registered) memory goes straight to the copy engine;
// pageable memory of a megabyte or more is copied block by block into a ring of pinned blocks by the context's workers,
// each block's transfer queued behind its copy -- the transfer of block i runs under the host copy of block i+1.
static cudaError_t h2d_any(dfb_ctx* ctx, cudaStream_t up, void* dst, const void* src, size_t bytes)
{
	if (bytes == 0) return cudaSuccess;
	bool pageable = false;
	if (bytes >= ((size_t)1 << 20))
	{
		cudaPointerAttributes attr;
		if (cudaPointerGetAttributes(&attr, src) == cudaSuccess) pageable = attr.type == cudaMemoryTypeUnregistered;
		else cudaGetLastError();
	}
	// (one copy engine carries 50 of the link's 55 GB/s on the boxes measured -- scripts/gpu_h2d_rate.py --, so a large
	// pinned upload stays one copy)
	if (!pageable) return cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, up);
	cudaError_t e = ctx->h_ring.ensure(dfb_ctx::kRingSlots * dfb_ctx::kRingBlock);
	if (e != cudaSuccess) return e;
	for (size_t off = 0; off < bytes; off += dfb_ctx::kRingBlock)
	{
		const size_t n = std::min(dfb_ctx::kRingBlock, bytes - off);
		const int slot = (int)(ctx->ring_next++ % dfb_ctx::kRingSlots);
		if (!ctx->ring_ev[slot])
		{
			if ((e = cudaEventCreateWithFlags(&ctx->ring_ev[slot], cudaEventDisableTiming)) != cudaSuccess) return e;
		}
		else if ((e = cudaEventSynchronize(ctx->ring_ev[slot])) != cudaSuccess) return e; // the block's last transfer is over
		uint8_t* stage = (uint8_t*)ctx->h_ring.p + (size_t)slot * dfb_ctx::kRingBlock;
		const uint8_t* from = (const uint8_t*)src + off;
		// (a thread per megabyte of the block; a thread per 512 or 256 KB made the matealign shape from pageable arrays
		// slower, 36 against 32 ms: call r04l)
		const int T = (int)std::max<size_t>(1, std::min<size_t>((size_t)ctx->host_threads, n >> 20));
		parallel_for(ctx->pool, T, [&](int tid) {
			const size_t a = n * (size_t)tid / (size_t)T, b = n * ((size_t)tid + 1) / (size_t)T;
			memcpy(stage + a, from + a, b - a);
		});
		if ((e = cudaMemcpyAsync((uint8_t*)dst + off, stage, n, cudaMemcpyHostToDevice, up)) != cudaSuccess) return e;
		if ((e = cudaEventRecord(ctx->ring_ev[slot], up)) != cudaSuccess) return e;
	}
	return cudaSuccess;
}

// Starts the copy of the raw sequence bytes before the host builds descriptors and jobs: with pinned
// caller buffers the transfer runs underneath that host work.  `dev_range` (device-resident tables): the bytes are
// device memory, [a0, a1) of table A's and [b0, b1) of table B's; they are copied device to device (the pack kernel
// reads whole 16-byte windows, so it never reads the caller's allocation itself).
static int upload_raw(dfb_plan* pl, const dfb_seq_table* a, const dfb_seq_table* b, const int64_t* dev_range = nullptr)
{
	dfb_ctx* ctx = pl->ctx;
	cudaStream_t up = pl->up ? pl->up : ctx->stream;
	const int64_t a0 = dev_range ? dev_range[0] : a->off[0], b0 = dev_range ? dev_range[2] : b->off[0];
	const int64_t na = (dev_range ? dev_range[1] : a->off[a->n]) - a0, nb = (dev_range ? dev_range[3] : b->off[b->n]) - b0;
	// 16 bytes of slack in front, 32 behind (the pack kernel reads whole 16-byte windows)
	CK(ctx, cudaMallocAsync((void**)&pl->d_raw, std::max<size_t>(256, (size_t)(na + nb + 48)), up));
	pl->raw_bytes = (unsigned long long)(na + nb + 48);
	if (dev_range)
	{
		if (na) CK(ctx, cudaMemcpyAsync(pl->d_raw + 16, a->bytes + a0, (size_t)na, cudaMemcpyDeviceToDevice, up));
		if (nb) CK(ctx, cudaMemcpyAsync(pl->d_raw + 16 + na, b->bytes + b0, (size_t)nb, cudaMemcpyDeviceToDevice, up));
		return DFB_OK;
	}
	if (na) CK(ctx, h2d_any(ctx, up, pl->d_raw + 16, a->bytes + a0, (size_t)na));
	if (nb) CK(ctx, h2d_any(ctx, up, pl->d_raw + 16 + na, b->bytes + b0, (size_t)nb));
	return DFB_OK;
}

static int upload_and_pack(dfb_plan* pl, const dfb_seq_table* a, int mode_a, const dfb_seq_table* b, int mode_b,
                           const Staging& st, uint32_t words_a_end, uint32_t total_words)
{
	dfb_ctx* ctx = pl->ctx;
	cudaStream_t up = pl->up ? pl->up : ctx->stream;
	const int64_t na = a->off[a->n] - a->off[0], nb = b->off[b->n] - b->off[0];
	CK(ctx, cudaMallocAsync((void**)&pl->d_stage, std::max<size_t>(256, st.total), up));
	CK(ctx, cudaMemcpyAsync(pl->d_stage, st.host, st.total, cudaMemcpyHostToDevice, up));
	// (slack: a 16-byte copy may take the word behind a sequence's last one)
	CK(ctx, cudaMallocAsync((void**)&pl->d_pool, ((size_t)total_words + 8) * sizeof(uint2), up));
	CK(ctx, cudaMallocAsync((void**)&pl->d_obytes, ((size_t)total_words + 8) * 16, up));
	pl->pool_words = (unsigned long long)total_words + 8;
	for (int k = 0; k < 3; k++)
		if (!pl->ev[k]) CK(ctx, cudaEventCreate(&pl->ev[k]));
	CK(ctx, cudaEventRecord(pl->ev[0], up));
	const SeqDesc* d_da = (const SeqDesc*)(pl->d_stage + st.off_desc_a);
	const SeqDesc* d_db = (const SeqDesc*)(pl->d_stage + st.off_desc_b);
	const int max_grid = ctx->prop.multiProcessorCount * 16;
	auto launch = [&](int mode, const SeqDesc* d, int64_t n, uint32_t w0, uint32_t w1) -> cudaError_t {
		if (n == 0 || w1 <= w0) return cudaSuccess;
		const int grid = (int)std::min<uint64_t>(((uint64_t)n * 16 + 255) / 256, (uint64_t)max_grid); // sixteen lanes per sequence
		if (mode == PACK_FWD)
			pack_kernel<PACK_FWD><<<grid, 256, 0, up>>>(pl->d_raw, d, (int)n, pl->d_pool, pl->d_obytes, pl->pool_words, pl->raw_bytes);
		else if (mode == PACK_REV_ODD)
			pack_kernel<PACK_REV_ODD><<<grid, 256, 0, up>>>(pl->d_raw, d, (int)n, pl->d_pool, pl->d_obytes, pl->pool_words, pl->raw_bytes);
		else
			pack_kernel<PACK_BOTH><<<grid, 256, 0, up>>>(pl->d_raw, d, (int)n, pl->d_pool, pl->d_obytes, pl->pool_words, pl->raw_bytes);
		return cudaGetLastError();
	};
	CK(ctx, launch(mode_a, d_da, a->n, 0, words_a_end));
	CK(ctx, launch(mode_b, d_db, b->n, words_a_end, total_words));
	CK(ctx, cudaEventRecord(pl->ev[1], up));
	pl->pack_timed = true;
	if (up != ctx->stream)
	{
		if (!pl->packed_ev) CK(ctx, cudaEventCreateWithFlags(&pl->packed_ev, cudaEventDisableTiming));
		CK(ctx, cudaEventRecord(pl->packed_ev, up));
	}
	pl->stats.h2d_bytes += (pl->dev_inputs ? 0 : na + nb) + (int64_t)st.total;
	pl->stats.raw_bytes = na * (mode_a == PACK_BOTH ? 2 : 1) + nb * (mode_b == PACK_BOTH ? 2 : 1);
	pl->stats.packed_bytes = (int64_t)total_words * 8;
	return DFB_OK;
}

static void fill_fast_params(dfb_plan* pl, int c, int m, int x, int g, int min_split)
{
	ClassWork& cw = pl->cls[c];
	FastParams& fp = cw.fp;
	memset(&fp, 0, sizeof(fp));
	fp.pool = pl->d_pool;
	fp.obytes = pl->d_obytes;
	fp.jobs = cw.d_jobs;
	fp.n_jobs = (int)cw.n_jobs;
	fp.m = m;
	fp.bias = pl->bias[c];
	fp.xm = (uint32_t)(x - m);
	fp.g2 = pack2(g);
	fp.gm2 = pack2(g - m);
	fp.min_split = min_split;
	fp.out = pl->d_out;
	fp.hit_count = cw.d_ctrl + 1;
	fp.hit_count_long = cw.d_ctrl + 3;
	fp.hitq = cw.d_hitq;
	fp.slot_task = cw.d_slot_task;
	fp.task_slot = pl->d_task_slot;
	fp.slot_base = (int)pl->job_base[c];
	fp.slot_ev = cw.d_slot_ev;
	fp.slot_n = cw.d_slot_n;
	fp.ntg = cw.d_ntg;
	fp.rdq = cw.d_rdq;
	fp.ckpt = cw.d_ckpt;
	fp.ckpt_blocks = cw.ckpt_blocks;
	fp.ckpt_words = cw.ckpt_words;
	fp.pool_words = pl->pool_words;
	fp.n_tasks = pl->n_tasks;
	// probe granules: 16 mask bits per half cover checkpoint blocks 0 .. ckpt_blocks
	fp.gran_shift = 0;
	while ((cw.ckpt_blocks >> fp.gran_shift) > 15) fp.gran_shift++;
	fp.slot_rng = cw.d_slot_rng;
	fp.events = pl->d_events;
	fp.ev_count = pl->d_ev_count;
	fp.ev_cap = pl->ev_cap;
	for (int k = 0; k < 32; k++) fp.ck[k] = pack2(m * (k + 1));
}

// device-side bookkeeping common to both plan kinds, after the job counts are known
static int alloc_work(dfb_plan* pl, JobPair* d_jobs_base, GenJob* d_gen_base, const int64_t* n_jobs_cls, bool split, uint32_t gen_max_R)
{
	dfb_ctx* ctx = pl->ctx;
	DALLOC(ctx, pl->d_ctrl, kNumClasses * 4 * sizeof(int));
	int64_t first = 0;
	size_t arena_need = 0;
	pl->sweep_in_arena = split && pl->early_release;
	for (int c = 0; c < kNumClasses; c++)
	{
		ClassWork& cw = pl->cls[c];
		cw.n_jobs = n_jobs_cls[c];
		cw.d_jobs = d_jobs_base + first;
		cw.d_ctrl = pl->d_ctrl + 4 * c;
		pl->job_base[c] = first;
		first += cw.n_jobs;
		pl->stats.fast_jobs += cw.n_jobs;
		if (split && cw.n_jobs)
		{
			const size_t n = (size_t)cw.n_jobs;
			DALLOC(ctx, cw.d_hitq, n * sizeof(int));
			DALLOC(ctx, cw.d_slot_task, n * sizeof(int32_t));
			DALLOC(ctx, cw.d_slot_n, n * sizeof(int));
			DALLOC(ctx, cw.d_slot_ev, n * DFB_SLOT_EVENTS * sizeof(uint2));
			DALLOC(ctx, cw.d_slot_rng, n * sizeof(uint32_t));
			// checkpoints every CK = ckpt_steps(G) steps of the wavefront (R + G - 1 steps)
			const int G = kClasses[c].G, CK = ckpt_steps(G);
			const size_t gs_bytes = n * (size_t)G * kClasses[c].S * sizeof(uint32_t);
			cw.ckpt_blocks = (int)(((int64_t)cw.max_R + G - 2) / CK);
			size_t ck_bytes = n * (size_t)cw.ckpt_blocks * (size_t)(kClasses[c].S + 2) * G * sizeof(uint32_t);
			if (!(cw.ckpt_blocks > 0 && ck_bytes <= (size_t)ctx->prop.totalGlobalMem / 4))
			{
				cw.ckpt_blocks = 0;
				ck_bytes = 0;
			}
			cw.ckpt_words = ck_bytes / sizeof(uint32_t);
			if (pl->sweep_in_arena)
			{
				// offsets now, pointers once the arena is known to hold every class
				cw.d_ntg = (uint32_t*)(uintptr_t)arena_need;
				arena_need = align_up(arena_need + gs_bytes, 256);
				cw.d_rdq = (uint32_t*)(uintptr_t)arena_need;
				arena_need = align_up(arena_need + gs_bytes, 256);
				cw.d_ckpt = (uint32_t*)(uintptr_t)arena_need;
				arena_need = align_up(arena_need + ck_bytes, 256);
			}
			else
			{
				DALLOC(ctx, cw.d_ntg, gs_bytes);
				DALLOC(ctx, cw.d_rdq, gs_bytes);
				if (ck_bytes) DALLOC(ctx, cw.d_ckpt, ck_bytes);
			}
		}
	}
	if (pl->sweep_in_arena)
	{
		if (arena_need > ctx->sweep_arena_cap)
		{
			// (stream-ordered on the compute stream like every use of it: the previous chunk's sweeps are done with the old
			// buffer when it goes)
			if (ctx->sweep_arena) cudaFreeAsync(ctx->sweep_arena, ctx->stream);
			ctx->sweep_arena = nullptr;
			ctx->sweep_arena_cap = 0;
			const size_t want = arena_need + arena_need / 8;
			CK(ctx, cudaMallocAsync((void**)&ctx->sweep_arena, want, ctx->stream));
			ctx->sweep_arena_cap = want;
		}
		for (int c = 0; c < kNumClasses; c++)
		{
			ClassWork& cw = pl->cls[c];
			if (!cw.n_jobs) continue;
			cw.d_ntg = (uint32_t*)(ctx->sweep_arena + (uintptr_t)cw.d_ntg);
			cw.d_rdq = (uint32_t*)(ctx->sweep_arena + (uintptr_t)cw.d_rdq);
			cw.d_ckpt = cw.ckpt_words ? (uint32_t*)(ctx->sweep_arena + (uintptr_t)cw.d_ckpt) : nullptr;
		}
	}
	if (pl->n_gen_jobs)
	{
		const size_t n = (size_t)pl->n_gen_jobs;
		pl->d_gen_jobs = d_gen_base;
		DALLOC(ctx, pl->d_gen_ctrl, 4 * sizeof(int));
		pl->gen_bnd_stride = (int64_t)gen_max_R + 2;
		pl->gen_grid = (int)std::min<size_t>((n + 3) / 4, (size_t)ctx->prop.multiProcessorCount * 4);
		DALLOC(ctx, pl->d_gen_bnd, (size_t)pl->gen_grid * 4 * 2 * pl->gen_bnd_stride * sizeof(int32_t));
		if (split)
		{
			DALLOC(ctx, pl->d_gen_rowmax, (size_t)std::max<int64_t>(pl->gen_rows_total, 1) * sizeof(int32_t));
			DALLOC(ctx, pl->d_gen_row_en, (size_t)std::max<int64_t>(pl->gen_rows_total, 1));
			CK(ctx, cudaMemsetAsync(pl->d_gen_row_en, 0, (size_t)std::max<int64_t>(pl->gen_rows_total, 1), ctx->stream));
			DALLOC(ctx, pl->d_gen_probe_flag, (n / 2 + 1) * sizeof(int));
		}
		pl->stats.generic_jobs += (int64_t)n;
	}
	DALLOC(ctx, pl->d_out, (size_t)std::max<int64_t>(pl->n_tasks, 1) * sizeof(int32_t));
	CK(ctx, cudaMemsetAsync(pl->d_out, 0, (size_t)std::max<int64_t>(pl->n_tasks, 1) * sizeof(int32_t), ctx->stream));
	if (split) DALLOC(ctx, pl->d_task_slot, (size_t)std::max<int64_t>(pl->n_tasks, 1) * sizeof(int32_t));
	if (split && first > 0)
	{
		// a task assembled on the device has at most DFB_SLOT_EVENTS columns, hence at most half as many rows
		pl->n_fast_tasks = first;
		pl->asm_blocks = (pl->n_tasks + DFB_ASM_BLOCK - 1) / DFB_ASM_BLOCK;
		DALLOC(ctx, pl->d_asm_rows, (size_t)first * (DFB_SLOT_EVENTS / 2) * sizeof(dfb_split_row));
		DALLOC(ctx, pl->d_asm_cols, (size_t)first * DFB_SLOT_EVENTS * sizeof(int32_t));
		DALLOC(ctx, pl->d_asm_sums, ((size_t)pl->asm_blocks + 1) * 2 * sizeof(unsigned long long));
	}
	return DFB_OK;
}

static int finish_create(dfb_plan* pl)
{
	dfb_ctx* ctx = pl->ctx;
	CK(ctx, cudaStreamSynchronize(ctx->stream));
	if (pl->pack_timed)
	{
		float ms = 0;
		if (cudaEventElapsedTime(&ms, pl->ev[0], pl->ev[1]) == cudaSuccess) pl->stats.ms_pack = ms;
	}
	return DFB_OK;
}

// ---- job lists built on the host ------------------------------------------------------------------

// One builder for both aligners (`simple`: SimpleAligner).  Table A holds the references (simple) or two windows per
// cluster (split), table B the sequences or reads; task_a / task_b name an entry of each, task_min_score is null for
// simple, whose `params` carry the scoring triple only.  Either table may be a view into a larger one (off[0] != 0)
// whose first entry is number `a_base` / `b_base` of the caller's numbering.  `up_stream` null: uploads on the compute
// stream and a final synchronisation; else uploads on `up_stream` and none (chunks of a pipelined batch).
static int plan_create_host(dfb_ctx* ctx, bool simple, const dfb_split_params* params, const dfb_seq_table* A,
                            const dfb_seq_table* B, const int32_t* task_a, const int32_t* task_b, const int32_t* task_min_score,
                            int64_t n_tasks, int32_t a_base, int32_t b_base, int stage_slot, cudaStream_t up_stream, dfb_plan** out,
                            bool bytes_on_device = false)
{
	*out = nullptr;
	int rc;
	CK(ctx, cudaSetDevice(ctx->device));
	dfb_plan* pl = new (std::nothrow) dfb_plan();
	if (!pl) return set_err(ctx, DFB_ERR_NOMEM, "out of host memory");
	auto fail = [&](int code) {
		dfb_plan_destroy(pl);
		return code;
	};
	pl->ctx = ctx;
	pl->split = !simple;
	pl->early_release = !simple && up_stream; // (a chunk of a pipelined batch: its sweep state lives in the context's arena)
	pl->sp = *params;
	pl->n_tasks = n_tasks;
	pl->stats.n_tasks = n_tasks;
	classify_params(pl, params->match, params->mismatch, params->gap, simple || (params->end_gaps == 0 && params->min_split_score >= 1));
	pl->up = up_stream;
	pl->dev_inputs = bytes_on_device;
	Trace tr;
	const int64_t range[4] = {A->off[0], A->off[A->n], B->off[0], B->off[B->n]};
	if ((rc = upload_raw(pl, A, B, bytes_on_device ? range : nullptr))) return fail(rc);
	tr.lap("host build: raw upload");

	// pass 1 (host threads): class and reference-length bin of every task, per-thread bin counts
	const int64_t n_a = simple ? A->n : A->n / 2; // references / clusters
	const int T = (int)std::max<int64_t>(1, std::min<int64_t>(ctx->host_threads, n_tasks / 65536 + 1));
	const size_t n_bins = (size_t)kNumClasses * kRBins;
	std::vector<int32_t> bin_of((size_t)n_tasks);
	std::vector<int64_t> bin_pos(n_bins * (size_t)T, 0); // [thread][bin]
	if (!simple) pl->task_L.resize((size_t)n_tasks);
	struct Part
	{
		int64_t cells = 0, n_gen = 0, bad = -1;
		uint32_t gen_max_R = 0;
		uint32_t cls_max_R[kNumClasses] = {0};
	};
	std::vector<Part> part((size_t)T);
	parallel_for(ctx->pool, T, [&](int tid) {
		Part& pt = part[(size_t)tid];
		int64_t* cnt = bin_pos.data() + n_bins * (size_t)tid;
		for (int64_t t = n_tasks * tid / T; t < n_tasks * (tid + 1) / T; t++)
		{
			const int64_t ia = (int64_t)task_a[t] - a_base, ib = (int64_t)task_b[t] - b_base;
			if (ia < 0 || ia >= n_a || ib < 0 || ib >= B->n)
			{
				if (pt.bad < 0) pt.bad = t;
				bin_of[t] = -1;
				continue;
			}
			// simple: the reference (R1); split: both windows, the longer one decides the bin and the class limit
			const int64_t a0 = simple ? ia : 2 * ia;
			const int64_t R1 = A->off[a0 + 1] - A->off[a0];
			const int64_t R2 = simple ? 0 : A->off[a0 + 2] - A->off[a0 + 1];
			const int64_t R = std::max(R1, R2);
			const int64_t L = B->off[ib + 1] - B->off[ib];
			if (!simple) pl->task_L[t] = (int32_t)L;
			pt.cells += (R1 + R2) * L;
			// no DP cell -- simple: score 0 (d_out is zero-initialised); split: an empty read, every row maximum is 0, no
			// split (SplitReadAligner.cpp:224-227)
			int32_t bin = -1;
			if (L > 0 && (R > 0 || !simple))
			{
				int c = (L <= kMaxFastRows && R <= 65535) ? class_for_rows((int)L) : -1;
				if (c >= 0 && !pl->fast_ok[c]) c = -1;
				if (c < 0)
				{
					bin = -2;
					pt.n_gen++;
					pt.gen_max_R = std::max<uint32_t>(pt.gen_max_R, (uint32_t)R);
				}
				else
				{
					bin = c * kRBins + (kRBins - 1 - (int)std::min<int64_t>(R >> 4, kRBins - 1));
					cnt[bin]++;
					pt.cls_max_R[c] = std::max<uint32_t>(pt.cls_max_R[c], (uint32_t)R);
				}
			}
			bin_of[t] = bin;
		}
	});
	int64_t n_gen_tasks = 0;
	uint32_t gen_max_R = 0;
	for (int k = 0; k < T; k++)
	{
		if (part[(size_t)k].bad >= 0) return fail(set_err(ctx, DFB_ERR_ARG, "task %lld: table index out of range", (long long)part[(size_t)k].bad));
		pl->stats.cells += part[(size_t)k].cells;
		n_gen_tasks += part[(size_t)k].n_gen;
		gen_max_R = std::max(gen_max_R, part[(size_t)k].gen_max_R);
		for (int c = 0; c < kNumClasses; c++) pl->cls[c].max_R = std::max(pl->cls[c].max_R, part[(size_t)k].cls_max_R[c]);
	}
	// counts -> positions inside the class: class by class, bin by bin, thread by thread (keeps task order inside a bin).
	// Simple: two tasks share a job (low / high half), task position p -> job p/2, half p%2.  Split: a job per task.
	int64_t n_jobs_cls[kNumClasses], job_base[kNumClasses];
	int64_t n_fast_jobs = 0;
	for (int c = 0; c < kNumClasses; c++)
	{
		int64_t tasks_c = 0;
		for (int bb = 0; bb < kRBins; bb++)
			for (int k = 0; k < T; k++)
			{
				int64_t& slot = bin_pos[n_bins * (size_t)k + (size_t)c * kRBins + bb];
				const int64_t cnt = slot;
				slot = tasks_c;
				tasks_c += cnt;
			}
		job_base[c] = n_fast_jobs;
		n_jobs_cls[c] = simple ? (tasks_c + 1) / 2 : tasks_c;
		n_fast_jobs += n_jobs_cls[c];
	}
	const int64_t gen_per_task = simple ? 1 : 2; // split: one generic job per window
	tr.lap("host build: classify");

	Staging st;
	cudaError_t e = stage_layout(ctx, stage_slot, st, A->n, B->n, n_fast_jobs, gen_per_task * n_gen_tasks);
	if (e != cudaSuccess) return fail(set_err(ctx, DFB_ERR_NOMEM, "pinned staging buffer: %s", cudaGetErrorString(e)));
	// split: reference 1 of every cluster forward, reference 2 reversed (SplitReadAligner.cpp:80-81); every read forward
	// and reversed (:84-85)
	const int mode_a = simple ? PACK_FWD : PACK_REV_ODD, mode_b = simple ? PACK_FWD : PACK_BOTH;
	uint32_t words_a_end = 0;
	bool overflow = false;
	const uint32_t total_words = layout_words(ctx, A, mode_a, B, mode_b, st.desc_a, st.desc_b, &words_a_end, &overflow);
	if (overflow) return fail(set_err(ctx, DFB_ERR_ARG, "batch too large: more than 2^32 packed words; split it"));
	tr.lap("host build: layout");
	// pass 2 (host threads): every task into its job slot
	if (simple)
		parallel_for(ctx->pool, T, [&](int tid) {
			for (int64_t j = n_fast_jobs * tid / T; j < n_fast_jobs * (tid + 1) / T; j++)
			{
				JobPair& jp = st.jobs[j];
				memset(&jp, 0, sizeof(jp));
				jp.out0 = jp.out1 = -1;
			}
		});
	parallel_for(ctx->pool, T, [&](int tid) {
		int64_t* pos = bin_pos.data() + n_bins * (size_t)tid;
		for (int64_t t = n_tasks * tid / T; t < n_tasks * (tid + 1) / T; t++)
		{
			const int32_t bin = bin_of[t];
			if (bin < 0) continue;
			const int64_t ia = (int64_t)task_a[t] - a_base;
			const SeqDesc& bd = st.desc_b[task_b[t] - b_base];
			const int64_t p = pos[bin]++;
			const int64_t j0 = job_base[bin / kRBins];
			if (simple)
			{
				JobPair& jp = st.jobs[j0 + (p >> 1)];
				const int h = (int)(p & 1);
				jp.ref_w[h] = st.desc_a[ia].word;
				jp.read_w[h] = bd.word;
				jp.R[h] = (uint16_t)st.desc_a[ia].len;
				jp.L[h] = (uint16_t)bd.len;
				if (h == 0) jp.out0 = (int32_t)t; else jp.out1 = (int32_t)t;
			}
			else
			{
				JobPair& jp = st.jobs[j0 + p];
				jp.ref_w[0] = st.desc_a[2 * ia].word;
				jp.ref_w[1] = st.desc_a[2 * ia + 1].word;
				jp.read_w[0] = bd.word;
				jp.read_w[1] = bd.word + (bd.len + 15) / 16;
				jp.R[0] = (uint16_t)st.desc_a[2 * ia].len;
				jp.R[1] = (uint16_t)st.desc_a[2 * ia + 1].len;
				jp.L[0] = jp.L[1] = (uint16_t)bd.len;
				jp.out0 = (int32_t)t;
				jp.out1 = task_min_score[t];
			}
		}
	});
	int64_t gi = 0;
	for (int64_t t = 0; n_gen_tasks && t < n_tasks; t++)
	{
		if (bin_of[t] != -2) continue;
		const int64_t ia = (int64_t)task_a[t] - a_base;
		const SeqDesc& bd = st.desc_b[task_b[t] - b_base];
		for (int h = 0; h < gen_per_task; h++)
		{
			const SeqDesc& ad = st.desc_a[simple ? ia : 2 * ia + h];
			GenJob& j = st.gen[gi++];
			j.ref_w = ad.word;
			j.read_w = h ? bd.word + (bd.len + 15) / 16 : bd.word;
			j.R = ad.len;
			j.L = bd.len;
			j.task = (int32_t)t;
			j.half = h;
			j.row_off = 0;
			if (!simple)
			{
				// (split: the row maxima of both windows, one row list per job)
				j.row_off = pl->gen_rows_total;
				pl->gen_rows_total += (int64_t)j.L + 1;
			}
		}
	}
	pl->n_gen_jobs = gi;
	tr.lap("host build: jobs");

	rc = upload_and_pack(pl, A, mode_a, B, mode_b, st, words_a_end, total_words);
	tr.lap("host build: enqueue h2d+pack");
	if (!rc && !simple)
	{
		pl->ev_cap = (unsigned long long)std::max<int64_t>(n_tasks, 1 << 20);
		cudaError_t e2 = dalloc(ctx, (void**)&pl->d_events, (size_t)pl->ev_cap * sizeof(Event));
		if (e2 == cudaSuccess) e2 = dalloc(ctx, (void**)&pl->d_ev_count, sizeof(unsigned long long));
		if (e2 == cudaSuccess && n_gen_tasks)
		{
			e2 = dalloc(ctx, (void**)&pl->d_task_min_score, (size_t)n_tasks * sizeof(int32_t));
			if (e2 == cudaSuccess)
				e2 = cudaMemcpyAsync(pl->d_task_min_score, task_min_score, (size_t)n_tasks * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream);
			pl->stats.h2d_bytes += n_tasks * (int64_t)sizeof(int32_t);
		}
		if (e2 != cudaSuccess) rc = set_err(ctx, DFB_ERR_CUDA, "output allocation failed: %s", cudaGetErrorString(e2));
	}
	if (!rc) rc = alloc_work(pl, (JobPair*)(pl->d_stage + st.off_jobs), (GenJob*)(pl->d_stage + st.off_gen), n_jobs_cls, !simple, gen_max_R);
	if (!rc)
	{
		for (int c = 0; c < kNumClasses; c++)
			if (pl->cls[c].n_jobs)
				fill_fast_params(pl, c, params->match, params->mismatch, params->gap, simple ? 0 : params->min_split_score);
		tr.lap("host build: alloc");
		if (!up_stream) rc = finish_create(pl);
		tr.lap("host build: sync");
	}
	if (rc) return fail(rc);
	*out = pl;
	return DFB_OK;
}

// The argument checks of a batch, shared by the resident plan and the one-call form of each aligner
static int check_simple_args(dfb_ctx* ctx, const dfb_simple_params* params, const dfb_seq_table* refs, const dfb_seq_table* seqs,
                             const int32_t* task_ref, const int32_t* task_seq, int64_t n_tasks)
{
	if (!params || n_tasks < 0 || (n_tasks > 0 && (!task_ref || !task_seq)))
		return set_err(ctx, DFB_ERR_ARG, "dfb_simple_plan_create: null argument");
	int rc;
	if ((rc = check_table_parallel(ctx, refs, "refs")) || (rc = check_table_parallel(ctx, seqs, "seqs"))) return rc;
	if (n_tasks > 0x7fffff00LL) return set_err(ctx, DFB_ERR_ARG, "too many tasks in one batch");
	return DFB_OK;
}

static int check_split_args(dfb_ctx* ctx, const dfb_split_params* params, const dfb_seq_table* refs, const dfb_seq_table* reads,
                            const int32_t* task_cluster, const int32_t* task_read, const int32_t* task_min_score, int64_t n_tasks)
{
	if (!params || n_tasks < 0 || (n_tasks > 0 && (!task_cluster || !task_read || !task_min_score)))
		return set_err(ctx, DFB_ERR_ARG, "dfb_split_plan_create: null argument");
	int rc;
	if ((rc = check_table_parallel(ctx, refs, "refs")) || (rc = check_table_parallel(ctx, reads, "reads"))) return rc;
	if (refs->n & 1) return set_err(ctx, DFB_ERR_ARG, "refs must hold two windows per cluster (n is odd)");
	if (n_tasks > 0x7fffff00LL) return set_err(ctx, DFB_ERR_ARG, "too many tasks in one batch");
	return DFB_OK;
}

static int dfb_simple_plan_create_body(dfb_ctx* ctx, const dfb_simple_params* params, const dfb_seq_table* refs,
                                      const dfb_seq_table* seqs, const int32_t* task_ref, const int32_t* task_seq,
                                      int64_t n_tasks, dfb_plan** out)
{
	if (!ctx) return DFB_ERR_ARG;
	if (!out) return set_err(ctx, DFB_ERR_ARG, "dfb_simple_plan_create: null argument");
	*out = nullptr;
	if (int rc = check_simple_args(ctx, params, refs, seqs, task_ref, task_seq, n_tasks)) return rc;
	const dfb_split_params sp{params->match, params->mismatch, params->gap, 0, 0};
	return plan_create_host(ctx, true, &sp, refs, seqs, task_ref, task_seq, nullptr, n_tasks, 0, 0, 0, nullptr, out);
}

static int dfb_split_plan_create_body(dfb_ctx* ctx, const dfb_split_params* params, const dfb_seq_table* refs,
                                     const dfb_seq_table* reads, const int32_t* task_cluster, const int32_t* task_read,
                                     const int32_t* task_min_score, int64_t n_tasks, dfb_plan** out)
{
	if (!ctx) return DFB_ERR_ARG;
	if (!out) return set_err(ctx, DFB_ERR_ARG, "dfb_split_plan_create: null argument");
	*out = nullptr;
	if (int rc = check_split_args(ctx, params, refs, reads, task_cluster, task_read, task_min_score, n_tasks)) return rc;
	return plan_create_host(ctx, false, params, refs, reads, task_cluster, task_read, task_min_score, n_tasks, 0, 0, 0, nullptr, out);
}

// ---- job lists built on the device (dfb_build.cuh) ----------------------------------------------------------
// Chunks of a pipelined batch of either aligner (`simple`, tables and tasks as for plan_create_host): the caller's
// offsets and task arrays are uploaded as they are; descriptors, class / length bins and the 32-byte job records are
// made by kernels.  One small read-back (jobs per class, longest reference per class, total pool words) separates the
// classify pass from the allocations that depend on it.  device_build_finish returns DFB_BUILD_ON_HOST when the chunk
// holds tasks only the s32 kernels can take: the caller builds that chunk on the host instead.
static const int DFB_BUILD_ON_HOST = 1000;

// The uploads go on ctx->upload_stream for every chunk.  The upload streams carry copies only, so one stream serves every
// chunk in order and chunk 0's upload has the link to itself (two alternating streams share it: the first sweep of a
// batch started 0.4 ms later on the split path, 5 ms later at the matealign shape).
static int device_build_enqueue(dfb_ctx* ctx, bool simple, const dfb_split_params* params, const dfb_seq_table* refs,
                                const dfb_seq_table* reads, const int32_t* task_cluster, const int32_t* task_read,
                                const int32_t* task_min_score, int64_t n_tasks, int32_t ref_base, int32_t read_base, int stage_slot,
                                dfb_plan** out, const int64_t* dev_range = nullptr)
{
	static_assert(kNumClasses <= DFB_BUILD_MAX_CLASSES && kRBins == DFB_BUILD_RBINS, "dfb_build.cuh tables");
	*out = nullptr;
	int rc;
	CK(ctx, cudaSetDevice(ctx->device));
	dfb_plan* pl = new (std::nothrow) dfb_plan();
	if (!pl) return set_err(ctx, DFB_ERR_NOMEM, "out of host memory");
	pl->ctx = ctx;
	pl->split = !simple;
	pl->early_release = !simple; // (always a chunk of a pipelined batch)
	pl->sp = *params;
	pl->n_tasks = n_tasks;
	pl->stats.n_tasks = n_tasks;
	// (dev_range: every input is device memory -- offsets, tasks, bytes --, [off[0], off[n]) of either table given)
	pl->dev_inputs = dev_range != nullptr;
	pl->h_read_off = dev_range ? nullptr : reads->off;
	pl->h_task_read = dev_range ? nullptr : task_read;
	pl->h_read_base = read_base;
	classify_params(pl, params->match, params->mismatch, params->gap, simple || (params->end_gaps == 0 && params->min_split_score >= 1));
	pl->up = ctx->upload_stream;
	cudaStream_t up = pl->up;
	auto fail = [&](int code) {
		dfb_plan_destroy(pl);
		return code;
	};
	Trace tr;
	if ((rc = upload_raw(pl, refs, reads, dev_range))) return fail(rc);

	// arena
	const int64_t na = refs->n, nb = reads->n;
	const size_t n_bins = (size_t)kNumClasses * kRBins;
	const int64_t blocks_a = (na + DFB_BUILD_BLOCK * DFB_BUILD_ITEMS - 1) / (DFB_BUILD_BLOCK * DFB_BUILD_ITEMS);
	const int64_t blocks_b = (nb + DFB_BUILD_BLOCK * DFB_BUILD_ITEMS - 1) / (DFB_BUILD_BLOCK * DFB_BUILD_ITEMS);
	size_t at = 0;
	auto take = [&](size_t bytes) {
		const size_t o = at;
		at = align_up(at + bytes, 256);
		return o;
	};
	const size_t o_off_a = take((size_t)(na + 1) * 8), o_off_b = take((size_t)(nb + 1) * 8);
	const size_t o_tc = take((size_t)n_tasks * 4), o_tr = take((size_t)n_tasks * 4), o_tm = take((size_t)n_tasks * 4);
	const size_t o_desc_a = take((size_t)na * sizeof(SeqDesc)), o_desc_b = take((size_t)nb * sizeof(SeqDesc));
	const size_t o_bin_of = take((size_t)n_tasks * 4);
	const size_t o_bins = take(2 * n_bins * 4);
	const size_t o_sums_a = take((size_t)(blocks_a + 1) * 8), o_sums_b = take((size_t)(blocks_b + 1) * 8);
	const size_t o_stats = take(sizeof(BuildStats) + 64);
	const size_t o_jobs = take(((size_t)n_tasks + 2 * kNumClasses) * sizeof(JobPair)); // (simple: ceil(tasks / 2) per class)
	CK(ctx, cudaMallocAsync((void**)&pl->d_build, std::max<size_t>(at, 256), up));
	uint8_t* base = pl->d_build;
	BuildStats* d_stats = (BuildStats*)(base + o_stats);
	unsigned long long* d_words_a_end = (unsigned long long*)(base + o_stats + sizeof(BuildStats));
	int* d_bad_table = &d_stats->bad_table;
	// pinned scratch: the initial statistics go up from it, the final ones come back into it
	PinnedBuf& hin = ctx->h_in[stage_slot];
	{
		cudaError_t e = hin.ensure(2 * sizeof(BuildStats) + 64);
		if (e != cudaSuccess) return fail(set_err(ctx, DFB_ERR_NOMEM, "pinned staging buffer: %s", cudaGetErrorString(e)));
	}
	BuildStats* h_init = (BuildStats*)hin.p;
	BuildStats* h_stats = h_init + 1;
	memset(h_init, 0, sizeof(*h_init));
	h_init->bad_task = ~0ull;
	auto cuda_fail = [&](cudaError_t e, const char* what) {
		return fail(set_err(ctx, DFB_ERR_CUDA, "%s failed: %s", what, cudaGetErrorString(e)));
	};
	cudaError_t e;
	if ((e = cudaMemcpyAsync(d_stats, h_init, sizeof(BuildStats), cudaMemcpyHostToDevice, up)) != cudaSuccess) return cuda_fail(e, "statistics upload");
	const cudaMemcpyKind kind = dev_range ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
	if ((e = cudaMemcpyAsync(base + o_off_a, refs->off, (size_t)(na + 1) * 8, kind, up)) != cudaSuccess ||
	    (e = cudaMemcpyAsync(base + o_off_b, reads->off, (size_t)(nb + 1) * 8, kind, up)) != cudaSuccess ||
	    (e = cudaMemcpyAsync(base + o_tc, task_cluster, (size_t)n_tasks * 4, kind, up)) != cudaSuccess ||
	    (e = cudaMemcpyAsync(base + o_tr, task_read, (size_t)n_tasks * 4, kind, up)) != cudaSuccess ||
	    (!simple && (e = cudaMemcpyAsync(base + o_tm, task_min_score, (size_t)n_tasks * 4, kind, up)) != cudaSuccess))
		return cuda_fail(e, "task upload");
	const int64_t raw_a = dev_range ? dev_range[1] - dev_range[0] : refs->off[refs->n] - refs->off[0];
	// descriptors: windows (one stored copy each), then reads (forward + reversed copy)
	DescParams da;
	da.off = (const int64_t*)(base + o_off_a);
	da.n = na;
	da.copies = 1;
	da.src_base = 0;
	da.desc = (SeqDesc*)(base + o_desc_a);
	da.block_sums = (unsigned long long*)(base + o_sums_a);
	da.word_base = nullptr;
	da.total = d_words_a_end;
	da.bad = d_bad_table;
	DescParams db = da;
	db.off = (const int64_t*)(base + o_off_b);
	db.n = nb;
	db.copies = simple ? 1 : 2;
	db.src_base = raw_a;
	db.desc = (SeqDesc*)(base + o_desc_b);
	db.block_sums = (unsigned long long*)(base + o_sums_b);
	db.word_base = d_words_a_end;
	db.total = &d_stats->total_words;
	SplitBuildParams bp;
	memset(&bp, 0, sizeof(bp));
	bp.desc_a = da.desc;
	bp.n_clusters = simple ? na : na / 2;
	bp.simple = simple ? 1 : 0;
	bp.ref_base = ref_base;
	bp.desc_b = db.desc;
	bp.n_reads = nb;
	bp.task_cluster = (const int32_t*)(base + o_tc);
	bp.task_read = (const int32_t*)(base + o_tr);
	bp.task_min_score = (const int32_t*)(base + o_tm);
	bp.n_tasks = n_tasks;
	bp.read_base = read_base;
	bp.bin_of = (int32_t*)(base + o_bin_of);
	bp.bin_count = (unsigned int*)(base + o_bins);
	bp.bin_fill = bp.bin_count + n_bins;
	bp.n_classes = kNumClasses;
	for (int c = 0; c < kNumClasses; c++)
	{
		bp.cls_rows[c] = kClasses[c].G * kClasses[c].S;
		bp.cls_ok[c] = pl->fast_ok[c] ? 1 : 0;
	}
	bp.max_fast_rows = kMaxFastRows;
	bp.stats = d_stats;
	bp.jobs = (JobPair*)(base + o_jobs);
	if ((e = cudaEventCreateWithFlags(&pl->pending.uploaded, trace_on() ? cudaEventDefault : cudaEventDisableTiming)) != cudaSuccess ||
	    (e = cudaEventRecord(pl->pending.uploaded, up)) != cudaSuccess)
		return cuda_fail(e, "cudaEventRecord");
	pl->pending.active = true;
	pl->pending.bp = bp;
	pl->pending.da = da;
	pl->pending.db = db;
	pl->pending.d_desc_a = da.desc;
	pl->pending.d_desc_b = db.desc;
	pl->pending.na = na;
	pl->pending.nb = nb;
	pl->pending.blocks_a = blocks_a;
	pl->pending.blocks_b = blocks_b;
	pl->pending.raw_a = raw_a;
	pl->pending.raw_b = dev_range ? dev_range[3] - dev_range[2] : reads->off[reads->n] - reads->off[0];
	pl->pending.d_stats = d_stats;
	pl->pending.d_words_a_end = d_words_a_end;
	pl->pending.h_stats = h_stats;
	tr.lap("device build: uploads queued");
	*out = pl;
	return DFB_OK;
}

// The build kernels of a chunk, on the COMPUTE stream: the sweeps are persistent grids that fill every SM, so a chain
// of small dependent kernels on another stream would wait for a kernel boundary per link.  Queued between the first
// sweep and the probe sweep of the previous chunk, the chain costs the GPU a few tens of microseconds and its class
// counts are back on the host long before that chunk's probe sweep ends.
static int device_build_kernels(dfb_plan* pl)
{
	dfb_ctx* ctx = pl->ctx;
	cudaStream_t cs = ctx->stream;
	auto& pd = pl->pending;
	CK(ctx, cudaStreamWaitEvent(cs, pd.uploaded, 0));
	// (a memset is a kernel: on the upload stream it would wait for an SM the persistent sweeps hold, and the copies
	// queued behind it with it -- the upload streams carry copies only)
	CK(ctx, cudaMemsetAsync(pd.bp.bin_count, 0, 2 * (size_t)kNumClasses * kRBins * 4, cs));
	if (pd.na)
	{
		desc_count_kernel<<<(unsigned)pd.blocks_a, DFB_BUILD_BLOCK, 0, cs>>>(pd.da);
		desc_scan_kernel<<<1, DFB_BUILD_BLOCK, 0, cs>>>(pd.da.block_sums, pd.blocks_a, pd.da.word_base, pd.da.total);
		desc_write_kernel<<<(unsigned)pd.blocks_a, DFB_BUILD_BLOCK, 0, cs>>>(pd.da);
	}
	else CK(ctx, cudaMemsetAsync(pd.d_words_a_end, 0, 8, cs));
	if (pd.nb)
	{
		desc_count_kernel<<<(unsigned)pd.blocks_b, DFB_BUILD_BLOCK, 0, cs>>>(pd.db);
		desc_scan_kernel<<<1, DFB_BUILD_BLOCK, 0, cs>>>(pd.db.block_sums, pd.blocks_b, pd.db.word_base, pd.db.total);
		desc_write_kernel<<<(unsigned)pd.blocks_b, DFB_BUILD_BLOCK, 0, cs>>>(pd.db);
	}
	else CK(ctx, cudaMemcpyAsync(&pd.d_stats->total_words, pd.d_words_a_end, 8, cudaMemcpyDeviceToDevice, cs));
	const unsigned task_blocks = (unsigned)((pl->n_tasks + DFB_BUILD_BLOCK - 1) / DFB_BUILD_BLOCK);
	if (pl->n_tasks) split_classify_kernel<<<task_blocks, DFB_BUILD_BLOCK, 0, cs>>>(pd.bp);
	bin_scan_kernel<<<1, 1024, 0, cs>>>(pd.bp.bin_count, kNumClasses, pd.d_stats);
	stats_to_host_kernel<<<1, 64, 0, cs>>>(pd.d_stats, pd.h_stats); // (pinned host memory is device-accessible under UVA)
	CK(ctx, cudaGetLastError());
	if (!pd.ready) CK(ctx, cudaEventCreateWithFlags(&pd.ready, cudaEventDisableTiming | cudaEventBlockingSync));
	CK(ctx, cudaEventRecord(pd.ready, cs));
	return DFB_OK;
}

// second half: the class counts are back (or will be: the wait sleeps); everything that depends on them
static int device_build_finish(dfb_plan* pl)
{
	dfb_ctx* ctx = pl->ctx;
	const dfb_split_params* params = &pl->sp;
	cudaStream_t up = ctx->stream; // (packing and the job scatter run on the compute stream, in front of the chunk's sweeps)
	auto fail = [&](int code) { return code; }; // (the caller destroys the plan)
	auto cuda_fail = [&](cudaError_t e, const char* what) {
		return set_err(ctx, DFB_ERR_CUDA, "%s failed: %s", what, cudaGetErrorString(e));
	};
	Trace tr;
	cudaError_t e;
	if ((e = wait_event(pl->pending.ready)) != cudaSuccess) return cuda_fail(e, "job build");
	pl->pending.active = false;
	const SplitBuildParams bp = pl->pending.bp;
	const int64_t na = pl->pending.na, nb = pl->pending.nb, raw_a = pl->pending.raw_a, raw_b = pl->pending.raw_b;
	const int64_t n_tasks = pl->n_tasks;
	const BuildStats* h_stats = pl->pending.h_stats;
	const unsigned task_blocks = (unsigned)((n_tasks + DFB_BUILD_BLOCK - 1) / DFB_BUILD_BLOCK);
	int rc;
	tr.lap("device build: classify done");
	if (h_stats->bad_table) return fail(set_err(ctx, DFB_ERR_ARG, "a table's offsets decrease or a sequence is too long"));
	if (h_stats->bad_task != ~0ull) return fail(set_err(ctx, DFB_ERR_ARG, "task %llu: table index out of range", h_stats->bad_task));
	if (h_stats->n_gen) return fail(DFB_BUILD_ON_HOST);
	if (h_stats->total_words >= 0xFFFFFFF0ull) return fail(set_err(ctx, DFB_ERR_ARG, "batch too large: more than 2^32 packed words; split it"));
	pl->stats.cells = (int64_t)h_stats->cells;
	const uint32_t total_words = (uint32_t)h_stats->total_words;
	int64_t n_jobs_cls[kNumClasses];
	for (int c = 0; c < kNumClasses; c++)
	{
		n_jobs_cls[c] = h_stats->cls_jobs[c];
		pl->cls[c].max_R = h_stats->cls_max_R[c];
	}
	// pool, packing, job scatter: still on the upload stream, underneath the previous chunk's sweeps
	if ((e = cudaMallocAsync((void**)&pl->d_pool, ((size_t)total_words + 8) * sizeof(uint2), up)) != cudaSuccess ||
	    (e = cudaMallocAsync((void**)&pl->d_obytes, ((size_t)total_words + 8) * 16, up)) != cudaSuccess)
		return fail(set_err(ctx, DFB_ERR_NOMEM, "packed pool of %u words: %s", total_words, cudaGetErrorString(e)));
	pl->pool_words = (unsigned long long)total_words + 8;
	for (int k = 0; k < 3; k++)
		if (!pl->ev[k] && (e = cudaEventCreate(&pl->ev[k])) != cudaSuccess) return cuda_fail(e, "cudaEventCreate");
	cudaEventRecord(pl->ev[0], up);
	const int max_grid = ctx->prop.multiProcessorCount * 16;
	const bool simple = bp.simple != 0;
	const int grid_a = (int)std::min<uint64_t>(((uint64_t)na * 16 + 255) / 256, (uint64_t)max_grid);
	const int grid_b = (int)std::min<uint64_t>(((uint64_t)nb * 16 + 255) / 256, (uint64_t)max_grid);
	if (na && simple) pack_kernel<PACK_FWD><<<grid_a, 256, 0, up>>>(pl->d_raw, pl->pending.d_desc_a, (int)na, pl->d_pool, pl->d_obytes, pl->pool_words, pl->raw_bytes);
	if (na && !simple) pack_kernel<PACK_REV_ODD><<<grid_a, 256, 0, up>>>(pl->d_raw, pl->pending.d_desc_a, (int)na, pl->d_pool, pl->d_obytes, pl->pool_words, pl->raw_bytes);
	if (nb && simple) pack_kernel<PACK_FWD><<<grid_b, 256, 0, up>>>(pl->d_raw, pl->pending.d_desc_b, (int)nb, pl->d_pool, pl->d_obytes, pl->pool_words, pl->raw_bytes);
	if (nb && !simple) pack_kernel<PACK_BOTH><<<grid_b, 256, 0, up>>>(pl->d_raw, pl->pending.d_desc_b, (int)nb, pl->d_pool, pl->d_obytes, pl->pool_words, pl->raw_bytes);
	cudaEventRecord(pl->ev[1], up);
	pl->pack_timed = true;
	if (simple)
	{
		// two tasks per job: jobs per class = ceil(tasks / 2); the scatter needs the first task position and first job of a class
		SplitBuildParams sb = bp;
		unsigned int first_task = 0, first_job = 0;
		for (int c = 0; c < kNumClasses; c++)
		{
			sb.cls_first_task[c] = first_task;
			sb.cls_first_job[c] = first_job;
			first_task += h_stats->cls_jobs[c];
			n_jobs_cls[c] = ((int64_t)h_stats->cls_jobs[c] + 1) / 2;
			first_job += (unsigned int)n_jobs_cls[c];
		}
		if (first_job) jobs_init_kernel<<<(unsigned)((first_job + DFB_BUILD_BLOCK - 1) / DFB_BUILD_BLOCK), DFB_BUILD_BLOCK, 0, up>>>(bp.jobs, (long long)first_job);
		if (n_tasks) simple_scatter_kernel<<<task_blocks, DFB_BUILD_BLOCK, 0, up>>>(sb);
	}
	else if (n_tasks) split_scatter_kernel<<<task_blocks, DFB_BUILD_BLOCK, 0, up>>>(bp);
	if ((e = cudaGetLastError()) != cudaSuccess) return cuda_fail(e, "pack / scatter kernels");
	if (pl->dev_inputs)
	{
		// (the statistics, both ways, are all that crosses)
		pl->stats.h2d_bytes += (int64_t)sizeof(BuildStats);
		pl->stats.d2h_bytes += (int64_t)sizeof(BuildStats);
	}
	else pl->stats.h2d_bytes += raw_a + raw_b + (na + 1 + nb + 1) * 8 + n_tasks * 12 + (int64_t)sizeof(BuildStats);
	pl->stats.raw_bytes = raw_a + (simple ? 1 : 2) * raw_b;
	pl->stats.packed_bytes = (int64_t)total_words * 8;

	if (!simple)
	{
		pl->ev_cap = (unsigned long long)std::max<int64_t>(n_tasks, 1 << 20);
		if ((e = dalloc(ctx, (void**)&pl->d_events, (size_t)pl->ev_cap * sizeof(Event))) != cudaSuccess ||
		    (e = dalloc(ctx, (void**)&pl->d_ev_count, sizeof(unsigned long long))) != cudaSuccess)
			return fail(set_err(ctx, DFB_ERR_CUDA, "output allocation failed: %s", cudaGetErrorString(e)));
	}
	if ((rc = alloc_work(pl, bp.jobs, nullptr, n_jobs_cls, !simple, 0))) return fail(rc);
	for (int c = 0; c < kNumClasses; c++)
		if (pl->cls[c].n_jobs) fill_fast_params(pl, c, params->match, params->mismatch, params->gap, simple ? 0 : params->min_split_score);
	tr.lap("device build: pack, scatter, alloc");
	return DFB_OK;
}

// ---- run / fetch -------------------------------------------------------------------------------

static GenParams gen_params(dfb_plan* pl, int cursor_slot)
{
	GenParams gp;
	memset(&gp, 0, sizeof(gp));
	gp.pool = pl->d_pool;
	gp.obytes = pl->d_obytes;
	gp.jobs = pl->d_gen_jobs;
	gp.n_jobs = (int)pl->n_gen_jobs;
	gp.cursor = pl->d_gen_ctrl + cursor_slot;
	gp.m = pl->sp.match;
	gp.x = pl->sp.mismatch;
	gp.g = pl->sp.gap;
	gp.end_gaps = pl->split ? pl->sp.end_gaps : 0;
	gp.out = pl->d_out;
	gp.rowmax = pl->d_gen_rowmax;
	gp.row_en = pl->d_gen_row_en;
	gp.probe_flag = pl->d_gen_probe_flag;
	gp.bnd = pl->d_gen_bnd;
	gp.bnd_stride = pl->gen_bnd_stride;
	gp.events = pl->d_events;
	gp.ev_count = pl->d_ev_count;
	gp.ev_cap = pl->ev_cap;
	return gp;
}

static int run_probe(dfb_plan* pl)
{
	dfb_ctx* ctx = pl->ctx;
	const int sm = ctx->prop.multiProcessorCount;
	CK(ctx, cudaMemsetAsync(pl->d_ev_count, 0, sizeof(unsigned long long), ctx->stream));
	for (int c = 0; c < kNumClasses; c++)
	{
		ClassWork& cw = pl->cls[c];
		if (!cw.n_jobs) continue;
		CK(ctx, cudaMemsetAsync(cw.d_ctrl + 2, 0, sizeof(int), ctx->stream));
		CK(ctx, cudaMemsetAsync(cw.d_slot_n, 0, (size_t)cw.n_jobs * sizeof(int), ctx->stream));
		FastParams fp = cw.fp;
		fp.cursor = cw.d_ctrl + 2;
		fp.events = pl->d_events;
		fp.ev_cap = pl->ev_cap;
		CK(ctx, launch_fast(c, MODE_PROBE, fp, sm, ctx->stream, (int)cw.n_jobs));
		pl->stats.kernel_launches++;
	}
	if (pl->n_gen_jobs)
	{
		CK(ctx, cudaMemsetAsync(pl->d_gen_ctrl + 1, 0, sizeof(int), ctx->stream));
		GenParams gp = gen_params(pl, 1);
		dp_generic_kernel<MODE_PROBE><<<pl->gen_grid, 128, 0, ctx->stream>>>(gp);
		CK(ctx, cudaGetLastError());
		pl->stats.kernel_launches++;
	}
	return DFB_OK;
}

// rows and column lists of the tasks whose arg-max columns all sit in their region, in task order (dfb_assemble.cuh)
static int run_assemble(dfb_plan* pl)
{
	dfb_ctx* ctx = pl->ctx;
	if (!pl->d_asm_rows) return DFB_OK;
	static_assert(kNumClasses <= DFB_ASM_MAX_CLASSES, "AsmParams class tables too small");
	AsmParams ap;
	memset(&ap, 0, sizeof(ap));
	ap.n_tasks = pl->n_tasks;
	ap.task_slot = pl->d_task_slot;
	ap.n_classes = kNumClasses;
	for (int c = 0; c < kNumClasses; c++)
	{
		const ClassWork& cw = pl->cls[c];
		ap.job_base[c] = pl->job_base[c];
		ap.slot_n[c] = cw.d_slot_n;
		ap.slot_ev[c] = cw.d_slot_ev;
		ap.hitq[c] = cw.d_hitq;
		ap.jobs[c] = cw.d_jobs;
	}
	ap.job_base[kNumClasses] = pl->n_fast_tasks;
	ap.block_sums = pl->d_asm_sums;
	ap.totals = pl->d_asm_sums + 2 * (size_t)pl->asm_blocks;
	ap.rows = pl->d_asm_rows;
	ap.cols = pl->d_asm_cols;
	ap.events = pl->d_events;
	ap.ev_count = pl->d_ev_count;
	ap.ev_cap = pl->ev_cap;
	ap.rows_cap = (unsigned long long)pl->n_fast_tasks * (DFB_SLOT_EVENTS / 2);
	ap.cols_cap = (unsigned long long)pl->n_fast_tasks * DFB_SLOT_EVENTS;
	asm_count_kernel<<<(unsigned)pl->asm_blocks, DFB_ASM_BLOCK, 0, ctx->stream>>>(ap);
	asm_scan_kernel<<<1, 1024, 0, ctx->stream>>>(ap.block_sums, pl->asm_blocks, ap.totals);
	asm_write_kernel<<<(unsigned)pl->asm_blocks, DFB_ASM_BLOCK, 0, ctx->stream>>>(ap);
	CK(ctx, cudaGetLastError());
	pl->stats.kernel_launches += 3;
	return DFB_OK;
}

// `between_sweeps`: work queued on the compute stream behind the first sweep and in front of the probe sweep (the
// pipelined batch puts the next chunk's job-build kernels there)
static int plan_run_impl(dfb_plan* pl, const std::function<int()>* between_sweeps)
{
	if (!pl) return DFB_ERR_ARG;
	dfb_ctx* ctx = pl->ctx;
	if (!pl->d_pool) return set_err(ctx, DFB_ERR_STATE, "plan's device buffers were released");
	CK(ctx, cudaSetDevice(ctx->device));
	const int sm = ctx->prop.multiProcessorCount;
	pl->stats.kernel_launches = 0;
	pl->fetched = false;
	pl->run_timed = false;
	if (pl->packed_ev) CK(ctx, cudaStreamWaitEvent(ctx->stream, pl->packed_ev, 0));
	if (pl->timing)
	{
		for (int k = 0; k < 3; k++)
			if (!pl->ev[k]) CK(ctx, cudaEventCreate(&pl->ev[k]));
		CK(ctx, cudaEventRecord(pl->ev[0], ctx->stream));
	}
	CK(ctx, cudaMemsetAsync(pl->d_ctrl, 0, kNumClasses * 4 * sizeof(int), ctx->stream));
	if (pl->split) CK(ctx, cudaMemsetAsync(pl->d_task_slot, 0xff, (size_t)std::max<int64_t>(pl->n_tasks, 1) * sizeof(int32_t), ctx->stream));
	for (int c = 0; c < kNumClasses; c++)
	{
		ClassWork& cw = pl->cls[c];
		if (!cw.n_jobs) continue;
		FastParams fp = cw.fp;
		fp.cursor = cw.d_ctrl;
		CK(ctx, launch_fast(c, pl->split ? MODE_SPLIT : MODE_SIMPLE, fp, sm, ctx->stream, (int)cw.n_jobs));
		pl->stats.kernel_launches++;
	}
	if (pl->n_gen_jobs)
	{
		CK(ctx, cudaMemsetAsync(pl->d_gen_ctrl, 0, 4 * sizeof(int), ctx->stream));
		GenParams gp = gen_params(pl, 0);
		if (pl->split)
		{
			dp_generic_kernel<MODE_SPLIT><<<pl->gen_grid, 128, 0, ctx->stream>>>(gp);
			CK(ctx, cudaGetLastError());
			GenReduceParams rp;
			rp.jobs = pl->d_gen_jobs;
			rp.n_tasks = (int)(pl->n_gen_jobs / 2);
			rp.task_min_score = pl->d_task_min_score;
			rp.min_split = pl->sp.min_split_score;
			rp.rowmax = pl->d_gen_rowmax;
			rp.row_en = pl->d_gen_row_en;
			rp.out_best = pl->d_out;
			rp.probe_flag = pl->d_gen_probe_flag;
			split_reduce_generic_kernel<<<(rp.n_tasks + 127) / 128, 128, 0, ctx->stream>>>(rp);
			CK(ctx, cudaGetLastError());
			pl->stats.kernel_launches += 2;
		}
		else
		{
			dp_generic_kernel<MODE_SIMPLE><<<pl->gen_grid, 128, 0, ctx->stream>>>(gp);
			CK(ctx, cudaGetLastError());
			pl->stats.kernel_launches++;
		}
	}
	if (pl->timing) CK(ctx, cudaEventRecord(pl->ev[1], ctx->stream));
	if (between_sweeps)
	{
		int rc = (*between_sweeps)();
		if (rc) return rc;
	}
	if (pl->split)
	{
		int rc = run_probe(pl);
		if (!rc && pl->early_release)
		{
			for (int c = 0; c < kNumClasses; c++)
			{
				ClassWork& cw = pl->cls[c];
				if (pl->sweep_in_arena) cw.d_ckpt = cw.d_ntg = cw.d_rdq = nullptr; // (the next chunk takes the arena over)
				dfree(ctx, cw.d_ckpt);
				dfree(ctx, cw.d_ntg);
				dfree(ctx, cw.d_rdq);
				cw.fp.ckpt = cw.fp.ntg = cw.fp.rdq = nullptr;
			}
			pl->sweep_state_released = true;
		}
		if (!rc) rc = run_assemble(pl);
		if (rc) return rc;
	}
	if (pl->timing)
	{
		CK(ctx, cudaEventRecord(pl->ev[2], ctx->stream));
		pl->run_timed = true;
	}
	// (blocking-sync event: the thread that waits for a chunk's kernels sleeps instead of spinning on a core the other
	// lanes -- or the other ranks of the host -- could use)
	if (!pl->done_ev) CK(ctx, cudaEventCreateWithFlags(&pl->done_ev, cudaEventDisableTiming | cudaEventBlockingSync));
	CK(ctx, cudaEventRecord(pl->done_ev, ctx->stream));
	pl->ran = true;
	return DFB_OK;
}

static int dfb_plan_run_body(dfb_plan* pl) { return plan_run_impl(pl, nullptr); }

extern "C" int dfb_plan_sync(dfb_plan* pl)
{
	if (!pl) return DFB_ERR_ARG;
	dfb_ctx* ctx = pl->ctx;
	CK(ctx, cudaSetDevice(ctx->device));
	CK(ctx, cudaStreamSynchronize(ctx->stream));
	if (int brc = bounds_check_status(ctx)) return brc;
	if (pl->run_timed)
	{
		float a = 0, b = 0;
		CK(ctx, cudaEventElapsedTime(&a, pl->ev[0], pl->ev[1]));
		CK(ctx, cudaEventElapsedTime(&b, pl->ev[1], pl->ev[2]));
		pl->stats.ms_sweep = a;
		pl->stats.ms_probe = b;
	}
	return DFB_OK;
}

extern "C" int dfb_plan_set_timing(dfb_plan* pl, int enable)
{
	if (!pl) return DFB_ERR_ARG;
	pl->timing = enable != 0;
	return DFB_OK;
}

extern "C" int dfb_simple_plan_fetch(dfb_plan* pl, int32_t* out_score)
{
	if (!pl) return DFB_ERR_ARG;
	dfb_ctx* ctx = pl->ctx;
	if (pl->split) return set_err(ctx, DFB_ERR_STATE, "dfb_simple_plan_fetch on a split plan");
	if (!pl->ran) return set_err(ctx, DFB_ERR_STATE, "dfb_simple_plan_fetch before dfb_plan_run");
	if (!out_score && pl->n_tasks) return set_err(ctx, DFB_ERR_ARG, "null output");
	CK(ctx, cudaSetDevice(ctx->device));
	if (pl->n_tasks)
		CK(ctx, cudaMemcpyAsync(out_score, pl->d_out, (size_t)pl->n_tasks * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
	CK(ctx, cudaStreamSynchronize(ctx->stream));
	if (int brc = bounds_check_status(ctx)) return brc;
	pl->stats.d2h_bytes = pl->n_tasks * (int64_t)sizeof(int32_t);
	pl->fetched = true;
	return DFB_OK;
}

// ---- split result assembly ---------------------------------------------------------------------

namespace
{
struct Chunk
{
	std::vector<dfb_split_row> rows;
	std::vector<int32_t> cols;
};

inline uint64_t wide_key(int half, int row, int col) { return ((uint64_t)half << 62) | ((uint64_t)row << 31) | (uint64_t)col; }
inline int key_row(uint64_t k) { return (int)((k >> 31) & 0x7fffffff); }

// rows of one task from its events sorted by (matrix, row, column): the nested loops of
// SplitReadAligner.cpp:233-269 walk tie rows, then columns1, then columns2, all ascending
void emit_task_rows(int task, int L, const uint64_t* key, const int32_t* score, int n, Chunk& out)
{
	int n0 = 0;
	while (n0 < n && (key[n0] >> 62) == 0) n0++;
	int i = 0;
	while (i < n0)
	{
		const int a = key_row(key[i]);
		int i_end = i;
		while (i_end < n0 && key_row(key[i_end]) == a) i_end++;
		const int want = L - a;
		int j = n0;
		while (j < n && key_row(key[j]) != want) j++;
		if (j < n)
		{
			int j_end = j;
			while (j_end < n && key_row(key[j_end]) == want) j_end++;
			dfb_split_row row;
			row.task = task;
			row.read_split = a;
			row.score1 = score[i];
			row.score2 = score[j];
			row.col_begin = (int64_t)out.cols.size();
			row.n1 = i_end - i;
			row.n2 = j_end - j;
			for (int k = i; k < i_end; k++) out.cols.push_back((int32_t)(key[k] & 0x7fffffff));
			for (int k = j; k < j_end; k++) out.cols.push_back((int32_t)(key[k] & 0x7fffffff));
			out.rows.push_back(row);
		}
		i = i_end;
	}
}
}  // namespace

// where a chunk of a pipelined batch leaves its rows: straight behind the previous chunks' in the batch's result arrays
struct ResultSink
{
	HostArr<dfb_split_row>* rows;
	HostArr<int32_t>* cols;
	size_t row_base, col_base; // filled so far
	int32_t task_shift;        // first task of the chunk in the batch's numbering
};

static int split_fetch_impl(dfb_plan* pl, int32_t* out_best, int64_t* n_rows, int64_t* n_cols, HostPool* pool, ResultSink* sink = nullptr);

static int dfb_split_plan_fetch_body(dfb_plan* pl, int32_t* out_best, int64_t* n_rows, int64_t* n_cols)
{
	if (!pl) return DFB_ERR_ARG;
	return split_fetch_impl(pl, out_best, n_rows, n_cols, pl->ctx->pool);
}

// Step 1 of a split fetch, once the plan's kernels are done (`cs` waits for them): the overflow-list length, the
// winning tasks per class (h_ctrl) and the row / column totals of the region assembly.  When the probe sweep found more
// arg-max columns than the overflow list holds, the list is sized exactly and the sweep run again.
static int fetch_counters(dfb_plan* pl, cudaStream_t cs, int* h_ctrl, unsigned long long* n_ov_out, unsigned long long* asm_totals)
{
	dfb_ctx* ctx = pl->ctx;
	unsigned long long n_ov = 0;
	for (int attempt = 0;; attempt++)
	{
		CK(ctx, cudaMemcpyAsync(&n_ov, pl->d_ev_count, sizeof(n_ov), cudaMemcpyDeviceToHost, cs));
		CK(ctx, cudaMemcpyAsync(h_ctrl, pl->d_ctrl, kNumClasses * 4 * sizeof(int), cudaMemcpyDeviceToHost, cs));
		if (pl->d_asm_sums)
			CK(ctx, cudaMemcpyAsync(asm_totals, pl->d_asm_sums + 2 * (size_t)pl->asm_blocks, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, cs));
		CK(ctx, cudaStreamSynchronize(cs));
		if (n_ov <= pl->ev_cap) break;
		if (attempt >= 2) return set_err(ctx, DFB_ERR_STATE, "event buffer overflow persists");
		// the probe sweep found more arg-max columns than the overflow list holds: size it exactly, redo the sweep
		dfree(ctx, pl->d_events);
		pl->ev_cap = n_ov + 1024;
		cudaError_t e = dalloc(ctx, (void**)&pl->d_events, (size_t)pl->ev_cap * sizeof(Event));
		if (e != cudaSuccess) return set_err(ctx, DFB_ERR_NOMEM, "event buffer of %llu entries: %s", pl->ev_cap, cudaGetErrorString(e));
		int rc;
		if (pl->sweep_state_released)
		{
			// (a chunk of a pipelined batch gave its checkpoints back behind the probe sweep: both sweeps again)
			pl->early_release = pl->sweep_state_released = pl->sweep_in_arena = false; // (buffers of its own this time)
			for (int c = 0; c < kNumClasses; c++)
			{
				ClassWork& cw = pl->cls[c];
				if (!cw.n_jobs) continue;
				const size_t n = (size_t)cw.n_jobs, gs = (size_t)kClasses[c].G * kClasses[c].S;
				DALLOC(ctx, cw.d_ntg, n * gs * sizeof(uint32_t));
				DALLOC(ctx, cw.d_rdq, n * gs * sizeof(uint32_t));
				if (cw.ckpt_blocks > 0) DALLOC(ctx, cw.d_ckpt, cw.ckpt_words * sizeof(uint32_t));
				cw.fp.ntg = cw.d_ntg;
				cw.fp.rdq = cw.d_rdq;
				cw.fp.ckpt = cw.d_ckpt;
			}
			rc = plan_run_impl(pl, nullptr);
		}
		else
		{
			rc = run_probe(pl);
			if (!rc) rc = run_assemble(pl);
			if (!rc) CK(ctx, cudaEventRecord(pl->done_ev, ctx->stream));
		}
		if (rc) return rc;
		CK(ctx, cudaStreamWaitEvent(cs, pl->done_ev, 0));
	}
	*n_ov_out = n_ov;
	return DFB_OK;
}

static int split_fetch_impl(dfb_plan* pl, int32_t* out_best, int64_t* n_rows, int64_t* n_cols, HostPool* pool, ResultSink* sink)
{
	dfb_ctx* ctx = pl->ctx;
	if (!pl->split) return set_err(ctx, DFB_ERR_STATE, "dfb_split_plan_fetch on a simple plan");
	if (!pl->ran) return set_err(ctx, DFB_ERR_STATE, "dfb_split_plan_fetch before dfb_plan_run");
	CK(ctx, cudaSetDevice(ctx->device));
	Trace tr;
	// result copies run on the copy stream, ordered behind this plan's kernels only (later batches may
	// already be queued on the compute stream)
	cudaStream_t cs = ctx->copy_stream;
	CK(ctx, wait_event(pl->done_ev));
	CK(ctx, cudaStreamWaitEvent(cs, pl->done_ev, 0));

	// 1. counters: overflow-list length and winning tasks per class
	int h_ctrl[kNumClasses * 4];
	unsigned long long n_ov = 0;
	unsigned long long asm_totals[2] = {0, 0}; // rows, columns assembled on the device
	if (int rc = fetch_counters(pl, cs, h_ctrl, &n_ov, asm_totals)) return rc;
	int64_t n_slots = 0;
	for (int c = 0; c < kNumClasses; c++)
		if (pl->cls[c].n_jobs) n_slots += (int64_t)h_ctrl[4 * c + 1] + h_ctrl[4 * c + 3]; // short- and long-window queue slots

	if (int brc = bounds_check_status(ctx)) return brc;
	tr.lap("split.fetch: wait kernels");
	// 2. bulk copy into pinned staging: best | device-assembled rows | their columns | overflow events
	const size_t g_rows = (size_t)asm_totals[0], g_cols = (size_t)asm_totals[1];
	const size_t off_best = 0;
	const size_t off_rows = align_up(off_best + (size_t)pl->n_tasks * 4, 256);
	const size_t off_cols = align_up(off_rows + g_rows * sizeof(dfb_split_row), 256);
	const size_t off_ov = align_up(off_cols + g_cols * sizeof(int32_t), 256);
	const size_t total = off_ov + (size_t)n_ov * sizeof(Event) + 256;
	{
		cudaError_t e = ctx->h_out.ensure(total);
		if (e != cudaSuccess) return set_err(ctx, DFB_ERR_NOMEM, "pinned result buffer: %s", cudaGetErrorString(e));
	}
	uint8_t* hb = (uint8_t*)ctx->h_out.p;
	int32_t* h_best = (int32_t*)(hb + off_best);
	const dfb_split_row* h_rows = (const dfb_split_row*)(hb + off_rows);
	const int32_t* h_cols = (const int32_t*)(hb + off_cols);
	Event* h_ov = (Event*)(hb + off_ov);
	int64_t d2h = 0;
	if (pl->n_tasks)
	{
		CK(ctx, cudaMemcpyAsync(h_best, pl->d_out, (size_t)pl->n_tasks * 4, cudaMemcpyDeviceToHost, cs));
		d2h += pl->n_tasks * 4;
	}
	if (g_rows) CK(ctx, cudaMemcpyAsync((void*)h_rows, pl->d_asm_rows, g_rows * sizeof(dfb_split_row), cudaMemcpyDeviceToHost, cs));
	if (g_cols) CK(ctx, cudaMemcpyAsync((void*)h_cols, pl->d_asm_cols, g_cols * sizeof(int32_t), cudaMemcpyDeviceToHost, cs));
	d2h += (int64_t)(g_rows * sizeof(dfb_split_row) + g_cols * sizeof(int32_t));
	if (n_ov) CK(ctx, cudaMemcpyAsync(h_ov, pl->d_events, (size_t)n_ov * sizeof(Event), cudaMemcpyDeviceToHost, cs));
	d2h += (int64_t)(n_ov * sizeof(Event));
	if (ctx->copied_ev)
	{
		CK(ctx, cudaEventRecord(ctx->copied_ev, cs));
		CK(ctx, wait_event(ctx->copied_ev)); // (sleeps through the transfer)
	}
	CK(ctx, cudaStreamSynchronize(cs));
	pl->stats.d2h_bytes = d2h;
	pl->stats.probe_jobs = n_slots;
	if (trace_on()) fprintf(stderr, "[dfb] fetch: %.1f MB device -> host\n", (double)d2h / 1e6);
	tr.lap("split.fetch: d2h");

	if (out_best && pl->n_tasks) memcpy(out_best, h_best, (size_t)pl->n_tasks * 4);

	// 3. overflow list = every arg-max column of the tie-heavy and generic-path tasks.  Its tasks are assembled here:
	//    events are dealt into buckets of consecutive tasks, every bucket is ordered by (task, matrix, row, column)
	//    and walked by one thread
	const int T = (int)std::max<int64_t>(1, std::min<int64_t>(pool ? pool->Size() : ctx->host_threads, (int64_t)(g_rows + n_ov) / 32768 + 1));
	std::vector<Chunk> host_part((size_t)T);
	if (n_ov)
	{
		std::vector<Event> bucketed((size_t)n_ov);
		std::vector<size_t> hist((size_t)T * (size_t)T, 0); // [thread][bucket]
		const int64_t n_tasks = std::max<int64_t>(pl->n_tasks, 1);
		auto bucket_of = [&](int32_t task) { return (int)((int64_t)task * T / n_tasks); };
		parallel_for(pool, T, [&](int tid) {
			size_t* h = hist.data() + (size_t)tid * (size_t)T;
			for (size_t k = n_ov * (size_t)tid / (size_t)T; k < n_ov * ((size_t)tid + 1) / (size_t)T; k++) h[bucket_of(h_ov[k].task)]++;
		});
		std::vector<size_t> bucket_begin((size_t)T + 1, 0);
		{
			size_t at = 0;
			for (int b = 0; b < T; b++)
			{
				bucket_begin[(size_t)b] = at;
				for (int tid = 0; tid < T; tid++)
				{
					size_t& h = hist[(size_t)tid * (size_t)T + (size_t)b];
					const size_t cnt = h;
					h = at;
					at += cnt;
				}
			}
			bucket_begin[(size_t)T] = at;
		}
		parallel_for(pool, T, [&](int tid) {
			size_t* h = hist.data() + (size_t)tid * (size_t)T;
			for (size_t k = n_ov * (size_t)tid / (size_t)T; k < n_ov * ((size_t)tid + 1) / (size_t)T; k++)
				bucketed[h[bucket_of(h_ov[k].task)]++] = h_ov[k];
		});
		parallel_for(pool, T, [&](int b) {
			Event* ov = bucketed.data() + bucket_begin[(size_t)b];
			Event* const last = bucketed.data() + bucket_begin[(size_t)b + 1];
			std::sort(ov, last, [](const Event& x, const Event& y) {
				if (x.task != y.task) return x.task < y.task;
				if (x.half_row != y.half_row) return x.half_row < y.half_row;
				return x.col < y.col;
			});
			Chunk& out = host_part[(size_t)b];
			std::vector<uint64_t> key;
			std::vector<int32_t> score;
			while (ov < last)
			{
				const int32_t t = ov->task;
				key.clear();
				score.clear();
				for (; ov < last && ov->task == t; ov++)
				{
					key.push_back(wide_key(ov->half_row >> 30, ov->half_row & 0x3fffffff, ov->col));
					score.push_back(ov->score);
				}
				int L_t;
				if (pl->h_read_off)
				{
					const int64_t rd = (int64_t)pl->h_task_read[t] - pl->h_read_base;
					L_t = (int)(pl->h_read_off[rd + 1] - pl->h_read_off[rd]);
				}
				else L_t = pl->task_L[(size_t)t];
				emit_task_rows((int)t, L_t, key.data(), score.data(), (int)key.size(), out);
			}
		});
	}
	size_t x_rows = 0, x_cols = 0; // assembled on the host
	std::vector<size_t> part_row((size_t)T + 1, 0), part_col((size_t)T + 1, 0);
	for (int k = 0; k < T; k++)
	{
		part_row[(size_t)k + 1] = (x_rows += host_part[(size_t)k].rows.size());
		part_col[(size_t)k + 1] = (x_cols += host_part[(size_t)k].cols.size());
	}
	pl->stats.events = (int64_t)(g_cols + x_cols);
	if (trace_on()) fprintf(stderr, "[dfb] fetch: %zu device rows, %llu overflow events -> %zu host rows\n", g_rows, n_ov, x_rows);
	tr.lap("split.fetch: assemble");

	// 4. result arrays (recycled): rows merged by task -- the two sources never share a task --, columns of the
	//    device part first, of the host part behind them
	const size_t tot_rows = g_rows + x_rows, tot_cols = g_cols + x_cols;
	dfb_split_row* out_rows = nullptr;
	int32_t* out_cols = nullptr;
	int32_t task_shift = 0;
	int64_t col_shift = 0;
	if (sink)
	{
		if (!sink->rows->ensure_keep(sink->row_base + tot_rows, sink->row_base) || !sink->cols->ensure_keep(sink->col_base + tot_cols, sink->col_base))
			return set_err(ctx, DFB_ERR_NOMEM, "out of host memory");
		out_rows = sink->rows->data() + sink->row_base;
		out_cols = sink->cols->data() + sink->col_base;
		task_shift = sink->task_shift;
		col_shift = (int64_t)sink->col_base;
		sink->row_base += tot_rows;
		sink->col_base += tot_cols;
	}
	else
	{
		if (pl->rows.cap < ctx->spare_rows.cap) pl->rows.swap(ctx->spare_rows);
		if (pl->cols.cap < ctx->spare_cols.cap) pl->cols.swap(ctx->spare_cols);
		if (!pl->rows.ensure(tot_rows) || !pl->cols.ensure(tot_cols)) return set_err(ctx, DFB_ERR_NOMEM, "out of host memory");
		out_rows = pl->rows.data();
		out_cols = pl->cols.data();
	}
	// host rows in one list (col_begin moved behind the device columns)
	std::vector<dfb_split_row> x((size_t)x_rows);
	for (int k = 0; k < T; k++)
	{
		const Chunk& c = host_part[(size_t)k];
		for (size_t r = 0; r < c.rows.size(); r++)
		{
			dfb_split_row row = c.rows[r];
			row.col_begin += (int64_t)(g_cols + part_col[(size_t)k]) + col_shift;
			row.task += task_shift;
			x[part_row[(size_t)k] + r] = row;
		}
		if (!c.cols.empty()) memcpy(out_cols + g_cols + part_col[(size_t)k], c.cols.data(), c.cols.size() * 4);
	}
	parallel_for(pool, T, [&](int tid) {
		// device rows [g0, g1) and the host rows that sort between them
		const size_t g0 = g_rows * (size_t)tid / (size_t)T, g1 = g_rows * ((size_t)tid + 1) / (size_t)T;
		auto before = [&](size_t g) -> size_t { // host rows with a task below device row g's
			if (g >= g_rows) return x_rows;
			const int32_t task = h_rows[g].task + task_shift;
			return (size_t)(std::lower_bound(x.begin(), x.end(), task, [](const dfb_split_row& r, int32_t t) { return r.task < t; }) - x.begin());
		};
		size_t h = tid == 0 ? 0 : before(g0);
		const size_t h1 = tid == T - 1 ? x_rows : before(g1);
		dfb_split_row* dst = out_rows + g0 + h;
		size_t g = g0;
		while (g < g1 || h < h1)
		{
			if (h < h1 && (g >= g1 || x[h].task < h_rows[g].task + task_shift))
				*dst++ = x[h++];
			else
			{
				// a run of device rows up to the next host task
				size_t run_end = g1;
				if (h < h1)
				{
					const int32_t stop = x[h].task - task_shift;
					run_end = (size_t)(std::lower_bound(h_rows + g, h_rows + g1, stop, [](const dfb_split_row& r, int32_t t) { return r.task < t; }) - h_rows);
				}
				for (; g < run_end; g++)
				{
					dfb_split_row row = h_rows[g];
					row.task += task_shift;
					row.col_begin += col_shift;
					*dst++ = row;
				}
			}
		}
		const size_t c0 = g_cols * (size_t)tid / (size_t)T, c1 = g_cols * ((size_t)tid + 1) / (size_t)T;
		if (c1 > c0) memcpy(out_cols + c0, h_cols + c0, (c1 - c0) * 4);
	});
	tr.lap("split.fetch: concatenate");
	if (n_rows) *n_rows = (int64_t)tot_rows;
	if (n_cols) *n_cols = (int64_t)tot_cols;
	pl->fetched = true;
	return DFB_OK;
}

extern "C" int dfb_split_plan_copy(const dfb_plan* pl, dfb_split_row* rows, int32_t* cols)
{
	if (!pl) return DFB_ERR_ARG;
	if (!pl->fetched || !pl->split) return set_err(pl->ctx, DFB_ERR_STATE, "dfb_split_plan_copy before dfb_split_plan_fetch");
	if (rows && !pl->rows.empty()) memcpy(rows, pl->rows.data(), pl->rows.size() * sizeof(dfb_split_row));
	if (cols && !pl->cols.empty()) memcpy(cols, pl->cols.data(), pl->cols.size() * sizeof(int32_t));
	return DFB_OK;
}

extern "C" int dfb_split_plan_view(const dfb_plan* pl, const dfb_split_row** rows, int64_t* n_rows, const int32_t** cols,
                                   int64_t* n_cols)
{
	if (!pl) return DFB_ERR_ARG;
	if (!pl->fetched || !pl->split) return set_err(pl->ctx, DFB_ERR_STATE, "dfb_split_plan_view before dfb_split_plan_fetch");
	if (rows) *rows = pl->rows.data();
	if (n_rows) *n_rows = (int64_t)pl->rows.size();
	if (cols) *cols = pl->cols.data();
	if (n_cols) *n_cols = (int64_t)pl->cols.size();
	return DFB_OK;
}

extern "C" int dfb_plan_get_stats(const dfb_plan* pl, dfb_plan_stats* stats)
{
	if (!pl || !stats) return DFB_ERR_ARG;
	*stats = pl->stats;
	return DFB_OK;
}

// ---- one-call forms -------------------------------------------------------------------------------

// Batches of at least this many tasks whose table-B indices (sequences, reads) do not decrease are cut into chunks
static int64_t pipeline_min_tasks()
{
	if (const char* e = getenv("DFB_PIPELINE_MIN_TASKS")) return std::max<long long>(2, atoll(e)); // tests
	return 1 << 18;
}

static bool env_on(const char* name)
{
	const char* e = getenv(name);
	return e && *e && *e != '0';
}

// Whether task array `b` does not decrease (*b_ok) and, if it does not, whether `a` does not either (*a_ok)
static void tasks_non_decreasing(dfb_ctx* ctx, const int32_t* b, const int32_t* a, int64_t n_tasks, bool* b_ok, bool* a_ok)
{
	const int T = (int)std::max<int64_t>(1, std::min<int64_t>(ctx->host_threads, n_tasks / 262144 + 1));
	std::vector<char> ok_b((size_t)T, 1), ok_a((size_t)T, 1);
	parallel_for(ctx->pool, T, [&](int tid) {
		const int64_t t0 = std::max<int64_t>(1, n_tasks * tid / T), t1 = n_tasks * (tid + 1) / T;
		bool mb = true, ma = true;
		for (int64_t t = t0; t < t1 && mb; t++)
		{
			mb = b[t] >= b[t - 1];
			ma = ma && a[t] >= a[t - 1];
		}
		ok_b[(size_t)tid] = mb;
		ok_a[(size_t)tid] = ma;
	});
	*b_ok = *a_ok = true;
	for (int k = 0; k < T; k++)
	{
		*b_ok = *b_ok && ok_b[(size_t)k];
		*a_ok = *a_ok && ok_a[(size_t)k];
	}
}

// First task of every chunk (and n_tasks behind the last): chunk k's share of the batch is weight[k] / sum(weight)
static std::vector<int64_t> chunk_starts(int64_t n_tasks, const std::vector<double>& weight)
{
	const int K = (int)weight.size();
	std::vector<int64_t> t0((size_t)K + 1, 0);
	double total = 0, run = 0;
	for (double w : weight) total += w;
	for (int k = 0; k < K; k++)
	{
		run += weight[(size_t)k];
		t0[(size_t)k + 1] = k + 1 == K ? n_tasks : (int64_t)((double)n_tasks * run / total);
	}
	return t0;
}

// Where the job lists of a chunked batch are built.  Never on the device when no class of the s16x2 kernels takes this
// scoring (every task is generic then and the host path lists them).  Simple: on the device otherwise -- a simple batch is
// host-bound on the host path (one pass over the tasks and two over the tables per chunk against 4 ms of sweep).  Split:
// on the device, 31 ms of host CPU time per 2 M-task batch, but the build kernels sit on the compute stream (0.2 ms per
// chunk with their launch gaps); on the host, 72 ms of CPU time over the context's workers, fully hidden under the GPU
// when the host has the threads -- 1.7 ms per batch faster then (A/B on one box, profiles/r03l_ab_e2e.txt).  So the
// device unless this context has 16 or more host threads to itself (one process per GPU on a shared host caps them with
// DFB_HOST_THREADS; bench.py does under torchrun).  DFB_DEVICE_BUILD / DFB_HOST_BUILD force either (tests).
static bool device_build_chosen(dfb_ctx* ctx, bool simple, const dfb_split_params* params)
{
	dfb_plan probe;
	classify_params(&probe, params->match, params->mismatch, params->gap, simple || (params->end_gaps == 0 && params->min_split_score >= 1));
	bool any_fast = false;
	for (int c = 0; c < kNumClasses; c++) any_fast = any_fast || probe.fast_ok[c];
	bool device = any_fast && (simple || ctx->host_threads < 16);
	if (env_on("DFB_DEVICE_BUILD")) device = any_fast;
	if (env_on("DFB_HOST_BUILD")) device = false;
	return device;
}

// A chunk of a pipelined batch: its views of the two tables, the caller's numbers of their first entries and, for
// device-resident tables, the byte ranges [a0, a1), [b0, b1) the views cover (null: host tables)
struct ChunkView
{
	dfb_seq_table a, b;
	int32_t a_lo = 0, b_lo = 0;
	const int64_t* range = nullptr;
};

// A batch of either aligner (tasks as for plan_create_host) cut into the chunks that start at t0.  view_of(k) gives chunk
// k's table views, host_plan(k) builds chunk k on the host.  Device-built chunks (`device_build`; three beats per chunk):
// the uploads of chunk k+1 are queued on the upload stream while chunk k is finished -- allocations, packing and job
// scatter once its class counts are back -- and launched; the job-build kernels of chunk k+1 ride on the compute stream
// between chunk k's two sweeps, so their counts are on the host before chunk k's probe sweep ends and the GPU never waits
// for this thread.  A chunk the device build hands back (DFB_BUILD_ON_HOST) is built by host_plan.  The plans land in
// `plans`; chunk_queued(k) runs once chunk k is on the GPU (a non-zero return stops the batch), batch_done(rc) once no
// more is queued: it waits for what is in flight and returns the batch's result.  The plans are destroyed on return.
static int pipeline_run(dfb_ctx* ctx, bool simple, const dfb_split_params* params, const int32_t* task_a, const int32_t* task_b,
                        const int32_t* task_min_score, const std::vector<int64_t>& t0, bool device_build,
                        const std::function<int(int, ChunkView&)>& view_of,
                        const std::function<int(int, const ChunkView&, dfb_plan**)>& host_plan, std::vector<dfb_plan*>& plans,
                        const std::function<int(int)>& chunk_queued, const std::function<int(int)>& batch_done)
{
	const int K = (int)t0.size() - 1;
	std::vector<dfb_plan*> staged((size_t)K, nullptr);
	auto upload = [&](int k) -> int {
		ChunkView v;
		const int64_t a = t0[(size_t)k];
		int rc = view_of(k, v);
		return rc ? rc : device_build_enqueue(ctx, simple, params, &v.a, &v.b, task_a + a, task_b + a, simple ? nullptr : task_min_score + a,
		                                      t0[(size_t)k + 1] - a, v.a_lo, v.b_lo, k, &staged[(size_t)k], v.range);
	};
	// DFB_TRACE: the device's side of the batch -- when every chunk's uploads, first sweep and (split) probe sweep +
	// assembly ended, measured from an event recorded on the (idle) compute stream now
	cudaEvent_t trace_base = nullptr;
	if (trace_on() && cudaEventCreate(&trace_base) == cudaSuccess) cudaEventRecord(trace_base, ctx->stream);
	int rc = DFB_OK;
	if (device_build && K)
	{
		rc = upload(0);
		if (!rc) rc = device_build_kernels(staged[0]); // (the GPU is idle: straight away)
	}
	for (int k = 0; k < K && !rc; k++)
	{
		if (device_build && k + 1 < K && (rc = upload(k + 1))) break;
		dfb_plan* pk = staged[(size_t)k];
		staged[(size_t)k] = nullptr;
		rc = DFB_BUILD_ON_HOST;
		if (pk && (rc = device_build_finish(pk)))
		{
			dfb_plan_destroy(pk);
			pk = nullptr;
		}
		if (rc == DFB_BUILD_ON_HOST)
		{
			ChunkView v;
			if (!(rc = view_of(k, v))) rc = host_plan(k, v, &pk);
		}
		if (rc) break;
		plans[(size_t)k] = pk;
		if (trace_base) pk->timing = true;
		// the next chunk's build kernels ride behind this chunk's first sweep on the compute stream
		dfb_plan* next = (k + 1 < K) ? staged[(size_t)k + 1] : nullptr;
		const std::function<int()> hook = [&]() -> int { return next ? device_build_kernels(next) : DFB_OK; };
		rc = plan_run_impl(pk, &hook);
		if (!rc) rc = chunk_queued(k);
	}
	for (dfb_plan* sp : staged)
		if (sp)
		{
			cudaStreamSynchronize(sp->up); // (its uploads read the caller's arrays)
			dfb_plan_destroy(sp);
		}
	rc = batch_done(rc);
	if (trace_base)
	{
		for (int k = 0; k < K && !rc; k++)
		{
			const dfb_plan* pk = plans[(size_t)k];
			float up = -1, a = -1, b = -1, c = -1;
			if (pk->pending.uploaded) cudaEventElapsedTime(&up, trace_base, pk->pending.uploaded);
			cudaEventElapsedTime(&a, trace_base, pk->ev[0]);
			cudaEventElapsedTime(&b, trace_base, pk->ev[1]);
			fprintf(stderr, "[dfb] device: chunk %d (%lld tasks) uploaded %.3f | %s %.3f .. %.3f", k, (long long)pk->n_tasks, up,
			        simple ? "sweep" : "first sweep", a, b);
			if (!simple)
			{
				cudaEventElapsedTime(&c, trace_base, pk->ev[2]);
				fprintf(stderr, " | probe + assembly .. %.3f", c);
			}
			fprintf(stderr, " ms\n");
		}
		cudaEventDestroy(trace_base);
	}
	for (dfb_plan* pk : plans)
		if (pk) dfb_plan_destroy(pk);
	return rc;
}

// pipeline_run over host tables, whose table-B indices do not decrease.  A chunk sees a view of table B (its own entries)
// and, when the batch's table-A indices do not decrease either (`a_monotone`), a view of table A too -- else the whole
// table.  Chunks the device does not build are built by plan_create_host.
static int pipeline_run_host(dfb_ctx* ctx, bool simple, const dfb_split_params* params, const dfb_seq_table* A, const dfb_seq_table* B,
                             const int32_t* task_a, const int32_t* task_b, const int32_t* task_min_score, bool a_monotone,
                             const std::vector<int64_t>& t0, std::vector<dfb_plan*>& plans, const std::function<int(int)>& chunk_queued,
                             const std::function<int(int)>& batch_done)
{
	const int64_t per = simple ? 1 : 2; // table-A entries per task index (split: the two windows of a cluster)
	auto view_of = [&](int k, ChunkView& v) -> int {
		const int64_t t_lo = t0[(size_t)k], t_hi = t0[(size_t)k + 1];
		if (t_hi <= t_lo) return set_err(ctx, DFB_ERR_STATE, "empty chunk in a pipelined batch");
		const int64_t b_lo = task_b[t_lo], b_hi = (int64_t)task_b[t_hi - 1] + 1;
		if (b_lo < 0 || b_hi > B->n) return set_err(ctx, DFB_ERR_ARG, "task %lld: table index out of range", (long long)t_lo);
		int64_t a_lo = 0, a_hi = A->n / per;
		if (a_monotone)
		{
			a_lo = task_a[t_lo];
			a_hi = (int64_t)task_a[t_hi - 1] + 1;
			if (a_lo < 0 || per * a_hi > A->n)
				return set_err(ctx, DFB_ERR_ARG, "task %lld: table index out of range", (long long)(simple || a_lo < 0 ? t_lo : t_hi - 1));
		}
		v.a = dfb_seq_table{A->bytes, A->off + per * a_lo, per * (a_hi - a_lo)};
		v.b = dfb_seq_table{B->bytes, B->off + b_lo, b_hi - b_lo};
		v.a_lo = (int32_t)a_lo;
		v.b_lo = (int32_t)b_lo;
		return DFB_OK;
	};
	auto host_plan = [&](int k, const ChunkView& v, dfb_plan** out) -> int {
		const int64_t a = t0[(size_t)k];
		return plan_create_host(ctx, simple, params, &v.a, &v.b, task_a + a, task_b + a, simple ? nullptr : task_min_score + a,
		                        t0[(size_t)k + 1] - a, v.a_lo, v.b_lo, k, (k & 1) ? ctx->upload_stream2 : ctx->upload_stream, out);
	};
	return pipeline_run(ctx, simple, params, task_a, task_b, task_min_score, t0, device_build_chosen(ctx, simple, params), view_of, host_plan,
	                    plans, chunk_queued, batch_done);
}

// Large batches whose task_seq is non-decreasing go through pipeline_run: chunk k+1 is uploaded and packed underneath
// chunk k's sweep, the scores of chunk k-1 go back on the copy stream meanwhile.  A chunk takes a view of the sequences it
// names; of the references too when task_ref is non-decreasing as well (matealign: one window per task), else the whole
// reference table (localalign: few references, named in any order).
static int simple_align_pipelined(dfb_ctx* ctx, const dfb_split_params* params, const dfb_seq_table* refs,
                                  const dfb_seq_table* seqs, const int32_t* task_ref, const int32_t* task_seq,
                                  int64_t n_tasks, bool refs_monotone, int32_t* out_score)
{
	// chunks: a batch whose references come in task order (matealign: one window per task) uploads every byte once however
	// it is cut, and is bound by the upload -- short chunks keep the wait for the first and the sweep of the last short;
	// one whose references are named in any order re-uploads the reference table with every chunk: fewer, longer chunks
	const int64_t per_chunk = refs_monotone ? 80000 : 150000;
	const int K = (int)std::max<int64_t>(2, std::min<int64_t>(dfb_ctx::kStageSlots, n_tasks / per_chunk));
	std::vector<double> weight((size_t)K, 1.0);
	weight[0] = 0.4; // a short first chunk puts the GPU to work early
	const std::vector<int64_t> t0 = chunk_starts(n_tasks, weight);
	std::vector<dfb_plan*> plans((size_t)K, nullptr);
	Trace trp;
	auto copy_scores = [&](int k) -> int {
		// scores straight into the caller's array, behind this chunk's kernels only
		const int64_t a = t0[(size_t)k], b = t0[(size_t)k + 1];
		cudaError_t e = cudaStreamWaitEvent(ctx->copy_stream, plans[(size_t)k]->done_ev, 0);
		if (e == cudaSuccess)
			e = cudaMemcpyAsync(out_score + a, plans[(size_t)k]->d_out, (size_t)(b - a) * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->copy_stream);
		return e == cudaSuccess ? DFB_OK : set_err(ctx, DFB_ERR_CUDA, "score copy failed: %s", cudaGetErrorString(e));
	};
	auto wait_all = [&](int rc) -> int {
		cudaError_t e = cudaStreamSynchronize(ctx->copy_stream);
		if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
		if (!rc && e != cudaSuccess) rc = set_err(ctx, DFB_ERR_CUDA, "pipelined batch failed: %s", cudaGetErrorString(e));
		if (!rc) rc = bounds_check_status(ctx);
		trp.lap("simple pipelined: done");
		return rc;
	};
	return pipeline_run_host(ctx, true, params, refs, seqs, task_ref, task_seq, nullptr, refs_monotone, t0, plans, copy_scores, wait_all);
}

static int dfb_simple_align_batch_body(dfb_ctx* ctx, const dfb_simple_params* params, const dfb_seq_table* refs,
                                      const dfb_seq_table* seqs, const int32_t* task_ref, const int32_t* task_seq,
                                      int64_t n_tasks, int32_t* out_score)
{
	if (!ctx) return DFB_ERR_ARG;
	int rc = check_simple_args(ctx, params, refs, seqs, task_ref, task_seq, n_tasks);
	if (rc) return rc;
	const dfb_split_params sp{params->match, params->mismatch, params->gap, 0, 0};
	if (n_tasks >= pipeline_min_tasks() && out_score)
	{
		bool seq_monotone, ref_monotone;
		tasks_non_decreasing(ctx, task_seq, task_ref, n_tasks, &seq_monotone, &ref_monotone);
		if (seq_monotone) return simple_align_pipelined(ctx, &sp, refs, seqs, task_ref, task_seq, n_tasks, ref_monotone, out_score);
	}
	dfb_plan* pl = nullptr;
	Trace tr;
	rc = plan_create_host(ctx, true, &sp, refs, seqs, task_ref, task_seq, nullptr, n_tasks, 0, 0, 0, nullptr, &pl);
	if (rc) return rc;
	tr.lap("simple: create");
	rc = dfb_plan_run(pl);
	if (!rc) rc = dfb_simple_plan_fetch(pl, out_score);
	tr.lap("simple: run + fetch");
	dfb_plan_destroy(pl);
	tr.lap("simple: destroy");
	return rc;
}

// Chunk boundaries of a pipelined split batch (both one-call forms cut a batch at the same tasks: the column pool
// holds each chunk's region-assembled columns in front of its overflow-list columns, so equal results need equal cuts)
static std::vector<int64_t> split_chunk_starts(int64_t n_tasks)
{
	const int K = (int)std::max<int64_t>(2, std::min<int64_t>(std::min<int64_t>(dfb_ctx::kStageSlots, n_tasks), n_tasks / 330000));
	// chunk boundaries: short chunks in front put the GPU to work early, chunks that taper off at the end keep the part
	// of the result assembly that nothing overlaps small (lane 2 finishes chunk k while the GPU runs chunk k+1); the
	// chunks in between share the rest
	std::vector<double> weight((size_t)K, 1.0);
	if (K >= 8)
	{
		// the fetch lane needs about 0.8 of a chunk's GPU time for that chunk: a tail that shrinks by no more than
		// that factor per chunk keeps it from falling behind, so only the last, smallest chunk's fetch is left uncovered
		weight[0] = 0.3;
		weight[1] = 0.7;
		weight[(size_t)K - 4] = 0.8;
		weight[(size_t)K - 3] = 0.62;
		weight[(size_t)K - 2] = 0.48;
		weight[(size_t)K - 1] = 0.36;
	}
	else if (K >= 6)
	{
		weight[0] = 0.25;
		weight[1] = 0.6;
		weight[(size_t)K - 2] = 0.6;
		weight[(size_t)K - 1] = 0.3;
	}
	else if (K >= 4)
	{
		weight[0] = 0.4;
		weight[(size_t)K - 1] = 0.45;
	}
	return chunk_starts(n_tasks, weight);
}

// Large batches whose task_read is non-decreasing (the usual case: reads are listed in task order) go through
// pipeline_run: chunks flow through the GPU back to back while the host builds the next chunk and assembles the previous
// one.  Results are merged into one task-ordered row list.  A chunk sees views of both tables: its own reads and -- when
// the batch's clusters do not decrease, the order dosplitalign emits -- its own window pairs, so that every window is
// uploaded and packed once per batch (plus one shared cluster per chunk boundary) instead of once per chunk.
static int split_align_pipelined(dfb_ctx* ctx, const dfb_split_params* params, const dfb_seq_table* refs,
                                 const dfb_seq_table* reads, const int32_t* task_cluster, const int32_t* task_read,
                                 const int32_t* task_min_score, int64_t n_tasks, int32_t* out_best, bool clusters_monotone)
{
	const std::vector<int64_t> t0 = split_chunk_starts(n_tasks);
	const int K = (int)t0.size() - 1;
	std::vector<dfb_plan*> plans((size_t)K, nullptr);
	{
		// the pinned buffer the chunks' results land in: sized for the largest chunk now (growing it chunk by chunk frees and
		// pins it again each time, at 0.6 ms per MB either way)
		int64_t largest = 0;
		for (int k = 0; k < K; k++) largest = std::max(largest, t0[(size_t)k + 1] - t0[(size_t)k]);
		ctx->h_out.ensure((size_t)largest * 72);
	}
	Trace trp;
	// the batch's result holder: every chunk's rows go straight behind the previous chunk's
	dfb_plan* holder = new (std::nothrow) dfb_plan();
	if (!holder) return set_err(ctx, DFB_ERR_NOMEM, "out of host memory");
	holder->ctx = ctx;
	holder->split = true;
	holder->n_tasks = n_tasks;
	holder->stats.n_tasks = n_tasks;
	if (holder->rows.cap < ctx->spare_rows.cap) holder->rows.swap(ctx->spare_rows);
	if (holder->cols.cap < ctx->spare_cols.cap) holder->cols.swap(ctx->spare_cols);
	holder->rows.n = holder->cols.n = 0;
	ResultSink sink{&holder->rows, &holder->cols, 0, 0, 0};
	// lane 2 (helper thread): waits for chunk k to be queued on the GPU, copies its results back and assembles its
	// rows -- while lane 1 (this thread) builds and queues the following chunks
	std::mutex mu;
	std::condition_variable cv;
	int queued = 0;      // chunks handed to the GPU so far
	bool abort = false;  // lane 1 failed: lane 2 stops after the chunks already queued
	std::atomic<int> fetch_rc{DFB_OK}; // (lane 1 looks at it between chunks: nothing more is queued behind a failed fetch)
	std::thread lane2([&] {
		try
		{
		for (int k = 0; k < K; k++)
		{
			{
				std::unique_lock<std::mutex> lk(mu);
				cv.wait(lk, [&] { return queued > k || abort; });
				if (queued <= k) return;
			}
			sink.task_shift = (int32_t)t0[k];
			int frc = split_fetch_impl(plans[k], out_best ? out_best + t0[k] : nullptr, nullptr, nullptr, ctx->pool_fetch, &sink);
			if (frc)
			{
				fetch_rc = frc;
				return;
			}
			// the chunk's device buffers go back to the pool now (stream-ordered): lane 1 stays about two chunks ahead
			// of the GPU, so the chunks still to be built reuse them and a batch never holds more than about half of
			// its chunks' checkpoints at a time
			release_device(plans[k]);
		}
		}
		catch (...)
		{
			fetch_rc = set_err(ctx, DFB_ERR_NOMEM, "out of host memory in the fetch lane");
		}
	});
	auto hand_to_lane2 = [&](int k) -> int {
		{
			std::lock_guard<std::mutex> lk(mu);
			queued = k + 1;
		}
		cv.notify_all();
		return fetch_rc.load();
	};
	auto join_lane2 = [&](int rc) -> int {
		{
			std::lock_guard<std::mutex> lk(mu);
			if (rc) abort = true;
		}
		cv.notify_all();
		trp.lap("pipelined: lane 1 done");
		lane2.join();
		trp.lap("pipelined: lane 2 joined");
		if (!rc) rc = fetch_rc.load();
		if (!rc)
		{
			holder->fetched = true;
			holder->ran = true;
			for (int k = 0; k < K; k++)
			{
				holder->stats.events += plans[k]->stats.events;
				holder->stats.probe_jobs += plans[k]->stats.probe_jobs;
				holder->stats.d2h_bytes += plans[k]->stats.d2h_bytes;
				holder->stats.h2d_bytes += plans[k]->stats.h2d_bytes;
				holder->stats.cells += plans[k]->stats.cells;
				holder->stats.fast_jobs += plans[k]->stats.fast_jobs;
				holder->stats.generic_jobs += plans[k]->stats.generic_jobs;
				holder->stats.kernel_launches += plans[k]->stats.kernel_launches;
				holder->stats.raw_bytes += plans[k]->stats.raw_bytes;
				holder->stats.packed_bytes += plans[k]->stats.packed_bytes;
			}
		}
		return rc;
	};
	const int rc = pipeline_run_host(ctx, false, params, refs, reads, task_cluster, task_read, task_min_score, clusters_monotone, t0, plans,
	                                 hand_to_lane2, join_lane2);
	trp.lap("pipelined: chunks destroyed");
	if (rc)
	{
		dfb_plan_destroy(holder);
		return rc;
	}
	ctx->last_split = holder;
	return DFB_OK;
}

static int dfb_split_align_batch_body(dfb_ctx* ctx, const dfb_split_params* params, const dfb_seq_table* refs,
                                     const dfb_seq_table* reads, const int32_t* task_cluster, const int32_t* task_read,
                                     const int32_t* task_min_score, int64_t n_tasks, int32_t* out_best)
{
	if (!ctx) return DFB_ERR_ARG;
	if (ctx->last_split)
	{
		dfb_plan_destroy(ctx->last_split);
		ctx->last_split = nullptr;
	}
	Trace tre;
	tre.lap("split: entry");
	int rc = check_split_args(ctx, params, refs, reads, task_cluster, task_read, task_min_score, n_tasks);
	if (rc) return rc;
	if (n_tasks >= pipeline_min_tasks())
	{
		bool monotone, clusters_monotone;
		tasks_non_decreasing(ctx, task_read, task_cluster, n_tasks, &monotone, &clusters_monotone);
		tre.lap("split: validated");
		if (monotone)
			return split_align_pipelined(ctx, params, refs, reads, task_cluster, task_read, task_min_score, n_tasks, out_best, clusters_monotone);
	}
	dfb_plan* pl = nullptr;
	rc = plan_create_host(ctx, false, params, refs, reads, task_cluster, task_read, task_min_score, n_tasks, 0, 0, 0, nullptr, &pl);
	if (rc) return rc;
	rc = dfb_plan_run(pl);
	if (!rc) rc = dfb_split_plan_fetch(pl, out_best, nullptr, nullptr);
	if (rc)
	{
		dfb_plan_destroy(pl);
		return rc;
	}
	// only the host-side rows are kept; the device buffers go back to the pool now
	release_device(pl);
	ctx->last_split = pl;
	return DFB_OK;
}

extern "C" int dfb_split_result_stats(const dfb_ctx* ctx, dfb_plan_stats* stats)
{
	if (!ctx || !stats) return DFB_ERR_ARG;
	if (!ctx->last_split) return set_err(ctx, DFB_ERR_STATE, "no split result on this context");
	*stats = ctx->last_split->stats;
	return DFB_OK;
}

extern "C" int dfb_split_result_size(const dfb_ctx* ctx, int64_t* n_rows, int64_t* n_cols)
{
	if (!ctx) return DFB_ERR_ARG;
	if (!ctx->last_split) return set_err(ctx, DFB_ERR_STATE, "no split result on this context");
	if (ctx->last_split->device_result)
		return set_err(ctx, DFB_ERR_STATE, "the last split result is in device memory: use dfb_split_result_copy_device");
	if (n_rows) *n_rows = (int64_t)ctx->last_split->rows.size();
	if (n_cols) *n_cols = (int64_t)ctx->last_split->cols.size();
	return DFB_OK;
}

extern "C" int dfb_split_result_copy(const dfb_ctx* ctx, dfb_split_row* rows, int32_t* cols)
{
	if (!ctx) return DFB_ERR_ARG;
	if (!ctx->last_split) return set_err(ctx, DFB_ERR_STATE, "no split result on this context");
	if (ctx->last_split->device_result)
		return set_err(ctx, DFB_ERR_STATE, "the last split result is in device memory: use dfb_split_result_copy_device");
	return dfb_split_plan_copy(ctx->last_split, rows, cols);
}

extern "C" int dfb_split_result_view(const dfb_ctx* ctx, const dfb_split_row** rows, int64_t* n_rows, const int32_t** cols,
                                     int64_t* n_cols)
{
	if (!ctx) return DFB_ERR_ARG;
	if (!ctx->last_split) return set_err(ctx, DFB_ERR_STATE, "no split result on this context");
	if (ctx->last_split->device_result)
		return set_err(ctx, DFB_ERR_STATE, "the last split result is in device memory: use dfb_split_result_copy_device");
	return dfb_split_plan_view(ctx->last_split, rows, n_rows, cols, n_cols);
}


// ---- exception barrier of the entry points that allocate batch-sized host memory --------------------------------

extern "C" int dfb_simple_plan_create(dfb_ctx* ctx, const dfb_simple_params* params, const dfb_seq_table* refs,
                                      const dfb_seq_table* seqs, const int32_t* task_ref, const int32_t* task_seq,
                                      int64_t n_tasks, dfb_plan** out)
{
	return guarded(ctx, [&] { return dfb_simple_plan_create_body(ctx, params, refs, seqs, task_ref, task_seq, n_tasks, out); });
}

extern "C" int dfb_split_plan_create(dfb_ctx* ctx, const dfb_split_params* params, const dfb_seq_table* refs,
                                     const dfb_seq_table* reads, const int32_t* task_cluster, const int32_t* task_read,
                                     const int32_t* task_min_score, int64_t n_tasks, dfb_plan** out)
{
	return guarded(ctx, [&] { return dfb_split_plan_create_body(ctx, params, refs, reads, task_cluster, task_read, task_min_score, n_tasks, out); });
}

extern "C" int dfb_plan_run(dfb_plan* pl)
{
	return guarded(pl ? pl->ctx : nullptr, [&] { return dfb_plan_run_body(pl); });
}

extern "C" int dfb_split_plan_fetch(dfb_plan* pl, int32_t* out_best, int64_t* n_rows, int64_t* n_cols)
{
	return guarded(pl ? pl->ctx : nullptr, [&] { return dfb_split_plan_fetch_body(pl, out_best, n_rows, n_cols); });
}

extern "C" int dfb_simple_align_batch(dfb_ctx* ctx, const dfb_simple_params* params, const dfb_seq_table* refs,
                                      const dfb_seq_table* seqs, const int32_t* task_ref, const int32_t* task_seq,
                                      int64_t n_tasks, int32_t* out_score)
{
	return guarded(ctx, [&] { return dfb_simple_align_batch_body(ctx, params, refs, seqs, task_ref, task_seq, n_tasks, out_score); });
}

extern "C" int dfb_split_align_batch(dfb_ctx* ctx, const dfb_split_params* params, const dfb_seq_table* refs,
                                     const dfb_seq_table* reads, const int32_t* task_cluster, const int32_t* task_read,
                                     const int32_t* task_min_score, int64_t n_tasks, int32_t* out_best)
{
	return guarded(ctx, [&] { return dfb_split_align_batch_body(ctx, params, refs, reads, task_cluster, task_read, task_min_score, n_tasks, out_best); });
}

// ---- device-resident one-call forms ------------------------------------------------------------------------------
// The batch, the outputs and the results stay in device memory: tables and tasks are read where they are, checked by
// kernels (dfb_build.cuh), copied device to device into the plan's raw buffer and built into job lists on the device;
// the overflow list is assembled by the kernels of dfb_assemble.cuh.  What crosses PCIe is counters: the check record,
// the build statistics and the overflow / assembly totals of every chunk, the batch's row and column totals.  Chunks that
// hold tasks only the s32 kernels take are built by the host builder from a host copy of their offsets and task arrays
// (never the bytes).

// Every array of a device-resident call must be memory of the context's device: host memory (pinned or not), managed
// memory and another GPU's memory are refused before anything is queued.
static bool is_ctx_device_memory(const dfb_ctx* ctx, const void* p)
{
	if (!p) return true; // (null pointers are judged by the argument checks of the host form)
	cudaPointerAttributes a;
	if (cudaPointerGetAttributes(&a, p) != cudaSuccess)
	{
		cudaGetLastError();
		return false;
	}
	return a.type == cudaMemoryTypeDevice && a.device == ctx->device;
}

// the kernels of check_device_args: the record is initialised, then both tables and the task arrays are checked
static void enqueue_device_checks(dfb_ctx* ctx, bool simple, const dfb_device_seq_table* A, const dfb_device_seq_table* B,
                                  const int32_t* ta, const int32_t* tb, int64_t n_tasks, DeviceCheck* d_chk)
{
	const dfb_device_seq_table* tabs[2] = {A, B};
	const int max_grid = ctx->prop.multiProcessorCount * 8;
	auto grid = [&](int64_t n) { return (unsigned)std::max<int64_t>(1, std::min<int64_t>((n + DFB_BUILD_BLOCK - 1) / DFB_BUILD_BLOCK, max_grid)); };
	device_check_init_kernel<<<1, 1, 0, ctx->stream>>>(d_chk);
	for (int k = 0; k < 2; k++) table_check_kernel<<<grid(tabs[k]->n), DFB_BUILD_BLOCK, 0, ctx->stream>>>(tabs[k]->off, tabs[k]->n, &d_chk->tab[k]);
	if (n_tasks)
		task_check_kernel<<<grid(n_tasks), DFB_BUILD_BLOCK, 0, ctx->stream>>>(ta, tb, n_tasks, simple ? A->n : A->n / 2, B->n, d_chk);
}

// the status and message of a check record read back from the device
static int device_check_status(dfb_ctx* ctx, bool simple, const dfb_device_seq_table* A, const dfb_device_seq_table* B, int64_t n_tasks,
                               const DeviceCheck& chk)
{
	const char* names[2] = {"refs", simple ? "seqs" : "reads"};
	const dfb_device_seq_table* tabs[2] = {A, B};
	for (int k = 0; k < 2; k++)
	{
		const TableCheck& c = chk.tab[k];
		if (tabs[k]->n > 0 && !tabs[k]->bytes && c.off_n > 0) return set_err(ctx, DFB_ERR_ARG, "%s: null table", names[k]);
		if (c.off0 != 0) return set_err(ctx, DFB_ERR_ARG, "%s: off[0] must be 0", names[k]);
		if (c.first_bad != ~0ull)
		{
			if (c.first_bad & 1) return set_err(ctx, DFB_ERR_ARG, "%s: sequence %lld too long", names[k], (long long)(c.first_bad >> 1));
			return set_err(ctx, DFB_ERR_ARG, "%s: offsets decrease at %lld", names[k], (long long)(c.first_bad >> 1));
		}
		if (c.off_n > tabs[k]->n_bytes)
			return set_err(ctx, DFB_ERR_ARG, "%s: off[n] = %lld exceeds n_bytes = %lld", names[k], (long long)c.off_n, (long long)tabs[k]->n_bytes);
	}
	if (!simple && (A->n & 1)) return set_err(ctx, DFB_ERR_ARG, "refs must hold two windows per cluster (n is odd)");
	if (n_tasks > 0x7fffff00LL) return set_err(ctx, DFB_ERR_ARG, "too many tasks in one batch");
	if (chk.bad_task != ~0ull) return set_err(ctx, DFB_ERR_ARG, "task %lld: table index out of range", (long long)chk.bad_task);
	return DFB_OK;
}

// The argument checks of the host form (check_simple_args / check_split_args, and the builders' task index check) with
// the same statuses and messages, run on the device; plus off[n] <= n_bytes.  *chk receives the record.
static int check_device_args(dfb_ctx* ctx, bool simple, const void* params, const dfb_device_seq_table* A, const dfb_device_seq_table* B,
                             const int32_t* ta, const int32_t* tb, const int32_t* tm, int64_t n_tasks, const void* out, DeviceCheck* chk)
{
	const char* names[2] = {"refs", simple ? "seqs" : "reads"};
	const dfb_device_seq_table* tabs[2] = {A, B};
	if (!params || n_tasks < 0 || (n_tasks > 0 && (!ta || !tb || (!simple && !tm))))
		return set_err(ctx, DFB_ERR_ARG, "%s: null argument", simple ? "dfb_simple_plan_create" : "dfb_split_plan_create");
	for (int k = 0; k < 2; k++)
		if (!tabs[k] || !tabs[k]->off || tabs[k]->n < 0 || tabs[k]->n_bytes < 0) return set_err(ctx, DFB_ERR_ARG, "%s: null table", names[k]);
	if (n_tasks > 0 && !out) return set_err(ctx, DFB_ERR_ARG, "null output");
	const void* ptrs[8] = {A->bytes, A->off, B->bytes, B->off, ta, tb, simple ? nullptr : tm, out};
	const char* what[8] = {"refs->bytes", "refs->off", simple ? "seqs->bytes" : "reads->bytes", simple ? "seqs->off" : "reads->off",
	                       simple ? "task_ref" : "task_cluster", simple ? "task_seq" : "task_read", "task_min_score",
	                       simple ? "out_score" : "out_best"};
	for (int k = 0; k < 8; k++)
		if (!is_ctx_device_memory(ctx, ptrs[k]))
			return set_err(ctx, DFB_ERR_ARG, "%s is not device memory of device %d", what[k], ctx->device);
	DeviceCheck* d_chk = nullptr;
	CK(ctx, dalloc(ctx, (void**)&d_chk, sizeof(DeviceCheck)));
	CK(ctx, ctx->h_out.ensure(sizeof(DeviceCheck)));
	DeviceCheck* h_chk = (DeviceCheck*)ctx->h_out.p;
	enqueue_device_checks(ctx, simple, A, B, ta, tb, n_tasks, d_chk);
	CK(ctx, cudaGetLastError());
	CK(ctx, cudaMemcpyAsync(h_chk, d_chk, sizeof(DeviceCheck), cudaMemcpyDeviceToHost, ctx->stream));
	cudaFreeAsync(d_chk, ctx->stream);
	CK(ctx, cudaStreamSynchronize(ctx->stream));
	*chk = *h_chk;
	return device_check_status(ctx, simple, A, B, n_tasks, *chk);
}

// Work on the upload and copy streams is ordered behind what the caller queued on the context's stream before the call
static int order_side_streams(dfb_ctx* ctx)
{
	cudaEvent_t ev;
	CK(ctx, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
	cudaError_t e = cudaEventRecord(ev, ctx->stream);
	if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->upload_stream, ev, 0);
	if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->upload_stream2, ev, 0);
	if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->copy_stream, ev, 0);
	cudaEventDestroy(ev);
	if (e != cudaSuccess) return set_err(ctx, DFB_ERR_CUDA, "stream ordering failed: %s", cudaGetErrorString(e));
	return DFB_OK;
}

static bool any_fast_class(bool simple, const dfb_split_params* params)
{
	dfb_plan probe;
	classify_params(&probe, params->match, params->mismatch, params->gap, simple || (params->end_gaps == 0 && params->min_split_score >= 1));
	for (int c = 0; c < kNumClasses; c++)
		if (probe.fast_ok[c]) return true;
	return false;
}

// A chunk with tasks only the s32 kernels take: its offsets and task arrays come to the host and the host builder makes
// its job lists; the raw bytes go device to device.  *d2h counts what crossed.
static int plan_create_from_device(dfb_ctx* ctx, bool simple, const dfb_split_params* params, const dfb_seq_table* A, const dfb_seq_table* B,
                                   const int32_t* ta, const int32_t* tb, const int32_t* tm, int64_t n_tasks, int32_t a_base, int32_t b_base,
                                   int stage_slot, cudaStream_t up_stream, int64_t* d2h, dfb_plan** out)
{
	std::vector<int64_t> ha((size_t)A->n + 1), hb((size_t)B->n + 1);
	std::vector<int32_t> hta((size_t)n_tasks), htb((size_t)n_tasks), htm(simple ? 0 : (size_t)n_tasks);
	cudaStream_t cs = ctx->copy_stream;
	CK(ctx, cudaMemcpyAsync(ha.data(), A->off, ha.size() * 8, cudaMemcpyDeviceToHost, cs));
	CK(ctx, cudaMemcpyAsync(hb.data(), B->off, hb.size() * 8, cudaMemcpyDeviceToHost, cs));
	if (n_tasks)
	{
		CK(ctx, cudaMemcpyAsync(hta.data(), ta, (size_t)n_tasks * 4, cudaMemcpyDeviceToHost, cs));
		CK(ctx, cudaMemcpyAsync(htb.data(), tb, (size_t)n_tasks * 4, cudaMemcpyDeviceToHost, cs));
		if (!simple) CK(ctx, cudaMemcpyAsync(htm.data(), tm, (size_t)n_tasks * 4, cudaMemcpyDeviceToHost, cs));
	}
	CK(ctx, cudaStreamSynchronize(cs));
	*d2h += (int64_t)(ha.size() + hb.size()) * 8 + n_tasks * (simple ? 8 : 12);
	const dfb_seq_table a{A->bytes, ha.data(), A->n}, b{B->bytes, hb.data(), B->n};
	return plan_create_host(ctx, simple, params, &a, &b, hta.data(), htb.data(), simple ? nullptr : htm.data(), n_tasks, a_base, b_base,
	                        stage_slot, up_stream, out, true);
}

static int dfb_simple_align_device_body(dfb_ctx* ctx, const dfb_simple_params* params, const dfb_device_seq_table* refs,
                                        const dfb_device_seq_table* seqs, const int32_t* task_ref, const int32_t* task_seq, int64_t n_tasks,
                                        int32_t* out_score)
{
	if (!ctx) return DFB_ERR_ARG;
	CK(ctx, cudaSetDevice(ctx->device));
	DeviceCheck chk;
	int rc = check_device_args(ctx, true, params, refs, seqs, task_ref, task_seq, nullptr, n_tasks, out_score, &chk);
	if (rc || n_tasks == 0) return rc;
	if ((rc = order_side_streams(ctx))) return rc;
	const dfb_split_params sp{params->match, params->mismatch, params->gap, 0, 0};
	const dfb_seq_table a{refs->bytes, refs->off, refs->n}, b{seqs->bytes, seqs->off, seqs->n};
	const int64_t range[4] = {0, chk.tab[0].off_n, 0, chk.tab[1].off_n};
	// one chunk: a simple batch keeps no first-sweep state
	dfb_plan* pl = nullptr;
	rc = DFB_BUILD_ON_HOST;
	if (any_fast_class(true, &sp))
	{
		rc = device_build_enqueue(ctx, true, &sp, &a, &b, task_ref, task_seq, nullptr, n_tasks, 0, 0, 0, &pl, range);
		if (!rc) rc = device_build_kernels(pl);
		if (!rc) rc = device_build_finish(pl);
		if (rc && pl)
		{
			dfb_plan_destroy(pl);
			pl = nullptr;
		}
	}
	int64_t d2h = 0;
	if (rc == DFB_BUILD_ON_HOST) rc = plan_create_from_device(ctx, true, &sp, &a, &b, task_ref, task_seq, nullptr, n_tasks, 0, 0, 0, nullptr, &d2h, &pl);
	if (!rc) rc = plan_run_impl(pl, nullptr);
	if (!rc)
	{
		cudaError_t e = cudaMemcpyAsync(out_score, pl->d_out, (size_t)n_tasks * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream);
		if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
		if (e != cudaSuccess) rc = set_err(ctx, DFB_ERR_CUDA, "simple device batch failed: %s", cudaGetErrorString(e));
	}
	if (!rc) rc = bounds_check_status(ctx);
	if (pl) dfb_plan_destroy(pl);
	return rc;
}

static int bit_width(unsigned long long v)
{
	int b = 0;
	while (v) { b++; v >>= 1; }
	return b;
}

// exclusive scan of v[0, n) in place on the context's stream; the total goes to *total (device)
static int scan_u64(dfb_ctx* ctx, unsigned long long* v, long long n, unsigned long long* sums, unsigned long long* total)
{
	const long long blocks = std::max<long long>(1, (n + DFB_BUILD_BLOCK * DFB_BUILD_ITEMS - 1) / (DFB_BUILD_BLOCK * DFB_BUILD_ITEMS));
	u64_scan_sums_kernel<<<(unsigned)blocks, DFB_BUILD_BLOCK, 0, ctx->stream>>>(v, n, sums);
	desc_scan_kernel<<<1, DFB_BUILD_BLOCK, 0, ctx->stream>>>(sums, blocks, nullptr, total);
	u64_scan_write_kernel<<<(unsigned)blocks, DFB_BUILD_BLOCK, 0, ctx->stream>>>(v, n, sums);
	CK(ctx, cudaGetLastError());
	return DFB_OK;
}

// The rows of chunk `pl` into the batch's arrays (dfb_assemble.cuh, "overflow list assembled on the device"): n_ov overflow
// events, g_rows / g_cols rows and columns of the region assembly; d_base holds the batch's totals before the chunk and
// is advanced past it.
static int assemble_chunk_device(dfb_plan* pl, unsigned long long n_ov, long long g_rows, long long g_cols, int32_t task_shift,
                                 const int64_t* read_off, const int32_t* task_read, OvKey key, int passes, unsigned long long* d_base,
                                 dfb_split_row* out_rows, int32_t* out_cols)
{
	dfb_ctx* ctx = pl->ctx;
	cudaStream_t s = ctx->stream;
	const long long n = (long long)n_ov, n_x_bound = n / 2 + 1;
	unsigned long long* scal = nullptr;
	dfb_split_row* x_rows = nullptr;
	Event* tmp = nullptr;
	unsigned long long *hist = nullptr, *head = nullptr, *sums = nullptr, *g_r = nullptr, *g_c = nullptr;
	long long* g_first = nullptr;
	int32_t *g_match = nullptr, *g_mb = nullptr;
	int rc = DFB_OK;
	auto cleanup = [&]() {
		dfree(ctx, scal);
		dfree(ctx, x_rows);
		dfree(ctx, tmp);
		dfree(ctx, hist);
		dfree(ctx, head);
		dfree(ctx, sums);
		dfree(ctx, g_r);
		dfree(ctx, g_c);
		dfree(ctx, g_first);
		dfree(ctx, g_match);
		dfree(ctx, g_mb);
	};
	if (n)
	{
		const long long nb = (n + DFB_OV_BLOCK - 1) / DFB_OV_BLOCK;
		const long long scan_len = std::max<long long>(256 * nb, n);
		cudaError_t e = cudaSuccess;
		auto take = [&](void** p, size_t bytes) {
			if (e == cudaSuccess) e = dalloc(ctx, p, bytes);
		};
		take((void**)&scal, 4 * sizeof(unsigned long long));
		take((void**)&x_rows, (size_t)n_x_bound * sizeof(dfb_split_row));
		take((void**)&tmp, (size_t)n * sizeof(Event));
		take((void**)&hist, (size_t)256 * nb * sizeof(unsigned long long));
		take((void**)&head, (size_t)n * sizeof(unsigned long long));
		take((void**)&sums, (size_t)(scan_len / (DFB_BUILD_BLOCK * DFB_BUILD_ITEMS) + 2) * sizeof(unsigned long long));
		take((void**)&g_r, (size_t)n * sizeof(unsigned long long));
		take((void**)&g_c, (size_t)n * sizeof(unsigned long long));
		take((void**)&g_first, (size_t)(n + 1) * sizeof(long long));
		take((void**)&g_match, (size_t)n * sizeof(int32_t));
		take((void**)&g_mb, (size_t)n * sizeof(int32_t));
		if (e != cudaSuccess)
		{
			cleanup();
			return set_err(ctx, DFB_ERR_NOMEM, "overflow assembly buffers for %lld events: %s", n, cudaGetErrorString(e));
		}
		// 1. radix sort: (matrix, row, column) passes, then task passes
		Event* src = pl->d_events;
		Event* dst = tmp;
		for (int pass = 0; pass < passes && !rc; pass++)
		{
			ov_hist_kernel<<<(unsigned)nb, DFB_OV_BLOCK, 0, s>>>(src, n, pass, key, hist, nb);
			rc = scan_u64(ctx, hist, 256 * nb, sums, scal + 3);
			ov_scatter_kernel<<<(unsigned)nb, DFB_OV_BLOCK, 0, s>>>(src, dst, n, pass, key, hist, nb);
			std::swap(src, dst);
		}
		OvAsmParams p;
		p.ev = src;
		p.n = n;
		p.head = head;
		p.scal = scal;
		p.g_first = g_first;
		p.g_match = g_match;
		p.g_matched_by = g_mb;
		p.g_rows = g_r;
		p.g_cols = g_c;
		p.read_off = read_off;
		p.task_read = task_read;
		p.task_base = task_shift;
		p.x_rows = x_rows;
		p.asm_cols = g_cols;
		p.cols = out_cols;
		p.base = d_base;
		// 2.-4. groups, pairs, rows, columns
		if (!rc)
		{
			ov_head_kernel<<<(unsigned)nb, DFB_OV_BLOCK, 0, s>>>(p);
			rc = scan_u64(ctx, head, n, sums, scal + 0);
		}
		if (!rc)
		{
			ov_group_kernel<<<(unsigned)nb, DFB_OV_BLOCK, 0, s>>>(p);
			cudaMemsetAsync(g_mb, 0xff, (size_t)n * sizeof(int32_t), s);
			ov_match_kernel<<<(unsigned)nb, DFB_OV_BLOCK, 0, s>>>(p);
			rc = scan_u64(ctx, g_r, n, sums, scal + 1);
		}
		if (!rc) rc = scan_u64(ctx, g_c, n, sums, scal + 2);
		if (!rc)
		{
			ov_rows_kernel<<<(unsigned)nb, DFB_OV_BLOCK, 0, s>>>(p);
			ov_cols_kernel<<<(unsigned)nb, DFB_OV_BLOCK, 0, s>>>(p);
		}
	}
	// 5. merge by task into the batch's arrays, columns of the region part first
	const long long items = g_rows + (n ? n_x_bound : 0) + g_cols;
	if (!rc && items)
		ov_place_kernel<<<(unsigned)((items + DFB_OV_BLOCK - 1) / DFB_OV_BLOCK), DFB_OV_BLOCK, 0, s>>>(
		    pl->d_asm_rows, g_rows, pl->d_asm_cols, g_cols, x_rows, n ? n_x_bound : 0, n ? scal : nullptr, task_shift, d_base, out_rows, out_cols);
	if (!rc) ov_advance_kernel<<<1, 1, 0, s>>>(d_base, g_rows, g_cols, n ? scal : nullptr);
	if (!rc)
	{
		cudaError_t e = cudaGetLastError();
		if (e != cudaSuccess) rc = set_err(ctx, DFB_ERR_CUDA, "overflow assembly kernels: %s", cudaGetErrorString(e));
	}
	cleanup();
	return rc;
}

// grows a device array of the batch's results (stream-ordered), keeping its first `cap` entries
template <class T>
static int grow_device(dfb_ctx* ctx, T*& p, int64_t& cap, int64_t need)
{
	if (need <= cap) return DFB_OK;
	const int64_t ncap = need + need / 2 + 1024;
	T* q = nullptr;
	CK(ctx, dalloc(ctx, (void**)&q, (size_t)ncap * sizeof(T)));
	if (p) CK(ctx, cudaMemcpyAsync(q, p, (size_t)cap * sizeof(T), cudaMemcpyDeviceToDevice, ctx->stream));
	dfree(ctx, p);
	p = q;
	cap = ncap;
	return DFB_OK;
}

static int dfb_split_align_device_body(dfb_ctx* ctx, const dfb_split_params* params, const dfb_device_seq_table* refs,
                                       const dfb_device_seq_table* reads, const int32_t* task_cluster, const int32_t* task_read,
                                       const int32_t* task_min_score, int64_t n_tasks, int32_t* out_best, int64_t* n_rows, int64_t* n_cols)
{
	if (!ctx) return DFB_ERR_ARG;
	if (ctx->last_split)
	{
		dfb_plan_destroy(ctx->last_split);
		ctx->last_split = nullptr;
	}
	CK(ctx, cudaSetDevice(ctx->device));
	DeviceCheck chk;
	int rc = check_device_args(ctx, false, params, refs, reads, task_cluster, task_read, task_min_score, n_tasks, out_best, &chk);
	if (rc) return rc;
	if ((rc = order_side_streams(ctx))) return rc;
	dfb_plan* holder = new (std::nothrow) dfb_plan();
	if (!holder) return set_err(ctx, DFB_ERR_NOMEM, "out of host memory");
	holder->ctx = ctx;
	holder->split = true;
	holder->n_tasks = n_tasks;
	holder->stats.n_tasks = n_tasks;
	holder->device_result = true;
	holder->stats.d2h_bytes = (int64_t)sizeof(DeviceCheck);
	auto fail = [&](int code) {
		dfb_plan_destroy(holder);
		return code;
	};
	// the host form's chunks (split_chunk_starts), so that the column pool comes out the same
	const bool chunked = n_tasks >= pipeline_min_tasks() && !chk.b_decreases;
	std::vector<int64_t> t0 = chunked ? split_chunk_starts(n_tasks) : std::vector<int64_t>{0, n_tasks};
	if (!n_tasks) t0.resize(1); // (no chunk)
	const int K = (int)t0.size() - 1;
	static_assert(dfb_ctx::kStageSlots <= DFB_MAX_CHUNKS, "ChunkStarts too small");
	// chunk views: a_lo, a_hi, b_lo, b_hi and their byte offsets
	std::vector<int64_t> bnd((size_t)std::max(K, 1) * 8, 0);
	if (chunked)
	{
		ChunkStarts cs;
		for (int k = 0; k <= K; k++) cs.t[k] = t0[(size_t)k];
		long long* d_bnd = nullptr;
		if (cudaError_t e = dalloc(ctx, (void**)&d_bnd, bnd.size() * sizeof(long long)))
			return fail(set_err(ctx, DFB_ERR_NOMEM, "chunk bounds: %s", cudaGetErrorString(e)));
		chunk_bounds_kernel<<<1, 32, 0, ctx->stream>>>(refs->off, refs->n / 2, 2, reads->off, task_cluster, task_read, cs, K,
		                                               chk.a_decreases ? 0 : 1, d_bnd);
		cudaError_t e = cudaMemcpyAsync(ctx->h_out.p, d_bnd, bnd.size() * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream);
		if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
		dfree(ctx, d_bnd);
		if (e != cudaSuccess) return fail(set_err(ctx, DFB_ERR_CUDA, "chunk bounds: %s", cudaGetErrorString(e)));
		memcpy(bnd.data(), ctx->h_out.p, bnd.size() * sizeof(long long));
		holder->stats.d2h_bytes += (int64_t)(bnd.size() * sizeof(long long));
	}
	else if (K)
	{
		const int64_t one[8] = {0, refs->n / 2, 0, reads->n, 0, (int64_t)chk.tab[0].off_n, 0, (int64_t)chk.tab[1].off_n};
		memcpy(bnd.data(), one, sizeof(one));
	}
	// chunk k's views: entries o[0] .. o[1] of the clusters and o[2] .. o[3] of the reads, bytes o[4] .. o[5] and o[6] .. o[7]
	auto view_of = [&](int k, ChunkView& v) -> int {
		const int64_t* o = bnd.data() + 8 * (size_t)k;
		v.a = dfb_seq_table{refs->bytes, refs->off + 2 * o[0], 2 * (o[1] - o[0])};
		v.b = dfb_seq_table{reads->bytes, reads->off + o[2], o[3] - o[2]};
		v.a_lo = (int32_t)o[0];
		v.b_lo = (int32_t)o[2];
		v.range = o + 4;
		return DFB_OK;
	};
	int64_t host_d2h = 0;
	auto host_plan = [&](int k, const ChunkView& v, dfb_plan** out) -> int {
		const int64_t a = t0[(size_t)k];
		return plan_create_from_device(ctx, false, params, &v.a, &v.b, task_cluster + a, task_read + a, task_min_score + a, t0[(size_t)k + 1] - a,
		                               v.a_lo, v.b_lo, k, ctx->upload_stream, &host_d2h, out);
	};
	// sort key widths of the overflow events: rows <= longest read, columns <= longest window
	OvKey key;
	key.rb = bit_width(chk.tab[1].max_len + 1);
	key.cb = bit_width(chk.tab[0].max_len + 1);
	key.sub_passes = (1 + key.rb + key.cb + 7) / 8;
	std::vector<dfb_plan*> plans((size_t)K, nullptr);
	unsigned long long* d_base = nullptr; // the batch's row and column totals so far
	int64_t rows_cap = 0, cols_cap = 0, rows_bound = 0, cols_bound = 0;
	if (cudaError_t e = dalloc(ctx, (void**)&d_base, 2 * sizeof(unsigned long long))) return fail(set_err(ctx, DFB_ERR_NOMEM, "%s", cudaGetErrorString(e)));
	if (cudaError_t e = cudaMemsetAsync(d_base, 0, 2 * sizeof(unsigned long long), ctx->stream)) rc = set_err(ctx, DFB_ERR_CUDA, "%s", cudaGetErrorString(e));
	auto collect = [&](int k) -> int {
		dfb_plan* pl = plans[(size_t)k];
		cudaStream_t cs = ctx->copy_stream;
		CK(ctx, wait_event(pl->done_ev));
		CK(ctx, cudaStreamWaitEvent(cs, pl->done_ev, 0));
		int h_ctrl[kNumClasses * 4];
		unsigned long long n_ov = 0, asm_totals[2] = {0, 0};
		if (int frc = fetch_counters(pl, cs, h_ctrl, &n_ov, asm_totals)) return frc;
		if (int brc = bounds_check_status(ctx)) return brc;
		holder->stats.d2h_bytes += (int64_t)(sizeof(n_ov) + sizeof(h_ctrl) + (pl->d_asm_sums ? sizeof(asm_totals) : 0));
		for (int c = 0; c < kNumClasses; c++)
			if (pl->cls[c].n_jobs) holder->stats.probe_jobs += (int64_t)h_ctrl[4 * c + 1] + h_ctrl[4 * c + 3];
		const int64_t a = t0[(size_t)k], nk = t0[(size_t)k + 1] - a;
		CK(ctx, cudaMemcpyAsync(out_best + a, pl->d_out, (size_t)nk * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
		rows_bound += (int64_t)asm_totals[0] + (int64_t)(n_ov / 2 + 1);
		cols_bound += (int64_t)asm_totals[1] + (int64_t)n_ov;
		int grc = grow_device(ctx, holder->d_res_rows, rows_cap, rows_bound);
		if (!grc) grc = grow_device(ctx, holder->d_res_cols, cols_cap, cols_bound);
		if (grc) return grc;
		const int64_t task_bits = bit_width((unsigned long long)std::max<int64_t>(nk - 1, 0));
		const int passes = key.sub_passes + (int)((task_bits + 7) / 8);
		int arc = assemble_chunk_device(pl, n_ov, (long long)asm_totals[0], (long long)asm_totals[1], (int32_t)a, reads->off, task_read, key,
		                                passes, d_base, holder->d_res_rows, holder->d_res_cols);
		holder->stats.cells += pl->stats.cells;
		holder->stats.fast_jobs += pl->stats.fast_jobs;
		holder->stats.generic_jobs += pl->stats.generic_jobs;
		holder->stats.kernel_launches += pl->stats.kernel_launches;
		holder->stats.h2d_bytes += pl->stats.h2d_bytes;
		holder->stats.d2h_bytes += pl->stats.d2h_bytes;
		holder->stats.raw_bytes += pl->stats.raw_bytes;
		holder->stats.packed_bytes += pl->stats.packed_bytes;
		release_device(pl);
		return arc;
	};
	// chunk k-1 is collected once chunk k is queued: its assembly runs behind chunk k's sweeps
	auto queued = [&](int k) -> int { return k ? collect(k - 1) : DFB_OK; };
	unsigned long long totals[2] = {0, 0};
	auto done = [&](int brc) -> int {
		if (!brc && K) brc = collect(K - 1);
		if (!brc)
		{
			cudaError_t e = cudaMemcpyAsync(ctx->h_out.p, d_base, sizeof(totals), cudaMemcpyDeviceToHost, ctx->stream);
			if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
			if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->copy_stream);
			if (e != cudaSuccess) brc = set_err(ctx, DFB_ERR_CUDA, "split device batch failed: %s", cudaGetErrorString(e));
			else memcpy(totals, ctx->h_out.p, sizeof(totals));
			holder->stats.d2h_bytes += (int64_t)sizeof(totals) + host_d2h;
		}
		if (!brc) brc = bounds_check_status(ctx);
		return brc;
	};
	Trace tr;
	if (!rc)
		rc = pipeline_run(ctx, false, params, task_cluster, task_read, task_min_score, t0, any_fast_class(false, params), view_of, host_plan,
		                  plans, queued, done);
	dfree(ctx, d_base);
	tr.lap("split device: done");
	if (rc) return fail(rc);
	holder->d_res_n_rows = (int64_t)totals[0];
	holder->d_res_n_cols = (int64_t)totals[1];
	holder->stats.events = (int64_t)totals[1];
	holder->ran = holder->fetched = true;
	if (n_rows) *n_rows = holder->d_res_n_rows;
	if (n_cols) *n_cols = holder->d_res_n_cols;
	ctx->last_split = holder;
	return DFB_OK;
}

extern "C" int dfb_split_result_copy_device(dfb_ctx* ctx, dfb_split_row* rows, int32_t* cols)
{
	if (!ctx) return DFB_ERR_ARG;
	const dfb_plan* h = ctx->last_split;
	if (!h || !h->device_result) return set_err(ctx, DFB_ERR_STATE, "no device-resident split result on this context");
	if ((h->d_res_n_rows && !rows) || (h->d_res_n_cols && !cols)) return set_err(ctx, DFB_ERR_ARG, "dfb_split_result_copy_device: null argument");
	CK(ctx, cudaSetDevice(ctx->device));
	if (!is_ctx_device_memory(ctx, rows)) return set_err(ctx, DFB_ERR_ARG, "rows is not device memory of device %d", ctx->device);
	if (!is_ctx_device_memory(ctx, cols)) return set_err(ctx, DFB_ERR_ARG, "cols is not device memory of device %d", ctx->device);
	if (h->d_res_n_rows)
		CK(ctx, cudaMemcpyAsync(rows, h->d_res_rows, (size_t)h->d_res_n_rows * sizeof(dfb_split_row), cudaMemcpyDeviceToDevice, ctx->stream));
	if (h->d_res_n_cols)
		CK(ctx, cudaMemcpyAsync(cols, h->d_res_cols, (size_t)h->d_res_n_cols * sizeof(int32_t), cudaMemcpyDeviceToDevice, ctx->stream));
	CK(ctx, cudaStreamSynchronize(ctx->stream));
	return DFB_OK;
}

extern "C" int dfb_simple_align_device(dfb_ctx* ctx, const dfb_simple_params* params, const dfb_device_seq_table* refs,
                                       const dfb_device_seq_table* seqs, const int32_t* task_ref, const int32_t* task_seq, int64_t n_tasks,
                                       int32_t* out_score)
{
	return guarded(ctx, [&] { return dfb_simple_align_device_body(ctx, params, refs, seqs, task_ref, task_seq, n_tasks, out_score); });
}

extern "C" int dfb_split_align_device(dfb_ctx* ctx, const dfb_split_params* params, const dfb_device_seq_table* refs,
                                      const dfb_device_seq_table* reads, const int32_t* task_cluster, const int32_t* task_read,
                                      const int32_t* task_min_score, int64_t n_tasks, int32_t* out_best, int64_t* n_rows, int64_t* n_cols)
{
	return guarded(ctx, [&] {
		return dfb_split_align_device_body(ctx, params, refs, reads, task_cluster, task_read, task_min_score, n_tasks, out_best, n_rows, n_cols);
	});
}

#include "dfb_trace.cuh"
#include "dfb_records.cuh"
