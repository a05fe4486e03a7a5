// Device code of the deFuse DP hot path for sm_100a.
//
// Replaces (batch form, bit-exact):
//   SplitReadAligner::FillMatrix / Align / FindMaxRowEntry / GetAlignments
//       /root/reference tools/SplitReadAligner.cpp:24-75, 77-89, 91-122, 156-298
//   SimpleAligner::Align
//       tools/SimpleAligner.cpp:23-63
//
// Design (see DESIGN.md): no DP matrix is ever stored.  A group of G lanes owns G*S read
// rows (S per lane, in registers) and sweeps the reference one column per step as a skewed
// wavefront; lane g hands the last row of its strip to lane g+1 with one SHFL per step.
// In the s16x2 kernel every 32-bit register holds TWO independent DPs (low/high half),
// advanced by DPX instructions: per register pair of cells the steady-state loop issues
// VIADDMNMX.U16x2 (mismatch indicator), IMAD (diagonal), VIADDMNMX.S16x2 x2 (the two maxima)
// and half a VIMNMX3.S16x2 (row-maximum sink, one per two columns).  Reference words reach
// shared memory by cp.async (LDGSTS) one ring block ahead of the wavefront.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>

namespace dfb
{

// -DDFB_BOUNDS_CHECK: every indexed global-memory access of the kernels is range-checked against the size of its buffer
// (compute-sanitizer is closed on the GPU pool this was developed on).  The first violation is recorded -- the access
// still happens -- and the host turns it into an error at the next fetch / sync.  Compiled out otherwise.
#ifdef DFB_BOUNDS_CHECK
__device__ int g_dfb_bounds_err = 0;
#define DFB_BC(cond, code)                                      \
	do                                                          \
	{                                                           \
		if (!(cond)) atomicCAS(&g_dfb_bounds_err, 0, (code));   \
	} while (0)
#else
#define DFB_BC(cond, code) \
	do                     \
	{                      \
	} while (0)
#endif

// ------------------------------------------------------------------------------------------
// HBM layout of sequences
// ------------------------------------------------------------------------------------------
// Every sequence (already in the orientation its DP consumes it) is stored 16 bases per
// "word":   pool[w] = { codes: 16 x 2 bit (A,C,G,T = 0..3, base n at bits 2n..2n+1),
//                       mask : bit n set  <=>  base n is NOT one of ACGT (exception plane) }
// and, for the exception plane only, obytes[16*w + n] keeps the raw byte so that equality is
// exact for every byte value (the reference compares raw bytes: SplitReadAligner.cpp:51,
// SimpleAligner.cpp:50).  A sequence starts on a word boundary.

struct SeqDesc
{
	int64_t src;   // offset of the first byte in the raw upload
	uint32_t len;  // bases
	uint32_t word; // first pool word of this sequence's (first) stored copy
};

enum
{
	PACK_FWD = 0,     // one forward copy per sequence
	PACK_REV_ODD = 1, // even table entries forward, odd entries reversed (reference2 of each cluster)
	PACK_BOTH = 2     // forward copy at `word`, reversed copy right behind it (reads of the split aligner)
};

// Sixteen lanes per sequence (a 100-bp read in both orientations is 14 words, a 340-bp window 22): the owner of a
// word is known without a search and a sequence's words are written side by side.  Per 16-base word: the 16-byte
// source window through five aligned 32-bit loads + funnel shifts (adjacent lanes read adjacent windows, so the
// sectors are fully used), four bytes at a time through the 2-bit code / exception test (SWAR, no per-byte loop),
// 8 bytes written.  The raw copy of a word is written only when it has an exception.  The raw upload is padded by
// 16 bytes in front and 32 behind so that the window never leaves the allocation.
__device__ __forceinline__ void pack4(uint32_t w, uint32_t valid, uint32_t& codes8, uint32_t& mask4)
{
	// A=0x41 C=0x43 G=0x47 T=0x54: bits 2..1 are 00 01 11 10 (Gray) -> code 0..3; exact iff the code decodes back
	const uint32_t gray = (w >> 1) & 0x03030303u;
	const uint32_t code = gray ^ ((gray >> 1) & 0x01010101u);
	const uint32_t c1 = code & 0x01010101u, c2 = (code >> 1) & 0x01010101u;
	const uint32_t back = 0x41414141u + 2u * c1 + 6u * c2 + 11u * (c1 & c2); // 'A' + {0, 2, 6, 0x13}
	const uint32_t diff = w ^ back;
	const uint32_t bad = ((diff | ((diff & 0x7F7F7F7Fu) + 0x7F7F7F7Fu)) >> 7) & 0x01010101u & valid; // 1 per byte that is not ACGT
	const uint32_t good = code & (valid * 3u) & ~(bad * 3u);
	codes8 = (good * 0x01041040u) >> 24; // byte k's two bits -> bits 2k..2k+1
	mask4 = (bad * 0x01020408u) >> 24;   // byte k's flag -> bit k
}

template <int MODE>
__global__ void __launch_bounds__(256) pack_kernel(const uint8_t* __restrict__ raw, const SeqDesc* __restrict__ descs,
                                                    int n_seqs, uint2* __restrict__ pool, uint8_t* __restrict__ obytes,
                                                    unsigned long long pool_words, unsigned long long raw_bytes)
{
	(void)pool_words;
	(void)raw_bytes;
	const uint32_t lane16 = threadIdx.x & 15u;
	const uint32_t n_groups = (gridDim.x * blockDim.x) >> 4;
	for (uint32_t lo = (blockIdx.x * blockDim.x + threadIdx.x) >> 4; lo < (uint32_t)n_seqs; lo += n_groups)
	{
		const SeqDesc sd = descs[lo];
		const uint32_t nw = (sd.len + 15u) >> 4;
		const uint32_t seq_words = nw * (MODE == PACK_BOTH ? 2u : 1u);
		for (uint32_t local_all = lane16; local_all < seq_words; local_all += 16u)
		{
			const uint32_t w = sd.word + local_all;
			uint32_t local = local_all;
			bool rev = false;
			if (MODE == PACK_REV_ODD) rev = (lo & 1u) != 0;
			if (MODE == PACK_BOTH && local >= nw) { rev = true; local -= nw; }
			const uint32_t first = local * 16u;
			const uint32_t n_valid = min(16u, sd.len - first);
			// source window: forward bytes [first, first+16); reversed bytes [len-first-16, len-first) read backwards
			const int64_t win = sd.src + (rev ? (int64_t)sd.len - (int64_t)first - 16 : (int64_t)first);
			const uintptr_t addr = reinterpret_cast<uintptr_t>(raw + win);
			const uint32_t* ap = reinterpret_cast<const uint32_t*>(addr & ~(uintptr_t)3);
			const uint32_t sh = (uint32_t)(addr & 3u) * 8u;
			const uint32_t a0 = __ldg(ap), a1 = __ldg(ap + 1), a2 = __ldg(ap + 2), a3 = __ldg(ap + 3), a4 = __ldg(ap + 4);
			uint32_t b[4];
			b[0] = __funnelshift_r(a0, a1, sh);
			b[1] = __funnelshift_r(a1, a2, sh);
			b[2] = __funnelshift_r(a2, a3, sh);
			b[3] = __funnelshift_r(a3, a4, sh);
			if (rev)
			{
				const uint32_t r0 = __byte_perm(b[3], 0, 0x0123), r1 = __byte_perm(b[2], 0, 0x0123);
				const uint32_t r2 = __byte_perm(b[1], 0, 0x0123), r3 = __byte_perm(b[0], 0, 0x0123);
				b[0] = r0; b[1] = r1; b[2] = r2; b[3] = r3;
			}
			uint32_t codes = 0, mask = 0;
#pragma unroll
			for (int q = 0; q < 4; q++)
			{
				// bytes of this quad inside the sequence: 0x01 per valid byte
				const int keep = (int)n_valid - 4 * q;
				const uint32_t valid = keep >= 4 ? 0x01010101u : (keep <= 0 ? 0u : (0x01010101u >> (8 * (4 - keep))));
				uint32_t c8, m4;
				pack4(b[q], valid, c8, m4);
				codes |= c8 << (8 * q);
				mask |= m4 << (4 * q);
				b[q] &= valid * 0xFFu; // the raw copy keeps zeros beyond the sequence end
			}
			DFB_BC((unsigned long long)w < pool_words && win >= 0 && (unsigned long long)(win + 20) <= raw_bytes, 101);
			pool[w] = make_uint2(codes, mask);
			if (mask) reinterpret_cast<uint4*>(obytes)[w] = make_uint4(b[0], b[1], b[2], b[3]);
		}
	}
}

// ------------------------------------------------------------------------------------------
// s16x2 wavefront kernel
// ------------------------------------------------------------------------------------------

// Two DPs ("halves") that travel in the low and high 16 bits of every register.
struct JobPair
{
	uint32_t ref_w[2];  // first pool word of each half's reference (already oriented)
	uint32_t read_w[2]; // first pool word of each half's read (already oriented)
	uint16_t R[2];      // reference lengths
	uint16_t L[2];      // read lengths
	int32_t out0;       // SIMPLE: task index of half 0 (-1: none).  SPLIT: task index
	int32_t out1;       // SIMPLE: task index of half 1 (-1: none).  SPLIT: minScore
};

struct Event
{
	int32_t task;
	int32_t half_row; // (half << 30) | row
	int32_t col;      // matrix column index i (1-based over the oriented reference)
	int32_t score;    // the row maximum this column attains
};

enum
{
	MODE_SIMPLE = 0, // SimpleAligner::Align: best interior cell
	MODE_SPLIT = 1,  // SplitReadAligner first sweep: per-row maxima -> best split -> probe queue
	MODE_PROBE = 2   // second sweep of the winning tasks: every column attaining a winning row max
};

struct FastParams
{
	const uint2* pool;
	const uint8_t* obytes;
	const JobPair* jobs;
	int n_jobs;
	int* cursor; // work queue position (SIMPLE/SPLIT: over jobs; PROBE: over hitq)
	// scoring, pre-packed for the two halves
	int m;           // match
	uint32_t bias;   // B: stored value = H - m*j + B, kept in [8, B]
	uint32_t xm;     // (mismatch - match) as a 32-bit multiplier of the 0/1 mismatch indicator
	uint32_t g2;     // gap in both halves
	uint32_t gm2;    // gap - match in both halves
	int min_split;   // SPLIT: minSplitScore
	// outputs
	int32_t* out;    // SIMPLE: score per task.  SPLIT: best per task
	int* hit_count;  // SPLIT (write) / PROBE (read): queued tasks with a one-block window (slots from the front)
	int* hit_count_long; // ... with a longer window (slots from the back), so that a warp's job pairs run equally long
	int* hitq;       // job index per queue slot
	uint32_t* ntg;   // [slot][S][G] negated row-max targets (or "row disabled")
	uint32_t* rdq;   // [slot][S][G] the lanes' (negated) read symbols, so that the probe does not decode them again
	uint32_t* ckpt;  // [job][ckpt_blocks][S+2][G] wavefront state (F[S], prev, Flast) in front of every CH-th step (null: off)
	int ckpt_blocks; // checkpoints per job in this launch
	int gran_shift;  // a probe granule is 1 << gran_shift checkpoint blocks (so that a class' longest wavefront has <= 16 granules)
	int slot_base;   // SPLIT: first global slot number of this class (slots are numbered class by class)
	uint32_t* slot_rng; // per queue slot: granules to re-sweep, a 16-bit mask per half
	int32_t* slot_task; // SPLIT (write): task index per queue slot
	int32_t* task_slot; // SPLIT (write): queue slot per task, -1 when the task needs no second sweep
	uint2* slot_ev;     // PROBE: [slot][DFB_SLOT_EVENTS] {key = half<<27 | row<<16 | col, score}
	int* slot_n;        // PROBE: events found per slot (may exceed DFB_SLOT_EVENTS: the rest is in `events`)
	Event* events;      // PROBE: overflow list
	unsigned long long* ev_count;
	unsigned long long ev_cap;
	uint32_t ck[32]; // SIMPLE: m*(k+1) in both halves
	// buffer sizes (bounds-check builds)
	unsigned long long pool_words; // pool / obytes entries allocated
	unsigned long long ckpt_words; // ckpt entries allocated
	long long n_tasks;             // entries of out / task_slot
};

#define DFB_SLOT_EVENTS 16

// Symbols in shared memory and registers: the raw byte of a base in a 16-bit field (equality of symbols is equality
// of bytes: SplitReadAligner.cpp:51), and two padding values that equal nothing.
#define DFB_READ_PAD 0x7FFEu // read rows beyond L: never equals a reference field
#define DFB_REF_PAD 0xFFFFu  // reference columns beyond R: never equals a read field; bit 15 doubles as the row-max mask

__device__ __forceinline__ uint32_t decode_base(uint2 w, uint32_t word_index, int n, const uint8_t* __restrict__ obytes)
{
	if ((w.y >> n) & 1u)
	{
		return __ldg(obytes + (size_t)word_index * 16 + n); // exception plane: raw byte
	}
	return (0x54474341u >> (8 * ((w.x >> (2 * n)) & 3u))) & 0xFFu; // "ACGT"
}

__device__ __forceinline__ void cp_async_16(void* smem_dst, const void* gmem_src)
{
	const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
	asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// (the PTX instruction itself: __byte_perm masks its selector first, one more ALU-pipe instruction per use)
__device__ __forceinline__ uint32_t prmt(uint32_t lo, uint32_t hi, uint32_t selector)
{
	uint32_t r;
	asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(lo), "r"(hi), "r"(selector));
	return r;
}

// 0xFFFF in every half of x whose bit 15 is set, 0 in the others (PRMT with sign replication: bytes 1, 1, 3, 3)
__device__ __forceinline__ uint32_t spread_bit15(uint32_t x)
{
	uint32_t r;
	asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(x), "r"(0u), "r"(0xBB99u));
	return r;
}

// One arg-max column found by the probe sweep: the task's fixed region first, the overflow list after.
__device__ __noinline__ void emit_probe_event(const FastParams& p, int item, int task, int h, int j, int col, int score)
{
	DFB_BC(item >= 0 && item < p.n_jobs && task >= 0 && task < p.n_tasks && col >= 0 && col < 65535 && j >= 1 && j <= 1024, 305);
	const int n = atomicAdd(p.slot_n + item, 1);
	if (n < DFB_SLOT_EVENTS)
	{
		p.slot_ev[(size_t)item * DFB_SLOT_EVENTS + n] =
		    make_uint2(((uint32_t)h << 27) | ((uint32_t)j << 16) | (uint32_t)(col + 1), (uint32_t)score);
		return;
	}
	const unsigned long long idx = atomicAdd(p.ev_count, 1ull);
	if (idx < p.ev_cap)
	{
		Event ev;
		ev.task = task;
		ev.half_row = (h << 30) | j;
		ev.col = col + 1;
		ev.score = score;
		p.events[idx] = ev;
	}
}

// Steps of the wavefront per checkpoint block: the first sweep's row-maximum fold and checkpoint interval, the probe
// sweep's resume granularity.  4G, but at least 32: a four-lane group would otherwise fold and checkpoint every 16
// steps, twice the per-cell cost of both.  A reference ring block is two checkpoint blocks (CH = 2 CK columns).
__host__ __device__ constexpr int ckpt_steps(int G) { return G >= 8 ? 4 * G : 32; }

// Decodes one ring block (CH = 2 ckpt_steps(G) reference columns of both halves) from the raw pool words cp.async left in
// shared memory into 32-bit {half 1, half 0} symbol pairs.  Lane g owns CPL = CH/G columns (8; 16 for G = 4) starting at
// CPL*g and stores them in an order rotated by the lane, so that the 32 lanes of the warp hit 32 different banks.  cw0 / cw1: pool word of ring column 0
// in either half's reference (negative in front of the reference: those columns are padding).  The last G-1 columns of the
// ring are stored a second time in front of it (ring[-1] = ring[RING-1] ...): lane g of the first sweep reads column u-g
// at ring_lane[u mod RING] with ring_lane = ring - g and a warp-uniform index that needs no mask (MIRROR; the probe sweep
// masks its index and does without).  Out of line: three call
// sites per kernel, and the instruction cache is what short probe rounds wait for.
template <int G, bool MIRROR>
__device__ __noinline__ void ring_decode_block(uint32_t* ring, const uint2* raw_slot, int blk, int cw0, int cw1, uint32_t R0, uint32_t R1,
                                               uint32_t ref_w0, uint32_t ref_w1, const uint8_t* __restrict__ obytes, int g,
                                               unsigned long long pool_words)
{
	(void)pool_words;
	constexpr int CH = 2 * ckpt_steps(G), RING = 2 * CH;
	constexpr int WB = CH / 16;  // pool words of one half in a ring block
	constexpr int CPL = CH / G;  // columns per lane
	static_assert(CPL == 8 || CPL == 16, "a lane decodes half a pool word or a whole one");
	// G >= 8 (rings RING + G = 8 mod 32 words apart): bank = 8 * (g + q * G / 8) + rotation (mod 32): distinct over the warp.
	// G = 4 (rings 4 mod 32 apart, 16 columns per lane): bank = 4q + 16g + ((n + g) mod 16) + 4 (mod 32) is (n + g) mod 4,
	// distinct over the four lanes of a group, and the eight groups shift it by 4q: each residue class once.
	constexpr int RSH = (G <= 8) ? 0 : (G == 16 ? 1 : 2);
	const int wl = (g * CPL) >> 4;   // the lane's pool word in the block
	const int bit0 = (g * CPL) & 15; // and its first base in that word
	const uint2 w0 = raw_slot[wl], w1 = raw_slot[WB + wl];
	const int wrel = blk * WB + wl;
	const int wi0 = cw0 + wrel, wi1 = cw1 + wrel;
	// the lane's CPL bases of either half: 2-bit codes, exception flags, and how many of them lie inside the reference
	const uint32_t c0 = w0.x >> (2 * bit0), c1 = w1.x >> (2 * bit0);
	const int nv0 = wi0 < 0 ? 0 : min(CPL, max(0, (int)R0 - (wi0 * 16 + bit0)));
	const int nv1 = wi1 < 0 ? 0 : min(CPL, max(0, (int)R1 - (wi1 * 16 + bit0)));
	const uint32_t m0 = (w0.y >> bit0) & ((1u << nv0) - 1u), m1 = (w1.y >> bit0) & ((1u << nv1) - 1u);
	DFB_BC(nv0 == 0 || (unsigned long long)ref_w0 + (unsigned long long)wi0 < pool_words, 201);
	DFB_BC(nv1 == 0 || (unsigned long long)ref_w1 + (unsigned long long)wi1 < pool_words, 202);
	const int rot = g >> RSH;
	// ring slot of the lane's first column: a multiple of CPL, so + nn never wraps
	const int base_idx = (int)(((uint32_t)blk * CH + (uint32_t)(CPL * g)) & (RING - 1));
	uint32_t* dst = ring + base_idx;
	const int mirror_from = MIRROR ? RING - G - base_idx : 8; // columns nn > mirror_from have a mirror slot (RING words below)
	// Both halves of a column with one PRMT: the 2-bit codes of the two references sit in the two halves of cc; the
	// selector {code0, 4, code1, 4} picks {"ACGT"[code0], 0, "ACGT"[code1], 0} out of ("ACGT", 0).
	// (16 columns per lane do not fit one register that way: the two codes are gathered one by one)
	const uint32_t cc = (c0 & 0xFFFFu) | (c1 << 16);
#pragma unroll
	for (int n = 0; n < CPL; n++)
	{
		const int nn = (n + rot) & (CPL - 1);
		const uint32_t x = CPL == 8 ? (cc >> (2 * nn)) & 0x00030003u : ((c0 >> (2 * nn)) & 3u) | (((c1 >> (2 * nn)) & 3u) << 16);
		const uint32_t word = prmt(0x54474341u, 0u, x | (x >> 8) | 0x4040u);
		dst[nn] = word;
		if (MIRROR && nn > mirror_from) dst[nn - RING] = word;
	}
	uint16_t* dst16 = reinterpret_cast<uint16_t*>(dst);
	if (nv0 < CPL || nv1 < CPL)
	{
		// columns in front of a reference or at and past its end equal no read symbol (only the blocks at a reference's
		// ends have any)
		for (int nn = 0; nn < CPL; nn++)
		{
			const int mirror = (MIRROR && nn > mirror_from) ? nn - RING : nn; // (the same slot again when the column has no mirror)
			if (nn >= nv0) dst16[2 * nn] = dst16[2 * mirror] = (uint16_t)DFB_REF_PAD;
			if (nn >= nv1) dst16[2 * nn + 1] = dst16[2 * mirror + 1] = (uint16_t)DFB_REF_PAD;
		}
	}
	if (m0 | m1)
	{
		// exception plane (rare): the raw byte replaces the decoded code
		for (int nn = 0; nn < CPL; nn++)
		{
			const int mirror = (MIRROR && nn > mirror_from) ? nn - RING : nn;
			if ((m0 >> nn) & 1u) dst16[2 * nn] = dst16[2 * mirror] = __ldg(obytes + ((size_t)ref_w0 + (size_t)wi0) * 16 + bit0 + nn);
			if ((m1 >> nn) & 1u) dst16[2 * nn + 1] = dst16[2 * mirror + 1] = __ldg(obytes + ((size_t)ref_w1 + (size_t)wi1) * 16 + bit0 + nn);
		}
	}
}

// Probe sweep, rare path: rows of this lane (bit k of hm0 / hm1: row j0+k+1 of half 0 / 1) reached their targets in the
// column the lane has just computed.  Out of line and loop-shaped: the unrolled form of this test was most of the probe
// kernel's code.  The score of an event is the row's target, read back from the list the first sweep wrote.
__device__ __noinline__ void emit_probe_hits(const FastParams& p, int item, int task, uint32_t hm0, uint32_t hm1, int j0, int col0, int col1,
                                             uint32_t R0, uint32_t R1, int L, int S, int G, int g)
{
	for (int h = 0; h < 2; h++)
	{
		uint32_t hm = h ? hm1 : hm0;
		const int col = h ? col1 : col0;
		if (col < 0 || col >= (int)(h ? R1 : R0)) continue;
		while (hm)
		{
			const int k = __ffs(hm) - 1;
			hm &= hm - 1;
			const int j = j0 + k + 1;
			if (j > L) continue;
			const uint32_t x = p.ntg[((size_t)item * S + k) * G + g];
			const int target = (int)((0u - (h ? (x >> 16) : x)) & 0xFFFFu); // stored value of the row maximum
			emit_probe_event(p, item, task, h, j, col, target - (int)p.bias + p.m * j);
		}
	}
}

// registers per thread the mode needs (arrays of S) decide how many CTAs we ask ptxas to fit per SM.  Four-lane groups
// (25-row strips, granule masks in shared memory) fit 168 registers in either mode with no local-memory traffic in the
// pair loop (at 128, ptxas spills hundreds of bytes in SPLIT mode): three CTAs.
template <int G, int S, int MODE>
struct FastOcc
{
	static constexpr int kArrays = (MODE == MODE_SPLIT) ? 5 : 2;
	static constexpr int kEst = kArrays * S + 48;
#ifndef DFB_OCC_SMALL
#define DFB_OCC_SMALL 4 // CTAs per SM asked of ptxas for the classes with short strips (build-time knob for A/B runs)
#endif
	static constexpr int kMinBlocks =
	    G == 4 ? 3 : (kEst <= 128 ? DFB_OCC_SMALL : (kEst <= 168 ? 3 : (kEst <= 255 ? 2 : 1)));
};

template <int G, int S, int MODE>
__global__ void __launch_bounds__(128, FastOcc<G, S, MODE>::kMinBlocks) dp_fast_kernel(const __grid_constant__ FastParams p)
{
	constexpr int NG = 32 / G;      // job pairs per warp
	constexpr int CK = ckpt_steps(G); // checkpoint interval (steps): probe windows are whole CK blocks
	constexpr int CH = 2 * CK;      // reference ring: block of CH columns, two blocks resident
	constexpr int RING = 2 * CH;
	// G words in front of every ring: the mirror of its last G-1 columns (ring_decode_block) -- and what puts the rings of a
	// warp's groups, which read the same index in the same step, into different banks
	constexpr int RING_STRIDE = RING + G;
	constexpr int ROWS = G * S;
	constexpr int RDW = (ROWS + 15) / 16;
	constexpr int WB = CH / 16;     // pool words of one half in a ring block
	static_assert(G >= 4 && (G & (G - 1)) == 0 && G <= 32, "group size");
	static_assert(S >= 1 && S <= 32, "strip height");
	static_assert(WB <= G && G - 1 <= CK, "one lane per cp.async chunk; a lane joins inside the first checkpoint block");

	__shared__ uint32_t s_ring[4][NG][RING_STRIDE];
	__shared__ uint32_t s_rows[4][NG][RDW * 16 + 1]; // (whole 16-base words: the read staging stores without a row test)
	__shared__ __align__(16) uint2 s_raw[4][NG][2][2][WB]; // [slot][half][word]: raw pool words of the ring blocks in flight (cp.async)
	// SPLIT, four-lane groups: the granule masks of the lane's rows (read and written only at the fold and in the epilogue)
	// live here rather than in 25 registers, which buys the third CTA per SM
	constexpr bool INFO_SMEM = MODE == MODE_SPLIT && G == 4;
	__shared__ uint32_t s_info[4][INFO_SMEM ? S : 1][32];

	const int lane = threadIdx.x & 31;
	const int warp = threadIdx.x >> 5;
	const int q = lane / G;
	const int g = lane % G;
	uint32_t* ring = s_ring[warp][q] + G;
	uint32_t* rows = s_rows[warp][q];
	uint16_t* rows16 = reinterpret_cast<uint16_t*>(rows);

	const uint32_t B = p.bias;
	const uint32_t Bp = B | (B << 16);
	const uint32_t gm16 = p.gm2 & 0xFFFFu;

	const int n_items = p.n_jobs;

	for (;;)
	{
		int base = 0;
		if (lane == 0) base = atomicAdd(p.cursor, NG);
		base = __shfl_sync(0xffffffffu, base, 0);
		if (base >= n_items) break;
		const bool have = base + q < n_items;
		const int jid = base + q;
		JobPair jp;
		jp.ref_w[0] = jp.ref_w[1] = jp.read_w[0] = jp.read_w[1] = 0;
		jp.R[0] = jp.R[1] = jp.L[0] = jp.L[1] = 0;
		jp.out0 = jp.out1 = -1;
		if (have) jp = p.jobs[jid];

		// ---- stage the reads: pool words -> 16-bit symbols -> S registers per lane ----
		__syncwarp();
		{
			for (int w = g; w < 2 * RDW; w += G)
			{
				const int h = w / RDW;
				const int wi = w % RDW;
				const uint32_t len = jp.L[h];
				uint2 pw = make_uint2(0, 0);
				const uint32_t widx = jp.read_w[h] + wi;
				DFB_BC((uint32_t)wi * 16u >= len || widx < p.pool_words, 205);
				if ((uint32_t)wi * 16u < len) pw = __ldg(p.pool + widx);
				// No per-base branches: every code is decoded -- a PRMT picks the NEGATED 16-bit symbol of the 2-bit code out
				// of an 8-byte table; (-read + ref) mod 2^16 is 0 exactly on a match, so one VIADDMNMX.U16x2 (add, min with 1)
				// yields the mismatch indicator in the sweep --, rows beyond the read are overwritten with the padding value,
				// the exception plane patches its bytes afterwards (rare).
				const int nv = min(16, max(0, (int)len - wi * 16)); // bases of this word inside the read
				uint16_t* dst = rows16 + 2 * (wi * 16) + h;
#pragma unroll
				for (int n = 0; n < 16; n++)
				{
					const uint32_t code = (pw.x >> (2 * n)) & 3u;
					// bytes 2c, 2c+1 of {0xFFBF (-'A'), 0xFFBD (-'C'), 0xFFB9 (-'G'), 0xFFAC (-'T')}
					dst[2 * n] = (uint16_t)prmt(0xFFBDFFBFu, 0xFFACFFB9u, code * 0x22u + 0x10u);
				}
				for (int n = nv; n < 16; n++) dst[2 * n] = (uint16_t)(0u - DFB_READ_PAD); // (only a read's last word has any)
				uint32_t ex = pw.y & (nv >= 16 ? 0xFFFFu : ((1u << nv) - 1u));
				while (ex)
				{
					const int n = __ffs(ex) - 1;
					ex &= ex - 1;
					dst[2 * n] = (uint16_t)(0u - (uint32_t)__ldg(p.obytes + (size_t)widx * 16 + n));
				}
			}
			__syncwarp();
		}
		uint32_t rd[S], F[S], X[S];
		const int j0 = g * S; // rows owned: j0+1 .. j0+S
#pragma unroll
		for (int k = 0; k < S; k++)
		{
			rd[k] = rows[j0 + k];
			// column i = 0: H(0,j) = j*gap  ->  stored value B + j*(gap - match)
			const uint32_t v = (B + (uint32_t)(j0 + k + 1) * gm16) & 0xFFFFu;
			F[k] = v | (v << 16);
			X[k] = 0;
		}
		const uint32_t v0 = (B + (uint32_t)j0 * gm16) & 0xFFFFu;
		uint32_t prev = v0 | (v0 << 16); // stored value of (i-1, j0); lane 0: row 0 is H = 0 -> B
		__syncwarp();

		// ---- the whole wavefront: steps u = 0 .. R+G-2, lane g at column u-g ----
		const int Rg = max((int)jp.R[0], (int)jp.R[1]);
		uint32_t Flast = F[S - 1];
		// steps this warp runs: the longest of its groups (every lane takes part in the shuffles)
		int T = Rg + G - 1;
#pragma unroll
		for (int o = 16; o >= 1; o >>= 1) T = max(T, __shfl_xor_sync(0xffffffffu, T, o));
		const bool ck_on = p.ckpt != nullptr;

		// ---- reference ring: two blocks of CH columns resident as 32-bit {half 1, half 0} symbol pairs; the pool words
		//      of the next block are copied into shared memory by cp.async while the wavefront crosses the current one ----
		const uint32_t R0 = jp.R[0], R1 = jp.R[1];
		uint2(*raw)[2][WB] = s_raw[warp][q];
		// lanes 0 .. WB-1 copy one 16-byte chunk (two pool words) each: WB/2 chunks per half
		auto issue_block = [&](int blk) {
			if (g < WB)
			{
				const int h = g / (WB / 2), c = g % (WB / 2);
				const uint32_t wi = (uint32_t)blk * WB + 2u * c;
				if (wi * 16u < (h ? R1 : R0))
				{
					DFB_BC((unsigned long long)jp.ref_w[h] + wi + 2 <= p.pool_words && ((jp.ref_w[h] + wi) & 1u) == 0, 203);
					cp_async_16(&raw[blk & 1][h][2 * c], p.pool + jp.ref_w[h] + wi);
				}
			}
			cp_async_commit();
		};
		auto decode_block = [&](int blk) {
			ring_decode_block<G, true>(ring, &raw[blk & 1][0][0], blk, 0, 0, R0, R1, jp.ref_w[0], jp.ref_w[1], p.obytes, g, p.pool_words);
		};
		const int ring_blocks = min(2, (T + CH - 1) / CH); // ring columns this warp will read: T steps
		issue_block(0);
		if (ring_blocks > 1) issue_block(1);
		cp_async_wait_all();
		__syncwarp();
		decode_block(0);
		if (ring_blocks > 1) decode_block(1);
		__syncwarp();
		int blk_next = 2;
		issue_block(2);

		uint32_t acc = 0x80008000u;
		uint32_t Y[(MODE == MODE_SPLIT) ? S : 1];    // SPLIT: row maxima inside the current checkpoint block
		uint32_t info_r[(MODE == MODE_SPLIT && !INFO_SMEM) ? S : 1]; // SPLIT: granules in which the row attains its maximum X, a 16-bit mask per half
		auto info = [&](int k) -> uint32_t& {
			if constexpr (INFO_SMEM) return s_info[warp][k][lane];
			else return info_r[k];
		};
		if (MODE == MODE_SPLIT)
		{
#pragma unroll
			for (int k = 0; k < S; k++) { Y[k] = 0; info(k) = 0; }
		}
		// the sweep, one checkpoint block (CK steps) at a time so that the per-block work (checkpoint,
		// ring refill, row-maximum bookkeeping) stays out of the per-step instruction stream
		// SPLIT: steps below the shorter reference of every job pair of the warp touch real columns only (lane g is at
		// column u-g <= u).  SIMPLE tolerates the padding columns: all steps.
		int u_paired = T;
		if (MODE == MODE_SPLIT)
		{
			u_paired = have ? min((int)jp.R[0], (int)jp.R[1]) : 0x7fffffff;
#pragma unroll
			for (int o = 16; o >= 1; o >>= 1) u_paired = min(u_paired, __shfl_xor_sync(0xffffffffu, u_paired, o));
		}
		// one step of one lane: the next reference column against the S rows of the strip, with an activity test (lane g
		// joins at step g and leaves after its last column) and the new column folded into the row state at once:
		// head and tail steps
		// (the boundary value of lane 0 comes in by a multiply-add on the FMA pipe, not by a select on the ALU pipe the
		// sweep is bound by)
		uint32_t lane_nz = g != 0 ? 1u : 0u, lane_add = g != 0 ? 0u : Bp;
		asm volatile("" : "+r"(lane_nz), "+r"(lane_add)); // (opaque, or the compiler turns the multiply-add back into a select)
		auto step = [&](const int u) {
			const uint32_t recv = __shfl_up_sync(0xffffffffu, Flast, 1, G) * lane_nz + lane_add;
			const int b = u - g; // column
			if ((unsigned)b < (unsigned)Rg)
			{
				const uint32_t rf = ring[b & (RING - 1)];
				uint32_t left = recv;
				uint32_t dg_in = prev;
				uint32_t pen = 0;
				if (MODE == MODE_SPLIT) pen = rf & 0x80008000u; // -32768 in a half that is past its reference end
#pragma unroll
				for (int k = 0; k < S; k++)
				{
					const uint32_t d = __viaddmin_u16x2(rd[k], rf, 0x00010001u); // min(ref - read, 1): 1 per half on mismatch
					const uint32_t dg = d * p.xm + dg_in;                         // diagonal: + (match ? 0 : x - m)
					const uint32_t fold = F[k];                                   // this row in the previous column
					dg_in = fold;
					const uint32_t e = __viaddmax_s16x2(fold, p.g2, dg);          // max(up + gap, diagonal)
					left = __viaddmax_s16x2(left, p.gm2, e);                      // max(left + gap - m, e)
					F[k] = left;
					if (MODE == MODE_SPLIT) Y[k] = __viaddmax_s16x2(left, pen, Y[k]);
					if (MODE == MODE_SIMPLE) acc = __viaddmax_s16x2(left, p.ck[k], acc);
				}
				prev = recv;
				Flast = left;
			}
		};
		// two steps of a lane whose columns are known to be in range (every lane has joined, none has left): no
		// activity test, and one three-input maximum folds both columns into the row state (half the sink issues)
		// (rp: this lane's two ring columns -- a pointer that walks the mirrored ring, no index arithmetic per step)
		auto step_pair = [&](const uint32_t* rp) {
			uint32_t Fe[S];
			{
				const uint32_t recv = __shfl_up_sync(0xffffffffu, Flast, 1, G) * lane_nz + lane_add;
				const uint32_t rf = rp[0];
				uint32_t left = recv;
				uint32_t dg_in = prev;
#pragma unroll
				for (int k = 0; k < S; k++)
				{
					const uint32_t d = __viaddmin_u16x2(rd[k], rf, 0x00010001u);
					const uint32_t dg = d * p.xm + dg_in;
					dg_in = F[k];
					const uint32_t e = __viaddmax_s16x2(F[k], p.g2, dg);
					left = __viaddmax_s16x2(left, p.gm2, e);
					Fe[k] = left;
				}
				prev = recv;
				Flast = left;
			}
			{
				const uint32_t recv = __shfl_up_sync(0xffffffffu, Flast, 1, G) * lane_nz + lane_add;
				const uint32_t rf = rp[1];
				uint32_t left = recv;
				uint32_t dg_in = prev;
#pragma unroll
				for (int k = 0; k < S; k++)
				{
					const uint32_t d = __viaddmin_u16x2(rd[k], rf, 0x00010001u);
					const uint32_t dg = d * p.xm + dg_in;
					dg_in = Fe[k];
					const uint32_t e = __viaddmax_s16x2(Fe[k], p.g2, dg);
					left = __viaddmax_s16x2(left, p.gm2, e);
					F[k] = left;
					if (MODE == MODE_SPLIT) Y[k] = __vimax3_s16x2(Y[k], Fe[k], left);
					if (MODE == MODE_SIMPLE) X[k] = __vimax3_s16x2(X[k], Fe[k], left);
				}
				prev = recv;
				Flast = left;
			}
		};
		int u = 0;
		for (int blkno = 0; u < T; blkno++)
		{
			if (MODE == MODE_SPLIT)
			{
				// checkpoint: the wavefront state in front of every CK-th step (same step for all lanes)
				if (ck_on && blkno > 0 && have)
				{
					const size_t cb = ((size_t)jid * p.ckpt_blocks + (size_t)(blkno - 1)) * (S + 2);
					DFB_BC(blkno - 1 < p.ckpt_blocks && (cb + S + 2) * G <= p.ckpt_words, 206);
#pragma unroll
					for (int k = 0; k < S; k++) p.ckpt[(cb + k) * G + g] = F[k];
					p.ckpt[(cb + S) * G + g] = prev;
					p.ckpt[(cb + S + 1) * G + g] = Flast;
				}
			}
			// ring block n+1 replaces ring block n-1 half way through ring block n (n >= 1): every lane is past block
			// n-1 by then (G-1 <= CK steps in) and none has reached n+1
			if (blkno >= 3 && (blkno & 1))
			{
				cp_async_wait_all();
				__syncwarp();
				decode_block(blk_next);
				blk_next++;
				__syncwarp();
				issue_block(blk_next);
			}
			const int u_end = min(T, (blkno + 1) * CK);
			// head: lanes are still joining (lane g at step g); then pairs of steps while every lane is inside the
			// references; the steps with an activity test take the rest
			const int u_head = min(u_end, G - 1);
#pragma unroll 1
			for (; u < u_head; u++) step(u);
			const int u_pair_end = min(u_end, u_paired);
			if (u + 1 < u_pair_end)
			{
				// (a checkpoint block never straddles the ring's end: RING = 4 CK)
				const uint32_t* rp = ring - g + (u & (RING - 1));
				const int n_pairs = (u_pair_end - u) >> 1;
				const uint32_t* const rp_end = rp + 2 * n_pairs;
#pragma unroll 1
				for (; rp != rp_end; rp += 2) step_pair(rp);
				u += 2 * n_pairs;
			}
#pragma unroll 1
			for (; u < u_end; u++) step(u);
			if (MODE == MODE_SPLIT)
			{
				// end of a checkpoint block (or of the sweep), same step for all lanes: fold the block maxima into the
				// row maxima and remember in which granules each row maximum occurs: a block that ties the row maximum
				// joins the row's granule set, one that beats it replaces the set.  No predicates (thirteen rows x four of
				// them made ptxas spill predicates into a register, 17 ALU-pipe instructions per row): with
				// xn = max(X, Y) both xn - X and xn - Y are non-negative in either half, so one 32-bit IADD3 per difference
				// (+ 0x7FFF per half) leaves bit 15 of a half set exactly when the difference is positive, and a PRMT that
				// replicates sign bits spreads it over the half -- 7 ALU-pipe instructions per row.
				const uint32_t bit2 = (1u << (blkno >> p.gran_shift)) * 0x00010001u;
#pragma unroll
				for (int k = 0; k < S; k++)
				{
					const uint32_t xn = __vmaxs2(X[k], Y[k]);
					const uint32_t beat = spread_bit15(xn - X[k] + 0x7FFF7FFFu);  // 0xFFFF per half whose block maximum > row maximum
					const uint32_t below = spread_bit15(xn - Y[k] + 0x7FFF7FFFu); // 0xFFFF per half whose block maximum < row maximum
					info(k) = (info(k) & ~beat) | (bit2 & ~below);
					X[k] = xn;
					Y[k] = 0;
				}
			}
		}
		// the copies of a block past the end of the sweep may still be in flight: the raw slots are reused by the next job
		cp_async_wait_all();

		// ---- epilogues ----
		if (MODE == MODE_SIMPLE)
		{
			// row maxima gathered by the paired steps, plus the last column of every lane (a lane whose last
			// step was the even one of a pair has not folded it yet)
#pragma unroll
			for (int k = 0; k < S; k++) acc = __viaddmax_s16x2(__vmaxs2(X[k], F[k]), p.ck[k], acc);
			int lo = (int)(short)(acc & 0xFFFFu);
			int hi = (int)(short)(acc >> 16);
			lo = lo - (int)B + p.m * j0;
			hi = hi - (int)B + p.m * j0;
#pragma unroll
			for (int o = G / 2; o >= 1; o >>= 1)
			{
				lo = max(lo, __shfl_xor_sync(0xffffffffu, lo, o, G));
				hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o, G));
			}
			if (g == 0 && have)
			{
				DFB_BC(jp.out0 < p.n_tasks && jp.out1 < p.n_tasks, 209);
				if (jp.out0 >= 0) p.out[jp.out0] = max(lo, 0);
				if (jp.out1 >= 0) p.out[jp.out1] = max(hi, 0);
			}
		}
		if (MODE == MODE_SPLIT)
		{
			const int L = jp.L[0];
			__syncwarp();
			// FindMaxRowEntry (SplitReadAligner.cpp:91-102): keep a row max only if >= minSplitScore and > 0
#pragma unroll
			for (int k = 0; k < S; k++)
			{
				const int j = j0 + k + 1;
				int v1 = (int)(X[k] & 0xFFFFu) - (int)B + p.m * j;
				int v2 = (int)(X[k] >> 16) - (int)B + p.m * j;
				if (!(v1 >= p.min_split && v1 > 0)) v1 = 0;
				if (!(v2 >= p.min_split && v2 > 0)) v2 = 0;
				rows[j] = (uint32_t)v1 | ((uint32_t)v2 << 16);
			}
			if (g == 0) rows[0] = 0;
			__syncwarp();
			// best split total over a = 0..L (SplitReadAligner.cpp:194-222)
			int best = 0;
#pragma unroll
			for (int k = 0; k < S; k++)
			{
				const int j = j0 + k + 1;
				if (j <= L) best = max(best, (int)(rows[j] & 0xFFFFu) + (int)(rows[L - j] >> 16));
			}
			if (g == 0) best = max(best, (int)(rows[L] >> 16)); // a = 0
#pragma unroll
			for (int o = G / 2; o >= 1; o >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, o, G));
			const int min_score = jp.out1;
			const bool hit = have && best >= min_score && best > 0;
			// rows that tie for the best AND have a non-empty column set on both sides need the
			// second sweep (SplitReadAligner.cpp:233-269); the others emit nothing.
			bool en_any = false;
			uint32_t ntg[S];
			uint32_t gr0 = 0, gr1 = 0; // granules the second sweep has to visit, per half
#pragma unroll
			for (int k = 0; k < S; k++)
			{
				const int j = j0 + k + 1;
				uint32_t tlo = 0x8001u, thi = 0x8001u;
				if (hit && j <= L)
				{
					const int a1 = (int)(rows[j] & 0xFFFFu), a2 = (int)(rows[L - j] >> 16);     // this row as matrix-1 row a=j
					const int b1 = (int)(rows[L - j] & 0xFFFFu), b2 = (int)(rows[j] >> 16);     // this row as matrix-2 row, a=L-j
					if (a1 > 0 && a2 > 0 && a1 + a2 == best)
					{
						tlo = (0u - (X[k] & 0xFFFFu)) & 0xFFFFu;
						en_any = true;
						gr0 |= info(k) & 0xFFFFu;
					}
					if (b1 > 0 && b2 > 0 && b1 + b2 == best)
					{
						thi = (0u - (X[k] >> 16)) & 0xFFFFu;
						en_any = true;
						gr1 |= info(k) >> 16;
					}
				}
				ntg[k] = tlo | (thi << 16);
			}
#pragma unroll
			for (int o = G / 2; o >= 1; o >>= 1)
			{
				gr0 |= __shfl_xor_sync(0xffffffffu, gr0, o, G);
				gr1 |= __shfl_xor_sync(0xffffffffu, gr1, o, G);
			}
			const uint32_t ballot = __ballot_sync(0xffffffffu, en_any);
			const uint32_t gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << (q * G));
			const bool group_en = (ballot & gmask) != 0;
			int slot = -1;
			if (g == 0 && have)
			{
				DFB_BC(jp.out0 >= 0 && jp.out0 < p.n_tasks, 207);
				p.out[jp.out0] = hit ? best : 0;
				if (group_en)
				{
					// one granule per half is the common case; jobs with more rounds go to the other end of the queue so
					// that the job pairs of a probe warp run equally many rounds
					const bool one_round = ck_on && __popc(gr0) <= 1 && __popc(gr1) <= 1;
					slot = (one_round ? atomicAdd(p.hit_count, 1) : p.n_jobs - 1 - atomicAdd(p.hit_count_long, 1)) + p.slot_base;
					DFB_BC(slot - p.slot_base >= 0 && slot - p.slot_base < p.n_jobs, 208);
					p.hitq[slot - p.slot_base] = jid;
					p.slot_task[slot - p.slot_base] = jp.out0;
					p.task_slot[jp.out0] = slot;
					p.slot_rng[slot - p.slot_base] = gr0 | (gr1 << 16);
					slot -= p.slot_base;
				}
			}
			slot = __shfl_sync(0xffffffffu, slot, q * G);
			if (group_en && have)
			{
#pragma unroll
				for (int k = 0; k < S; k++)
				{
					p.ntg[((size_t)slot * S + k) * G + g] = ntg[k];
					p.rdq[((size_t)slot * S + k) * G + g] = rd[k];
				}
			}
		}
	}
}

// ------------------------------------------------------------------------------------------
// Probe sweep: the arg-max column sets of the winning split rows (second half of GetAlignments,
// SplitReadAligner.cpp:229-269).  The first sweep left, per winning task, the negated row maxima of
// its winning rows (ntg), the lanes' read symbols (rdq) and, per half, a 16-bit mask of the
// checkpoint granules in which those rows attain their maxima.  A job is swept in rounds: round r
// visits the r-th marked granule of either half -- the two halves of the registers resume from two
// different checkpoints -- and records every column at which an enabled row reaches its target.
// ------------------------------------------------------------------------------------------
// (four-lane groups: 25-row strips spill 104 bytes at 128 registers, 36 at 168 -- outside the step loop: three CTAs)
template <int G, int S>
struct ProbeOcc
{
	static constexpr int kEst = 3 * S + 44;
#ifndef DFB_PROBE_OCC6_EST
#define DFB_PROBE_OCC6_EST 60 // strips up to this register estimate ask ptxas for six CTAs per SM (build-time knob for A/B runs)
#endif
	static constexpr int kMinBlocks =
	    G == 4 ? 3 : (kEst <= DFB_PROBE_OCC6_EST ? 6 : (kEst <= 100 ? 5 : (kEst <= 128 ? 4 : (kEst <= 168 ? 3 : 2))));
};

template <int G, int S>
__global__ void __launch_bounds__(128, ProbeOcc<G, S>::kMinBlocks) dp_probe_kernel(const __grid_constant__ FastParams p)
{
	constexpr int NG = 32 / G;
	constexpr int CK = ckpt_steps(G);
	constexpr int CH = 2 * CK;
	constexpr int RING = 2 * CH;
	// G words in front of every ring: the mirror of its last G-1 columns (ring_decode_block) -- and what puts the rings of a
	// warp's groups, which read the same index in the same step, into different banks
	constexpr int RING_STRIDE = RING + G;
	constexpr int WB = CH / 16; // pool words of one half in a ring block
	constexpr int PRE = 32; // ring columns in front of a round's first step (>= G-1, two whole pool words)
	static_assert(G >= 4 && (G & (G - 1)) == 0 && G <= 32 && WB <= G, "group size");
	static_assert(G - 1 <= PRE && PRE + CK <= CH, "a one-block round fits one ring block");

	__shared__ uint32_t s_ring[4][NG][RING_STRIDE];
	__shared__ __align__(16) uint2 s_raw[4][NG][2][2][WB];

	const int lane = threadIdx.x & 31;
	const int warp = threadIdx.x >> 5;
	const int q = lane / G;
	const int g = lane % G;
	uint32_t* ring = s_ring[warp][q] + G;
	uint2(*raw)[2][WB] = s_raw[warp][q];

	const uint32_t B = p.bias;
	const uint32_t Bp = B | (B << 16);
	const uint32_t gm16 = p.gm2 & 0xFFFFu;
	const int gs = p.gran_shift;
	const int n_short = *p.hit_count;
	const int n_items = n_short + *p.hit_count_long;
	const int j0 = g * S; // rows owned: j0+1 .. j0+S

	auto claim = [&]() -> int {
		int b = 0;
		if (lane == 0) b = atomicAdd(p.cursor, NG);
		return __shfl_sync(0xffffffffu, b, 0);
	};
	// queue position -> slot (one-round jobs were queued from the front, the others from the back)
	auto slot_of = [&](int idx) -> int { return (idx >= n_short) ? p.n_jobs - 1 - (idx - n_short) : idx; };
	for (;;)
	{
		const int base = claim();
		if (base >= n_items) break;
		const bool have = base + q < n_items;
		const int item = slot_of(base + q);
		int jid = 0;
		uint32_t rng = 0;
		if (have)
		{
			jid = p.hitq[item];
			rng = p.slot_rng[item];
		}
		JobPair jp;
		jp.ref_w[0] = jp.ref_w[1] = jp.read_w[0] = jp.read_w[1] = 0;
		jp.R[0] = jp.R[1] = jp.L[0] = jp.L[1] = 0;
		jp.out0 = jp.out1 = -1;
		uint32_t m0 = 0, m1 = 0;
		if (have)
		{
			DFB_BC(item >= 0 && item < p.n_jobs, 301);
			DFB_BC(jid >= 0 && jid < p.n_jobs, 302);
			jp = p.jobs[jid];
			m0 = rng & 0xFFFFu;
			m1 = rng >> 16;
		}
		uint32_t rd[S], X[S]; // read symbols; negated targets of the rows being enumerated (0x8001: row not enumerated)
#pragma unroll
		for (int k = 0; k < S; k++)
		{
			rd[k] = have ? p.rdq[((size_t)item * S + k) * G + g] : 0u;
			X[k] = have ? p.ntg[((size_t)item * S + k) * G + g] : 0x80018001u;
		}
		// without checkpoints (the class' references are too long to keep them): one round over the whole wavefront
		const bool whole = p.ckpt == nullptr;
		int Tr = CK << gs; // steps per round
		if (whole)
		{
			m0 = m1 = have ? 1u : 0u;
			Tr = max((int)jp.R[0], (int)jp.R[1]) + G - 1;
		}
		int rounds = max(__popc(m0), __popc(m1));
#pragma unroll
		for (int o = 16; o >= 1; o >>= 1)
		{
			rounds = max(rounds, __shfl_xor_sync(0xffffffffu, rounds, o));
			Tr = max(Tr, __shfl_xor_sync(0xffffffffu, Tr, o));
		}

		for (int r = 0; r < rounds; r++)
		{
			// the granule either half visits in this round; a half that has none left idles on padding
			const bool on0 = r < __popc(m0), on1 = r < __popc(m1);
			uint32_t mr0 = m0, mr1 = m1; // masks without their r lowest set bits
			for (int i = 0; i < r; i++) { mr0 &= mr0 - 1; mr1 &= mr1 - 1; }
			const int b0 = on0 ? ((__ffs(mr0) - 1) << gs) : 0; // first checkpoint block of the granule
			const int b1 = on1 ? ((__ffs(mr1) - 1) << gs) : 0;
			const uint32_t R0 = on0 ? jp.R[0] : 0u, R1 = on1 ? jp.R[1] : 0u;
			// ring index = relative column + PRE; relative column 0 = absolute column b * CK of the half
			const int c0 = b0 * CK - PRE, c1 = b1 * CK - PRE; // absolute column of ring column 0 (negative in block 0)
			auto issue_block = [&](int blk) {
				if (g < WB)
				{
					const int h = g / (WB / 2), c = g % (WB / 2);
					const int wi = ((h ? c1 : c0) >> 4) + blk * WB + 2 * c; // (c0, c1 are multiples of 32: arithmetic shift is exact)
					if (wi >= 0 && (uint32_t)wi * 16u < (h ? R1 : R0))
					{
						DFB_BC((unsigned long long)jp.ref_w[h] + (unsigned)wi + 2 <= p.pool_words && ((jp.ref_w[h] + (unsigned)wi) & 1u) == 0, 204);
						cp_async_16(&raw[blk & 1][h][2 * c], p.pool + jp.ref_w[h] + wi);
					}
				}
				cp_async_commit();
			};
			auto decode_block = [&](int blk) {
				ring_decode_block<G, false>(ring, &raw[blk & 1][0][0], blk, c0 >> 4, c1 >> 4, R0, R1, jp.ref_w[0], jp.ref_w[1], p.obytes, g, p.pool_words); // (the probe masks its ring index: no mirror)
			};
			__syncwarp(); // (the previous round's ring reads are over)
			const int ring_blocks = min(2, (Tr + PRE + CH - 1) / CH);
			issue_block(0);
			if (ring_blocks > 1) issue_block(1);

			// wavefront state in front of the round's first step: the checkpoint of the block before it, or the
			// boundary column H(0,j) = j*gap (stored B + j*(gap - match)) in block 0 -- per half
			uint32_t F[S], prev, Flast;
			// (an idle half starts from the boundary column too: every field must stay a valid stored value, the 32-bit
			// diagonal IMAD borrows from the other half otherwise)
			const uint32_t keep0 = (on0 && b0 > 0) ? 0x0000FFFFu : 0u, keep1 = (on1 && b1 > 0) ? 0xFFFF0000u : 0u;
			const uint32_t init0 = keep0 ^ 0x0000FFFFu, init1 = keep1 ^ 0xFFFF0000u;
			// halves whose lanes join one by one (lane g at step g)
			const uint32_t jm = whole ? 0u : (((on0 && b0 == 0) ? 0x0000FFFFu : 0u) | ((on1 && b1 == 0) ? 0xFFFF0000u : 0u));
			const size_t cb0 = ((size_t)jid * p.ckpt_blocks + (size_t)max(b0 - 1, 0)) * (S + 2);
			const size_t cb1 = ((size_t)jid * p.ckpt_blocks + (size_t)max(b1 - 1, 0)) * (S + 2);
			auto boundary = [&](int j) -> uint32_t { // stored value of column 0, row j, in both halves
				const uint32_t v = (B + (uint32_t)j * gm16) & 0xFFFFu;
				return v | (v << 16);
			};
			DFB_BC(!keep0 || (b0 - 1 < p.ckpt_blocks && (cb0 + S + 2) * G <= p.ckpt_words), 303);
			DFB_BC(!keep1 || (b1 - 1 < p.ckpt_blocks && (cb1 + S + 2) * G <= p.ckpt_words), 304);
#pragma unroll
			for (int k = 0; k < S + 2; k++)
			{
				uint32_t v = 0;
				if (keep0) v |= p.ckpt[(cb0 + k) * G + g] & keep0;
				if (keep1) v |= p.ckpt[(cb1 + k) * G + g] & keep1;
				// k < S: row j0+k+1; k = S: the diagonal input (row j0); k = S+1: the hand-off value (row j0+S)
				v |= boundary(k < S ? j0 + k + 1 : (k == S ? j0 : j0 + S)) & (init0 | init1);
				if (k < S) F[k] = v;
				else if (k == S) prev = v;
				else Flast = v;
			}
			cp_async_wait_all();
			__syncwarp();
			decode_block(0);
			if (ring_blocks > 1) decode_block(1);
			__syncwarp();
			int blk_next = 2;
			if (Tr + PRE > 2 * CH) issue_block(2);

			// whole-wavefront rounds: lane g joins at step g and leaves after its last column (activity test);
			// checkpointed rounds: every lane runs every step, a half that starts in block 0 is put back to the
			// boundary column after each step its lane has not joined yet
			const int act_off = whole ? g : 0;
			const int Rg = whole ? max((int)jp.R[0], (int)jp.R[1]) : Tr;
			auto step = [&](const int u) {
				uint32_t recv = __shfl_up_sync(0xffffffffu, Flast, 1, G);
				if (g == 0) recv = Bp;
				const int b = u - g;
				if ((unsigned)(u - act_off) < (unsigned)Rg)
				{
					const uint32_t rf = ring[(b + PRE) & (RING - 1)];
					uint32_t left = recv;
					uint32_t dg_in = prev;
					uint32_t acc = 0x80008000u;
#pragma unroll
					for (int k = 0; k < S; k++)
					{
						const uint32_t d = __viaddmin_u16x2(rd[k], rf, 0x00010001u);
						const uint32_t dg = d * p.xm + dg_in;
						dg_in = F[k];
						const uint32_t e = __viaddmax_s16x2(F[k], p.g2, dg);
						left = __viaddmax_s16x2(left, p.gm2, e);
						F[k] = left;
						acc = __viaddmax_s16x2(left, X[k], acc);
					}
					prev = recv;
					Flast = left;
					// a half of acc is >= 0 only when some enumerated row reached its target here (a row that is not
					// enumerated has the target 0x8001, which no stored value cancels)
					if ((~acc) & 0x80008000u)
					{
						uint32_t hm0 = 0, hm1 = 0;
#pragma unroll
						for (int k = 0; k < S; k++)
						{
							if (((F[k] + X[k]) & 0xFFFFu) == 0) hm0 |= 1u << k;
							if ((((F[k] >> 16) + (X[k] >> 16)) & 0xFFFFu) == 0) hm1 |= 1u << k;
						}
						if (!on0) hm0 = 0;
						if (!on1) hm1 = 0;
						if (hm0 | hm1)
							emit_probe_hits(p, item, jp.out0, hm0, hm1, j0, b0 * CK + b, b1 * CK + b, jp.R[0], jp.R[1], (int)jp.L[0], S, G, g);
					}
				}
			};
			int u = 0;
			for (int blkno = 0; u < Tr; blkno++)
			{
				if (blkno >= 3 && (blkno & 1))
				{
					cp_async_wait_all();
					__syncwarp();
					decode_block(blk_next);
					blk_next++;
					__syncwarp();
					issue_block(blk_next);
				}
				const int u_end = min(Tr, (blkno + 1) * CK);
#pragma unroll 1
				for (; u < u_end; u++)
				{
					step(u);
					if (jm && u < g)
					{
						// this lane has not joined the half that starts in block 0 yet: back to the boundary column
#pragma unroll
						for (int k = 0; k < S; k++) F[k] = (F[k] & ~jm) | (boundary(j0 + k + 1) & jm);
						prev = (prev & ~jm) | (boundary(j0) & jm);
						Flast = (Flast & ~jm) | (boundary(j0 + S) & jm);
					}
				}
			}
			cp_async_wait_all();
		}
	}
}

// ------------------------------------------------------------------------------------------
// s32 generic kernels: any scoring triple (positive gaps, endGaps, minSplitScore <= 0 ...),
// any read / reference length.  One warp per DP, 8 rows per lane, the read tiled 256 rows at
// a time with the tile boundary row kept in a per-warp HBM scratch line.  Same wavefront as
// above, plain 32-bit max/add, H stored directly.  Rarely selected (see host dispatch);
// exactness over speed.
// ------------------------------------------------------------------------------------------

struct GenJob
{
	uint32_t ref_w;  // first pool word of the (oriented) reference
	uint32_t read_w; // first pool word of the (oriented) read
	uint32_t R;
	uint32_t L;
	int32_t task;    // output index
	int32_t half;    // SPLIT/PROBE: 0 = matrix 1, 1 = matrix 2
	int64_t row_off; // SPLIT/PROBE: first entry of this DP's row arrays (L + 1 entries)
};

struct GenParams
{
	const uint2* pool;
	const uint8_t* obytes;
	const GenJob* jobs;
	int n_jobs;
	int* cursor;
	int m, x, g, end_gaps;
	int32_t* out;          // SIMPLE: score per task
	int32_t* rowmax;       // SPLIT: raw row maxima over i = 0..R     PROBE: target per row
	const uint8_t* row_en; // PROBE: 1 = enumerate the columns of this row
	const int* probe_flag; // PROBE: per task (jobs 2t, 2t+1): 0 = nothing to enumerate, skip
	int32_t* bnd;          // per-warp scratch: 2 * bnd_stride ints
	int64_t bnd_stride;
	Event* events;
	unsigned long long* ev_count;
	unsigned long long ev_cap;
};

#define DFB_GEN_S 8
#define DFB_GEN_TILE (32 * DFB_GEN_S)

__device__ __forceinline__ void emit_event(const GenParams& p, int task, int half, int row, int col, int score)
{
	const unsigned long long idx = atomicAdd(p.ev_count, 1ull);
	if (idx < p.ev_cap)
	{
		Event ev;
		ev.task = task;
		ev.half_row = (half << 30) | row;
		ev.col = col;
		ev.score = score;
		p.events[idx] = ev;
	}
}

template <int MODE>
__global__ void __launch_bounds__(128) dp_generic_kernel(const __grid_constant__ GenParams p)
{
	constexpr int S = DFB_GEN_S;
	const int lane = threadIdx.x & 31;
	const int gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	int32_t* bnd_a = p.bnd + (int64_t)gwarp * 2 * p.bnd_stride;
	int32_t* bnd_b = bnd_a + p.bnd_stride;
	const int col0_step = p.end_gaps ? 0 : p.g; // H(0,j) = j * col0_step  (SplitReadAligner.cpp:44-48)

	for (;;)
	{
		int jid = 0;
		if (lane == 0) jid = atomicAdd(p.cursor, 1);
		jid = __shfl_sync(0xffffffffu, jid, 0);
		if (jid >= p.n_jobs) break;
		if (MODE == MODE_PROBE && p.probe_flag[jid >> 1] == 0) continue;
		const GenJob job = p.jobs[jid];
		const int R = (int)job.R, L = (int)job.L;
		auto base_at = [&](uint32_t first_word, int pos) -> int {
			const uint32_t widx = first_word + ((uint32_t)pos >> 4);
			return (int)decode_base(__ldg(p.pool + widx), widx, pos & 15, p.obytes);
		};
		int best = INT32_MIN; // SIMPLE: max over interior cells

		if (MODE == MODE_PROBE)
		{
			// row 0 is H(i,0) = 0 for every i
			if (p.row_en[job.row_off] && p.rowmax[job.row_off] == 0)
			{
				for (int i = lane; i <= R; i += 32) emit_event(p, job.task, job.half, 0, i, 0);
			}
		}
		if (MODE == MODE_SPLIT)
		{
			if (lane == 0) p.rowmax[job.row_off] = 0;
		}

		const int n_tiles = (L + DFB_GEN_TILE - 1) / DFB_GEN_TILE;
		for (int tile = 0; tile < n_tiles; tile++)
		{
			const int jbase = tile * DFB_GEN_TILE; // rows jbase+1 .. jbase+256
			const int j0 = jbase + lane * S;
			const bool first_tile = tile == 0;
			const bool last_tile = tile == n_tiles - 1;
			const int32_t* bin = (tile & 1) ? bnd_b : bnd_a;  // row jbase of every column (written by the previous tile)
			int32_t* bout = (tile & 1) ? bnd_a : bnd_b;
			int rd[S], H[S], X[S], tg[S];
			bool en[S];
#pragma unroll
			for (int k = 0; k < S; k++)
			{
				const int j = j0 + k + 1;
				rd[k] = (j <= L) ? base_at(job.read_w, j - 1) : -1;
				H[k] = j * col0_step;
				X[k] = H[k];
				tg[k] = 0;
				en[k] = false;
				if (MODE == MODE_PROBE && j <= L)
				{
					en[k] = p.row_en[job.row_off + j] != 0;
					tg[k] = p.rowmax[job.row_off + j];
					if (en[k] && H[k] == tg[k]) emit_event(p, job.task, job.half, j, 0, tg[k]); // column i = 0
				}
			}
			int prev = j0 * col0_step; // H(0, j0); for lane 0 of tile 0 this is H(0,0) = 0
			int Hlast = H[S - 1];
			const int T = R + 31;
			__syncwarp();
			for (int tau = 0; tau < T; tau++)
			{
				int recv = __shfl_up_sync(0xffffffffu, Hlast, 1);
				const int b = tau - lane;
				if (lane == 0) recv = (first_tile || b >= R) ? 0 : __ldcg(bin + b + 1);
				if (b >= 0 && b < R)
				{
					const int rf = base_at(job.ref_w, b);
					int left = recv;
					int dg_in = prev;
#pragma unroll
					for (int k = 0; k < S; k++)
					{
						const int dg = dg_in + ((rd[k] == rf) ? p.m : p.x);
						dg_in = H[k];
						const int e = max(H[k] + p.g, dg);
						left = max(left + p.g, e);
						H[k] = left;
						const int j = j0 + k + 1;
						if (MODE == MODE_SIMPLE) { if (j <= L) best = max(best, left); }
						if (MODE == MODE_SPLIT) X[k] = max(X[k], left);
						if (MODE == MODE_PROBE) { if (en[k] && left == tg[k]) emit_event(p, job.task, job.half, j, b + 1, left); }
					}
					prev = recv;
					Hlast = left;
					if (lane == 31 && !last_tile) bout[b + 1] = left;
				}
			}
			if (MODE == MODE_SPLIT)
			{
#pragma unroll
				for (int k = 0; k < S; k++)
				{
					const int j = j0 + k + 1;
					if (j <= L) p.rowmax[job.row_off + j] = X[k];
				}
			}
			__syncwarp();
			__threadfence_block();
		}
		if (MODE == MODE_SIMPLE)
		{
#pragma unroll
			for (int o = 16; o >= 1; o >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, o));
			if (lane == 0) p.out[job.task] = max(best, 0);
		}
	}
}

// Per split task (generic path): turn the raw row maxima of both matrices into the best split
// total and the per-row probe targets.  One thread per task; rows are few thousand at most.
struct GenReduceParams
{
	const GenJob* jobs; // two consecutive jobs per task: matrix 1, matrix 2
	int n_tasks;
	const int32_t* task_min_score; // indexed by jobs[2t].task
	int min_split;
	int32_t* rowmax;  // in: raw maxima; out: FindMaxRowEntry value (0 when not accepted)
	uint8_t* row_en;  // out
	int32_t* out_best;
	int* probe_flag;  // out per task pair index: 1 = needs the probe sweep
};

__global__ void __launch_bounds__(128) split_reduce_generic_kernel(const GenReduceParams p)
{
	const int t = blockIdx.x * blockDim.x + threadIdx.x;
	if (t >= p.n_tasks) return;
	const GenJob j1 = p.jobs[2 * t], j2 = p.jobs[2 * t + 1];
	const int L = (int)j1.L;
	int32_t* r1 = p.rowmax + j1.row_off;
	int32_t* r2 = p.rowmax + j2.row_off;
	uint8_t* e1 = p.row_en + j1.row_off;
	uint8_t* e2 = p.row_en + j2.row_off;
	// FindMaxRowEntry (SplitReadAligner.cpp:91-102): values below minSplitScore or not above 0 give 0
	for (int j = 0; j <= L; j++)
	{
		int v1 = r1[j], v2 = r2[j];
		if (!(v1 >= p.min_split && v1 > 0)) v1 = 0;
		if (!(v2 >= p.min_split && v2 > 0)) v2 = 0;
		r1[j] = v1;
		r2[j] = v2;
		e1[j] = 0;
		e2[j] = 0;
	}
	const int min_score = p.task_min_score[j1.task];
	int best = 0;
	for (int a = 0; a <= L; a++)
	{
		const int tot = r1[a] + r2[L - a];
		if (tot >= min_score && tot > best) best = tot;
	}
	p.out_best[j1.task] = best;
	int need = 0;
	if (best != 0)
	{
		// a row with maximum 0 still has columns when 0 >= minSplitScore (the == branch of
		// SplitReadAligner.cpp:111-121 with max == 0)
		const bool zero_ok = p.min_split <= 0;
		for (int a = 0; a <= L; a++)
		{
			if (r1[a] + r2[L - a] == best && (r1[a] > 0 || zero_ok) && (r2[L - a] > 0 || zero_ok))
			{
				e1[a] = 1;
				e2[L - a] = 1;
				need = 1;
			}
		}
	}
	p.probe_flag[t] = need;
}

}  // namespace dfb
