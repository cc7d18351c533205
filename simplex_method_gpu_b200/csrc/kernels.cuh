// Device code of the B200 dense revised-simplex engine (sm_100a).
//
// One pivot of the reference loop (src/v4_cub_reduction.cu:286-359) is three
// phases separated by grid-wide barriers; all of them live in ONE persistent
// cooperative kernel (simplex_persistent), so there is no host round trip per
// pivot.  The same phase functions are also wrapped as stand-alone kernels for
// unit tests and for the one-launch-per-phase mode.
//
//   price          e_j = y.A_j - c_j fused with the argmin           (v4:289-296)
//                  its prologue applies the O(m) updates of the PREVIOUS pivot
//                  (x_b, y, c_b, b_ixs: v4:339-356) when y fits in shared memory
//   update_ftran   B^-1 += E_q (x) row_q  AND  alpha = B^-1_new a_p  (v4:333 + v4:307-308)
//                  -> B^-1 crosses HBM once per pivot (read + write);
//                  the CTA that completes the last tile of a row group sums the group's
//                  chunk partials and runs the ratio test on those rows (v4:311-325)
//                  while the other CTAs keep streaming
//   book1          row_q gather, E_q, the two O(m) dot products      (v4:331-332, 347, 354)
//   (book2         x_b, y, c_b, b_ixs as a phase of its own: large m, window end)
//
// Layout: everything column-major like the reference (v4:59-60).  The leading
// dimension ld is m rounded up to one warp-wide 16-byte vector row (64 doubles
// / 128 floats = 512 B) and the padding rows are zero, so every warp access is
// a full, aligned 512 B segment without predicates.
//
// Summation orders are fixed by the problem size only (never by the grid or
// the tile shape), so results are bit-identical for every launch geometry:
//   pricing dot ..... thread t of 256 owns vectors t, t+256, ...; per-slot fma
//                     chains, slots left to right, warp butterfly, 8 warp sums
//                     left to right, then "- c_j"
//   FTRAN ........... 32-column sub-blocks (one fma chain each), pairwise tree
//                     over the 8 sub-blocks of a 256-column chunk, chunks left
//                     to right
//   O(m) dots ....... 256-element slices (thread t owns element t), warp
//                     butterfly, 8 warp sums left to right, slices left to right
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <math_constants.h>

namespace b200lp {

constexpr int NT = 256;       // threads per CTA
constexpr int NWARP = NT / 32;
constexpr int CHUNK = 256;    // FTRAN partial-sum chunk (columns)
constexpr int SUBW = 32;      // FTRAN sub-block (columns)
constexpr int SLICE = 256;    // O(m) dot slice (elements)
constexpr int PRICE_NC = 4;   // most columns priced together by one CTA (Dev::price_nc = 4 or 2 per problem)
constexpr int PRICE_UNIT = NT * 16;                   // ring allocation unit: one vector (y or a column) of one row block
constexpr int DYN_SMEM_BYTES = 20 * PRICE_UNIT;       // pricing ring: 4 stages of y + 4 columns (or 6 stages of y + 2 columns);
                                                      // its first 12 KB double as the update+FTRAN staging area.
                                                      // Measured: a 5th stage (100 KB) does not speed pricing up and slows the
                                                      // update+FTRAN pass by 17 % — two CTAs would leave only ~23 KB of L1, and
                                                      // the pass keeps 64 KB of loads per SM in flight through L1
constexpr int UF_SMEM_BYTES = 2 * CHUNK * 8 + NWARP * 32 * 4 * 8; // row_q/a_p chunk + cross-warp combine
constexpr int PRICE_MAX_STAGES = 8;
// Measured on B200: a block is latency bound (about 2 us from TMA issue to landing under load), so the ring must
// keep ~48 KB of A per CTA in flight; single-column blocks cannot (half the streaming rate), two-column blocks with
// six stages can.  Narrow groups shorten the tail of the pass when a CTA gets only a few groups (sharded, m <= 8192).
constexpr int MIN_CTAS = 2;   // resident CTAs per SM the persistent kernel is compiled for
constexpr int MAXR = 8;       // ranks (GPUs) of one NVSwitch box

template <typename T> struct VecT;
template <> struct VecT<double> { using V = double2; static constexpr int N = 2; };
template <> struct VecT<float>  { using V = float4;  static constexpr int N = 4; };

// (value, index) candidate of a distributed argmin; value kept as double for
// both dtypes (float -> double is exact and order preserving)
struct Cand {
	double val;
	long long idx;
};

struct Ctl {
	unsigned long long bar;   // grid barrier arrivals (reset by the host before a launch)
	long long iter;           // iterations done ("# Iteration" lines, v4:287)
	long long pivots;
	long long it_end;         // this launch stops at iter == it_end
	int status;               // B200LP_STATUS_*
	int pending;              // rank-1 update (E_q, row_q) not yet applied to B^-1
	int done;                 // optimum / unbounded reached
	int bad;                  // a wait timed out (sharded mode)
	unsigned long long xarr[2];       // arrivals at the exchanges X1 / X2 (reset by the host before a launch)
	unsigned int price_ctr;   // dynamic work tickets of the pricing phase (column groups)
	unsigned int upd_ctr;     // dynamic work tickets of the update+FTRAN phase (tiles)
	unsigned long long xepoch; // cross-GPU barrier epoch, monotonic over the engine's life
	int abort_req;            // host: stop at the next iteration boundary (b200lp_abort); written while the kernel runs
	int abort_latched;        // CTA 0's copy of abort_req, taken before it arrives at the pricing barrier
	int aborted;              // the last launch ended because of abort_req
	int se_pending;           // steepest edge: the weight recurrence of the last pivot is still to be applied
	unsigned int btran_ctr;   // dynamic work tickets of the BTRAN pass (steepest edge)
	int pad0;
	long long leaving;        // steepest edge: variable that left the basis in the last pivot
	double alpha_q;           // steepest edge: pivot element of the last pivot
	long long p, q;           // last entering column / leaving row
	double min_e;             // last pricing minimum
	double c_b_q;             // c_b[q] before the swap (v4:339)
	double z;                 // c_b . x_b (v4:365)
};

template <typename T>
struct Dev {
	long long m, n, ns, ld;   // ns = dense (structural) columns; the n - ns others are unit vectors
	int nchunk, nslice;
	const T* A;               // ld x ns, read-only while solving
	T* B;                     // ld x m   (B^-1)
	const T* b;               // ld
	const T* c;               // n
	T *y, *x_b, *c_b, *alpha, *E_q, *row_q; // ld each
	T* alpha_part;            // nchunk x ld
	T* dpart;                 // 2 x nslice
	int* b_ixs;               // m
	Cand* cand;               // one per CTA
	long long* cnt;           // eligible rows, one per CTA
	Cand* cand2;              // steepest edge: per-CTA (-e^2/gamma, index) candidate
	T* gamma;                 // steepest edge: weights 1 + |B^-1 a_j|^2 of all n columns
	T* vbt;                   // steepest edge: v = B^-T alpha (ld)
	int pricing_rule;         // 0 Dantzig (v4:288-302), 1 steepest edge with the Goldfarb-Reid recurrence (README.md:16-17)
	Cand* rcand;              // ratio-test candidate of every row group of the update+FTRAN pass
	long long* rcnt;          // eligible rows of every row group
	unsigned int* grp_done;   // tiles finished per row group (reset by the finisher)
	int rg;                   // row tiles per row group
	int ngrp;                 // row groups of the local row block
	int fuse_ratio;           // 1: ratio test per row group inside the update+FTRAN pass; 0: a phase of its own after a barrier
	int fuse_book2;           // 1: the O(m) updates of a pivot ride in the prologue of the next pricing pass (y in shared memory)
	int price_tail;           // columns at the end of the local block priced one at a time (shorter tail of the pass)
	double pivot_tol;         // ratio-test eligibility alpha > pivot_tol (0 = the reference's strict test, v4:203)
	int res_maxG;             // resident kernel: CTAs available (one per SM)
	int ratio_mode;           // 0 textbook (v4:199-208), 1 bounded (x_b clamped at 0), 2 Harris two-pass
	double harris_delta;      // Harris: feasibility tolerance of the first pass
	Ctl* ctl;
	int2* trace;
	long long trace_cap;
	double eps;
	// ---- sharding over the GPUs of one box (single GPU: rank 0 of 1, row0 = 0, ldb = ld, col0 = 0, nsl = ns)
	// B^-1 is row-block sharded (B holds rows [row0, row0+ldb) with leading dimension ldb),
	// A is column-block sharded (A holds dense columns [col0, col0+nsl), ld rows each),
	// every O(m) vector is replicated.
	int rank, nranks;
	long long row0, ldb;
	long long col0, nsl;
	long long k0, k1;                 // share of the unit (slack) columns priced on this rank
	int price_nc;                     // pricing group width of the TMA ring: 4 (or 2, option)
	int price_direct;                 // 1: register-staged pricing without the ring (the A shard is L2 resident)
	long long colstart[MAXR + 1], rowstart[MAXR + 1];
	unsigned long long* prof;         // optional phase stamps (globaltimer ns), NSTAMP per iteration of a launch
	long long prof_cap;               // iterations the buffer holds (0 = profiling off)
	const T* A_peer[MAXR];            // every rank's A shard (peer-mapped over NVLink)
	unsigned char* mbox_peer[MAXR];   // every rank's mailbox: [XHdr][alpha ld][row_q ld][rqb nslice]; alpha/row_q above point into our own
	long long vpart_off;              // steepest edge, sharded: element offset (from alpha) of the R partial-v vectors in a mailbox
	const T* dpart0;                  // row_q.b slice partials: dpart on one GPU, the mailbox's rqb when sharded
	T* acol;                          // local copy of the entering column (sharded mode only)
};

// head of a rank's mailbox; peers store into it over NVLink.  Every record carries its own flag
// (= the serial number of the pricing round it belongs to, monotonic over the engine's life), so
// receiving a record is one acquire-load spin and needs no separate barrier.
struct XCand {
	double val;
	long long idx;
	long long cnt;
	double val2;                      // steepest edge: the weighted candidate (-e^2/gamma, index) rides beside (min e, index)
	long long idx2;
	unsigned long long flag;
};
struct XHdr {
	XCand pc[2][MAXR];                // X1: pricing candidate of rank r (double buffered by round parity)
	XCand rc[MAXR];                   // X2: ratio candidate + eligible count of rank r's rows; flag also says "alpha slice stored"
	unsigned long long rflag;         // X3: row q and its row_q.b slice partials are stored
	unsigned long long vflag[MAXR];   // X4 (steepest edge): rank r's partial of v = B^-T alpha is stored
	unsigned long long pad[7];
};
static_assert(sizeof(XHdr) % 256 == 0, "mailbox vectors must stay 16-byte aligned");

// ---------------------------------------------------------------- memory ops

template <typename T> struct Mem;
template <> struct Mem<double> {
	using V = double2;
	// read-only stream (A): non-coherent path, do not allocate in L1
	static __device__ __forceinline__ V ld_nc(const double* p) {
		V v;
		asm("ld.global.nc.L1::no_allocate.v2.f64 {%0,%1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
		return v;
	}
	// read-write stream (B^-1): coherent, do not allocate in L1
	static __device__ __forceinline__ V ld_stream(const double* p) {
		V v;
		asm volatile("ld.global.L1::no_allocate.v2.f64 {%0,%1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p) : "memory");
		return v;
	}
	static __device__ __forceinline__ void st_stream(double* p, V v) {
		asm volatile("st.global.L1::no_allocate.v2.f64 [%0], {%1,%2};" ::"l"(p), "d"(v.x), "d"(v.y) : "memory");
	}
	static __device__ __forceinline__ double get(const V& v, int k) { return k == 0 ? v.x : v.y; }
	static __device__ __forceinline__ void set(V& v, int k, double s) { if (k == 0) v.x = s; else v.y = s; }
};
template <> struct Mem<float> {
	using V = float4;
	static __device__ __forceinline__ V ld_nc(const float* p) {
		V v;
		asm("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
		return v;
	}
	static __device__ __forceinline__ V ld_stream(const float* p) {
		V v;
		asm volatile("ld.global.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
		return v;
	}
	static __device__ __forceinline__ void st_stream(float* p, V v) {
		asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
	}
	static __device__ __forceinline__ float get(const V& v, int k) { return k == 0 ? v.x : k == 1 ? v.y : k == 2 ? v.z : v.w; }
	static __device__ __forceinline__ void set(V& v, int k, float s) { if (k == 0) v.x = s; else if (k == 1) v.y = s; else if (k == 2) v.z = s; else v.w = s; }
};

__device__ __forceinline__ double fma_t(double a, double b, double c) { return fma(a, b, c); }
__device__ __forceinline__ float fma_t(float a, float b, float c) { return fmaf(a, b, c); }
// a product rounded on its own (never contracted into an fma)
__device__ __forceinline__ double mul_rn_t(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float mul_rn_t(float a, float b) { return __fmul_rn(a, b); }

template <typename T>
__device__ __forceinline__ T warp_butterfly_sum(T s) {
#pragma unroll
	for (int off = 16; off >= 1; off >>= 1) s = s + __shfl_xor_sync(0xffffffffu, s, off);
	return s;
}

// numerator of the ratio test: x_b itself (v4:205), or clamped at zero in the bounded / Harris modes
template <typename T>
__device__ __forceinline__ T ratio_num(T xb, int mode) { return mode >= 1 && xb < T(0) ? T(0) : xb; }

// lexicographic (value, index): the lowest index wins ties, like cub ArgMin (v4:294, 324)
__device__ __forceinline__ bool cand_better(double v, long long i, double bv, long long bi) {
	return v < bv || (v == bv && i < bi);
}

__device__ __forceinline__ void warp_argmin(double& v, long long& i) {
#pragma unroll
	for (int off = 16; off >= 1; off >>= 1) {
		const double ov = __shfl_xor_sync(0xffffffffu, v, off);
		const long long oi = __shfl_xor_sync(0xffffffffu, i, off);
		if (cand_better(ov, oi, v, i)) { v = ov; i = oi; }
	}
}

struct Smem {
	double red_v[NWARP];
	long long red_i[NWARP];
	long long red_c[NWARP];
	double wsum[2][PRICE_NC * 3][NWARP];  // pricing: warp sums (steepest edge: three dots per column), double buffered
	double dsum[3][NWARP];            // O(m) dots
	double bc_v;                      // broadcasts
	long long bc_c;
	double bc_s[3];
	long long tk;                     // update_ftran: next dynamic tile
	double xv[MAXR];                  // sharded: records gathered from the mailbox
	long long xi[MAXR];
	long long xc[MAXR];
	double xv2[MAXR];
	long long xi2[MAXR];
	// pricing ring: TMA bulk copies land in dynamic shared memory, one mbarrier pair per stage
	unsigned long long full[PRICE_MAX_STAGES];
	unsigned long long empty[PRICE_MAX_STAGES];
	long long ring_group[PRICE_MAX_STAGES];   // column group held by the stage, -1 = end of stream
};

// ---------------------------------------------------------------- TMA bulk copy + mbarrier (sm_90+/sm_100a PTX)

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
	asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
	asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long* bar, unsigned bytes) {
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
	const unsigned a = smem_u32(bar);
	asm volatile(
		"{\n"
		".reg .pred p;\n"
		"WAIT_%=:\n"
		"mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
		"@p bra DONE_%=;\n"
		"bra WAIT_%=;\n"
		"DONE_%=:\n"
		"}\n" ::"r"(a), "r"(parity) : "memory");
}
// orders this thread's earlier generic-proxy global accesses (and those it has acquired) with later
// async-proxy ones (TMA reads of y, which the previous pivot wrote with plain stores)
__device__ __forceinline__ void fence_proxy_async_global() {
	asm volatile("fence.proxy.async.global;" ::: "memory");
}
// all state spaces: also orders earlier generic-proxy use of the ring's shared memory (it doubles as the
// update+FTRAN staging area) with the TMA writes that follow
__device__ __forceinline__ void fence_proxy_async_all() {
	asm volatile("fence.proxy.async;" ::: "memory");
}
// global -> shared bulk copy (TMA, 1-D): completes `bytes` transaction bytes on `bar`; 16-byte aligned everything
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_gmem, unsigned bytes, unsigned long long* bar) {
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
		::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// same copy carrying an L2 eviction-priority hint (read-once streams must not push B^-1 out of L2)
__device__ __forceinline__ void tma_load_1d_hint(void* dst_smem, const void* src_gmem, unsigned bytes, unsigned long long* bar,
		unsigned long long policy) {
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
		::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(policy) : "memory");
}
__device__ __forceinline__ unsigned long long l2_policy_evict_first() {
	unsigned long long pol;
	asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
	return pol;
}

// ring position, identical in every thread of the CTA; survives from one pricing phase to the next
struct Ring {
	int stage;
	unsigned phase;
	int nstages;
	__device__ __forceinline__ void advance() { if (++stage == nstages) { stage = 0; phase ^= 1u; } }
};

__device__ __forceinline__ void ring_init(Smem& sh, Ring& cons, Ring& prod, int price_nc) {
	if (threadIdx.x == 0) {
		for (int s = 0; s < PRICE_MAX_STAGES; ++s) { mbar_init(&sh.full[s], 1); mbar_init(&sh.empty[s], NWARP); }
		mbar_fence_init();
	}
	cons.stage = prod.stage = 0;
	cons.phase = prod.phase = 0;
	const int ns = DYN_SMEM_BYTES / ((price_nc + 1) * PRICE_UNIT);
	cons.nstages = prod.nstages = ns < PRICE_MAX_STAGES ? ns : PRICE_MAX_STAGES;
	__syncthreads();
}

// block-wide argmin; result valid in every thread
__device__ __forceinline__ void block_argmin(double& v, long long& i, Smem& sh) {
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	warp_argmin(v, i);
	__syncthreads();
	if (lane == 0) { sh.red_v[warp] = v; sh.red_i[warp] = i; }
	__syncthreads();
	v = sh.red_v[0]; i = sh.red_i[0];
#pragma unroll
	for (int w = 1; w < NWARP; ++w)
		if (cand_better(sh.red_v[w], sh.red_i[w], v, i)) { v = sh.red_v[w]; i = sh.red_i[w]; }
}

// ---------------------------------------------------------------- phase stamps

constexpr int NSTAMP = 16;
// interval j runs from stamp j to stamp j+1 (the last one to stamp 0 of the next iteration)
#define PROFILE_NAMES_JSON \
	"{\"single\": [\"price (+ book2 prologue)\", \"barrier + argmin p\", \"update + FTRAN + ratio groups\", \"barrier\", " \
	"\"argmin q\", \"book1 (row_q, E_q, dots)\", \"barrier\", \"book2 (x_b, y) [unfused only]\", \"barrier [unfused only]\", \"loop\"], " \
	"\"resident\": [\"price (shared memory)\", \"barrier + argmin p\", \"a_p from L2, update + FTRAN + ratio (shared memory)\", " \
	"\"barrier\", \"argmin q\", \"E_q, products, owner: row q out\", \"barrier\", \"row_q / products in, dots, y, x_b\", \"loop\", \"-\"], " \
	"\"sharded\": [\"price\", \"X1: arrive, publish candidate, gather\", \"fetch a_p + barrier\", " \
	"\"update + FTRAN\", \"X2: barrier, alpha + ratio of local rows, publish, gather\", " \
	"\"book1 (E_q, dots; owner: row_q push)\", \"barrier + X3 flag\", \"book2 (x_b, y)\", \"barrier\", \"loop\"]}"

__device__ __forceinline__ unsigned long long globaltimer_ns() {
	unsigned long long t;
	asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
	return t;
}

// CTA 0 / thread 0 stamps the time at which it passes point k of iteration `itl` of this launch
template <typename T>
__device__ __forceinline__ void stamp(const Dev<T>& d, long long itl, int k, int me = 0) {
	if (d.prof_cap > 0 && me == 0 && threadIdx.x == 0 && itl < d.prof_cap)
		d.prof[itl * NSTAMP + k] = globaltimer_ns();
}

// ---------------------------------------------------------------- grid barrier

// All CTAs are co-resident (cooperative launch).  One arrival per CTA on a monotonically increasing counter:
// a release reduction (fire and forget: nobody waits for the old value) and an acquire-load spin, so the
// arrival costs one fence and the wake-up one L2 round trip.  The acquire also invalidates L1, so plain loads
// after the barrier see fresh data.
__device__ __forceinline__ void grid_barrier(Ctl* ctl, unsigned long long& epoch, int G) {
	epoch += G;
	if (G == 1) { __syncthreads(); return; }
	__syncthreads();
	if (threadIdx.x == 0) {
		asm volatile("red.release.gpu.global.add.u64 [%0], 1;" ::"l"(&ctl->bar) : "memory");
		unsigned long long v;
		do {
			asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(&ctl->bar) : "memory");
		} while (v < epoch);
	}
	__syncthreads();
}

// every CTA reduces the per-CTA candidates redundantly -> same answer everywhere
__device__ __forceinline__ void reduce_cands(const Cand* cand, int ncand, double& v, long long& i, Smem& sh) {
	v = CUDART_INF; i = LLONG_MAX;
	for (int k = threadIdx.x; k < ncand; k += NT) {
		const double cv = __ldcg(&cand[k].val);
		const long long ci = __ldcg(&cand[k].idx);
		if (cand_better(cv, ci, v, i)) { v = cv; i = ci; }
	}
	block_argmin(v, i, sh);
}

__device__ __forceinline__ long long reduce_counts(const long long* cnt, int n, Smem& sh) {
	long long c = 0;
	for (int k = threadIdx.x; k < n; k += NT) c += __ldcg(&cnt[k]);
#pragma unroll
	for (int off = 16; off >= 1; off >>= 1) c += __shfl_xor_sync(0xffffffffu, c, off);
	__syncthreads();
	if ((threadIdx.x & 31) == 0) sh.red_c[threadIdx.x >> 5] = c;
	__syncthreads();
	c = 0;
#pragma unroll
	for (int w = 0; w < NWARP; ++w) c += sh.red_c[w];
	return c;
}

// argmin over the per-CTA candidates and the sum of their counts in one pass (one set of loads and barriers)
__device__ __forceinline__ long long reduce_cands_counts(const Cand* cand, const long long* cnt, int n, double& v, long long& i, Smem& sh) {
	v = CUDART_INF; i = LLONG_MAX;
	long long c = 0;
	for (int k = threadIdx.x; k < n; k += NT) {
		const double cv = __ldcg(&cand[k].val);
		const long long ci = __ldcg(&cand[k].idx);
		c += __ldcg(&cnt[k]);
		if (cand_better(cv, ci, v, i)) { v = cv; i = ci; }
	}
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	warp_argmin(v, i);
#pragma unroll
	for (int off = 16; off >= 1; off >>= 1) c += __shfl_xor_sync(0xffffffffu, c, off);
	__syncthreads();
	if (lane == 0) { sh.red_v[warp] = v; sh.red_i[warp] = i; sh.red_c[warp] = c; }
	__syncthreads();
	v = sh.red_v[0]; i = sh.red_i[0]; c = sh.red_c[0];
#pragma unroll
	for (int w = 1; w < NWARP; ++w) {
		if (cand_better(sh.red_v[w], sh.red_i[w], v, i)) { v = sh.red_v[w]; i = sh.red_i[w]; }
		c += sh.red_c[w];
	}
	return c;
}

// ---------------------------------------------------------------- phase: pricing

// e_j = y.A_j - c_j for the ns dense columns, e_j = y_k - c_j for the unit columns, fused
// with the argmin.  Replaces cublasSgemm(M=1) + cub::DeviceReduce::ArgMin (v4:289-294).
//
// A is streamed through a shared-memory ring (4 or 6 stages) by TMA bulk copies
// (cp.async.bulk + mbarrier complete_tx): one block = y + price_nc columns x RB rows, RB = NT
// 16-byte vectors, i.e. one row step of the whole CTA.  Warp 0 is the producer and runs
// nstages-1 blocks ahead of the consumers (all NT threads, itself included), across
// column-group boundaries, so HBM requests never drain while a group is being reduced.
// Column groups are handed out dynamically: the first one is the CTA's index, the others
// come from a ticket counter, which evens out slow and fast SMs.  Groups are price_nc columns
// wide; a ragged remainder goes one column at a time.
// The summation order of a column does not depend on any of this (see the file header).
template <typename T>
__device__ void price_phase(const Dev<T>& d, Smem& sh, unsigned char* ringbuf, Ring& cons, Ring& prod, int part, int nparts) {
	using V = typename VecT<T>::V;
	constexpr int VN = VecT<T>::N;
	constexpr int RB = NT * VN;               // rows per block
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const long long ld = d.ld;
	const int NCW = d.price_nc;                                  // group width (2 or 4)
	const int stage_bytes = (NCW + 1) * PRICE_UNIT;
	const long long nquad = d.nsl / NCW;                         // full-width groups
	const long long ngroups = nquad + (d.nsl - nquad * NCW);     // + single columns
	const int nrb = (int)((ld + RB - 1) / RB);

	double best_v = CUDART_INF;
	long long best_i = LLONG_MAX;

	// ---- producer: warp 0, all lanes in step (same cursor in every lane).  One thread issuing a block alone
	// needs ~0.3 us of dependent scalar work per block, more than a 2-column block takes to stream; spread over
	// the lanes (lane 0: barrier bookkeeping, lane 1: y, lanes 2..: one column each) it is a third of that.
	const unsigned long long pol_stream = l2_policy_evict_first();   // A is read once per pivot
	long long pg = part, pnext = ngroups;
	int prb = 0;
	bool pend = false;
	auto produce = [&]() {
		mbar_wait(&sh.empty[prod.stage], prod.phase ^ 1u);       // consumers have released the stage
		if (pg >= ngroups) {
			if (lane == 0) {
				sh.ring_group[prod.stage] = -1;                    // end of this CTA's stream
				mbar_arrive(&sh.full[prod.stage]);
			}
			pend = true;
		} else {
			if (prb == 0 && lane == 0) pnext = (long long)nparts + atomicAdd(&d.ctl->price_ctr, 1u);   // used nrb blocks later
			const long long r0 = (long long)prb * RB;
			const unsigned colbytes = (unsigned)((ld - r0 < RB ? ld - r0 : RB) * (long long)sizeof(T));
			const int nc = pg < nquad ? NCW : 1;
			const long long c0 = pg < nquad ? pg * NCW : nquad * NCW + (pg - nquad);
			unsigned char* dst = ringbuf + prod.stage * stage_bytes;
			if (lane == 0) {
				sh.ring_group[prod.stage] = pg;
				// the phase cannot complete before this arrival, whatever the order of the copies' complete_tx
				mbar_arrive_expect_tx(&sh.full[prod.stage], (unsigned)(nc + 1) * colbytes);
			} else if (lane == 1) {
				tma_load_1d(dst, d.y + r0, colbytes, &sh.full[prod.stage]);
			} else if (lane < nc + 2) {
				const int k = lane - 2;
				tma_load_1d_hint(dst + (k + 1) * PRICE_UNIT, d.A + (c0 + k) * ld + r0, colbytes, &sh.full[prod.stage], pol_stream);
			}
			if (++prb == nrb) { prb = 0; pg = __shfl_sync(0xffffffffu, pnext, 0); }
		}
		prod.advance();
	};
	__syncthreads();
	if (warp == 0) {
		fence_proxy_async_all();
		for (int k = 0; k < prod.nstages - 1 && !pend; ++k) produce();
	}

	// ---- consumers
	T acc[PRICE_NC][VN];
	int crb = 0, buf = 0;
	while (true) {
		if (warp == 0 && !pend) produce();
		const bool act = (long long)crb * RB + (long long)tid * VN < ld;
		mbar_wait(&sh.full[cons.stage], cons.phase);
		const long long g = sh.ring_group[cons.stage];
		const int nc = g < nquad ? NCW : 1;
		if (g >= 0) {
			if (crb == 0) {
#pragma unroll
				for (int k = 0; k < PRICE_NC; ++k)
#pragma unroll
					for (int v = 0; v < VN; ++v) acc[k][v] = T(0);
			}
			if (act) {
				const unsigned char* src = ringbuf + cons.stage * stage_bytes + tid * 16;
				const V yv = *reinterpret_cast<const V*>(src);
#pragma unroll
				for (int k = 0; k < PRICE_NC; ++k) {
					if (k < nc) {
						const V av = *reinterpret_cast<const V*>(src + (k + 1) * PRICE_UNIT);
#pragma unroll
						for (int v = 0; v < VN; ++v) acc[k][v] = fma_t(Mem<T>::get(av, v), Mem<T>::get(yv, v), acc[k][v]);
					}
				}
			}
		}
		__syncwarp();
		if (lane == 0) mbar_arrive(&sh.empty[cons.stage]);         // this warp is done with the stage
		cons.advance();
		if (g < 0) break;
		if (++crb == nrb) {
			crb = 0;
#pragma unroll
			for (int k = 0; k < PRICE_NC; ++k) {
				if (k < nc) {
					T s = acc[k][0];
#pragma unroll
					for (int v = 1; v < VN; ++v) s = s + acc[k][v];
					s = warp_butterfly_sum(s);
					if (lane == 0) sh.wsum[buf][k][warp] = (double)s;
				}
			}
			__syncthreads();
			if (tid < nc) {
				T s = (T)sh.wsum[buf][tid][0];
#pragma unroll
				for (int w = 1; w < NWARP; ++w) s = s + (T)sh.wsum[buf][tid][w];
				const long long c0 = g < nquad ? g * NCW : nquad * NCW + (g - nquad);
				const long long j = d.col0 + c0 + tid;               // global column index
				const double e = (double)(s - d.c[j]);
				if (cand_better(e, j, best_v, best_i)) { best_v = e; best_i = j; }
			}
			buf ^= 1;
		}
	}

	// unit (slack) columns: e_j = y_k - c_j, no matrix bytes (the reference reads
	// the identity block through the same GEMM; 0*y terms vanish exactly)
	for (long long k = d.k0 + (long long)part * NT + tid; k < d.k1; k += (long long)nparts * NT) {
		const double e = (double)(d.y[k] - d.c[d.ns + k]);
		const long long j = d.ns + k;
		if (cand_better(e, j, best_v, best_i)) { best_v = e; best_i = j; }
	}

	block_argmin(best_v, best_i, sh);
	if (tid == 0) { d.cand[part].val = best_v; d.cand[part].idx = best_i; }
}

// Pricing without the ring.  For LPs whose A shard is L2 resident (m <= ~2048) there is nothing to stream from
// HBM, a pass is a few microseconds and the ring's start-up (first TMA round trip, barrier handshakes) would be a
// third of it; measured, this path also wins by ~6 % of the pass at m = 8192 and ties with the ring above that, so
// the host selects it up to a 2 GB A shard (Engine::set_columns).  Register-staged 16-byte loads, 16 in flight per thread; the per-column summation order is
// the one of price_phase (thread t owns vectors t, t+256, ...), so both give the same bits.
//
// Work items are handed out by the ticket counter (first item = CTA index), like the tiles of the update pass:
// fast and slow SMs even out, results do not depend on who prices a column.  Items are groups of PRICE_NC columns
// except for the last d.price_tail columns of the block, which go one at a time: the pass ends when the slowest CTA
// finishes its last item, and a single column is a quarter of a group (measured on 8 GPUs, m = 32768: a group is
// ~40 us of a ~170 us pass).

// dot products of NC consecutive columns (base, leading dimension ldm, nrows rows) with NV vectors: per-thread
// partial sums reduced to one value per warp in sh.wsum[buf][k * NV + w][warp].  UR row steps are unrolled so that
// NC * UR 16-byte loads are in flight per thread.  COHERENT: the matrix is written by this kernel (B^-1), use the
// coherent path; otherwise the read-only non-coherent one (A).  The summation order of every dot is the pricing
// order of the file header, whatever NC / UR / NV.
template <typename T, int NC, int UR, int NV, bool COHERENT>
__device__ __forceinline__ void column_dots(const T* base, long long ldm, long long nrows, const T* const (&vec)[3], Smem& sh, int buf) {
	using M = Mem<T>;
	using V = typename VecT<T>::V;
	constexpr int VN = VecT<T>::N;
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	T acc[NC][NV][VN];
#pragma unroll
	for (int k = 0; k < NC; ++k)
#pragma unroll
		for (int w = 0; w < NV; ++w)
#pragma unroll
			for (int v = 0; v < VN; ++v) acc[k][w][v] = T(0);
#pragma unroll UR
	for (long long i = (long long)tid * VN; i < nrows; i += (long long)NT * VN) {
		V av[NC];
#pragma unroll
		for (int k = 0; k < NC; ++k) av[k] = COHERENT ? M::ld_stream(base + k * ldm + i) : M::ld_nc(base + k * ldm + i);
#pragma unroll
		for (int w = 0; w < NV; ++w) {
			const V yv = *reinterpret_cast<const V*>(vec[w] + i);
#pragma unroll
			for (int k = 0; k < NC; ++k)
#pragma unroll
				for (int v = 0; v < VN; ++v) acc[k][w][v] = fma_t(M::get(av[k], v), M::get(yv, v), acc[k][w][v]);
		}
	}
#pragma unroll
	for (int k = 0; k < NC; ++k)
#pragma unroll
		for (int w = 0; w < NV; ++w) {
			T s = acc[k][w][0];
#pragma unroll
			for (int v = 1; v < VN; ++v) s = s + acc[k][w][v];
			s = warp_butterfly_sum(s);
			if (lane == 0) sh.wsum[buf][k * NV + w][warp] = (double)s;
		}
}

// the 8 warp sums of dot `slot`, left to right
template <typename T>
__device__ __forceinline__ T warp_sums(const Smem& sh, int buf, int slot) {
	T s = (T)sh.wsum[buf][slot][0];
#pragma unroll
	for (int w = 1; w < NWARP; ++w) s = s + (T)sh.wsum[buf][slot][w];
	return s;
}

// ysm: y staged in shared memory by book2_prologue (nullptr: read d.y through L1/L2)
template <typename T>
__device__ void price_phase_direct(const Dev<T>& d, Smem& sh, const T* ysm, int part, int nparts) {
	const int tid = threadIdx.x;
	double best_v = CUDART_INF;
	long long best_i = LLONG_MAX;

	const long long c1 = d.nsl;
	const long long tail = d.price_tail < c1 ? d.price_tail : c1;
	const long long nq = (c1 - tail) / PRICE_NC;              // full groups
	const long long nitems = nq + (c1 - nq * PRICE_NC);       // + single columns
	int buf = 0;
	for (long long g = part; g < nitems; buf ^= 1) {
		if (tid == 0) sh.tk = (long long)nparts + atomicAdd(&d.ctl->price_ctr, 1u);   // read after the barrier below
		const bool quad = g < nq;
		const long long col = quad ? g * PRICE_NC : nq * PRICE_NC + (g - nq);
		const T* const vec[3] = {ysm ? ysm : d.y, nullptr, nullptr};
		if (quad) column_dots<T, PRICE_NC, 4, 1, false>(d.A + col * d.ld, d.ld, d.ld, vec, sh, buf);
		else      column_dots<T, 1, 16, 1, false>(d.A + col * d.ld, d.ld, d.ld, vec, sh, buf);
		__syncthreads();
		g = sh.tk;
		if (tid < (quad ? PRICE_NC : 1)) {
			const T s = warp_sums<T>(sh, buf, tid);
			const long long j = d.col0 + col + tid;     // global column index
			const double e = (double)(s - d.c[j]);
			if (cand_better(e, j, best_v, best_i)) { best_v = e; best_i = j; }
		}
		__syncthreads();                              // sh.tk is rewritten at the top of the next item
	}

	const T* yp = ysm ? ysm : d.y;
	for (long long k = d.k0 + (long long)part * NT + tid; k < d.k1; k += (long long)nparts * NT) {   // unit (slack) columns
		const double e = (double)(yp[k] - d.c[d.ns + k]);
		const long long j = d.ns + k;
		if (cand_better(e, j, best_v, best_i)) { best_v = e; best_i = j; }
	}

	block_argmin(best_v, best_i, sh);
	if (tid == 0) { d.cand[part].val = best_v; d.cand[part].idx = best_i; }
}

// ---------------------------------------------------------------- steepest-edge pricing (README.md:16-17)
//
// p = argmax e_j^2 / gamma_j over the attractive columns e_j < -eps (lowest index on ties), gamma_j = 1 + |B^-1 a_j|^2
// kept exact by the Goldfarb-Reid recurrence.  The recurrence of the PREVIOUS pivot rides in this pass: besides
// e_j = y.a_j - c_j every column also gets  r_j = row_q.a_j  and  w_j = v.a_j  (v = B^-T alpha) from the same
// bytes of A, then
//     t = r_j / alpha_q,   gamma_j <- max(gamma_j - 2 t w_j + t^2 gamma_p, 1 + t^2),
// the entering column of that pivot is set to 2 and its leaving variable to max(gamma_p / alpha_q^2, 1 + 1/alpha_q^2).
// The optimality test is the reference's (min e_j >= -eps, v4:299), so both candidates are reduced.
// Mirrored by the oracle (oracle/simplex_oracle_impl.h, pricing_rule = 1) with the same arithmetic.

struct SeUpd {
	bool on;                 // a pivot's recurrence is pending
	long long p, leaving;    // its entering column / leaving variable (global column indices)
	double alpha_q, gamma_p;
};

template <typename T>
__device__ __forceinline__ T se_weight(const Dev<T>& d, const SeUpd& u, long long j, T r, T w) {
	T g = d.gamma[j];
	if (u.on) {
		const T aq = (T)u.alpha_q, gp = (T)u.gamma_p;
		if (j == u.p) g = T(2);
		else if (j == u.leaving) {
			const T ia = T(1) / aq;
			const T g1 = gp * (ia * ia), g2 = fma_t(ia, ia, T(1));
			g = g1 > g2 ? g1 : g2;
		} else {
			const T t = r / aq;
			const T g1 = fma_t(t * t, gp, fma_t(T(-2) * t, w, g));
			const T g2 = fma_t(t, t, T(1));
			g = g1 > g2 ? g1 : g2;
		}
		d.gamma[j] = g;
	}
	return g;
}

// vec = {y, row_q, v}: shared-memory copies where they fit, global otherwise
template <typename T>
__device__ void price_phase_se(const Dev<T>& d, Smem& sh, const T* const (&vec)[3], const SeUpd& u, int part, int nparts) {
	const int tid = threadIdx.x;
	double best_v = CUDART_INF, se_v = CUDART_INF;      // (min e, index) and (min -e^2/gamma, index)
	long long best_i = LLONG_MAX, se_i = LLONG_MAX;
	const double neg_eps = -d.eps;
	auto consider = [&](long long j, T e, T r, T w) {
		const T g = se_weight<T>(d, u, j, r, w);
		if (cand_better((double)e, j, best_v, best_i)) { best_v = (double)e; best_i = j; }
		if ((double)e < neg_eps) {
			const double sc = -(double)((e * e) / g);
			if (cand_better(sc, j, se_v, se_i)) { se_v = sc; se_i = j; }
		}
	};

	const long long c1 = d.nsl;
	const long long nq = c1 / PRICE_NC;
	const long long nitems = nq + (c1 - nq * PRICE_NC);
	int buf = 0;
	for (long long g = part; g < nitems; buf ^= 1) {
		if (tid == 0) sh.tk = (long long)nparts + atomicAdd(&d.ctl->price_ctr, 1u);
		const bool quad = g < nq;
		const long long col = quad ? g * PRICE_NC : nq * PRICE_NC + (g - nq);
		const T* base = d.A + col * d.ld;
		if (u.on) {
			if (quad) column_dots<T, PRICE_NC, 2, 3, false>(base, d.ld, d.ld, vec, sh, buf);
			else      column_dots<T, 1, 8, 3, false>(base, d.ld, d.ld, vec, sh, buf);
		} else {
			if (quad) column_dots<T, PRICE_NC, 4, 1, false>(base, d.ld, d.ld, vec, sh, buf);
			else      column_dots<T, 1, 16, 1, false>(base, d.ld, d.ld, vec, sh, buf);
		}
		__syncthreads();
		g = sh.tk;
		if (tid < (quad ? PRICE_NC : 1)) {
			const long long j = d.col0 + col + tid;
			const int nv = u.on ? 3 : 1;
			const T e = warp_sums<T>(sh, buf, tid * nv) - d.c[j];
			const T r = u.on ? warp_sums<T>(sh, buf, tid * nv + 1) : T(0);
			const T w = u.on ? warp_sums<T>(sh, buf, tid * nv + 2) : T(0);
			consider(j, e, r, w);
		}
		__syncthreads();
	}
	for (long long k = d.k0 + (long long)part * NT + tid; k < d.k1; k += (long long)nparts * NT)   // unit (slack) columns
		consider(d.ns + k, vec[0][k] - d.c[d.ns + k], u.on ? vec[1][k] : T(0), u.on ? vec[2][k] : T(0));

	block_argmin(best_v, best_i, sh);
	block_argmin(se_v, se_i, sh);
	if (tid == 0) {
		d.cand[part].val = best_v; d.cand[part].idx = best_i;
		d.cand2[part].val = se_v; d.cand2[part].idx = se_i;
	}
}

// v = B^-T alpha: the column dots of B^-1 with alpha, in the pricing order (one extra read of B^-1 per pivot,
// the price of exact steepest-edge weights).  Column groups come from ctl->btran_ctr.
template <typename T>
__device__ void btran_phase(const Dev<T>& d, Smem& sh, const T* alpha_vec, int part, int nparts) {
	const int tid = threadIdx.x;
	const long long c1 = d.m;
	const long long nq = c1 / PRICE_NC;
	const long long nitems = nq + (c1 - nq * PRICE_NC);
	const T* const vec[3] = {alpha_vec, nullptr, nullptr};
	int buf = 0;
	for (long long g = part; g < nitems; buf ^= 1) {
		if (tid == 0) sh.tk = (long long)nparts + atomicAdd(&d.ctl->btran_ctr, 1u);
		const bool quad = g < nq;
		const long long col = quad ? g * PRICE_NC : nq * PRICE_NC + (g - nq);
		if (quad) column_dots<T, PRICE_NC, 4, 1, true>(d.B + col * d.ldb, d.ldb, d.ldb, vec, sh, buf);
		else      column_dots<T, 1, 16, 1, true>(d.B + col * d.ldb, d.ldb, d.ldb, vec, sh, buf);
		__syncthreads();
		g = sh.tk;
		if (tid < (quad ? PRICE_NC : 1)) d.vbt[col + tid] = warp_sums<T>(sh, buf, tid);
		__syncthreads();
	}
}

// ---------------------------------------------------------------- phase: update + FTRAN

// alpha_i = sum over the FTRAN chunks of alpha_part[ck][i], strictly left to right; the loads of
// 16 chunks are issued together (predicated, no serial remainder), only the adds are ordered
template <typename T>
__device__ __forceinline__ T sum_chunk_partials(const T* part0, long long stride, int nchunk) {
	T a = __ldcg(part0);
	for (int c0 = 1; c0 < nchunk; c0 += 16) {
		T v[16];
#pragma unroll
		for (int u = 0; u < 16; ++u) v[u] = c0 + u < nchunk ? __ldcg(part0 + (long long)(c0 + u) * stride) : T(0);
#pragma unroll
		for (int u = 0; u < 16; ++u)
			if (c0 + u < nchunk) a = a + v[u];
	}
	return a;
}


// The same sums for 32 consecutive local rows [il0, il0 + 32) by the whole CTA: warp w loads chunks w, w + 8, ...
// (one coalesced 32-row segment each, all loads of the CTA in flight together) into `stage` (nchunk x 32), then
// threads 0..31 add their row's partials left to right from shared memory.  One L2 round trip instead of
// nchunk / 16 dependent ones per thread; same association as sum_chunk_partials.  Result valid in threads 0..31.
template <typename T>
__device__ __forceinline__ T sum_partials_rows32(const Dev<T>& d, T* stage, long long il0) {
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const bool in = il0 + lane < d.ldb;
	for (int c = warp; c < d.nchunk; c += NWARP)
		stage[c * 32 + lane] = in ? __ldcg(d.alpha_part + (long long)c * d.ldb + il0 + lane) : T(0);
	__syncthreads();
	T a = T(0);
	if (tid < 32) {
		a = stage[lane];
		for (int c = 1; c < d.nchunk; ++c) a = a + stage[c * 32 + lane];
	}
	__syncthreads();
	return a;
}

template <typename T> __device__ __forceinline__ T* xalpha(const Dev<T>& d, int r);

// tile count of a row group: release at gpu scope (the tile's alpha_part stores, made by other threads of the
// CTA before a barrier, are visible at L2 before the count is).  A release atom is one MEMBAR.ALL.GPU + ATOM;
// __threadfence() would be an SC fence plus an L1 invalidation (MEMBAR.SC + ERRBAR + CCTL.IVALL) per tile.
__device__ __forceinline__ unsigned int post_tile(unsigned int* ctr) {
	unsigned int old;
	asm volatile("atom.add.release.gpu.global.u32 %0, [%1], 1;" : "=r"(old) : "l"(ctr) : "memory");
	return old + 1u;
}

// Ratio test of one finished row group (v4:199-208, 311-325): alpha of the group's rows = sum of their chunk
// partials (left to right), stored into every rank's alpha vector (one rank: our own), masked (theta, index)
// argmin over alpha > pivot_tol + eligible count -> rcand[g] / rcnt[g].  Run by the CTA that completed the
// group's last tile while the other CTAs keep streaming B^-1.
template <typename T>
__device__ void finish_row_group(const Dev<T>& d, Smem& sh, long long g, long long grows) {
	const int tid = threadIdx.x;
	double best_v = CUDART_INF;
	long long best_i = LLONG_MAX;
	long long elig = 0;
	const T tol = (T)d.pivot_tol;
	for (long long r = tid; r < grows; r += NT) {
		const long long il = g * grows + r;
		if (il >= d.ldb) break;
		const T a = sum_chunk_partials(d.alpha_part + il, d.ldb, d.nchunk);
		const long long i = d.row0 + il;
		for (int k = 0; k < d.nranks; ++k) xalpha(d, k)[i] = a;
		if (i < d.m && a > tol) {
			++elig;
			const double th = (double)(ratio_num(d.x_b[i], d.ratio_mode) / a);
			if (cand_better(th, i, best_v, best_i)) { best_v = th; best_i = i; }
		}
	}
	block_argmin(best_v, best_i, sh);
#pragma unroll
	for (int off = 16; off >= 1; off >>= 1) elig += __shfl_xor_sync(0xffffffffu, elig, off);
	__syncthreads();
	if ((tid & 31) == 0) sh.red_c[tid >> 5] = elig;
	__syncthreads();
	if (tid == 0) {
		long long c = 0;
#pragma unroll
		for (int w = 0; w < NWARP; ++w) c += sh.red_c[w];
		d.rcand[g].val = best_v;
		d.rcand[g].idx = best_i;
		d.rcnt[g] = c;
	}
}

// One pass over B^-1:  (UPDATE) B^-1 += E_q (x) row_q   [cublasSger, v4:333]
//                      (FTRAN)  alpha = B^-1_new a_p     [cublasSgemv, v4:307-308 of the NEXT iteration]
// Thread owns VN consecutive rows (one 16-byte vector), a warp 32*VN rows, the
// CTA's 8 warps are arranged WR (rows) x WC (columns) over a tile of
// WR*32*VN rows x CHUNK columns.  row_q[chunk] and a_p[chunk] are staged in
// shared memory.  alpha_part[chunk][row] receives the chunk partial.
// Tiles are handed out chunk by chunk, row tile fastest (measured: concurrent CTAs must sweep whole columns — a
// group-major order that leaves only 2 KB of a column contiguous costs 8 % of the pass).  FINISH (row groups of
// d.rg row tiles = 256+ rows): a CTA counts its tile on the group's counter; whoever completes the group sums its
// chunk partials and runs the ratio test of its rows (finish_row_group), so the ratio test of the reference
// (v4:311-325) needs neither a phase nor a grid barrier of its own.  The count of tile k is posted behind the
// first loads of tile k+1 and looked at after tile k+1 has been streamed.  Measured on one GPU the release
// (one MEMBAR.GPU round trip per tile in one warp, ~0.65 us per tile) costs more than the phase and barrier it
// saves — 14 tiles per CTA at m = 8192, 55 on a 2-GPU shard of m = 32768 — so FINISH is an option
// (options.fuse_ratio = 1), not the default, on one GPU and in the sharded loop alike.
template <typename T, int WC, bool UPDATE, bool FTRAN, bool FINISH>
__device__ void update_ftran_phase(const Dev<T>& d, Smem& sh, unsigned char* dyn, const T* acol, long long uk, bool reverse, int part, int nparts) {
	using M = Mem<T>;
	using V = typename VecT<T>::V;
	constexpr int VN = VecT<T>::N;
	constexpr int WR = NWARP / WC;
	constexpr int TR = WR * 32 * VN;      // tile rows
	constexpr int SUBS = (CHUNK / SUBW) / WC; // sub-blocks per warp
	static_assert(SUBS >= 1, "bad WC");

	static_assert(NT == CHUNK, "staging assumes one thread per chunk column");
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const int wr = warp % WR, wc = warp / WR;
	const long long ld = d.ldb, m = d.m;   // local row block
	const long long ntr = (ld + TR - 1) / TR;
	const long long ntiles = ntr * d.nchunk;
	const long long RG = d.rg;                               // row tiles per row group (the last group may be shorter)
	// staging area in dynamic shared memory (aliases the idle pricing ring): row_q chunk, a_p chunk, combine
	T* stage_rq = reinterpret_cast<T*>(dyn);
	T* stage_a = reinterpret_cast<T*>(dyn + CHUNK * 8);
	double (*comb)[32][4] = reinterpret_cast<double (*)[32][4]>(dyn + 2 * CHUNK * 8);
	const bool unit = acol == nullptr;     // entering column is the unit vector e_uk

	// tiles are handed out dynamically: the first one is the CTA's index, the others come from a
	// ticket counter (results do not depend on which CTA computes a tile).  Every other pass walks
	// the tiles backwards, so the part of B^-1 that is still in L2 from the previous pass (up to
	// the L2 capacity, dirty lines included) is touched first and never makes the trip to HBM.
	long long ticket = part;
	long long prev_grp = -1;               // group of the tile this CTA finished last, not yet counted
	unsigned int prev_target = 0, prev_done = 0;
	constexpr int POSTER = 32;             // the thread that posts tile counts (warp 1, lane 0; thread 0 draws the tickets)
	while (ticket < ntiles) {
		const long long tile = reverse ? ntiles - 1 - ticket : ticket;
		const long long rt = tile % ntr, ck = tile / ntr;     // row tile fastest: concurrent CTAs sweep whole columns
		const long long grp = rt / RG;
		const long long rgg = ntr - grp * RG < RG ? ntr - grp * RG : RG;   // row tiles of this group
		const long long j0 = ck * CHUNK;
		__syncthreads();
		if (tid == 0) sh.tk = (long long)nparts + atomicAdd(&d.ctl->upd_ctr, 1u);
		{
			const long long j = j0 + tid;     // NT == CHUNK
			T r = T(0), a = T(0);
			if (j < m) {
				if (UPDATE) r = __ldcg(d.row_q + j);      // mailbox data (peer-written when sharded): read at L2
				if (FTRAN) a = unit ? (j == uk ? T(1) : T(0)) : acol[j];   // plain load: acol may have been written by this kernel
			}
			stage_rq[tid] = r;
			stage_a[tid] = a;
		}
		__syncthreads();
		const long long next_ticket = sh.tk;
		bool post = FINISH && prev_grp >= 0 && tid == POSTER;   // count the previous tile on its group (see below)

		const long long row = rt * TR + (long long)wr * 32 * VN + (long long)lane * VN;
		const bool active = row < ld;     // warp uniform (ld is a multiple of 32*VN)
		T wpart[VN];
#pragma unroll
		for (int v = 0; v < VN; ++v) wpart[v] = T(0);

		if (active) {
			V Ev;
			if (UPDATE) Ev = *reinterpret_cast<const V*>(d.E_q + d.row0 + row);
			// pairwise tree over this warp's sub-blocks, kept as a binary-counter stack so
			// at most log2(SUBS)+1 partials are live
			T stk[4][VN];
#pragma unroll
			for (int s = 0; s < SUBS; ++s) {
				const int jb = wc * (CHUNK / WC) + s * SUBW;   // offset inside the chunk
				T acc[VN];
#pragma unroll
				for (int v = 0; v < VN; ++v) acc[v] = T(0);
				T* bp = d.B + (j0 + jb) * ld + row;
				long long ncols = m - (j0 + jb);
				if (ncols >= SUBW) {
#pragma unroll
					for (int u0 = 0; u0 < SUBW; u0 += 8) {
						V v8[8];
#pragma unroll
						for (int u = 0; u < 8; ++u) v8[u] = M::ld_stream(bp + (long long)(u0 + u) * ld);
#pragma unroll
						for (int u = 0; u < 8; ++u) {
							const T r = stage_rq[jb + u0 + u], a = stage_a[jb + u0 + u];
#pragma unroll
							for (int v = 0; v < VN; ++v) {
								T x = M::get(v8[u], v);
								if (UPDATE) { x = fma_t(M::get(Ev, v), r, x); M::set(v8[u], v, x); }
								if (FTRAN) acc[v] = fma_t(x, a, acc[v]);
							}
							if (UPDATE) M::st_stream(bp + (long long)(u0 + u) * ld, v8[u]);
						}
					}
				} else {
					for (int u = 0; u < ncols; ++u) {
						V vv = M::ld_stream(bp + (long long)u * ld);
						const T r = stage_rq[jb + u], a = stage_a[jb + u];
#pragma unroll
						for (int v = 0; v < VN; ++v) {
							T x = M::get(vv, v);
							if (UPDATE) { x = fma_t(M::get(Ev, v), r, x); M::set(vv, v, x); }
							if (FTRAN) acc[v] = fma_t(x, a, acc[v]);
						}
						if (UPDATE) M::st_stream(bp + (long long)u * ld, vv);
					}
				}
				int lvl = 0;
#pragma unroll
				for (; lvl < 3; ++lvl) {
					if (!((s >> lvl) & 1)) break;
#pragma unroll
					for (int v = 0; v < VN; ++v) acc[v] = stk[lvl][v] + acc[v];
				}
#pragma unroll
				for (int v = 0; v < VN; ++v) stk[lvl][v] = acc[v];
			}
			constexpr int TOP = SUBS == 8 ? 3 : SUBS == 4 ? 2 : SUBS == 2 ? 1 : 0;
#pragma unroll
			for (int v = 0; v < VN; ++v) wpart[v] = stk[TOP][v];
		}

		if (FTRAN) {
			if (WC == 1) {
				if (active) {
					V o;
#pragma unroll
					for (int v = 0; v < VN; ++v) M::set(o, v, wpart[v]);
					*reinterpret_cast<V*>(d.alpha_part + ck * ld + row) = o;
				}
			} else {
				// continue the same pairwise tree across the WC warps that share these rows
#pragma unroll
				for (int v = 0; v < VN; ++v) comb[warp][lane][v] = (double)wpart[v];
				__syncthreads();
				if (wc == 0 && active) {
					T t[WC][VN];
#pragma unroll
					for (int c = 0; c < WC; ++c)
#pragma unroll
						for (int v = 0; v < VN; ++v) t[c][v] = (T)comb[c * WR + wr][lane][v];
#pragma unroll
					for (int w = 1; w < WC; w <<= 1)
#pragma unroll
						for (int c = 0; c + w < WC; c += 2 * w)
#pragma unroll
							for (int v = 0; v < VN; ++v) t[c][v] = t[c][v] + t[c + w][v];
					V o;
#pragma unroll
					for (int v = 0; v < VN; ++v) M::set(o, v, t[0][v]);
					*reinterpret_cast<V*>(d.alpha_part + ck * ld + row) = o;
				}
			}
		}
		if (FINISH) {
			if (prev_grp >= 0) {               // CTA uniform
				if (post) prev_done = post_tile(&d.grp_done[prev_grp]);   // (inactive rows / ragged chunk: the fast path above was not taken)
				if (tid == POSTER) {
					const bool last = prev_done == prev_target;
					if (last) { d.grp_done[prev_grp] = 0; __threadfence(); }   // acquire side: the group's partials are complete at L2
					sh.bc_c = last;
				}
				__syncthreads();
				const bool fin = sh.bc_c != 0;
				__syncthreads();
				if (fin) finish_row_group<T>(d, sh, prev_grp, RG * TR);
			}
			prev_grp = grp;
			prev_target = (unsigned int)(rgg * d.nchunk);
		}
		ticket = next_ticket;
	}
	if (FINISH && prev_grp >= 0) {             // this CTA's last tile: post and look at once
		__syncthreads();
		if (tid == POSTER) {
			const bool last = post_tile(&d.grp_done[prev_grp]) == prev_target;
			if (last) { d.grp_done[prev_grp] = 0; __threadfence(); }
			sh.bc_c = last;
		}
		__syncthreads();
		const bool fin = sh.bc_c != 0;
		__syncthreads();
		if (fin) finish_row_group<T>(d, sh, prev_grp, RG * TR);
	}
}

// ---------------------------------------------------------------- phase: ratio test

// alpha_i = sum of the chunk partials (left to right); theta_i = x_b_i/alpha_i
// over alpha_i > 0 (strict, v4:203); masked argmin + eligible-row count.
// Replaces cudaMemset + compute_theta + D2H + cub ArgMin (v4:311-325).
template <typename T, bool FROM_PARTIALS>
__device__ void ratio_phase(const Dev<T>& d, Smem& sh, int part, int nparts, T* stage = nullptr) {
	const int tid = threadIdx.x;
	double best_v = CUDART_INF;
	long long best_i = LLONG_MAX;
	long long elig = 0;
	auto consider = [&](long long i, T a) {
		if (a > (T)d.pivot_tol) {
			++elig;
			const T xb = ratio_num(d.x_b[i], d.ratio_mode);
			// Harris, first pass: the widest step the tolerance allows (the row is chosen by harris_phase2)
			const double th = d.ratio_mode == 2 ? (double)((xb + (T)d.harris_delta) / a) : (double)(xb / a);
			if (cand_better(th, i, best_v, best_i)) { best_v = th; best_i = i; }
		}
	};
	const long long nblk = (d.m + 31) / 32;
	if (FROM_PARTIALS && stage && nblk <= 2 * (long long)nparts) {
		// blocks of 32 rows, the CTA's warps load the chunk partials together (sum_partials_rows32); only while
		// every CTA gets at most two blocks (measured at m = 32768 on one GPU, 3.5 blocks per CTA: 20.7 us against
		// 12.8 us for one row per thread)
		for (long long blk = part; blk < nblk; blk += nparts) {
			const T a = sum_partials_rows32<T>(d, stage, blk * 32);
			const long long i = blk * 32 + tid;
			if (tid < 32 && i < d.m) {
				d.alpha[i] = a;
				consider(i, a);
			}
		}
	} else {
		for (long long i = (long long)part * NT + tid; i < d.m; i += (long long)nparts * NT) {
			T a;
			if (FROM_PARTIALS) {
				a = sum_chunk_partials(d.alpha_part + i, d.ldb, d.nchunk);
				d.alpha[i] = a;
			} else {
				a = d.alpha[i];   // already exchanged between the ranks
			}
			consider(i, a);
		}
	}
	block_argmin(best_v, best_i, sh);
	// block-wide eligible count
#pragma unroll
	for (int off = 16; off >= 1; off >>= 1) elig += __shfl_xor_sync(0xffffffffu, elig, off);
	__syncthreads();
	if ((tid & 31) == 0) sh.red_c[tid >> 5] = elig;
	__syncthreads();
	if (tid == 0) {
		long long c = 0;
#pragma unroll
		for (int w = 0; w < NWARP; ++w) c += sh.red_c[w];
		d.cand[part].val = best_v;
		d.cand[part].idx = best_i;
		d.cnt[part] = c;
	}
}

// Harris ratio test, second pass: among the eligible rows whose step max(x_b,0)/alpha does not exceed theta_max,
// the one with the LARGEST pivot element alpha (lowest index on ties) -> cand2[part] as (-alpha, index)
template <typename T>
__device__ void harris_phase2(const Dev<T>& d, Smem& sh, double theta_max, int part, int nparts) {
	const int tid = threadIdx.x;
	double best_v = CUDART_INF;
	long long best_i = LLONG_MAX;
	for (long long i = (long long)part * NT + tid; i < d.m; i += (long long)nparts * NT) {
		const T a = d.alpha[i];
		if (a > (T)d.pivot_tol && (double)(ratio_num(d.x_b[i], 2) / a) <= theta_max && cand_better(-(double)a, i, best_v, best_i)) {
			best_v = -(double)a;
			best_i = i;
		}
	}
	block_argmin(best_v, best_i, sh);
	if (tid == 0) { d.cand2[part].val = best_v; d.cand2[part].idx = best_i; }
}

// ---------------------------------------------------------------- phase: bookkeeping 1

// row_q = B^-1[q,:] (old), E_q from alpha (v4:331-332, 210-215) and the slice
// partials of  row_q.b  (v4:347)  and  c_b_new.E_q  (v4:354; c_b[q] already
// replaced by c[p], v4:340).
// SE: also the slice partials of alpha.alpha (gamma_p = 1 + |alpha|^2) and the pivot's alpha_q / leaving variable
template <typename T, bool SE = false>
__device__ void book1_phase(const Dev<T>& d, Smem& sh, long long p, long long q, int part, int nparts) {
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const T alpha_q = d.alpha[q];
	const T c_p = d.c[p];
	for (long long s = part; s < d.nslice; s += nparts) {
		const long long i = s * SLICE + tid;
		T t1 = T(0), t2 = T(0), t3 = T(0);
		if (i < d.m) {
			const T rq = d.B[q + i * d.ldb];
			const T al = d.alpha[i];
			const T eq = (i != q) ? (-al / alpha_q) : (T)(1.0 / (double)alpha_q - 1.0);
			d.row_q[i] = rq;
			d.E_q[i] = eq;
			T cb = d.c_b[i];
			if (i == q) {
				d.ctl->c_b_q = (double)cb; cb = c_p;
				if (SE) { d.ctl->alpha_q = (double)alpha_q; d.ctl->leaving = d.b_ixs[q]; }
			}
			t1 = fma_t(rq, d.b[i], T(0));
			t2 = fma_t(cb, eq, T(0));
			if (SE) t3 = fma_t(al, al, T(0));
		}
		t1 = warp_butterfly_sum(t1);
		t2 = warp_butterfly_sum(t2);
		if (SE) t3 = warp_butterfly_sum(t3);
		__syncthreads();
		if (lane == 0) { sh.dsum[0][warp] = (double)t1; sh.dsum[1][warp] = (double)t2; if (SE) sh.dsum[2][warp] = (double)t3; }
		__syncthreads();
		if (tid < (SE ? 3 : 2)) {
			T a = T(0);
#pragma unroll
			for (int w = 0; w < NWARP; ++w) a = a + (T)sh.dsum[tid][w];
			d.dpart[(long long)tid * d.nslice + s] = a;
		}
	}
}

// ---------------------------------------------------------------- phase: bookkeeping 2

// the two scalars of the linear updates: s_x = row_q.b (v4:347), s_y = c_b_new.E_q + (c_p - c_b_q) (v4:354-355);
// slice partials summed left to right (loads of 32 slices together).  Valid in every thread afterwards.
// SE: also gamma_p = 1 + alpha.alpha of the last pivot (steepest edge).
template <typename T, bool SE = false>
__device__ __forceinline__ void book2_scalars(const Dev<T>& d, Smem& sh, long long p, T& sx, T& sy, T* gp = nullptr) {
	const int tid = threadIdx.x;
	__syncthreads();
	if (tid < (SE ? 3 : 2)) {
		T a = T(0);
		const T* part = tid == 0 ? d.dpart0 : d.dpart + (long long)tid * d.nslice;
		for (int s0 = 0; s0 < d.nslice; s0 += 32) {
			T v[32];
#pragma unroll
			for (int u = 0; u < 32; ++u) v[u] = s0 + u < d.nslice ? __ldcg(part + s0 + u) : T(0);
#pragma unroll
			for (int u = 0; u < 32; ++u)
				if (s0 + u < d.nslice) a = a + v[u];
		}
		if (tid == 1) a += d.c[p] - (T)__ldcg(&d.ctl->c_b_q);
		if (tid == 2) a = T(1) + a;
		sh.bc_s[tid] = (double)a;
	}
	__syncthreads();
	sx = (T)sh.bc_s[0];
	sy = (T)sh.bc_s[1];
	if (SE && gp) *gp = (T)sh.bc_s[2];
}

// x_b += (row_q.b) E_q (v4:348);  y += ((c_b_new.E_q) + (c_p - c_b_q)) row_q (v4:355-356);
// c_b[q] = c[p], b_ixs[q] = p (v4:340-342)
template <typename T>
__device__ void book2_phase(const Dev<T>& d, Smem& sh, long long p, long long q, int part, int nparts) {
	const int tid = threadIdx.x;
	T sx, sy;
	book2_scalars<T>(d, sh, p, sx, sy);
	for (long long i = (long long)part * NT + tid; i < d.m; i += (long long)nparts * NT) {
		const T eq = d.E_q[i], rq = __ldcg(d.row_q + i);
		d.x_b[i] = fma_t(sx, eq, d.x_b[i]);
		d.y[i] = fma_t(sy, rq, d.y[i]);
		if (i == q) { d.c_b[i] = d.c[p]; d.b_ixs[i] = (int)p; }
	}
	fence_proxy_async_global();     // y is read by TMA (async proxy) in the next pricing phase
}

// The same updates as the PROLOGUE of the next pricing pass (d.fuse_book2: y fits in shared memory).  Every CTA
// builds the whole new y in shared memory (ysm, ld elements) from the old y and row_q — the pricing pass then
// reads y from there and never from L1/L2 — and applies its slice of the x_b / c_b / b_ixs updates in global
// memory.  The global y is NOT touched here (other CTAs may still be reading the old one): y_flush does it after
// the pricing barrier.  apply = false: no pivot pending, ysm = y.  Returns s_y for y_flush.
// SE (steepest edge): gp receives gamma_p; row_q and v are staged behind y while they fit (nstage = 1..3 vectors).
template <typename T, bool SE = false>
__device__ T book2_prologue(const Dev<T>& d, Smem& sh, T* ysm, bool apply, long long p, long long q, int part, int nparts,
		T* gp = nullptr, int nstage = 1) {
	using V = typename VecT<T>::V;
	constexpr int VN = VecT<T>::N;
	const int tid = threadIdx.x;
	T sx = T(0), sy = T(0);
	if (apply) {
		book2_scalars<T, SE>(d, sh, p, sx, sy, gp);
		for (long long i = (long long)part * NT + tid; i < d.m; i += (long long)nparts * NT) {
			d.x_b[i] = fma_t(sx, d.E_q[i], d.x_b[i]);
			if (i == q) { d.c_b[i] = d.c[p]; d.b_ixs[i] = (int)p; }
		}
	}
	for (long long i = (long long)tid * VN; i < d.ld; i += (long long)NT * VN) {
		V yv = __ldcg(reinterpret_cast<const V*>(d.y + i));
		if (apply) {
			const V rq = __ldcg(reinterpret_cast<const V*>(d.row_q + i));
#pragma unroll
			for (int v = 0; v < VN; ++v) Mem<T>::set(yv, v, fma_t(sy, Mem<T>::get(rq, v), Mem<T>::get(yv, v)));
		}
		*reinterpret_cast<V*>(ysm + i) = yv;
		if (SE && nstage > 1) *reinterpret_cast<V*>(ysm + d.ld + i) = __ldcg(reinterpret_cast<const V*>(d.row_q + i));
		if (SE && nstage > 2) *reinterpret_cast<V*>(ysm + 2 * d.ld + i) = __ldcg(reinterpret_cast<const V*>(d.vbt + i));
	}
	__syncthreads();
	return sy;
}

// global y += s_y row_q for this CTA's slice; legal once every CTA is past its pricing pass (nobody reads the old y)
template <typename T>
__device__ __forceinline__ void y_flush(const Dev<T>& d, T sy, int part, int nparts) {
	for (long long i = (long long)part * NT + threadIdx.x; i < d.m; i += (long long)nparts * NT)
		d.y[i] = fma_t(sy, __ldcg(d.row_q + i), d.y[i]);
}

// z = c_b . x_b in slice order (v4:365); single CTA
template <typename T>
__device__ double objective(const Dev<T>& d, Smem& sh) {
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	T z = T(0);
	for (long long s = 0; s < d.nslice; ++s) {
		const long long i = s * SLICE + tid;
		T t = i < d.m ? fma_t(d.c_b[i], d.x_b[i], T(0)) : T(0);
		t = warp_butterfly_sum(t);
		__syncthreads();
		if (lane == 0) sh.dsum[0][warp] = (double)t;
		__syncthreads();
		T a = T(0);
#pragma unroll
		for (int w = 0; w < NWARP; ++w) a = a + (T)sh.dsum[0][w];
		z = z + a;
	}
	return (double)z;
}

// ---------------------------------------------------------------- the persistent kernel

// The whole loop of v4:286-359 on the device.  Every CTA takes the same
// branches because every decision is recomputed from the same global data.
// Three grid barriers per pivot:
//   price (+ prologue: x_b / y / c_b / b_ixs of the previous pivot when d.fuse_book2)   | B1 -> p, optimality
//   update + FTRAN (+ ratio test of every row group as it completes)                     | B2 -> q, unboundedness
//   book1 (row_q, E_q, dot partials)                                                     | B3
// Without fuse_book2 (y does not fit in shared memory, or the TMA-ring pricing path reads it from global memory)
// book2 stays a phase of its own with a fourth barrier.
// SE: steepest-edge pricing (price_phase_se), one more read of B^-1 per pivot for v = B^-T alpha (btran_phase, in
// the same barrier interval as book1).
template <typename T, int WC, bool SE = false>
__global__ void __launch_bounds__(NT, MIN_CTAS) simplex_persistent(Dev<T> d) {
	__shared__ Smem sh;
	extern __shared__ __align__(128) unsigned char ringbuf[];
	Ring rcons, rprod;
	ring_init(sh, rcons, rprod, d.price_nc);
	Ctl* ctl = d.ctl;
	const int G = gridDim.x, me = blockIdx.x;
	unsigned long long epoch = 0;

	long long it = ctl->iter, pivots = ctl->pivots;
	const long long it_end = ctl->it_end;
	int pending = ctl->pending;
	int status = 0, done = 0, aborted = 0;
	long long p = ctl->p, q = ctl->q;
	double min_e = ctl->min_e;
	const bool fuse = d.fuse_book2 != 0;
	T* ysm = reinterpret_cast<T*>(ringbuf);
	bool pend2 = false;                 // book2 of the last pivot still to be applied (fuse only; never across launches)
	T sy_keep = T(0);
	bool pendg = SE && ctl->se_pending != 0;   // steepest edge: weight recurrence of the last pivot still to be applied
	// steepest edge: how many of {y, row_q, v} fit in the staging area (fuse: at least y does)
	const int nstage = SE && fuse ? (int)((long long)DYN_SMEM_BYTES / (d.ld * (long long)sizeof(T)) < 3 ? (long long)DYN_SMEM_BYTES / (d.ld * (long long)sizeof(T)) : 3) : 0;

	const long long it0 = it;
	while (it < it_end) {
		// ---- pricing + entering column (v4:288-302)
		stamp(d, it - it0, 0);
		if (SE) {
			SeUpd u;
			u.on = pendg;
			u.p = p;
			u.leaving = pendg ? __ldcg(&ctl->leaving) : -1;
			u.alpha_q = pendg ? __ldcg(&ctl->alpha_q) : 1.0;
			T gp = T(0);
			if (fuse) {
				sy_keep = book2_prologue<T, true>(d, sh, ysm, pend2, p, q, me, G, &gp, nstage);
				if (pendg && !pend2) { T sx_, sy_; book2_scalars<T, true>(d, sh, p, sx_, sy_, &gp); }
			} else if (pendg) { T sx_, sy_; book2_scalars<T, true>(d, sh, p, sx_, sy_, &gp); }
			u.gamma_p = (double)gp;
			const T* const vec[3] = {fuse ? ysm : d.y, nstage > 1 ? ysm + d.ld : d.row_q, nstage > 2 ? ysm + 2 * d.ld : d.vbt};
			price_phase_se<T>(d, sh, vec, u, me, G);
		} else if (fuse) {
			sy_keep = book2_prologue<T>(d, sh, ysm, pend2, p, q, me, G);
			price_phase_direct<T>(d, sh, ysm, me, G);
		} else if (d.price_direct) price_phase_direct<T>(d, sh, nullptr, me, G);
		else                       price_phase<T>(d, sh, ringbuf, rcons, rprod, me, G);
		stamp(d, it - it0, 1);
		if (me == 0 && threadIdx.x == 0) ctl->abort_latched = *(volatile int*)&ctl->abort_req;   // before CTA 0 arrives: one value for all
		grid_barrier(ctl, epoch, G);
		if (me == 0 && threadIdx.x == 0) { ctl->price_ctr = 0; if (SE) ctl->btran_ctr = 0; }   // every CTA is past pricing; next use is barriers away
		reduce_cands(d.cand, G, min_e, p, sh);
		if (SE) {                                                 // optimality from min e (v4:299), the pivot from the weighted candidate
			double sc; long long pse;
			reduce_cands(d.cand2, G, sc, pse, sh);
			if (pse != LLONG_MAX) p = pse;
			pendg = false;                                         // the recurrence has been applied by this pass
		}
		if (pend2) { y_flush<T>(d, sy_keep, me, G); pend2 = false; }   // read again two barriers from here at the earliest
		stamp(d, it - it0, 2);
		if (__ldcg(&ctl->abort_latched)) { aborted = 1; break; }
		if (min_e >= -d.eps) { status = 1; done = 1; ++it; break; }

		// ---- pending rank-1 update fused with the FTRAN of column p and the ratio test (v4:333, 307-308, 311-325)
		const T* acol = p < d.ns ? d.A + p * d.ld : nullptr;
		double th;
		long long elig;
		if (d.fuse_ratio) {
			if (pending) update_ftran_phase<T, WC, true, true, true>(d, sh, ringbuf, acol, p - d.ns, pivots & 1, me, G);
			else         update_ftran_phase<T, WC, false, true, true>(d, sh, ringbuf, acol, p - d.ns, pivots & 1, me, G);
			stamp(d, it - it0, 3);
			grid_barrier(ctl, epoch, G);
			if (me == 0 && threadIdx.x == 0) ctl->upd_ctr = 0;
			stamp(d, it - it0, 4);
			reduce_cands(d.rcand, d.ngrp, th, q, sh);
			elig = reduce_counts(d.rcnt, d.ngrp, sh);
		} else {
			if (pending) update_ftran_phase<T, WC, true, true, false>(d, sh, ringbuf, acol, p - d.ns, pivots & 1, me, G);
			else         update_ftran_phase<T, WC, false, true, false>(d, sh, ringbuf, acol, p - d.ns, pivots & 1, me, G);
			stamp(d, it - it0, 3);
			grid_barrier(ctl, epoch, G);
			if (me == 0 && threadIdx.x == 0) ctl->upd_ctr = 0;
			ratio_phase<T, true>(d, sh, me, G, reinterpret_cast<T*>(ringbuf));
			grid_barrier(ctl, epoch, G);
			stamp(d, it - it0, 4);
			reduce_cands(d.cand, G, th, q, sh);
			elig = reduce_counts(d.cnt, G, sh);
			if (d.ratio_mode == 2 && elig > 0) {        // Harris: th is theta_max, now pick the largest pivot inside it
				harris_phase2<T>(d, sh, th, me, G);
				grid_barrier(ctl, epoch, G);
				double na;
				reduce_cands(d.cand2, G, na, q, sh);
			}
		}
		pending = 0;
		if (elig == 0) { status = 2; done = 1; ++it; break; }
		stamp(d, it - it0, 5);

		// ---- pivot (v4:331-356)
		book1_phase<T, SE>(d, sh, p, q, me, G);
		if (SE) { btran_phase<T>(d, sh, d.alpha, me, G); pendg = true; }
		stamp(d, it - it0, 6);
		grid_barrier(ctl, epoch, G);
		stamp(d, it - it0, 7);
		if (me == 0 && threadIdx.x == 0 && pivots < d.trace_cap) d.trace[pivots] = make_int2((int)p, (int)q);
		if (fuse && it + 1 < it_end) {
			pend2 = true;               // rides in the prologue of the next pricing pass
		} else {
			book2_phase<T>(d, sh, p, q, me, G);
			stamp(d, it - it0, 8);
			grid_barrier(ctl, epoch, G);
			stamp(d, it - it0, 9);
		}
		pending = 1;
		++pivots;
		++it;
	}

	if (me == 0) {
		const double z = objective<T>(d, sh);
		if (threadIdx.x == 0) {
			ctl->iter = it; ctl->pivots = pivots; ctl->pending = pending;
			ctl->status = status; ctl->done = done; ctl->aborted = aborted;
			ctl->p = p; ctl->q = q; ctl->min_e = min_e; ctl->z = z;
			if (SE) ctl->se_pending = pendg ? 1 : 0;
		}
	}
}

// ---------------------------------------------------------------- dual simplex (options.algorithm = 1)
//
// For LPs whose slack basis is dual feasible (every e_j = y.a_j - c_j >= 0, e.g. c <= 0) but primal infeasible
// (some b_i < 0).  One iteration:
//   r = argmin (x_b_i, i)                                     leaving row
//   e_j = y.a_j - c_j and, when x_b_r < -eps, alpha_rj = rho.a_j from the same bytes of A, rho = row r of B^-1
//       after the pending rank-1 update (rho_j = fma(E_q[r], row_q[j], B[r,j]), the update pass's own fma)
//   min e < -eps -> NOT_DUAL_FEASIBLE;  x_b_r >= -eps -> OPTIMUM
//   p = argmin (max(e_j, 0) / -alpha_rj, j) over the NONBASIC columns with alpha_rj < -pivot_tol; none -> INFEASIBLE
//   basis change with q = r: the primal pivot's update + FTRAN, chunk sums of alpha, book1 and book2, unchanged.
// The nonbasic mask is needed: with product-form rounding a basic column can get alpha_rj ~ -1e-17 and ratio 0.
// Sums keep the primal kernel's associations (file header), both argmins are lexicographic.
//
// Phases and grid barriers per pivot (the primal loop has four; the two streaming passes are the same bytes):
//   reduce the leaving-row candidates -> r;  rho gather (only when x_b_r < -eps)              | D1
//   price_phase_dual: e_j, alpha_rj, min-e and ratio candidates per CTA                      | D2 -> statuses, p
//   update + FTRAN of a_p                                                                     | D3
//   alpha = chunk sums                                                                        | D4
//   book1 (row_q, E_q, dot partials)                                                          | D5
//   book2 (x_b, y, c_b, b_ixs), nonbasic mask, leaving-row candidates of the new x_b          | D6
template <typename T>
struct DualDev {
	unsigned char* nb;        // n flags: 1 = column j is nonbasic (upload / reset: the first n - m columns)
	T* rho;                   // ld: row r of B^-1 (padding rows zero)
	Cand* lcand;              // one per CTA: (min x_b, row) over the CTA's rows
};

// (min x_b_i, i) over rows part*NT + tid, stride nparts*NT: the rows book2_phase updates in this thread, so it
// runs right behind it without a barrier
template <typename T>
__device__ void dual_leave_cands(const Dev<T>& d, const DualDev<T>& dd, Smem& sh, int part, int nparts) {
	double best_v = CUDART_INF;
	long long best_i = LLONG_MAX;
	for (long long i = (long long)part * NT + threadIdx.x; i < d.m; i += (long long)nparts * NT) {
		const double v = (double)d.x_b[i];
		if (cand_better(v, i, best_v, best_i)) { best_v = v; best_i = i; }
	}
	block_argmin(best_v, best_i, sh);
	if (threadIdx.x == 0) { dd.lcand[part].val = best_v; dd.lcand[part].idx = best_i; }
}

// rho = row r of B^-1 with the pending rank-1 update applied on the fly (bit-identical to a flushed B^-1)
template <typename T>
__device__ void dual_rho_phase(const Dev<T>& d, const DualDev<T>& dd, long long r, bool pending, int part, int nparts) {
	const T er = pending ? d.E_q[r] : T(0);
	for (long long j = (long long)part * NT + threadIdx.x; j < d.m; j += (long long)nparts * NT) {
		const T bj = d.B[r + j * d.ldb];
		dd.rho[j] = pending ? fma_t(er, __ldcg(d.row_q + j), bj) : bj;
	}
}

// e_j = y.a_j - c_j (+ alpha_rj = rho.a_j when want_alpha) for all n columns, one read of A; per CTA the
// (min e, index) candidate -> cand[part] and the dual ratio candidate (max(e,0) / -alpha, index) over the nonbasic
// columns with alpha < -pivot_tol -> cand2[part]
template <typename T>
__device__ void price_phase_dual(const Dev<T>& d, const DualDev<T>& dd, Smem& sh, bool want_alpha, int part, int nparts) {
	const int tid = threadIdx.x;
	double best_v = CUDART_INF, rat_v = CUDART_INF;
	long long best_i = LLONG_MAX, rat_i = LLONG_MAX;
	const T tol = (T)d.pivot_tol;
	auto consider = [&](long long j, T e, T a) {
		if (cand_better((double)e, j, best_v, best_i)) { best_v = (double)e; best_i = j; }
		if (want_alpha && dd.nb[j] && a < -tol) {
			const double rt = (double)((e > T(0) ? e : T(0)) / -a);
			if (cand_better(rt, j, rat_v, rat_i)) { rat_v = rt; rat_i = j; }
		}
	};

	const T* const vec[3] = {d.y, dd.rho, nullptr};
	const long long c1 = d.nsl;
	const long long nq = c1 / PRICE_NC;
	const long long nitems = nq + (c1 - nq * PRICE_NC);
	int buf = 0;
	for (long long g = part; g < nitems; buf ^= 1) {
		if (tid == 0) sh.tk = (long long)nparts + atomicAdd(&d.ctl->price_ctr, 1u);
		const bool quad = g < nq;
		const long long col = quad ? g * PRICE_NC : nq * PRICE_NC + (g - nq);
		const T* base = d.A + col * d.ld;
		if (want_alpha) {
			if (quad) column_dots<T, PRICE_NC, 2, 2, false>(base, d.ld, d.ld, vec, sh, buf);
			else      column_dots<T, 1, 8, 2, false>(base, d.ld, d.ld, vec, sh, buf);
		} else {
			if (quad) column_dots<T, PRICE_NC, 4, 1, false>(base, d.ld, d.ld, vec, sh, buf);
			else      column_dots<T, 1, 16, 1, false>(base, d.ld, d.ld, vec, sh, buf);
		}
		__syncthreads();
		g = sh.tk;
		if (tid < (quad ? PRICE_NC : 1)) {
			const long long j = d.col0 + col + tid;
			const int nv = want_alpha ? 2 : 1;
			const T e = warp_sums<T>(sh, buf, tid * nv) - d.c[j];
			const T a = want_alpha ? warp_sums<T>(sh, buf, tid * nv + 1) : T(0);
			consider(j, e, a);
		}
		__syncthreads();
	}
	for (long long k = d.k0 + (long long)part * NT + tid; k < d.k1; k += (long long)nparts * NT)   // unit (slack) columns
		consider(d.ns + k, d.y[k] - d.c[d.ns + k], want_alpha ? dd.rho[k] : T(0));

	block_argmin(best_v, best_i, sh);
	block_argmin(rat_v, rat_i, sh);
	if (tid == 0) {
		d.cand[part].val = best_v; d.cand[part].idx = best_i;
		d.cand2[part].val = rat_v; d.cand2[part].idx = rat_i;
	}
}

// alpha_i = the chunk partials of row i summed left to right (ratio_phase<T, true> without its ratio test)
template <typename T>
__device__ void dual_alpha_phase(const Dev<T>& d, int part, int nparts) {
	for (long long i = (long long)part * NT + threadIdx.x; i < d.m; i += (long long)nparts * NT)
		d.alpha[i] = sum_chunk_partials(d.alpha_part + i, d.ldb, d.nchunk);
}

template <typename T, int WC>
__global__ void __launch_bounds__(NT, MIN_CTAS) simplex_dual(Dev<T> d, DualDev<T> dd) {
	__shared__ Smem sh;
	extern __shared__ __align__(128) unsigned char dyn[];   // update+FTRAN staging (UF_SMEM_BYTES)
	Ctl* ctl = d.ctl;
	const int G = gridDim.x, me = blockIdx.x;
	unsigned long long epoch = 0;

	long long it = ctl->iter, pivots = ctl->pivots;
	const long long it_end = ctl->it_end;
	int pending = ctl->pending;
	int status = 0, done = 0, aborted = 0;
	long long p = ctl->p, q = ctl->q;
	double min_e = ctl->min_e;
	const long long it0 = it;

	dual_leave_cands<T>(d, dd, sh, me, G);     // later ones ride behind book2
	grid_barrier(ctl, epoch, G);
	while (it < it_end) {
		// ---- leaving row, rho
		stamp(d, it - it0, 0);
		double xr;
		long long r;
		reduce_cands(dd.lcand, G, xr, r, sh);
		const bool want_alpha = xr < -d.eps;
		if (want_alpha) {
			dual_rho_phase<T>(d, dd, r, pending != 0, me, G);
			grid_barrier(ctl, epoch, G);
		}
		// ---- column pass: reduced costs, row r of B^-1 A, both candidates
		stamp(d, it - it0, 1);
		price_phase_dual<T>(d, dd, sh, want_alpha, me, G);
		stamp(d, it - it0, 2);
		if (me == 0 && threadIdx.x == 0) ctl->abort_latched = *(volatile int*)&ctl->abort_req;
		grid_barrier(ctl, epoch, G);
		if (me == 0 && threadIdx.x == 0) ctl->price_ctr = 0;
		stamp(d, it - it0, 3);
		long long pmin, pe;
		double rt;
		reduce_cands(d.cand, G, min_e, pmin, sh);
		reduce_cands(d.cand2, G, rt, pe, sh);
		if (__ldcg(&ctl->abort_latched)) { aborted = 1; break; }
		if (min_e < -d.eps) { status = 5; done = 1; ++it; break; }   // B200LP_STATUS_NOT_DUAL_FEASIBLE
		if (!want_alpha) { status = 1; done = 1; ++it; break; }      // x_b >= -eps everywhere: optimum
		if (pe == LLONG_MAX) { status = 4; done = 1; ++it; break; }  // row r is a Farkas certificate: infeasible
		p = pe;
		q = r;

		// ---- basis change with the primal pivot's phases
		const T* acol = p < d.ns ? d.A + p * d.ld : nullptr;
		if (pending) update_ftran_phase<T, WC, true, true, false>(d, sh, dyn, acol, p - d.ns, pivots & 1, me, G);
		else         update_ftran_phase<T, WC, false, true, false>(d, sh, dyn, acol, p - d.ns, pivots & 1, me, G);
		pending = 0;
		stamp(d, it - it0, 4);
		grid_barrier(ctl, epoch, G);
		if (me == 0 && threadIdx.x == 0) ctl->upd_ctr = 0;
		dual_alpha_phase<T>(d, me, G);
		const long long leaving = d.b_ixs[q];      // b_ixs[q] is rewritten by book2, barriers from here
		stamp(d, it - it0, 5);
		grid_barrier(ctl, epoch, G);
		book1_phase<T>(d, sh, p, q, me, G);
		stamp(d, it - it0, 6);
		grid_barrier(ctl, epoch, G);
		if (me == 0 && threadIdx.x == 0) {
			if (pivots < d.trace_cap) d.trace[pivots] = make_int2((int)p, (int)q);
			dd.nb[p] = 0;
			dd.nb[leaving] = 1;
		}
		stamp(d, it - it0, 7);
		book2_phase<T>(d, sh, p, q, me, G);
		dual_leave_cands<T>(d, dd, sh, me, G);
		stamp(d, it - it0, 8);
		grid_barrier(ctl, epoch, G);
		pending = 1;
		++pivots;
		++it;
	}

	if (me == 0) {
		const double z = objective<T>(d, sh);
		if (threadIdx.x == 0) {
			ctl->iter = it; ctl->pivots = pivots; ctl->pending = pending;
			ctl->status = status; ctl->done = done; ctl->aborted = aborted;
			ctl->p = p; ctl->q = q; ctl->min_e = min_e; ctl->z = z;
		}
	}
}

// ---------------------------------------------------------------- tiny LPs: everything in shared memory
//
// Klee-Minty (m = 20, 2^20 - 1 pivots) and friends: the matrices fit in one SM's shared memory and a pivot is
// pure latency.  One CTA, state loaded once, ~10 __syncthreads per pivot, no global round trip inside the loop
// (the general kernel with a 1-CTA grid spends ~19 us per pivot on ~20 dependent L2 round trips).
// Condition (host): ld == one warp-wide vector row (m <= 64 doubles / 128 floats) and A, B^-1 fit.
// Every sum is associated exactly as in the general kernel (see the file header), so results are bit-identical:
//   pricing dot ... the column's 32 vectors sit in warp 0's slots; the other 7 warp sums are +0
//   FTRAN ......... 8 sub-blocks of 32 columns, one fma chain each (empty ones stay +0), the same pairwise tree
//   O(m) dots ..... a single 256-element slice
// State is read from and written back to the same global buffers, so windows, downloads and the phase entry
// points see no difference.
template <typename T>
struct TinyLayout {
	static constexpr int VN = VecT<T>::N;
	static constexpr int LD = 32 * VN;
	// element offsets into the dynamic shared memory (all multiples of LD, hence 16-byte aligned)
	long long A, B, y, x_b, c_b, alpha, E_q, row_q, b, part, c, end;
	int* b_ixs;
	__host__ __device__ TinyLayout(long long m, long long n, long long ns) {
		long long o = 0;
		A = o; o += LD * ns;
		B = o; o += LD * m;
		y = o; o += LD; x_b = o; o += LD; c_b = o; o += LD; alpha = o; o += LD;
		E_q = o; o += LD; row_q = o; o += LD; b = o; o += LD;
		part = o; o += 8 * LD;
		c = o; o += (n + 3) / 4 * 4;
		end = o;
		b_ixs = nullptr;
	}
	__host__ __device__ size_t bytes(long long m) const { return (size_t)end * sizeof(T) + (size_t)m * sizeof(int) + 16; }
};

// Shared-memory pointers of one tiny LP (TinyLayout) and its sizes.
template <typename T>
struct TinyLP {
	T *A, *B, *y, *x_b, *c_b, *alpha, *E_q, *row_q, *b, *part, *c;
	int* b_ixs;
	int m, n, ns;
	__device__ __forceinline__ TinyLP(T* S, const TinyLayout<T>& L, int m_, int n_, int ns_)
		: A(S + L.A), B(S + L.B), y(S + L.y), x_b(S + L.x_b), c_b(S + L.c_b), alpha(S + L.alpha), E_q(S + L.E_q),
		  row_q(S + L.row_q), b(S + L.b), part(S + L.part), c(S + L.c), b_ixs(reinterpret_cast<int*>(S + L.end)),
		  m(m_), n(n_), ns(ns_) {}
};

// The pricing dot of the tiny kernels: the column's 32 vectors are the lanes of one warp (av, yv: this lane's
// vector of the column and of y), the association of the general kernel's pricing dot.  Valid in every lane.
template <typename T>
__device__ __forceinline__ T tiny_dot(const typename VecT<T>::V& av, const typename VecT<T>::V& yv) {
	using M = Mem<T>;
	T s = fma_t(M::get(av, 0), M::get(yv, 0), T(0));
#pragma unroll
	for (int v = 1; v < VecT<T>::N; ++v) s = s + fma_t(M::get(av, v), M::get(yv, v), T(0));
	s = warp_butterfly_sum(s);
	return s + T(0);                               // + the seven empty warp sums of the general kernel
}

// Pending rank-1 update fused with the FTRAN of column p (v4:333 + v4:307-308): alpha = B^-1 a_p after
// B^-1 += E_q (x) row_q when `pending`.  Shared by the primal and the dual loop; ends with a barrier.
template <typename T>
__device__ __forceinline__ void tiny_update_ftran(const TinyLP<T>& s, long long p, int pending) {
	using V = typename VecT<T>::V;
	using M = Mem<T>;
	constexpr int VN = VecT<T>::N;
	constexpr int LD = 32 * VN;
	T *sA = s.A, *sB = s.B, *sal = s.alpha, *sE = s.E_q, *srq = s.row_q, *spart = s.part;
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const int m = s.m, ns = s.ns;
	{
		const int j0 = warp * SUBW;                // this warp's 32-column sub-block
		T acc[VN];
		V Ev = *reinterpret_cast<const V*>(sE + lane * VN);
#pragma unroll
		for (int v = 0; v < VN; ++v) acc[v] = T(0);
		const int jend = j0 + SUBW < m ? j0 + SUBW : m;
		for (int j = j0; j < jend; ++j) {
			V x = *reinterpret_cast<const V*>(sB + (long long)j * LD + lane * VN);
			const T a = p < ns ? sA[(long long)p * LD + j] : (j == (int)(p - ns) ? T(1) : T(0));
			if (pending) {
				const T r = srq[j];
#pragma unroll
				for (int v = 0; v < VN; ++v) M::set(x, v, fma_t(M::get(Ev, v), r, M::get(x, v)));
				*reinterpret_cast<V*>(sB + (long long)j * LD + lane * VN) = x;
			}
#pragma unroll
			for (int v = 0; v < VN; ++v) acc[v] = fma_t(M::get(x, v), a, acc[v]);
		}
#pragma unroll
		for (int v = 0; v < VN; ++v) spart[(warp * 32 + lane) * VN + v] = acc[v];
	}
	__syncthreads();
	if (warp == 0) {
		T t[NWARP][VN];
#pragma unroll
		for (int c = 0; c < NWARP; ++c)
#pragma unroll
			for (int v = 0; v < VN; ++v) t[c][v] = spart[(c * 32 + lane) * VN + v];
#pragma unroll
		for (int w = 1; w < NWARP; w <<= 1)
#pragma unroll
			for (int c = 0; c + w < NWARP; c += 2 * w)
#pragma unroll
				for (int v = 0; v < VN; ++v) t[c][v] = t[c][v] + t[c + w][v];
#pragma unroll
		for (int v = 0; v < VN; ++v) sal[lane * VN + v] = t[0][v];
	}
	__syncthreads();
}

// The basis change on (p, q) (v4:331-356: book1 and book2 of the general kernel, one 256-element slice): row_q, E_q,
// x_b, y, c_b[q], b_ixs[q] and the trace entry of pivot `pivots`.  Needs alpha = B^-1 a_p; leaves the rank-1 update
// pending.  Shared by the primal and the dual loop; ends with a barrier.
template <typename T>
__device__ __forceinline__ void tiny_pivot(const TinyLP<T>& s, Smem& sh, long long p, long long q, int2* trace,
		long long trace_cap, long long pivots) {
	constexpr int LD = 32 * VecT<T>::N;
	T *sB = s.B, *sy = s.y, *sx = s.x_b, *scb = s.c_b, *sal = s.alpha, *sE = s.E_q, *srq = s.row_q, *sb = s.b, *sc = s.c;
	int* sbix = s.b_ixs;
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const int m = s.m;
	const T alpha_q = sal[q];
	const T c_p = sc[p];
	T t1 = T(0), t2 = T(0), eq = T(0), rq = T(0);
	const int i = tid;
	if (i < m) {
		rq = sB[(long long)i * LD + q];
		eq = (i != q) ? (-sal[i] / alpha_q) : (T)(1.0 / (double)alpha_q - 1.0);
		T cb = scb[i];
		if (i == q) { sh.bc_v = (double)cb; cb = c_p; }
		t1 = fma_t(rq, sb[i], T(0));
		t2 = fma_t(cb, eq, T(0));
	}
	t1 = warp_butterfly_sum(t1);
	t2 = warp_butterfly_sum(t2);
	__syncthreads();
	if (lane == 0) { sh.dsum[0][warp] = (double)t1; sh.dsum[1][warp] = (double)t2; }
	if (i < LD) { srq[i] = i < m ? rq : T(0); sE[i] = i < m ? eq : T(0); }
	__syncthreads();
	T sxv = T(0), syv = T(0);
#pragma unroll
	for (int w = 0; w < NWARP; ++w) { sxv = sxv + (T)sh.dsum[0][w]; syv = syv + (T)sh.dsum[1][w]; }
	sxv = T(0) + sxv;                              // book2 of the general kernel starts its slice sum from 0
	syv = T(0) + syv;
	syv += c_p - (T)sh.bc_v;
	if (i < m) {
		sx[i] = fma_t(sxv, eq, sx[i]);
		sy[i] = fma_t(syv, rq, sy[i]);
		if (i == q) { scb[i] = c_p; sbix[i] = (int)p; }
	}
	if (tid == 0 && pivots < trace_cap) trace[pivots] = make_int2((int)p, (int)q);
	__syncthreads();
}

// The pivot loop of the tiny kernels (simplex_tiny, simplex_tiny_batch): iterations [it, it_end) on the LP in
// shared memory, the scalar state in registers of every thread.  Leaves after the last iteration or at
// optimum / unbounded (status, done set, the final iteration counted like the general kernel does).
template <typename T>
__device__ __forceinline__ void tiny_pivots(const TinyLP<T>& s, Smem& sh, double eps, double pivot_tol, int ratio_mode,
		int2* trace, long long trace_cap, long long& it, const long long it_end, long long& pivots, int& pending,
		int& status, int& done, long long& p, long long& q, double& min_e) {
	using V = typename VecT<T>::V;
	constexpr int VN = VecT<T>::N;
	constexpr int LD = 32 * VN;
	T *sA = s.A, *sy = s.y, *sx = s.x_b, *sal = s.alpha, *sc = s.c;
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const int m = s.m, n = s.n, ns = s.ns;
	while (it < it_end) {
		// ---- pricing (v4:288-302): warp w takes columns w, w+8, ...; the column's 32 vectors are this warp's lanes
		double best_v = CUDART_INF;
		long long best_i = LLONG_MAX;
		const V yv = *reinterpret_cast<const V*>(sy + lane * VN);
		for (int col = warp; col < ns; col += NWARP) {
			const V av = *reinterpret_cast<const V*>(sA + (long long)col * LD + lane * VN);
			const double e = (double)(tiny_dot<T>(av, yv) - sc[col]);
			if (lane == 0 && cand_better(e, col, best_v, best_i)) { best_v = e; best_i = col; }
		}
		for (int k = tid; k < n - ns; k += NT) {       // unit (slack) columns
			const double e = (double)(sy[k] - sc[ns + k]);
			if (cand_better(e, ns + k, best_v, best_i)) { best_v = e; best_i = ns + k; }
		}
		block_argmin(best_v, best_i, sh);
		min_e = best_v;
		p = best_i;
		if (min_e >= -eps) { status = 1; done = 1; ++it; break; }

		tiny_update_ftran(s, p, pending);
		pending = 0;

		// ---- ratio test (v4:311-325)
		best_v = CUDART_INF;
		best_i = LLONG_MAX;
		long long elig = 0;
		for (int i = tid; i < m; i += NT) {
			const T a = sal[i];
			if (a > (T)pivot_tol) {
				++elig;
				const double th = (double)(ratio_num(sx[i], ratio_mode) / a);
				if (cand_better(th, i, best_v, best_i)) { best_v = th; best_i = i; }
			}
		}
		block_argmin(best_v, best_i, sh);
		q = best_i;
#pragma unroll
		for (int off = 16; off >= 1; off >>= 1) elig += __shfl_xor_sync(0xffffffffu, elig, off);
		__syncthreads();
		if (lane == 0) sh.red_c[warp] = elig;
		__syncthreads();
		elig = 0;
#pragma unroll
		for (int w = 0; w < NWARP; ++w) elig += sh.red_c[w];
		if (elig == 0) { status = 2; done = 1; ++it; break; }

		tiny_pivot(s, sh, p, q, trace, trace_cap, pivots);
		pending = 1;
		++pivots;
		++it;
	}
}

// The dual loop of the tiny batch kernel (simplex_tiny_batch_dual): simplex_dual's iteration (see above it) on one LP
// in shared memory, with the same numbers in the same order:
//   r = argmin (x_b_i, i) as double;  rho = row r of B^-1 after the pending update (dual_rho_phase's fma), held in
//   alpha, which is dead until this iteration's FTRAN;  e_j and alpha_rj with the pricing dot (tiny_dot), unit
//   columns y_k - c_j and rho_k (price_phase_dual);  the statuses in simplex_dual's order;  the pivot on (p, q = r)
//   through the primal loop's own update+FTRAN and pivot blocks.  nb: the nonbasic mask (n bytes).
template <typename T>
__device__ __forceinline__ void tiny_dual_pivots(const TinyLP<T>& s, unsigned char* nb, Smem& sh, double eps,
		double pivot_tol, int2* trace, long long trace_cap, long long& it, const long long it_end, long long& pivots,
		int& pending, int& status, int& done, long long& p, long long& q, double& min_e) {
	using V = typename VecT<T>::V;
	constexpr int VN = VecT<T>::N;
	constexpr int LD = 32 * VN;
	T *sA = s.A, *sB = s.B, *sy = s.y, *sx = s.x_b, *rho = s.alpha, *sc = s.c;
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const int m = s.m, n = s.n, ns = s.ns;
	const T tol = (T)pivot_tol;
	while (it < it_end) {
		// ---- leaving row, rho
		double xr = CUDART_INF;
		long long r = LLONG_MAX;
		for (int i = tid; i < m; i += NT)
			if (cand_better((double)sx[i], i, xr, r)) { xr = (double)sx[i]; r = i; }
		block_argmin(xr, r, sh);
		const bool want_alpha = xr < -eps;
		if (want_alpha) {
			if (tid < LD) {
				const T bj = tid < m ? sB[r + (long long)tid * LD] : T(0);    // padding rows +0, as in DualDev::rho
				rho[tid] = pending && tid < m ? fma_t(s.E_q[r], s.row_q[tid], bj) : bj;
			}
			__syncthreads();
		}

		// ---- column pass: reduced costs, row r of B^-1 A, both candidates
		double best_v = CUDART_INF, rat_v = CUDART_INF;
		long long best_i = LLONG_MAX, rat_i = LLONG_MAX;
		auto consider = [&](int j, T e, T a) {
			if (cand_better((double)e, j, best_v, best_i)) { best_v = (double)e; best_i = j; }
			if (want_alpha && nb[j] && a < -tol) {
				const double rt = (double)((e > T(0) ? e : T(0)) / -a);
				if (cand_better(rt, j, rat_v, rat_i)) { rat_v = rt; rat_i = j; }
			}
		};
		const V yv = *reinterpret_cast<const V*>(sy + lane * VN);
		const V rv = *reinterpret_cast<const V*>(rho + lane * VN);
		for (int col = warp; col < ns; col += NWARP) {
			const V av = *reinterpret_cast<const V*>(sA + (long long)col * LD + lane * VN);
			const T e = tiny_dot<T>(av, yv) - sc[col];
			const T a = want_alpha ? tiny_dot<T>(av, rv) : T(0);
			if (lane == 0) consider(col, e, a);
		}
		for (int k = tid; k < n - ns; k += NT)          // unit (slack) columns
			consider(ns + k, sy[k] - sc[ns + k], want_alpha ? rho[k] : T(0));
		block_argmin(best_v, best_i, sh);
		block_argmin(rat_v, rat_i, sh);
		min_e = best_v;
		if (min_e < -eps) { status = 5; done = 1; ++it; break; }        // B200LP_STATUS_NOT_DUAL_FEASIBLE
		if (!want_alpha) { status = 1; done = 1; ++it; break; }         // x_b >= -eps everywhere: optimum
		if (rat_i == LLONG_MAX) { status = 4; done = 1; ++it; break; }  // row r is a Farkas certificate: infeasible
		p = rat_i;
		q = r;

		// ---- basis change with the primal loop's blocks
		if (tid == 0) { nb[p] = 0; nb[s.b_ixs[q]] = 1; }   // b_ixs[q] before tiny_pivot rewrites it
		tiny_update_ftran(s, p, pending);
		pending = 0;
		tiny_pivot(s, sh, p, q, trace, trace_cap, pivots);
		pending = 1;
		++pivots;
		++it;
	}
}

// z = c_b . x_b in slice order (v4:365); the sum is valid in thread 0
template <typename T>
__device__ __forceinline__ T tiny_objective(const T* scb, const T* sx, int m, Smem& sh) {
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	T t = tid < m ? fma_t(scb[tid], sx[tid], T(0)) : T(0);
	t = warp_butterfly_sum(t);
	__syncthreads();
	if (lane == 0) sh.dsum[0][warp] = (double)t;
	__syncthreads();
	T a = T(0);
	if (tid == 0) {
#pragma unroll
		for (int w = 0; w < NWARP; ++w) a = a + (T)sh.dsum[0][w];
	}
	return T(0) + a;
}

template <typename T>
__global__ void __launch_bounds__(NT, 1) simplex_tiny(Dev<T> d) {
	constexpr int LD = TinyLayout<T>::LD;
	__shared__ Smem sh;
	extern __shared__ __align__(128) unsigned char dynraw[];
	T* S = reinterpret_cast<T*>(dynraw);
	const TinyLayout<T> L(d.m, d.n, d.ns);
	const TinyLP<T> s(S, L, (int)d.m, (int)d.n, (int)d.ns);
	T *sA = s.A, *sB = s.B, *sy = s.y, *sx = s.x_b, *scb = s.c_b, *sal = s.alpha, *sE = s.E_q, *srq = s.row_q, *sb = s.b,
	  *sc = s.c;
	int* sbix = s.b_ixs;
	const int tid = threadIdx.x;
	const int m = (int)d.m, n = (int)d.n, ns = (int)d.ns;
	Ctl* ctl = d.ctl;

	// ---- state in
	for (long long e = tid; e < (long long)LD * ns; e += NT) sA[e] = d.A[e];
	for (long long e = tid; e < (long long)LD * m; e += NT) sB[e] = d.B[e];
	for (int i = tid; i < LD; i += NT) {
		sy[i] = d.y[i]; sx[i] = d.x_b[i]; scb[i] = d.c_b[i]; sal[i] = d.alpha[i];
		sE[i] = d.E_q[i]; srq[i] = d.row_q[i]; sb[i] = d.b[i];
	}
	for (int j = tid; j < n; j += NT) sc[j] = d.c[j];
	for (int i = tid; i < m; i += NT) sbix[i] = d.b_ixs[i];
	long long it = ctl->iter, pivots = ctl->pivots;
	const long long it_end = ctl->it_end;
	int pending = ctl->pending;
	int status = 0, done = 0;
	long long p = ctl->p, q = ctl->q;
	double min_e = ctl->min_e;
	__syncthreads();

	tiny_pivots(s, sh, d.eps, d.pivot_tol, d.ratio_mode, d.trace, d.trace_cap, it, it_end, pivots, pending, status, done,
		p, q, min_e);

	// ---- state out
	__syncthreads();
	for (long long e = tid; e < (long long)LD * m; e += NT) d.B[e] = sB[e];
	for (int k = tid; k < LD; k += NT) {
		d.y[k] = sy[k]; d.x_b[k] = sx[k]; d.c_b[k] = scb[k]; d.alpha[k] = sal[k]; d.E_q[k] = sE[k]; d.row_q[k] = srq[k];
	}
	for (int k = tid; k < m; k += NT) d.b_ixs[k] = sbix[k];
	const T z = tiny_objective(scb, sx, m, sh);
	if (tid == 0) {
		ctl->iter = it; ctl->pivots = pivots; ctl->pending = pending;
		ctl->status = status; ctl->done = done;
		ctl->p = p; ctl->q = q; ctl->min_e = min_e; ctl->z = (double)z; ctl->c_b_q = sh.bc_v;
	}
}

// ---------------------------------------------------------------- many tiny LPs of one shape: one CTA per LP
//
// b200lp_solve_batch_*: the LPs of a batch are independent, so every CTA of a persistent grid solves whole LPs
// with the loop of simplex_tiny (tiny_pivots, NT threads, the same summation orders: the same bits as a single
// call).  CTAs take LP indices from a ticket counter because pivot counts differ by orders of magnitude between
// LPs; the order of hand-out changes no bit.  Each LP starts from the slack basis built in shared memory exactly
// as upload / reset leave it for simplex_tiny (k_reset); nothing per LP lives in HBM besides inputs and outputs.
constexpr int TINY_BATCH_MIN_CTAS = 2;   // 104 registers x 256 threads (f64): two CTAs per SM by registers

// one LP's outcome (the per-LP fields of b200lp_result)
struct TinyBatchRec {
	long long iterations, pivots;
	double z, min_e;
	int status, pad;
};

template <typename T>
struct TinyBatch {
	long long batch, m, n;
	const T* A;               // batch x (m x n column-major, leading dimension m)
	const T* b;               // batch x m
	const T* c;               // batch x n
	const int* ns;            // structural (stored, priced as dense) columns of every LP: n - m or n
	long long it_end;         // max_iter, per LP
	double eps, pivot_tol;
	int ratio_mode;
	T* x_b;                   // batch x m
	T* y;                     // batch x m, or null
	int* b_ixs;               // batch x m
	int2* trace;              // batch x trace_cap (p, q), or null
	long long trace_cap;
	TinyBatchRec* rec;        // batch
	unsigned long long* ticket; // next LP to hand out (zeroed by the host before the launch)
	int cost_shift;           // simplex_tiny_batch_dual: 1 = composite method (options.cost_shift)
	T delta;                  // its shift (options.shift_delta, 0 -> 1e-7, rounded to T as Engine does)
};

// state in: LP k's slack basis in shared memory, as k_reset leaves it for simplex_tiny, padding rows +0
template <typename T>
__device__ __forceinline__ void tiny_batch_load(const TinyBatch<T>& bt, long long k, const TinyLP<T>& s) {
	constexpr int LD = TinyLayout<T>::LD;
	const int tid = threadIdx.x;
	const int m = s.m, n = s.n, ns = s.ns;
	const T* Ak = bt.A + (size_t)k * (size_t)m * (size_t)n;
	const T* bk = bt.b + (size_t)k * m;
	const T* ck = bt.c + (size_t)k * n;
	for (long long e = tid; e < (long long)LD * ns; e += NT) {
		const int i = (int)(e % LD);
		s.A[e] = i < m ? Ak[(e / LD) * m + i] : T(0);
	}
	for (long long e = tid; e < (long long)LD * m; e += NT) s.B[e] = e % LD == e / LD ? T(1) : T(0);
	for (int i = tid; i < LD; i += NT) {
		const bool in = i < m;
		const T cb = in ? ck[n - m + i] : T(0);
		const T bi = in ? bk[i] : T(0);
		s.y[i] = cb; s.c_b[i] = cb; s.x_b[i] = bi; s.b[i] = bi;
		s.alpha[i] = T(0); s.E_q[i] = T(0); s.row_q[i] = T(0);
	}
	for (int j = tid; j < n; j += NT) s.c[j] = ck[j];
	for (int i = tid; i < m; i += NT) s.b_ixs[i] = n - m + i;
}

// state out: LP k's rows of x_b, b_ixs (and y), and its record with z = c_b . x_b; ends with the barrier after
// which the next LP may overwrite shared memory
template <typename T>
__device__ __forceinline__ void tiny_batch_store(const TinyBatch<T>& bt, long long k, const TinyLP<T>& s, Smem& sh,
		long long it, long long pivots, double min_e, int status) {
	const int tid = threadIdx.x;
	const int m = s.m;
	__syncthreads();
	for (int i = tid; i < m; i += NT) {
		bt.x_b[(size_t)k * m + i] = s.x_b[i];
		bt.b_ixs[(size_t)k * m + i] = s.b_ixs[i];
		if (bt.y) bt.y[(size_t)k * m + i] = s.y[i];
	}
	const T z = tiny_objective(s.c_b, s.x_b, m, sh);
	if (tid == 0) {
		TinyBatchRec r;
		r.iterations = it; r.pivots = pivots; r.z = (double)z; r.min_e = min_e; r.status = status; r.pad = 0;
		bt.rec[k] = r;
	}
	__syncthreads();                               // shared memory (ticket, LP) is reused by the next LP
}

template <typename T>
__global__ void __launch_bounds__(NT, TINY_BATCH_MIN_CTAS) simplex_tiny_batch(TinyBatch<T> bt) {
	__shared__ Smem sh;
	__shared__ long long s_k;
	extern __shared__ __align__(128) unsigned char dynraw[];
	T* S = reinterpret_cast<T*>(dynraw);
	const int tid = threadIdx.x;
	const int m = (int)bt.m, n = (int)bt.n;
	for (;;) {
		if (tid == 0) s_k = (long long)atomicAdd(bt.ticket, 1ULL);
		__syncthreads();
		const long long k = s_k;
		if (k >= bt.batch) break;
		const int ns = bt.ns[k];
		const TinyLayout<T> L(m, n, ns);
		const TinyLP<T> s(S, L, m, n, ns);
		tiny_batch_load(bt, k, s);
		long long it = 0, pivots = 0, p = 0, q = 0;
		int pending = 0, status = 0, done = 0;
		double min_e = 0;
		__syncthreads();

		int2* tr = bt.trace ? bt.trace + (size_t)k * bt.trace_cap : nullptr;
		tiny_pivots(s, sh, bt.eps, bt.pivot_tol, bt.ratio_mode, tr, tr ? bt.trace_cap : 0, it, bt.it_end, pivots, pending,
			status, done, p, q, min_e);
		tiny_batch_store(bt, k, s, sh, it, pivots, min_e, status);
	}
}

// Shared memory of simplex_tiny_batch_dual: TinyLayout (rho lives in alpha) and the nonbasic mask after b_ixs.
template <typename T>
struct TinyDualLayout : TinyLayout<T> {
	__host__ __device__ TinyDualLayout(long long m, long long n, long long ns) : TinyLayout<T>(m, n, ns) {}
	__host__ __device__ size_t nb(long long m) const { return (size_t)this->end * sizeof(T) + (size_t)m * sizeof(int); }
	__host__ __device__ size_t bytes(long long m, long long n) const { return TinyLayout<T>::bytes(m) + (size_t)n; }
};

// The dual simplex (options.algorithm = 1) and the composite method (cost_shift = 1) on many tiny LPs: the grid,
// tickets, state in and state out of simplex_tiny_batch, and per LP the single call's sequence in one CTA:
//   cost_shift: k_cost_shift from the slack basis (y = c_b) over the stored nonbasic columns j < n - m, s = y.a_j
//     in the pricing association, c_j <- s - mul_rn(delta, 1 + |c_j|) where (double)(s - c_j) < -eps
//   phase 1: tiny_dual_pivots (simplex_dual) from the mask of k_nonbasic_init
//   after a phase-1 OPTIMUM with a shifted column, Engine::hand_over: flush the pending update (the update block's
//     fma), c from the caller's c, c_b = c[b_ixs], y_j = c_b.B^-1[:, j] (k_btran_vec's pricing association) when
//     phase 1 pivoted, status MAX_ITER; then phase 2: tiny_pivots with the rest of max_iter.  z is c_b . x_b of
//     whatever basis the LP stops in, which after a budget ending on the phase-1 optimum is hand_over's k_objective.
template <typename T>
__global__ void __launch_bounds__(NT, TINY_BATCH_MIN_CTAS) simplex_tiny_batch_dual(TinyBatch<T> bt) {
	using V = typename VecT<T>::V;
	constexpr int VN = VecT<T>::N;
	constexpr int LD = TinyLayout<T>::LD;
	__shared__ Smem sh;
	__shared__ long long s_k;
	extern __shared__ __align__(128) unsigned char dynraw[];
	T* S = reinterpret_cast<T*>(dynraw);
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const int m = (int)bt.m, n = (int)bt.n;
	for (;;) {
		if (tid == 0) s_k = (long long)atomicAdd(bt.ticket, 1ULL);
		__syncthreads();
		const long long k = s_k;
		if (k >= bt.batch) break;
		const int ns = bt.ns[k];
		const TinyDualLayout<T> L(m, n, ns);
		const TinyLP<T> s(S, L, m, n, ns);
		unsigned char* nb = dynraw + L.nb(m);
		tiny_batch_load(bt, k, s);
		for (int j = tid; j < n; j += NT) nb[j] = j < n - m ? 1 : 0;
		long long it = 0, pivots = 0, p = 0, q = 0;
		int pending = 0, status = 0, done = 0;
		double min_e = 0;
		__syncthreads();

		int shifted = 0;
		if (bt.cost_shift) {
			const V yv = *reinterpret_cast<const V*>(s.y + lane * VN);
			for (int col = warp; col < n - m; col += NWARP) {
				const T sd = tiny_dot<T>(*reinterpret_cast<const V*>(s.A + (long long)col * LD + lane * VN), yv);
				if (lane == 0) {
					const T cj = s.c[col];
					if ((double)(sd - cj) < -bt.eps) {
						s.c[col] = sd - mul_rn_t(bt.delta, T(1) + (cj < T(0) ? -cj : cj));
						shifted = 1;
					}
				}
			}
			shifted = __syncthreads_or(shifted);
		}

		int2* tr = bt.trace ? bt.trace + (size_t)k * bt.trace_cap : nullptr;
		tiny_dual_pivots(s, nb, sh, bt.eps, bt.pivot_tol, tr, tr ? bt.trace_cap : 0, it, bt.it_end, pivots, pending,
			status, done, p, q, min_e);

		if (shifted && done && status == 1) {          // hand-over to the primal loop
			if (pending) {
				for (long long e = tid; e < (long long)LD * m; e += NT)
					s.B[e] = fma_t(s.E_q[e % LD], s.row_q[e / LD], s.B[e]);
				pending = 0;
			}
			const T* ck = bt.c + (size_t)k * n;
			for (int j = tid; j < n; j += NT) s.c[j] = ck[j];
			__syncthreads();
			for (int i = tid; i < m; i += NT) s.c_b[i] = s.c[s.b_ixs[i]];
			__syncthreads();
			if (pivots > 0) {
				const V cv = *reinterpret_cast<const V*>(s.c_b + lane * VN);
				for (int col = warp; col < m; col += NWARP) {
					const T yj = tiny_dot<T>(*reinterpret_cast<const V*>(s.B + (long long)col * LD + lane * VN), cv);
					if (lane == 0) s.y[col] = yj;
				}
				__syncthreads();
			}
			status = 0;                                // B200LP_STATUS_MAX_ITER
			done = 0;
			tiny_pivots(s, sh, bt.eps, bt.pivot_tol, bt.ratio_mode, tr, tr ? bt.trace_cap : 0, it, bt.it_end, pivots,
				pending, status, done, p, q, min_e);
		}
		tiny_batch_store(bt, k, s, sh, it, pivots, min_e, status);
	}
}

// ---------------------------------------------------------------- mid-size LPs: B^-1 and A resident in shared memory
//
// m ~ 256 ... 1500 (BASELINE config 2: m = 1024): A and B^-1 fit in the 126 MB L2, but a pivot of the general
// kernel is ~20 us of tile / barrier latency for ~3 us of L2 streaming (64 tiles for 148 SMs, ~20 dependent L2
// round trips).  Here the whole LP lives in the shared memory of the grid: CTA c owns rpc consecutive ROWS of B^-1
// (row-major, every 32-column sub-block padded to 33 so that the per-(row, sub-block) fma chains of a warp hit
// different banks) and cpc consecutive COLUMNS of A, plus private copies of y, b and the pivot row.  A pivot is
//   pricing of the own columns (shared memory)                              | B1 -> p
//   entering column from global A (L2), rank-1 update + FTRAN + ratio test
//   on the own rows (shared memory)                                         | B2 -> q, alpha_q
//   E_q of the own rows, products c_b E_q, owner: row q -> global (8 KB)     | B3
//   every CTA: row_q.b, c_b.E_q, y (own full copy), x_b / c_b / b_ixs (own rows)
// i.e. three grid barriers and three small L2 exchanges; no matrix byte leaves shared memory inside the loop.
// Every sum is associated exactly as in the general kernel (file header), so the results are bit-identical to it
// and to the oracle's order = 1.  State is read from and written back to the same global buffers (same deferred
// rank-1 update semantics), so windows, downloads, check_basis and the phase entry points see no difference.

template <typename T>
struct ResLayout {
	static constexpr int SBP = SUBW + 1;     // padded sub-block
	long long rpc, cpc, nsb, G;              // rows / columns per CTA, sub-blocks per row, CTAs in use
	long long Bs, As, y, b, rowq, prod, rowqP, apP, part, xb, cb, al, eq, cown, cunit, end;   // element offsets (T)
	__host__ __device__ static long long r4(long long x) { return (x + 3) / 4 * 4; }
	__host__ __device__ ResLayout(long long m, long long ld, long long ns, long long maxG) {
		rpc = (m + maxG - 1) / maxG;
		G = (m + rpc - 1) / rpc;
		cpc = (ns + G - 1) / G;
		nsb = (m + SUBW - 1) / SUBW;
		long long o = 0;
		As = o; o += r4(cpc * ld);
		y = o; o += ld; b = o; o += ld; rowq = o; o += ld; prod = o; o += ld;
		rowqP = o; o += r4(nsb * SBP); apP = o; o += r4(nsb * SBP);     // row_q / a_p in the padded sub-block layout of Bs
		Bs = o; o += r4(rpc * nsb * SBP);
		part = o; o += r4(rpc * nsb);
		xb = o; o += r4(rpc); cb = o; o += r4(rpc); al = o; o += r4(rpc); eq = o; o += r4(rpc);
		cown = o; o += r4(cpc);                                   // costs of the own structural columns
		cunit = o; o += r4(((m > ns ? m : ns) + G - 1) / G + 1);  // costs of the own share of the unit columns
		end = o;
	}
	__host__ __device__ size_t bytes() const { return (size_t)end * sizeof(T) + (size_t)r4(rpc) * sizeof(int) + 16; }
};

// sum of a vector of m values held in shared memory in the order of the O(m) dots (256-element slices: thread t
// owns element t, warp butterfly, 8 warp sums left to right; slices left to right); PROD: the elements are
// x[i] * y[i] formed by one fma each, otherwise x[i] as they are.  Result in every thread.
// two such sums at once: s1 = sum of x[i] * y[i] (one fma each), s2 = sum of z[i]; six slices (m <= 1536) share
// one barrier
template <typename T>
__device__ __forceinline__ void res_sliced_sums(const T* x, const T* y, const T* z, long long m, Smem& sh, T& s1, T& s2) {
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	constexpr int SPB = 6;                                    // slices per barrier: 2 * SPB <= the 12 slots of a wsum buffer
	s1 = T(0); s2 = T(0);
	int buf = 0;
	for (long long s0 = 0; s0 < m; s0 += (long long)SPB * SLICE, buf ^= 1) {
#pragma unroll
		for (int k = 0; k < SPB; ++k) {
			const long long i = s0 + (long long)k * SLICE + tid;
			if (s0 + (long long)k * SLICE < m) {               // CTA uniform
				T t1 = T(0), t2 = T(0);
				if (i < m) { t1 = fma_t(x[i], y[i], T(0)); t2 = z[i]; }
				t1 = warp_butterfly_sum(t1);
				t2 = warp_butterfly_sum(t2);
				if (lane == 0) { sh.wsum[buf][2 * k][warp] = (double)t1; sh.wsum[buf][2 * k + 1][warp] = (double)t2; }
			}
		}
		__syncthreads();
#pragma unroll
		for (int k = 0; k < SPB; ++k) {
			if (s0 + (long long)k * SLICE < m) {
				T a1 = T(0), a2 = T(0);
#pragma unroll
				for (int w = 0; w < NWARP; ++w) { a1 = a1 + (T)sh.wsum[buf][2 * k][w]; a2 = a2 + (T)sh.wsum[buf][2 * k + 1][w]; }
				s1 = s1 + a1;
				s2 = s2 + a2;
			}
		}
	}
	__syncthreads();
}

template <typename T>
__global__ void __launch_bounds__(NT, 1) simplex_resident(Dev<T> d) {
	using V = typename VecT<T>::V;
	using M = Mem<T>;
	constexpr int VN = VecT<T>::N;
	constexpr int SBP = ResLayout<T>::SBP;
	__shared__ Smem sh;
	extern __shared__ __align__(128) unsigned char dynraw[];
	T* S = reinterpret_cast<T*>(dynraw);
	const ResLayout<T> L(d.m, d.ld, d.ns, d.res_maxG);
	T *sA = S + L.As, *sy = S + L.y, *sb = S + L.b, *srq = S + L.rowq, *srqP = S + L.rowqP, *sapP = S + L.apP, *sprod = S + L.prod, *sB = S + L.Bs,
	  *spart = S + L.part, *sxb = S + L.xb, *scb = S + L.cb, *sal = S + L.al, *seq = S + L.eq, *scown = S + L.cown, *scunit = S + L.cunit;
	int* sbix = reinterpret_cast<int*>(S + L.end);
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const int G = gridDim.x, me = blockIdx.x;          // G == L.G
	const long long m = d.m, ld = d.ld, ns = d.ns, nsb = L.nsb;
	const long long r0 = (long long)me * L.rpc, nr = r0 < m ? (m - r0 < L.rpc ? m - r0 : L.rpc) : 0;   // own rows
	const long long c0 = (long long)me * L.cpc, nc = c0 < ns ? (ns - c0 < L.cpc ? ns - c0 : L.cpc) : 0; // own columns
	const long long nunit = d.n - ns, k0 = nunit * me / G, k1 = nunit * (me + 1) / G;                   // own unit columns
	Ctl* ctl = d.ctl;
	unsigned long long epoch = 0;

	// ---- state in
	for (long long e = tid; e < nc * ld; e += NT) sA[e] = d.A[c0 * ld + e];
	for (long long e = tid; e < nr * m; e += NT) {
		const long long r = e % nr, j = e / nr;           // consecutive threads: consecutive rows of one column
		sB[(r * nsb + j / SUBW) * SBP + j % SUBW] = d.B[(r0 + r) + j * d.ldb];
	}
	for (long long i = tid; i < ld; i += NT) {
		sy[i] = d.y[i]; sb[i] = d.b[i]; sprod[i] = T(0);
		const T rq = d.row_q[i];
		srq[i] = rq;
		if (i < m) srqP[(i / SUBW) * SBP + i % SUBW] = rq;
	}
	for (long long r = tid; r < nr; r += NT) {
		sxb[r] = d.x_b[r0 + r]; scb[r] = d.c_b[r0 + r]; sal[r] = d.alpha[r0 + r]; seq[r] = d.E_q[r0 + r]; sbix[r] = d.b_ixs[r0 + r];
	}
	for (long long k = tid; k < nc; k += NT) scown[k] = d.c[c0 + k];
	for (long long k = k0 + tid; k < k1; k += NT) scunit[k - k0] = d.c[ns + k];
	long long it = ctl->iter, pivots = ctl->pivots;
	const long long it_end = ctl->it_end;
	int pending = ctl->pending;
	int status = 0, done = 0, aborted = 0;
	long long p = ctl->p, q = ctl->q;
	double min_e = ctl->min_e;
	const T tol = (T)d.pivot_tol;
	__syncthreads();

	const long long it0 = it;
	while (it < it_end) {
		// ---- pricing of the own columns (v4:288-302): the dots of price_phase, operands in shared memory
		stamp(d, it - it0, 0, me);
		double best_v = CUDART_INF;
		long long best_i = LLONG_MAX;
		int buf = 0;
		for (long long kq = 0; kq < nc; kq += PRICE_NC, buf ^= 1) {
			T acc[PRICE_NC][VN];
#pragma unroll
			for (int k = 0; k < PRICE_NC; ++k)
#pragma unroll
				for (int v = 0; v < VN; ++v) acc[k][v] = T(0);
			for (long long i = (long long)tid * VN; i < ld; i += (long long)NT * VN) {
				const V yv = *reinterpret_cast<const V*>(sy + i);
#pragma unroll
				for (int k = 0; k < PRICE_NC; ++k) {
					if (kq + k < nc) {
						const V av = *reinterpret_cast<const V*>(sA + (kq + k) * ld + i);
#pragma unroll
						for (int v = 0; v < VN; ++v) acc[k][v] = fma_t(M::get(av, v), M::get(yv, v), acc[k][v]);
					}
				}
			}
#pragma unroll
			for (int k = 0; k < PRICE_NC; ++k) {
				T s = acc[k][0];
#pragma unroll
				for (int v = 1; v < VN; ++v) s = s + acc[k][v];
				s = warp_butterfly_sum(s);
				if (lane == 0) sh.wsum[buf][k][warp] = (double)s;
			}
			__syncthreads();
			if (tid < PRICE_NC && kq + tid < nc) {
				const long long j = c0 + kq + tid;
				const double e = (double)(warp_sums<T>(sh, buf, tid) - scown[kq + tid]);
				if (cand_better(e, j, best_v, best_i)) { best_v = e; best_i = j; }
			}
		}
		for (long long k = k0 + tid; k < k1; k += NT) {      // unit (slack) columns
			const double e = (double)(sy[k] - scunit[k - k0]);
			if (cand_better(e, ns + k, best_v, best_i)) { best_v = e; best_i = ns + k; }
		}
		block_argmin(best_v, best_i, sh);
		if (tid == 0) { d.cand[me].val = best_v; d.cand[me].idx = best_i; }
		if (me == 0 && tid == 0) ctl->abort_latched = *(volatile int*)&ctl->abort_req;
		stamp(d, it - it0, 1, me);
		grid_barrier(ctl, epoch, G);
		reduce_cands(d.cand, G, min_e, p, sh);
		stamp(d, it - it0, 2, me);
		if (__ldcg(&ctl->abort_latched)) { aborted = 1; break; }
		if (min_e >= -d.eps) { status = 1; done = 1; ++it; break; }

		// ---- entering column (L2), then the pending rank-1 update fused with the FTRAN on the own rows (v4:333, 307-308)
		for (long long j = tid; j < m; j += NT)
			sapP[(j / SUBW) * SBP + j % SUBW] = p < ns ? __ldcg(d.A + p * ld + j) : (j == p - ns ? T(1) : T(0));
		__syncthreads();
		for (long long w = tid; w < nr * nsb; w += NT) {
			const long long r = w / nsb, sbk = w % nsb;
			T* bp = sB + w * SBP;
			const long long jb = sbk * SUBW;
			const int ncols = (int)(m - jb < SUBW ? m - jb : SUBW);
			const T er = seq[r];
			const T *rqp = srqP + sbk * SBP, *app = sapP + sbk * SBP;   // consecutive lanes: stride 33 -> no bank conflicts
			T acc = T(0);
			if (ncols == SUBW) {
#pragma unroll
				for (int u0 = 0; u0 < SUBW; u0 += 8) {
					T x8[8], r8[8], a8[8];
#pragma unroll
					for (int u = 0; u < 8; ++u) { x8[u] = bp[u0 + u]; r8[u] = rqp[u0 + u]; a8[u] = app[u0 + u]; }
#pragma unroll
					for (int u = 0; u < 8; ++u) {
						if (pending) { x8[u] = fma_t(er, r8[u], x8[u]); bp[u0 + u] = x8[u]; }
						acc = fma_t(x8[u], a8[u], acc);
					}
				}
			} else {
				for (int u = 0; u < ncols; ++u) {
					T x = bp[u];
					if (pending) { x = fma_t(er, rqp[u], x); bp[u] = x; }
					acc = fma_t(x, app[u], acc);
				}
			}
			spart[w] = acc;
		}
		pending = 0;
		__syncthreads();
		// alpha of the own rows: pairwise tree over the 8 sub-blocks of a chunk, chunks left to right; ratio test (v4:311-325)
		double rv = CUDART_INF;
		long long ri = LLONG_MAX, elig = 0;
		if (tid < nr) {
			const T* pr = spart + (long long)tid * nsb;
			T a = T(0);
			for (long long c8 = 0; c8 < nsb; c8 += CHUNK / SUBW) {
				T t8[CHUNK / SUBW];
#pragma unroll
				for (int k = 0; k < CHUNK / SUBW; ++k) t8[k] = c8 + k < nsb ? pr[c8 + k] : T(0);
				const T ck = ((t8[0] + t8[1]) + (t8[2] + t8[3])) + ((t8[4] + t8[5]) + (t8[6] + t8[7]));
				a = c8 == 0 ? ck : a + ck;
			}
			sal[tid] = a;
			if (a > tol) {
				elig = 1;
				rv = (double)(ratio_num(sxb[tid], d.ratio_mode) / a);
				ri = r0 + tid;
			}
		}
		block_argmin(rv, ri, sh);
		elig = __syncthreads_count(elig != 0);
		if (tid == 0) {
			// (not d.cand: a slow CTA may still be reducing the pricing candidates of this iteration)
			d.cand2[me].val = rv; d.cand2[me].idx = ri; d.cnt[me] = elig;
			d.cand2[G + me].val = ri != LLONG_MAX ? (double)sal[ri - r0] : 0.0;      // alpha at this CTA's candidate
		}
		const T c_p = d.c[p];                                 // (in flight across the barrier)
		stamp(d, it - it0, 3, me);
		grid_barrier(ctl, epoch, G);
		stamp(d, it - it0, 4, me);
		// one pass: argmin of the candidates, sum of the eligible counts, and alpha at the winner (thread k holds CTA k's record)
		double th = CUDART_INF, aq = 0.0;
		q = LLONG_MAX;
		long long el = 0;
		for (int k = tid; k < G; k += NT) {
			const double cv = __ldcg(&d.cand2[k].val), ca = __ldcg(&d.cand2[G + k].val);
			const long long ci = __ldcg(&d.cand2[k].idx);
			el += __ldcg(&d.cnt[k]);
			if (cand_better(cv, ci, th, q)) { th = cv; q = ci; aq = ca; }
		}
#pragma unroll
		for (int off = 16; off >= 1; off >>= 1) {
			const double ov = __shfl_xor_sync(0xffffffffu, th, off), oa = __shfl_xor_sync(0xffffffffu, aq, off);
			const long long oi = __shfl_xor_sync(0xffffffffu, q, off);
			el += __shfl_xor_sync(0xffffffffu, el, off);
			if (cand_better(ov, oi, th, q)) { th = ov; q = oi; aq = oa; }
		}
		__syncthreads();
		if (lane == 0) { sh.red_v[warp] = th; sh.red_i[warp] = q; sh.red_c[warp] = el; sh.dsum[2][warp] = aq; }
		__syncthreads();
		th = sh.red_v[0]; q = sh.red_i[0]; el = sh.red_c[0]; aq = sh.dsum[2][0];
#pragma unroll
		for (int w = 1; w < NWARP; ++w) {
			if (cand_better(sh.red_v[w], sh.red_i[w], th, q)) { th = sh.red_v[w]; q = sh.red_i[w]; aq = sh.dsum[2][w]; }
			el += sh.red_c[w];
		}
		if (el == 0) { status = 2; done = 1; ++it; break; }
		const int owner = (int)(q / L.rpc);
		const T alpha_q = (T)aq;
		stamp(d, it - it0, 5, me);

		// ---- E_q of the own rows, products c_b_new E_q; the owner of row q publishes it (v4:331-332, 340, 354)
		if (tid < nr) {
			const long long i = r0 + tid;
			const T eqv = (i != q) ? (-sal[tid] / alpha_q) : (T)(1.0 / (double)alpha_q - 1.0);
			seq[tid] = eqv;
			T cb = scb[tid];
			if (i == q) { ctl->c_b_q = (double)cb; cb = c_p; }
			d.E_q[i] = fma_t(cb, eqv, T(0));                  // (E_q doubles as the exchange buffer of the products; rewritten at exit)
		}
		if (me == owner) {
			const T* brow = sB + (q - r0) * nsb * SBP;
			for (long long j = tid; j < m; j += NT) d.row_q[j] = brow[(j / SUBW) * SBP + j % SUBW];
		}
		stamp(d, it - it0, 6, me);
		grid_barrier(ctl, epoch, G);
		stamp(d, it - it0, 7, me);

		// ---- every CTA: row_q.b, c_b.E_q, y (own full copy); own rows: x_b, c_b, b_ixs (v4:339-356)
		const T c_b_q = (T)__ldcg(&ctl->c_b_q);            // issued with the vector loads below
		for (long long j = tid; j < ld; j += NT) {
			const T rq = j < m ? __ldcg(d.row_q + j) : T(0);
			srq[j] = rq;
			if (j < m) srqP[(j / SUBW) * SBP + j % SUBW] = rq;
			sprod[j] = j < m ? __ldcg(d.E_q + j) : T(0);
		}
		__syncthreads();
		T sx, syv;
		res_sliced_sums<T>(srq, sb, sprod, m, sh, sx, syv);
		syv += c_p - c_b_q;
		for (long long j = tid; j < m; j += NT) sy[j] = fma_t(syv, srq[j], sy[j]);
		if (tid < nr) {
			sxb[tid] = fma_t(sx, seq[tid], sxb[tid]);
			if (r0 + tid == q) { scb[tid] = c_p; sbix[tid] = (int)p; }
		}
		if (me == 0 && tid == 0 && pivots < d.trace_cap) d.trace[pivots] = make_int2((int)p, (int)q);
		pending = 1;
		++pivots;
		stamp(d, it - it0, 8, me);
		++it;
		__syncthreads();
		// (the next exchange through d.E_q / d.row_q is two barriers away: no barrier needed here)
	}

	// ---- state out (every CTA is past its last read of the exchange buffers after this barrier)
	grid_barrier(ctl, epoch, G);
	for (long long e = tid; e < nr * m; e += NT) {
		const long long r = e % nr, j = e / nr;
		d.B[(r0 + r) + j * d.ldb] = sB[(r * nsb + j / SUBW) * SBP + j % SUBW];
	}
	for (long long r = tid; r < nr; r += NT) {
		d.x_b[r0 + r] = sxb[r]; d.c_b[r0 + r] = scb[r]; d.alpha[r0 + r] = sal[r]; d.E_q[r0 + r] = seq[r]; d.b_ixs[r0 + r] = sbix[r];
	}
	if (me == 0) for (long long i = tid; i < m; i += NT) { d.y[i] = sy[i]; d.row_q[i] = srq[i]; }
	grid_barrier(ctl, epoch, G);
	if (me == 0) {
		const double z = objective<T>(d, sh);
		if (tid == 0) {
			ctl->iter = it; ctl->pivots = pivots; ctl->pending = pending;
			ctl->status = status; ctl->done = done; ctl->aborted = aborted;
			ctl->p = p; ctl->q = q; ctl->min_e = min_e; ctl->z = z;
		}
	}
}

// ---------------------------------------------------------------- sharded (multi-GPU) loop
//
// One process per GPU, the same persistent kernel on every rank.  B^-1 is row-block
// sharded, A column-block sharded, every O(m) vector (y, x_b, c_b, alpha, E_q, row_q,
// b_ixs) is replicated, so all ranks take identical decisions and the per-row / per-column
// sums are exactly the single-GPU ones (results are bit-identical for every GPU count).
// Three exchanges per pivot, all direct peer stores over NVLink into the receivers'
// mailboxes — no NCCL call and no host on the data path:
//   X1  pricing candidate (value, index) of the local column block      (replaces the global cub ArgMin)
//   X2  alpha of the local row block (m/R values) + the ratio-test candidate of those rows
//   X3  row q of B^-1 from its owner (m values) + the slice partials of row_q.b  (replaces cublasScopy, v4:331)
// Each record carries its own flag: the LAST CTA of the sending rank to finish the producing
// phase stores the record with a release at system scope, and every CTA of every rank spins
// on the flags in its own mailbox.  That spin is the barrier — a pivot costs three NVLink
// hops and four local grid barriers.  Ordering: payload stores by any CTA -> gpu-scope fence +
// arrival (barrier or counter) -> acquired by the publishing thread -> st.release.sys of the
// flag -> ld.acquire.sys by the receiver; release/acquire are cumulative in the PTX memory
// model, so exactly ONE system-scope fence sits on the critical path of an exchange.  The entering column a_p is pulled from its owner's A
// shard with peer loads.

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
	unsigned long long v;
	asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
	return v;
}
__device__ __forceinline__ unsigned long long ld_acquire_gpu(const unsigned long long* p) {
	unsigned long long v;
	asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
	return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
	asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

constexpr unsigned long long XWAIT_NS = 20000000000ULL;   // 20 s: a peer died

// spin until *flag >= want; false on time-out
__device__ __forceinline__ bool wait_flag_sys(const unsigned long long* flag, unsigned long long want) {
	if (ld_acquire_sys(flag) >= want) return true;
	const unsigned long long t0 = globaltimer_ns();
	while (ld_acquire_sys(flag) < want)
		if (globaltimer_ns() - t0 > XWAIT_NS) return false;
	return true;
}

// local grid barrier with a time-out (a CTA that gave up on a dead peer must not hang the others)
__device__ __forceinline__ bool grid_barrier_t(Ctl* ctl, unsigned long long& epoch, Smem& sh, int G) {
	epoch += G;
	__syncthreads();
	if (threadIdx.x == 0) {
		bool ok = true;
		if (G > 1) {
			asm volatile("red.release.gpu.global.add.u64 [%0], 1;" ::"l"(&ctl->bar) : "memory");
			if (ld_acquire_gpu(&ctl->bar) < epoch) {
				const unsigned long long t0 = globaltimer_ns();
				while (ld_acquire_gpu(&ctl->bar) < epoch)
					if (globaltimer_ns() - t0 > XWAIT_NS) { ok = false; break; }
			}
		}
		sh.bc_c = ok;
	}
	__syncthreads();
	return sh.bc_c != 0;
}

// one arrival per CTA on a monotonic counter; true (in every thread) for the CTA that arrives last.
// Data written before the call by any CTA is visible to the last one after it.
__device__ __forceinline__ bool arrive_last(unsigned long long* ctr, unsigned long long target, Smem& sh) {
	__syncthreads();
	if (threadIdx.x == 0) {
		__threadfence();
		const bool last = atomicAdd(ctr, 1ULL) + 1 == target;
		__threadfence();
		sh.bc_c = last;
	}
	__syncthreads();
	const bool last = sh.bc_c != 0;
	__syncthreads();
	return last;
}

template <typename T> __device__ __forceinline__ XHdr* xhdr(const Dev<T>& d, int r) { return reinterpret_cast<XHdr*>(d.mbox_peer[r]); }
template <typename T> __device__ __forceinline__ T* xalpha(const Dev<T>& d, int r) { return reinterpret_cast<T*>(d.mbox_peer[r] + sizeof(XHdr)); }
template <typename T> __device__ __forceinline__ T* xrowq(const Dev<T>& d, int r) { return xalpha(d, r) + d.ld; }
template <typename T> __device__ __forceinline__ T* xrqb(const Dev<T>& d, int r) { return xalpha(d, r) + 2 * d.ld; }
// rank `src`'s partial of v = B^-T alpha in rank `dst`'s mailbox (steepest edge)
template <typename T> __device__ __forceinline__ T* xvpart(const Dev<T>& d, int dst, int src) { return xalpha(d, dst) + d.vpart_off + (long long)src * d.ld; }

// collect the R records of one exchange from our own mailbox and reduce them: lexicographic
// argmin over (val, idx), sum of cnt.  Same fixed order on every rank and CTA.
template <typename T>
__device__ __forceinline__ bool gather_records(const Dev<T>& d, const XCand* rec, unsigned long long e, Smem& sh,
		double& v, long long& i, long long& c, double* v2 = nullptr, long long* i2 = nullptr) {
	if (threadIdx.x < d.nranks) {
		const XCand* r = rec + threadIdx.x;
		const bool ok = wait_flag_sys(&r->flag, e);
		sh.xv[threadIdx.x] = __ldcg(&r->val);
		sh.xi[threadIdx.x] = __ldcg(&r->idx);
		sh.xc[threadIdx.x] = ok ? __ldcg(&r->cnt) : -1;
		if (v2) { sh.xv2[threadIdx.x] = __ldcg(&r->val2); sh.xi2[threadIdx.x] = __ldcg(&r->idx2); }
	}
	__syncthreads();
	v = CUDART_INF; i = LLONG_MAX; c = 0;
	if (v2) { *v2 = CUDART_INF; *i2 = LLONG_MAX; }
	bool ok = true;
	for (int r = 0; r < d.nranks; ++r) {
		if (sh.xc[r] < 0) ok = false;
		if (cand_better(sh.xv[r], sh.xi[r], v, i)) { v = sh.xv[r]; i = sh.xi[r]; }
		if (v2 && cand_better(sh.xv2[r], sh.xi2[r], *v2, *i2)) { *v2 = sh.xv2[r]; *i2 = sh.xi2[r]; }
		c += sh.xc[r];
	}
	__syncthreads();
	return ok;
}

// the last CTA of this rank reduces the rank's candidates (per CTA for pricing, per row group for the ratio
// test) and stores the record into every mailbox.  cnts == nullptr: the count field carries `extra`
// (X1: this rank's abort request, so that all ranks stop in the same iteration).
template <typename T>
__device__ __forceinline__ void publish(const Dev<T>& d, Smem& sh, int which, int par, unsigned long long e,
		const Cand* cands, int ncand, const long long* cnts, long long extra, const Cand* cands2 = nullptr) {
	double v, v2 = CUDART_INF; long long i, i2 = LLONG_MAX;
	reduce_cands(cands, ncand, v, i, sh);
	if (cands2) reduce_cands(cands2, ncand, v2, i2, sh);
	const long long c = cnts ? reduce_counts(cnts, ncand, sh) : extra;
	if (threadIdx.x < d.nranks) {
		XHdr* h = xhdr(d, threadIdx.x);
		XCand* dst = which == 0 ? &h->pc[par][d.rank] : &h->rc[d.rank];
		dst->val = v;
		dst->idx = i;
		dst->cnt = c;
		dst->val2 = v2;
		dst->idx2 = i2;
		st_release_sys(&dst->flag, e);     // orders the three stores above (and, cumulatively, everything
		                                   // the other CTAs fenced before they arrived) before the flag
	}
}

// pull the entering column from its owner's A shard into the local staging vector
template <typename T>
__device__ void fetch_column(const Dev<T>& d, long long p, int part, int nparts) {
	using M = Mem<T>;
	using V = typename VecT<T>::V;
	constexpr int VN = VecT<T>::N;
	int o = 0;
	while (o + 1 < d.nranks && p >= d.colstart[o + 1]) ++o;
	const T* src = d.A_peer[o] + (p - d.colstart[o]) * d.ld;
	for (long long i = ((long long)part * NT + threadIdx.x) * VN; i < d.ld; i += (long long)nparts * NT * VN)
		*reinterpret_cast<V*>(d.acol + i) = M::ld_nc(src + i);
}

// X2 producer: alpha of the local rows = sum of the chunk partials (left to right), stored into
// every rank's alpha; the ratio test of those rows (v4:199-208) gives this CTA's candidate.
template <typename T>
__device__ void push_alpha_ratio(const Dev<T>& d, Smem& sh, T* stage, int part, int nparts) {
	const int tid = threadIdx.x;
	double best_v = CUDART_INF;
	long long best_i = LLONG_MAX;
	long long elig = 0;
	auto take = [&](long long il, T a) {
		const long long i = d.row0 + il;
		for (int r = 0; r < d.nranks; ++r) xalpha(d, r)[i] = a;
		if (i < d.m && a > (T)d.pivot_tol) {
			++elig;
			const double th = (double)(ratio_num(d.x_b[i], d.ratio_mode) / a);
			if (cand_better(th, i, best_v, best_i)) { best_v = th; best_i = i; }
		}
	};
	const long long nblk = (d.ldb + 31) / 32;           // blocks of 32 local rows
	if (nblk <= 2 * (long long)nparts) {                // the CTA's warps load a block's chunk partials together
		for (long long blk = part; blk < nblk; blk += nparts) {
			const T a = sum_partials_rows32<T>(d, stage, blk * 32);
			const long long il = blk * 32 + tid;
			if (tid < 32 && il < d.ldb) take(il, a);
		}
	} else {                                            // many rows per CTA: one row per thread
		for (long long il = (long long)part * NT + tid; il < d.ldb; il += (long long)nparts * NT)
			take(il, sum_chunk_partials(d.alpha_part + il, d.ldb, d.nchunk));
	}
	block_argmin(best_v, best_i, sh);
#pragma unroll
	for (int off = 16; off >= 1; off >>= 1) elig += __shfl_xor_sync(0xffffffffu, elig, off);
	__syncthreads();
	if ((tid & 31) == 0) sh.red_c[tid >> 5] = elig;
	__syncthreads();
	if (tid == 0) {
		long long c = 0;
#pragma unroll
		for (int w = 0; w < NWARP; ++w) c += sh.red_c[w];
		d.cand[part].val = best_v;
		d.cand[part].idx = best_i;
		d.cnt[part] = c;
	}
}

// book1, sharded: E_q and the c_b.E_q slice partials on every rank (replicated data);
// X3 producer: the owner of row q gathers it from its B^-1 block, forms the row_q.b slice
// partials and stores both into every rank's mailbox.
template <typename T, bool SE = false>
__device__ void book1_sharded(const Dev<T>& d, Smem& sh, long long p, long long q, int part, int nparts) {
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const T alpha_q = __ldcg(d.alpha + q);     // mailbox data: read at L2
	const T c_p = d.c[p];
	const bool owner = q >= d.row0 && q < d.row0 + d.ldb;
	for (long long s = part; s < d.nslice; s += nparts) {
		const long long i = s * SLICE + tid;
		T t1 = T(0), t2 = T(0), t3 = T(0);
		if (i < d.m) {
			const T al = __ldcg(d.alpha + i);
			const T eq = (i != q) ? (-al / alpha_q) : (T)(1.0 / (double)alpha_q - 1.0);
			d.E_q[i] = eq;
			T cb = d.c_b[i];
			if (i == q) {
				d.ctl->c_b_q = (double)cb; cb = c_p;
				if (SE) { d.ctl->alpha_q = (double)alpha_q; d.ctl->leaving = d.b_ixs[q]; }
			}
			t2 = fma_t(cb, eq, T(0));
			if (SE) t3 = fma_t(al, al, T(0));
			if (owner) {
				const T rq = d.B[(q - d.row0) + i * d.ldb];
				t1 = fma_t(rq, d.b[i], T(0));
				for (int r = 0; r < d.nranks; ++r) xrowq(d, r)[i] = rq;
			}
		}
		t1 = warp_butterfly_sum(t1);
		t2 = warp_butterfly_sum(t2);
		if (SE) t3 = warp_butterfly_sum(t3);
		__syncthreads();
		if (lane == 0) { sh.dsum[0][warp] = (double)t1; sh.dsum[1][warp] = (double)t2; if (SE) sh.dsum[2][warp] = (double)t3; }
		__syncthreads();
		if (tid == 0) {
			T a1 = T(0), a2 = T(0), a3 = T(0);
#pragma unroll
			for (int w = 0; w < NWARP; ++w) { a1 = a1 + (T)sh.dsum[0][w]; a2 = a2 + (T)sh.dsum[1][w]; if (SE) a3 = a3 + (T)sh.dsum[2][w]; }
			d.dpart[(long long)d.nslice + s] = a2;
			if (SE) d.dpart[2LL * d.nslice + s] = a3;
			if (owner)
				for (int r = 0; r < d.nranks; ++r) xrqb(d, r)[s] = a1;
		}
	}
}

// steepest edge, sharded: this rank's partial of v = B^-T alpha — the column dots of its row block of B^-1 with its
// slice of alpha (pricing order over the local rows) — stored into every rank's mailbox (X4)
template <typename T>
__device__ void btran_partial_push(const Dev<T>& d, Smem& sh, int part, int nparts) {
	const int tid = threadIdx.x;
	const long long c1 = d.m;
	const long long nq = c1 / PRICE_NC;
	const long long nitems = nq + (c1 - nq * PRICE_NC);
	const T* const vec[3] = {d.alpha + d.row0, nullptr, nullptr};
	int buf = 0;
	for (long long g = part; g < nitems; buf ^= 1) {
		if (tid == 0) sh.tk = (long long)nparts + atomicAdd(&d.ctl->btran_ctr, 1u);
		const bool quad = g < nq;
		const long long col = quad ? g * PRICE_NC : nq * PRICE_NC + (g - nq);
		if (quad) column_dots<T, PRICE_NC, 4, 1, true>(d.B + col * d.ldb, d.ldb, d.ldb, vec, sh, buf);
		else      column_dots<T, 1, 16, 1, true>(d.B + col * d.ldb, d.ldb, d.ldb, vec, sh, buf);
		__syncthreads();
		g = sh.tk;
		if (tid < (quad ? PRICE_NC : 1)) {
			const T v = warp_sums<T>(sh, buf, tid);
			for (int r = 0; r < d.nranks; ++r) xvpart(d, r, d.rank)[col + tid] = v;
		}
		__syncthreads();
	}
}

// One rank's loop.  G / me: size of this rank's CTA group and the CTA's index in it (the whole grid on a real
// multi-GPU run; a slice of the grid when several ranks are emulated on one device).
// Per pivot: X1 after pricing, the entering column fetch + one local barrier, the update + FTRAN pass whose row
// groups push their alpha slices to every rank and run their ratio test as they complete, X2 (one record per
// rank), book1 + local barrier + X3, book2 + local barrier.
// SE: steepest-edge pricing (section "steepest-edge pricing" above).  gamma is column-sharded like A, so the weight
// recurrence needs no exchange; v = B^-T alpha does (X4): every rank pushes the column sums over ITS rows to all ranks
// beside book1, the v-flag goes out with the X3 flag, and book2 adds the R partials in rank order.
template <typename T, int WC, bool SE>
__device__ void sharded_loop(const Dev<T>& d, Smem& sh, unsigned char* ringbuf, Ring& rcons, Ring& rprod, const int G, const int me) {
	Ctl* ctl = d.ctl;
	const int tid = threadIdx.x;
	unsigned long long epoch = 0;
	unsigned long long xe = ctl->xepoch;            // serial number of the last pricing round
	unsigned long long n1 = 0, n2 = 0;              // arrival targets of X1 / X2 in this launch

	long long it = ctl->iter, pivots = ctl->pivots;
	const long long it_end = ctl->it_end;
	int pending = ctl->pending;
	int status = 0, done = 0, bad = 0, aborted = 0;
	long long p = ctl->p, q = ctl->q;
	double min_e = ctl->min_e;
	const XHdr* mine = xhdr(d, d.rank);
	bool pendg = SE && ctl->se_pending != 0;

	const long long it0 = it;
	while (it < it_end) {
		// ---- pricing over the local column block; X1
		stamp(d, it - it0, 0, me);
		++xe;
		const int par = (int)(xe & 1);
		if (SE) {
			SeUpd u;
			u.on = pendg;
			u.p = p;
			u.leaving = pendg ? __ldcg(&ctl->leaving) : -1;
			u.alpha_q = pendg ? __ldcg(&ctl->alpha_q) : 1.0;
			T gp = T(0);
			if (pendg) { T sx_, sy_; book2_scalars<T, true>(d, sh, p, sx_, sy_, &gp); }
			u.gamma_p = (double)gp;
			const T* const vec[3] = {d.y, d.row_q, d.vbt};
			price_phase_se<T>(d, sh, vec, u, me, G);
		} else if (d.price_direct) price_phase_direct<T>(d, sh, nullptr, me, G);
		else                       price_phase<T>(d, sh, ringbuf, rcons, rprod, me, G);
		stamp(d, it - it0, 1, me);
		if (arrive_last(&ctl->xarr[0], n1 += G, sh))
			publish(d, sh, 0, par, xe, d.cand, G, nullptr, (long long)*(volatile int*)&ctl->abort_req, SE ? d.cand2 : nullptr);
		long long stop;
		double sc;
		long long pse;
		if (!gather_records(d, mine->pc[par], xe, sh, min_e, p, stop, SE ? &sc : nullptr, SE ? &pse : nullptr)) { bad = 1; break; }
		if (SE) { if (pse != LLONG_MAX) p = pse; pendg = false; }
		if (me == 0 && tid == 0) { ctl->price_ctr = 0; if (SE) ctl->btran_ctr = 0; }   // every local CTA is past pricing
		stamp(d, it - it0, 2, me);
		if (stop > 0) { aborted = 1; break; }              // some rank was asked to stop: all ranks see the same sum
		if (min_e >= -d.eps) { status = 1; done = 1; ++it; break; }

		// ---- entering column from its owner, then the fused update + FTRAN + ratio test on the local rows
		const bool dense = p < d.ns;
		if (dense) {
			fetch_column<T>(d, p, me, G);
			if (!grid_barrier_t(ctl, epoch, sh, G)) { bad = 1; break; }
		}
		stamp(d, it - it0, 3, me);
		const T* acol = dense ? d.acol : nullptr;
		if (d.fuse_ratio) {
			// (experiment, off by default: the per-tile release of the group counts costs more than it saves)
			if (pending) update_ftran_phase<T, WC, true, true, true>(d, sh, ringbuf, acol, p - d.ns, pivots & 1, me, G);
			else         update_ftran_phase<T, WC, false, true, true>(d, sh, ringbuf, acol, p - d.ns, pivots & 1, me, G);
			stamp(d, it - it0, 4, me);
			if (arrive_last(&ctl->xarr[1], n2 += G, sh)) publish(d, sh, 1, 0, xe, d.rcand, d.ngrp, d.rcnt, 0);
		} else {
			if (pending) update_ftran_phase<T, WC, true, true, false>(d, sh, ringbuf, acol, p - d.ns, pivots & 1, me, G);
			else         update_ftran_phase<T, WC, false, true, false>(d, sh, ringbuf, acol, p - d.ns, pivots & 1, me, G);
			stamp(d, it - it0, 4, me);
			if (!grid_barrier_t(ctl, epoch, sh, G)) { bad = 1; break; }
			// ---- X2: alpha slices to every rank together with the ratio test of the local rows (v4:311-325)
			push_alpha_ratio<T>(d, sh, reinterpret_cast<T*>(ringbuf), me, G);
			if (arrive_last(&ctl->xarr[1], n2 += G, sh)) publish(d, sh, 1, 0, xe, d.cand, G, d.cnt, 0);
		}
		pending = 0;
		double th;
		long long elig;
		if (!gather_records(d, mine->rc, xe, sh, th, q, elig)) { bad = 1; break; }
		if (me == 0 && tid == 0) ctl->upd_ctr = 0;         // every local CTA has left the update pass
		stamp(d, it - it0, 5, me);
		if (elig == 0) { status = 2; done = 1; ++it; break; }

		// ---- pivot: E_q everywhere, X3 row q from its owner, then the replicated O(m) updates
		book1_sharded<T, SE>(d, sh, p, q, me, G);
		if (SE) btran_partial_push<T>(d, sh, me, G);       // X4 payload: v-partials of the local rows into every mailbox
		stamp(d, it - it0, 6, me);
		if (!grid_barrier_t(ctl, epoch, sh, G)) { bad = 1; break; }
		// owner: the row and its partials were stored by all local CTAs before the barrier; one
		// system-scope release covers them (release is cumulative over what the barrier acquired)
		if (me == 0 && tid < d.nranks && q >= d.row0 && q < d.row0 + d.ldb) st_release_sys(&xhdr(d, tid)->rflag, xe);
		if (SE && me == 0 && tid < d.nranks) st_release_sys(&xhdr(d, tid)->vflag[d.rank], xe);   // X4: same barrier, same release
		if (tid == 0) sh.bc_c = wait_flag_sys(&mine->rflag, xe);
		__syncthreads();
		if (!sh.bc_c) { bad = 1; break; }
		if (SE) {
			__syncthreads();
			if (tid == 0) sh.bc_c = 1;
			__syncthreads();
			if (tid < d.nranks && !wait_flag_sys(&mine->vflag[tid], xe)) sh.bc_c = 0;
			__syncthreads();
			if (!sh.bc_c) { bad = 1; break; }
			// v = sum of the R partials in rank order (same on every rank); read again a barrier from here
			for (long long j = (long long)me * NT + tid; j < d.m; j += (long long)G * NT) {
				T a = __ldcg(xvpart(d, d.rank, 0) + j);
				for (int r = 1; r < d.nranks; ++r) a = a + __ldcg(xvpart(d, d.rank, r) + j);
				d.vbt[j] = a;
			}
			pendg = true;
		}
		stamp(d, it - it0, 7, me);
		book2_phase<T>(d, sh, p, q, me, G);
		if (me == 0 && tid == 0 && pivots < d.trace_cap) d.trace[pivots] = make_int2((int)p, (int)q);
		pending = 1;
		++pivots;
		stamp(d, it - it0, 8, me);
		++it;
		if (!grid_barrier_t(ctl, epoch, sh, G)) { bad = 1; break; }
		stamp(d, it - 1 - it0, 9, me);
	}

	if (bad) { if (tid == 0) ctl->bad = 1; return; }
	if (me == 0) {
		const double z = objective<T>(d, sh);
		if (tid == 0) {
			ctl->iter = it; ctl->pivots = pivots; ctl->pending = pending;
			ctl->status = status; ctl->done = done; ctl->xepoch = xe; ctl->aborted = aborted;
			ctl->p = p; ctl->q = q; ctl->min_e = min_e; ctl->z = z;
			if (SE) ctl->se_pending = pendg ? 1 : 0;
		}
	}
}

template <typename T, int WC, bool SE = false>
__global__ void __launch_bounds__(NT, MIN_CTAS) simplex_persistent_sharded(Dev<T> d) {
	__shared__ Smem sh;
	extern __shared__ __align__(128) unsigned char ringbuf[];
	Ring rcons, rprod;
	ring_init(sh, rcons, rprod, d.price_nc);
	sharded_loop<T, WC, SE>(d, sh, ringbuf, rcons, rprod, gridDim.x, blockIdx.x);
}

// Several ranks on ONE device (tests on a single-GPU box, b200lp_create_multi with a repeated device): the
// ranks' CTA groups are slices of one cooperative grid, so they are co-resident by construction — separate
// launches that spin on each other must never share a GPU.  Same loop, same mailboxes, same flags; the "peer"
// pointers are plain device pointers.  R ranks x (gridDim.x / R) CTAs.
template <typename T, int WC, bool SE = false>
__global__ void __launch_bounds__(NT, MIN_CTAS) simplex_persistent_sharded_emu(const Dev<T>* devs, int R) {
	__shared__ Smem sh;
	extern __shared__ __align__(128) unsigned char ringbuf[];
	const int Gr = gridDim.x / R;
	const Dev<T>& d = devs[blockIdx.x / Gr];
	Ring rcons, rprod;
	ring_init(sh, rcons, rprod, d.price_nc);
	sharded_loop<T, WC, SE>(d, sh, ringbuf, rcons, rprod, Gr, blockIdx.x % Gr);
}

// ---------------------------------------------------------------- stand-alone phase kernels
// (unit tests, one-launch-per-phase mode, sharded driver).  p / q are passed by
// the host or read from ctl by the caller.

template <typename T>
__global__ void __launch_bounds__(NT) k_price(Dev<T> d) {
	__shared__ Smem sh;
	extern __shared__ __align__(128) unsigned char ringbuf[];
	Ring rcons, rprod;
	ring_init(sh, rcons, rprod, d.price_nc);
	if (d.price_direct) price_phase_direct<T>(d, sh, nullptr, blockIdx.x, gridDim.x);
	else                price_phase<T>(d, sh, ringbuf, rcons, rprod, blockIdx.x, gridDim.x);
}

// final argmin over the per-CTA candidates -> ctl->p / ctl->min_e (kind 0) or ctl->q + eligible (kind 1)
template <typename T>
__global__ void __launch_bounds__(NT) k_pick(Dev<T> d, int ncand, int kind) {
	__shared__ Smem sh;
	double v; long long i;
	reduce_cands(d.cand, ncand, v, i, sh);
	if (kind == 0) {
		if (threadIdx.x == 0) { d.ctl->p = i; d.ctl->min_e = v; }
	} else {
		const long long el = reduce_counts(d.cnt, ncand, sh);
		if (threadIdx.x == 0) { d.ctl->q = i; d.ctl->min_e = v; d.cnt[ncand] = el; }
	}
}

template <typename T, int WC, bool UPDATE, bool FTRAN>
__global__ void __launch_bounds__(NT) k_update_ftran(Dev<T> d, long long p, int reverse) {
	__shared__ Smem sh;
	extern __shared__ __align__(128) unsigned char dyn[];
	update_ftran_phase<T, WC, UPDATE, FTRAN, false>(d, sh, dyn, p < d.ns ? d.A + p * d.ld : nullptr, p - d.ns, reverse != 0, blockIdx.x, gridDim.x);
}

// alpha_part <- chunk partials of B^-1 v for an arbitrary device vector v (length ld): the FTRAN pass alone
template <typename T, int WC>
__global__ void __launch_bounds__(NT) k_ftran_vec(Dev<T> d, const T* v) {
	__shared__ Smem sh;
	extern __shared__ __align__(128) unsigned char dyn[];
	update_ftran_phase<T, WC, false, true, false>(d, sh, dyn, v, 0, false, blockIdx.x, gridDim.x);
}

// out[il] = sum of the chunk partials of local row il (left to right), il < ldb
template <typename T>
__global__ void __launch_bounds__(NT) k_sum_partials(Dev<T> d, T* out) {
	for (long long il = (long long)blockIdx.x * NT + threadIdx.x; il < d.ldb; il += (long long)gridDim.x * NT)
		out[il] = sum_chunk_partials(d.alpha_part + il, d.ldb, d.nchunk);
}

// out[j] = vec . B^-1[:, j] for the m columns of B^-1 (pricing order of the dot): y = c_b^T B^-1 after a refactorisation
template <typename T>
__global__ void __launch_bounds__(NT) k_btran_vec(Dev<T> d, const T* vec, T* out) {
	__shared__ Smem sh;
	const T* const v3[3] = {vec, nullptr, nullptr};
	int buf = 0;
	for (long long col = blockIdx.x; col < d.m; col += gridDim.x, buf ^= 1) {
		column_dots<T, 1, 16, 1, true>(d.B + col * d.ldb, d.ldb, d.ldb, v3, sh, buf);
		__syncthreads();
		if (threadIdx.x == 0) out[col] = warp_sums<T>(sh, buf, 0);
		__syncthreads();
	}
}

// dst[i] = src[i] for i < n (device vectors)
template <typename T>
__global__ void k_copy(T* dst, const T* src, long long n) {
	for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) dst[i] = src[i];
}

// B^-1 = I on the local row block (start of a refactorisation; the O(m) vectors stay)
template <typename T>
__global__ void k_identity(Dev<T> d) {
	const long long tot = d.ldb * d.m;
	for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < tot; e += (long long)gridDim.x * blockDim.x)
		d.B[e] = (d.row0 + e % d.ldb == e / d.ldb) ? T(1) : T(0);
}

template <typename T>
__global__ void __launch_bounds__(NT) k_ratio(Dev<T> d) {
	__shared__ Smem sh;
	ratio_phase<T, true>(d, sh, blockIdx.x, gridDim.x);
}

template <typename T>
__global__ void __launch_bounds__(NT) k_book1(Dev<T> d, long long p, long long q) {
	__shared__ Smem sh;
	book1_phase<T>(d, sh, p, q, blockIdx.x, gridDim.x);
}

template <typename T>
__global__ void __launch_bounds__(NT) k_book2(Dev<T> d, long long p, long long q) {
	__shared__ Smem sh;
	book2_phase<T>(d, sh, p, q, blockIdx.x, gridDim.x);
}

template <typename T>
__global__ void __launch_bounds__(NT) k_objective(Dev<T> d) {
	__shared__ Smem sh;
	const double z = objective<T>(d, sh);
	if (threadIdx.x == 0) d.ctl->z = z;
}

// ---------------------------------------------------------------- setup kernels

// steepest-edge reference framework = the slack basis (B^-1 = I): gamma_j = 1 + |a_j|^2 in the pricing order of
// the dots; unit (slack) columns 2.  One pass over the local A block.
template <typename T>
__global__ void __launch_bounds__(NT) k_gamma_init(Dev<T> d) {
	__shared__ Smem sh;
	using M = Mem<T>;
	using V = typename VecT<T>::V;
	constexpr int VN = VecT<T>::N;
	const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	for (long long col = blockIdx.x; col < d.nsl; col += gridDim.x) {
		const T* a = d.A + col * d.ld;
		T acc[VN];
#pragma unroll
		for (int v = 0; v < VN; ++v) acc[v] = T(0);
		for (long long i = (long long)tid * VN; i < d.ld; i += (long long)NT * VN) {
			const V av = M::ld_nc(a + i);
#pragma unroll
			for (int v = 0; v < VN; ++v) acc[v] = fma_t(M::get(av, v), M::get(av, v), acc[v]);
		}
		T s = acc[0];
#pragma unroll
		for (int v = 1; v < VN; ++v) s = s + acc[v];
		s = warp_butterfly_sum(s);
		__syncthreads();
		if (lane == 0) sh.wsum[0][0][warp] = (double)s;
		__syncthreads();
		if (tid == 0) d.gamma[d.col0 + col] = T(1) + warp_sums<T>(sh, 0, 0);
	}
	for (long long k = d.k0 + (long long)blockIdx.x * NT + tid; k < d.k1; k += (long long)gridDim.x * NT) d.gamma[d.ns + k] = T(2);
}

// slack-basis initial state (v4:272-277): B^-1 = I, c_b = c[n-m..n), x_b = b,
// b_ixs[j] = n-m+j, y = c_b; padding rows zero.
template <typename T>
__global__ void k_reset(Dev<T> d) {
	const long long tot = d.ldb * d.m;
	const long long stride = (long long)gridDim.x * blockDim.x;
	for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < tot; e += stride) {
		const long long i = d.row0 + e % d.ldb, j = e / d.ldb;
		d.B[e] = (i == j) ? T(1) : T(0);
	}
	for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < d.ld; i += stride) {
		const bool in = i < d.m;
		const T cb = in ? d.c[d.n - d.m + i] : T(0);
		d.c_b[i] = cb;
		d.y[i] = cb;
		d.x_b[i] = in ? d.b[i] : T(0);
		d.alpha[i] = T(0);
		d.E_q[i] = T(0);
		d.row_q[i] = T(0);
		if (in) d.b_ixs[i] = (int)(d.n - d.m + i);
	}
}

// nonbasic mask of the slack basis (dual simplex): the first n - m columns are nonbasic, the last m basic
__global__ void k_nonbasic_init(unsigned char* nb, long long n, long long m) {
	for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (long long)gridDim.x * blockDim.x)
		nb[j] = j < n - m ? 1 : 0;
}

// Cost shift of the composite method (options.cost_shift), from the slack basis: for every stored nonbasic column,
// s = y.a_j in the pricing association and e_j = s - c_j (the dual pricing's own numbers); where e_j < -eps,
// c_j <- s - delta (1 + |c_j|) (a product rounded on its own, never fused into the subtraction) and the column is
// counted.  Unit (slack) columns are basic at the start and are not visited.  c is rewritten in place: the caller
// keeps the original.
template <typename T>
__global__ void __launch_bounds__(NT) k_cost_shift(Dev<T> d, T* c, const unsigned char* nb, T delta,
		unsigned long long* shifted) {
	__shared__ Smem sh;
	const T* const v3[3] = {d.y, nullptr, nullptr};
	int buf = 0;
	for (long long col = blockIdx.x; col < d.nsl; col += gridDim.x, buf ^= 1) {
		const long long j = d.col0 + col;
		if (!nb[j]) continue;                         // the same for the whole CTA
		column_dots<T, 1, 16, 1, false>(d.A + col * d.ld, d.ld, d.ld, v3, sh, buf);
		__syncthreads();
		if (threadIdx.x == 0) {
			const T s = warp_sums<T>(sh, buf, 0);
			const T cj = c[j];
			if ((double)(s - cj) < -d.eps) {
				c[j] = s - mul_rn_t(delta, T(1) + (cj < T(0) ? -cj : cj));
				atomicAdd(shifted, 1ull);
			}
		}
		__syncthreads();
	}
}

// c_b[i] = c[b_ixs[i]] (hand-over of the composite method: the basis costs of the original c)
template <typename T>
__global__ void k_gather_cb(T* c_b, const T* c, const int* b_ixs, long long m) {
	for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += (long long)gridDim.x * blockDim.x)
		c_b[i] = c[b_ixs[i]];
}

__host__ __device__ __forceinline__ uint64_t mix64(uint64_t z) {
	z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
	z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
	return z ^ (z >> 31);
}
__host__ __device__ __forceinline__ double u01(uint64_t seed, uint64_t stream, uint64_t idx) {
	uint64_t z = mix64(seed * 0x9E3779B97F4A7C15ULL + stream * 0xD1B54A32D192ED03ULL + 0x632BE59BD9B4E019ULL);
	z = mix64(z + idx * 0x9E3779B97F4A7C15ULL);
	return (double)(z >> 11) * (1.0 / 9007199254740992.0);
}

// dense synthetic LP (same numbers as oracle/lpgen_dense_*): A_s ~ U(0,1),
// b = (ns/2) U(1,2), c_s ~ U(0.5,1.5), slack costs 0
template <typename T>
__global__ void k_generate_dense(T* A, T* b, T* c, long long m, long long n, long long ns, long long ld, uint64_t seed,
		long long col0, long long nsl) {
	const long long stride = (long long)gridDim.x * blockDim.x;
	const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
	const long long tot = ld * nsl;           // this rank's column block [col0, col0 + nsl)
	for (long long e = g; e < tot; e += stride) {
		const long long i = e % ld, j = col0 + e / ld;
		A[e] = i < m ? (T)u01(seed, 0, (uint64_t)(i * ns + j)) : T(0);
	}
	for (long long i = g; i < ld; i += stride) b[i] = i < m ? (T)(0.5 * (double)ns * (1.0 + u01(seed, 1, (uint64_t)i))) : T(0);
	for (long long j = g; j < n; j += stride) c[j] = j < ns ? (T)(0.5 + u01(seed, 2, (uint64_t)j)) : T(0);
}

// zero the padding rows [m, ld) of an ld x ncols column-major matrix
template <typename T>
__global__ void k_zero_pad(T* X, long long m, long long ld, long long ncols) {
	const long long pad = ld - m;
	const long long tot = pad * ncols;
	const long long stride = (long long)gridDim.x * blockDim.x;
	for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < tot; e += stride) {
		const long long i = m + e % pad, j = e / pad;
		X[i + j * ld] = T(0);
	}
}

} // namespace b200lp
