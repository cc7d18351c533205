// Host side of the B200 dense revised-simplex engine and its C ABI
// (include/b200lp.h).  Replaces the host half of the reference's solve()
// (src/v4_cub_reduction.cu:219-380): allocation (v4:245-264), H2D + initial
// state (v4:269-279), the loop driver (v4:286-359, here ONE cooperative
// launch) and the read-back (v4:362-368).  No cuBLAS, no CUB, no CPU fallback.
#include "../../include/b200lp.h"
#include "kernels.cuh"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

using namespace b200lp;

static thread_local std::string g_err;

static int fail(int code, const std::string& msg) {
	g_err = msg;
	return code;
}

#define CU(call)                                                                          \
	do {                                                                                  \
		cudaError_t e_ = (call);                                                          \
		if (e_ != cudaSuccess)                                                            \
			return fail(B200LP_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
	} while (0)

struct b200lp_engine {
	virtual ~b200lp_engine() {}
	virtual int upload(const void* A, const void* b, const void* c) = 0;
	virtual int upload_unchecked(const void* A, const void* b, const void* c) = 0;
	virtual bool slack_is_identity(const void* A) const = 0;
	virtual int upload_columns(const void* Acols, int64_t col0, int64_t ncols, const void* b, const void* c) = 0;
	virtual int shard_columns(int64_t* col0, int64_t* ncols) = 0;
	virtual int generate_dense(uint64_t seed) = 0;
	virtual int reset() = 0;
	virtual int run_async(int64_t iters) = 0;
	virtual int wait(b200lp_result* res) = 0;
	virtual int download(void* x_b, int32_t* b_ixs, void* y) = 0;
	virtual int download_binv(void* Binv) = 0;
	virtual int download_trace(int32_t* pq, int64_t cap, int64_t* n_out) = 0;
	virtual int phase_price(int64_t* p, double* min_e) = 0;
	virtual int phase_update_ftran(int64_t p) = 0;
	virtual int phase_ratio(int64_t* q, int64_t* eligible) = 0;
	virtual int phase_pivot_update(int64_t p, int64_t q) = 0;
	virtual int download_vector(int32_t which, void* out) = 0;
	virtual int64_t bytes_per_pivot() const = 0;
	virtual int ipc_export(void* out) = 0;
	virtual int ipc_import(const void* all, int nranks) = 0;
	virtual int shard_rows(int64_t* row0, int64_t* rows) = 0;
	virtual int download_profile(uint64_t* out, int64_t cap_iters, int64_t* n_iters) = 0;
	virtual int check_basis(double* xb_err, double* xb_scale) = 0;
	virtual int abort() = 0;
	virtual int refactor(double rel_pivot_tol, int64_t* replayed) = 0;
	// composite method (options.cost_shift): only the single-GPU engine has phases
	virtual int phase_info(int32_t* phase, int64_t* shifted, int64_t* phase1_pivots) {
		if (phase) *phase = 0;
		if (shifted) *shifted = 0;
		if (phase1_pivots) *phase1_pivots = 0;
		return B200LP_OK;
	}
	cudaStream_t stream = nullptr;
	int rank = 0, nranks = 1;
	int grid = 0;
	long long ns = 0;
	double ms_upload = 0;
};

namespace {

template <typename T> class MultiEngine;
template <typename T> class BatchCall;

// tiny LPs: ld is one warp-wide vector row (m <= 64 doubles / 128 floats) and A (ns stored columns), B^-1 and the
// vectors fit in one CTA's shared memory.  Asked by the single engine (simplex_tiny) and by the batched call
// (simplex_tiny_batch, ns = the largest of the batch).
template <typename T>
bool tiny_fits(long long m, long long n, long long ns) {
	if (m > TinyLayout<T>::LD) return false;
	return TinyLayout<T>(m, n, ns).bytes(m) <= (size_t)200 * 1024;
}

// the same question for simplex_tiny_batch_dual (dual simplex / composite batches), whose layout adds the nonbasic
// mask: a shape can fit tiny_fits and not this
template <typename T>
bool tiny_dual_fits(long long m, long long n, long long ns) {
	if (m > TinyLayout<T>::LD) return false;
	return TinyDualLayout<T>(m, n, ns).bytes(m, n) <= (size_t)200 * 1024;
}

// options.algorithm against the rest of the options and the number of GPUs; host only, before any device call
int check_algorithm(const b200lp_options& o, int ngpus) {
	if (o.algorithm != 0 && o.algorithm != 1) return fail(B200LP_ERR_ARG, "algorithm must be 0 (primal) or 1 (dual)");
	if (o.algorithm == 0) return B200LP_OK;
	if (o.pricing_rule != 0) return fail(B200LP_ERR_ARG, "the dual simplex (algorithm = 1) needs pricing_rule = 0");
	if (o.ratio_mode != 0) return fail(B200LP_ERR_ARG, "the dual simplex (algorithm = 1) needs ratio_mode = 0");
	if (o.mode != 0) return fail(B200LP_ERR_ARG, "the dual simplex (algorithm = 1) needs the persistent kernel (mode = 0)");
	if (o.fuse_ratio > 0) return fail(B200LP_ERR_ARG, "the dual simplex (algorithm = 1) has no fused ratio test (fuse_ratio > 0)");
	if (ngpus > 1) return fail(B200LP_ERR_ARG, "the dual simplex (algorithm = 1) runs on one GPU");
	return B200LP_OK;
}

// options.cost_shift / shift_delta (composite method: dual phase on shifted costs, then primal); after check_algorithm
int check_cost_shift(const b200lp_options& o) {
	if (o.cost_shift != 0 && o.cost_shift != 1) return fail(B200LP_ERR_ARG, "cost_shift must be 0 (off) or 1 (on)");
	if (!(o.shift_delta >= 0)) return fail(B200LP_ERR_ARG, "shift_delta must be >= 0 (0 = default) and not NaN");
	if (o.cost_shift == 1 && o.algorithm != 1) return fail(B200LP_ERR_ARG, "cost_shift = 1 needs the dual simplex (algorithm = 1)");
	return B200LP_OK;
}

template <typename T>
class Engine final : public b200lp_engine {
	friend class MultiEngine<T>;
	friend class BatchCall<T>;
public:
	Engine(int64_t m, int64_t n, const b200lp_options& o, int rank_, int nranks_) : opt(o) {
		std::memset(&d, 0, sizeof(d));
		std::memset(&dd, 0, sizeof(dd));
		std::memset(&hc, 0, sizeof(hc));
		rank = rank_;
		nranks = nranks_;
		d.m = m;
		d.n = n;
		constexpr long long rowq = 32 * VecT<T>::N;
		d.ld = (m + rowq - 1) / rowq * rowq;
		// row blocks of B^-1: equal multiples of one warp-wide vector row, the tail ranks may own fewer (or no) rows
		d.rank = rank;
		d.nranks = nranks;
		const long long rpr = ((d.ld + nranks - 1) / nranks + rowq - 1) / rowq * rowq;
		for (int r = 0; r <= nranks; ++r) d.rowstart[r] = std::min<long long>(d.ld, (long long)r * rpr);
		d.row0 = d.rowstart[rank];
		d.ldb = d.rowstart[rank + 1] - d.rowstart[rank];
		d.nchunk = (int)((m + CHUNK - 1) / CHUNK);
		d.nslice = (int)((m + SLICE - 1) / SLICE);
		d.eps = sizeof(T) == 4 ? (double)(float)o.eps : o.eps;
		d.trace_cap = std::max<int64_t>(1, std::min<int64_t>(o.max_iter, (int64_t)1 << 22));
	}

	~Engine() override { release(); }

	int init() {
		CU(cudaSetDevice(opt.device));
		cudaDeviceProp prop;
		CU(cudaGetDeviceProperties(&prop, opt.device));
		if (prop.major < 10)
			return fail(B200LP_ERR_NO_GPU, std::string("device is sm_") + std::to_string(prop.major * 10 + prop.minor) +
				", the engine is built for sm_100a only");
		num_sms = prop.multiProcessorCount;
		CU(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
		CU(cudaEventCreate(&ev0));
		CU(cudaEventCreate(&ev1));

		const size_t ld = (size_t)d.ld, m = (size_t)d.m;
		// B^-1 (the big one: 8 GB at m = 32768) is allocated at first use, i.e. AFTER the upload of A has been put on
		// the wire, so that the allocation overlaps the DMA instead of preceding it (ensure_B)
		T* vecs[6];
		for (auto& v : vecs) CU(alloc(&v, ld));
		d.b = vecs[0]; hb = vecs[0];
		d.y = vecs[1]; d.x_b = vecs[2]; d.c_b = vecs[3]; d.E_q = vecs[4]; d.acol = vecs[5];
		// mailbox: [XHdr][alpha ld][row_q ld][row_q.b slice partials]; peers store into it in sharded mode (IPC-exported)
		// steepest edge on several ranks: + R partial vectors of v = B^-T alpha (X4)
		const size_t rqb_len = ((size_t)d.nslice + 64 + 3) / 4 * 4;
		d.vpart_off = (long long)(2 * ld + rqb_len);
		mbox_bytes = sizeof(XHdr) + (2 * ld + rqb_len + (opt.pricing_rule == 1 && nranks > 1 ? (size_t)nranks * ld : 0)) * sizeof(T);
		CU(alloc(&mbox, mbox_bytes));
		CU(cudaMemsetAsync(mbox, 0, mbox_bytes, stream));
		d.alpha = reinterpret_cast<T*>(mbox + sizeof(XHdr));
		d.row_q = d.alpha + ld;
		for (int r = 0; r < MAXR; ++r) { d.mbox_peer[r] = nullptr; d.A_peer[r] = nullptr; }
		d.mbox_peer[rank] = mbox;
		CU(alloc(&hcst, (size_t)d.n));
		d.c = hcst;
		CU(alloc(&d.alpha_part, (size_t)d.nchunk * (size_t)d.ldb));
		CU(alloc(&d.dpart, (size_t)3 * d.nslice));
		d.pricing_rule = opt.pricing_rule;
		if (opt.pricing_rule == 1) {
			if (opt.mode != 0) return fail(B200LP_ERR_ARG, "steepest-edge pricing needs the persistent kernel (mode = 0)");
			CU(alloc(&d.gamma, (size_t)d.n));
			CU(alloc(&d.vbt, ld));
			CU(cudaMemsetAsync(d.vbt, 0, ld * sizeof(T), stream));
		} else if (opt.pricing_rule != 0) return fail(B200LP_ERR_ARG, "pricing_rule must be 0 (Dantzig) or 1 (steepest edge)");
		d.dpart0 = nranks > 1 ? d.row_q + ld : d.dpart;
		CU(alloc(&d.b_ixs, m));
		CU(alloc(&d.ctl, 1));
		CU(alloc(&d.trace, (size_t)d.trace_cap));
		CU(cudaMemsetAsync(d.ctl, 0, sizeof(Ctl), stream));
		CU(cudaMallocHost(&pinned, sizeof(Ctl) + 64));
		if (opt.profile > 0) {
			d.prof_cap = std::min<int64_t>(opt.profile, 1 << 16);
			CU(alloc(&d.prof, (size_t)d.prof_cap * NSTAMP));
		}

		// L2 residency: pin the head of B^-1 in the persisting part of L2 so that it never makes the trip to HBM
		// (B^-1 is read and rewritten once per pivot; A streams through with evict_first)
		if (opt.l2_persist_mb >= 0) {
			CU(ensure_B());
			int max_persist = 0, max_window = 0;
			CU(cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, opt.device));
			CU(cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, opt.device));
			size_t want = opt.l2_persist_mb > 0 ? (size_t)opt.l2_persist_mb << 20 : (size_t)max_persist;
			want = std::min({want, (size_t)max_persist, (size_t)max_window, (size_t)d.ldb * m * sizeof(T)});
			if (want >= ((size_t)4 << 20) && (size_t)d.ldb * m * sizeof(T) > ((size_t)64 << 20)) {
				CU(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want));
				cudaStreamAttrValue av;
				std::memset(&av, 0, sizeof(av));
				av.accessPolicyWindow.base_ptr = d.B;
				av.accessPolicyWindow.num_bytes = want;
				av.accessPolicyWindow.hitRatio = 1.0f;
				av.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
				av.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
				CU(cudaStreamSetAttribute(stream, cudaStreamAttributeAccessPolicyWindow, &av));
				l2_persist_bytes = want;
			}
		}

		// persistent grid: co-resident CTAs only (cooperative launch)
		// the pricing ring lives in dynamic shared memory (above the 48 KB default limit)
		for (const void* fn : {(const void*)simplex_persistent<T, 1>, (const void*)simplex_persistent<T, 2>,
				(const void*)simplex_persistent<T, 4>, (const void*)simplex_persistent<T, 8>,
				(const void*)simplex_persistent_sharded<T, 1>, (const void*)simplex_persistent_sharded<T, 2>,
				(const void*)simplex_persistent_sharded<T, 4>, (const void*)simplex_persistent_sharded<T, 8>,
				(const void*)simplex_persistent_sharded<T, 1, true>, (const void*)simplex_persistent_sharded<T, 2, true>,
				(const void*)simplex_persistent_sharded<T, 4, true>, (const void*)simplex_persistent_sharded<T, 8, true>,
				(const void*)simplex_persistent<T, 1, true>, (const void*)simplex_persistent<T, 2, true>,
				(const void*)simplex_persistent<T, 4, true>, (const void*)simplex_persistent<T, 8, true>,
				(const void*)k_price<T>})
			CU(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, DYN_SMEM_BYTES));
		int occ = 0;
		if (opt.algorithm == 1 && opt.cost_shift == 1) {   // phase 2 launches the primal kernel on the same grid
			int occ2 = 0;
			CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, simplex_dual<T, 1>, NT, UF_SMEM_BYTES));
			CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ2, simplex_persistent<T, 1>, NT, DYN_SMEM_BYTES));
			occ = std::min(occ, occ2);
		}
		else if (opt.algorithm == 1) CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, simplex_dual<T, 1>, NT, UF_SMEM_BYTES));
		else if (nranks > 1 && opt.pricing_rule == 1) CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, simplex_persistent_sharded<T, 1, true>, NT, DYN_SMEM_BYTES));
		else if (nranks > 1) CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, simplex_persistent_sharded<T, 1>, NT, DYN_SMEM_BYTES));
		else if (opt.pricing_rule == 1) CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, simplex_persistent<T, 1, true>, NT, DYN_SMEM_BYTES));
		else            CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, simplex_persistent<T, 1>, NT, DYN_SMEM_BYTES));
		if (occ < 1) return fail(B200LP_ERR_CUDA, "persistent kernel does not fit on an SM");
		max_grid = occ * num_sms;
		const double work = (double)d.ld * (double)d.n / nranks;
		int g;
		if (opt.grid_ctas > 0) g = opt.grid_ctas;
		else if (work <= 64.0 * 1024) g = 1;                       // tiny LPs: barriers are pure latency
		else if (work <= 4.0 * 1024 * 1024) g = num_sms;
		else g = num_sms * std::min(occ, 4);
		grid = std::max(1, std::min(g, max_grid));
		CU(alloc(&d.cand, (size_t)max_grid + 2));
		CU(alloc(&d.cand2, (size_t)2 * (max_grid + 2)));
		CU(alloc(&d.cnt, (size_t)max_grid + 2));
		if (opt.algorithm == 1) {                         // dual simplex: nonbasic mask, rho, leaving-row candidates
			CU(alloc(&dd.nb, (size_t)d.n));
			CU(alloc(&dd.rho, ld));
			CU(cudaMemsetAsync(dd.rho, 0, ld * sizeof(T), stream));
			CU(alloc(&dd.lcand, (size_t)max_grid + 2));
		}
		if (opt.cost_shift == 1) {                        // composite method: the original c, the shifted-column count
			CU(alloc(&c_orig, (size_t)d.n));
			CU(alloc(&d_shifted, 1));
		}

		// tile shape of the update+FTRAN pass: tiles are handed out dynamically, so the tallest row
		// tile that still leaves every CTA ~100 tiles keeps the tail of the pass well under 1 %
		// (measured: C3 best with 64-row tiles, C4 with 128-row tiles)
		wc = 8;
		for (int cand_wc : {1, 2, 4, 8}) {
			const long long tr = (long long)(NWARP / cand_wc) * 32 * VecT<T>::N;
			const long long tiles = (d.ldb + tr - 1) / tr * d.nchunk;
			if (tiles >= 96LL * grid) { wc = cand_wc; break; }
		}
		if (opt.tile_shape == 1 || opt.tile_shape == 2 || opt.tile_shape == 4 || opt.tile_shape == 8) wc = opt.tile_shape;
		// row groups of the update+FTRAN pass: the ratio test of a group runs as soon as its last tile is done
		{
			const long long tr = (long long)(NWARP / wc) * 32 * VecT<T>::N;
			const long long ntr = (d.ldb + tr - 1) / tr;
			const long long want = opt.ratio_group_rows > 0 ? opt.ratio_group_rows : 256;
			d.rg = (int)std::max<long long>(1, want / tr);
			d.ngrp = (int)((ntr + d.rg - 1) / d.rg);              // 0: this rank owns no rows (more ranks than row blocks)
			CU(alloc(&d.rcand, (size_t)d.ngrp + 1));
			CU(alloc(&d.rcnt, (size_t)d.ngrp + 1));
			CU(alloc(&d.grp_done, (size_t)d.ngrp + 1));
			CU(cudaMemsetAsync(d.grp_done, 0, ((size_t)d.ngrp + 1) * sizeof(unsigned int), stream));
		}
		d.pivot_tol = sizeof(T) == 4 ? (double)(float)opt.pivot_tol : opt.pivot_tol;
		d.ratio_mode = opt.ratio_mode;
		d.harris_delta = sizeof(T) == 4 ? (double)(float)opt.harris_delta : opt.harris_delta;
		if (opt.ratio_mode < 0 || opt.ratio_mode > 2) return fail(B200LP_ERR_ARG, "ratio_mode must be 0, 1 or 2");
		if (opt.ratio_mode == 2 && (nranks > 1 || opt.mode != 0 || opt.fuse_ratio > 0))
			return fail(B200LP_ERR_ARG, "the Harris ratio test (ratio_mode = 2) needs the single-GPU persistent kernel with the ratio test as its own phase");
		d.fuse_ratio = opt.fuse_ratio > 0 ? 1 : 0;    // measured: the per-tile release costs more than the phase it saves
		return B200LP_OK;
	}

	// ---- data in -------------------------------------------------------

	int upload(const void* Av, const void* bv, const void* cv) override {
		const T* A = static_cast<const T*>(Av);
		const long long m = d.m, n = d.n;
		CU(cudaSetDevice(opt.device));
		// Is the last m x m block the identity the reference assumes (v4:272)?  If so those columns are
		// priced and FTRAN'd as unit vectors and never stored.  The check reads m*m host elements (8.6 GB at
		// m = 32768), so the structural columns are put on the wire first and the check runs on the host
		// threads while the DMA engine works (pinned memory; a pageable copy simply finishes first).
		if (opt.check_slack) {
			CU(set_columns(n - m));
			int rc = enqueue_block(A + (size_t)d.col0 * m, bv, cv);
			if (rc) return rc;
			if (host_is_identity(A + (size_t)(n - m) * m, m)) return finish_upload();
			CU(cudaStreamSynchronize(stream));       // rare: the block is data, store and price all n columns
		}
		CU(set_columns(opt.check_slack ? n : n - m));
		return upload_block(A + (size_t)d.col0 * m, bv, cv);
	}

	// the structural columns only, trusting the identity slack block for now (solve_once checks it while the
	// GPU is already pivoting and starts over in the rare case that the block is data)
	int upload_unchecked(const void* Av, const void* bv, const void* cv) override {
		const T* A = static_cast<const T*>(Av);
		CU(cudaSetDevice(opt.device));
		CU(set_columns(d.n - d.m));
		return upload_block(A + (size_t)d.col0 * d.m, bv, cv);
	}

	bool slack_is_identity(const void* Av) const override {
		return host_is_identity(static_cast<const T*>(Av) + (size_t)(d.n - d.m) * d.m, d.m);
	}

	// sharded front door: the caller hands over only this rank's structural columns
	// [col0, col0 + ncols) (column-major m x ncols) and vouches for the identity slack block
	int upload_columns(const void* Acols, int64_t col0, int64_t ncols, const void* bv, const void* cv) override {
		CU(cudaSetDevice(opt.device));
		CU(set_columns(d.n - d.m));
		if (col0 != d.col0 || ncols != d.nsl)
			return fail(B200LP_ERR_ARG, "upload_columns: block is not this rank's column shard (see b200lp_shard_columns)");
		return upload_block(Acols, bv, cv);
	}

	// multi-GPU front door inside one process: the caller holds the whole host matrix and says how many of its
	// leading columns are data (n - m with an identity slack block, n otherwise); this rank takes its block
	int upload_shard(const void* A_full, long long ns_new, const void* bv, const void* cv) {
		CU(cudaSetDevice(opt.device));
		if (int rc = settle()) return rc;
		CU(set_columns(ns_new));
		return upload_block(static_cast<const T*>(A_full) + (size_t)d.col0 * d.m, bv, cv);
	}

	int upload_block(const void* Av, const void* bv, const void* cv) {
		int rc = enqueue_block(Av, bv, cv);
		return rc ? rc : finish_upload();
	}

	// H2D of this rank's column block, b and c: enqueued on the engine's stream, not waited for
	int enqueue_block(const void* Av, const void* bv, const void* cv) {
		const T* A = static_cast<const T*>(Av);          // first column of this rank's block
		const T* b = static_cast<const T*>(bv);
		const T* c = static_cast<const T*>(cv);
		const long long m = d.m, n = d.n, ld = d.ld;
		if (int rc = settle()) return rc;              // a composite run in flight may still write c (hand-over)
		CU(cudaEventRecord(ev0, stream));
		if (d.nsl > 0)
			CU(cudaMemcpy2DAsync(hA, ld * sizeof(T), A, m * sizeof(T), m * sizeof(T), (size_t)d.nsl,
				cudaMemcpyHostToDevice, stream));
		CU(cudaMemsetAsync(hb, 0, ld * sizeof(T), stream));
		CU(cudaMemcpyAsync(hb, b, m * sizeof(T), cudaMemcpyHostToDevice, stream));
		CU(cudaMemcpyAsync(hcst, c, n * sizeof(T), cudaMemcpyHostToDevice, stream));
		c_shifted = false;
		if (ld > m && d.nsl > 0) {
			k_zero_pad<T><<<num_sms * 4, 256, 0, stream>>>(hA, m, ld, d.nsl);
			launches++;
		}
		CU(cudaEventRecord(ev1, stream));
		CU(ensure_B());                 // while the copies are on the wire
		return B200LP_OK;
	}

	// slack-basis initial state, then wait for the copies
	int finish_upload() {
		have_data = true;
		int rc = reset();
		if (rc) return rc;
		CU(cudaStreamSynchronize(stream));
		float ms = 0;
		CU(cudaEventElapsedTime(&ms, ev0, ev1));
		ms_upload = ms;
		return B200LP_OK;
	}

	int generate_dense(uint64_t seed) override {
		CU(cudaSetDevice(opt.device));
		if (int rc = settle()) return rc;
		CU(set_columns(d.n - d.m));
		k_generate_dense<T><<<num_sms * 8, 256, 0, stream>>>(hA, hb, hcst, d.m, d.n, d.ns, d.ld, seed, d.col0, d.nsl);
		launches++;
		CU(cudaGetLastError());
		c_shifted = false;
		have_data = true;
		return reset();
	}

	cudaError_t ensure_B() {
		if (d.B) return cudaSuccess;
		return alloc(&d.B, (size_t)d.ldb * (size_t)d.m);
	}

	// a launch may still be running: the host mirror of the control block (pending, xepoch, counters) is only
	// valid after wait()
	int settle() { return in_flight ? wait(nullptr) : B200LP_OK; }

	int reset() override {
		if (!have_data) return fail(B200LP_ERR_STATE, "reset before upload/generate");
		CU(cudaSetDevice(opt.device));
		if (int rc = settle()) return rc;
		CU(ensure_B());
		if (c_shifted) {                                   // composite method: back to the original c before c_b, y
			CU(cudaMemcpyAsync(hcst, c_orig, (size_t)d.n * sizeof(T), cudaMemcpyDeviceToDevice, stream));
			c_shifted = false;
		}
		phase = 0;
		shifted_cols = ph1_pivots = 0;
		k_reset<T><<<num_sms * 8, 256, 0, stream>>>(d);
		launches++;
		if (opt.pricing_rule == 1) {                       // steepest edge: the weights start over with the slack basis
			k_gamma_init<T><<<num_sms * 4, NT, 0, stream>>>(d);
			launches++;
		}
		if (opt.algorithm == 1) {                          // dual simplex: the slack basis's nonbasic columns
			k_nonbasic_init<<<num_sms, 256, 0, stream>>>(dd.nb, d.n, d.m);
			launches++;
		}
		CU(cudaGetLastError());
		const unsigned long long xe = hc.xepoch;    // the peer-barrier epoch outlives a reset
		std::memset(&hc, 0, sizeof(hc));
		hc.xepoch = xe;
		CU(push_ctl());
		return B200LP_OK;
	}

	// ---- the loop ------------------------------------------------------

	// everything of run_async up to the launch: 1 = nothing to launch (done / no iterations), 0 = go, < 0 error
	int prepare_run(int64_t iters) {
		if (!have_data) return fail(B200LP_ERR_STATE, "run before upload/generate");
		CU(cudaSetDevice(opt.device));
		if (int rc = settle()) return rc;
		in_flight = true;
		if (hc.done || iters <= 0) {
			CU(cudaEventRecord(ev0, stream));
			CU(cudaEventRecord(ev1, stream));
			return 1;
		}
		if (opt.mode == 1 && nranks == 1) { int rc = run_phases(iters); return rc ? rc : 1; }
		if (tiny_ok()) { int rc = run_tiny(iters); return rc ? rc : 1; }
		if (resident_ok()) { int rc = run_resident(iters); return rc ? rc : 1; }
		hc.it_end = hc.iter + iters;
		CU(push_ctl());
		if (d.prof_cap > 0) CU(cudaMemsetAsync(d.prof, 0, (size_t)d.prof_cap * NSTAMP * sizeof(unsigned long long), stream));
		prof_iter0 = hc.iter;
		CU(cudaEventRecord(ev0, stream));
		if (opt.cost_shift == 1 && phase == 0) {           // first run from the slack basis: shift, then phase 1
			if (int rc = shift_costs()) return rc;
		}
		return 0;
	}

	int run_async(int64_t iters) override {
		const int pr = prepare_run(iters);
		if (pr != 0) return pr < 0 ? pr : B200LP_OK;
		void* args[] = {&d};
		const void* fn;
		if (!primal_loop()) {                      // dual simplex: its own loop kernel at every size
			void* dargs[] = {&d, &dd};
			fn = wc == 1 ? (const void*)simplex_dual<T, 1>
			   : wc == 2 ? (const void*)simplex_dual<T, 2>
			   : wc == 4 ? (const void*)simplex_dual<T, 4>
			             : (const void*)simplex_dual<T, 8>;
			CU(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(NT), dargs, UF_SMEM_BYTES, stream));
			launches++;
			CU(cudaEventRecord(ev1, stream));
			return B200LP_OK;
		}
		if (nranks > 1) {
			if (!peers_mapped) return fail(B200LP_ERR_STATE, "sharded engine: peers are not mapped (ipc_import / create_multi)");
			if (opt.pricing_rule == 1)
				fn = wc == 1 ? (const void*)simplex_persistent_sharded<T, 1, true>
				   : wc == 2 ? (const void*)simplex_persistent_sharded<T, 2, true>
				   : wc == 4 ? (const void*)simplex_persistent_sharded<T, 4, true>
				             : (const void*)simplex_persistent_sharded<T, 8, true>;
			else
				fn = wc == 1 ? (const void*)simplex_persistent_sharded<T, 1>
				   : wc == 2 ? (const void*)simplex_persistent_sharded<T, 2>
				   : wc == 4 ? (const void*)simplex_persistent_sharded<T, 4>
				             : (const void*)simplex_persistent_sharded<T, 8>;
		} else if (opt.pricing_rule == 1) {
			fn = wc == 1 ? (const void*)simplex_persistent<T, 1, true>
			   : wc == 2 ? (const void*)simplex_persistent<T, 2, true>
			   : wc == 4 ? (const void*)simplex_persistent<T, 4, true>
			             : (const void*)simplex_persistent<T, 8, true>;
		} else {
			fn = wc == 1 ? (const void*)simplex_persistent<T, 1>
			   : wc == 2 ? (const void*)simplex_persistent<T, 2>
			   : wc == 4 ? (const void*)simplex_persistent<T, 4>
			             : (const void*)simplex_persistent<T, 8>;
		}
		CU(cudaLaunchCooperativeKernel(fn, dim3(grid), dim3(NT), args, DYN_SMEM_BYTES, stream));
		launches++;
		CU(cudaEventRecord(ev1, stream));
		return B200LP_OK;
	}

	// ask the running loop to stop at its next iteration boundary: one word written by a copy on a second stream
	int abort() override {
		CU(cudaSetDevice(opt.device));
		if (!in_flight) return B200LP_OK;
		abort_asked = true;                        // also keeps wait() from starting phase 2 of the composite method
		if (!abort_stream) CU(cudaStreamCreateWithFlags(&abort_stream, cudaStreamNonBlocking));
		int* one = reinterpret_cast<int*>(static_cast<unsigned char*>(pinned) + sizeof(Ctl));
		*one = 1;
		CU(cudaMemcpyAsync(reinterpret_cast<unsigned char*>(d.ctl) + offsetof(Ctl, abort_req), one, sizeof(int),
			cudaMemcpyHostToDevice, abort_stream));
		CU(cudaStreamSynchronize(abort_stream));
		return B200LP_OK;
	}

	int wait(b200lp_result* res) override {
		CU(cudaSetDevice(opt.device));
		CU(cudaStreamSynchronize(stream));
		CU(cudaGetLastError());
		float ms = 0;
		bool was_aborted = false;
		if (in_flight) {
			CU(cudaEventElapsedTime(&ms, ev0, ev1));
			CU(pull_ctl());
			was_aborted = hc.aborted != 0;
			hc.abort_req = hc.abort_latched = hc.aborted = 0;
		}
		in_flight = false;
		if (hc.bad) return fail(B200LP_ERR_CUDA, "sharded engine: a peer GPU did not answer within 20 s (the engine must be destroyed)");
		ms_run += ms;
		if (opt.cost_shift == 1 && phase == 1) {
			if (shift_unread) {
				unsigned long long k = 0;
				CU(cudaMemcpy(&k, d_shifted, sizeof(k), cudaMemcpyDeviceToHost));
				shifted_cols = (int64_t)k;
				shift_unread = false;
			}
			ph1_pivots = hc.pivots;
			// phase 1 at the optimum of c': hand over to the primal loop, and run it with what is left of the budget
			if (hc.done && hc.status == B200LP_STATUS_OPTIMUM && shifted_cols > 0) {
				if (int rc = hand_over()) return rc;
				if (abort_asked) was_aborted = true;
				else if (hc.it_end > hc.iter) {
					if (int rc = run_async(hc.it_end - hc.iter)) return rc;
					return wait(res);
				}
			}
		}
		abort_asked = false;
		if (res) {
			std::memset(res, 0, sizeof(*res));
			res->status = hc.status;
			res->aborted = was_aborted ? 1 : 0;
			res->iterations = hc.iter;
			res->pivots = hc.pivots;
			res->z = hc.z;
			res->min_reduced_cost = hc.min_e;
			res->ms_solve = ms_run;
			res->ms_upload = ms_upload;
			res->kernel_launches = launches;
		}
		ms_run = 0;
		return B200LP_OK;
	}

	int phase_info(int32_t* ph, int64_t* shifted, int64_t* phase1_pivots) override {
		if (ph) *ph = phase;
		if (shifted) *shifted = shifted_cols;
		if (phase1_pivots) *phase1_pivots = ph1_pivots;
		return B200LP_OK;
	}

	// ---- data out ------------------------------------------------------

	int download(void* x_b, int32_t* b_ixs, void* y) override {
		CU(cudaSetDevice(opt.device));
		CU(cudaStreamSynchronize(stream));
		if (x_b) CU(cudaMemcpy(x_b, d.x_b, d.m * sizeof(T), cudaMemcpyDeviceToHost));
		if (b_ixs) CU(cudaMemcpy(b_ixs, d.b_ixs, d.m * sizeof(int), cudaMemcpyDeviceToHost));
		if (y) CU(cudaMemcpy(y, d.y, d.m * sizeof(T), cudaMemcpyDeviceToHost));
		return B200LP_OK;
	}

	int download_binv(void* Binv) override {
		CU(cudaSetDevice(opt.device));
		if (int rc = settle()) return rc;
		CU(cudaStreamSynchronize(stream));
		if (hc.pending) {
			launch_update_ftran(true, false, 0);
			CU(cudaGetLastError());
			hc.pending = 0;
			CU(push_ctl());
		}
		CU(cudaStreamSynchronize(stream));
		// the local row block [row0, row0 + rows) as a rows x m column-major matrix (all of B^-1 on one GPU)
		const long long rows = std::max<long long>(0, std::min<long long>(d.m, d.row0 + d.ldb) - d.row0);
		if (rows > 0)
			CU(cudaMemcpy2D(Binv, rows * sizeof(T), d.B, d.ldb * sizeof(T), rows * sizeof(T), (size_t)d.m, cudaMemcpyDeviceToHost));
		return B200LP_OK;
	}

	// numerical health of the product-form inverse: max_i |(B^-1 b)_i - x_b_i| over the rows this engine owns
	// (all of them on one GPU).  One extra pass over the local block of B^-1, between runs.
	int check_basis(double* xb_err, double* xb_scale) override {
		if (!have_data) return fail(B200LP_ERR_STATE, "check_basis before upload/generate");
		CU(cudaSetDevice(opt.device));
		if (int rc = settle()) return rc;
		if (hc.pending) {
			launch_update_ftran(true, false, 0);
			CU(cudaGetLastError());
			hc.pending = 0;
			CU(push_ctl());
		}
		CU(zero_tickets());
		const long long tr = (long long)(NWARP / wc) * 32 * VecT<T>::N;
		const long long tiles = (d.ldb + tr - 1) / tr * d.nchunk;
		const int g = (int)std::max<long long>(1, std::min<long long>(tiles, grid));
		if (wc == 1) k_ftran_vec<T, 1><<<g, NT, UF_SMEM_BYTES, stream>>>(d, d.b);
		else if (wc == 2) k_ftran_vec<T, 2><<<g, NT, UF_SMEM_BYTES, stream>>>(d, d.b);
		else if (wc == 4) k_ftran_vec<T, 4><<<g, NT, UF_SMEM_BYTES, stream>>>(d, d.b);
		else k_ftran_vec<T, 8><<<g, NT, UF_SMEM_BYTES, stream>>>(d, d.b);
		k_sum_partials<T><<<num_sms, NT, 0, stream>>>(d, d.acol);     // (B^-1 b) of the local rows -> scratch
		launches += 2;
		CU(cudaGetLastError());
		const long long rows = std::max<long long>(0, std::min<long long>(d.m, d.row0 + d.ldb) - d.row0);
		std::vector<T> a((size_t)std::max<long long>(rows, 1)), x((size_t)std::max<long long>(rows, 1));
		if (rows > 0) {
			CU(cudaMemcpyAsync(a.data(), d.acol, rows * sizeof(T), cudaMemcpyDeviceToHost, stream));
			CU(cudaMemcpyAsync(x.data(), d.x_b + d.row0, rows * sizeof(T), cudaMemcpyDeviceToHost, stream));
		}
		CU(cudaStreamSynchronize(stream));
		double err = 0, scale = 0;
		for (long long i = 0; i < rows; ++i) {
			err = std::max(err, std::fabs((double)a[i] - (double)x[i]));
			scale = std::max(scale, std::fabs((double)x[i]));
		}
		if (xb_err) *xb_err = err;
		if (xb_scale) *xb_scale = scale;
		return B200LP_OK;
	}

	// Refactorisation (the reference lists it as open, README.md:29-30; it never rebuilds its product-form inverse):
	// B^-1 is rebuilt from the basis alone.  Start from the identity (the slack basis) and replay one pivot per basis
	// position whose column is not that position's slack: FTRAN of the column through the inverse built so far,
	// pivot on the position's own row, rank-1 update fused into the next FTRAN pass — the same kernels as the loop,
	// m' <= m passes over B^-1.  A position whose pivot element is too small for now (|alpha_q| < rel_pivot_tol * max|alpha|)
	// goes to the back of the queue.  Then x_b = B^-1 b and y = c_b^T B^-1 are recomputed from the fresh inverse, so
	// the drift of the linear updates (v4:347-356) is gone as well.  Single GPU.
	int refactor(double rel_pivot_tol, int64_t* replayed) override {
		if (!have_data) return fail(B200LP_ERR_STATE, "refactor before upload/generate");
		if (nranks > 1) return fail(B200LP_ERR_STATE, "refactor is single-GPU only");
		CU(cudaSetDevice(opt.device));
		if (int rc = settle()) return rc;
		const long long m = d.m;
		std::vector<int> bix((size_t)m);
		CU(cudaMemcpy(bix.data(), d.b_ixs, m * sizeof(int), cudaMemcpyDeviceToHost));
		// steepest edge: the weight recurrence of the last pivot may still be pending (it rides in the next pricing pass
		// and reads row_q and the alpha.alpha slice partials); the replay below reuses both buffers, so keep copies
		T* keep = nullptr;
		const size_t keep_n = (size_t)d.ld + (size_t)3 * d.nslice;
		if (hc.se_pending) {
			CU(cudaMalloc((void**)&keep, keep_n * sizeof(T)));
			CU(cudaMemcpyAsync(keep, d.row_q, (size_t)d.ld * sizeof(T), cudaMemcpyDeviceToDevice, stream));
			CU(cudaMemcpyAsync(keep + d.ld, d.dpart, (size_t)3 * d.nslice * sizeof(T), cudaMemcpyDeviceToDevice, stream));
		}
		struct Free { T* p; ~Free() { if (p) cudaFree(p); } } keep_guard{keep};
		k_identity<T><<<num_sms * 8, 256, 0, stream>>>(d);
		launches++;
		hc.pending = 0;
		std::vector<long long> queue;
		for (long long i = 0; i < m; ++i)
			if (bix[(size_t)i] != (int)(d.ns + i) || d.ns == d.n) queue.push_back(i);   // (slack block not recognised: every position is replayed)
		std::vector<T> al((size_t)m);
		int64_t done = 0;
		size_t stalled = 0;
		const double tol = rel_pivot_tol > 0 ? rel_pivot_tol : 1e-9;
		while (!queue.empty()) {
			const long long q = queue.front();
			queue.erase(queue.begin());
			const long long p = bix[(size_t)q];
			launch_update_ftran(hc.pending != 0, true, p);
			hc.pending = 0;
			k_sum_partials<T><<<num_sms, NT, 0, stream>>>(d, d.alpha);
			launches++;
			CU(cudaMemcpyAsync(al.data(), d.alpha, m * sizeof(T), cudaMemcpyDeviceToHost, stream));
			CU(cudaStreamSynchronize(stream));
			double amax = 0;
			for (long long i = 0; i < m; ++i) amax = std::max(amax, std::fabs((double)al[(size_t)i]));
			if (!(std::fabs((double)al[(size_t)q]) >= tol * amax) || amax == 0) {
				queue.push_back(q);                      // not now: the rows this column needs are not in place yet
				if (++stalled > queue.size()) return fail(B200LP_ERR_STATE, "refactor: no admissible pivot order (basis singular to working precision); reset the engine");
				continue;
			}
			stalled = 0;
			k_book1<T><<<grid, NT, 0, stream>>>(d, p, q);   // row_q, E_q of this replay pivot (its dot partials are not used)
			launches++;
			hc.pending = 1;
			++done;
		}
		if (hc.pending) { launch_update_ftran(true, false, 0); hc.pending = 0; }
		CU(cudaGetLastError());
		// x_b = B^-1 b, y = c_b^T B^-1
		CU(zero_tickets());
		const long long tr = (long long)(NWARP / wc) * 32 * VecT<T>::N;
		const long long tiles = (d.ldb + tr - 1) / tr * d.nchunk;
		const int g = (int)std::max<long long>(1, std::min<long long>(tiles, grid));
		if (wc == 1) k_ftran_vec<T, 1><<<g, NT, UF_SMEM_BYTES, stream>>>(d, d.b);
		else if (wc == 2) k_ftran_vec<T, 2><<<g, NT, UF_SMEM_BYTES, stream>>>(d, d.b);
		else if (wc == 4) k_ftran_vec<T, 4><<<g, NT, UF_SMEM_BYTES, stream>>>(d, d.b);
		else k_ftran_vec<T, 8><<<g, NT, UF_SMEM_BYTES, stream>>>(d, d.b);
		k_sum_partials<T><<<num_sms, NT, 0, stream>>>(d, d.x_b);
		k_btran_vec<T><<<num_sms * 2, NT, 0, stream>>>(d, d.c_b, d.acol);
		k_copy<T><<<num_sms, 256, 0, stream>>>(d.y, d.acol, m);
		launches += 4;
		CU(cudaGetLastError());
		if (keep) {                       // (the steepest-edge weights themselves depend on the basis only: untouched)
			CU(cudaMemcpyAsync(d.row_q, keep, (size_t)d.ld * sizeof(T), cudaMemcpyDeviceToDevice, stream));
			CU(cudaMemcpyAsync(d.dpart, keep + d.ld, (size_t)3 * d.nslice * sizeof(T), cudaMemcpyDeviceToDevice, stream));
			CU(cudaStreamSynchronize(stream));
		}
		CU(push_ctl());
		if (replayed) *replayed = done;
		return B200LP_OK;
	}

	int download_trace(int32_t* pq, int64_t cap, int64_t* n_out) override {
		CU(cudaSetDevice(opt.device));
		CU(cudaStreamSynchronize(stream));
		const int64_t k = std::max<int64_t>(0, std::min<int64_t>({cap, (int64_t)hc.pivots, (int64_t)d.trace_cap}));
		if (k > 0 && pq) CU(cudaMemcpy(pq, d.trace, (size_t)k * sizeof(int2), cudaMemcpyDeviceToHost));
		if (n_out) *n_out = k;
		return B200LP_OK;
	}

	int download_vector(int32_t which, void* out) override {
		const T* src = which == 0 ? d.alpha : which == 1 ? d.E_q : which == 2 ? d.row_q
		             : which == 3 ? d.x_b : which == 4 ? d.y : which == 5 ? d.c_b : nullptr;
		if (!src || !out) return fail(B200LP_ERR_ARG, "download_vector: bad selector");
		CU(cudaSetDevice(opt.device));
		CU(cudaStreamSynchronize(stream));
		CU(cudaMemcpy(out, src, d.m * sizeof(T), cudaMemcpyDeviceToHost));
		return B200LP_OK;
	}

	// ---- one launch per phase (tests, mode 1) ---------------------------

	int phase_price(int64_t* p, double* min_e) override {
		if (!have_data) return fail(B200LP_ERR_STATE, "phase before upload/generate");
		if (nranks > 1) return fail(B200LP_ERR_STATE, "phase entry points are single-GPU only");
		if (in_flight && !phase_loop) { if (int rc = settle()) return rc; }
		CU(cudaSetDevice(opt.device));
		CU(zero_tickets());
		k_price<T><<<grid, NT, DYN_SMEM_BYTES, stream>>>(d);
		k_pick<T><<<1, NT, 0, stream>>>(d, grid, 0);
		launches += 2;
		CU(cudaGetLastError());
		CU(pull_ctl_fields());
		if (p) *p = hc.p;
		if (min_e) *min_e = hc.min_e;
		return B200LP_OK;
	}

	int phase_update_ftran(int64_t p) override {
		if (!have_data) return fail(B200LP_ERR_STATE, "phase before upload/generate");
		if (nranks > 1) return fail(B200LP_ERR_STATE, "phase entry points are single-GPU only");
		if (in_flight && !phase_loop) { if (int rc = settle()) return rc; }
		if (p < 0 || p >= d.n) return fail(B200LP_ERR_ARG, "entering column out of range");
		CU(cudaSetDevice(opt.device));
		launch_update_ftran(hc.pending != 0, true, p);
		CU(cudaGetLastError());
		hc.pending = 0;
		hc.p = p;
		CU(cudaStreamSynchronize(stream));
		return B200LP_OK;
	}

	int phase_ratio(int64_t* q, int64_t* eligible) override {
		if (!have_data) return fail(B200LP_ERR_STATE, "phase before upload/generate");
		if (nranks > 1) return fail(B200LP_ERR_STATE, "phase entry points are single-GPU only");
		if (in_flight && !phase_loop) { if (int rc = settle()) return rc; }
		CU(cudaSetDevice(opt.device));
		k_ratio<T><<<grid, NT, 0, stream>>>(d);
		k_pick<T><<<1, NT, 0, stream>>>(d, grid, 1);
		launches += 2;
		CU(cudaGetLastError());
		CU(pull_ctl_fields());
		long long el = 0;
		CU(cudaMemcpy(&el, d.cnt + grid, sizeof(long long), cudaMemcpyDeviceToHost));
		if (q) *q = hc.q;
		if (eligible) *eligible = el;
		return B200LP_OK;
	}

	int phase_pivot_update(int64_t p, int64_t q) override {
		if (!have_data) return fail(B200LP_ERR_STATE, "phase before upload/generate");
		if (nranks > 1) return fail(B200LP_ERR_STATE, "phase entry points are single-GPU only");
		if (in_flight && !phase_loop) { if (int rc = settle()) return rc; }
		if (p < 0 || p >= d.n || q < 0 || q >= d.m) return fail(B200LP_ERR_ARG, "pivot out of range");
		CU(cudaSetDevice(opt.device));
		k_book1<T><<<grid, NT, 0, stream>>>(d, p, q);
		k_book2<T><<<grid, NT, 0, stream>>>(d, p, q);
		launches += 2;
		CU(cudaGetLastError());
		if (hc.pivots < d.trace_cap) {
			const int2 pq = make_int2((int)p, (int)q);
			CU(cudaMemcpyAsync(d.trace + hc.pivots, &pq, sizeof(int2), cudaMemcpyHostToDevice, stream));
		}
		CU(cudaStreamSynchronize(stream));
		hc.pending = 1;
		hc.pivots++;
		hc.iter++;
		hc.p = p;
		hc.q = q;
		return B200LP_OK;
	}

	int shard_columns(int64_t* col0, int64_t* ncols) override {
		const long long nsg = d.n - d.m;      // with the identity slack block recognised
		if (col0) *col0 = nsg * rank / nranks;
		if (ncols) *ncols = nsg * (rank + 1) / nranks - nsg * rank / nranks;
		return B200LP_OK;
	}

	int shard_rows(int64_t* row0, int64_t* rows) override {
		if (row0) *row0 = d.row0;
		if (rows) *rows = std::max<long long>(0, std::min<long long>(d.m, d.row0 + d.ldb) - d.row0);
		return B200LP_OK;
	}

	// phase stamps of the last persistent launch: NSTAMP globaltimer values per iteration
	int download_profile(uint64_t* out, int64_t cap_iters, int64_t* n_iters) override {
		if (d.prof_cap == 0) return fail(B200LP_ERR_STATE, "engine was created without options.profile");
		CU(cudaSetDevice(opt.device));
		CU(cudaStreamSynchronize(stream));
		const int64_t k = std::max<int64_t>(0, std::min<int64_t>({cap_iters, (int64_t)d.prof_cap, (int64_t)(hc.iter - prof_iter0)}));
		if (k > 0 && out) CU(cudaMemcpy(out, d.prof, (size_t)k * NSTAMP * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
		if (n_iters) *n_iters = k;
		return B200LP_OK;
	}

	// algorithmic bytes: B^-1 read + written once, the structural columns read once; steepest edge reads B^-1 once
	// more (v = B^-T alpha)
	int64_t bytes_per_pivot() const override {
		return (int64_t)sizeof(T) * ((opt.pricing_rule == 1 ? 3 : 2) * d.m * d.m + d.m * (d.n - d.m));
	}

	// ---- sharded mode: peer mapping of the A shards and mailboxes (CUDA IPC over NVLink) ----

	int ipc_export(void* out) override {
		if (!have_data) return fail(B200LP_ERR_STATE, "ipc_export before upload/generate (the A shard is allocated there)");
		CU(cudaSetDevice(opt.device));
		cudaIpcMemHandle_t h[2];
		CU(cudaIpcGetMemHandle(&h[0], (void*)hA));
		CU(cudaIpcGetMemHandle(&h[1], (void*)mbox));
		std::memcpy(out, h, sizeof(h));
		return B200LP_OK;
	}

	int ipc_import(const void* all, int n) override {
		if (n != nranks) return fail(B200LP_ERR_ARG, "ipc_import: handle count differs from the engine's rank count");
		if (!have_data) return fail(B200LP_ERR_STATE, "ipc_import before upload/generate");
		CU(cudaSetDevice(opt.device));
		const cudaIpcMemHandle_t* h = static_cast<const cudaIpcMemHandle_t*>(all);
		for (int r = 0; r < nranks; ++r) {
			if (r == rank) { d.A_peer[r] = hA; d.mbox_peer[r] = mbox; continue; }
			void *pa = nullptr, *pm = nullptr;
			CU(cudaIpcOpenMemHandle(&pa, h[2 * r], cudaIpcMemLazyEnablePeerAccess));
			CU(cudaIpcOpenMemHandle(&pm, h[2 * r + 1], cudaIpcMemLazyEnablePeerAccess));
			opened.push_back(pa);
			opened.push_back(pm);
			d.A_peer[r] = static_cast<const T*>(pa);
			d.mbox_peer[r] = static_cast<unsigned char*>(pm);
		}
		peers_mapped = true;
		return B200LP_OK;
	}

private:
	// (re)allocate the local A shard for `ns_new` global dense columns
	cudaError_t set_columns(long long ns_new) {
		for (int r = 0; r <= nranks; ++r) d.colstart[r] = ns_new * r / nranks;
		const long long nsl_new = d.colstart[rank + 1] - d.colstart[rank];
		if (!hA || nsl_new != d.nsl) {
			if (hA) cudaFree(hA);
			hA = nullptr;
			cudaError_t e = cudaMalloc((void**)&hA, std::max<size_t>(1, (size_t)d.ld * nsl_new) * sizeof(T));
			if (e != cudaSuccess) return e;
		}
		d.A = hA;
		d.A_peer[rank] = hA;
		d.ns = ns_new;
		d.nsl = nsl_new;
		d.col0 = d.colstart[rank];
		// pricing group width
		// (measured on B200: 2-column blocks run at ~60 % of the streaming rate of 4-column blocks, which costs
		// more than their shorter tail saves, so auto is always 4)
		d.price_nc = (opt.price_cols == 2 || opt.price_cols == 4) ? opt.price_cols : 4;
		// Pricing path (measured, DESIGN.md 3): register-staged loads win clearly while the A shard is L2 resident
		// (the ring's start-up is a third of such a pass) and by ~6 % of the pass at m = 8192.  At 8 GB (m = 32768 on
		// one GPU) the TMA ring was on a par in round 1 (1215 us against 1243 us per pass); in the round-2 kernel its
		// loop state no longer fits the 128 registers next to the rest of the loop (ptxas spills it: 1323 us) while
		// the register-staged pass runs at 1233 us, so auto = register-staged everywhere and the ring is price_mode = 1.
		d.price_direct = opt.price_mode == 1 ? 0 : 1;
		if (opt.pricing_rule == 1) d.price_direct = 1;      // the steepest-edge pass is register-staged
		// x_b / y / c_b / b_ixs updates in the prologue of the next pricing pass: y must fit in the (idle) ring memory
		// and pricing must read y from there (register-staged path); single GPU only
		d.fuse_book2 = (opt.fuse_book2 >= 0 && nranks == 1 && d.price_direct && opt.mode == 0 &&
		                (size_t)d.ld * sizeof(T) <= (size_t)DYN_SMEM_BYTES) ? 1 : 0;
		// single-column work items at the end of the pricing pass: only where one column alone keeps 16 loads per
		// thread in flight (ld >= 16 row steps of the CTA), two per CTA
		d.price_tail = opt.price_tail < 0 ? 0 : opt.price_tail > 0 ? opt.price_tail
		             : (d.ld >= 16LL * NT * VecT<T>::N ? 2 * grid : 0);
		// unit (slack) columns priced without matrix bytes: none when the slack block was not recognised
		const long long nunit = d.n - ns_new;
		d.k0 = nunit * rank / nranks;
		d.k1 = nunit * (rank + 1) / nranks;
		ns = ns_new;
		return cudaSuccess;
	}

	template <typename U>
	cudaError_t alloc(U** p, size_t count) {
		cudaError_t e = cudaMalloc((void**)p, std::max<size_t>(count, 1) * sizeof(U));
		if (e == cudaSuccess) owned.push_back((void*)*p);
		return e;
	}

	void release() {
		cudaSetDevice(opt.device);
		if (stream) cudaStreamSynchronize(stream);
		if (l2_persist_bytes) cudaCtxResetPersistingL2Cache();
		for (void* p : opened) cudaIpcCloseMemHandle(p);
		opened.clear();
		// newest first: the allocator gets its blocks back in the reverse order it handed them out
		for (auto it = owned.rbegin(); it != owned.rend(); ++it) cudaFree(*it);
		if (hA) cudaFree(hA);
		owned.clear();
		if (pinned) cudaFreeHost(pinned);
		if (ev0) cudaEventDestroy(ev0);
		if (ev1) cudaEventDestroy(ev1);
		if (stream) cudaStreamDestroy(stream);
		if (abort_stream) cudaStreamDestroy(abort_stream);
	}

	// Is S (m x m, column-major, host) the identity?  A streaming OR over the raw bits of every column (sign bit
	// shifted out so that -0.0 passes like in a == comparison) with the diagonal entry checked apart: the loop
	// vectorises and runs at memory speed, which matters because it reads m*m elements (8.6 GB at m = 32768)
	// while the upload is on the wire.
	static bool host_is_identity(const T* S, long long m) {
		using U = typename std::conditional<sizeof(T) == 8, uint64_t, uint32_t>::type;
		const unsigned hw = std::max(1u, std::min(32u, std::thread::hardware_concurrency()));
		const unsigned nt = (unsigned)std::max<long long>(1, std::min<long long>(hw, m / 64));
		std::atomic<bool> ok{true};
		auto work = [&](long long j0, long long j1) {
			for (long long j = j0; j < j1 && ok.load(std::memory_order_relaxed); ++j) {
				const T* col = S + (size_t)j * m;
				if (col[j] != T(1)) { ok.store(false, std::memory_order_relaxed); return; }
				const U* bits = reinterpret_cast<const U*>(col);
				U acc = 0;
				for (long long i = 0; i < j; ++i) acc |= bits[i];
				for (long long i = j + 1; i < m; ++i) acc |= bits[i];
				if ((U)(acc << 1) != 0) { ok.store(false, std::memory_order_relaxed); return; }
			}
		};
		if (nt == 1) { work(0, m); return ok; }
		std::vector<std::thread> th;
		for (unsigned t = 0; t < nt; ++t) th.emplace_back(work, m * t / nt, m * (t + 1) / nt);
		for (auto& t : th) t.join();
		return ok;
	}

	cudaError_t push_ctl() {
		Ctl* st = static_cast<Ctl*>(pinned);
		*st = hc;
		st->bar = 0;
		st->price_ctr = st->upd_ctr = st->btran_ctr = 0;
		st->xarr[0] = st->xarr[1] = 0;
		cudaError_t e = cudaMemcpyAsync(d.ctl, st, sizeof(Ctl), cudaMemcpyHostToDevice, stream);
		if (e != cudaSuccess) return e;
		// the staging buffer is reused: make sure the copy has been consumed
		return cudaStreamSynchronize(stream);
	}

	cudaError_t pull_ctl() {
		return cudaMemcpy(&hc, d.ctl, sizeof(Ctl), cudaMemcpyDeviceToHost);
	}

	// phase mode: only p / q / min_e come from the device, counters live on the host
	cudaError_t pull_ctl_fields() {
		Ctl t;
		cudaError_t e = cudaStreamSynchronize(stream);
		if (e != cudaSuccess) return e;
		e = cudaMemcpy(&t, d.ctl, sizeof(Ctl), cudaMemcpyDeviceToHost);
		if (e != cudaSuccess) return e;
		hc.p = t.p; hc.q = t.q; hc.min_e = t.min_e;
		return cudaSuccess;
	}

	// work-ticket counters of the pricing / update phases (the persistent kernel resets them itself)
	cudaError_t zero_tickets() {
		static_assert(offsetof(Ctl, upd_ctr) == offsetof(Ctl, price_ctr) + sizeof(unsigned int), "adjacent counters");
		return cudaMemsetAsync(reinterpret_cast<unsigned char*>(d.ctl) + offsetof(Ctl, price_ctr), 0, 2 * sizeof(unsigned int), stream);
	}

	void launch_update_ftran(bool update, bool ftran, long long p) {
		zero_tickets();
		const long long tr = (long long)(NWARP / wc) * 32 * VecT<T>::N;
		const long long tiles = (d.ldb + tr - 1) / tr * d.nchunk;
		const int g = (int)std::max<long long>(1, std::min<long long>(tiles, grid));
		const int rev = (int)(hc.pivots & 1);
#define LAUNCH_UF(WC_)                                                                                    \
		do {                                                                                              \
			if (update && ftran) k_update_ftran<T, WC_, true, true><<<g, NT, UF_SMEM_BYTES, stream>>>(d, p, rev);          \
			else if (update)     k_update_ftran<T, WC_, true, false><<<g, NT, UF_SMEM_BYTES, stream>>>(d, p, rev);         \
			else                 k_update_ftran<T, WC_, false, true><<<g, NT, UF_SMEM_BYTES, stream>>>(d, p, rev);         \
		} while (0)
		if (wc == 1) LAUNCH_UF(1); else if (wc == 2) LAUNCH_UF(2); else if (wc == 4) LAUNCH_UF(4); else LAUNCH_UF(8);
#undef LAUNCH_UF
		launches++;
	}

	// the primal loop runs: algorithm = 0, or phase 2 of the composite method (algorithm = 1, cost_shift = 1)
	bool primal_loop() const { return opt.algorithm == 0 || phase == 2; }

	// composite method, first run from the slack basis: keep the original c, shift the nonbasic columns with
	// e_j < -eps (k_cost_shift), then phase 1 (the dual loop) prices with c'.  The count is read by wait().
	int shift_costs() {
		CU(cudaMemcpyAsync(c_orig, hcst, (size_t)d.n * sizeof(T), cudaMemcpyDeviceToDevice, stream));
		CU(cudaMemsetAsync(d_shifted, 0, sizeof(unsigned long long), stream));
		const T delta = (T)(opt.shift_delta > 0 ? opt.shift_delta : 1e-7);
		k_cost_shift<T><<<num_sms * 4, NT, 0, stream>>>(d, hcst, dd.nb, delta, d_shifted);
		launches++;
		CU(cudaGetLastError());
		c_shifted = true;
		shift_unread = true;
		phase = 1;
		return B200LP_OK;
	}

	// composite method, after a phase-1 OPTIMUM with shifted columns: flush the pending rank-1 update (as check_basis
	// and refactor do), restore c, c_b = c[b_ixs], y = c_b^T B^-1 (as refactor does; B^-1 = I and y unchanged when
	// phase 1 made no pivot), z for the original c, and a control block as a primal window boundary leaves it:
	// nothing pending, not done.  simplex_persistent / _tiny / _resident read iter, pivots, pending, p, q and min_e at
	// entry; p and q are used only with a pending book2 (fuse_book2 never carries one across launches) or the
	// steepest-edge recurrence (pricing_rule = 0 here).
	int hand_over() {
		if (hc.pending) { launch_update_ftran(true, false, 0); hc.pending = 0; }
		CU(cudaMemcpyAsync(hcst, c_orig, (size_t)d.n * sizeof(T), cudaMemcpyDeviceToDevice, stream));
		c_shifted = false;
		k_gather_cb<T><<<num_sms, 256, 0, stream>>>(d.c_b, d.c, d.b_ixs, d.m);
		launches++;
		if (hc.pivots > 0) {
			k_btran_vec<T><<<num_sms * 2, NT, 0, stream>>>(d, d.c_b, d.acol);
			k_copy<T><<<num_sms, 256, 0, stream>>>(d.y, d.acol, d.m);
			launches += 2;
		}
		k_objective<T><<<1, NT, 0, stream>>>(d);
		launches++;
		CU(cudaGetLastError());
		CU(cudaStreamSynchronize(stream));
		Ctl t;
		CU(cudaMemcpy(&t, d.ctl, sizeof(Ctl), cudaMemcpyDeviceToHost));
		hc.z = t.z;
		hc.done = 0;
		hc.status = B200LP_STATUS_MAX_ITER;
		phase = 2;
		CU(push_ctl());
		return B200LP_OK;
	}

	// tiny LPs (one warp-wide vector row, everything fits in shared memory): the shared-memory-resident kernel.
	// Only with the automatic grid: an explicit grid_ctas asks for the general kernel.
	bool tiny_ok() const {
		if (nranks != 1 || opt.grid_ctas > 0 || opt.mode != 0 || d.prof_cap > 0 || opt.pricing_rule != 0 || opt.ratio_mode == 2 ||
				!primal_loop())
			return false;
		return tiny_fits<T>(d.m, d.n, d.ns);
	}

	// mid-size LPs whose A and B^-1 fit in the shared memory of the whole grid (one CTA per SM): the resident kernel.
	// Only with the automatic configuration (an explicit grid, tile shape or pricing path asks for the general kernel).
	bool resident_ok() const {
		if (nranks != 1 || opt.grid_ctas > 0 || opt.mode != 0 || opt.pricing_rule != 0 || opt.ratio_mode == 2 ||
				opt.tile_shape != 0 || opt.price_mode != 0 || opt.fuse_ratio > 0 || opt.resident < 0 || !primal_loop())
			return false;
		if (d.m < 128) return false;                     // a handful of CTAs: the general kernel on a small grid is as good
		const ResLayout<T> L(d.m, d.ld, d.ns, num_sms);
		return L.bytes() <= (size_t)200 * 1024 && L.G <= num_sms && L.G <= max_grid;
	}

	int run_resident(int64_t iters) {
		hc.it_end = hc.iter + iters;
		CU(push_ctl());
		if (d.prof_cap > 0) CU(cudaMemsetAsync(d.prof, 0, (size_t)d.prof_cap * NSTAMP * sizeof(unsigned long long), stream));
		prof_iter0 = hc.iter;
		d.res_maxG = num_sms;
		const ResLayout<T> L(d.m, d.ld, d.ns, num_sms);
		const size_t smem = L.bytes();
		CU(cudaFuncSetAttribute(simplex_resident<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
		CU(cudaEventRecord(ev0, stream));
		void* args[] = {&d};
		CU(cudaLaunchCooperativeKernel((const void*)simplex_resident<T>, dim3((unsigned)L.G), dim3(NT), args, smem, stream));
		launches++;
		CU(cudaEventRecord(ev1, stream));
		return B200LP_OK;
	}

	int run_tiny(int64_t iters) {
		hc.it_end = hc.iter + iters;
		CU(push_ctl());
		const size_t smem = TinyLayout<T>(d.m, d.n, d.ns).bytes(d.m);
		CU(cudaFuncSetAttribute(simplex_tiny<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
		CU(cudaEventRecord(ev0, stream));
		simplex_tiny<T><<<1, NT, smem, stream>>>(d);
		launches++;
		CU(cudaGetLastError());
		CU(cudaEventRecord(ev1, stream));
		return B200LP_OK;
	}

	// mode 1: the loop of v4:286-359 driven from the host, one launch per phase and
	// one blocking read-back per decision (what the reference does, minus the libraries)
	int run_phases(int64_t iters) {
		struct Guard { bool& f; Guard(bool& g) : f(g) { f = true; } ~Guard() { f = false; } } guard(phase_loop);
		CU(cudaEventRecord(ev0, stream));
		const long long it_end = hc.iter + iters;
		hc.status = B200LP_STATUS_MAX_ITER;
		while (hc.iter < it_end) {
			int64_t p = 0, q = 0, el = 0;
			double mn = 0;
			int rc = phase_price(&p, &mn);
			if (rc) return rc;
			if (mn >= -d.eps) { hc.status = B200LP_STATUS_OPTIMUM; hc.done = 1; hc.iter++; break; }
			if ((rc = phase_update_ftran(p))) return rc;
			if ((rc = phase_ratio(&q, &el))) return rc;
			if (el == 0) { hc.status = B200LP_STATUS_UNBOUNDED; hc.done = 1; hc.iter++; break; }
			if ((rc = phase_pivot_update(p, q))) return rc;
		}
		k_objective<T><<<1, NT, 0, stream>>>(d);
		launches++;
		CU(cudaEventRecord(ev1, stream));
		CU(cudaStreamSynchronize(stream));
		Ctl t;
		CU(cudaMemcpy(&t, d.ctl, sizeof(Ctl), cudaMemcpyDeviceToHost));
		hc.z = t.z;
		CU(push_ctl());
		return B200LP_OK;
	}

	b200lp_options opt;
	Dev<T> d;
	DualDev<T> dd;             // dual simplex state (options.algorithm = 1)
	T* c_orig = nullptr;       // composite method (options.cost_shift): the original c while d.c holds c'
	unsigned long long* d_shifted = nullptr;   // columns k_cost_shift moved
	int phase = 0;             // composite method: 0 not started, 1 dual loop on c', 2 primal loop on c
	int64_t shifted_cols = 0, ph1_pivots = 0;
	bool c_shifted = false;    // d.c holds c' (c_orig the original)
	bool shift_unread = false; // d_shifted not read back yet
	std::atomic<bool> abort_asked{false};
	double ms_run = 0;         // device time of the phases of the current run
	Ctl hc;                    // host mirror of the control block
	T* hA = nullptr;           // mutable aliases of the const members of d
	T* hb = nullptr;
	T* hcst = nullptr;
	unsigned char* mbox = nullptr;
	size_t mbox_bytes = 0;
	void* pinned = nullptr;
	std::vector<void*> owned, opened;
	bool peers_mapped = false;
	cudaEvent_t ev0 = nullptr, ev1 = nullptr;
	int num_sms = 0, max_grid = 0, wc = 1;
	bool have_data = false, in_flight = false, phase_loop = false;
	cudaStream_t abort_stream = nullptr;
	int64_t launches = 0;
	long long prof_iter0 = 0;
	size_t l2_persist_bytes = 0;
};

// ---------------------------------------------------------------------------------------------
// Several GPUs behind ONE handle (b200lp_create_multi / b200lp_solve_*_multi): one rank of the sharded engine per
// listed device, all in this process.  Peers are mapped with cudaDeviceEnablePeerAccess and plain pointers (the
// multi-process front end exchanges CUDA IPC handles instead); launches, copies and waits fan out from the
// calling host thread, uploads run on one host thread per rank so that every GPU's PCIe link is busy.
// A device listed more than once hosts several ranks: they must share ONE cooperative launch
// (simplex_persistent_sharded_emu), because kernels that spin on each other may never be separate launches on one GPU.
template <typename T>
class MultiEngine final : public b200lp_engine {
public:
	MultiEngine(int64_t m, int64_t n) : m_(m), n_(n) {}
	~MultiEngine() override {
		for (auto* e : eng) delete e;
		if (devs_d) { cudaSetDevice(devices[0]); cudaFree(devs_d); }
		if (done_ev) cudaEventDestroy(done_ev);
	}

	int init(const b200lp_options& o, const int32_t* devs, int ndev) {
		R = ndev;
		devices.assign(devs, devs + ndev);
		int same = 0;
		for (int r = 0; r < R; ++r) same += devices[r] == devices[0];
		emu = R > 1 && same == R;
		if (!emu)
			for (int r = 0; r < R; ++r)
				for (int q = 0; q < r; ++q)
					if (devices[q] == devices[r])
						return fail(B200LP_ERR_ARG, "devices: either all distinct, or one device repeated for every rank");
		for (int r = 0; r < R; ++r) {
			b200lp_options orr = o;
			orr.device = devices[r];
			if (emu && orr.tile_shape == 0) orr.tile_shape = 8;   // one kernel instance serves all ranks
			auto* e = new Engine<T>(m_, n_, orr, r, R);
			eng.push_back(e);
			if (int rc = e->init()) return rc;
		}
		if (emu) {
			CU(cudaSetDevice(devices[0]));
			int occ = 0;
			CU(cudaFuncSetAttribute(emu_fn(), cudaFuncAttributeMaxDynamicSharedMemorySize, DYN_SMEM_BYTES));
			CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, emu_fn(), NT, DYN_SMEM_BYTES));
			if (occ < 1) return fail(B200LP_ERR_CUDA, "emulated multi-rank kernel does not fit on an SM");
			int gr = std::max(1, std::min(eng[0]->grid, occ * eng[0]->num_sms / R));
			for (auto* e : eng) e->grid = gr;
			CU(cudaMalloc((void**)&devs_d, sizeof(Dev<T>) * R));
			CU(cudaEventCreateWithFlags(&done_ev, cudaEventDisableTiming));
		} else {
			for (int r = 0; r < R; ++r) {
				CU(cudaSetDevice(devices[r]));
				for (int q = 0; q < R; ++q) {
					if (q == r) continue;
					int can = 0;
					CU(cudaDeviceCanAccessPeer(&can, devices[r], devices[q]));
					if (!can) return fail(B200LP_ERR_CUDA, "devices cannot access each other's memory (no NVLink / P2P)");
					cudaError_t e_ = cudaDeviceEnablePeerAccess(devices[q], 0);
					if (e_ == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
					else if (e_ != cudaSuccess) return fail(B200LP_ERR_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e_));
				}
			}
		}
		stream = eng[0]->stream;
		grid = eng[0]->grid;
		return B200LP_OK;
	}

	// ---- data in
	int upload(const void* A, const void* b, const void* c) override {
		// the identity check of the slack block (m*m host reads) runs beside the copies of the structural columns
		bool ident = true;
		std::thread chk([&] { ident = !eng[0]->opt.check_slack || Engine<T>::host_is_identity(static_cast<const T*>(A) + (size_t)(n_ - m_) * m_, m_); });
		int rc = upload_all(A, n_ - m_, b, c);
		chk.join();
		if (rc) return rc;
		if (!ident && (rc = upload_all(A, n_, b, c))) return rc;   // rare: the block is data, all n columns are stored
		return connect();
	}
	int upload_unchecked(const void* A, const void* b, const void* c) override { return upload(A, b, c); }
	bool slack_is_identity(const void*) const override { return true; }
	int upload_columns(const void*, int64_t, int64_t, const void*, const void*) override { return only_single("upload_columns"); }
	int shard_columns(int64_t* col0, int64_t* ncols) override { if (col0) *col0 = 0; if (ncols) *ncols = n_ - m_; return B200LP_OK; }
	int shard_rows(int64_t* row0, int64_t* rows) override { if (row0) *row0 = 0; if (rows) *rows = m_; return B200LP_OK; }
	int generate_dense(uint64_t seed) override {
		for (auto* e : eng) if (int rc = e->generate_dense(seed)) return rc;
		return connect();
	}
	int reset() override {
		for (auto* e : eng) if (int rc = e->reset()) return rc;
		return B200LP_OK;
	}

	// ---- the loop
	int run_async(int64_t iters) override {
		if (!connected) return fail(B200LP_ERR_STATE, "run before upload/generate");
		if (!emu) {
			for (auto* e : eng) if (int rc = e->run_async(iters)) return rc;
			return B200LP_OK;
		}
		int go = 0;
		for (auto* e : eng) {
			const int pr = e->prepare_run(iters);
			if (pr < 0) return pr;
			go += pr == 0;
		}
		if (go == 0) return B200LP_OK;
		if (go != R) return fail(B200LP_ERR_STATE, "ranks disagree on whether there is work left");
		CU(cudaSetDevice(devices[0]));
		std::vector<Dev<T>> h;
		for (auto* e : eng) h.push_back(e->d);
		for (int r = 1; r < R; ++r) CU(cudaStreamSynchronize(eng[r]->stream));
		CU(cudaMemcpyAsync(devs_d, h.data(), sizeof(Dev<T>) * R, cudaMemcpyHostToDevice, stream));
		CU(cudaStreamSynchronize(stream));              // h goes out of scope
		CU(cudaEventRecord(eng[0]->ev0, stream));
		int Rarg = R;
		void* args[] = {&devs_d, &Rarg};
		CU(cudaLaunchCooperativeKernel(emu_fn(), dim3(eng[0]->grid * R), dim3(NT), args, DYN_SMEM_BYTES, stream));
		eng[0]->launches++;
		CU(cudaEventRecord(eng[0]->ev1, stream));
		CU(cudaEventRecord(done_ev, stream));
		for (int r = 1; r < R; ++r) {                    // the other ranks' streams wait for the shared launch
			CU(cudaStreamWaitEvent(eng[r]->stream, done_ev, 0));
			CU(cudaEventRecord(eng[r]->ev1, eng[r]->stream));
		}
		return B200LP_OK;
	}
	int wait(b200lp_result* res) override {
		b200lp_result first;
		std::memset(&first, 0, sizeof(first));
		double ms = 0;
		int rc_all = B200LP_OK;
		for (int r = 0; r < R; ++r) {
			b200lp_result rr;
			const int rc = eng[r]->wait(&rr);
			if (rc && !rc_all) rc_all = rc;
			if (r == 0) first = rr;
			ms = std::max(ms, rr.ms_solve);
		}
		first.ms_solve = ms;
		int64_t l = 0;
		for (auto* e : eng) l += e->launches;
		first.kernel_launches = l;
		if (res) *res = first;
		return rc_all;
	}
	int abort() override {
		for (auto* e : eng) if (int rc = e->abort()) return rc;
		return B200LP_OK;
	}

	// ---- data out (every O(m) vector is replicated: rank 0 answers)
	int download(void* x_b, int32_t* b_ixs, void* y) override { if (int rc = settle_all()) return rc; return eng[0]->download(x_b, b_ixs, y); }
	int download_trace(int32_t* pq, int64_t cap, int64_t* n_out) override { if (int rc = settle_all()) return rc; return eng[0]->download_trace(pq, cap, n_out); }
	int download_vector(int32_t which, void* out) override { if (int rc = settle_all()) return rc; return eng[0]->download_vector(which, out); }
	int download_profile(uint64_t* out, int64_t cap, int64_t* n) override { return eng[0]->download_profile(out, cap, n); }
	int download_binv(void* Binv) override {
		T* out = static_cast<T*>(Binv);
		for (auto* e : eng) {
			int64_t r0 = 0, rows = 0;
			e->shard_rows(&r0, &rows);
			if (rows <= 0) continue;
			std::vector<T> blk((size_t)rows * m_);
			if (int rc = e->download_binv(blk.data())) return rc;
			for (int64_t j = 0; j < m_; ++j)
				std::memcpy(out + (size_t)j * m_ + r0, blk.data() + (size_t)j * rows, (size_t)rows * sizeof(T));
		}
		return B200LP_OK;
	}
	int check_basis(double* xb_err, double* xb_scale) override {
		double err = 0, scale = 0;
		for (auto* e : eng) {
			double a = 0, b = 0;
			if (int rc = e->check_basis(&a, &b)) return rc;
			err = std::max(err, a);
			scale = std::max(scale, b);
		}
		if (xb_err) *xb_err = err;
		if (xb_scale) *xb_scale = scale;
		return B200LP_OK;
	}
	int refactor(double, int64_t*) override { return only_single("refactor"); }
	int phase_price(int64_t*, double*) override { return only_single("phase_price"); }
	int phase_update_ftran(int64_t) override { return only_single("phase_update_ftran"); }
	int phase_ratio(int64_t*, int64_t*) override { return only_single("phase_ratio"); }
	int phase_pivot_update(int64_t, int64_t) override { return only_single("phase_pivot_update"); }
	int ipc_export(void*) override { return only_single("ipc_export"); }
	int ipc_import(const void*, int) override { return only_single("ipc_import"); }
	int64_t bytes_per_pivot() const override { return eng[0]->bytes_per_pivot(); }

private:
	static int only_single(const char* what) { return fail(B200LP_ERR_STATE, std::string(what) + " is not available on a multi-GPU handle"); }
	int settle_all() { for (auto* e : eng) if (int rc = e->settle()) return rc; return B200LP_OK; }

	const void* emu_fn() const {
		return eng[0]->opt.pricing_rule == 1 ? (const void*)simplex_persistent_sharded_emu<T, 8, true>
		                                      : (const void*)simplex_persistent_sharded_emu<T, 8>;
	}

	int upload_all(const void* A, long long ns_new, const void* b, const void* c) {
		std::vector<int> rcs(R, 0);
		std::vector<std::string> errs(R);
		std::vector<std::thread> th;
		for (int r = 0; r < R; ++r)
			th.emplace_back([&, r] { rcs[r] = eng[r]->upload_shard(A, ns_new, b, c); if (rcs[r]) errs[r] = g_err; });
		for (auto& t : th) t.join();
		for (int r = 0; r < R; ++r) if (rcs[r]) return fail(rcs[r], errs[r]);
		ns = ns_new;
		return B200LP_OK;
	}

	// every rank learns every rank's A shard and mailbox (same address space: plain pointers)
	int connect() {
		for (auto* e : eng) {
			for (int q = 0; q < R; ++q) { e->d.A_peer[q] = eng[q]->hA; e->d.mbox_peer[q] = eng[q]->mbox; }
			e->peers_mapped = true;
		}
		connected = true;
		ms_upload = 0;
		for (auto* e : eng) ms_upload = std::max(ms_upload, e->ms_upload);
		return B200LP_OK;
	}

	int64_t m_, n_;
	int R = 0;
	bool emu = false, connected = false;
	std::vector<int> devices;
	std::vector<Engine<T>*> eng;
	Dev<T>* devs_d = nullptr;
	cudaEvent_t done_ev = nullptr;
};

template <typename T>
int create_engine(int64_t m, int64_t n, const b200lp_options* opt, b200lp_engine** out, int rank = 0, int nranks = 1) {
	if (!out) return fail(B200LP_ERR_ARG, "out is NULL");
	*out = nullptr;
	if (nranks < 1 || nranks > MAXR || rank < 0 || rank >= nranks) return fail(B200LP_ERR_ARG, "need 0 <= rank < nranks <= 8");
	if (m <= 0 || n <= 0 || m > n) return fail(B200LP_ERR_ARG, "need 0 < m <= n (v4:402)");
	if (n >= ((int64_t)1 << 31)) return fail(B200LP_ERR_ARG, "n must fit a 32-bit basis index");
	b200lp_options o;
	if (opt) o = *opt; else b200lp_default_options(&o);
	if (int rc = check_algorithm(o, nranks)) return rc;
	if (int rc = check_cost_shift(o)) return rc;
	int ndev = 0;
	if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
		cudaGetLastError();
		return fail(B200LP_ERR_NO_GPU, "no CUDA device: the engine has no CPU fallback");
	}
	if (o.device < 0 || o.device >= ndev) return fail(B200LP_ERR_ARG, "device ordinal out of range");
	auto* e = new Engine<T>(m, n, o, rank, nranks);
	int rc = e->init();
	if (rc) { delete e; return rc; }
	*out = e;
	return B200LP_OK;
}

template <typename T>
int create_multi(int64_t m, int64_t n, const b200lp_options* opt, const int32_t* devices, int ndev, b200lp_engine** out) {
	if (!out) return fail(B200LP_ERR_ARG, "out is NULL");
	*out = nullptr;
	if (!devices || ndev < 1 || ndev > MAXR) return fail(B200LP_ERR_ARG, "need 1 <= ndev <= 8 device ordinals");
	b200lp_options o;
	if (opt) o = *opt; else b200lp_default_options(&o);
	if (int rc = check_algorithm(o, ndev)) return rc;
	if (int rc = check_cost_shift(o)) return rc;
	if (ndev == 1) {
		o.device = devices[0];
		return create_engine<T>(m, n, &o, out);
	}
	if (m <= 0 || n <= 0 || m > n) return fail(B200LP_ERR_ARG, "need 0 < m <= n (v4:402)");
	if (n >= ((int64_t)1 << 31)) return fail(B200LP_ERR_ARG, "n must fit a 32-bit basis index");
	int have = 0;
	if (cudaGetDeviceCount(&have) != cudaSuccess || have == 0) {
		cudaGetLastError();
		return fail(B200LP_ERR_NO_GPU, "no CUDA device: the engine has no CPU fallback");
	}
	for (int r = 0; r < ndev; ++r)
		if (devices[r] < 0 || devices[r] >= have) return fail(B200LP_ERR_ARG, "device ordinal out of range");
	auto* e = new MultiEngine<T>(m, n);
	int rc = e->init(o, devices, ndev);
	if (rc) { delete e; return rc; }
	*out = e;
	return B200LP_OK;
}

// the one-call solve over several GPUs: create, upload (slack check beside the copies), run, read back, destroy
template <typename T>
int solve_multi(const T* A, const T* b, const T* c, int64_t m, int64_t n, const b200lp_options* opt,
		const int32_t* devices, int ndev, T* x_b, int32_t* b_ixs, int32_t* trace_pq, int64_t trace_cap, b200lp_result* res) {
	if (!A || !b || !c) return fail(B200LP_ERR_ARG, "A, b, c must not be NULL");
	b200lp_options o;
	if (opt) o = *opt; else b200lp_default_options(&o);
	b200lp_engine* e = nullptr;
	int rc = create_multi<T>(m, n, &o, devices, ndev, &e);
	if (rc) return rc;
	b200lp_result r;
	std::memset(&r, 0, sizeof(r));
	do {
		if ((rc = e->upload(A, b, c))) break;
		if ((rc = e->run_async(o.max_iter))) break;
		if ((rc = e->wait(&r))) break;
		r.ms_upload = e->ms_upload;
		if ((rc = e->download(x_b, b_ixs, nullptr))) break;
		if (trace_pq && trace_cap > 0 && (rc = e->download_trace(trace_pq, trace_cap, nullptr))) break;
	} while (0);
	if (res) *res = r;
	delete e;
	return rc;
}

// One engine kept between calls of b200lp_solve_* (b200lp_set_memory_cache): creating and destroying 16 GB of
// device buffers costs 40-500 ms per call (cudaFree alone was measured at 31-449 ms), the solve of a 192-pivot
// window 740 ms.  Off by default: like the reference, a call then leaves no device memory behind.
struct EngineCache {
	std::mutex mu;
	bool on = false;
	b200lp_engine* e = nullptr;
	int dtype = -1;
	int64_t m = 0, n = 0;
	b200lp_options opt;
};
static EngineCache g_cache;

template <typename T>
int solve_once(const T* A, const T* b, const T* c, int64_t m, int64_t n, const b200lp_options* opt,
		T* x_b, int32_t* b_ixs, int32_t* trace_pq, int64_t trace_cap, b200lp_result* res) {
	if (!A || !b || !c) return fail(B200LP_ERR_ARG, "A, b, c must not be NULL");
	b200lp_options o;
	if (opt) o = *opt; else b200lp_default_options(&o);
	const int dtype = sizeof(T) == 8 ? B200LP_F64 : B200LP_F32;
	using Clk = std::chrono::steady_clock;
	auto ms_since = [](Clk::time_point t) { return std::chrono::duration<double, std::milli>(Clk::now() - t).count(); };
	const bool timing = std::getenv("B200LP_TIMING") != nullptr;    // host wall-clock split of the call on stderr
	auto t_all = Clk::now(), t = t_all;
	double ms_create = 0, ms_up = 0, ms_run = 0, ms_down = 0;
	b200lp_engine* e = nullptr;
	{
		std::lock_guard<std::mutex> lk(g_cache.mu);
		if (g_cache.on && g_cache.e && g_cache.dtype == dtype && g_cache.m == m && g_cache.n == n &&
				std::memcmp(&g_cache.opt, &o, sizeof(o)) == 0) {
			e = g_cache.e;                 // take it out of the cache for the duration of the call
			g_cache.e = nullptr;
		}
	}
	int rc = B200LP_OK;
	if (!e && (rc = create_engine<T>(m, n, &o, &e))) return rc;
	ms_create = ms_since(t);
	b200lp_result r;
	std::memset(&r, 0, sizeof(r));
	cudaEvent_t t0 = nullptr, t1 = nullptr;
	do {
		t = Clk::now();
		if (o.check_slack) {
			// optimistic: ship the structural columns and start pivoting; the m x m slack block (8.6 GB of host
			// memory at m = 32768) is verified by host threads while the GPU works
			if ((rc = e->upload_unchecked(A, b, c))) break;
			ms_up = ms_since(t);
			t = Clk::now();
			if ((rc = e->run_async(o.max_iter))) break;
			if (!e->slack_is_identity(A)) {           // rare: the block is data -> store and price all n columns
				if ((rc = e->abort())) break;            // the optimistic run stops at its next iteration boundary
				if ((rc = e->wait(nullptr))) break;
				if ((rc = e->upload(A, b, c))) break;
				if ((rc = e->run_async(o.max_iter))) break;
			}
		} else {
			if ((rc = e->upload(A, b, c))) break;
			ms_up = ms_since(t);
			t = Clk::now();
			if ((rc = e->run_async(o.max_iter))) break;
		}
		if ((rc = e->wait(&r))) break;
		ms_run = ms_since(t);
		t = Clk::now();
		cudaEventCreate(&t0);
		cudaEventCreate(&t1);
		cudaEventRecord(t0, e->stream);
		if ((rc = e->download(x_b, b_ixs, nullptr))) break;
		if (trace_pq && trace_cap > 0 && (rc = e->download_trace(trace_pq, trace_cap, nullptr))) break;
		cudaEventRecord(t1, e->stream);
		cudaEventSynchronize(t1);
		float ms = 0;
		cudaEventElapsedTime(&ms, t0, t1);
		r.ms_download = ms;
		ms_down = ms_since(t);
	} while (0);
	if (t0) cudaEventDestroy(t0);
	if (t1) cudaEventDestroy(t1);
	if (res) *res = r;
	t = Clk::now();
	{
		std::lock_guard<std::mutex> lk(g_cache.mu);
		if (g_cache.on && rc == B200LP_OK && !g_cache.e) {
			g_cache.e = e;
			g_cache.dtype = dtype;
			g_cache.m = m;
			g_cache.n = n;
			g_cache.opt = o;
			e = nullptr;
		}
	}
	delete e;
	if (timing)
		std::fprintf(stderr, "[b200lp] solve %lldx%lld: create %.1f ms, upload %.1f ms (copy %.1f), run %.1f ms (kernel %.1f), "
			"download %.1f ms, destroy %.1f ms, total %.1f ms\n", (long long)m, (long long)n, ms_create, ms_up, r.ms_upload,
			ms_run, r.ms_solve, ms_down, ms_since(t), ms_since(t_all));
	return rc;
}

// Many LPs of one shape in one call (b200lp_solve_batch_*).  Tiny shapes run in one kernel, one CTA per LP on a
// persistent grid fed by a ticket counter: simplex_tiny_batch for the primal Dantzig rule with a one-pass ratio test,
// simplex_tiny_batch_dual for the dual simplex and the composite method (algorithm = 1, with or without cost_shift).
// Everything else, and max_iter <= 0, runs the LPs one after another on one engine (upload, run, download per LP).
// Either way record k and row k of every output are bit-identical to b200lp_solve_* on LP k alone.
template <typename T>
class BatchCall {
public:
	BatchCall(const T* A, const T* b, const T* c, int64_t batch, int64_t m, int64_t n, const b200lp_options& o,
			T* x_b, int32_t* b_ixs, T* y, int32_t* trace_pq, int64_t trace_cap, b200lp_result* res)
		: A(A), b(b), c(c), batch(batch), m(m), n(n), o(o), x_b(x_b), b_ixs(b_ixs), y(y), trace_pq(trace_pq),
		  trace_cap(trace_pq ? trace_cap : 0), res(res) {}

	~BatchCall() {
		for (void* p : owned) cudaFree(p);
		if (stream) cudaStreamDestroy(stream);
		for (cudaEvent_t e : ev) if (e) cudaEventDestroy(e);
	}

	int run() {
		// structural columns per LP: the rule of Engine::upload (check_slack), slack blocks checked on host threads
		std::vector<int> ns((size_t)batch);
		{
			const unsigned nt = (unsigned)std::max<int64_t>(1, std::min<int64_t>(std::max(1u, std::thread::hardware_concurrency()), batch));
			auto work = [&](int64_t k0, int64_t k1) {
				for (int64_t k = k0; k < k1; ++k)
					ns[k] = (int)(!o.check_slack || Engine<T>::host_is_identity(A + (size_t)k * m * n + (size_t)(n - m) * m, m) ? n - m : n);
			};
			std::vector<std::thread> th;
			for (unsigned t = 0; t < nt; ++t) th.emplace_back(work, batch * t / nt, batch * (t + 1) / nt);
			for (auto& t : th) t.join();
		}
		const int ns_max = *std::max_element(ns.begin(), ns.end());
		if (o.max_iter > 0 && o.algorithm == 1 && tiny_dual_fits<T>(m, n, ns_max))   // check_algorithm: Dantzig, textbook ratio
			return run_kernel(ns, ns_max);
		if (o.max_iter > 0 && o.pricing_rule == 0 && o.ratio_mode != 2 && o.algorithm == 0 && tiny_fits<T>(m, n, ns_max))
			return run_kernel(ns, ns_max);
		return run_engine();
	}

private:
	template <typename U>
	cudaError_t alloc(U** p, size_t count) {
		void* v = nullptr;
		cudaError_t e = cudaMalloc(&v, std::max<size_t>(count, 1) * sizeof(U));
		if (e == cudaSuccess) owned.push_back(v);
		*p = static_cast<U*>(v);
		return e;
	}

	int run_kernel(const std::vector<int>& ns, int ns_max) {
		CU(cudaSetDevice(o.device));
		cudaDeviceProp prop;
		CU(cudaGetDeviceProperties(&prop, o.device));
		if (prop.major < 10)
			return fail(B200LP_ERR_NO_GPU, std::string("device is sm_") + std::to_string(prop.major * 10 + prop.minor) +
				", the engine is built for sm_100a only");
		CU(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
		for (auto& e : ev) CU(cudaEventCreate(&e));
		const size_t bm = (size_t)batch * m, bn = (size_t)batch * n;
		TinyBatch<T> bt;
		std::memset(&bt, 0, sizeof(bt));
		T *dA, *db, *dc, *dx, *dy = nullptr;
		int *dns, *dbix;
		int2* dtr = nullptr;
		TinyBatchRec* drec;
		unsigned long long* dticket;
		CU(alloc(&dA, bm * n));
		CU(alloc(&db, bm));
		CU(alloc(&dc, bn));
		CU(alloc(&dns, (size_t)batch));
		CU(alloc(&dx, bm));
		CU(alloc(&dbix, bm));
		if (y) CU(alloc(&dy, bm));
		if (trace_cap > 0) CU(alloc(&dtr, (size_t)batch * trace_cap));
		CU(alloc(&drec, (size_t)batch));
		CU(alloc(&dticket, 1));
		CU(cudaEventRecord(ev[0], stream));
		CU(cudaMemcpyAsync(dA, A, bm * n * sizeof(T), cudaMemcpyHostToDevice, stream));
		CU(cudaMemcpyAsync(db, b, bm * sizeof(T), cudaMemcpyHostToDevice, stream));
		CU(cudaMemcpyAsync(dc, c, bn * sizeof(T), cudaMemcpyHostToDevice, stream));
		CU(cudaMemcpyAsync(dns, ns.data(), (size_t)batch * sizeof(int), cudaMemcpyHostToDevice, stream));
		CU(cudaMemsetAsync(dticket, 0, sizeof(unsigned long long), stream));
		if (dtr) CU(cudaMemsetAsync(dtr, 0xff, (size_t)batch * trace_cap * sizeof(int2), stream));   // -1: no pivot
		CU(cudaEventRecord(ev[1], stream));

		bt.batch = batch; bt.m = m; bt.n = n;
		bt.A = dA; bt.b = db; bt.c = dc; bt.ns = dns;
		bt.it_end = o.max_iter;
		bt.eps = sizeof(T) == 4 ? (double)(float)o.eps : o.eps;                  // as Engine does
		bt.pivot_tol = sizeof(T) == 4 ? (double)(float)o.pivot_tol : o.pivot_tol;
		bt.ratio_mode = o.ratio_mode;
		bt.x_b = dx; bt.y = dy; bt.b_ixs = dbix; bt.trace = dtr; bt.trace_cap = trace_cap; bt.rec = drec; bt.ticket = dticket;
		bt.cost_shift = o.cost_shift;
		bt.delta = (T)(o.shift_delta > 0 ? o.shift_delta : 1e-7);                // as Engine::shift_costs does
		const bool dual = o.algorithm == 1;
		const void* fn = dual ? (const void*)simplex_tiny_batch_dual<T> : (const void*)simplex_tiny_batch<T>;
		const size_t smem = dual ? TinyDualLayout<T>(m, n, ns_max).bytes(m, n) : TinyLayout<T>(m, n, ns_max).bytes(m);
		CU(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
		int occ = 0;
		CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, NT, smem));
		if (occ < 1) return fail(B200LP_ERR_CUDA, "the tiny batch kernel does not fit on an SM");
		const int grid = (int)std::min<int64_t>(batch, (int64_t)occ * prop.multiProcessorCount);
		if (dual) simplex_tiny_batch_dual<T><<<grid, NT, smem, stream>>>(bt);
		else      simplex_tiny_batch<T><<<grid, NT, smem, stream>>>(bt);
		CU(cudaGetLastError());
		CU(cudaEventRecord(ev[2], stream));

		std::vector<TinyBatchRec> rec((size_t)batch);
		CU(cudaMemcpyAsync(rec.data(), drec, (size_t)batch * sizeof(TinyBatchRec), cudaMemcpyDeviceToHost, stream));
		CU(cudaMemcpyAsync(x_b, dx, bm * sizeof(T), cudaMemcpyDeviceToHost, stream));
		CU(cudaMemcpyAsync(b_ixs, dbix, bm * sizeof(int), cudaMemcpyDeviceToHost, stream));
		if (y) CU(cudaMemcpyAsync(y, dy, bm * sizeof(T), cudaMemcpyDeviceToHost, stream));
		if (dtr) CU(cudaMemcpyAsync(trace_pq, dtr, (size_t)batch * trace_cap * sizeof(int2), cudaMemcpyDeviceToHost, stream));
		CU(cudaEventRecord(ev[3], stream));
		CU(cudaStreamSynchronize(stream));
		float up = 0, solve = 0, down = 0;
		CU(cudaEventElapsedTime(&up, ev[0], ev[1]));
		CU(cudaEventElapsedTime(&solve, ev[1], ev[2]));
		CU(cudaEventElapsedTime(&down, ev[2], ev[3]));
		for (int64_t k = 0; k < batch; ++k) {
			b200lp_result& r = res[k];
			std::memset(&r, 0, sizeof(r));
			r.status = rec[k].status;
			r.iterations = rec[k].iterations;
			r.pivots = rec[k].pivots;
			r.z = rec[k].z;
			r.min_reduced_cost = rec[k].min_e;
			r.ms_upload = up;
			r.ms_solve = solve;
			r.ms_download = down;
			r.kernel_launches = 1;
		}
		return B200LP_OK;
	}

	// any other shape or option: the LPs one after another on one engine, i.e. exactly the single call's path
	int run_engine() {
		b200lp_engine* e = nullptr;
		if (int rc = create_engine<T>(m, n, &o, &e)) return rc;
		std::unique_ptr<b200lp_engine> own(e);
		double up = 0, solve = 0, down = 0;
		using Clk = std::chrono::steady_clock;
		for (int64_t k = 0; k < batch; ++k) {
			b200lp_result& r = res[k];
			if (int rc = e->upload(A + (size_t)k * m * n, b + (size_t)k * m, c + (size_t)k * n)) return rc;
			if (int rc = e->run_async(o.max_iter)) return rc;
			if (int rc = e->wait(&r)) return rc;
			const auto t = Clk::now();
			if (int rc = e->download(x_b + (size_t)k * m, b_ixs + (size_t)k * m, y ? y + (size_t)k * m : nullptr)) return rc;
			if (trace_cap > 0) {
				int32_t* tr = trace_pq + (size_t)k * trace_cap * 2;
				int64_t got = 0;
				if (int rc = e->download_trace(tr, trace_cap, &got)) return rc;
				std::fill(tr + 2 * got, tr + 2 * trace_cap, -1);
			}
			down += std::chrono::duration<double, std::milli>(Clk::now() - t).count();
			up += r.ms_upload;
			solve += r.ms_solve;
		}
		const int64_t launches = res[batch - 1].kernel_launches;    // the engine's count covers the whole call
		for (int64_t k = 0; k < batch; ++k) {
			res[k].aborted = 0;
			res[k].ms_upload = up;
			res[k].ms_solve = solve;
			res[k].ms_download = down;
			res[k].kernel_launches = launches;
		}
		return B200LP_OK;
	}

	const T *A, *b, *c;
	int64_t batch, m, n;
	b200lp_options o;
	T* x_b;
	int32_t* b_ixs;
	T* y;
	int32_t* trace_pq;
	int64_t trace_cap;
	b200lp_result* res;
	std::vector<void*> owned;
	cudaStream_t stream = nullptr;
	cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
};

template <typename T>
int solve_batch(const T* A, const T* b, const T* c, int64_t batch, int64_t m, int64_t n, const b200lp_options* opt,
		T* x_b, int32_t* b_ixs, T* y, int32_t* trace_pq, int64_t trace_cap, b200lp_result* res) {
	if (batch <= 0) return fail(B200LP_ERR_ARG, "batch must be positive");
	if (m <= 0 || n <= 0 || m > n) return fail(B200LP_ERR_ARG, "need 0 < m <= n (v4:402)");
	if (n >= ((int64_t)1 << 31)) return fail(B200LP_ERR_ARG, "n must fit a 32-bit basis index");
	if (!A || !b || !c) return fail(B200LP_ERR_ARG, "A, b, c must not be NULL");
	if (!x_b || !b_ixs || !res) return fail(B200LP_ERR_ARG, "x_b, b_ixs, res must not be NULL");
	if (trace_cap < 0) return fail(B200LP_ERR_ARG, "trace_cap must not be negative");
	b200lp_options o;
	if (opt) o = *opt; else b200lp_default_options(&o);
	if (o.pricing_rule != 0 && o.pricing_rule != 1) return fail(B200LP_ERR_ARG, "pricing_rule must be 0 (Dantzig) or 1 (steepest edge)");
	if (o.ratio_mode < 0 || o.ratio_mode > 2) return fail(B200LP_ERR_ARG, "ratio_mode must be 0, 1 or 2");
	if (int rc = check_algorithm(o, 1)) return rc;
	if (int rc = check_cost_shift(o)) return rc;
	int ndev = 0;
	if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
		cudaGetLastError();
		return fail(B200LP_ERR_NO_GPU, "no CUDA device: the engine has no CPU fallback");
	}
	if (o.device < 0 || o.device >= ndev) return fail(B200LP_ERR_ARG, "device ordinal out of range");
	BatchCall<T> call(A, b, c, batch, m, n, o, x_b, b_ixs, y, trace_pq, trace_cap, res);
	return call.run();
}

} // namespace

// host-side twin of k_generate_dense (same counter-based numbers), threaded over columns
template <typename T>
static void lpgen_host(T* A, T* b, T* c, int64_t m, int64_t n, int64_t col0, int64_t ncols, uint64_t seed) {
	const int64_t ns = n - m;
	if (A && ncols > 0) {
		const unsigned nt = (unsigned)std::max<int64_t>(1, std::min<int64_t>(std::max(1u, std::thread::hardware_concurrency()), ncols));
		auto work = [&](int64_t j0, int64_t j1) {
			for (int64_t jj = j0; jj < j1; ++jj) {
				const int64_t j = col0 + jj;
				T* col = A + (size_t)jj * m;
				if (j < ns) for (int64_t i = 0; i < m; ++i) col[i] = (T)u01(seed, 0, (uint64_t)(i * ns + j));
				else        for (int64_t i = 0; i < m; ++i) col[i] = (T)(i == j - ns);
			}
		};
		std::vector<std::thread> th;
		for (unsigned t = 0; t < nt; ++t) th.emplace_back(work, ncols * t / nt, ncols * (t + 1) / nt);
		for (auto& t : th) t.join();
	}
	if (b) for (int64_t i = 0; i < m; ++i) b[i] = (T)(0.5 * (double)ns * (1.0 + u01(seed, 1, (uint64_t)i)));
	if (c) for (int64_t j = 0; j < n; ++j) c[j] = j < ns ? (T)(0.5 + u01(seed, 2, (uint64_t)j)) : T(0);
}

// ------------------------------------------------------------------ C ABI

extern "C" {

// used by the other translation units of the library (lp_io.cpp); not part of the public ABI
int b200lp_internal_fail(int code, const char* msg) { return fail(code, msg ? msg : ""); }

int b200lp_lpgen_dense_host(int32_t dtype, void* A_cols, void* b, void* c, int64_t m, int64_t n,
		int64_t col0, int64_t ncols, uint64_t seed) {
	if (m <= 0 || n < m || col0 < 0 || ncols < 0 || col0 + ncols > n) return fail(B200LP_ERR_ARG, "lpgen: bad shape");
	if (dtype == B200LP_F64) lpgen_host<double>((double*)A_cols, (double*)b, (double*)c, m, n, col0, ncols, seed);
	else if (dtype == B200LP_F32) lpgen_host<float>((float*)A_cols, (float*)b, (float*)c, m, n, col0, ncols, seed);
	else return fail(B200LP_ERR_ARG, "dtype must be B200LP_F32 or B200LP_F64");
	return B200LP_OK;
}

void b200lp_default_options(b200lp_options* opt) {
	if (!opt) return;
	std::memset(opt, 0, sizeof(*opt));
	opt->eps = 1e-4;      // v4:18
	opt->max_iter = 5;    // v4:19
	opt->device = 0;
	opt->check_slack = 1;
	opt->l2_persist_mb = -1;
}

int b200lp_solve_f64(const double* A, const double* b, const double* c, int64_t m, int64_t n,
		const b200lp_options* opt, double* x_b, int32_t* b_ixs, int32_t* trace_pq, int64_t trace_cap, b200lp_result* res) {
	return solve_once<double>(A, b, c, m, n, opt, x_b, b_ixs, trace_pq, trace_cap, res);
}

int b200lp_solve_f32(const float* A, const float* b, const float* c, int64_t m, int64_t n,
		const b200lp_options* opt, float* x_b, int32_t* b_ixs, int32_t* trace_pq, int64_t trace_cap, b200lp_result* res) {
	return solve_once<float>(A, b, c, m, n, opt, x_b, b_ixs, trace_pq, trace_cap, res);
}

int b200lp_solve_batch_f64(const double* A, const double* b, const double* c, int64_t batch, int64_t m, int64_t n,
		const b200lp_options* opt, double* x_b, int32_t* b_ixs, double* y, int32_t* trace_pq, int64_t trace_cap,
		b200lp_result* res) {
	return solve_batch<double>(A, b, c, batch, m, n, opt, x_b, b_ixs, y, trace_pq, trace_cap, res);
}

int b200lp_solve_batch_f32(const float* A, const float* b, const float* c, int64_t batch, int64_t m, int64_t n,
		const b200lp_options* opt, float* x_b, int32_t* b_ixs, float* y, int32_t* trace_pq, int64_t trace_cap,
		b200lp_result* res) {
	return solve_batch<float>(A, b, c, batch, m, n, opt, x_b, b_ixs, y, trace_pq, trace_cap, res);
}

int b200lp_solve_f64_multi(const double* A, const double* b, const double* c, int64_t m, int64_t n,
		const b200lp_options* opt, const int32_t* devices, int32_t ndev, double* x_b, int32_t* b_ixs,
		int32_t* trace_pq, int64_t trace_cap, b200lp_result* res) {
	if (!devices || ndev < 1 || ndev > MAXR) return fail(B200LP_ERR_ARG, "need 1 <= ndev <= 8 device ordinals");
	if (ndev == 1) {
		b200lp_options o;
		if (opt) o = *opt; else b200lp_default_options(&o);
		o.device = devices[0];
		return solve_once<double>(A, b, c, m, n, &o, x_b, b_ixs, trace_pq, trace_cap, res);
	}
	return solve_multi<double>(A, b, c, m, n, opt, devices, ndev, x_b, b_ixs, trace_pq, trace_cap, res);
}

int b200lp_solve_f32_multi(const float* A, const float* b, const float* c, int64_t m, int64_t n,
		const b200lp_options* opt, const int32_t* devices, int32_t ndev, float* x_b, int32_t* b_ixs,
		int32_t* trace_pq, int64_t trace_cap, b200lp_result* res) {
	if (!devices || ndev < 1 || ndev > MAXR) return fail(B200LP_ERR_ARG, "need 1 <= ndev <= 8 device ordinals");
	if (ndev == 1) {
		b200lp_options o;
		if (opt) o = *opt; else b200lp_default_options(&o);
		o.device = devices[0];
		return solve_once<float>(A, b, c, m, n, &o, x_b, b_ixs, trace_pq, trace_cap, res);
	}
	return solve_multi<float>(A, b, c, m, n, opt, devices, ndev, x_b, b_ixs, trace_pq, trace_cap, res);
}

int b200lp_create_multi(int32_t dtype, int64_t m, int64_t n, const int32_t* devices, int32_t ndev,
		const b200lp_options* opt, b200lp_engine** out) {
	if (dtype == B200LP_F64) return create_multi<double>(m, n, opt, devices, ndev, out);
	if (dtype == B200LP_F32) return create_multi<float>(m, n, opt, devices, ndev, out);
	return fail(B200LP_ERR_ARG, "dtype must be B200LP_F32 or B200LP_F64");
}

int b200lp_create(int32_t dtype, int64_t m, int64_t n, const b200lp_options* opt, b200lp_engine** out) {
	if (dtype == B200LP_F64) return create_engine<double>(m, n, opt, out);
	if (dtype == B200LP_F32) return create_engine<float>(m, n, opt, out);
	return fail(B200LP_ERR_ARG, "dtype must be B200LP_F32 or B200LP_F64");
}

int b200lp_create_sharded(int32_t dtype, int64_t m, int64_t n, int32_t rank, int32_t nranks, const b200lp_options* opt,
		b200lp_engine** out) {
	if (dtype == B200LP_F64) return create_engine<double>(m, n, opt, out, rank, nranks);
	if (dtype == B200LP_F32) return create_engine<float>(m, n, opt, out, rank, nranks);
	return fail(B200LP_ERR_ARG, "dtype must be B200LP_F32 or B200LP_F64");
}

#define NEED(e) do { if (!(e)) return fail(B200LP_ERR_ARG, "engine is NULL"); } while (0)

int b200lp_ipc_handle_bytes(void) { return (int)(2 * sizeof(cudaIpcMemHandle_t)); }
int b200lp_ipc_export(b200lp_engine* e, void* out) { NEED(e); if (!out) return fail(B200LP_ERR_ARG, "out is NULL"); return e->ipc_export(out); }
int b200lp_ipc_import(b200lp_engine* e, const void* all, int32_t nranks) { NEED(e); if (!all) return fail(B200LP_ERR_ARG, "handles are NULL"); return e->ipc_import(all, nranks); }
int b200lp_shard_rows(b200lp_engine* e, int64_t* row0, int64_t* rows) { NEED(e); return e->shard_rows(row0, rows); }
int b200lp_shard_columns(b200lp_engine* e, int64_t* col0, int64_t* ncols) { NEED(e); return e->shard_columns(col0, ncols); }
int b200lp_check_basis(b200lp_engine* e, double* xb_err, double* xb_scale) { NEED(e); return e->check_basis(xb_err, xb_scale); }
int b200lp_profile_stamps(void) { return NSTAMP; }
const char* b200lp_profile_names(void) { return PROFILE_NAMES_JSON; }
int b200lp_download_profile(b200lp_engine* e, uint64_t* out, int64_t cap_iters, int64_t* n_iters) { NEED(e); return e->download_profile(out, cap_iters, n_iters); }
int b200lp_upload_columns(b200lp_engine* e, const void* Acols, int64_t col0, int64_t ncols, const void* b, const void* c) {
	NEED(e);
	if (!Acols || !b || !c) return fail(B200LP_ERR_ARG, "Acols, b, c must not be NULL");
	return e->upload_columns(Acols, col0, ncols, b, c);
}

int b200lp_set_memory_cache(int32_t on) {
	b200lp_engine* drop = nullptr;
	int prev;
	{
		std::lock_guard<std::mutex> lk(g_cache.mu);
		prev = g_cache.on ? 1 : 0;
		g_cache.on = on != 0;
		if (!g_cache.on) { drop = g_cache.e; g_cache.e = nullptr; }
	}
	delete drop;
	return prev;
}

int b200lp_destroy(b200lp_engine* e) { delete e; return B200LP_OK; }
int b200lp_upload(b200lp_engine* e, const void* A, const void* b, const void* c) {
	NEED(e);
	if (!A || !b || !c) return fail(B200LP_ERR_ARG, "A, b, c must not be NULL");
	return e->upload(A, b, c);
}
int b200lp_generate_dense(b200lp_engine* e, uint64_t seed) { NEED(e); return e->generate_dense(seed); }
int b200lp_reset(b200lp_engine* e) { NEED(e); return e->reset(); }
int b200lp_run(b200lp_engine* e, int64_t iterations, b200lp_result* res) {
	NEED(e);
	int rc = e->run_async(iterations);
	if (rc) return rc;
	return e->wait(res);
}
int b200lp_run_async(b200lp_engine* e, int64_t iterations) { NEED(e); return e->run_async(iterations); }
int b200lp_wait(b200lp_engine* e, b200lp_result* res) { NEED(e); return e->wait(res); }
int b200lp_phase_info(b200lp_engine* e, int32_t* phase, int64_t* shifted_columns, int64_t* phase1_pivots) {
	NEED(e);
	return e->phase_info(phase, shifted_columns, phase1_pivots);
}
int b200lp_abort(b200lp_engine* e) { NEED(e); return e->abort(); }
int b200lp_refactor(b200lp_engine* e, double rel_pivot_tol, int64_t* replayed) { NEED(e); return e->refactor(rel_pivot_tol, replayed); }

// run() in windows with a drift check after each; refactorise when |B^-1 b - x_b| exceeds drift_tol * max|x_b|
int b200lp_run_guarded(b200lp_engine* e, int64_t iterations, int64_t window, double drift_tol, b200lp_result* res,
		int64_t* refactorisations) {
	NEED(e);
	if (window <= 0) return fail(B200LP_ERR_ARG, "window must be positive");
	int64_t left = iterations, nref = 0;
	b200lp_result r;
	std::memset(&r, 0, sizeof(r));
	double ms = 0;
	while (left > 0) {
		const int64_t w = std::min(left, window);
		int rc = e->run_async(w);
		if (!rc) rc = e->wait(&r);
		if (rc) return rc;
		ms += r.ms_solve;
		left -= w;
		if (r.status != B200LP_STATUS_MAX_ITER || r.aborted) break;
		double err = 0, scale = 0;
		if ((rc = e->check_basis(&err, &scale))) return rc;
		if (err > drift_tol * std::max(scale, 1.0)) {
			if ((rc = e->refactor(0, nullptr))) return rc;
			++nref;
		}
	}
	r.ms_solve = ms;
	if (res) *res = r;
	if (refactorisations) *refactorisations = nref;
	return B200LP_OK;
}
int b200lp_download(b200lp_engine* e, void* x_b, int32_t* b_ixs, void* y) { NEED(e); return e->download(x_b, b_ixs, y); }
int b200lp_download_binv(b200lp_engine* e, void* Binv) { NEED(e); if (!Binv) return fail(B200LP_ERR_ARG, "Binv is NULL"); return e->download_binv(Binv); }
int b200lp_download_trace(b200lp_engine* e, int32_t* pq, int64_t cap, int64_t* n_out) { NEED(e); return e->download_trace(pq, cap, n_out); }
int b200lp_phase_price(b200lp_engine* e, int64_t* p, double* min_e) { NEED(e); return e->phase_price(p, min_e); }
int b200lp_phase_update_ftran(b200lp_engine* e, int64_t p) { NEED(e); return e->phase_update_ftran(p); }
int b200lp_phase_ratio(b200lp_engine* e, int64_t* q, int64_t* eligible) { NEED(e); return e->phase_ratio(q, eligible); }
int b200lp_phase_pivot_update(b200lp_engine* e, int64_t p, int64_t q) { NEED(e); return e->phase_pivot_update(p, q); }
int b200lp_download_vector(b200lp_engine* e, int32_t which, void* out) { NEED(e); return e->download_vector(which, out); }

void* b200lp_stream(b200lp_engine* e) { return e ? (void*)e->stream : nullptr; }
int b200lp_grid_ctas(b200lp_engine* e) { return e ? e->grid : 0; }
int b200lp_dense_columns(b200lp_engine* e) { return e ? (int)e->ns : 0; }
int64_t b200lp_bytes_per_pivot(b200lp_engine* e) { return e ? e->bytes_per_pivot() : 0; }
const char* b200lp_last_error(void) { return g_err.c_str(); }
const char* b200lp_version(void) { return "b200lp 0.2 (sm_100a)"; }
int b200lp_sizeof_options(void) { return (int)sizeof(b200lp_options); }
int b200lp_sizeof_result(void) { return (int)sizeof(b200lp_result); }

} // extern "C"
