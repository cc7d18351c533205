/*
 * b200lp — C ABI of the B200-native dense revised-simplex engine.
 *
 * Drop-in boundary for the reference's solver entry point
 *     std::pair<real, SolveStatus> solve(real* A, real* b, real* c, real* x_b,
 *                                        int* b_ixs, int m, int n, TimeStruct& t)
 * (reference: src/v4_cub_reduction.cu:219, called once from main at :423).
 * Plain pointers and sizes only; no C++/torch types cross this boundary.
 *
 * Conventions shared with the reference:
 *   - A is column-major m x n (v4:59-60), n counts ALL columns, the slack
 *     (identity) block is the LAST m columns (v4:272-277); requires m <= n
 *     (v4:402).
 *   - standard form  max c'x  s.t.  Ax <= b, x >= 0, slack starting basis.
 *   - entering column: most negative reduced cost over all n columns, lowest
 *     index on ties (v4:288-302); optimal iff min >= -eps (v4:299).
 *   - leaving row: min x_b/alpha over alpha > 0 (strict), lowest index on
 *     ties; unbounded iff no row is eligible (v4:199-208, 319-325).
 *   - x_b / b_ixs are returned in basis order, slack variables included
 *     (v4:366-367, printed at v4:429-430).
 *
 * Every function returns B200LP_OK (0) or a negative error code; nothing in
 * the library calls exit() (the reference does, v4:67-92).  Solver outcomes
 * are statuses, not errors (v4:426-445).
 */
#ifndef B200LP_H
#define B200LP_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- solver outcome: mirrors `enum class SolveStatus` (v4:49-54) ---- */
#define B200LP_STATUS_MAX_ITER       0
#define B200LP_STATUS_OPTIMUM        1
#define B200LP_STATUS_UNBOUNDED      2
#define B200LP_STATUS_THETA_OVERFLOW 3 /* unreachable, kept for enum parity (v1 only) */
/* dual simplex only (options.algorithm = 1): */
#define B200LP_STATUS_INFEASIBLE     4 /* no entering column for the leaving row r: row r of B^-1 proves Ax <= b,
                                          x >= 0 infeasible (rho.b = x_b[r] < 0, rho.a_j >= 0 for every nonbasic j) */
#define B200LP_STATUS_NOT_DUAL_FEASIBLE 5 /* some reduced cost e_j < -eps: the dual method cannot start (or continue)
                                          from this basis; the primal method (algorithm = 0) applies */

/* ---- error codes ---- */
#define B200LP_OK            0
#define B200LP_ERR_ARG      -1 /* bad sizes / NULL pointers / m > n (v4:402) */
#define B200LP_ERR_CUDA     -2 /* CUDA runtime failure, see b200lp_last_error() */
#define B200LP_ERR_NO_GPU   -3 /* no sm_100 device: there is no CPU fallback */
#define B200LP_ERR_STATE    -4 /* call order (e.g. run before upload) */

/* ---- scalar type of an engine (`using real = float`, v4:12) ---- */
#define B200LP_F32 0
#define B200LP_F64 1

typedef struct b200lp_engine b200lp_engine; /* opaque */

typedef struct {
	double  eps;          /* optimality tolerance, reference EPS = 1e-4 (v4:18) */
	int64_t max_iter;     /* iteration cap, reference MAX_ITER = 5 (v4:19) */
	int32_t device;       /* CUDA device ordinal */
	int32_t grid_ctas;    /* persistent grid size; 0 = auto (multiple of the SM count) */
	int32_t tile_shape;   /* update+FTRAN tile: 0 = auto, else warps along columns 1|2|4|8 */
	int32_t check_slack;  /* 1: verify that the last m columns are the identity (default);
	                         0: trust the caller like the reference does (v4:272) */
	int32_t mode;         /* 0 = persistent cooperative kernel, 1 = one launch per phase */
	int32_t profile;      /* > 0: record phase time stamps for the first `profile` iterations of every
	                         persistent launch (b200lp_download_profile); 0 = off (default) */
	int32_t price_cols;   /* pricing group width: 0 = auto, else 2 | 4 columns per TMA block */
	int32_t l2_persist_mb; /* pin the head of B^-1 in the persisting part of L2: -1 = off (default), 0 = as much as
	                          the device allows, else MiB */
	int32_t price_mode;   /* 0 = auto (register-staged loads), 1 = TMA ring (cp.async.bulk + mbarrier), 2 = register-staged */
	int32_t ratio_group_rows; /* rows of B^-1 whose ratio test runs as one unit inside the update+FTRAN pass: 0 = auto (256) */
	double  pivot_tol;    /* ratio-test eligibility alpha > pivot_tol; 0 (default) = the reference's strict test (v4:203) */
	int32_t price_tail;   /* columns at the end of a pricing pass handed out one at a time: 0 = auto, -1 = none, else count */
	int32_t fuse_book2;   /* x_b / y / c_b / b_ixs updates in the prologue of the next pricing pass (4 grid barriers per
	                         pivot instead of 5): 0 = auto (when y fits in shared memory), -1 = off */
	int32_t fuse_ratio;   /* ratio test of every row group inside the update+FTRAN pass as the group completes:
	                         0 = auto (off: measured slower, DESIGN.md 3), 1 = on, -1 = off (the ratio test is a
	                         phase of its own after a grid barrier) */
	int32_t pricing_rule; /* 0 = Dantzig, the reference's rule (v4:288-302); 1 = steepest edge with the Goldfarb-Reid
	                         recurrence (the reference's to-do list, README.md:16-17): a different pivot sequence, far
	                         fewer pivots, one more read of B^-1 per pivot (and, sharded, one more exchange); persistent kernels */
	int32_t ratio_mode;   /* ratio test (the reference's open items, README.md:29-30): 0 = textbook, the reference's
	                         (v4:199-208); 1 = bounded: theta = max(x_b, 0) / alpha, a slightly negative x_b never
	                         yields a negative step; 2 = Harris two-pass: theta_max = min (max(x_b,0) + harris_delta) / alpha,
	                         then the LARGEST alpha among the rows with max(x_b,0)/alpha <= theta_max (one more O(m) pass
	                         and grid barrier; single GPU).  Mirrored by the oracle (oracle_opts). */
	int32_t resident;     /* mid-size LPs (m ~ 128 ... 1500): keep A and B^-1 in the shared memory of the whole grid
	                         (simplex_resident): 0 = auto (when they fit), -1 = never */
	double  harris_delta; /* ratio_mode 2: feasibility tolerance of the first pass (e.g. 1e-9) */
	int32_t algorithm;    /* 0 = primal simplex (default, everything above); 1 = dual simplex from the slack basis, for
	                         LPs with "<=" rows of negative b (">=" constraints) and a dual feasible start (e.g. c <= 0).
	                         One iteration:
	                           r = argmin (x_b[i], i), lowest index on ties;
	                           e_j = y.a_j - c_j for all n columns and, when x_b[r] < -eps, alpha_rj = rho.a_j with
	                             rho = row r of B^-1, from the same pass over A;
	                           min e_j < -eps -> B200LP_STATUS_NOT_DUAL_FEASIBLE; x_b[r] >= -eps -> OPTIMUM;
	                           p = argmin (max(e_j, 0) / -alpha_rj, j) over the nonbasic columns with
	                             alpha_rj < -pivot_tol; none -> B200LP_STATUS_INFEASIBLE;
	                           pivot on (p, q = r) exactly like the primal loop.
	                         iterations, pivots, trace, z and min_reduced_cost (min e_j of the last pass) keep their
	                         primal meaning.  Single GPU, general persistent kernel at every size (simplex_dual;
	                         tiny batches of b200lp_solve_batch_*: simplex_tiny_batch_dual, the same bits);
	                         needs pricing_rule = 0, ratio_mode = 0, mode = 0 and fuse_ratio <= 0, else B200LP_ERR_ARG
	                         (checked before any device call, like algorithm outside {0, 1} and ndev > 1). */
	int32_t cost_shift;   /* 1 (with algorithm = 1): composite method for LPs whose slack basis is neither primal
	                         feasible (some b_i < 0) nor dual feasible (some c_j > 0), e.g. max c.x with ">=" rows.
	                         No columns are added; both phases are the existing loops.
	                           shift: at the first run after upload / generate_dense / reset (slack basis, y = c_b),
	                             e_j = y.a_j - c_j for every nonbasic column (the dual pricing's association); where
	                             e_j < -eps, c'_j = y.a_j - delta_j with delta_j = shift_delta * (1 + |c_j|), else c'_j = c_j.
	                             Slack columns are basic and never shifted.  The engine keeps the original c apart.
	                           phase 1: the dual loop above on c' (its start is dual feasible by construction).
	                             INFEASIBLE ends the run (feasibility does not depend on c); NOT_DUAL_FEASIBLE is only
	                             possible through rounding drift and is reported as is.  OPTIMUM with no shifted
	                             column ends the run: it is the plain algorithm = 1 run, status included.
	                           hand-over (after a phase-1 OPTIMUM with a shifted column): the pending rank-1 update
	                             is applied, c is restored, c_b[i] = c[b_ixs[i]], and y = c_b^T B^-1 when phase 1 made
	                             a pivot (B^-1 = I otherwise and y stays).
	                           phase 2: the primal loop (Dantzig, textbook ratio test, pivot_tol) from that basis with
	                             the original c, in whichever primal kernel algorithm = 0 would pick.  It ends in
	                             OPTIMUM, UNBOUNDED or MAX_ITER.
	                         iterations, pivots and the trace run across both phases; max_iter and b200lp_run(e, k)
	                         count the total; the phase-1 check that finds x_b >= -eps is one iteration.  A window that
	                         ends on the phase-1 OPTIMUM performs the hand-over and reports MAX_ITER with z = c_b.x_b for
	                         the original c.  z and min_reduced_cost are the current phase's: after a stop inside phase 1
	                         they refer to c'.  Needs algorithm = 1 (and so everything algorithm = 1 needs), else
	                         B200LP_ERR_ARG before any device call.  0 = off (default). */
	double  shift_delta;  /* cost_shift: relative size of the shift (delta_j above); 0 = default 1e-7; < 0 or NaN:
	                         B200LP_ERR_ARG */
} b200lp_options;

typedef struct {
	int32_t status;       /* B200LP_STATUS_* */
	int32_t aborted;      /* 1: the run ended early because of b200lp_abort() (status stays MAX_ITER) */
	int64_t iterations;   /* number of "# Iteration k" lines the reference prints (v4:287) */
	int64_t pivots;
	double  z;            /* c_b . x_b (v4:365) */
	double  min_reduced_cost; /* last pricing minimum */
	double  ms_upload;    /* host->device, CUDA events */
	double  ms_solve;     /* pivot loop on the device, CUDA events */
	double  ms_download;  /* device->host */
	int64_t kernel_launches;
} b200lp_result;

/* defaults: eps 1e-4, max_iter 5 (the reference's constants), device 0, auto grid, algorithm 0, cost_shift 0 (off),
 * shift_delta 0 (= 1e-7 when cost_shift is on) */
void b200lp_default_options(b200lp_options* opt);

/*
 * One-call replacement of the reference's solve() (v4:219): host buffers in,
 * host buffers out; allocates and frees all device state per call like the
 * reference (v4:245-264, 370-377).  x_b (m) and b_ixs (m) are written for
 * every status (the reference only fills them on OptimumFound, v4:363-368).
 * trace_pq (optional) receives (p, q) per pivot, 2*trace_cap ints.
 */
int b200lp_solve_f64(const double* A, const double* b, const double* c, int64_t m, int64_t n,
		const b200lp_options* opt, double* x_b, int32_t* b_ixs,
		int32_t* trace_pq, int64_t trace_cap, b200lp_result* res);
int b200lp_solve_f32(const float* A, const float* b, const float* c, int64_t m, int64_t n,
		const b200lp_options* opt, float* x_b, int32_t* b_ixs,
		int32_t* trace_pq, int64_t trace_cap, b200lp_result* res);

/*
 * The same call over several GPUs of one box (SURVEY.md 8(b2): `devices, ndev`): one process, one persistent kernel
 * per device, B^-1 row-sharded and A column-sharded across them, peer access instead of CUDA IPC.  `devices` lists
 * ndev CUDA ordinals (1..8).  A device may be repeated: its ranks then share one cooperative launch (used by the
 * tests on single-GPU boxes; it buys no speed).  Results are bit-identical to the single-GPU call.
 */
int b200lp_solve_f64_multi(const double* A, const double* b, const double* c, int64_t m, int64_t n,
		const b200lp_options* opt, const int32_t* devices, int32_t ndev, double* x_b, int32_t* b_ixs,
		int32_t* trace_pq, int64_t trace_cap, b200lp_result* res);
int b200lp_solve_f32_multi(const float* A, const float* b, const float* c, int64_t m, int64_t n,
		const b200lp_options* opt, const int32_t* devices, int32_t ndev, float* x_b, int32_t* b_ixs,
		int32_t* trace_pq, int64_t trace_cap, b200lp_result* res);

/*
 * Many independent LPs of ONE shape in one call (scenario subproblems, parameter sweeps, per-sample LPs).
 *
 * Layout: A is `batch` consecutive column-major m x n matrices (leading dimension m), b is batch x m, c is
 * batch x n.  x_b, b_ixs and y are batch x m; trace_pq is batch x trace_cap x 2 ints, entries past an LP's
 * pivots are -1.  y and trace_pq may be NULL; a non-NULL trace_pq with trace_cap = 0 receives nothing.
 * res points to `batch` records: status, iterations, pivots, z and min_reduced_cost are LP k's, aborted is 0;
 * ms_upload / ms_solve / ms_download / kernel_launches are the whole call's, repeated in every record.
 * max_iter applies to every LP on its own; check_slack decides per LP whether its last m columns are priced as
 * unit vectors (identity) or stored like the rest (data), as in the single call.
 *
 * Contract: record k and row k of every output are bit-identical to b200lp_solve_f64 / _f32 called on LP k alone
 * with the same options (y: to b200lp_download after such a run).
 *
 * Selection: the LPs run in one kernel, one CTA per LP on a persistent grid with all of an LP in shared memory,
 * when m <= 64 (f64) / 128 (f32), A, B^-1 and the vectors of the LP with the most stored columns fit in 200 KB of
 * shared memory and max_iter > 0: simplex_tiny_batch for algorithm = 0 with pricing_rule = 0 and ratio_mode != 2,
 * simplex_tiny_batch_dual for algorithm = 1 with or without cost_shift (the dual's layout adds one byte per
 * column, its nonbasic mask, to the 200 KB test).  That kernel runs the single call's sequence per LP: the cost shift,
 * the dual loop, the hand-over and the primal loop.  Otherwise the LPs run one after another on
 * one engine (the single call's path without its per-call allocation), so the call accepts every shape and option
 * b200lp_solve_* accepts.  The single-engine tuning options grid_ctas, tile_shape, mode, profile, price_cols,
 * price_mode, price_tail, fuse_book2, fuse_ratio, ratio_group_rows, resident and l2_persist_mb affect only that
 * fallback; eps, max_iter, device, check_slack, pivot_tol, pricing_rule, ratio_mode, harris_delta, algorithm,
 * cost_shift and shift_delta apply to both.
 *
 * Argument errors (B200LP_ERR_ARG, before any device call): batch <= 0, m <= 0, m > n, NULL A / b / c / x_b /
 * b_ixs / res, trace_cap < 0, an algorithm the options do not allow (see b200lp_options.algorithm).  No device:
 * B200LP_ERR_NO_GPU.
 */
int b200lp_solve_batch_f64(const double* A, const double* b, const double* c, int64_t batch, int64_t m, int64_t n,
		const b200lp_options* opt, double* x_b, int32_t* b_ixs, double* y,
		int32_t* trace_pq, int64_t trace_cap, b200lp_result* res);
int b200lp_solve_batch_f32(const float* A, const float* b, const float* c, int64_t batch, int64_t m, int64_t n,
		const b200lp_options* opt, float* x_b, int32_t* b_ixs, float* y,
		int32_t* trace_pq, int64_t trace_cap, b200lp_result* res);

/* Keep the device buffers of the last b200lp_solve_* call for the next call of the same shape, dtype and options
 * (on != 0), or release them and go back to the reference's behaviour of leaving nothing behind (on == 0, the
 * default).  Creating and freeing 16 GB of device memory costs 40-500 ms per call at m = 32768.  Returns the
 * previous setting.  Thread safe; one engine is kept per process. */
int b200lp_set_memory_cache(int32_t on);

/* ---- handle API: device state survives between calls (bench, windows, tests) ---- */

/* allocates A_N, B^-1 and all vectors for an m x n problem (v4:245-264) */
int b200lp_create(int32_t dtype, int64_t m, int64_t n, const b200lp_options* opt, b200lp_engine** out);
/* the same engine spread over ndev GPUs of this process (see b200lp_solve_f64_multi); every handle call below
 * works on it except the per-phase entry points and the IPC calls */
int b200lp_create_multi(int32_t dtype, int64_t m, int64_t n, const int32_t* devices, int32_t ndev,
		const b200lp_options* opt, b200lp_engine** out);
int b200lp_destroy(b200lp_engine* e);

/* H2D of A (col-major m x n), b (m), c (n) (v4:269-271) followed by the slack-basis
 * initial state (v4:272-279).  Pointers are host memory of the engine's dtype. */
int b200lp_upload(b200lp_engine* e, const void* A, const void* b, const void* c);

/* synthetic dense LP generated on the device (bench; same numbers as oracle/lpgen_dense_*) */
int b200lp_generate_dense(b200lp_engine* e, uint64_t seed);

/* back to the slack basis: B^-1 = I, x_b = b, y = c_b = c[n-m..n) (v4:272-277) */
int b200lp_reset(b200lp_engine* e);

/* run at most `iterations` more iterations of the loop at v4:286-359 (blocking) */
int b200lp_run(b200lp_engine* e, int64_t iterations, b200lp_result* res);
/* same, without waiting: returns after the launch; pair with b200lp_wait() */
int b200lp_run_async(b200lp_engine* e, int64_t iterations);
int b200lp_wait(b200lp_engine* e, b200lp_result* res);
/* composite method (options.cost_shift = 1): phase 0 (no run since upload / generate_dense / reset), 1 (dual loop on
 * the shifted costs) or 2 (primal loop on the original costs); shifted_columns counts the columns the shift moved,
 * phase1_pivots the pivots of phase 1.  Any pointer may be NULL.  Engines without cost_shift report 0, 0, 0. */
int b200lp_phase_info(b200lp_engine* e, int32_t* phase, int64_t* shifted_columns, int64_t* phase1_pivots);
/* touched columns of B^-1: from the slack basis only the columns of the rows that have left the basis (K) differ
 * from e_j, so the single-GPU persistent kernel's update + FTRAN pass (and the steepest-edge BTRAN) can stream K's
 * columns alone, with the same bits.  k = 0: auto (m >= 4096 and |K| <= m / 8, the default), -1: off (every pass streams
 * all of B^-1), > 0: while |K| <= k.  Applies from the next run.  Never used with the fused ratio test, on sharded
 * engines (B200LP_ERR_STATE), for m > 262144, for stored columns with an inf or NaN, and after a non-finite pivot
 * row or alpha until the next reset / refactor.  k < -1: B200LP_ERR_ARG. */
int b200lp_set_binv_sparse(b200lp_engine* e, int32_t k);
/* the touched-column state since the last reset / refactor: columns of B^-1 that may differ from e_j, and how many
 * update + FTRAN passes of the persistent kernel streamed only those.  Sharded engines report 0, 0. */
int b200lp_binv_info(b200lp_engine* e, int64_t* touched, int64_t* sparse_passes);
/* ask a running loop (b200lp_run_async, or b200lp_run on another thread) to stop at its next iteration boundary;
 * state stays consistent and the run can be continued.  The kernel polls one word per iteration. */
int b200lp_abort(b200lp_engine* e);

/* D2H of the basis-ordered solution (v4:366-367); any pointer may be NULL */
int b200lp_download(b200lp_engine* e, void* x_b, int32_t* b_ixs, void* y);
/* D2H of B^-1 (col-major m x m) after flushing a pending rank-1 update (tests) */
int b200lp_download_binv(b200lp_engine* e, void* Binv);
/* (p, q) of the first min(pivots, cap) pivots */
int b200lp_download_trace(b200lp_engine* e, int32_t* trace_pq, int64_t cap, int64_t* n_out);

/* ---- per-phase entry points (unit tests, sharded multi-GPU driver) ----
 * Each runs ONE phase of the pivot as its own launch on the engine's stream and
 * waits for it.  Order within a pivot: price -> update_ftran -> ratio -> pivot_update.  These are the phases of the
 * primal loop, whatever options.algorithm says. */
/* pricing fused with argmin (replaces cublasSgemm + cub ArgMin, v4:289-296) */
int b200lp_phase_price(b200lp_engine* e, int64_t* p, double* min_e);
/* pending rank-1 update of B^-1 fused with alpha = B^-1 A[:,p] (v4:307-308 + v4:333 of the previous pivot) */
int b200lp_phase_update_ftran(b200lp_engine* e, int64_t p);
/* fused masked-argmin ratio test (v4:311-325); eligible = number of rows with alpha > 0 */
int b200lp_phase_ratio(b200lp_engine* e, int64_t* q, int64_t* eligible);
/* row extract, E_q, c_b/b_ixs bookkeeping, x_b and y updates (v4:331-332, 339-356) */
int b200lp_phase_pivot_update(b200lp_engine* e, int64_t p, int64_t q);
/* device vectors for inspection: which = 0 alpha, 1 E_q, 2 row_q, 3 x_b, 4 y, 5 c_b (length m); steepest edge
 * (pricing_rule = 1) only: 6 v = B^-T alpha of the last pivot (length m), 7 the weights gamma (length n) */
int b200lp_download_vector(b200lp_engine* e, int32_t which, void* out);

/* ---- sharded engine: one process per GPU of one NVSwitch box (SURVEY.md 8(e)) ----
 * B^-1 is row-block sharded, A column-block sharded, all O(m) vectors replicated; every
 * rank runs the same persistent kernel and the three per-pivot exchanges (pricing
 * candidates, FTRAN result slices, pivot row) are direct peer stores over NVLink into
 * IPC-mapped mailboxes.  The reference is single-GPU (v4:219-380 has no peer, stream or
 * NCCL call), so these entry points have no counterpart there.
 * Call order on EVERY rank: create_sharded -> upload | generate_dense -> ipc_export ->
 * (all-gather the handle blobs with any host transport) -> ipc_import -> run (same
 * iteration count on all ranks) -> download.  Results are replicated and bit-identical
 * to the single-GPU engine. */
int b200lp_create_sharded(int32_t dtype, int64_t m, int64_t n, int32_t rank, int32_t nranks,
		const b200lp_options* opt, b200lp_engine** out);
int b200lp_ipc_handle_bytes(void);                       /* size of one rank's handle blob */
int b200lp_ipc_export(b200lp_engine* e, void* out);      /* this rank's blob */
int b200lp_ipc_import(b200lp_engine* e, const void* all, int32_t nranks); /* nranks blobs, rank order */
int b200lp_shard_rows(b200lp_engine* e, int64_t* row0, int64_t* rows);    /* B^-1 rows owned here */
int b200lp_shard_columns(b200lp_engine* e, int64_t* col0, int64_t* ncols); /* structural columns of A owned here */
/* H2D of this rank's column block only (col-major m x ncols, starting at column col0 of A);
 * the caller vouches for the identity slack block, which is never transferred */
int b200lp_upload_columns(b200lp_engine* e, const void* Acols, int64_t col0, int64_t ncols,
		const void* b, const void* c);

/* ---- numerical health (the reference lists refactorisation / small-pivot guards as open, README.md:29-30) ----
 * max_i |(B^-1 b)_i - x_b_i| and max_i |x_b_i| after flushing a pending rank-1 update: how far the product-form
 * inverse and the linearly updated x_b (v4:347-348) have drifted apart.  One extra pass over B^-1; call it between
 * runs (it overwrites alpha).  Changes nothing the loop reads afterwards.  On a sharded engine (one rank of a
 * multi-process run) the maxima are over the rank's own rows; b200lp_create_multi engines return the global ones. */
int b200lp_check_basis(b200lp_engine* e, double* xb_err, double* xb_scale);

/* Refactorisation: rebuild B^-1 from the current basis alone (identity + one replayed pivot per non-slack basis
 * position, the loop's own update + FTRAN kernel), then x_b = B^-1 b and y = c_b^T B^-1 from the fresh inverse.
 * The reference never does this (README.md:29-30 lists the numerical guards as open); nothing in the parity runs
 * calls it.  rel_pivot_tol: a replay pivot needs |alpha_q| >= rel_pivot_tol * max|alpha| (<= 0: 1e-9); positions that
 * do not qualify yet are retried later.  replayed (optional) receives the number of replayed pivots.  Single GPU.
 * After it the basis (b_ixs, c_b) is unchanged, the pivot counters too. */
int b200lp_refactor(b200lp_engine* e, double rel_pivot_tol, int64_t* replayed);
/* b200lp_run in windows of `window` iterations with b200lp_check_basis after each one and b200lp_refactor whenever
 * the drift exceeds drift_tol * max|x_b|.  refactorisations (optional) counts them. */
int b200lp_run_guarded(b200lp_engine* e, int64_t iterations, int64_t window, double drift_tol, b200lp_result* res,
		int64_t* refactorisations);

/* ---- in-kernel phase profile (options.profile > 0) ----
 * CTA 0 of the persistent kernel stamps %globaltimer (ns) at every phase boundary; one record of
 * b200lp_profile_stamps() values per iteration of the LAST launch (0 = point not reached).
 * Replaces the reference's unsynchronised host chrono timers (v4:293-297, 330-357, 456-471). */
int b200lp_profile_stamps(void);
const char* b200lp_profile_names(void);   /* JSON: interval names of the single-GPU and the sharded loop */
int b200lp_download_profile(b200lp_engine* e, uint64_t* out, int64_t cap_iters, int64_t* n_iters);

/* ---- synthetic input (bench / tests) ----
 * Host-side twin of b200lp_generate_dense: columns [col0, col0 + ncols) of the full
 * [A_s, I_m] matrix (col-major m x ncols) and, when non-NULL, b (m) and c (n). */
int b200lp_lpgen_dense_host(int32_t dtype, void* A_cols, void* b, void* c, int64_t m, int64_t n,
		int64_t col0, int64_t ncols, uint64_t seed);

/* ---- introspection ---- */
void*       b200lp_stream(b200lp_engine* e);     /* cudaStream_t the engine launches on */
int         b200lp_grid_ctas(b200lp_engine* e);
int         b200lp_dense_columns(b200lp_engine* e); /* n - m when the slack block was recognised */
int64_t     b200lp_bytes_per_pivot(b200lp_engine* e); /* algorithmic bytes: s*(2 m^2 + m (n-m)) */
const char* b200lp_last_error(void);
const char* b200lp_version(void);
/* sizeof(b200lp_options) / sizeof(b200lp_result) of the library build: lets a binding check its mirror of the structs */
int         b200lp_sizeof_options(void);
int         b200lp_sizeof_result(void);

#ifdef __cplusplus
}
#endif
#endif /* B200LP_H */
