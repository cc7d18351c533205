/*
 * TEST INFRASTRUCTURE — NOT PRODUCT CODE.
 *
 * CPU reference of the dual simplex loop (options.algorithm = 1 of include/b200lp.h) and of the composite method
 * built on it (options.cost_shift = 1), included twice by dual_oracle.c (REAL = double / float).  The basis change,
 * the FTRAN and every bookkeeping sum are the primal oracle's (oracle/simplex_oracle_impl.h), in both orders:
 *   order 0 ... plain left-to-right fma chains
 *   order 1 ... the B200 engine's associations (dot_block256 for the column dots, dot_sliced for the O(m) dots,
 *               32-column sub-blocks and 256-column chunks for the FTRAN), so engine results compare bit for bit.
 * The inverse here is always flushed, so rho = row r of Binv is what the engine forms as
 * fma(E_q[r], row_q[j], B[r,j]) from its deferred rank-1 update.
 *
 * One dual iteration:
 *   r = argmin (x_b[i], i)                                      leaving row, lowest index on ties
 *   e_j = y.a_j - c_j; alpha_j = rho.a_j when x_b[r] < -eps     rho = row r of Binv; slack columns need no dot
 *   min e < -eps -> NOT_DUAL_FEASIBLE (5); x_b[r] >= -eps -> OPTIMUM (1)
 *   p = argmin (max(e_j,0) / -alpha_j, j) over nonbasic j with alpha_j < -pivot_tol; none -> INFEASIBLE (4)
 *   pivot on (p, q = r) exactly like the primal loop
 *
 * Composite method (cost_shift = 1):
 *   shift     from the slack basis (y = c_b): s = y.a_j, e_j = s - c_j for the nonbasic columns (the dual pricing's
 *             association); e_j < -eps -> c'_j = s - shift_delta * (1 + |c_j|), counted
 *   phase 1   the dual loop above on c'
 *   hand-over after a phase-1 OPTIMUM with a shifted column (the check counts as one iteration): c restored,
 *             c_b[i] = c[b_ixs[i]], y_j = c_b . Binv[:, j] when phase 1 pivoted (k_btran_vec's association)
 *   phase 2   the primal loop: Dantzig pricing, textbook ratio test alpha > pivot_tol, lowest index on ties
 */

#define CAT_(a, b) a##b
#define CAT(a, b) CAT_(a, b)
#define FN(name) CAT(name, SUFFIX)

/* alpha = Binv a_p (the primal oracle's FTRAN, both orders) */
static void FN(dual_ftran)(const REAL* Binv, const REAL* a_p, REAL* alpha, long m, int order) {
	if (order == 0) {
		for (long i = 0; i < m; ++i) alpha[i] = (REAL)0;
		#pragma omp parallel for schedule(static)
		for (long i0 = 0; i0 < m; i0 += 512) {
			long i1 = i0 + 512 < m ? i0 + 512 : m;
			for (long j = 0; j < m; ++j) {
				const REAL aj = a_p[j];
				const REAL* bc = Binv + j * m;
				for (long i = i0; i < i1; ++i) alpha[i] = FMA(bc[i], aj, alpha[i]);
			}
		}
		return;
	}
	#pragma omp parallel for schedule(static)
	for (long i0 = 0; i0 < m; i0 += 256) {
		long i1 = i0 + 256 < m ? i0 + 256 : m;
		REAL tot[256], sub[8][256];
		for (long j0 = 0; j0 < m; j0 += 256) {
			for (int sb = 0; sb < 8; ++sb) {
				for (long i = i0; i < i1; ++i) sub[sb][i - i0] = (REAL)0;
				long ja = j0 + sb * 32, jb = ja + 32 < m ? ja + 32 : m;
				for (long j = ja; j < jb; ++j) {
					const REAL aj = a_p[j];
					const REAL* bc = Binv + j * m;
					for (long i = i0; i < i1; ++i) sub[sb][i - i0] = FMA(bc[i], aj, sub[sb][i - i0]);
				}
			}
			for (long i = i0; i < i1; ++i) {
				const long rr = i - i0;
				const REAL c8 = ((sub[0][rr] + sub[1][rr]) + (sub[2][rr] + sub[3][rr]))
				              + ((sub[4][rr] + sub[5][rr]) + (sub[6][rr] + sub[7][rr]));
				tot[rr] = j0 == 0 ? c8 : tot[rr] + c8;
			}
		}
		for (long i = i0; i < i1; ++i) alpha[i] = tot[i - i0];
	}
}

/* basis change on (p, q): row extract + E_q + rank-1 update, bookkeeping, nonbasic mask, x_b and y (the primal
 * oracle's pivot, costs c) */
static void FN(dual_pivot)(const REAL* b, const REAL* c, long m, int order, long p, long q, REAL* Binv,
		const REAL* alpha, REAL* row_q, REAL* E_q, REAL* c_b, int* b_ixs, unsigned char* nb, REAL* x_b, REAL* y) {
	const REAL alpha_q = alpha[q];
	for (long j = 0; j < m; ++j) row_q[j] = Binv[q + j * m];
	for (long i = 0; i < m; ++i)
		E_q[i] = (i != q) ? (-alpha[i] / alpha_q) : (REAL)(1.0 / (double)alpha_q - 1.0);
	#pragma omp parallel for schedule(static)
	for (long j = 0; j < m; ++j) {
		const REAL rq = row_q[j];
		REAL* bc = Binv + j * m;
		for (long i = 0; i < m; ++i) bc[i] = FMA(E_q[i], rq, bc[i]);
	}

	const REAL c_b_q = c_b[q];
	const long leaving = b_ixs[q];
	c_b[q] = c[p];
	b_ixs[q] = (int)p;
	nb[p] = 0;
	nb[leaving] = 1;

	REAL s = order == 0 ? FN(dot_seq)(row_q, b, m, (REAL)0) : FN(dot_sliced)(row_q, b, m);
	for (long i = 0; i < m; ++i) x_b[i] = FMA(s, E_q[i], x_b[i]);
	s = order == 0 ? FN(dot_seq)(c_b, E_q, m, (REAL)0) : FN(dot_sliced)(c_b, E_q, m);
	s += c[p] - c_b_q;
	for (long i = 0; i < m; ++i) y[i] = FMA(s, row_q[i], y[i]);
}

int FN(dual_solve)(const REAL* A, const REAL* b, const REAL* c_in, long m, long n,
		REAL eps, long max_iter, int order, double pivot_tol_d, int cost_shift, double shift_delta,
		REAL* x_b_out, int* b_ixs_out, REAL* y_out, REAL* Binv_out,
		int* trace_p, int* trace_q, double* trace_gap_p, double* trace_gap_q,
		long trace_cap, dual_result* res) {
	if (m <= 0 || n <= 0 || m > n) return -1;
	const REAL pivot_tol = (REAL)pivot_tol_d;
	REAL* Binv = (REAL*)calloc((size_t)m * m, sizeof(REAL));
	REAL* c = (REAL*)malloc(sizeof(REAL) * n);       /* the costs priced with: c' in phase 1 of the composite method */
	REAL* c_b = (REAL*)malloc(sizeof(REAL) * m);
	REAL* x_b = (REAL*)malloc(sizeof(REAL) * m);
	REAL* y = (REAL*)malloc(sizeof(REAL) * m);
	REAL* e = (REAL*)malloc(sizeof(REAL) * n);
	REAL* ar = (REAL*)malloc(sizeof(REAL) * n);      /* alpha_rj = rho . a_j */
	REAL* rho = (REAL*)malloc(sizeof(REAL) * m);
	REAL* alpha = (REAL*)malloc(sizeof(REAL) * m);
	REAL* row_q = (REAL*)malloc(sizeof(REAL) * m);
	REAL* E_q = (REAL*)malloc(sizeof(REAL) * m);
	int* b_ixs = (int*)malloc(sizeof(int) * m);
	unsigned char* nb = (unsigned char*)malloc((size_t)n);
	if (!Binv || !c || !c_b || !x_b || !y || !e || !ar || !rho || !alpha || !row_q || !E_q || !b_ixs || !nb) return -2;

	memcpy(c, c_in, sizeof(REAL) * n);
	for (long i = 0; i < m; ++i) {
		Binv[i + i * m] = (REAL)1;
		c_b[i] = c[n - m + i];
		x_b[i] = b[i];
		b_ixs[i] = (int)(n - m + i);
		y[i] = c_b[i];
	}
	for (long j = 0; j < n; ++j) nb[j] = j < n - m;

	long ns = n;
	if (order == 1) {
		int ident = 1;
		for (long j = 0; j < m && ident; ++j)
			for (long i = 0; i < m; ++i)
				if (A[i + (n - m + j) * m] != (REAL)(i == j)) { ident = 0; break; }
		if (ident) ns = n - m;
	}

	/* ---- composite method: the cost shift from the slack basis */
	int phase = 0;
	long shifted = 0;
	if (cost_shift) {
		const REAL delta = (REAL)(shift_delta > 0 ? shift_delta : 1e-7);
		phase = 1;
		for (long j = 0; j < ns; ++j) {
			if (!nb[j]) continue;
			const REAL* col = A + j * m;
			const REAL s = order == 0 ? FN(dot_seq)(y, col, m, (REAL)0) : FN(dot_block256)(col, y, m);
			const REAL ej = order == 0 ? FN(dot_seq)(y, col, m, -c[j]) : s - c[j];
			if (ej < -eps) {
				const REAL cj = c[j];
				const REAL dj = delta * ((REAL)1 + (cj < (REAL)0 ? -cj : cj));
				c[j] = s - dj;
				++shifted;
			}
		}
	}

	int status = 0;
	long it = 0, pivots = 0, phase1_pivots = 0;
	double min_e = 0;
	do {
		if (phase == 2) {
			/* ---- primal iteration: Dantzig pricing over all n columns */
			#pragma omp parallel for schedule(static)
			for (long j = 0; j < n; ++j) {
				const REAL* col = A + j * m;
				if (order == 0) e[j] = FN(dot_seq)(y, col, m, -c[j]);
				else if (j < ns) e[j] = FN(dot_block256)(col, y, m) - c[j];
				else e[j] = y[j - ns] - c[j];
			}
			long p = 0;
			REAL mn = e[0];
			for (long j = 1; j < n; ++j)
				if (e[j] < mn) { mn = e[j]; p = j; }
			min_e = (double)mn;
			if (mn >= -eps) { status = 1; ++it; break; }
			double gap_p = INFINITY;
			for (long j = 0; j < n; ++j)
				if (j != p && (double)e[j] - (double)mn < gap_p) gap_p = (double)e[j] - (double)mn;

			FN(dual_ftran)(Binv, A + p * m, alpha, m, order);

			/* ---- textbook ratio test, lowest index on ties */
			long q = -1;
			REAL best = (REAL)INFINITY;
			for (long i = 0; i < m; ++i) {
				if (!(alpha[i] > pivot_tol)) continue;
				const REAL th = x_b[i] / alpha[i];
				if (q < 0 || th < best) { best = th; q = i; }
			}
			if (q < 0) { status = 2; ++it; break; }
			double gap_q = INFINITY;
			for (long i = 0; i < m; ++i)
				if (i != q && alpha[i] > pivot_tol && (double)(x_b[i] / alpha[i]) - (double)best < gap_q)
					gap_q = (double)(x_b[i] / alpha[i]) - (double)best;

			if (pivots < trace_cap) {
				if (trace_p) trace_p[pivots] = (int)p;
				if (trace_q) trace_q[pivots] = (int)q;
				if (trace_gap_p) trace_gap_p[pivots] = gap_p;
				if (trace_gap_q) trace_gap_q[pivots] = gap_q;
			}
			FN(dual_pivot)(b, c, m, order, p, q, Binv, alpha, row_q, E_q, c_b, b_ixs, nb, x_b, y);
			++pivots;
			continue;
		}

		/* ---- leaving row */
		long r = 0;
		REAL xr = x_b[0];
		for (long i = 1; i < m; ++i)
			if (x_b[i] < xr) { xr = x_b[i]; r = i; }
		double gap_q = INFINITY;
		for (long i = 0; i < m; ++i)
			if (i != r && (double)x_b[i] - (double)xr < gap_q) gap_q = (double)x_b[i] - (double)xr;
		const int want = xr < -eps;
		if (want)
			for (long j = 0; j < m; ++j) rho[j] = Binv[r + j * m];

		/* ---- column pass */
		#pragma omp parallel for schedule(static)
		for (long j = 0; j < n; ++j) {
			const REAL* col = A + j * m;
			if (order == 0) {
				e[j] = FN(dot_seq)(y, col, m, -c[j]);
				ar[j] = want ? FN(dot_seq)(rho, col, m, (REAL)0) : (REAL)0;
			} else if (j < ns) {
				e[j] = FN(dot_block256)(col, y, m) - c[j];
				ar[j] = want ? FN(dot_block256)(col, rho, m) : (REAL)0;
			} else {
				e[j] = y[j - ns] - c[j];
				ar[j] = want ? rho[j - ns] : (REAL)0;
			}
		}
		REAL mn = e[0];
		for (long j = 1; j < n; ++j)
			if (e[j] < mn) mn = e[j];
		min_e = (double)mn;
		if (mn < -eps) { status = 5; ++it; break; }
		if (!want) {
			if (phase == 1 && shifted > 0) {
				/* ---- hand-over to the primal loop on the original costs (this check was one iteration) */
				phase1_pivots = pivots;
				memcpy(c, c_in, sizeof(REAL) * n);
				for (long i = 0; i < m; ++i) c_b[i] = c[b_ixs[i]];
				if (pivots > 0)
					for (long j = 0; j < m; ++j)
						y[j] = order == 0 ? FN(dot_seq)(c_b, Binv + j * m, m, (REAL)0) : FN(dot_block256)(Binv + j * m, c_b, m);
				phase = 2;
				continue;
			}
			status = 1; ++it; break;
		}

		/* ---- entering column: dual ratio test over the nonbasic columns */
		long p = -1;
		REAL best = (REAL)0, second = (REAL)INFINITY;
		for (long j = 0; j < n; ++j) {
			if (!nb[j] || !(ar[j] < -pivot_tol)) continue;
			const REAL rt = (e[j] > (REAL)0 ? e[j] : (REAL)0) / -ar[j];
			if (p < 0 || rt < best) { if (p >= 0) second = best; best = rt; p = j; }
			else if (rt < second) second = rt;
		}
		if (p < 0) { status = 4; ++it; break; }
		const double gap_p = isinf((double)second) ? INFINITY : (double)second - (double)best;
		const long q = r;

		FN(dual_ftran)(Binv, A + p * m, alpha, m, order);

		if (pivots < trace_cap) {
			if (trace_p) trace_p[pivots] = (int)p;
			if (trace_q) trace_q[pivots] = (int)q;
			if (trace_gap_p) trace_gap_p[pivots] = gap_p;
			if (trace_gap_q) trace_gap_q[pivots] = gap_q;
		}
		FN(dual_pivot)(b, c, m, order, p, q, Binv, alpha, row_q, E_q, c_b, b_ixs, nb, x_b, y);
		++pivots;
	} while (++it < max_iter);
	if (phase == 1) phase1_pivots = pivots;

	REAL z = order == 0 ? FN(dot_seq)(c_b, x_b, m, (REAL)0) : FN(dot_sliced)(c_b, x_b, m);
	if (res) {
		res->status = status;
		res->iterations = it;
		res->pivots = pivots;
		res->z = (double)z;
		res->min_e = min_e;
		res->phase = phase;
		res->shifted = shifted;
		res->phase1_pivots = phase1_pivots;
	}
	if (x_b_out) memcpy(x_b_out, x_b, sizeof(REAL) * m);
	if (b_ixs_out) memcpy(b_ixs_out, b_ixs, sizeof(int) * m);
	if (y_out) memcpy(y_out, y, sizeof(REAL) * m);
	if (Binv_out) memcpy(Binv_out, Binv, sizeof(REAL) * (size_t)m * m);

	free(Binv); free(c); free(c_b); free(x_b); free(y); free(e); free(ar); free(rho); free(alpha);
	free(row_q); free(E_q); free(b_ixs); free(nb);
	return 0;
}

#undef FN
#undef CAT
#undef CAT_
