/*
 * TEST INFRASTRUCTURE — NOT PRODUCT CODE.
 * CPU reference of the dual simplex loop and of the composite method (see dual_oracle_impl.h).  The summation-order helpers (dot_seq,
 * dot_block256, dot_sliced) are the primal oracle's own, taken from oracle/simplex_oracle_impl.h unchanged.
 * Build: see __init__.py (gcc -O3 -fopenmp -ffp-contract=off, the primal oracle's flags)
 */
#include "../oracle/simplex_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

typedef struct {
	int status;      /* 0 max_iter, 1 optimum, 4 infeasible, 5 not dual feasible */
	long iterations;
	long pivots;
	double z;
	double min_e;    /* min e_j of the last column pass */
	int phase;       /* composite method: 1 dual loop on the shifted costs, 2 primal loop; 0 without cost_shift */
	long shifted;    /* columns the cost shift moved */
	long phase1_pivots;
} dual_result;

#define REAL double
#define SUFFIX _f64
#define FMA(a, b, c) fma((a), (b), (c))
#include "../oracle/simplex_oracle_impl.h"
#include "dual_oracle_impl.h"
#undef REAL
#undef SUFFIX
#undef FMA

#define REAL float
#define SUFFIX _f32
#define FMA(a, b, c) fmaf((a), (b), (c))
#include "../oracle/simplex_oracle_impl.h"
#include "dual_oracle_impl.h"
#undef REAL
#undef SUFFIX
#undef FMA
