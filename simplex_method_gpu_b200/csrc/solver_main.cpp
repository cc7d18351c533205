// CLI with the driver contract of the reference's main() (src/v4_cub_reduction.cu:384-474):
//   solver.out <lp.txt | lp.b200lp> [--f64] [--eps E] [--max-iter N] [--device D] [--gpus N | --devices a,b,..] [--dual]
//              [--cost-shift]
// --dual: the dual simplex from the slack basis (options.algorithm = 1; negative b, dual feasible start), which can
// also print "Problem infeasible." or "Start not dual feasible.".
// --cost-shift (with --dual): the composite method (options.cost_shift = 1) for LPs with both negative b and positive c:
// the dual loop on shifted costs, then the primal loop on the original ones.
// Same input text format (v4:401-420; parsed by b200lp_read_lp, which also accepts the binary twin), same stdout: one "# Iteration k" line per
// iteration (v4:287), the result block (v4:426-445) and the timing block
// (v4:456-471, same labels and number format).  Defaults reproduce the reference's
// compile-time constants: real = float, EPS = 1e-4, MAX_ITER = 5 (v4:12, 18-19).
// All numerics run in libb200lp.so through the C ABI.
#include "b200lp.h"
#include "b200lp_io.h"

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iomanip>
#include <iostream>
#include <string>
#include <vector>

using Clock = std::chrono::high_resolution_clock;

static double secs(Clock::time_point a, Clock::time_point b) {
	return std::chrono::duration<double>(b - a).count();
}

// "<label>: " right-aligned in 19 columns, seconds with 2 decimals in 6 (v4:151-157)
static void print_time(const char* label, double s) {
	std::cout << std::setw(19) << (std::string(label) + ": ");
	std::cout << std::fixed << std::setprecision(2) << std::setw(6) << s << '\n';
}

static std::vector<int32_t> g_devices;   // --gpus / --devices: more than one entry = the sharded multi-GPU solve

template <typename T>
static int run(const char* path, b200lp_options opt, Clock::time_point t_start) {
	// the reference allocates its pinned host arrays first and then parses into them (v4:407-420);
	// here the reader does both, so "Host alloc" is the output arrays only
	auto t_host_alloc = Clock::now();
	auto t_read = Clock::now();
	b200lp_problem lp;
	if (b200lp_read_lp(path, sizeof(T) == 8 ? B200LP_F64 : B200LP_F32, 1, &lp) != B200LP_OK) {
		std::cerr << b200lp_last_error() << "\n";
		return 1;                                    // v4:398, 404; a short file exits with EXIT_FAILURE = 1 too (v4:100)
	}
	const long m = (long)lp.m, n = (long)lp.n;
	const T *A = (const T*)lp.A, *b = (const T*)lp.b, *c = (const T*)lp.c;
	std::vector<T> x_b((size_t)m);
	std::vector<int32_t> b_ixs((size_t)m);

	auto t_solve = Clock::now();
	b200lp_result r;
	int rc;
	if (g_devices.size() > 1) {
		if (sizeof(T) == 8)
			rc = b200lp_solve_f64_multi((const double*)A, (const double*)b, (const double*)c, m, n, &opt, g_devices.data(),
					(int32_t)g_devices.size(), (double*)x_b.data(), b_ixs.data(), nullptr, 0, &r);
		else
			rc = b200lp_solve_f32_multi((const float*)A, (const float*)b, (const float*)c, m, n, &opt, g_devices.data(),
					(int32_t)g_devices.size(), (float*)x_b.data(), b_ixs.data(), nullptr, 0, &r);
	} else if (sizeof(T) == 8)
		rc = b200lp_solve_f64((const double*)A, (const double*)b, (const double*)c, m, n, &opt,
				(double*)x_b.data(), b_ixs.data(), nullptr, 0, &r);
	else
		rc = b200lp_solve_f32((const float*)A, (const float*)b, (const float*)c, m, n, &opt,
				(float*)x_b.data(), b_ixs.data(), nullptr, 0, &r);
	if (rc != B200LP_OK) {
		std::cerr << "b200lp failed (" << rc << "): " << b200lp_last_error() << "\n";
		return EXIT_FAILURE;
	}

	auto t_print = Clock::now();
	for (int64_t i = 0; i < r.iterations; ++i) std::cout << "# Iteration " << (i + 1) << '\n';
	switch (r.status) {
	case B200LP_STATUS_OPTIMUM:
		std::cout << "Optimum found: " << (T)r.z << '\n';
		for (long i = 0; i < m; ++i) std::cout << "\tx_" << b_ixs[i] << " = " << x_b[i] << "\n";
		break;
	case B200LP_STATUS_UNBOUNDED: std::cout << "Problem unbounded.\n"; break;
	case B200LP_STATUS_THETA_OVERFLOW: std::cout << "Theta overflow.\n"; break;
	case B200LP_STATUS_INFEASIBLE: std::cout << "Problem infeasible.\n"; break;
	case B200LP_STATUS_NOT_DUAL_FEASIBLE: std::cout << "Start not dual feasible.\n"; break;
	default: std::cout << "MAX_ITER exceeded.\n"; break;
	}
	std::cout << '\n';

	auto t_free = Clock::now();
	b200lp_free_problem(&lp);
	auto t_end = Clock::now();

	// the pivot loop is one fused kernel, so the reference's per-phase host timers
	// (y / p / B_inv / x_b, launch overhead only there, v4:293-357) have no counterpart;
	// "Solve call" carries the whole device time
	print_time("Total", secs(t_start, t_end));
	std::cout << '\n';
	print_time("y", 0.0);
	print_time("p", 0.0);
	print_time("B_inv", r.ms_solve * 1e-3);
	print_time("x_b", 0.0);
	std::cout << '\n';
	print_time("Alloc", 0.0);
	print_time("Init", r.ms_upload * 1e-3);
	print_time("Dealloc", 0.0);
	std::cout << '\n';
	print_time("Host alloc", secs(t_host_alloc, t_read));
	print_time("Read file", secs(t_read, t_solve));
	print_time("Solve call", secs(t_solve, t_print));
	print_time("Print result", secs(t_print, t_free));
	print_time("Host free", secs(t_free, t_end));
	return 0;
}

int main(int argc, char* argv[]) {
	std::ios_base::sync_with_stdio(false);
	if (argc < 2) {
		std::cerr << "Please, specify an input file.\n";
		return 1;
	}
	auto t_start = Clock::now();

	b200lp_options opt;
	b200lp_default_options(&opt);
	bool f64 = false;
	for (int i = 2; i < argc; ++i) {
		if (!std::strcmp(argv[i], "--f64")) f64 = true;
		else if (!std::strcmp(argv[i], "--f32")) f64 = false;
		else if (!std::strcmp(argv[i], "--eps") && i + 1 < argc) opt.eps = std::atof(argv[++i]);
		else if (!std::strcmp(argv[i], "--max-iter") && i + 1 < argc) opt.max_iter = std::atoll(argv[++i]);
		else if (!std::strcmp(argv[i], "--device") && i + 1 < argc) opt.device = std::atoi(argv[++i]);
		else if (!std::strcmp(argv[i], "--dual")) opt.algorithm = 1;
		else if (!std::strcmp(argv[i], "--cost-shift")) opt.cost_shift = 1;
		else if (!std::strcmp(argv[i], "--gpus") && i + 1 < argc) {
			g_devices.clear();
			for (int k = 0, nk = std::atoi(argv[++i]); k < nk; ++k) g_devices.push_back(k);
		}
		else if (!std::strcmp(argv[i], "--devices") && i + 1 < argc) {
			g_devices.clear();
			for (const char* p = argv[++i]; *p;) {
				g_devices.push_back((int32_t)std::strtol(p, const_cast<char**>(&p), 10));
				if (*p == ',') ++p;
				else if (*p) { std::cerr << "Bad device list.\n"; return 1; }
			}
		}
		else {
			std::cerr << "Unknown option " << argv[i] << "\n";
			return 1;
		}
	}

	if (g_devices.size() == 1) opt.device = g_devices[0];
	return f64 ? run<double>(argv[1], opt, t_start) : run<float>(argv[1], opt, t_start);
}
