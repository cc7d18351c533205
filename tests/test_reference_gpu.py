"""The reference's OWN v4 build pins the CPU oracle and the engine.

  v4_stock.out      the reference exactly as shipped (float, EPS 1e-4, MAX_ITER 5)
  libv4ref_f64.so   v4 + the documented minimal patches, real = double
That build (oracle/_ref, made by oracle/make_ref.sh from the reference's source) is not part of the repository.
Where it is absent, the tests compare with stored results in tests/golden/reference.json
(tests/golden/make_reference_golden.py), whose "source" field names what computed them.  As committed, that is the
CPU oracle, which these tests pin to the reference wherever the build is present.  The oracle is held only on LPs
whose pivot sequence cannot depend on summation order.  Printed output is checked against the reference main()'s
print format as its source defines it.
"""
import json
import os
import subprocess
from types import SimpleNamespace

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
TIE = 1e-12
# main()'s timing block as the reference's source prints it (v4:151-157; solver_main.cpp prints the same): groups
# separated by blank lines, each line "<label>: " right-aligned in 19 columns, then seconds with 2 decimals in 6
TIMING_LABELS = [["Total"], ["y", "p", "B_inv", "x_b"], ["Alloc", "Init", "Dealloc"],
                 ["Host alloc", "Read file", "Solve call", "Print result", "Host free"]]


def _stored(*keys, dtype=np.float64):
    """A solver result stored in tests/golden/reference.json."""
    with open(os.path.join(GOLDEN, "reference.json")) as f:
        g = json.load(f)
    for k in keys:
        g = g[k]
    return SimpleNamespace(status=g["status"], iterations=g["iterations"], pivots=g["pivots"], z=g["z"],
                           x_b=np.array(g["x_b"], dtype), b_ixs=np.array(g["b_ixs"], np.int32),
                           trace_p=np.array(g["trace_p"], np.int32), trace_q=np.array(g["trace_q"], np.int32))


def _reference_or_stored(oracle, live, *keys, dtype=np.float64):
    """live() on the reference's own build where present, otherwise the stored result."""
    return live() if oracle.ref_available(dtype) else _stored(*keys, dtype=dtype)


def _timing_block(s):   # same labels, same layout, values differ
    blk = s[s.index("\n\n") + 2:]
    return [(ln.split(":")[0], len(ln)) for ln in blk.splitlines()]


def _reference_timing_block():
    layout = []
    for i, group in enumerate(TIMING_LABELS):
        if i:
            layout.append(("", 0))
        layout += [(f"{label}: ".rjust(19).split(":")[0], 25) for label in group]
    return layout


def _result_block(stdout):
    """main()'s stdout before the timing block -> (iteration lines, status line, [(basis index, value)])."""
    lines = stdout.partition("\n\n")[0].splitlines()
    k = sum(ln.startswith("# Iteration ") for ln in lines)
    xs = [(int(ln.split("x_")[1].split(" = ")[0]), float(ln.split(" = ")[1])) for ln in lines[k + 1:]]
    return k, lines[k], xs


def test_stock_reference_binary_on_sample_matches_cli(oracle, engine_lib):
    """Byte-for-byte stdout parity with the unmodified reference up to the timing values.  Without its build, the
    reference's known stdout on its own fixture and its print format."""
    exe = oracle.ref_stock_binary()
    sample = os.path.join(GOLDEN, "sample.txt")
    head = "# Iteration 1\n# Iteration 2\n# Iteration 3\nOptimum found: 9\n\tx_1 = 3\n\tx_0 = 1\n\n"
    ours = subprocess.run([os.path.join(ROOT, "bin", "solver.out"), sample], capture_output=True, text=True, timeout=300)
    assert ours.returncode == 0, ours.stderr
    assert ours.stdout.startswith(head)
    if exe is None:
        assert _timing_block(ours.stdout) == _reference_timing_block()
        return
    ref = subprocess.run([exe, sample], capture_output=True, text=True, timeout=300)
    assert ref.returncode == 0, ref.stderr
    assert _timing_block(ref.stdout) == _timing_block(ours.stdout)
    if not ref.stdout.startswith(head):
        # The shipped v4 sets CUBLAS_POINTER_MODE_DEVICE and then passes HOST stack scalars
        # (v4:225, 243, 289-290): on a box without pageable-memory access the GEMM never runs,
        # `e` stays uninitialised and v4 reports a bogus optimum in iteration 1.  That is the
        # reference's bug (fixed by patch P5 in make_ref.sh), not a parity failure of the engine.
        assert ref.stdout.startswith("# Iteration 1\n")
        pytest.xfail("stock v4 is broken on this box by its device-pointer-mode bug: " + ref.stdout.split("\n")[1])


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_patched_reference_on_sample(oracle, dtype):
    """The reference's result on its own fixture.  Without its build, the CPU oracle, which stands in for it in the
    stored results, is held to that same result."""
    import simplex_method_gpu_b200 as lp
    A, b, c = lp.read_lp(os.path.join(GOLDEN, "sample.txt"), dtype=dtype)
    solve = oracle.ref_solve if oracle.ref_available(dtype) else oracle.solve
    r = solve(A, b, c, eps=1e-4, max_iter=5)
    assert r.status == oracle.OPTIMUM and r.iterations == 3 and r.z == 9.0
    assert r.trace_p.tolist() == [0, 1] and r.trace_q.tolist() == [1, 0]
    assert r.b_ixs.tolist() == [1, 0] and r.x_b.tolist() == [3.0, 1.0]


@pytest.mark.parametrize("m,n,seed", [(64, 128, 1), (256, 512, 1), (300, 700, 2), (1024, 2048, 1)])
def test_oracle_and_engine_match_reference_f64(oracle, engine_lib, m, n, seed):
    """The oracle is pinned by the reference itself, and the engine walks the same path.  Without the reference build
    both are compared with the stored results, so the oracle half then only guards against a change of the oracle."""
    import simplex_method_gpu_b200 as lp
    A, b, c = oracle.gen_dense(m, n, seed)
    ref = _reference_or_stored(oracle, lambda: oracle.ref_solve(A, b, c, eps=1e-9, max_iter=1 << 20), "dense_f64", f"{m}x{n}_s{seed}")
    cpu = oracle.solve(A, b, c, eps=1e-9, max_iter=1 << 20)
    sol = lp.solve(A, b, c, eps=1e-9, max_iter=1 << 20)
    assert ref.status == oracle.OPTIMUM
    for name, tp, tq, z, xb, bi, it in (("oracle", cpu.trace_p, cpu.trace_q, cpu.z, cpu.x_b, cpu.b_ixs, cpu.iterations),
                                        ("engine", sol.trace[:, 0], sol.trace[:, 1], sol.z, sol.x_b, sol.b_ixs, sol.iterations)):
        k = min(len(tp), len(ref.trace_p))
        same = (tp[:k] == ref.trace_p[:k]) & (tq[:k] == ref.trace_q[:k])
        if not same.all():
            first = int(np.argmin(same))
            gap = min(cpu.gap_p[first], cpu.gap_q[first])
            assert gap <= TIE, f"{name}: diverges from the reference at pivot {first} with runner-up gap {gap:g}"
        else:
            assert len(tp) == len(ref.trace_p) and it == ref.iterations, name
            assert np.array_equal(bi, ref.b_ixs), name
            assert np.abs(xb - ref.x_b).max() <= 1e-9 * max(1.0, np.abs(ref.x_b).max()), name
        assert abs(z - ref.z) <= 1e-9 * abs(ref.z), name


@pytest.mark.parametrize("m,n,seed", [(64, 160, 2), (200, 456, 3)])
def test_engine_matches_reference_f32(oracle, engine_lib, m, n, seed):
    """The reference's stock scalar type (`using real = float`, v4:12).  fp32 sums differ in the last bits between
    cuBLAS and the engine, so near-ties may swap pivots; the optimum must agree to fp32 accuracy and the first
    pivots (large gaps) must be the same."""
    import simplex_method_gpu_b200 as lp
    A, b, c = oracle.gen_dense(m, n, seed, dtype=np.float32)
    ref = _reference_or_stored(oracle, lambda: oracle.ref_solve(A, b, c, eps=1e-4, max_iter=100000),
                               "dense_f32", f"{m}x{n}_s{seed}", dtype=np.float32)
    sol = lp.solve(A, b, c, eps=1e-4, max_iter=100000)
    assert ref.status == oracle.OPTIMUM and sol.status == lp.SolveStatus.OptimumFound
    assert abs(sol.z - ref.z) <= 5e-4 * abs(ref.z)
    k = min(8, len(ref.trace_p), len(sol.trace))
    assert sol.trace[:k, 0].tolist() == ref.trace_p[:k].tolist() and sol.trace[:k, 1].tolist() == ref.trace_q[:k].tolist()


def test_reference_exact_problems(oracle, engine_lib):
    import simplex_method_gpu_b200 as lp
    A, b, c = oracle.gen_klee_minty(10)
    ref = _reference_or_stored(oracle, lambda: oracle.ref_solve(A, b, c, eps=1e-4, max_iter=1 << 20), "klee_minty_10")
    sol = lp.solve(A, b, c, eps=1e-4, max_iter=1 << 20)
    assert ref.status == oracle.OPTIMUM and ref.pivots == 1023 and ref.z == 5.0 ** 10
    assert sol.trace[:, 0].tolist() == ref.trace_p.tolist() and sol.trace[:, 1].tolist() == ref.trace_q.tolist()
    assert np.array_equal(sol.x_b, ref.x_b) and np.array_equal(sol.b_ixs, ref.b_ixs) and sol.z == ref.z
    A, b, c, w = oracle.gen_assignment(16, 1)        # n - m > m: needs the v4:277 length fix
    ref = _reference_or_stored(oracle, lambda: oracle.ref_solve(A, b, c, eps=1e-4, max_iter=1 << 20), "assignment_16")
    sol = lp.solve(A, b, c, eps=1e-4, max_iter=1 << 20)
    assert sol.trace[:, 0].tolist() == ref.trace_p.tolist() and sol.trace[:, 1].tolist() == ref.trace_q.tolist()
    assert sol.z == ref.z and np.array_equal(sol.x_b, ref.x_b)


# ---------------------------------------------------------------- the two big named configurations (BASELINE.json configs 3 and 4)

def _trace_sha(tp, tq):
    import hashlib
    a = np.stack([np.asarray(tp, np.int32), np.asarray(tq, np.int32)], axis=1)
    return hashlib.sha256(np.ascontiguousarray(a).astype("<i4").tobytes()).hexdigest()


def _runner_up_gap(lp, A, b, c, k, which):
    """Gap between the best and the second-best candidate of the pricing (which='p') or of the ratio test ('q') of
    pivot k, from the engine's own state after k pivots (host arithmetic on the downloaded vectors)."""
    m, n = A.shape
    with lp.Engine(m, n, np.float64, eps=1e-9, max_iter=1 << 40) as e:
        e.upload(A, b, c)
        if k:
            e.run(k)
        y = e.vector("y")
        p, _ = e.phase_price()
        if which == "p":
            red = np.concatenate([y @ A[:, :n - m] - c[:n - m], y - c[n - m:]])
            two = np.partition(red, 1)[:2]
            return float(two[1] - two[0])
        e.phase_update_ftran(p)
        e.phase_ratio()
        alpha, x_b = e.vector("alpha"), e.vector("x_b")
        th = np.where(alpha > 0, x_b / np.where(alpha > 0, alpha, 1.0), np.inf)
        two = np.partition(th, 1)[:2]
        return float(two[1] - two[0])


@pytest.mark.parametrize("name,m,n,iters", [("C3", 8192, 16384, 1 << 30), ("C4", 32768, 65536, 1024)])
def test_named_config_pivot_sequence_matches_reference(oracle, engine_lib, name, m, n, iters):
    """north_star: identical entering/leaving sequence with the reference's own CUDA path in fp64 (ties within 1e-12
    excepted), objective and x within 1e-9 relative.  C3 is solved to the optimum (37 395 pivots), C4 over its first
    1024 pivots (the reference needs 43 GB of device memory there; it fits).  The committed CPU-oracle digests
    (tests/golden/trace_digests.json) pin the same windows a third time; they equal the reference's own digests of
    those windows, so the engine is held to them on every run, also where the reference build is absent."""
    import json
    import simplex_method_gpu_b200 as lp
    A, b, c = oracle.gen_dense(m, n, 1)
    sol = lp.solve(A, b, c, eps=1e-9, max_iter=iters)
    tp, tq = sol.trace[:, 0], sol.trace[:, 1]
    with open(os.path.join(GOLDEN, "trace_digests.json")) as f:
        gold = json.load(f)[name]["windows"]
    for P, g in gold.items():
        assert int(P) <= len(tp) and _trace_sha(tp[:int(P)], tq[:int(P)]) == g["trace_sha256"], (name, P)
    if not oracle.ref_available():
        return
    ref = oracle.ref_solve(A, b, c, eps=1e-9, max_iter=iters, always_readback=True)
    k = min(len(tp), len(ref.trace_p))
    same = (tp[:k] == ref.trace_p[:k]) & (tq[:k] == ref.trace_q[:k])
    if not same.all():
        first = int(np.argmin(same))
        which = "p" if tp[first] != ref.trace_p[first] else "q"
        gap = _runner_up_gap(lp, A, b, c, first, which)
        assert gap <= TIE, f"{name}: diverges from the reference at pivot {first} ({which}) with runner-up gap {gap:g}"
        pytest.skip(f"{name}: tie within 1e-12 at pivot {first}; sequences may legitimately differ from there")
    assert len(tp) == len(ref.trace_p) and sol.iterations == ref.iterations and int(sol.status) == ref.status
    assert np.array_equal(sol.b_ixs, ref.b_ixs)
    assert abs(sol.z - ref.z) <= 1e-9 * abs(ref.z)
    assert np.abs(sol.x_b - ref.x_b).max() <= 1e-9 * max(1.0, np.abs(ref.x_b).max())
    for P, g in gold.items():
        assert _trace_sha(ref.trace_p[:int(P)], ref.trace_q[:int(P)]) == g["trace_sha256"], (name, P)
    if name == "C3":
        assert ref.status == oracle.OPTIMUM and sol.pivots == ref.pivots


# ---------------------------------------------------------------- the drop-in, compiled against the reference's own main()

def _split_stdout(s):
    head, _, blk = s.partition("\n\n")
    return head, [(ln.split(":")[0], len(ln)) for ln in blk.splitlines()]


def test_dropin_shim_with_reference_main(oracle, engine_lib, tmp_path):
    """oracle/_ref/v4_shim.out = the reference's unmodified main() (v4:384-474) + integration/v4_b200.inc + libb200lp.so
    (no cuBLAS on the link line).  Same stdout as bin/solver.out and as the reference itself, up to the timing values.
    Without that build, bin/solver.out is held to the reference's known result lines and main()'s print format."""
    import simplex_method_gpu_b200 as lp
    shim = oracle.ref_binary("v4_shim.out")
    cli = os.path.join(ROOT, "bin", "solver.out")

    def main_split(path, head):     # the reference main()'s stdout, split as _split_stdout does
        if shim is None:
            return head, _reference_timing_block()
        a = subprocess.run([shim, path], capture_output=True, text=True, timeout=300)
        assert a.returncode == 0, a.stderr
        return _split_stdout(a.stdout)

    sample = os.path.join(GOLDEN, "sample.txt")
    head = "# Iteration 1\n# Iteration 2\n# Iteration 3\nOptimum found: 9\n\tx_1 = 3\n\tx_0 = 1"
    a = main_split(sample, head)
    b = subprocess.run([cli, sample], capture_output=True, text=True, timeout=300)
    assert b.returncode == 0, b.stderr
    assert a[0] == head and a == _split_stdout(b.stdout)
    # stock constants (float, MAX_ITER = 5) on a 64 x 128 LP: five iteration lines and the MAX_ITER message
    A, bb, c = oracle.gen_dense(64, 128, 3, dtype=np.float32)
    path = str(tmp_path / "lp64.txt")
    lp.write_lp(path, A, bb, c)
    head = "".join(f"# Iteration {i}\n" for i in range(1, 6)) + "MAX_ITER exceeded."
    a = main_split(path, head)
    b = subprocess.run([cli, path], capture_output=True, text=True, timeout=300)
    assert b.returncode == 0 and a == _split_stdout(b.stdout)
    assert a[0] == head
    # error contract of main() is untouched (v4:387-405)
    bad = subprocess.run([shim or cli, str(tmp_path / "missing.txt")], capture_output=True, text=True, timeout=60)
    assert bad.returncode == 1 and "Could not open" in bad.stderr


@pytest.mark.parametrize("sfx,flag", [("f64", "--f64"), ("f32", "--f32")])
def test_dropin_shim_solves_like_the_patched_reference(oracle, engine_lib, tmp_path, sfx, flag):
    """Beyond 5 iterations: the patched reference program (run-time EPS / MAX_ITER, its own cuBLAS solve()) against the
    same main() bound to the engine, and against bin/solver.out: identical result block on a 64 x 128 LP.  Without
    those builds, the numbers bin/solver.out prints are compared with the stored result of the same LP."""
    import simplex_method_gpu_b200 as lp
    shim, ref = oracle.ref_binary(f"v4_shim_env_{sfx}.out"), oracle.ref_binary(f"v4_cli_{sfx}.out")
    dt = np.float64 if sfx == "f64" else np.float32
    eps = "1e-9" if sfx == "f64" else "1e-4"
    A, bb, c = oracle.gen_dense(64, 128, 5, dtype=dt)
    path = str(tmp_path / "lp64.txt")
    lp.write_lp(path, A, bb, c)
    o = subprocess.run([os.path.join(ROOT, "bin", "solver.out"), path, flag, "--eps", eps, "--max-iter", "100000"],
                       capture_output=True, text=True, timeout=300)
    assert o.returncode == 0, o.stderr
    if shim is None or ref is None:
        stored = _stored("dense_" + sfx, "64x128_s5", dtype=dt)
        iters, status, xs = _result_block(o.stdout)
        z = float(status.split("Optimum found: ")[1])
        assert stored.status == oracle.OPTIMUM and status.startswith("Optimum found: ")
        assert _split_stdout(o.stdout)[1] == _reference_timing_block()
        if sfx == "f64":    # printed with 6 significant digits (ostream defaults)
            assert iters == stored.iterations and abs(z - stored.z) <= 1e-5 * abs(stored.z)
            assert [ix for ix, _ in xs] == stored.b_ixs.tolist()
            assert np.allclose([v for _, v in xs], stored.x_b, rtol=1e-5, atol=1e-12)
        else:               # fp32: the live comparison's tolerance (the iteration count may differ)
            assert abs(z - stored.z) <= 5e-4 * abs(stored.z)
        return
    env = dict(os.environ, V4_EPS=eps, V4_MAX_ITER="100000")
    r = subprocess.run([ref, path], capture_output=True, text=True, timeout=300, env=env)
    s = subprocess.run([shim, path], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0 and s.returncode == 0, (r.stderr, s.stderr)
    assert "Optimum found" in r.stdout
    assert _split_stdout(s.stdout) == _split_stdout(o.stdout)
    if sfx == "f64":
        assert _split_stdout(r.stdout) == _split_stdout(s.stdout)
    else:   # fp32 sums differ in the last bits between cuBLAS and the engine: same iteration count is not guaranteed
        zr = float(r.stdout.split("Optimum found: ")[1].split()[0])
        zs = float(s.stdout.split("Optimum found: ")[1].split()[0])
        assert abs(zr - zs) <= 5e-4 * abs(zr)
