"""GPU parity: the CUDA tape through the C-ABI vs (a) the live-reference golden vectors and
(b) the CPU oracle on fresh seeded points.  Structures bit-exact, values rel 1e-10 (fp64)."""
import numpy as np
import pytest

from golden_util import Golden, assert_close, golden_names
from oracle.dnlp_oracle import RefOracles

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu_mod():
    from dnlp_b200.oracles import GpuOracles
    return GpuOracles


@pytest.mark.parametrize("name", golden_names())
def test_gpu_matches_reference_golden(name, gpu_mod):
    g = Golden(name)
    o = gpu_mod(g.problem)
    try:
        jr, jc = o.jacobianstructure()
        hr, hc = o.hessianstructure()
        assert jr.dtype == np.int32 and hr.dtype == np.int32
        np.testing.assert_array_equal(jr, g.jac_rows)
        np.testing.assert_array_equal(jc, g.jac_cols)
        np.testing.assert_array_equal(hr, g.hess_rows)
        np.testing.assert_array_equal(hc, g.hess_cols)
        for i, p in enumerate(g.points):
            assert_close(o.objective(p["x"]), p["f"], "f[%d]" % i)
            assert_close(o.gradient(p["x"]), p["grad"], "grad[%d]" % i)
            assert_close(o.constraints(p["x"]), p["g"], "g[%d]" % i)
            assert_close(o.jacobian(p["x"]), p["jac"], "jac[%d]" % i)
            assert_close(o.hessian(p["x"], p["lam"], float(p["sigma"])), p["hess"], "hess[%d]" % i)
        # interleaved call order with the x-keyed cache active (IPOPT's pattern: same x, five calls)
        for p in reversed(g.points):
            assert_close(o.hessian(p["x"], p["lam"], float(p["sigma"])), p["hess"], "hess/cached")
            assert_close(o.jacobian(p["x"]), p["jac"], "jac/cached")
            assert_close(o.objective(p["x"]), p["f"], "f/cached")
        p = g.points[-1]
        res = o.eval_all(p["x"], p["lam"], float(p["sigma"]))
        for k in ("f", "grad", "g", "jac", "hess"):
            assert_close(res[k], p[k], "eval_all/" + k)
    finally:
        o.close()


@pytest.mark.parametrize("name", ["c3_logistic_small", "c5_microbench_small", "matmul_with_atom_operand",
                                  "clnlbeam", "rel_entr_vector", "hyperbolic_mix"])
def test_gpu_matches_oracle_on_fresh_points(name, gpu_mod):
    g = Golden(name)
    ref = RefOracles(g.problem)
    ref.jacobianstructure(), ref.hessianstructure()
    o = gpu_mod(g.problem)
    rng = np.random.default_rng(1234)
    try:
        x0 = g.points[0]["x"]
        with np.errstate(all="ignore"):
            for _ in range(5):
                x = x0 * (1 + 0.02 * rng.standard_normal(x0.size)) + 0.01 * rng.standard_normal(x0.size)
                lam = rng.standard_normal(g.problem.m)
                sigma = float(rng.uniform(0.1, 2.0))
                assert_close(o.objective(x), ref.objective(x), "f")
                assert_close(o.gradient(x), ref.gradient(x), "grad")
                assert_close(o.constraints(x), ref.constraints(x), "g")
                assert_close(o.jacobian(x), ref.jacobian(x), "jac")
                assert_close(o.hessian(x, lam, sigma), ref.hessian(x, lam, sigma), "hess")
    finally:
        o.close()


@pytest.mark.parametrize("name", ["c2_eigen_qcqp_small", "c3_logistic_small", "c4_qcqp_small",
                                  "c5_microbench_small", "portfolio_socp", "matmul_var_var"])
def test_gpu_optimised_emission_paths(name, gpu_mod, monkeypatch):
    """Large-problem kernels (two-stage reductions, SCALE, one-term POLY, scatter-accumulate) forced on."""
    from dnlp_b200.rules import Builder
    monkeypatch.setattr(Builder, "LAYER_MIN", 2)
    monkeypatch.setattr(Builder, "LONG_ROW", 3)
    monkeypatch.setattr(Builder, "CHUNK", 2)
    g = Golden(name)
    o = gpu_mod(g.problem)
    try:
        for i, p in enumerate(g.points):
            assert_close(o.objective(p["x"]), p["f"], "f[%d]" % i)
            assert_close(o.gradient(p["x"]), p["grad"], "grad[%d]" % i)
            assert_close(o.constraints(p["x"]), p["g"], "g[%d]" % i)
            assert_close(o.jacobian(p["x"]), p["jac"], "jac[%d]" % i)
            assert_close(o.hessian(p["x"], p["lam"], float(p["sigma"])), p["hess"], "hess[%d]" % i)
    finally:
        o.close()


def _cmp_with_oracle(prob, gpu_mod, npoints=2, seed=0):
    ref = RefOracles(prob)
    jr, jc = ref.jacobianstructure()
    hr, hc = ref.hessianstructure()
    o = gpu_mod(prob)
    try:
        np.testing.assert_array_equal(o.jacobianstructure()[0], jr)
        np.testing.assert_array_equal(o.jacobianstructure()[1], jc)
        np.testing.assert_array_equal(o.hessianstructure()[0], hr)
        np.testing.assert_array_equal(o.hessianstructure()[1], hc)
        rng = np.random.default_rng(seed)
        with np.errstate(all="ignore"):
            for _ in range(npoints):
                x = prob.x0 * (1 + 0.01 * rng.standard_normal(prob.n))
                lam = rng.standard_normal(prob.m)
                sigma = float(rng.uniform(0.5, 1.5))
                assert_close(o.objective(x), ref.objective(x), "f")
                assert_close(o.gradient(x), ref.gradient(x), "grad")
                if prob.m:          # the reference's np.concatenate([]) raises without constraints
                    assert_close(o.constraints(x), ref.constraints(x), "g", atol=1e-9)
                assert_close(o.jacobian(x), ref.jacobian(x), "jac")
                assert_close(o.hessian(x, lam, sigma), ref.hessian(x, lam, sigma), "hess")
                res = o.eval_all(x, lam, sigma)
                assert_close(res["hess"], ref.hessian(x, lam, sigma), "eval_all/hess")
                if prob.m:
                    assert_close(res["g"], ref.constraints(x), "eval_all/g", atol=1e-9)
    finally:
        o.close()


@pytest.mark.parametrize("n", [1500, 1501])
def test_gpu_medium_eigen_qcqp(n, gpu_mod):
    """Sizes that reach the production kernels: CTA-per-row GEMV (even n) / warp-per-row GEMV
    (odd n), SCALE + scatter-accumulate Hessian, grid-wide single-row reduction."""
    from dnlp_b200 import workloads as W
    _cmp_with_oracle(W.eigen_qcqp(n), gpu_mod)


def test_gpu_medium_logistic(gpu_mod):
    from dnlp_b200 import workloads as W
    At, x0 = W.logistic_data(30000, 64, 16)
    _cmp_with_oracle(W.logistic_regression(At, x0), gpu_mod)


def test_gpu_medium_microbench(gpu_mod):
    from dnlp_b200 import workloads as W
    A, x0 = W.microbench_data(80000, 40000, 10)
    _cmp_with_oracle(W.microbench(A, x0), gpu_mod)


@pytest.mark.parametrize("name", ["c3_logistic_small", "clnlbeam", "portfolio_socp", "hs071", "c2_eigen_qcqp_small"])
def test_gpu_constant_entry_elision(name, gpu_mod, monkeypatch):
    """Compact D2H of only the x/lambda-dependent entries (affine rows cached, reference quirk Q5)."""
    monkeypatch.setattr(gpu_mod, "ELIDE_MIN", 1)
    monkeypatch.setattr(gpu_mod, "ELIDE_MAX_FRACTION", 1.0)
    g = Golden(name)
    o = gpu_mod(g.problem)
    try:
        assert o._dyn, "elision not active"
        for i, p in enumerate(g.points):
            assert_close(o.gradient(p["x"]), p["grad"], "grad[%d]" % i)
            assert_close(o.constraints(p["x"]), p["g"], "g[%d]" % i)
            assert_close(o.jacobian(p["x"]), p["jac"], "jac[%d]" % i)
            assert_close(o.hessian(p["x"], p["lam"], float(p["sigma"])), p["hess"], "hess[%d]" % i)
    finally:
        o.close()


def test_gpu_unconstrained_and_scalar_edge_cases(gpu_mod):
    """m = 0 (no constraints: empty g / J / lambda), n = 1, and an objective that is constant."""
    from dnlp_b200 import ir
    x = ir.Variable(5)
    p0 = ir.ProblemIR(ir.sum(ir.exp(x)) + ir.sum(ir.power(x, 4)), [], x0=np.linspace(-1, 1, 5))
    _cmp_with_oracle(p0, gpu_mod)
    o = gpu_mod(p0)
    try:
        assert o.constraints(p0.x0).size == 0 and o.jacobian(p0.x0).size == 0
        assert o.jacobianstructure()[0].size == 0
    finally:
        o.close()
    s = ir.Variable(1)
    p1 = ir.ProblemIR(ir.sum(ir.logistic(s)), [ir.sum(ir.power(s, 2)) + (-1.0)], x0=np.array([0.3]))
    _cmp_with_oracle(p1, gpu_mod)
    y = ir.Variable(3)
    p2 = ir.ProblemIR(ir.Constant(0.0), [ir.sum(ir.exp(y)) + (-3.0), y[0] + (-1.0) * y[1]], x0=np.array([0.1, 0.2, 0.3]))
    _cmp_with_oracle(p2, gpu_mod)


def test_gpu_knitro_style_calls(gpu_mod):
    """Knitro's wrappers pass Python lists and may pass sigma = 0 (knitro_nlpif.py:272-289)."""
    g = Golden("hs071")
    ref = RefOracles(g.problem)
    ref.jacobianstructure(), ref.hessianstructure()
    o = gpu_mod(g.problem)
    try:
        p = g.points[1]
        x, lam = list(p["x"]), list(p["lam"])
        assert_close(o.objective(x), ref.objective(np.array(x)), "f")
        assert_close(o.hessian(x, lam, 0.0), ref.hessian(np.array(x), np.array(lam), 0.0), "hess sigma=0")
        # Knitro's lambda_ carries constraint AND variable-bound multipliers (length m + n); the reference
        # only slices the first m (nlp_solver.py:405-411)
        long_lam = lam + [9.0] * len(x)
        assert_close(o.hessian(x, long_lam, 1.0), ref.hessian(np.array(x), np.array(long_lam), 1.0), "hess m+n duals")
        assert o.gradient(x) is o.gradient(x)        # same buffer object every call (nlp_solver.py:184,235)
        o.intermediate(0, 7, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0)
        assert o.iterations == 7
        with pytest.raises(ValueError):
            o.objective(np.zeros(3))
    finally:
        o.close()
    # a closed oracle raises instead of crashing the process (compile-cache eviction, uninstall())
    with pytest.raises(RuntimeError, match="closed"):
        o.objective(p["x"])
    with pytest.raises(RuntimeError, match="closed"):
        o.hessian(p["x"], p["lam"], 1.0)


@pytest.mark.parametrize("name,B", [("c4_qcqp_small", 37), ("c2_eigen_qcqp_small", 64), ("c5_microbench_small", 5),
                                    ("hs071", 33), ("rel_entr_vector", 8), ("matmul_var_var", 3),
                                    ("quad_over_lin_var_denominator", 40)])
def test_gpu_batched_multistart_matches_per_start_oracle(name, B):
    """BatchedOracles (B starts in lock step, DMMA GEMM for dense quad_form) vs the CPU oracle run
    start by start."""
    from dnlp_b200.multistart import BatchedOracles
    g = Golden(name)
    ref = RefOracles(g.problem)
    ref.jacobianstructure(), ref.hessianstructure()
    rng = np.random.default_rng(99)
    x0 = g.points[0]["x"]
    X = x0[None, :] * (1 + 0.05 * rng.standard_normal((B, x0.size)))
    LAM = rng.standard_normal((B, g.problem.m))
    SIG = rng.uniform(0.5, 1.5, B)
    o = BatchedOracles(g.problem, B)
    try:
        res = o.eval(X, LAM, SIG)
        with np.errstate(all="ignore"):
            for b in range(B):
                assert_close(res["f"][b], ref.objective(X[b]), "f[%d]" % b)
                assert_close(res["grad"][b], ref.gradient(X[b]), "grad[%d]" % b)
                assert_close(res["g"][b], ref.constraints(X[b]), "g[%d]" % b)
                assert_close(res["jac"][b], ref.jacobian(X[b]), "jac[%d]" % b)
                assert_close(res["hess"][b], ref.hessian(X[b], LAM[b], float(SIG[b])), "hess[%d]" % b)
        only = o.eval(X, want=("f", "g"))
        assert_close(only["f"], res["f"], "f only")
    finally:
        o.close()


def test_gpu_batched_medium_qcqp_dmma():
    """n = 200 (not a multiple of the 64 x 64 GEMM tile), k = 3, B = 100: exercises tile edges."""
    from dnlp_b200 import workloads as W
    from dnlp_b200.multistart import BatchedOracles
    P, q, rng = W.qcqp_data(200, 3)
    prob = W.qcqp(P, q)
    ref = RefOracles(prob)
    ref.jacobianstructure(), ref.hessianstructure()
    B = 100
    X = rng.uniform(-1, 1, (B, 200))
    LAM = rng.standard_normal((B, 3))
    SIG = np.ones(B)
    o = BatchedOracles(prob, B)
    try:
        res = o.eval(X, LAM, SIG)
        for b in (0, 1, 50, 99):
            assert_close(res["f"][b], ref.objective(X[b]), "f")
            assert_close(res["grad"][b], ref.gradient(X[b]), "grad")
            assert_close(res["g"][b], ref.constraints(X[b]), "g")
            assert_close(res["jac"][b], ref.jacobian(X[b]), "jac")
            assert_close(res["hess"][b], ref.hessian(X[b], LAM[b], 1.0), "hess")
    finally:
        o.close()


def _atom_names():
    from golden_util import atom_golden_names
    return atom_golden_names()


@pytest.mark.parametrize("name", _atom_names())
def test_gpu_atom_rules(name, gpu_mod):
    """Raw per-atom rules (no Dnlp2Smooth) through the CUDA path vs the live-reference goldens."""
    from golden_util import AtomGolden
    g = AtomGolden(name)
    if g.jac_error:
        with pytest.raises(getattr(__import__("builtins"), g.jac_error)):
            gpu_mod(g.problem, with_hessian=False)
        return
    o = gpu_mod(g.problem, with_hessian=not g.hess_error)
    try:
        np.testing.assert_array_equal(o.jacobianstructure()[0], g.jac_rows)
        np.testing.assert_array_equal(o.jacobianstructure()[1], g.jac_cols)
        if not g.hess_error:
            np.testing.assert_array_equal(o.hessianstructure()[0], g.hess_rows)
            np.testing.assert_array_equal(o.hessianstructure()[1], g.hess_cols)
        for p in g.points:
            assert_close(o.objective(p["x"]), p["f"], "f")
            assert_close(o.constraints(p["x"]), p["g"], "g")
            assert_close(o.gradient(p["x"]), p["grad"], "grad")
            assert_close(o.jacobian(p["x"]), p["jac"], "jac")
            if not g.hess_error:
                assert_close(o.hessian(p["x"], p["lam"], float(p["sigma"])), p["hess"], "hess")
    finally:
        o.close()


@pytest.mark.parametrize("graphs", [True, False])
def test_gpu_graph_replay_on_and_off(graphs, gpu_mod):
    """Launch sequences are replayed as CUDA graphs by default; results must not depend on it, and the
    IPOPT call pattern (five callbacks per iterate, many iterates) must hit the replay path."""
    g = Golden("clnlbeam")
    o = gpu_mod(g.problem)
    o.set_graphs(graphs)
    try:
        for rep in range(3):
            for i, p in enumerate(g.points):
                assert_close(o.objective(p["x"]), p["f"], "f")
                assert_close(o.gradient(p["x"]), p["grad"], "grad")
                assert_close(o.constraints(p["x"]), p["g"], "g")
                assert_close(o.jacobian(p["x"]), p["jac"], "jac")
                assert_close(o.hessian(p["x"], p["lam"], float(p["sigma"])), p["hess"], "hess")
        ms = o.run_device(iters=3)
        assert ms > 0
        assert_close(o.read_output("hess"), g.points[-1]["hess"], "hess after run_device")
    finally:
        o.close()


def test_gpu_cabi_error_paths():
    """Errors come back as return codes + dnlp_last_error text, never as crashes."""
    import ctypes as C
    from dnlp_b200 import _cabi
    from dnlp_b200.compiler import compile_problem
    L = _cabi.lib()
    g = Golden("hs071")
    tape = compile_problem(g.problem)
    td, keep = _cabi.make_tape_desc(tape)
    bad = np.array([0, 10 ** 6], dtype=np.int32)            # a program that references a missing instruction
    td.prog[0] = bad.ctypes.data_as(_cabi.c_i32p)
    td.prog_len[0] = 2
    h = C.c_void_p()
    assert L.dnlp_create(C.byref(td), 0, C.byref(h)) != 0
    assert b"unknown instruction" in L.dnlp_last_error(None)
    assert not h.value
    with pytest.raises(RuntimeError):
        _cabi.DeviceTape(tape, device=10 ** 4)                # no such device
    dev = _cabi.DeviceTape(tape)
    pos = np.array([10 ** 6], dtype=np.int32)
    assert L.dnlp_set_dynamic(dev.h, 4, pos.ctypes.data_as(_cabi.c_i32p), 1) != 0
    assert b"out of range" in L.dnlp_last_error(dev.h)
    assert L.dnlp_eval_dyn(dev.h, 0, None, None, 1.0, None) != 0     # program id without a dynamic form
    dev.close()
    from dnlp_b200.multistart import BatchedOracles
    with pytest.raises(RuntimeError):
        BatchedOracles(g.problem, 0)
    o = BatchedOracles(g.problem, 4)
    try:
        with pytest.raises(ValueError):
            o.eval(np.zeros((3, g.problem.n)))
        with pytest.raises(ValueError):
            o.eval(np.zeros((4, g.problem.n)), want=("hess",))
    finally:
        o.close()


@pytest.mark.parametrize("name", ["c1_readme_toy", "c2_eigen_qcqp_small", "c3_logistic_small",
                                  "c5_microbench_small", "c5_lifted_small", "clnlbeam", "nmf_kl_graph_form"])
def test_gpu_parallel_graph_branches_equal_serial(name, gpu_mod):
    """Independent instructions are captured as parallel graph branches (data-dependency edges only).
    Results must be bit-identical to the serial launch order, for single callbacks, for the fused
    five-program sequence of the device loop, and with CUDA graphs switched off."""
    g = Golden(name)
    p = g.points[-1]
    outs = {}
    for mode in ("parallel", "serial", "nographs"):
        o = gpu_mod(g.problem)
        try:
            if mode == "serial":
                o.set_parallel(False)
            if mode == "nographs":
                o.set_graphs(False)
            res = []
            for _ in range(2):      # second round replays the captured graphs
                o.set_cache(False)
                o.set_cache(True)
                r = o.eval_all(p["x"], p["lam"], float(p["sigma"]))
                res.append({k: np.array(np.asarray(r[k]).reshape(-1), copy=True) for k in r})
            o.upload_point(p["x"], p["lam"], float(p["sigma"]))
            o.run_device(iters=3)
            dev = {k: o.read_output(k) for k in ("f", "grad", "g", "jac", "hess")}
            outs[mode] = (res, dev)
        finally:
            o.close()
    for k in ("f", "grad", "g", "jac", "hess"):
        assert_close(outs["parallel"][0][0][k], p[k], "parallel/" + k)
        for mode in ("serial", "nographs"):
            for rnd in range(2):
                np.testing.assert_array_equal(outs["parallel"][0][rnd][k], outs[mode][0][rnd][k], err_msg=mode + "/" + k)
            np.testing.assert_array_equal(outs["parallel"][1][k], outs[mode][1][k], err_msg=mode + "/device/" + k)
        np.testing.assert_array_equal(outs["parallel"][1][k], outs["parallel"][0][0][k], err_msg="device vs host/" + k)


def test_gpu_medium_logistic_window(gpu_mod):
    """C3 shape at a size where the window is chosen by the production rule (>= 2^18 terms)."""
    from dnlp_b200 import workloads as W
    At, x0 = W.logistic_data(40000, 512, 16)
    prob = W.logistic_regression(At, x0)
    _cmp_with_oracle(prob, gpu_mod)
    o = gpu_mod(prob)
    try:
        o.constraints(prob.x0)
        assert any(o.instr_kernel(i).startswith("poly_flat_kernel<0, 0") for i in range(len(o.tape.instrs)))
        plain = np.array(o.constraints(prob.x0), copy=True)
        o.set_windows(True)                 # off by default (slower on B200); same bits when switched on
        o.set_cache(False)
        o.set_cache(True)
        np.testing.assert_array_equal(plain, o.constraints(prob.x0))
        assert any(o.instr_kernel(i).startswith("poly_flat_kernel<0, 1") for i in range(len(o.tape.instrs)))
    finally:
        o.close()


def test_gpu_fused_elementwise_families(gpu_mod):
    """phi / phi' / phi'' of sin, cos, logistic and tanh segments share their transcendental calls in
    the one-launch elementwise sweep of eval_all; per-callback evaluation runs each formula on its
    own.  Both must match the CPU oracle, also at arguments where exp overflows / underflows, and
    integer powers (evaluated as products) must match pow()."""
    from dnlp_b200 import ir
    n = 4100                                     # two tiles + a ragged tail
    rng = np.random.default_rng(5)
    extreme = np.array([0.0, -0.0, 1e-300, -1e-300, 36.0, -36.0, 709.0, -709.0, 720.0, -745.0, 1e4, -1e4, 1e-8])
    def point():
        v = rng.uniform(-3, 3, n)
        v[:extreme.size] = extreme
        return v
    a, b, c, d, e = (ir.Variable(n) for _ in range(5))
    obj = (ir.sum(ir.logistic(a)) + ir.sum(ir.tanh(b)) + ir.sum(ir.sin(c)) + ir.sum(ir.cos(d))
           + ir.sum(ir.power(e, 3)) + ir.sum(ir.power(e, 2)) + ir.sum(ir.power(e, 4)))
    cons = [ir.sum(ir.logistic(a)) + ir.sum(ir.cos(c)) + (-1.0), ir.sum(ir.tanh(b)) + ir.sum(ir.power(e, 2.5)) + (-2.0)]
    x0 = np.concatenate([point(), np.clip(point(), -30, 30), point(), point(), np.abs(point()) + 0.1])
    prob = ir.ProblemIR(obj, cons, x0=x0)
    ref = RefOracles(prob)
    ref.jacobianstructure(), ref.hessianstructure()
    o = gpu_mod(prob)
    try:
        lam = np.array([0.7, -1.3])
        with np.errstate(all="ignore"):
            want = {"f": ref.objective(x0), "grad": ref.gradient(x0).copy(), "g": ref.constraints(x0),
                    "jac": np.asarray(ref.jacobian(x0)).ravel(), "hess": np.asarray(ref.hessian(x0, lam, 0.9)).ravel()}
        fused = o.eval_all(x0, lam, 0.9)
        for k in want:
            assert_close(fused[k], want[k], "fused/" + k)
        o.set_cache(False)
        o.set_cache(True)
        assert_close(o.gradient(x0), want["grad"], "separate/grad")
        assert_close(o.jacobian(x0), want["jac"], "separate/jac")
        assert_close(o.hessian(x0, lam, 0.9), want["hess"], "separate/hess")
        assert_close(o.objective(x0), want["f"], "separate/f")
    finally:
        o.close()


@pytest.mark.parametrize("name", ["c3_logistic_small", "c5_microbench_small", "c5_lifted_small", "portfolio_socp",
                                  "matmul_const_sides", "nmf_kl_graph_form", "clnlbeam", "c4_qcqp_small"])
@pytest.mark.parametrize("layered", [False, True])
def test_gpu_flat_term_streaming_kernel(name, layered, gpu_mod, monkeypatch):
    """poly_flat_kernel (chunked term streaming + in-CTA segmented row sums) forced on for every
    multi-term instruction, with and without the shared-memory window, plain and through the
    scatter-accumulate second layer of large outputs."""
    monkeypatch.setenv("DNLP_FLAT_MIN_TERMS", "1")
    monkeypatch.setenv("DNLP_WIN_MIN_TERMS", "1")
    if layered:
        from dnlp_b200.rules import Builder
        monkeypatch.setattr(Builder, "LAYER_MIN", 2)
    g = Golden(name)
    o = gpu_mod(g.problem)
    o.set_windows(True)                   # first round with the window, second without
    try:
        for rnd in range(2):
            for i, p in enumerate(g.points):
                assert_close(o.objective(p["x"]), p["f"], "f[%d]" % i)
                assert_close(o.gradient(p["x"]), p["grad"], "grad[%d]" % i)
                assert_close(o.constraints(p["x"]), p["g"], "g[%d]" % i)
                assert_close(o.jacobian(p["x"]), p["jac"], "jac[%d]" % i)
                assert_close(o.hessian(p["x"], p["lam"], float(p["sigma"])), p["hess"], "hess[%d]" % i)
            used = [o.instr_kernel(i) for i in range(len(o.tape.instrs))]
            o.set_windows(False)          # second round: the variant without the window
    finally:
        o.close()
    if name.startswith("c"):
        assert any(u.startswith("poly_flat_kernel") for u in used), used


def test_gpu_flat_kernel_long_short_and_empty_rows(gpu_mod, monkeypatch):
    """Rows that fill almost a whole 256-term chunk mixed with many short ragged rows and empty rows,
    odd chunk starts (windows are aligned down to an even term), a partial last window; rows longer
    than a chunk make the instruction fall back to the row kernel."""
    from dnlp_b200 import ir
    import scipy.sparse as sp
    monkeypatch.setenv("DNLP_FLAT_MIN_TERMS", "1")
    rng = np.random.default_rng(11)
    for n, expect_flat in ((240, True), (300, False)):
        x = ir.Variable(n)
        A = rng.standard_normal((6, n))
        A[1, 100:] = 0.0                                   # one short dense row between the long ones
        B = rng.standard_normal((300, n)) * (rng.random((300, n)) < 0.02)
        cons = [ir.matmul(ir.Constant(A), x) + ir.Constant(-np.ones(6)),
                ir.matmul(ir.Constant(sp.csr_matrix(B)), ir.exp(x)) + ir.Constant(-np.ones(300))]
        prob = ir.ProblemIR(ir.sum(ir.power(x, 2)), cons, x0=rng.uniform(-1, 1, n))
        _cmp_with_oracle(prob, gpu_mod, npoints=2)
        o = gpu_mod(prob)
        try:
            a = np.array(o.constraints(prob.x0), copy=True)
            o.hessian(prob.x0, np.ones(306), 1.0)
            g_instr = [i.id for i in o.tape.instrs if i.dst_space == 3]
            assert all(o.instr_kernel(i).startswith("poly_flat_kernel") == expect_flat for i in g_instr), \
                [o.instr_kernel(i) for i in g_instr]
            for _ in range(3):                             # identical bits on every run
                o.set_cache(False)
                o.set_cache(True)
                np.testing.assert_array_equal(a, o.constraints(prob.x0))
        finally:
            o.close()


@pytest.mark.parametrize("name", ["c3_logistic_small", "c5_microbench_small", "c5_lifted_small", "hyperbolic_mix"])
def test_gpu_short_and_long_elementwise_batches(name, gpu_mod, monkeypatch):
    """The one-launch elementwise sweep is split into a short-segment and a long-segment batch so that
    consumers of a short segment do not wait for multi-million-element sweeps; here the split point
    is lowered so that small problems produce both batches."""
    monkeypatch.setenv("DNLP_BATCH_SPLIT", "100")
    g = Golden(name)
    o = gpu_mod(g.problem)
    try:
        for p in g.points:
            res = o.eval_all(p["x"], p["lam"], float(p["sigma"]))
            for k in ("f", "grad", "g", "jac", "hess"):
                assert_close(res[k], p[k], "eval_all/" + k)
            o.upload_point(p["x"], p["lam"], float(p["sigma"]))
            o.run_device(iters=2)
            for k in ("f", "grad", "g", "jac", "hess"):
                assert_close(o.read_output(k), p[k], "device/" + k)
    finally:
        o.close()


@pytest.mark.parametrize("name", ["c2_eigen_qcqp_small", "c4_qcqp_small", "portfolio_quadform", "hs071",
                                  "c3_logistic_small", "qcp_three_scalars"])
@pytest.mark.parametrize("layered", [False, True])
def test_gpu_sigma_only_hessian_entries_are_kept_between_calls(name, layered, gpu_mod, monkeypatch):
    """Hessian entries of the form c * sigma (dense quad_form objective) are fetched only when the
    objective factor changes; the instructions that produce them stay cached on the device until
    then.  Any interleaving of new x, new lambda and new sigma must still match the CPU oracle."""
    monkeypatch.setattr(gpu_mod, "ELIDE_MIN", 1)
    monkeypatch.setattr(gpu_mod, "ELIDE_MAX_FRACTION", 1.0)
    if layered:
        from dnlp_b200.rules import Builder
        monkeypatch.setattr(Builder, "LAYER_MIN", 2)
    g = Golden(name)
    ref = RefOracles(g.problem)
    ref.jacobianstructure(), ref.hessianstructure()
    o = gpu_mod(g.problem)
    rng = np.random.default_rng(3)
    try:
        x0, m = g.points[0]["x"], g.problem.m
        xs = [x0 * (1 + 0.03 * rng.standard_normal(x0.size)) for _ in range(3)]
        lams = [rng.standard_normal(m) for _ in range(3)]
        seq = [(0, 0, 1.0), (1, 1, 1.0), (1, 2, 1.0), (2, 2, 1.0), (2, 2, 0.5), (0, 1, 0.5), (0, 1, 0.0), (1, 0, 1.0),
               (1, 0, 1.0), (2, 1, 1.0)]
        with np.errstate(all="ignore"):
            for step, (xi, li, sg) in enumerate(seq):
                if step % 3 == 1:
                    assert_close(o.jacobian(xs[xi]), ref.jacobian(xs[xi]), "jac@%d" % step)
                got = o.hessian(xs[xi], lams[li], sg)
                assert_close(got, ref.hessian(xs[xi], lams[li], sg), "hess@%d" % step)
                assert got is o._hess
        if name in ("c2_eigen_qcqp_small", "portfolio_quadform"):
            assert o._hess_sigma_class and o._dyn["hess"][0].size < o.nnz_hess
        if name == "c2_eigen_qcqp_small" and layered:
            # the 2*sigma*Q layer is not re-launched while sigma stays the same: a new lambda costs the
            # diagonal update and the compaction kernel only
            o.hessian(xs[0], lams[0], 0.75)
            k0 = o.kernel_launches()
            o.hessian(xs[0], lams[1], 0.75)
            k1 = o.kernel_launches()
            o.hessian(xs[0], lams[1], 0.25)
            k2 = o.kernel_launches()
            assert k1 - k0 == 2 and k2 - k1 >= 2, (k0, k1, k2)
    finally:
        o.close()


@pytest.mark.parametrize("flat", [True, False])
def test_gpu_fused_spmv_jacobian(flat, gpu_mod, monkeypatch):
    """SPMVJ: g = A phi(x) and J = A o phi'(x) in one pass over A with 16-byte pair gathers (the union
    program), against the CPU oracle; per-callback programs (plain SpMV / Jacobian fill on the strided pair
    slots) too.  Both the chunked warp kernel and the row fallback."""
    from dnlp_b200 import tape as T
    from dnlp_b200 import workloads as W
    from dnlp_b200.rules import Builder
    monkeypatch.setattr(Builder, "PAIRING", True)        # off by default (measured slower at the C5 size)
    monkeypatch.setattr(Builder, "PAIR_MIN_NNZ", 1)
    monkeypatch.setenv("DNLP_FLAT_MIN_TERMS", "1" if flat else str(1 << 40))
    monkeypatch.setenv("DNLP_BATCH_SPLIT", "3000")
    A, x0 = W.microbench_data(40000, 15313, 7, seed=3)
    prob = W.microbench(A, x0)
    ref = RefOracles(prob)
    ref.jacobianstructure(), ref.hessianstructure()
    o = gpu_mod(prob)
    try:
        fused = [i for i in o.tape.instrs if i.kind == T.K_SPMVJ]
        assert len(fused) == 1
        rng = np.random.default_rng(2)
        for it in range(2):
            x = prob.x0 * (1 + 0.01 * rng.standard_normal(prob.n))
            lam = rng.standard_normal(prob.m)
            res = o.eval_all(x, lam, 0.8)                       # union program: the fused instruction
            assert_close(res["f"], ref.objective(x), "f")
            assert_close(res["grad"], ref.gradient(x), "grad")
            assert_close(res["g"], ref.constraints(x), "g", atol=1e-11)
            assert_close(res["jac"], ref.jacobian(x), "jac")
            assert_close(res["hess"], ref.hessian(x, lam, 0.8), "hess")
            assert_close(o.constraints(x), ref.constraints(x), "g alone", atol=1e-11)
            assert_close(o.jacobian(x), ref.jacobian(x), "jac alone")
        assert o.instr_kernel(fused[0].id) == ("spmvj_flat_kernel<0>" if flat else "spmvj_rows_kernel") or \
            o.instr_kernel(fused[0].id).startswith("spmvj_flat_kernel")
        o.upload_point(x, lam, 0.8)
        assert o.run_device(iters=2) > 0
        assert_close(o.read_output("jac"), ref.jacobian(x), "jac after device loop")
        assert_close(o.read_output("g"), ref.constraints(x), "g after device loop", atol=1e-11)
    finally:
        o.close()


@pytest.mark.parametrize("name", ["c3_logistic_small", "hs071", "c5_microbench_small", "c2_eigen_qcqp_small"])
def test_gpu_eager_delivery_random_callback_orders(name, gpu_mod, monkeypatch):
    """Eager delivery (dnlp_bind_outputs): at a new x every x-only output is computed and copied on a second
    stream.  Any interleaving of callbacks and points - IPOPT's order, line-search points that ask for f and g
    only, repeated calls, x changing while copies are in flight - must return exactly what the one-program
    path returns."""
    g = Golden(name)
    ref = RefOracles(g.problem)
    ref.jacobianstructure(), ref.hessianstructure()
    monkeypatch.setattr(gpu_mod, "ELIDE_MIN", 8)           # compact (dynamic-entry) delivery on these small problems too
    o = gpu_mod(g.problem, eager=True)
    plain = gpu_mod(g.problem, eager=False)
    try:
        assert o.eager and not plain.eager
        rng = np.random.default_rng(5)
        pts = [p["x"] * (1 + 0.01 * rng.standard_normal(p["x"].size)) for p in g.points for _ in range(2)]
        lam0 = g.points[0]["lam"]
        calls = ["f", "grad", "g", "jac", "hess"]
        for step in range(60):
            x = pts[rng.integers(len(pts))] if step % 3 else pts[step % len(pts)].copy()
            for c in rng.permutation(calls)[:rng.integers(1, 6)]:
                lam = lam0 * rng.uniform(0.5, 1.5)
                if c == "f":
                    assert_close(o.objective(x), ref.objective(x), "f")
                elif c == "grad":
                    assert_close(o.gradient(x), ref.gradient(x), "grad")
                elif c == "g":
                    assert_close(o.constraints(x), ref.constraints(x), "g", atol=1e-11)
                elif c == "jac":
                    assert_close(o.jacobian(x), ref.jacobian(x), "jac")
                else:
                    assert_close(o.hessian(x, lam, 0.9), ref.hessian(x, lam, 0.9), "hess")
                    assert_close(plain.hessian(x, lam, 0.9), ref.hessian(x, lam, 0.9), "hess/plain")
        # IPOPT's order at one iterate costs ONE launch sequence for the four x-only outputs
        x = pts[0] * 1.001
        l0 = o.kernel_launches()
        o.objective(x)
        l1 = o.kernel_launches()
        o.gradient(x), o.constraints(x), o.jacobian(x)
        assert o.kernel_launches() == l1 > l0
    finally:
        o.close(), plain.close()


@pytest.mark.parametrize("eager", [False, True])
def test_gpu_parameter_sweep_without_recompiling(eager, gpu_mod):
    """Parameter slots (SURVEY 8f item 3; expressions/constants/parameter.py:35): a sweep over parameter
    values on ONE compiled oracle - every output must equal the CPU oracle of the problem with the
    parameters folded at their current values, and only parameter-dependent work is repeated."""
    from dnlp_b200 import ir
    rng = np.random.default_rng(3)
    n = 300
    A = rng.standard_normal((40, n))
    x, t = ir.Variable(n), ir.Variable(40)
    gamma, b, w = ir.Parameter((), 0.5), ir.Parameter(n, rng.standard_normal(n)), ir.Parameter(40, rng.uniform(0.5, 2, 40))
    # smooth form (atoms on bare variables): parameters as a scalar weight, an elementwise weight, a linear
    # coefficient vector and right-hand sides
    obj = ir.sum(ir.exp(x)) + ir.multiply(gamma, ir.sum(ir.power(x, 2))) + ir.sum(ir.multiply(b, x))
    cons = [ir.multiply(w, ir.logistic(t)) + ir.neg(ir.promote(gamma, (40,))),
            t + ir.neg(ir.matmul(A, x)),
            ir.sum(ir.multiply(b, ir.power(x, 3))) + ir.neg(gamma)]
    prob = ir.ProblemIR(obj, cons, [x, t], x0=0.1 * rng.standard_normal(n + 40))
    assert prob.n_params == 1 + n + 40
    o = gpu_mod(prob, eager=eager)           # eager delivery must re-deliver the x-only outputs after new parameters
    try:
        assert o.tape.n_params == prob.n_params and o.eager == eager
        xv = prob.x0 * 1.1
        lam = rng.standard_normal(prob.m)
        for trial in range(4):
            if trial:
                gamma.attrs["value"] = np.asarray(rng.uniform(0.1, 3.0))
                b.attrs["value"] = rng.standard_normal(n)
                w.attrs["value"] = rng.uniform(0.5, 2, 40)
                o.set_parameters(prob.param_values())
            ref = RefOracles(prob.folded())
            np.testing.assert_array_equal(o.jacobianstructure()[0], ref.jacobianstructure()[0])
            np.testing.assert_array_equal(o.hessianstructure()[1], ref.hessianstructure()[1])
            assert_close(o.objective(xv), ref.objective(xv), "f")
            assert_close(o.gradient(xv), ref.gradient(xv), "grad")
            assert_close(o.constraints(xv), ref.constraints(xv), "g")
            assert_close(o.jacobian(xv), ref.jacobian(xv), "jac")
            assert_close(o.hessian(xv, lam, 0.6), ref.hessian(xv, lam, 0.6), "hess")
            res = o.eval_all(xv, lam, 0.6)
            assert_close(res["jac"], ref.jacobian(xv), "eval_all/jac")
        # same x, same parameters: nothing x- or parameter-dependent is launched again
        o.objective(xv)
        l0 = o.kernel_launches()
        o.objective(xv)
        assert o.kernel_launches() - l0 <= 1
        with pytest.raises(ValueError):
            o.set_parameters(np.zeros(3))
    finally:
        o.close()


@pytest.mark.parametrize("workload,scale", [("c3", 0.002), ("c4", 0.05)])
def test_gpu_bench_dump_outputs_are_the_last_device_step(workload, scale, tmp_path, monkeypatch):
    """bench.py --dump-outputs on the device: what the timed device steps left in HBM, read back after the timed
    window, equals the CPU oracle at the bench's seeded inputs (single oracle and batched multi-start path)."""
    import argparse
    import os

    import bench
    from workload_cases import bench_dump_expected
    monkeypatch.setattr(bench, "DUMP_MAX_ENTRIES", 4096)
    monkeypatch.setenv("DNLP_C4_BATCH", "5")
    args = argparse.Namespace(gpus=1, steps=2, warmup=3, workload=workload, scale=scale, impl="ours", no_cpu_baseline=True,
                              device_only=True, dump_outputs=str(tmp_path))
    run = bench.bench_multistart if workload == "c4" else (lambda a, *r: bench.bench_single(workload, a, *r))
    run(args, bench.Group(0, 1, 0), 6545.0, "test")
    want = bench_dump_expected(workload, scale, 4096)
    assert sorted(os.listdir(tmp_path)) == sorted("%s_%s.npy" % (workload, p) for p in bench.PROGS)
    for p in bench.PROGS:
        got = np.load(tmp_path / ("%s_%s.npy" % (workload, p)))
        assert got.dtype == np.float64
        assert_close(got, want[p], p, atol=1e-9 if p == "g" else 1e-12)
