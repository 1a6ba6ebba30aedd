"""``prob.solve(nlp=True, solver=cp.IPOPT)`` END TO END through the unmodified reference: reduction chain, ``Oracles``
(or, after ``install()``, ``GpuOracles``), ``IPOPT.solve_via_data`` (ipopt_nlpif.py:143-173), ``invert`` and
``unpack_results`` - with the cyipopt PROTOCOL stand-in of tests/cyipopt_standin.py where cyipopt itself would be
(not installed anywhere; the stand-in is not IPOPT, see its header).  What this pins is the drop-in boundary of SURVEY
8(b) as the reference's own solver interface exercises it: fresh x arrays per callback, ``np.array(ret).flatten()`` on
every return value, ``intermediate`` / ``iterations``, options, the info dict, dual recovery - and that swapping the
oracle changes nothing the user sees: same status, same iteration count, optimum within 1e-8.

CPU tier: GpuOracles on the interpreter-backed stand-in device.  GPU tier (the real device):
tests/test_zz_gpu_prob_solve.py.
The whole reference test-suite goes through the same path in tools/run_reference_nlp_suite.sh (build container only);
its last run is tests/golden/refsuite_prob_solve.*.log."""
import sys
import types

import numpy as np
import pytest

import cyipopt_standin

README_OPTIMUM = 11.950810853979528          # lambda_max(A), reference README.md:34-54


def _cvxpy():
    if "cvxpy" in sys.modules:
        return sys.modules["cvxpy"]
    from oracle import ref_driver as R
    if not R.available():
        pytest.skip("no reference to drive: oracle/_ref is missing")
    return R.load_reference()


@pytest.fixture
def cp():
    mod = _cvxpy()
    cyipopt_standin.install()
    yield mod
    cyipopt_standin.uninstall()


def readme_toy(cp):
    np.random.seed(0)
    n = 3
    A = np.random.randn(n, n)
    A = A.T @ A
    x = cp.Variable(n)
    x.value = np.ones(n)
    con = cp.sum_squares(x) == 1
    return cp.Problem(cp.Maximize(cp.quad_form(x, A)), [con]), x, con


def hs071(cp):
    x = cp.Variable(4, bounds=[1, 5])
    x.value = np.array([1.0, 5.0, 5.0, 1.0])
    cons = [x[0] * x[1] * x[2] * x[3] >= 25, cp.sum(cp.square(x)) == 40]
    return cp.Problem(cp.Minimize(x[0] * x[3] * (x[0] + x[1] + x[2]) + x[2]), cons), x, cons[1]


def entropy_simplex(cp):
    rng = np.random.default_rng(3)
    n = 12
    q = rng.uniform(0.1, 1.0, n)
    x = cp.Variable(n, nonneg=True)
    x.value = np.full(n, 1.0 / n)
    con = cp.sum(x) == 1
    return cp.Problem(cp.Maximize(cp.sum(cp.entr(x)) - q @ x), [con, x[0] + x[1] <= 0.1]), x, con


def _solve(cp, build, **kw):
    prob, x, con = build(cp)
    spied = []
    ctor = cyipopt_standin.Problem.__init__

    def spy(p, *a, **k):
        ctor(p, *a, **k)
        spied.append(p)
    cyipopt_standin.Problem.__init__ = spy
    try:
        prob.solve(nlp=True, solver=cp.IPOPT, **kw)
    finally:
        cyipopt_standin.Problem.__init__ = ctor
    return types.SimpleNamespace(status=prob.status, value=prob.value, iters=prob.solver_stats.num_iters,
                                 x=np.array(x.value, dtype=float), dual=con.dual_value, nlps=spied, prob=prob)


def _both_arms(cp, build, monkeypatch, standin_device, **kw):
    import dnlp_b200.nlp_solver as gpu
    from dnlp_b200.oracles import GpuOracles
    ref = _solve(cp, build, **kw)
    assert type(ref.nlps[0].obj).__name__ == "Oracles"
    if standin_device:
        import host_logic_device
        host_logic_device.install(monkeypatch)
    with gpu.gpu_oracle():
        ours = _solve(cp, build, **kw)
    assert isinstance(ours.nlps[0].obj, GpuOracles)
    assert ours.status == ref.status == "optimal"
    assert ours.iters == ref.iters and ours.iters > 0
    assert ours.nlps[0].calls == ref.nlps[0].calls                      # the same callbacks, the same number of times
    assert abs(ours.value - ref.value) <= 1e-8 * max(1.0, abs(ref.value))
    np.testing.assert_allclose(ours.x, ref.x, rtol=0, atol=1e-7)
    return ref, ours


CASES = {"readme_toy": readme_toy, "hs071": hs071, "entropy_simplex": entropy_simplex}


@pytest.mark.parametrize("name", sorted(CASES))
def test_prob_solve_is_unchanged_by_the_oracle_swap(name, cp, monkeypatch):
    ref, ours = _both_arms(cp, CASES[name], monkeypatch, standin_device=True)
    if name == "readme_toy":
        assert abs(ours.value - README_OPTIMUM) < 1e-7 and abs(ref.value - README_OPTIMUM) < 1e-7
        # dual recovery (install() default): the multiplier of x'x == 1 at the top eigenpair is lambda_max
        assert ref.dual is None and abs(abs(float(ours.dual)) - README_OPTIMUM) < 1e-5
    if name == "hs071":
        assert abs(ours.value - 17.0140173) < 1e-6


def test_solver_options_and_quasi_newton_reach_the_oracle(cp, monkeypatch):
    """``hessian_approximation='limited-memory'`` (a user option the reference forwards, ipopt_nlpif.py:152-166): the
    solver then never asks for the Hessian; ``max_iter`` stops the solve and the status maps to user_limit."""
    ref, ours = _both_arms(cp, hs071, monkeypatch, standin_device=True, hessian_approximation="limited-memory")
    assert ours.nlps[0].calls["hessian"] == 0 and ours.nlps[0].options["hessian_approximation"] == "limited-memory"
    import dnlp_b200.nlp_solver as gpu
    with gpu.gpu_oracle():
        short = _solve(cp, hs071, max_iter=2)
    assert short.status == "user_limit" and short.iters == 2


def test_best_of_loop_of_the_reference_compiles_once(cp, monkeypatch):
    """``best_of=N`` (problem.py:1249-1275): the reference re-applies the chain and solves per start; with install()
    the N starts share one compiled oracle and the objective set is the reference's."""
    import host_logic_device

    import dnlp_b200.nlp_solver as gpu
    from dnlp_b200 import compiler

    def build(cp):
        rng = np.random.default_rng(5)
        A = rng.standard_normal((4, 4))
        A = A + A.T
        x = cp.Variable(4, bounds=[-2, 2])
        con = cp.sum_squares(x) == 1
        return cp.Problem(cp.Minimize(cp.quad_form(x, A, assume_PSD=True)), [con]), x, con
    np.random.seed(11)
    ref = _solve(cp, build, best_of=4)
    host_logic_device.install(monkeypatch)
    compiles = []
    orig = compiler.compile_problem
    monkeypatch.setattr("dnlp_b200.oracles.compile_problem",
                        lambda *a, **k: (compiles.append(1), orig(*a, **k))[1], raising=False)
    np.random.seed(11)
    with gpu.gpu_oracle():
        ours = _solve(cp, build, best_of=4)
    a = ref.prob.solver_stats.extra_stats["all_objs_from_best_of"]
    b = ours.prob.solver_stats.extra_stats["all_objs_from_best_of"]
    np.testing.assert_allclose(b, a, rtol=1e-8, atol=1e-10)
    assert len(ours.nlps) == 4 and len({id(p.obj) for p in ours.nlps}) == 1      # one resident oracle, re-armed
    assert len(compiles) <= 1


def test_solve_best_of_with_per_start_solver_instances(cp, monkeypatch):
    """``dnlp_b200.best_of.solve_best_of(..., solver="ipopt")``: one chain application per start for the reference's
    own sampler, ONE compiled oracle, per-start ``solve_via_data``; same objective set and winner as the reference's
    loop (problem.py:1249-1275), Maximize and a constant objective term included."""
    import host_logic_device

    import dnlp_b200.nlp_solver as gpu
    from dnlp_b200.best_of import solve_best_of

    def build():
        rng = np.random.default_rng(8)
        A = rng.standard_normal((5, 5))
        A = A + A.T
        x = cp.Variable(5, bounds=[-3, 3])
        return cp.Problem(cp.Maximize(3.5 - cp.quad_form(x, A, assume_PSD=True) + cp.sum(x)),
                          [cp.sum_squares(x) == 2, x[0] + x[1] <= 1]), x
    np.random.seed(21)
    pr, xr = build()
    pr.solve(nlp=True, solver=cp.IPOPT, best_of=5)
    want = pr.solver_stats.extra_stats["all_objs_from_best_of"]
    host_logic_device.install(monkeypatch)
    np.random.seed(21)
    po, xo = build()
    with gpu.gpu_oracle():
        value = solve_best_of(po, 5, solver="ipopt")
    got = po.solver_stats.extra_stats["all_objs_from_best_of"]
    np.testing.assert_allclose(got, want, rtol=1e-8, atol=1e-9)
    assert abs(value - pr.value) <= 1e-8 * max(1.0, abs(pr.value))
    np.testing.assert_allclose(xo.value, xr.value, atol=1e-7)


def test_parameter_sweep_solves_without_recompiling(cp, monkeypatch):
    """A user's parameter sweep: the same Problem solved at three Parameter values.  The reference re-reads
    ``Parameter.value`` inside its rules on every callback (expressions/constants/parameter.py:35); with install()
    the values are slots of the resident tape: ONE compile, the same optimum / iteration count per setting."""
    import host_logic_device

    import dnlp_b200.nlp_solver as gpu
    from dnlp_b200 import oracles as oracles_mod

    def build():
        rng = np.random.default_rng(2)
        A = rng.standard_normal((8, 5))
        b = cp.Parameter(8)
        w = cp.Parameter(5, nonneg=True)        # (a 0-d Parameter crashes the reference's own multiply._hess_vec)
        x = cp.Variable(5, bounds=[-4, 4])
        x.value = np.zeros(5)
        prob = cp.Problem(cp.Minimize(cp.sum(cp.logistic(A @ x - b)) + cp.sum(cp.multiply(w, cp.square(x)))), [cp.sum(x) == 1])
        return prob, x, b, w
    settings = [(np.linspace(-1, 1, 8), 0.5), (np.linspace(1, -2, 8), 0.1), (np.full(8, 0.3), 2.0)]

    def sweep(prob, x, b, w):
        out = []
        for bv, wv in settings:
            b.value, w.value = bv, np.full(5, wv)
            x.value = np.zeros(5)
            prob.solve(nlp=True, solver=cp.IPOPT)
            out.append((prob.status, prob.value, prob.solver_stats.num_iters, np.array(x.value)))
        return out
    want = sweep(*build())
    host_logic_device.install(monkeypatch)
    compiles = []
    orig = oracles_mod.compile_problem
    monkeypatch.setattr(oracles_mod, "compile_problem", lambda *a, **k: (compiles.append(1), orig(*a, **k))[1])
    with gpu.gpu_oracle():
        got = sweep(*build())
    assert len(compiles) == 1
    for (s1, v1, i1, x1), (s2, v2, i2, x2) in zip(want, got):
        assert s1 == s2 == "optimal" and i1 == i2
        assert abs(v1 - v2) <= 1e-8 * max(1.0, abs(v1))
        np.testing.assert_allclose(x2, x1, atol=1e-7)
    assert len({round(v, 6) for _, v, _, _ in got}) == 3           # the three settings really differ


def test_install_and_uninstall_leave_the_reference_as_they_found_it(cp):
    """install() rebinds ``Oracles`` and wraps ``solve_via_data`` (write-back of the last evaluated point) / ``invert``
    / ``_prepare_data_and_inv_data`` (dual recovery); uninstall() must restore every one of them."""
    import importlib

    import dnlp_b200.nlp_solver as gpu
    mod = importlib.import_module("cvxpy.reductions.solvers.nlp_solvers.nlp_solver")
    ipopt = importlib.import_module("cvxpy.reductions.solvers.nlp_solvers.ipopt_nlpif").IPOPT
    knitro = importlib.import_module("cvxpy.reductions.solvers.nlp_solvers.knitro_nlpif").KNITRO
    before = (mod.Oracles, mod.NLPsolver._prepare_data_and_inv_data, ipopt.solve_via_data, ipopt.invert,
              knitro.solve_via_data)
    with gpu.gpu_oracle():
        assert mod.Oracles is gpu.gpu_oracles
        assert ipopt.solve_via_data is not before[2] and knitro.solve_via_data is not before[4]
        with gpu.gpu_oracle():                    # nested / repeated install keeps ONE layer of wrapping
            pass
    after = (mod.Oracles, mod.NLPsolver._prepare_data_and_inv_data, ipopt.solve_via_data, ipopt.invert,
             knitro.solve_via_data)
    assert after == before


def test_misaligned_bounds_of_the_reference_fail_the_same_way(cp, monkeypatch):
    """Reference quirk Q8 (DESIGN.md section 2; found by tests/golden/fuzz_live_solve.py): ``Bounds`` lays out lb / ub /
    x0 in the variable order of the problem BEFORE ``lower_ineq_to_nonneg`` rewrites ``a <= b`` as ``b - a >= 0``,
    ``Oracles`` reads x in the order after.  Here that puts the bounded ``v1`` on an auxiliary variable's slots; the
    reference's validating setter then raises ValueError in the first callback.  install() validates the initial
    point once with the reference's own validator: the same exception type and message."""
    import host_logic_device

    import dnlp_b200.nlp_solver as gpu

    def build():
        v1 = cp.Variable((3, 3), name="v1", bounds=[0.1, 2.0])
        v2 = cp.Variable(name="v2")
        v2.value = 0.5
        return cp.Problem(cp.Minimize(cp.atanh(0.9 * v2 + 0.08)),
                          [0.11 <= cp.minimum(v1, 0.7), 0.12 <= cp.asinh(1.18 * v2 + 0.1), 0.05 <= v1])
    with pytest.raises(ValueError, match="Variable value must be in bounds") as ref:
        build().solve(nlp=True, solver=cp.IPOPT)
    host_logic_device.install(monkeypatch)
    with gpu.gpu_oracle():
        with pytest.raises(ValueError, match="Variable value must be in bounds") as ours:
            build().solve(nlp=True, solver=cp.IPOPT)
    assert str(ours.value) == str(ref.value)
