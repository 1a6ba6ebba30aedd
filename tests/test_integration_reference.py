"""Drop-in boundary against the LIVE reference (runs only where oracle/make_ref.sh has installed it as oracle/_ref).

`install()` rebinds the one name the reference's solver interface instantiates; the reduction
chain then yields a GpuOracles object whose structures equal the reference Oracles' bit for bit.
The device upload is stubbed here (no GPU in the build container); the CUDA path itself is
covered by tests/test_gpu_parity.py."""
import types

import numpy as np
import pytest

from oracle import ref_driver as R

pytestmark = pytest.mark.skipif(not R.available(), reason="reference not present (oracle/_ref)")


@pytest.fixture(scope="module")
def cp():
    return R.load_reference()


def _chain(cp, prob):
    from cvxpy.reductions.cvx_attr2constr import CvxAttr2Constr
    from cvxpy.reductions.dnlp2smooth.dnlp2smooth import Dnlp2Smooth
    from cvxpy.reductions.flip_objective import FlipObjective
    from cvxpy.reductions.solvers.nlp_solvers.ipopt_nlpif import IPOPT
    from cvxpy.reductions.solvers.solving_chain import SolvingChain
    red = ([FlipObjective()] if type(prob.objective) == cp.Maximize else []) + \
        [CvxAttr2Constr(reduce_bounds=False), Dnlp2Smooth(), IPOPT()]
    return SolvingChain(reductions=red).apply(problem=prob)[0]


def test_install_swaps_the_oracle_and_structures_match(cp, monkeypatch):
    import dnlp_b200.nlp_solver as gpu
    from dnlp_b200 import _cabi
    from dnlp_b200.oracles import GpuOracles

    class FakeDevice:                       # no GPU here: keep the compile, skip the upload
        def __init__(self, tape, device=0):
            self.tape = tape

        def close(self):
            pass

        def bind_outputs(self, *a, **k):
            pass
    monkeypatch.setattr(_cabi, "DeviceTape", FakeDevice)
    monkeypatch.setattr(_cabi, "pinned_empty", lambda k: (np.empty(k), types.SimpleNamespace(free=lambda: None)))

    def build():
        np.random.seed(0)
        x = cp.Variable(4, bounds=[0, 6])
        x.value = np.array([1.0, 5.0, 5.0, 1.0])
        return cp.Problem(cp.Minimize(x[0] * x[3] * (x[0] + x[1] + x[2]) + x[2]),
                          [x[0] * x[1] * x[2] * x[3] >= 25, cp.sum(cp.square(x)) == 40])

    ref = _chain(cp, build())["oracles"]
    with gpu.gpu_oracle():
        data = _chain(cp, build())
    ours = data["oracles"]
    assert isinstance(ours, GpuOracles)
    assert type(ref).__name__ == "Oracles"
    for a, b in zip(ours.jacobianstructure(), ref.jacobianstructure()):
        assert a.dtype == np.int32
        np.testing.assert_array_equal(a, b)
    for a, b in zip(ours.hessianstructure(), ref.hessianstructure()):
        np.testing.assert_array_equal(a, b)
    # the bound methods the solver interfaces read from `data` exist with the reference's names
    for name in ("objective", "gradient", "constraints", "jacobian", "jacobianstructure",
                 "hessian", "hessianstructure"):
        assert callable(data[name])
    assert hasattr(ours, "intermediate") and ours.iterations == 0
    # after the context manager the reference's own class is back
    import cvxpy.reductions.solvers.nlp_solvers.nlp_solver as mod
    assert mod.Oracles is type(ref)


def test_best_of_style_reapplied_chain_reuses_the_compiled_oracle(cp, monkeypatch):
    """The reference's best_of loop re-applies the reduction chain per start (problem.py:1249-1275):
    fresh auxiliary variables and ids every time, same smooth problem.  The factory must hand back
    the oracle that is already compiled, re-armed with the new initial point."""
    import dnlp_b200.nlp_solver as gpu
    from dnlp_b200 import _cabi

    class FakeDevice:
        def __init__(self, tape, device=0):
            self.tape = tape

        def close(self):
            pass

        def bind_outputs(self, *a, **k):
            pass
    monkeypatch.setattr(_cabi, "DeviceTape", FakeDevice)
    monkeypatch.setattr(_cabi, "pinned_empty", lambda k: (np.empty(k), types.SimpleNamespace(free=lambda: None)))

    def build(start, rhs=1.0):
        np.random.seed(0)
        A = np.random.randn(5, 5)
        x = cp.Variable(5)
        x.value = start
        return cp.Problem(cp.Minimize(cp.sum(cp.logistic(A @ x)) + cp.sum(cp.exp(-x))), [cp.sum_squares(x) == rhs])

    with gpu.gpu_oracle():
        gpu.ORACLE_CACHE.hits = gpu.ORACLE_CACHE.misses = 0
        d1 = _chain(cp, build(np.ones(5)))
        o1 = d1["oracles"]
        x0_first = np.array(o1.initial_point, copy=True)
        d2 = _chain(cp, build(np.full(5, 0.25)))
        o2 = d2["oracles"]
        assert o2 is o1 and (gpu.ORACLE_CACHE.hits, gpu.ORACLE_CACHE.misses) == (1, 1)
        assert not np.array_equal(o2.initial_point, x0_first)            # re-armed with the new start
        np.testing.assert_array_equal(o2.initial_point, d2["x0"])
        o2.intermediate(0, 9, 0, 0, 0, 0, 0, 0, 0, 0, 0)
        d3 = _chain(cp, build(np.ones(5)))
        assert d3["oracles"] is o1 and d3["oracles"].iterations == 0
        d4 = _chain(cp, build(np.ones(5), rhs=2.0))                      # another constant: another oracle
        assert d4["oracles"] is not o1


def test_reference_best_of_loop_compiles_once(cp, monkeypatch):
    """The reference's own best_of problem (tests/NLP_tests/test_best_of.py:11-33) driven the way
    Problem._solve drives it (problems/problem.py:1262-1266): a random initial point per run, the
    chain re-applied every time.  One compile, best_of - 1 cache hits, the same structures throughout."""
    import dnlp_b200.nlp_solver as gpu
    from dnlp_b200 import _cabi

    class FakeDevice:
        def __init__(self, tape, device=0):
            self.tape = tape

        def close(self):
            pass

        def bind_outputs(self, *a, **k):
            pass
    monkeypatch.setattr(_cabi, "DeviceTape", FakeDevice)
    monkeypatch.setattr(_cabi, "pinned_empty", lambda k: (np.empty(k), types.SimpleNamespace(free=lambda: None)))
    rng = np.random.default_rng(5)
    n = 5
    radius = rng.uniform(1.0, 3.0, n)
    centers = cp.Variable((n, 2), name="c")
    constraints = []
    for i in range(n - 1):
        constraints += [cp.sum((centers[i, :] - centers[i + 1:, :]) ** 2, axis=1) >= (radius[i] + radius[i + 1:]) ** 2]
    prob = cp.Problem(cp.Minimize(cp.max(cp.norm_inf(centers, axis=1) + radius)), constraints)
    centers.sample_bounds = [-5.0, 5.0]
    n_runs = 4
    with gpu.gpu_oracle():
        gpu.ORACLE_CACHE.hits = gpu.ORACLE_CACHE.misses = 0
        seen, starts = [], []
        for run in range(n_runs):
            prob.set_random_NLP_initial_point(run)
            data = _chain(cp, prob)
            seen.append(data["oracles"])
            starts.append(np.array(data["x0"], copy=True))
            np.testing.assert_array_equal(data["oracles"].initial_point, data["x0"])
        assert all(o is seen[0] for o in seen)
        assert (gpu.ORACLE_CACHE.hits, gpu.ORACLE_CACHE.misses) == (n_runs - 1, 1)
        assert not np.array_equal(starts[0], starts[1])
    ref = _chain(cp, prob)["oracles"]                                   # the reference's own object again
    for a, b in zip(seen[0].jacobianstructure(), ref.jacobianstructure()):
        np.testing.assert_array_equal(a, b)
    for a, b in zip(seen[0].hessianstructure(), ref.hessianstructure()):
        np.testing.assert_array_equal(a, b)


def test_parameters_are_value_slots_no_recompile(cp, monkeypatch):
    """cvxpy Parameters (expressions/constants/parameter.py:35) in sums and elementwise products become value
    SLOTS of the tape: a new value re-arms the resident oracle (one small upload) instead of compiling a new
    one, and every output follows the new value exactly as the reference's `.value`-reading rules do.  A
    Parameter in a position that changes coefficient arrays (the matrix of a product with variables) is
    frozen instead: a new value there is a new fingerprint."""
    import dnlp_b200.nlp_solver as gpu
    from dnlp_b200 import _cabi
    from oracle.dnlp_oracle import RefOracles
    from tape_interp import TapeInterp

    uploads = []

    class FakeDevice:
        def __init__(self, tape, device=0):
            self.tape = tape

        def close(self):
            pass

        def bind_outputs(self, *a, **k):
            pass

        def set_params(self, values):
            uploads.append(np.array(values, copy=True))
    monkeypatch.setattr(_cabi, "DeviceTape", FakeDevice)
    monkeypatch.setattr(_cabi, "pinned_empty", lambda k: (np.empty(k), types.SimpleNamespace(free=lambda: None)))
    gamma = cp.Parameter(nonneg=True)
    b = cp.Parameter(3)
    x = cp.Variable(3)
    x.value = np.array([0.3, 0.5, 0.2])
    prob = cp.Problem(cp.Minimize(cp.sum(cp.exp(x)) + gamma * cp.sum_squares(x - b)),
                      [cp.sum(x) == 1, cp.multiply(b, cp.exp(x)) <= 9 + gamma])
    xv = np.array([0.3, 0.5, 0.2])
    with gpu.gpu_oracle():
        gpu.ORACLE_CACHE.hits = gpu.ORACLE_CACHE.misses = 0
        # (np.float64, not float: the reference's multiply._hess_vec calls x.value.flatten, binary_operators.py:517)
        gamma.value, b.value = np.float64(0.5), np.array([1.0, 2.0, 3.0])
        d1 = _chain(cp, prob)
        o1 = d1["oracles"]
        assert o1.tape.n_params == 4
        it = TapeInterp(o1.tape)
        ref = _chain_reference(cp, prob)
        xv = np.asarray(d1["x0"], dtype=np.float64) * 1.05 + 0.01      # the smooth problem's point (aux variables too)
        lam = np.linspace(-0.4, 0.6, len(d1["cl"]))
        for gval, bval in ((0.5, [1.0, 2.0, 3.0]), (2.0, [1.0, 2.0, 3.0]), (0.1, [3.0, -1.0, 0.5])):
            gamma.value, b.value = np.float64(gval), np.array(bval)
            d = _chain(cp, prob)                                        # what prob.solve() does per solve
            assert d["oracles"] is o1                                    # re-armed, never recompiled
            np.testing.assert_array_equal(uploads[-1], np.concatenate([[gval], bval]) if o1.problem.params[0].size == 1
                                          else np.concatenate([bval, [gval]]))
            it.set_params(uploads[-1])
            r = _chain_reference(cp, prob)["oracles"]
            r.jacobianstructure(), r.hessianstructure()
            np.testing.assert_allclose(it.eval("f", xv), r.objective(xv), rtol=1e-12)
            np.testing.assert_allclose(it.eval("grad", xv), r.gradient(xv), rtol=1e-12)
            np.testing.assert_allclose(it.eval("g", xv), r.constraints(xv), rtol=1e-12)
            np.testing.assert_allclose(it.eval("jac", xv), np.asarray(r.jacobian(xv)).ravel(), rtol=1e-12)
            np.testing.assert_allclose(it.eval("hess", xv, lam, 0.7), np.asarray(r.hessian(xv, lam, 0.7)).ravel(), rtol=1e-12)
            # the CPU oracle sees the folded problem (parameters at their current values)
            ro = RefOracles(d["oracles"].problem.folded())
            np.testing.assert_allclose(ro.objective(xv), r.objective(xv), rtol=1e-12)
        assert gpu.ORACLE_CACHE.misses == 1
        # a parameter MATRIX multiplying variables is frozen: new value -> new tape
        P = cp.Parameter((2, 3))
        P.value = np.arange(6.0).reshape(2, 3)
        prob2 = cp.Problem(cp.Minimize(cp.sum(cp.exp(P @ x))), [cp.sum(x) == 1])
        oa = _chain(cp, prob2)["oracles"]
        assert oa.tape.n_params == 0
        P.value = P.value + 1.0
        assert _chain(cp, prob2)["oracles"] is not oa


def _chain_reference(cp, prob):
    """The reference's own Oracles for the same problem (install() not active)."""
    import importlib
    mod = importlib.import_module("cvxpy.reductions.solvers.nlp_solvers.nlp_solver")
    import dnlp_b200.nlp_solver as gpu
    saved = mod.Oracles
    mod.Oracles = gpu._saved.get("Oracles", saved)
    try:
        return _chain(cp, prob)
    finally:
        mod.Oracles = saved


def test_dual_recovery_through_the_reference_chain(cp):
    """SURVEY 8f item 4: the reference returns no duals (ipopt_nlpif.py:100).  With install_dual_recovery()
    the solver's constraint multipliers travel back through the reference's own invert chain
    (canonicalization.py:76-84) to `constraint.dual_value`.  IPOPT is not installed, so the multipliers come
    from the Newton-KKT stand-in driving the reference's own Oracles (same Lagrangian f + mult_g' g); the
    recovered duals must make the ORIGINAL problem's Lagrangian stationary, with cvxpy's signs."""
    import dnlp_b200.nlp_solver as gpu
    import kkt_newton
    from cvxpy.reductions.cvx_attr2constr import CvxAttr2Constr
    from cvxpy.reductions.dnlp2smooth.dnlp2smooth import Dnlp2Smooth
    from cvxpy.reductions.solvers.nlp_solvers.ipopt_nlpif import IPOPT
    from cvxpy.reductions.solvers.solving_chain import SolvingChain
    rng = np.random.default_rng(0)
    n = 6
    A = rng.standard_normal((2, n))
    x = cp.Variable(n)
    x.value = np.full(n, 0.3)
    eq = A @ x == np.array([0.5, -0.2])
    ineq = cp.sum(cp.exp(x)) >= 6.5                      # active at the optimum (treated as an equality by the stand-in)
    prob = cp.Problem(cp.Minimize(cp.sum(cp.logistic(x)) + cp.sum_squares(x)), [eq, ineq])
    gpu.install_dual_recovery()
    try:
        chain = SolvingChain(reductions=[CvxAttr2Constr(reduce_bounds=False), Dnlp2Smooth(), IPOPT()])
        data, inverse_data = chain.apply(problem=prob)
        o = data["oracles"]
        xs, lam, f, iters = kkt_newton.solve(o, data["x0"], tol=1e-11)
        info = {"status": 0, "x": xs, "obj_val": f, "mult_g": lam, "iterations": iters}
        prob.unpack_results(info, chain, inverse_data)               # runs chain.invert: solver stage first
    finally:
        gpu.uninstall()
    nu, mu = np.asarray(eq.dual_value, float), float(ineq.dual_value)
    assert nu.shape == (2,) and mu > 0                   # an active inequality: nonnegative dual
    xv = np.asarray(x.value, float)
    assert abs(np.exp(xv).sum() - 6.5) < 1e-8
    # stationarity of f + nu'(A x - b) + mu (6.5 - sum exp(x)) in the ORIGINAL variables
    grad_f = np.exp(xv) / (1 + np.exp(xv)) + 2 * xv
    resid = grad_f + A.T @ nu - mu * np.exp(xv)
    assert np.linalg.norm(resid, np.inf) < 1e-7, resid
    # without the hook the reference hands back no duals at all
    data, inverse_data = chain.apply(problem=prob)
    sol = chain.invert({"status": 0, "x": xs, "obj_val": f, "mult_g": lam, "iterations": iters}, inverse_data)
    assert not sol.dual_vars
