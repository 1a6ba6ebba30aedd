"""Batched best_of (SURVEY 8f item 1; reference loop: cvxpy/problems/problem.py:1249-1275, objective set:
ipopt_nlpif.py:87-89).  All starts advance in lock step over one compiled tape; the per-start results must be
the serial loop's, start by start."""
import numpy as np
import pytest

import kkt_newton
from dnlp_b200 import workloads as W
from dnlp_b200.best_of import best_of_lockstep, lockstep_newton_kkt
from oracle import ref_driver as R
from oracle.dnlp_oracle import RefOracles


class CpuBatch:
    """Test stand-in for BatchedOracles: the CPU oracle evaluated start by start."""

    def __init__(self, prob, B):
        self.r = RefOracles(prob)
        self.n, self.m, self.B = prob.n, prob.m, B
        self.js, self.hs = self.r.jacobianstructure(), self.r.hessianstructure()

    def jacobianstructure(self):
        return self.js

    def hessianstructure(self):
        return self.hs

    def eval(self, X, LAM, SIG):
        r = self.r
        out = {k: [] for k in ("f", "grad", "g", "jac", "hess")}
        for x, lam, s in zip(X, LAM, SIG):
            out["f"].append(float(r.objective(x)))
            out["grad"].append(np.array(r.gradient(x), float).ravel().copy())
            out["g"].append(np.array(r.constraints(x), float).ravel().copy())
            out["jac"].append(np.array(r.jacobian(x), float).ravel().copy())
            out["hess"].append(np.array(r.hessian(x, lam, s), float).ravel().copy())
        return {k: np.array(v) for k, v in out.items()}

    def close(self):
        pass


def test_lockstep_equals_serial_newton_start_by_start():
    prob = W.eigen_qcqp(8)
    rng = np.random.default_rng(0)
    X0 = rng.uniform(-1, 1, (12, 8))
    out = best_of_lockstep(prob, X0, evaluator=CpuBatch(prob, 12))
    assert out["converged"].all()
    eig = np.linalg.eigvalsh(W.eigen_qcqp_data(8))
    for b in range(12):
        x, lam, f, it = kkt_newton.solve(RefOracles(prob), X0[b])
        assert it == out["iterations"][b]
        np.testing.assert_allclose(out["x"][b], x, rtol=1e-9, atol=1e-11)
        assert abs(out["f"][b] - f) < 1e-9
        assert np.min(np.abs(-out["f"][b] - eig)) < 1e-8           # every start lands on an eigenpair
    assert out["best"] == int(np.argmin(out["all_objs"]))


@pytest.mark.skipif(not R.available(), reason="reference not present (oracle/_ref)")
def test_solve_best_of_reproduces_the_reference_loop():
    """The reference's loop, emulated with the stand-in solver (IPOPT is not installed): same sampler stream,
    chain re-applied per start, one solve per start.  solve_best_of must return the same objective set, the
    same best value, and leave them where the reference leaves them (extra_stats)."""
    cp = R.load_reference()
    from cvxpy.reductions.cvx_attr2constr import CvxAttr2Constr
    from cvxpy.reductions.dnlp2smooth.dnlp2smooth import Dnlp2Smooth
    from cvxpy.reductions.flip_objective import FlipObjective
    from cvxpy.reductions.solvers.nlp_solvers.ipopt_nlpif import IPOPT
    from cvxpy.reductions.solvers.solving_chain import SolvingChain
    from dnlp_b200.best_of import solve_best_of
    np.random.seed(0)
    n = 6
    A = np.random.randn(n, n)
    A = A.T @ A

    def build():
        x = cp.Variable(n)
        x.sample_bounds = [-1.0, 1.0]
        return x, cp.Problem(cp.Maximize(cp.quad_form(x, A, assume_PSD=True)), [cp.sum_squares(x) == 1])

    N = 7
    # the reference's loop (problem.py:1262-1275) with the Newton-KKT stand-in in place of IPOPT
    x, prob = build()
    chain = SolvingChain(reductions=[FlipObjective(), CvxAttr2Constr(reduce_bounds=False), Dnlp2Smooth(), IPOPT()])
    np.random.seed(11)
    want = []
    for run in range(N):
        prob.set_random_NLP_initial_point(run)
        data, inv = chain.apply(problem=prob)
        xs, lam, f, it = kkt_newton.solve(data["oracles"], data["x0"])
        want.append(-f)
    # ours: one compile, all starts in lock step
    x2, prob2 = build()
    np.random.seed(11)
    # the problem's own sense: the largest objective wins, values reported with their own sign
    val = solve_best_of(prob2, N, evaluator_factory=lambda pir, B: CpuBatch(pir, B), faithful=False)
    got = prob2.solver_stats.extra_stats["all_objs_from_best_of"]
    np.testing.assert_allclose(got, want, rtol=1e-9)
    assert abs(val - max(want)) < 1e-9 and abs(prob2.value - max(want)) < 1e-9
    # default = the reference's loop as written (problem.py:1262-1272; observed by running it end to end in
    # tests/test_prob_solve_end_to_end.py): `obj_value < best_obj` on the Maximize objective's own value keeps the
    # SMALLEST one, and the reported set is negated
    x3, prob3 = build()
    np.random.seed(11)
    val3 = solve_best_of(prob3, N, evaluator_factory=lambda pir, B: CpuBatch(pir, B))
    np.testing.assert_allclose(prob3.solver_stats.extra_stats["all_objs_from_best_of"], -np.asarray(want), rtol=1e-9)
    assert abs(val3 - min(want)) < 1e-9
    assert abs(np.sum(np.asarray(x2.value) ** 2) - 1.0) < 1e-9
    assert abs(float(np.asarray(x2.value) @ A @ np.asarray(x2.value)) - val) < 1e-8


@pytest.mark.gpu
def test_gpu_lockstep_best_of_on_batched_oracles():
    """BatchedOracles as the evaluator: 64 starts of the eigen-QCQP n = 24, one kernel sequence per iteration
    for all starts; per-start results equal the serial stand-in on the CPU oracle."""
    prob = W.eigen_qcqp(24)
    rng = np.random.default_rng(1)
    X0 = rng.uniform(-1, 1, (64, 24))
    out = best_of_lockstep(prob, X0)
    assert out["converged"].all()
    eig = np.linalg.eigvalsh(W.eigen_qcqp_data(24))
    for b in (0, 1, 17, 63):
        x, lam, f, it = kkt_newton.solve(RefOracles(prob), X0[b])
        assert it == out["iterations"][b]
        assert abs(out["f"][b] - f) <= 1e-8 * max(1.0, abs(f))
    assert np.all(np.min(np.abs(-out["f"][:, None] - eig[None, :]), axis=1) < 1e-7)
    assert abs(-out["f"][out["best"]] - max(-out["f"])) < 1e-12
