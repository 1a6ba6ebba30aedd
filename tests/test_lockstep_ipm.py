"""Lock-step interior-point best_of (dnlp_b200/lockstep_ipm.py) for problems with bounds and inequality rows.

CPU tier: the oracle port evaluated start by start stands in for BatchedOracles and a NumPy implementation of the
device's KKT factorisation (LDL' without pivoting, one refinement step) stands in for the device backend.  The serial
reference is the test-suite's barrier solver (cyipopt_standin.Problem) on RefOracles.
GPU tier: the device KKT kernels against the NumPy backend, and the driver end to end on BatchedOracles."""
import numpy as np
import pytest
import scipy.linalg as sla

import cyipopt_standin
from golden_util import REFPROBLEMS_DIR, Golden
from dnlp_b200 import workloads as W
from dnlp_b200.lockstep_ipm import lockstep_ipm
from oracle import ref_driver as R
from oracle.dnlp_oracle import RefOracles

TOL = 1e-8


class CpuBatch:
    """Test stand-in for BatchedOracles: the CPU oracle evaluated start by start."""

    def __init__(self, prob):
        self.r = RefOracles(prob)
        self.n, self.m = prob.n, prob.m
        self.js, self.hs = self.r.jacobianstructure(), self.r.hessianstructure()

    def jacobianstructure(self):
        return self.js

    def hessianstructure(self):
        return self.hs

    def eval(self, X, LAM=None, SIGMA=None, want=("f", "grad", "g", "jac", "hess")):
        r = self.r
        fn = {"f": lambda x, l, s: float(r.objective(x)), "grad": lambda x, l, s: r.gradient(x),
              "g": lambda x, l, s: r.constraints(x), "jac": lambda x, l, s: r.jacobian(x),
              "hess": lambda x, l, s: r.hessian(x, l, s)}
        out = {}
        for k in want:
            rows = [np.array(fn[k](np.array(X[b], dtype=np.float64), None if LAM is None else LAM[b],
                                   None if SIGMA is None else float(SIGMA[b])), dtype=np.float64).ravel().copy()
                    for b in range(len(X))]
            out[k] = np.array(rows).reshape(len(X), -1)
        if "f" in out:
            out["f"] = out["f"].reshape(len(X))
        return out


def kkt_targets(n, m, ns, slack_rows, jr, jc, hr, hc):
    """The device's scatter map (csrc/dnlp_batch.cu dnlp_batch_kkt_setup): lower-triangle targets of K in row-major
    order, each with its sources in pattern order (id < nnzH: HESS, id >= nnzH: JAC, -1: the slack column's -1)."""
    N, M = n + ns, n + ns + m
    nnzH = len(hr)
    tgt = {(i, i): [] for i in range(M)}
    for k, (r, c) in enumerate(zip(hr, hc)):
        tgt.setdefault((max(r, c), min(r, c)), []).append(k)
    for k, (r, c) in enumerate(zip(jr, jc)):
        tgt.setdefault((N + r, c), []).append(nnzH + k)
    for s, r in enumerate(slack_rows):
        tgt.setdefault((N + r, n + s), []).append(-1)
    return sorted(tgt.items())


def assemble(targets, N, M, nnzH, jac, hess, sigma, dw, dc):
    """K and the Hessian diagonal W_ii of one start, summed in the device's order: ((W_ii + Sigma_i) + dw)."""
    K, Wd = np.zeros((M, M)), np.zeros(N)
    for (i, j), srcs in targets:
        v = 0.0
        for s in srcs:
            v += -1.0 if s < 0 else (hess[s] if s < nnzH else jac[s - nnzH])
        if i == j:
            if i < N:
                Wd[i] = v
                v = (v + sigma[i]) + dw
            else:
                v = -dc
        K[i, j] = K[j, i] = v
    return K, Wd


def ldl_nopivot(K):
    """K = L D L' without pivoting; a zero pivot gives inf / NaN further on, as on the device.  Also returns the scale
    of every pivot, |K_jj| + sum_k L_jk^2 |d_k|: the magnitude of the terms whose sum it is."""
    A = np.array(K, dtype=np.float64)
    M = A.shape[0]
    d = np.zeros(M)
    scale = np.abs(np.diag(A)).copy()
    with np.errstate(all="ignore"):
        for j in range(M):
            d[j] = A[j, j]
            lcol = A[j + 1:, j] / d[j]
            A[j + 1:, j + 1:] -= np.outer(lcol, lcol * d[j])
            A[j + 1:, j] = lcol
            scale[j + 1:] += lcol * lcol * abs(d[j])
    return np.tril(A, -1) + np.eye(M), d, scale


def inertia_of(d, scale):
    """(n+, n-, n0) from the signs of D; a pivot within 1e-11 of its own scale (its terms cancelled) counts as zero."""
    zero = ~(np.abs(d) > 1e-11 * scale)
    pos, neg = int(np.sum(~zero & (d > 0))), int(np.sum(~zero & (d < 0)))
    return pos, neg, d.size - pos - neg


def ldl_solve(K, Wd, N, rhs):
    """The device's solve: factor, inertia, solve + one refinement step, normwise backward error <= 1e-8, dz' W dz."""
    M = K.shape[0]
    Lf, d, scale = ldl_nopivot(K)
    inert = inertia_of(d, scale)
    nan = np.full(M, np.nan)
    if inert != (N, M - N, 0):
        return nan, inert, np.nan
    with np.errstate(all="ignore"):
        def apply(v):
            y = sla.solve_triangular(Lf, v, lower=True, unit_diagonal=True, check_finite=False) / d
            return sla.solve_triangular(Lf.T, y, lower=False, unit_diagonal=True, check_finite=False)
        x = apply(rhs)
        x = x + apply(rhs - K @ x)
        r = rhs - K @ x
        den = np.abs(K).sum(axis=1).max() * np.abs(x).max(initial=0.0) + np.abs(rhs).max(initial=0.0)
        eta = np.abs(r).max(initial=0.0) / den if den > 0 else np.abs(r).max(initial=0.0)
        if not (np.all(np.isfinite(x)) and np.isfinite(eta) and eta <= 1e-8):
            return nan, inert, np.nan
        Wm = K[:N, :N].copy()
        Wm[np.diag_indices(N)] = Wd
        dz = x[:N]
        return x, inert, float(dz @ (Wm @ dz))


class NumpyKKT:
    """KKT backend of the CPU tests: the device algorithm in NumPy, start by start."""

    def __init__(self, ev):
        self.ev = ev

    def setup(self, slack_rows):
        jr, jc = (np.asarray(a, dtype=np.int64) for a in self.ev.jacobianstructure())
        hr, hc = (np.asarray(a, dtype=np.int64) for a in self.ev.hessianstructure())
        self.ns = len(slack_rows)
        self.N, self.M = self.ev.n + self.ns, self.ev.n + self.ns + self.ev.m
        self.nnzH = len(hr)
        self.targets = kkt_targets(self.ev.n, self.ev.m, self.ns, list(slack_rows), jr, jc, hr, hc)

    def load(self, X, LAM):
        r = self.ev.eval(X, LAM, np.ones(len(X)), want=("jac", "hess"))
        self.jac, self.hess = r["jac"], r["hess"]

    def matrix(self, b, sigma, dw, dc):
        return assemble(self.targets, self.N, self.M, self.nnzH, self.jac[b], self.hess[b], sigma, dw, dc)

    def solve(self, starts, sigma, dw, dc, rhs):
        sol, inert, wq = np.empty((len(starts), self.M)), np.empty((len(starts), 3), dtype=np.int64), np.empty(len(starts))
        for c, b in enumerate(starts):
            K, Wd = self.matrix(b, sigma[c], dw[c], dc[c])
            sol[c], inert[c], wq[c] = ldl_solve(K, Wd, self.N, rhs[c])
        return sol, inert, wq


# ---- fixtures ---------------------------------------------------------------------------------------------
def qcqp_fixture(n=16, k=3, B=12):
    P, q, rng = W.qcqp_data(n, k)
    return W.qcqp(P, q), rng.uniform(-1, 1, (B, n))


def refp007_fixture(B=8):
    """The reference's best_of test problem (test_best_of.py::test_circle_packing_best_of): n=36, 35 inequality rows."""
    prob = Golden("refp_007", REFPROBLEMS_DIR).problem
    rng = np.random.default_rng(7)
    return prob, prob.x0[None, :] + 0.1 * rng.standard_normal((B, prob.n))


def twosided_fixture(B=8):
    """A QCQP whose rows are two-sided (0 <= 1 - x'P_i x - q_i'x <= 2.5) and whose variables are boxed both ways."""
    P, q, rng = W.qcqp_data(10, 3, seed=3)
    prob = W.qcqp(P, q)
    prob.cu = np.full(3, 2.5)
    prob.lb, prob.ub = np.full(10, -0.8), np.full(10, 1.2)
    return prob, rng.uniform(-0.8, 1.2, (B, 10))


FIXTURES = {"qcqp16": qcqp_fixture, "refp007": refp007_fixture, "twosided": twosided_fixture}


def bounds(prob):
    return dict(lb=prob.lb, ub=prob.ub, cl=prob.cl, cu=prob.cu)


def run_lockstep(prob, X0, **kw):
    ev = CpuBatch(prob)
    return lockstep_ipm(ev, NumpyKKT(ev), X0, **bounds(prob), **kw)


class _KeepPoints:
    """RefOracles that holds on to every point it is given: the stand-in asserts that each callback gets a fresh array
    (by id), and a freed array's id can be handed out again."""

    def __init__(self, prob):
        self.r, self.kept = RefOracles(prob), []

    def __getattr__(self, name):
        fn = getattr(self.r, name)
        if name in ("objective", "gradient", "constraints", "jacobian", "hessian"):
            def call(x, *a):
                self.kept.append(x)
                return fn(x, *a)
            return call
        return fn


def run_standin(prob, x0):
    n, m = prob.n, prob.m
    b = {k: (None if v is None else np.where(np.isinf(v), np.sign(v) * 2e19, v)) for k, v in bounds(prob).items()}
    p = cyipopt_standin.Problem(n, m, problem_obj=_KeepPoints(prob), lb=b["lb"], ub=b["ub"], cl=b["cl"], cu=b["cu"])
    return cyipopt_standin._BarrierSolver(p).run(np.asarray(x0, dtype=np.float64))   # Problem.solve without the info dict


_cache = {}


def lockstep_result(name):
    if name not in _cache:
        prob, X0 = FIXTURES[name]()
        _cache[name] = (prob, X0, run_lockstep(prob, X0))
    return _cache[name]


def check_optimality(prob, x, lam, zL, zU, what):
    """Primal feasibility, stationarity of the Lagrangian and complementarity, recomputed from RefOracles at the
    returned point and multipliers, against the solver's tolerance (IPOPT's scaled optimality error, tol = 1e-8)."""
    r = RefOracles(prob)
    n, m = prob.n, prob.m
    lb = np.full(n, -np.inf) if prob.lb is None else prob.lb
    ub = np.full(n, np.inf) if prob.ub is None else prob.ub
    cl = np.full(m, -np.inf) if prob.cl is None else prob.cl
    cu = np.full(m, np.inf) if prob.cu is None else prob.cu
    g = np.asarray(r.constraints(x), float).ravel() if m else np.zeros(0)
    viol = max(np.max(lb - x, initial=0.0), np.max(x - ub, initial=0.0), np.max(cl - g, initial=0.0),
               np.max(g - cu, initial=0.0))
    eq = cl == cu
    viol = max(viol, np.max(np.abs(g[eq] - cl[eq]), initial=0.0))
    assert viol <= TOL * (1 + 1e-6), "%s: primal infeasibility %.3e" % (what, viol)
    jr, jc = r.jacobianstructure()
    J = np.zeros((m, n))
    np.add.at(J, (np.asarray(jr), np.asarray(jc)), np.asarray(r.jacobian(x), float).ravel())
    grad = np.asarray(r.gradient(x), float).ravel()
    # the slack bound multipliers (not returned) equal |lam| on the inequality rows at a solution
    sd = max(100.0, (2 * np.abs(lam).sum() + zL.sum() + zU.sum()) / max(m + 2 * (n + np.sum(~eq)), 1)) / 100.0
    stat = np.abs(grad + J.T @ lam - zL + zU).max(initial=0.0)
    assert stat <= TOL * sd * (1 + 1e-6), "%s: stationarity %.3e" % (what, stat)
    with np.errstate(invalid="ignore"):            # inf * 0 on the absent bounds, masked out
        comp = _complementarity(x, g, lb, ub, cl, cu, eq, lam, zL, zU)
    assert comp <= 10 * TOL * sd, "%s: complementarity %.3e" % (what, comp)


def _complementarity(x, g, lb, ub, cl, cu, eq, lam, zL, zU):
    return max(np.max(np.where(np.isfinite(lb), (x - lb) * zL, 0.0), initial=0.0),
               np.max(np.where(np.isfinite(ub), (ub - x) * zU, 0.0), initial=0.0),
               np.max(np.where(~eq & np.isfinite(cl), (g - cl) * np.maximum(-lam, 0.0), 0.0), initial=0.0),
               np.max(np.where(~eq & np.isfinite(cu), (cu - g) * np.maximum(lam, 0.0), 0.0), initial=0.0))


# ---- CPU tier ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["qcqp16", "refp007"])
def test_lockstep_equals_start_by_start(name):
    """Masks and line-search rounds do not leak between starts: B starts at once give bit-identical per-start
    results to the same driver run on each start alone."""
    prob, X0, out = lockstep_result(name)
    for b in range(len(X0)):
        one = run_lockstep(prob, X0[b:b + 1])
        assert one["status"][0] == out["status"][b] and one["iterations"][0] == out["iterations"][b], b
        for k in ("x", "lam", "zL", "zU"):
            assert np.array_equal(one[k][0], out[k][b]), (b, k)
        assert one["f"][0] == out["f"][b]


# Starts whose inertia decisions differ from the stand-in's.  The stand-in counts a Bunch-Kaufman pivot as zero below
# 1e-11 max(1, max|d|); the no-pivot factorisation compares every pivot with its own scale (csrc/dnlp_batch_kkt.cuh).
# qcqp16 start 5: late in the solve Sigma spans ~1e-12 .. 1e11; the stand-in's global threshold then reads the small
# constraint-block pivots as zero, raises dw until the system cannot be regularised and stops with -3 at iteration 45;
# the lock-step driver converges at iteration 39 to the same objective.
STANDIN_DIFFERS = {("qcqp16", 5): (0, 39)}


@pytest.mark.parametrize("name", ["qcqp16", "twosided"])
def test_agrees_with_the_serial_standin(name):
    """Per start: the stand-in's status and iteration count; where both converge, the objective within 1e-8 relative
    and x within 1e-6."""
    prob, X0, out = lockstep_result(name)
    for b in range(len(X0)):
        ref = run_standin(prob, X0[b])
        if (name, b) in STANDIN_DIFFERS:
            assert (out["status"][b], out["iterations"][b]) == STANDIN_DIFFERS[name, b]
            assert ref["status"] == -3
            continue
        assert out["status"][b] == ref["status"], (b, out["status"][b], ref["status"])
        assert out["iterations"][b] == ref["iterations"], (b, out["iterations"][b], ref["iterations"])
        if ref["status"] == 0:
            assert abs(out["f"][b] - ref["f"]) <= 1e-8 * max(1.0, abs(ref["f"])), b
            np.testing.assert_allclose(out["x"][b], ref["x"], rtol=0, atol=1e-6)


def test_refp007_converges_where_the_standin_does():
    """The circle-packing problem is nonconvex with many local optima.  The two solvers regularise at different
    iterations there (see STANDIN_DIFFERS), so they follow different paths: the stand-in ends 4 of these 8 starts
    with -3 or -1, the lock-step driver 1.  Asserted: every start the stand-in solves, the driver solves too."""
    prob, X0, out = lockstep_result("refp007")
    ref = [run_standin(prob, x)["status"] for x in X0]
    for b in range(len(X0)):
        if ref[b] == 0:
            assert out["status"][b] == 0, b
    assert np.sum(out["status"] == 0) >= np.sum(np.array(ref) == 0)


@pytest.mark.parametrize("name", ["qcqp16", "refp007", "twosided"])
def test_independent_optimality(name):
    prob, X0, out = lockstep_result(name)
    conv = np.flatnonzero(out["status"] == 0)
    assert conv.size > 0
    for b in conv:
        check_optimality(prob, out["x"][b], out["lam"][b], out["zL"][b], out["zU"][b], "%s start %d" % (name, b))


def test_numpy_ldl_inertia_matches_eigenvalues():
    """The no-pivot LDL' of the NumPy backend reads the inertia of a quasi-definite K off D (Sylvester)."""
    rng = np.random.default_rng(5)
    N, m = 30, 7
    H = rng.standard_normal((N, N))
    H = H + H.T + 12 * np.eye(N)
    A = rng.standard_normal((m, N))
    K = np.block([[H, A.T], [A, -1e-9 * np.eye(m)]])
    _, d, scale = ldl_nopivot(K)
    ev = np.linalg.eigvalsh(K)
    assert inertia_of(d, scale) == (int(np.sum(ev > 0)), int(np.sum(ev < 0)), 0) == (N, m, 0)
    rhs = rng.standard_normal(N + m)
    x, inert, _ = ldl_solve(K, np.diag(H).copy(), N, rhs)
    np.testing.assert_allclose(K @ x, rhs, rtol=0, atol=1e-9 * np.abs(rhs).max())


@pytest.mark.skipif(not R.available(), reason="reference not present (oracle/_ref)")
def test_solve_best_of_with_bounds_and_inequalities():
    """solve_best_of on a live reference problem with variable bounds and <= rows: a value instead of
    NotImplementedError, and all_objs_from_best_of equal to the serial stand-in run start by start on the reference's
    own sampler stream."""
    cp = R.load_reference()
    from cvxpy.reductions.cvx_attr2constr import CvxAttr2Constr
    from cvxpy.reductions.dnlp2smooth.dnlp2smooth import Dnlp2Smooth
    from cvxpy.reductions.solvers.nlp_solvers.ipopt_nlpif import IPOPT
    from cvxpy.reductions.solvers.solving_chain import SolvingChain
    from dnlp_b200.best_of import solve_best_of

    def build():
        x = cp.Variable(4, bounds=[-2.0, 2.0])
        x.sample_bounds = [-1.0, 1.0]
        A = np.array([[1.0, 2.0, 0.0, -1.0], [0.5, -1.0, 1.0, 0.0]])
        obj = cp.Minimize(cp.sum(cp.exp(x)) - cp.sum_squares(x) / 4)
        return x, cp.Problem(obj, [A @ x <= 1.0, cp.sum_squares(x) <= 3.0])

    N = 5
    x, prob = build()
    chain = SolvingChain(reductions=[CvxAttr2Constr(reduce_bounds=False), Dnlp2Smooth(), IPOPT()])
    np.random.seed(3)
    want = []
    for run in range(N):
        prob.set_random_NLP_initial_point(run)
        data, inv = chain.apply(problem=prob)
        p = cyipopt_standin.Problem(len(data["x0"]), len(data["cl"]), problem_obj=data["oracles"], lb=data["lb"],
                                    ub=data["ub"], cl=data["cl"], cu=data["cu"])
        want.append(p.solve(data["x0"])[1]["obj_val"])
    x2, prob2 = build()
    np.random.seed(3)

    val = solve_best_of(prob2, N, evaluator_factory=lambda pir, B: CpuBatch(pir), kkt_factory=NumpyKKT)
    np.testing.assert_allclose(prob2.solver_stats.extra_stats["all_objs_from_best_of"], want, rtol=1e-8)
    assert abs(val - min(want)) <= 1e-8 * max(1.0, abs(min(want)))


# ---- GPU tier ----------------------------------------------------------------------------------------------
def _random_kkt_inputs(ev, slack_rows, count, rng):
    """A random point with LAM spread wide (indefinite W), Sigma spanning 1e-8 .. 1e8."""
    N = ev.n + len(slack_rows)
    X = rng.uniform(-1, 1, (ev.batch, ev.n))
    LAM = 3.0 * rng.standard_normal((ev.batch, ev.m))
    sigma = 10.0 ** rng.uniform(-8, 8, (count, N))
    dw = np.where(rng.uniform(size=count) < 0.5, 0.0, 10.0 ** rng.uniform(-4, 2, count))
    dc = 10.0 ** rng.uniform(-9, -6, count)
    rhs = rng.standard_normal((count, N + ev.m))
    return X, LAM, sigma, dw, dc, rhs


def _device_vs_numpy(prob, B, starts, seed):
    from dnlp_b200.multistart import BatchedOracles
    rng = np.random.default_rng(seed)
    ev = BatchedOracles(prob, B)
    try:
        cl = np.full(prob.m, -np.inf) if prob.cl is None else prob.cl
        cu = np.full(prob.m, np.inf) if prob.cu is None else prob.cu
        slack = np.flatnonzero(cl != cu)
        ev.kkt_setup(slack)
        X, LAM, sigma, dw, dc, rhs = _random_kkt_inputs(ev, slack, len(starts), rng)
        ev.upload(X, LAM, np.ones(B))
        ev.run_device(("jac", "hess"))
        sol, inert, wq = ev.kkt_solve(starts, sigma, dw, dc, rhs)
        host = CpuBatch(prob)
        ref = NumpyKKT(host)
        ref.setup(slack)
        ref.load(X, LAM)
        N = ref.N
        jr = np.asarray(host.jacobianstructure()[0])
        for c, b in enumerate(starts):
            K, Wd = ref.matrix(b, sigma[c], dw[c], dc[c])
            # the device oracle and the port may differ in the last bit of an entry: compare the scatter on the
            # device's own HESS / JAC values
            Kd = ev.kkt_matrix(b)
            hv, jv = ev.read_output("hess")[b], ev.read_output("jac")[b]
            Kh, Wdh = assemble(ref.targets, N, ref.M, ref.nnzH, jv, hv, sigma[c], dw[c], dc[c])
            assert np.array_equal(Kd, Kh), "start %d: assembled K differs from the host scatter" % b
            np.testing.assert_allclose(Kd, K, rtol=1e-12, atol=1e-12 * np.abs(K).max())
            s_ref, i_ref, w_ref = ldl_solve(Kh, Wdh, N, rhs[c])
            assert tuple(inert[c]) == tuple(i_ref), (b, inert[c], i_ref)
            if np.isfinite(s_ref).all():
                assert np.isfinite(sol[c]).all(), b
                np.testing.assert_allclose(sol[c], s_ref, rtol=1e-10, atol=1e-10 * np.abs(s_ref).max())
                dz = s_ref[:N]
                Wm = np.abs(Kh[:N, :N])
                Wm[np.diag_indices(N)] = np.abs(Wdh)
                assert abs(wq[c] - w_ref) <= 1e-10 * (np.abs(dz) @ Wm @ np.abs(dz)), b
            else:
                assert not np.isfinite(sol[c]).any(), b
        return inert
    finally:
        ev.close()


@pytest.mark.gpu
def test_gpu_kkt_matches_numpy_refp007():
    """N + m = 126 (refp_007: 35 slack rows), 48 of 64 starts in a non-contiguous order."""
    prob, _ = refp007_fixture()
    starts = np.random.default_rng(11).permutation(64)[:48]
    inert = _device_vs_numpy(prob, 64, starts, seed=1)
    assert len({tuple(i) for i in inert}) >= 2          # both right and wrong inertia occur


@pytest.mark.gpu
def test_gpu_kkt_matches_numpy_c4_shape():
    """N + m = 528: the C4 QCQP (n = 512, k = 8 slack rows), B = 64, a non-contiguous subset of starts."""
    P, q, _ = W.qcqp_data(512, 8)
    prob = W.qcqp(P, q)
    starts = np.array([63, 0, 5, 17, 18, 40, 2, 33, 9, 50])
    _device_vs_numpy(prob, 64, starts, seed=2)


@pytest.mark.gpu
def test_gpu_kkt_rank_deficient_jacobian():
    """Two identical constraint rows (J rank deficient): dc > 0 keeps K solvable, and the inertia agrees."""
    P, q, _ = W.qcqp_data(24, 2, seed=4)
    P = [P[0], P[1], P[1]]
    q = np.vstack([q[0], q[1], q[1]])
    prob = W.qcqp(P, q)
    _device_vs_numpy(prob, 16, np.arange(15, -1, -2), seed=3)


def _end_to_end(prob, X0, cpu_check):
    from dnlp_b200.lockstep_ipm import DeviceKKT
    from dnlp_b200.multistart import BatchedOracles
    ev = BatchedOracles(prob, len(X0))
    try:
        out = lockstep_ipm(ev, DeviceKKT(ev), X0, **bounds(prob))
    finally:
        ev.close()
    cpu = run_lockstep(prob, X0[cpu_check])
    assert np.array_equal(out["status"][cpu_check], cpu["status"])
    both = (cpu["status"] == 0)
    fo, fc = out["f"][cpu_check][both], cpu["f"][both]
    assert np.all(np.abs(fo - fc) <= 1e-8 * np.maximum(1.0, np.abs(fc)))
    for b in np.flatnonzero(out["status"] == 0):
        check_optimality(prob, out["x"][b], out["lam"][b], out["zL"][b], out["zU"][b], "start %d" % b)
    return out


@pytest.mark.gpu
def test_gpu_end_to_end_qcqp64():
    P, q, rng = W.qcqp_data(64, 4)
    prob = W.qcqp(P, q)
    X0 = rng.uniform(-1, 1, (256, 64))
    out = _end_to_end(prob, X0, np.arange(0, 256, 8))     # the CPU run on every 8th start: the port is slow
    assert np.sum(out["status"] == 0) > 0


@pytest.mark.gpu
def test_gpu_end_to_end_refp007():
    prob, X0 = refp007_fixture(64)
    out = _end_to_end(prob, X0, np.arange(0, 64, 4))
    assert np.sum(out["status"] == 0) > 0


@pytest.mark.gpu
def test_gpu_full_c4_shape(record_property):
    """n = 512, k = 8, B = 4096 starts drawn as bench.py draws them: the driver completes and at least one start
    converges; a sample of the converged starts passes the independent optimality check."""
    from dnlp_b200.lockstep_ipm import DeviceKKT
    from dnlp_b200.multistart import BatchedOracles
    P, q, rng = W.qcqp_data(512, 8)
    prob = W.qcqp(P, q)
    X0 = rng.uniform(-1, 1, (4096, 512))
    ev = BatchedOracles(prob, 4096)
    try:
        out = lockstep_ipm(ev, DeviceKKT(ev), X0, **bounds(prob))
    finally:
        ev.close()
    st, cnt = np.unique(out["status"], return_counts=True)
    record_property("status_histogram", dict(zip(st.tolist(), cnt.tolist())))
    record_property("iterations_histogram", np.bincount(out["iterations"]).tolist())
    print("C4 lock-step IPM: status histogram", dict(zip(st.tolist(), cnt.tolist())), "iterations min / median / max",
          out["iterations"].min(), np.median(out["iterations"]), out["iterations"].max())
    conv = np.flatnonzero(out["status"] == 0)
    assert conv.size > 0
    for b in conv[:: max(1, conv.size // 16)]:
        check_optimality(prob, out["x"][b], out["lam"][b], out["zL"][b], out["zU"][b], "start %d" % b)
