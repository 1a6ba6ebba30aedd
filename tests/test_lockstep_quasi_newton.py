"""Quasi-Newton mode of the lock-step interior-point best_of (hessian_approximation="limited-memory").

The driver keeps one dense damped-BFGS matrix per start instead of the Hessian of the Lagrangian (the update of the
test-suite's serial stand-in, tests/cyipopt_standin.py).  CPU tier: the oracle port start by start and a NumPy backend
that applies the device's update formula in its expression order; the serial reference is the stand-in with the same
option.  GPU tier: the device update against a long-double reference, the quasi-Newton KKT assembly against the NumPy
scatter, and the driver end to end on BatchedOracles."""
import numpy as np
import pytest

import cyipopt_standin
from dnlp_b200 import workloads as W
from dnlp_b200.lockstep_ipm import lockstep_ipm
from oracle import ref_driver as R
from test_lockstep_ipm import (FIXTURES, CpuBatch, NumpyKKT, _KeepPoints, assemble, bounds, check_optimality,
                               kkt_targets, ldl_solve, refp007_fixture)

LM = "limited-memory"
U = 2.0 ** -53


def bfgs_update(Wm, S, Y):
    """The device's update (csrc/dnlp_batch_qn.cuh) on full (count, n, n) matrices, sums in the same order.
    Returns the updated matrices and the mask of the starts it applies to (s'Ws > 0)."""
    c, n = S.shape
    Bs = np.zeros((c, n))
    for j in range(n):
        Bs = Bs + Wm[:, :, j] * S[:, j:j + 1]
    sBs, sy = np.zeros(c), np.zeros(c)
    for i in range(n):
        sBs = sBs + S[:, i] * Bs[:, i]
        sy = sy + S[:, i] * Y[:, i]
    with np.errstate(all="ignore"):
        ok = sBs > 0
        theta = np.where(sy >= 0.2 * sBs, 1.0, 0.8 * sBs / (sBs - sy))
        Rv = theta[:, None] * Y + (1.0 - theta)[:, None] * Bs
        sr = np.zeros(c)
        for i in range(n):
            sr = sr + S[:, i] * Rv[:, i]
        Wn = (Wm - (Bs[:, :, None] * Bs[:, None, :]) / sBs[:, None, None]) + \
            (Rv[:, :, None] * Rv[:, None, :]) / sr[:, None, None]
    return np.where(ok[:, None, None], Wn, Wm), ok


class NumpyQNKKT(NumpyKKT):
    """Quasi-Newton KKT backend of the CPU tests: the scatter map of the device's quasi-Newton mode (the packed lower
    triangle of W as the x-block's sources), W_b per start on the host, the NumPy factorisation of NumpyKKT."""
    quasi_newton = True

    def __init__(self, ev, quasi_newton=True):
        assert quasi_newton
        super().__init__(ev)
        self.W = None

    def setup(self, slack_rows):
        n = self.ev.n
        jr, jc = (np.asarray(a, dtype=np.int64) for a in self.ev.jacobianstructure())
        self.tril = np.tril_indices(n)                  # row-major: the packed order i(i+1)/2 + j
        self.ns = len(slack_rows)
        self.N, self.M = n + self.ns, n + self.ns + self.ev.m
        self.nnzH = self.tril[0].size
        self.targets = kkt_targets(n, self.ev.m, self.ns, list(slack_rows), jr, jc, *self.tril)
        self.W = None

    def load(self, X, LAM):
        if self.W is None:
            self.W = np.tile(np.eye(self.ev.n), (len(X), 1, 1))
        self.jac = self.ev.eval(X, want=("jac",))["jac"] if self.ev.m else np.zeros((len(X), 0))

    def matrix(self, b, sigma, dw, dc):
        return assemble(self.targets, self.N, self.M, self.nnzH, self.jac[b], self.W[b][self.tril], sigma, dw, dc)

    def update(self, starts, S, Y):
        starts = np.asarray(starts)
        Wn, ok = bfgs_update(self.W[starts], np.asarray(S, dtype=np.float64), np.asarray(Y, dtype=np.float64))
        self.W[starts] = Wn
        return ok


def run_lockstep_qn(prob, X0, **kw):
    ev = CpuBatch(prob)
    return lockstep_ipm(ev, NumpyQNKKT(ev), X0, **bounds(prob), hessian_approximation=LM, **kw)


def run_standin_qn(prob, x0):
    """The serial stand-in with hessian_approximation = limited-memory (its damped-BFGS branch)."""
    n, m = prob.n, prob.m
    b = {k: (None if v is None else np.where(np.isinf(v), np.sign(v) * 2e19, v)) for k, v in bounds(prob).items()}
    p = cyipopt_standin.Problem(n, m, problem_obj=_KeepPoints(prob), lb=b["lb"], ub=b["ub"], cl=b["cl"], cu=b["cu"])
    p.add_option("hessian_approximation", LM)
    return cyipopt_standin._BarrierSolver(p).run(np.asarray(x0, dtype=np.float64))


_cache = {}


def qn_result(name, max_iter=500):
    if (name, max_iter) not in _cache:
        prob, X0 = FIXTURES[name]()
        _cache[name, max_iter] = (prob, X0, run_lockstep_qn(prob, X0, max_iter=max_iter))
    return _cache[name, max_iter]


# ---- CPU tier ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,max_iter", [("qcqp16", 500), ("refp007", 60)])
def test_qn_lockstep_equals_start_by_start(name, max_iter):
    """B starts at once give bit-identical per-start results (x, lam, zL, zU, f, status, iterations) to the same
    driver run on each start alone: the BFGS matrices and their updates do not leak between starts."""
    prob, X0, out = qn_result(name, max_iter)
    for b in range(len(X0)):
        one = run_lockstep_qn(prob, X0[b:b + 1], max_iter=max_iter)
        assert one["status"][0] == out["status"][b] and one["iterations"][0] == out["iterations"][b], b
        for k in ("x", "lam", "zL", "zU"):
            assert np.array_equal(one[k][0], out[k][b]), (b, k)
        assert one["f"][0] == out["f"][b]


# Starts whose iteration count differs from the stand-in's (same status, objective and x), with (driver, stand-in)
# iterations.  In both the cause is the zero-pivot rule (csrc/dnlp_batch_kkt.cuh): late in the solve the stand-in's
# global threshold 1e-11 max(1, max|d|) reads small constraint-block pivots as zero and regularises, the driver's
# per-pivot rule keeps dw = 0 throughout.
# qcqp16 start 7: at iteration 30 the stand-in raises dw to 1.0 and meets the tolerance at 31; the driver at 32.
# twosided start 1: from iteration 28 the stand-in takes dw = 1e-2, 2.7e-2, 7.1e-2 and stops at 30; the driver at 31.
ITERATIONS_DIFFER = {("qcqp16", 7): (32, 31), ("twosided", 1): (31, 30)}


@pytest.mark.parametrize("name", ["qcqp16", "twosided"])
def test_qn_agrees_with_the_serial_standin(name):
    """Every start the stand-in solves with limited-memory, the driver solves, with the objective within 1e-8 relative
    and x within 1e-6, in the same number of iterations except for the starts in ITERATIONS_DIFFER.  Where the stand-in
    ends with -3 (its global zero-pivot threshold), the driver converges."""
    prob, X0, out = qn_result(name)
    for b in range(len(X0)):
        ref = run_standin_qn(prob, X0[b])
        if ref["status"] == -3:
            assert out["status"][b] == 0, b
            continue
        assert out["status"][b] == ref["status"], (b, out["status"][b], ref["status"])
        if (name, b) in ITERATIONS_DIFFER:
            assert (out["iterations"][b], ref["iterations"]) == ITERATIONS_DIFFER[name, b]
        else:
            assert out["iterations"][b] == ref["iterations"], (b, out["iterations"][b], ref["iterations"])
        if ref["status"] == 0:
            assert abs(out["f"][b] - ref["f"]) <= 1e-8 * max(1.0, abs(ref["f"])), b
            np.testing.assert_allclose(out["x"][b], ref["x"], rtol=0, atol=1e-6)


@pytest.mark.parametrize("name", ["qcqp16", "twosided"])
def test_qn_independent_optimality(name):
    prob, X0, out = qn_result(name)
    conv = np.flatnonzero(out["status"] == 0)
    assert conv.size > 0
    for b in conv:
        check_optimality(prob, out["x"][b], out["lam"][b], out["zL"][b], out["zU"][b], "%s start %d" % (name, b))


class _Recording(CpuBatch):
    def __init__(self, prob):
        super().__init__(prob)
        self.wanted = set()

    def eval(self, X, LAM=None, SIGMA=None, want=("f", "grad", "g", "jac", "hess")):
        self.wanted |= set(want)
        return super().eval(X, LAM, SIGMA, want)


def test_qn_never_asks_for_the_hessian(monkeypatch):
    def exact_load(self, X, LAM):
        raise AssertionError("the exact-Hessian load ran in quasi-Newton mode")
    monkeypatch.setattr(NumpyKKT, "load", exact_load)
    prob, X0 = FIXTURES["twosided"](4)
    ev = _Recording(prob)
    out = lockstep_ipm(ev, NumpyQNKKT(ev), X0, **bounds(prob), hessian_approximation=LM)
    assert "hess" not in ev.wanted and {"f", "grad", "g", "jac"} <= ev.wanted
    assert np.any(out["status"] == 0)


def test_qn_equality_only_problem_goes_through_the_ipm():
    """max x'Ax s.t. |x|^2 = 1 has no bound and no inequality row; with limited-memory best_of_lockstep still runs
    lockstep_ipm (the Newton-KKT iteration needs the Hessian) and every converged start is an eigenpair of A."""
    from dnlp_b200.best_of import best_of_lockstep
    prob = W.eigen_qcqp(8)
    A = W.eigen_qcqp_data(8)
    X0 = np.random.default_rng(2).standard_normal((6, 8))
    ev = CpuBatch(prob)
    out = best_of_lockstep(prob, X0, evaluator=ev, kkt=NumpyQNKKT(ev), hessian_approximation=LM)
    assert "status" in out
    conv = np.flatnonzero(out["status"] == 0)
    assert conv.size > 0
    for b in conv:
        x = out["x"][b]
        assert abs(x @ x - 1.0) <= 1e-8
        lam = x @ A @ x
        assert np.abs(A @ x - lam * x).max() <= 1e-6 * np.abs(A).max(), b


def test_unknown_hessian_approximation_is_a_value_error():
    from dnlp_b200.best_of import best_of_lockstep
    prob, X0 = FIXTURES["twosided"](2)
    ev = CpuBatch(prob)
    with pytest.raises(ValueError, match="'exact' or 'limited-memory'"):
        lockstep_ipm(ev, NumpyKKT(ev), X0, **bounds(prob), hessian_approximation="bfgs")
    with pytest.raises(ValueError, match="'exact' or 'limited-memory'"):
        best_of_lockstep(prob, X0, evaluator=ev, kkt=NumpyKKT(ev), hessian_approximation="bfgs")
    with pytest.raises(ValueError, match="quasi_newton"):          # a backend built for the other mode
        lockstep_ipm(ev, NumpyKKT(ev), X0, **bounds(prob), hessian_approximation=LM)


@pytest.mark.skipif(not R.available(), reason="reference not present (oracle/_ref)")
def test_solve_best_of_limited_memory():
    """solve_best_of forwards hessian_approximation through solver_opts: a value instead of TypeError, and
    all_objs_from_best_of equal to the serial stand-in with the same option run start by start on the reference's own
    sampler stream.  An unknown value raises ValueError."""
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
        p.add_option("hessian_approximation", LM)
        want.append(p.solve(data["x0"])[1]["obj_val"])
    x2, prob2 = build()
    np.random.seed(3)
    val = solve_best_of(prob2, N, evaluator_factory=lambda pir, B: CpuBatch(pir), kkt_factory=NumpyQNKKT,
                        hessian_approximation=LM)
    np.testing.assert_allclose(prob2.solver_stats.extra_stats["all_objs_from_best_of"], want, rtol=1e-8)
    assert abs(val - min(want)) <= 1e-8 * max(1.0, abs(min(want)))
    x3, prob3 = build()
    with pytest.raises(ValueError, match="'exact' or 'limited-memory'"):
        solve_best_of(prob3, 2, evaluator_factory=lambda pir, B: CpuBatch(pir), kkt_factory=NumpyQNKKT,
                      hessian_approximation="bfgs")


def test_qn_entry_points_reject_a_null_handle():
    from dnlp_b200 import _cabi, build
    build.build()
    L = _cabi.lib()
    i32 = np.zeros(4, dtype=np.int32)
    pi = i32.ctypes.data_as(_cabi.c_i32p)
    d = np.zeros(16)
    pd = d.ctypes.data_as(_cabi.c_f64p)
    ms = np.zeros(1, dtype=np.float32)
    assert L.dnlp_batch_kkt_setup_qn(None, 0, pi, pi, pi) != 0
    assert L.dnlp_batch_qn_update(None, 1, pi, pd, pd, pi, ms.ctypes.data_as(_cabi.c_f32p)) != 0
    assert L.dnlp_batch_qn_matrix(None, 0, pd) != 0
    assert b"NULL" in L.dnlp_batch_last_error(None)


# ---- GPU tier ----------------------------------------------------------------------------------------------
def _ld_update(Wm, s, y):
    """One start's update in long double with an absolute error magnitude per entry (first-order propagation of
    every rounding through the sums, the damping factor and the two divisions, in units of u)."""
    L = np.longdouble
    Wl, sl, yl = Wm.astype(L), s.astype(L), y.astype(L)
    aW, asl, ayl = np.abs(Wl), np.abs(sl), np.abs(yl)
    Bs = Wl @ sl
    eBs = aW @ asl                                        # |Bs_i| error / (n u)
    sBs, sy = sl @ Bs, sl @ yl
    esBs = asl @ (np.abs(Bs) + eBs)
    esy = asl @ ayl
    if not sBs > 0:
        return None, None
    if sy >= L(0.2) * sBs:
        theta, eth = L(1), L(0)
    else:
        theta = L(0.8) * sBs / (sBs - sy)
        eth = abs(theta) * (esBs / abs(sBs) + (esBs + esy) / abs(sBs - sy) + 4)
    r = theta * yl + (1 - theta) * Bs
    er = eth * (ayl + np.abs(Bs)) + abs(theta) * ayl + abs(1 - theta) * (np.abs(Bs) + eBs)
    sr = sl @ r
    esr = asl @ (np.abs(r) + er)
    T1 = np.outer(Bs, Bs) / sBs
    T2 = np.outer(r, r) / sr
    eT1 = (np.outer(eBs, np.abs(Bs)) + np.outer(np.abs(Bs), eBs)) / abs(sBs) + np.abs(T1) * (esBs / abs(sBs) + 2)
    eT2 = (np.outer(er, np.abs(r)) + np.outer(np.abs(r), er)) / abs(sr) + np.abs(T2) * (esr / abs(sr) + 2)
    return (Wl - T1) + T2, aW + np.abs(T1) + np.abs(T2) + eT1 + eT2


def _step_pair(Wm, kind, rng):
    """(s, y) for one start: 0 undamped (sy ~ 2 sBs), 1 damped with 0 < sy = 0.1 sBs, 2 damped with sy = -0.5 sBs,
    3 skipped (s = 0), 4 skipped (NaN in s)."""
    n = Wm.shape[0]
    s = rng.standard_normal(n)
    Ws = Wm @ s
    noise = rng.standard_normal(n)
    noise = noise - (noise @ s) / (s @ s) * s            # orthogonal to s (zero for n = 1)
    if kind == 0:
        y = 2.0 * Ws + 0.1 * rng.standard_normal(n) * np.abs(Ws).max()
        if s @ y < 0.5 * (s @ Ws):
            y = 2.0 * Ws
    elif kind == 1:
        y = 0.1 * Ws + 0.3 * noise * np.abs(Ws).max() / max(np.abs(noise).max(), 1e-300)
    elif kind == 2:
        y = -0.5 * Ws + 0.3 * noise * np.abs(Ws).max() / max(np.abs(noise).max(), 1e-300)
    elif kind == 3:
        s, y = np.zeros(n), rng.standard_normal(n)
    else:
        s[rng.integers(n)] = np.nan
        y = rng.standard_normal(n)
    return s, y


def _qn_handle(n, B):
    from dnlp_b200.multistart import BatchedOracles
    P, q, _ = W.qcqp_data(n, 1, seed=n)
    ev = BatchedOracles(W.qcqp(P, q), B)
    ev.kkt_setup(np.array([0]), quasi_newton=True)
    return ev


QN_UPDATE_CASES = [(1, 1), (2, 7), (31, 64), (32, 300), (33, 7), (63, 1), (64, 64), (65, 300), (127, 7), (128, 64),
                   (129, 300), (512, 64), (512, 7)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,B", QN_UPDATE_CASES, ids=["n%d_B%d" % c for c in QN_UPDATE_CASES])
def test_gpu_qn_update_against_long_double(n, B):
    """Five successive rounds on a non-contiguous subset of the starts; each round gives every selected start an
    undamped, a damped (0 <= sy < 0.2 sBs or sy < 0) or a skipped (s = 0, NaN in s) update in turn.  Each updated W_b
    is within 8 (n + 4) u of its long-double magnitude of the update applied to the device's previous W_b, entry by
    entry; W_b is bitwise symmetric; skipped and unselected starts are bitwise unchanged and skipped starts report
    applied = 0.  A second handle that updates one start alone ends bit-identical to it."""
    rng = np.random.default_rng(1000 * n + B)
    sel = np.sort(rng.permutation(B)[:max(1, (2 * B) // 3)])[::-1].copy() if B > 1 else np.array([0])
    if B > 2:
        sel = sel[sel != sel[len(sel) // 2]]                  # a hole in the middle
    alone = int(sel[0])
    ev = _qn_handle(n, B)
    ev1 = _qn_handle(n, B)
    try:
        prev = {b: ev.qn_matrix(b) for b in range(B)}
        for b in range(B):
            assert np.array_equal(prev[b], np.eye(n)), b
        for rnd in range(5):
            pairs = [_step_pair(prev[b], (b + rnd) % 5, rng) for b in sel]
            S = np.array([p[0] for p in pairs]).reshape(len(sel), n)
            Y = np.array([p[1] for p in pairs]).reshape(len(sel), n)
            applied = ev.qn_update(sel, S, Y)
            c1 = int(np.flatnonzero(sel == alone)[0])
            ev1.qn_update([alone], S[c1:c1 + 1], Y[c1:c1 + 1])
            assert ev.qn_ms >= 0.0
            for c, b in enumerate(sel):
                Wd = ev.qn_matrix(b)
                assert np.array_equal(Wd, Wd.T), (rnd, b)
                ref, mag = _ld_update(prev[b], S[c], Y[c])
                if ref is None:
                    assert not applied[c], (rnd, b)
                    assert np.array_equal(Wd, prev[b]), (rnd, b)
                else:
                    assert applied[c], (rnd, b)
                    err = np.abs(Wd.astype(np.longdouble) - ref)
                    bound = 8 * (n + 4) * U * mag
                    assert np.all(err <= bound), (rnd, b, float(np.max(err / bound)))
                prev[b] = Wd
            for b in set(range(B)) - set(sel.tolist()):
                assert np.array_equal(ev.qn_matrix(b), np.eye(n)), (rnd, b)
            assert np.array_equal(ev1.qn_matrix(alone), prev[alone]), rnd
    finally:
        ev.close()
        ev1.close()


def _qn_assembly_case(prob, B, starts, seed):
    """K in quasi-Newton mode against the NumPy scatter of qn_matrix(b) and the device's JAC, bit for bit; inertia,
    solution and dz'W dz against ldl_solve."""
    from dnlp_b200.multistart import BatchedOracles
    rng = np.random.default_rng(seed)
    ev = BatchedOracles(prob, B)
    try:
        cl = np.full(prob.m, -np.inf) if prob.cl is None else prob.cl
        cu = np.full(prob.m, np.inf) if prob.cu is None else prob.cu
        slack = np.flatnonzero(cl != cu)
        ev.kkt_setup(slack, quasi_newton=True)
        n = prob.n
        for rnd in range(3):                                  # W away from I: three undamped or damped updates
            sub = np.sort(rng.permutation(B)[:max(1, B // 2)])
            S = rng.standard_normal((sub.size, n))
            Y = S * rng.uniform(-0.5, 3.0, (sub.size, 1)) + 0.3 * rng.standard_normal((sub.size, n))
            ev.qn_update(sub, S, Y)
        X = rng.uniform(-1, 1, (B, n))
        LAM = 3.0 * rng.standard_normal((B, prob.m))
        ev.upload(X, LAM, np.ones(B))
        ev.run_device(("jac",))
        N, M = n + slack.size, n + slack.size + prob.m
        sigma = 10.0 ** rng.uniform(-8, 8, (len(starts), N))
        dw = np.where(rng.uniform(size=len(starts)) < 0.5, 0.0, 10.0 ** rng.uniform(-4, 2, len(starts)))
        dc = 10.0 ** rng.uniform(-9, -6, len(starts))
        rhs = rng.standard_normal((len(starts), M))
        sol, inert, wq = ev.kkt_solve(starts, sigma, dw, dc, rhs)
        jr, jc = (np.asarray(a, dtype=np.int64) for a in ev.jacobianstructure())
        tril = np.tril_indices(n)
        targets = kkt_targets(n, prob.m, slack.size, list(slack), jr, jc, *tril)
        jac = ev.read_output("jac")
        ok = 0
        for c, b in enumerate(starts):
            Wb = ev.qn_matrix(b)
            Kd = ev.kkt_matrix(b)
            Kh, Wdh = assemble(targets, N, M, tril[0].size, jac[b], Wb[tril], sigma[c], dw[c], dc[c])
            assert np.array_equal(Kd, Kh), "start %d: assembled K differs from the host scatter" % b
            s_ref, i_ref, w_ref = ldl_solve(Kh, Wdh, N, rhs[c])
            assert tuple(inert[c]) == tuple(i_ref), (b, inert[c], i_ref)
            if np.isfinite(s_ref).all():
                ok += 1
                assert np.isfinite(sol[c]).all(), b
                np.testing.assert_allclose(sol[c], s_ref, rtol=1e-10, atol=1e-10 * np.abs(s_ref).max())
                dz = s_ref[:N]
                Wm = np.abs(Kh[:N, :N])
                Wm[np.diag_indices(N)] = np.abs(Wdh)
                assert abs(wq[c] - w_ref) <= 1e-10 * (np.abs(dz) @ Wm @ np.abs(dz)), b
            else:
                assert not np.isfinite(sol[c]).any(), b
        return ok
    finally:
        ev.close()


QN_KKT_SHAPES = [(29, 1), (30, 1), (31, 1), (62, 1), (63, 1)]       # (n, k): M = n + 2k = 31, 32, 33, 64, 65


@pytest.mark.gpu
@pytest.mark.parametrize("n,k", QN_KKT_SHAPES, ids=["M%d" % (n + 2 * k) for n, k in QN_KKT_SHAPES])
def test_gpu_qn_kkt_assembly_and_solve(n, k):
    P, q, _ = W.qcqp_data(n, k, seed=n)
    _qn_assembly_case(W.qcqp(P, q), 16, np.array([15, 0, 3, 4, 9, 7, 12]), seed=n)


@pytest.mark.gpu
def test_gpu_qn_kkt_refp007():
    prob, _ = refp007_fixture()
    _qn_assembly_case(prob, 64, np.random.default_rng(11).permutation(64)[:40], seed=1)


@pytest.mark.gpu
def test_gpu_qn_kkt_c4_shape():
    """N + m = 528: the C4 QCQP (n = 512, k = 8 slack rows), B = 64, a non-contiguous subset of starts."""
    P, q, _ = W.qcqp_data(512, 8)
    _qn_assembly_case(W.qcqp(P, q), 64, np.array([63, 0, 5, 17, 18, 40, 2, 33, 9, 50]), seed=2)


def _hess_only_instrs(tape):
    others = set()
    for name in ("f", "grad", "g", "jac"):
        others |= set(np.asarray(tape.programs.get(name, []), dtype=np.int64).tolist())
    return sorted(set(np.asarray(tape.programs["hess"], dtype=np.int64).tolist()) - others)


@pytest.mark.gpu
def test_gpu_qn_never_runs_the_hess_program():
    """After a quasi-Newton solve of qcqp16 on a fresh handle no instruction that belongs only to the HESS program has
    run; after an exact solve on another fresh handle they all have."""
    from dnlp_b200.lockstep_ipm import DeviceKKT
    from dnlp_b200.multistart import BatchedOracles
    prob, X0 = FIXTURES["qcqp16"]()
    names = {}
    for mode in ("exact", LM):
        ev = BatchedOracles(prob, len(X0))
        try:
            hess_only = _hess_only_instrs(ev.tape)
            assert hess_only
            out = lockstep_ipm(ev, DeviceKKT(ev, quasi_newton=mode == LM), X0, **bounds(prob),
                               hessian_approximation=mode)
            assert np.any(out["status"] == 0)
            names[mode] = [ev.instr_kernel(i) for i in hess_only]
        finally:
            ev.close()
    assert all(nm != "" for nm in names["exact"]), names["exact"]
    assert all(nm == "" for nm in names[LM]), names[LM]


@pytest.mark.gpu
def test_gpu_qn_end_to_end_qcqp64():
    """The QCQP n = 64, k = 4, B = 256 in quasi-Newton mode on the device against the CPU lock-step driver (NumPy
    quasi-Newton backend) on every 8th start: same status, objective within 1e-8, optimality of every converged
    start."""
    from dnlp_b200.lockstep_ipm import DeviceKKT
    from dnlp_b200.multistart import BatchedOracles
    P, q, rng = W.qcqp_data(64, 4)
    prob = W.qcqp(P, q)
    X0 = rng.uniform(-1, 1, (256, 64))
    ev = BatchedOracles(prob, len(X0))
    try:
        kkt = DeviceKKT(ev, quasi_newton=True)
        out = lockstep_ipm(ev, kkt, X0, **bounds(prob), hessian_approximation=LM)
    finally:
        ev.close()
    assert kkt.qn_calls > 0 and kkt.qn_ms > 0.0
    check = np.arange(0, 256, 8)
    cpu = run_lockstep_qn(prob, X0[check])
    assert np.array_equal(out["status"][check], cpu["status"])
    both = cpu["status"] == 0
    fo, fc = out["f"][check][both], cpu["f"][both]
    assert np.all(np.abs(fo - fc) <= 1e-8 * np.maximum(1.0, np.abs(fc)))
    conv = np.flatnonzero(out["status"] == 0)
    assert conv.size > 0
    for b in conv:
        check_optimality(prob, out["x"][b], out["lam"][b], out["zL"][b], out["zU"][b], "start %d" % b)


@pytest.mark.gpu
def test_gpu_qn_setup_refuses_what_does_not_fit():
    """sum x^2 with n = 2048, m = 0 (bounds only), 16384 starts: the dense systems need 16384 * 2048^2 * 8 = 550 GB and
    the quasi-Newton matrices 16384 * 2098176 * 8 = 275 GB.  kkt_setup raises naming both terms and keeps nothing
    (qn_update and kkt_solve then ask for the setup); a small batch of the same problem then sets up with W = I, takes
    an update with a closed-form result and solves its diagonal systems."""
    from dnlp_b200 import ir
    from dnlp_b200.multistart import BatchedOracles
    n = 2048
    x = ir.Variable(n)
    prob = ir.ProblemIR(ir.sum(ir.power(x, 2)), [], [x], lb=-np.ones(n), ub=np.ones(n), x0=np.zeros(n))
    ev = BatchedOracles(prob, 16384)
    try:
        with pytest.raises(RuntimeError, match=r"B\*\(N\+m\)\^2\*8 = 16384\*2048\^2\*8 = .* "
                                               r"B\*n\(n\+1\)/2\*8 = 16384\*2098176\*8"):
            ev.kkt_setup(np.zeros(0, dtype=np.int32), quasi_newton=True)
        with pytest.raises(RuntimeError, match="kkt_setup_qn first"):
            ev.qn_update([0], np.ones((1, n)), np.ones((1, n)))
        ev.kkt_N = n
        with pytest.raises(RuntimeError, match="kkt_setup first"):
            ev.kkt_solve([0], np.ones((1, n)), [0.0], [0.0], np.ones((1, n)))
    finally:
        ev.close()
    ev = BatchedOracles(prob, 2)
    try:
        ev.kkt_setup(np.zeros(0, dtype=np.int32), quasi_newton=True)
        e0 = np.zeros((1, n))
        e0[0, 0] = 1.0
        # s = e0, y = 2 e0: Bs = e0, s'Bs = 1, s'y = 2 (undamped), r = y, s'r = 2: W_00 = (1 - 1) + 4 / 2 = 2
        assert ev.qn_update([1], e0, 2.0 * e0).tolist() == [True]
        W1 = np.eye(n)
        W1[0, 0] = 2.0
        assert np.array_equal(ev.qn_matrix(1), W1)
        assert np.array_equal(ev.qn_matrix(0), np.eye(n))
        rng = np.random.default_rng(1)
        sigma, rhs = rng.uniform(0.1, 1.0, (2, n)), rng.standard_normal((2, n))
        sol, inert, wq = ev.kkt_solve([1, 0], sigma[::-1], [1e-3, 0.0], [0.0, 0.0], rhs[::-1])
        for c, b in enumerate([1, 0]):
            d = (np.diag(W1 if b == 1 else np.eye(n)) + sigma[b]) + (1e-3 if c == 0 else 0.0)
            assert tuple(inert[c]) == (n, 0, 0)
            np.testing.assert_allclose(sol[c], rhs[b] / d, rtol=4 * U, atol=0)
    finally:
        ev.close()
