"""The batched engine (csrc/dnlp_batch*.cu) at the edges of its blocked kernels, against closed forms.

A QCQP  min x'P0x + q0'x  s.t.  g_i = 1 - x'P_i x - q_i'x >= 0 (or = 0)  has closed forms for all five oracle outputs
and for the KKT matrix of the lock-step interior-point driver.  They are computed here in np.longdouble from P and q
alone, so they share no code with the device kernels, with the oracle port or with the NumPy LDL' of
test_lockstep_ipm.py.  Every entry comes with its componentwise magnitude (the sum of the absolute values of the terms
it sums), and the tolerances are multiples of that magnitude times the unit roundoff.

CPU tier: the closed forms equal RefOracles and the device scatter map of test_lockstep_ipm.py, so a wrong closed form
fails before any GPU run.
GPU tier:
- KKT: assembly, LDL' (32-wide panels, 64 x 64 trailing tiles, 32-row solve blocks) and solve at sizes around every
  block edge, with m = 0, with constraint blocks that straddle a panel, and with indefinite, singular, zero-pivot and
  NaN-poisoned systems next to good ones; the refusal of a batch whose systems do not fit.
- Oracle dispatch: every variant `dnlp_batch::launch` picks (bsmallk<L, NB>, the three long-row kernels, bpoly, the
  DMMA GEMM), named by the engine itself (BatchedOracles.instr_kernel), checked entry by entry."""
import numpy as np
import pytest
import scipy.linalg as sla

from dnlp_b200 import tape as T
from dnlp_b200 import workloads as W
from oracle.dnlp_oracle import RefOracles
from test_lockstep_ipm import _device_vs_numpy, assemble, kkt_targets

LD = np.longdouble
U = 2.0 ** -53                 # unit roundoff of float64
C_ORACLE = 2                   # see within_bound


# ---- the problems ----------------------------------------------------------------------------------------------
def qcqp_case(n, k_in, k_eq, seed=0, P=None, q=None):
    """W.qcqp with k_eq equality rows (cu = cl = 0) FIRST and k_in inequality rows after them, so that slack s belongs
    to constraint row k_eq + s, not to row s.  Returns (prob, P, q, slack_rows)."""
    if P is None:
        P, q, _ = W.qcqp_data(n, k_in + k_eq, seed=seed)
    prob = W.qcqp(P, q)
    cu = np.full(k_in + k_eq, np.inf)
    cu[:k_eq] = 0.0
    prob.cu = cu
    return prob, P, q, np.arange(k_eq, k_eq + k_in)


class ClosedForm:
    """f, grad, g, J, H and K of a QCQP in long double, each with its componentwise magnitude."""

    def __init__(self, P, q, hess_pattern, jac_pattern):
        self.P = np.array(P, dtype=LD)                 # (k + 1, n, n)
        self.q = np.array(q, dtype=LD)                 # (k + 1, n)
        self.k, self.n = self.P.shape[0] - 1, self.P.shape[1]
        self.hr, self.hc = (np.asarray(a, dtype=np.int64) for a in hess_pattern)
        self.jr, self.jc = (np.asarray(a, dtype=np.int64) for a in jac_pattern)

    def oracles(self, X, LAM, SIGMA):
        """{name: (value, magnitude)}, each (B, len), for the points X (B, n), multipliers LAM (B, k), factors SIGMA."""
        X, LAM, S = np.asarray(X, LD), np.asarray(LAM, LD).reshape(len(X), self.k), np.asarray(SIGMA, LD)
        aX, aP, aq = np.abs(X), np.abs(self.P), np.abs(self.q)
        Y = np.einsum("inj,bj->ibn", self.P, X)        # Y[i, b] = P_i x_b
        aY = np.einsum("inj,bj->ibn", aP, aX)
        f = np.sum(X * Y[0], axis=1) + X @ self.q[0]
        fm = np.sum(aX * aY[0], axis=1) + aX @ aq[0]
        grad, gradm = 2 * Y[0] + self.q[0], 2 * aY[0] + aq[0]
        g = 1 - np.einsum("bn,ibn->bi", X, Y[1:]) - X @ self.q[1:].T
        gm = 1 + np.einsum("bn,ibn->bi", aX, aY[1:]) + aX @ aq[1:].T
        i, c = self.jr + 1, self.jc
        jac, jacm = -(2 * Y[i, :, c] + self.q[i, c][:, None]).T, (2 * aY[i, :, c] + aq[i, c][:, None]).T
        Ph, aPh = self.P[:, self.hr, self.hc], aP[:, self.hr, self.hc]              # (k + 1, nnzH)
        hess = 2 * (S[:, None] * Ph[0] - LAM @ Ph[1:])
        hessm = 2 * (np.abs(S)[:, None] * aPh[0] + np.abs(LAM) @ aPh[1:])
        return {"f": (f, fm), "grad": (grad, gradm), "g": (g, gm), "jac": (jac, jacm), "hess": (hess, hessm)}

    # the number of rounded operations an output entry goes through on the device (a sum of T products is
    # within T u of its magnitude): f and g are x'(P x) + q'x (n + 2n terms), grad and J one row of P x plus q
    TERMS = {"f": lambda n, k: 3 * n + 2, "grad": lambda n, k: n + 2, "g": lambda n, k: 3 * n + 3,
             "jac": lambda n, k: n + 2, "hess": lambda n, k: k + 2}

    def hessian_matrix(self, x, lam, sigma):
        """The dense W_xx = 2 (sigma P0 - sum lam_i P_i) and its magnitude, (n, n)."""
        lam = np.asarray(lam, LD)
        W_ = 2 * (LD(sigma) * self.P[0] - np.tensordot(lam, self.P[1:], 1))
        Wm = 2 * (abs(LD(sigma)) * np.abs(self.P[0]) + np.tensordot(np.abs(lam), np.abs(self.P[1:]), 1))
        return W_, Wm

    def kkt(self, x, lam, sigma_obj, slack_rows, sigma, dw, dc):
        """K = [[W + diag(Sigma) + dw I, A'], [A, -dc I]], A = [J, -P_slack] in z = (x, slacks), built directly from
        P and q, with its magnitude; (M, M) long double."""
        n, m, ns = self.n, self.k, len(slack_rows)
        N, M = n + ns, n + ns + m
        x = np.asarray(x, LD)
        W_, Wm = self.hessian_matrix(x, lam, sigma_obj)
        Px = np.einsum("inj,j->in", self.P[1:], x)
        J = -(2 * Px + self.q[1:])
        Jm = 2 * np.einsum("inj,j->in", np.abs(self.P[1:]), np.abs(x)) + np.abs(self.q[1:])
        K, Km = np.zeros((M, M), LD), np.zeros((M, M), LD)
        K[:n, :n], Km[:n, :n] = W_, Wm
        d = np.arange(N)
        K[d, d] += np.asarray(sigma, LD) + LD(dw)
        Km[d, d] += np.abs(np.asarray(sigma, LD)) + abs(LD(dw))
        A, Am = np.zeros((m, N), LD), np.zeros((m, N), LD)
        A[:, :n], Am[:, :n] = J, Jm
        for s, r in enumerate(slack_rows):
            A[r, n + s], Am[r, n + s] = -1, 1
        K[N:, :N], K[:N, N:], Km[N:, :N], Km[:N, N:] = A, A.T, Am, Am.T
        K[N + np.arange(m), N + np.arange(m)] = -LD(dc)
        Km[N + np.arange(m), N + np.arange(m)] = abs(LD(dc))
        return K, Km


def closed_form(prob, P, q):
    r = RefOracles(prob)
    return ClosedForm(P, q, r.hessianstructure(), r.jacobianstructure())


def within_bound(got, ref, mag, terms, what):
    """|got - ref| <= C_ORACLE * terms * u * magnitude, componentwise (a NaN fails).  terms * u * magnitude bounds
    the rounding error of a sum of `terms` rounded products; C_ORACLE = 2 covers the products rounded before they
    are summed (x_i times a rounded (P x)_i) and the final store."""
    got = np.asarray(got, dtype=np.float64)
    err = np.abs(got.astype(LD) - ref)
    bound = C_ORACLE * terms * U * mag
    bad = ~(err <= bound)
    if bad.any():
        idx = np.argwhere(bad)[:5]
        pts = ["%s: got %.17g want %.17g bound %.3g" % (tuple(i), got[tuple(i)], float(ref[tuple(i)]),
                                                         float(bound[tuple(i)])) for i in idx]
        raise AssertionError("%s: %d of %d entries off; %s" % (what, bad.sum(), bad.size, "; ".join(pts)))


# ---- KKT shapes: (n, inequality rows, equality rows) -> M = n + 2 k_in + k_eq -----------------------------------------
KKT_SHAPES = [
    (1, 0, 0),       # M = 1, m = 0
    (1, 1, 0),       # M = 3
    (29, 1, 0),      # M = 31
    (30, 1, 0),      # M = 32: one full panel
    (32, 0, 1),      # M = 33: the x block is exactly one panel, the constraint row opens the next
    (61, 1, 0),      # M = 63
    (64, 0, 0),      # M = 64: bounds only, one full trailing tile
    (64, 0, 1),      # M = 65: N = 64, the constraint block starts a new panel and a new tile
    (62, 2, 3),      # M = 69: N = 64 with two slack columns, five constraint rows from row 64
    (28, 2, 3),      # M = 35: the constraint block (rows 30..34) straddles row 32
    (30, 3, 2),      # M = 38: the slack columns (30..32) straddle row 32
    (90, 3, 0),      # M = 96
    (95, 0, 2),      # M = 97
    (120, 4, 0),     # M = 128
    (127, 1, 0),     # M = 129
    (250, 3, 0),     # M = 256
    (255, 0, 2),     # M = 257
]
KKT_M_REQUIRED = {1, 3, 31, 32, 33, 63, 64, 65, 96, 97, 128, 129, 256, 257}


def shape_M(s):
    n, ki, ke = s
    return n + 2 * ki + ke


def shape_id(s):
    return "n%d_in%d_eq%d_M%d" % (s + (shape_M(s),))


# ---- oracle dispatch cases: (n, k, B, {role: kernel}) on a 148-SM B200 ---------------------------------------------
# role: the instructions writing output f / grad / g / jac / hess, or "gemm" (the dense P_i x maps).  The gradient and
# Jacobian rows (two terms each) always run bpoly_kernel<0>.
DISPATCH = [
    (1, 0, 7, {"gemm": "bgemm_dmma_kernel<0>", "f": "bpoly_kernel<1>", "hess": "bpoly_kernel<0>"}),   # a lone GEMV, K = 1
    (1, 2, 8, {"gemm": "bgemm_dmma_kernel<0>", "f": "bpoly_kernel<1>", "g": "bpoly_kernel<1>"}),
    (13, 3, 31, {"gemm": "bgemm_dmma_kernel<0>", "f": "bpoly_kernel<1>", "hess": "bpoly_kernel<0>"}),  # K < 16, odd
    (45, 1, 100, {"gemm": "bgemm_dmma_kernel<0>", "hess": "bsmallk_kernel<2, 1>"}),     # 1035 Hessian rows (odd)
    (45, 2, 300, {"hess": "bsmallk_kernel<3, 2>", "g": "bpoly_kernel<1>"}),
    (45, 8, 333, {"hess": "bsmallk_kernel<9, 2>"}),
    (45, 15, 777, {"gemm": "bgemm_dmma_kernel<0>", "hess": "bsmallk_kernel<16, 4>"}),
    (64, 2, 63, {"gemm": "bgemm_dmma_kernel<0>", "f": "bpoly_long_split_kernel<1, 8>", "hess": "bsmallk_kernel<3, 1>"}),
    (64, 8, 512, {"f": "bpoly_long_split_kernel<1, 8>", "g": "bpoly_long_split_kernel<1, 8>",
                  "hess": "bsmallk_kernel<9, 2>"}),
    (64, 8, 1024, {"g": "bpoly_long_kernel<1, 16>", "hess": "bsmallk_kernel<9, 4>"}),
    (64, 8, 2048, {"g": "bpoly_long_kernel<1, 8>", "hess": "bsmallk_kernel<9, 4>"}),
    # the bench's per-GPU slices of C4 (8 and 4 GPUs), checked on every 37th start
    (512, 8, 512, {"g": "bpoly_long_split_kernel<1, 8>", "hess": "bsmallk_kernel<9, 2>"}),
    (512, 8, 1024, {"g": "bpoly_long_kernel<1, 16>", "hess": "bsmallk_kernel<9, 4>"}),
]
REQUIRED_VARIANTS = {"bsmallk_kernel<2, 1>", "bsmallk_kernel<3, 2>", "bsmallk_kernel<9, 2>", "bsmallk_kernel<16, 4>",
                     "bpoly_long_split_kernel<1, 8>", "bpoly_long_kernel<1, 16>", "bpoly_long_kernel<1, 8>",
                     "bpoly_kernel<0>", "bpoly_kernel<1>", "bgemm_dmma_kernel<0>"}
_ROLE = {1: "f", 2: "grad", 3: "g", 4: "jac", 5: "hess"}


def dispatch_id(c):
    return "n%d_k%d_B%d" % c[:3]


def oracle_inputs(n, k, B, seed):
    rng = np.random.default_rng(seed)
    return rng.uniform(-1, 1, (B, n)), rng.standard_normal((B, k)), rng.uniform(0.5, 2.0, B)


# ---- CPU tier ----------------------------------------------------------------------------------------------------
def test_shape_tables_hit_the_block_edges():
    assert KKT_M_REQUIRED <= {shape_M(s) for s in KKT_SHAPES}
    assert any(n + ki == 64 and ki + ke > 0 for n, ki, ke in KKT_SHAPES)           # N = 64, constraint block at row 64
    assert any(n + ki < 32 < shape_M((n, ki, ke)) - 1 for n, ki, ke in KKT_SHAPES)  # constraint block straddles 32
    seen = {name for *_, want in DISPATCH for name in want.values()} | {"bpoly_kernel<0>"}
    assert REQUIRED_VARIANTS <= seen


_CPU_SHAPES = sorted({(n, ki, ke) for n, ki, ke in KKT_SHAPES} | {(n, k, 0) for n, k, _, _ in DISPATCH})


@pytest.mark.parametrize("shape", _CPU_SHAPES, ids=shape_id)
def test_closed_form_equals_reforacles(shape):
    """The closed-form f, grad, g, J, H (in RefOracles' pattern order) equal the oracle port to 1e-12 of their
    magnitude, with the equality rows (cu = 0) in place."""
    n, ki, ke = shape
    prob, P, q, _ = qcqp_case(n, ki, ke)
    cf, r = closed_form(prob, P, q), RefOracles(prob)
    r.hessianstructure()                # (the port returns the pattern's entries once it has been asked for it)
    X, LAM, S = oracle_inputs(n, ki + ke, 1 if n > 200 else 2, seed=n)
    got = cf.oracles(X, LAM, S)
    for b in range(len(X)):
        m = ki + ke                     # (the port has no constraint callbacks for m = 0)
        ref = {"f": np.array([r.objective(X[b])]), "grad": r.gradient(X[b]),
               "g": r.constraints(X[b]) if m else np.zeros(0), "jac": r.jacobian(X[b]) if m else np.zeros(0),
               "hess": r.hessian(X[b], LAM[b], S[b])}
        for name, (v, mag) in got.items():
            want = np.asarray(ref[name], dtype=np.float64).ravel()
            assert want.size == v[b].size, name
            err = np.abs(want.astype(LD) - v[b])
            assert np.all(err <= 1e-12 * mag[b]), (name, b, float(np.max(err / np.maximum(mag[b], 1e-300))))


@pytest.mark.parametrize("shape", [s for s in KKT_SHAPES if shape_M(s) <= 129], ids=shape_id)
def test_direct_kkt_equals_the_scatter_map(shape):
    """K built directly from P and q equals assemble() (the device's scatter map replayed on the host) fed the
    closed-form J and H: the map, the -1 of the slack columns and the diagonal terms agree."""
    n, ki, ke = shape
    prob, P, q, slack = qcqp_case(n, ki, ke)
    cf = closed_form(prob, P, q)
    m, N = ki + ke, n + ki
    rng = np.random.default_rng(n + 7)
    X, LAM, S = oracle_inputs(n, m, 1, seed=n)
    o = cf.oracles(X, LAM, S)
    sigma, dw, dc = rng.uniform(0.1, 2.0, N), 1e-3, 1e-2
    targets = kkt_targets(n, m, len(slack), list(slack), cf.jr, cf.jc, cf.hr, cf.hc)
    Ka, _ = assemble(targets, N, N + m, len(cf.hr), o["jac"][0][0].astype(np.float64),
                     o["hess"][0][0].astype(np.float64), sigma, dw, dc)
    K, Km = cf.kkt(X[0], LAM[0], S[0], slack, sigma, dw, dc)
    assert np.all(np.abs(Ka.astype(LD) - K) <= 4 * U * Km)
    assert np.array_equal(Ka != 0, K != 0)


# ---- GPU tier: KKT -------------------------------------------------------------------------------------------------
B_KKT = 8
C_BACKWARD = 4


def _kkt_params(cf, X, LAM, S, slack, rng, quasi_definite=True):
    """Per start: Sigma, dw, dc.  Quasi-definite: Sigma_x lifts W_xx + diag(Sigma_x) above 0.1 (eigenvalues of the
    closed-form W_xx), Sigma_slack > 0, dc > 0."""
    n, ns, m = cf.n, len(slack), cf.k
    B = len(X)
    sigma = np.empty((B, n + ns))
    for b in range(B):
        W_, _ = cf.hessian_matrix(X[b], LAM[b], S[b])
        shift = max(0.0, -float(np.linalg.eigvalsh(W_.astype(np.float64))[0])) if n else 0.0
        sigma[b, :n] = shift + rng.uniform(0.1, 1.0, n)
        sigma[b, n:] = rng.uniform(0.1, 1.0, ns)
    dw = np.where(np.arange(B) % 2 == 0, 0.0, 1e-3)
    dc = 10.0 ** rng.uniform(-4, -1, B)
    rhs = rng.standard_normal((B, n + ns + m))
    return sigma, dw, dc, rhs


class KktRun:
    """A BatchedOracles of B_KKT starts with the KKT systems set up, the oracles evaluated at (X, LAM, S)."""

    def __init__(self, prob, slack, X, LAM, S):
        from dnlp_b200.multistart import BatchedOracles
        self.ev = BatchedOracles(prob, len(X))
        self.ev.kkt_setup(slack)
        self.load(X, LAM, S)

    def load(self, X, LAM, S):
        self.ev.upload(X, LAM, S)
        self.ev.run_device(("jac", "hess"))

    def solve(self, starts, sigma, dw, dc, rhs):
        st = np.asarray(starts)
        return self.ev.kkt_solve(st, sigma[st], dw[st], dc[st], rhs[st])

    def close(self):
        self.ev.close()


def _inertia_by_eigenvalues(K):
    ev = np.linalg.eigvalsh(K)
    tol = 1e-13 * np.abs(ev).max(initial=0.0)
    return int(np.sum(ev > tol)), int(np.sum(ev < -tol)), int(np.sum(np.abs(ev) <= tol))


def _check_quasi_definite(cf, X, LAM, S, slack, K_dev, sol, inert, wq, sigma, dw, dc, rhs, what):
    n, m = cf.n, cf.k
    N, M = n + len(slack), n + len(slack) + m
    K, Km = cf.kkt(X, LAM, S, slack, sigma, dw, dc)
    # the assembled K is the closed-form K (oracle rounding only)
    terms = n + m + 4
    within_bound(K_dev, K, Km, terms, what + ": assembled K")
    assert tuple(inert) == _inertia_by_eigenvalues(K_dev) == (N, m, 0), (what, tuple(inert))
    assert np.all(np.isfinite(sol)) and np.isfinite(wq), what
    # normwise backward error in long double against the assembled K.  One step of refinement in working precision
    # leaves a residual of at most about (M + 1) u (|K| |x| + |b|) (Higham, Accuracy and Stability of Numerical
    # Algorithms, 2nd ed., Thm. 12.3); C_BACKWARD = 4 leaves a factor of two for the 1 / (1 - O(M u)) terms.
    Kl, xl, bl = K_dev.astype(LD), sol.astype(LD), rhs.astype(LD)
    r = np.abs(bl - Kl @ xl).max()
    eta = r / (np.abs(Kl).sum(axis=1).max() * np.abs(xl).max() + np.abs(bl).max())
    assert eta <= C_BACKWARD * M * U, "%s: backward error %.3e > %.3e" % (what, float(eta), C_BACKWARD * M * U)
    xs = sla.solve(K_dev, rhs)
    cond = np.linalg.cond(K_dev)
    assert np.abs(sol - xs).max() <= cond * 1e-15 * np.abs(xs).max(), (what, cond)
    # dz' W dz with the closed-form W (zero on the slack block)
    W_, Wm = cf.hessian_matrix(X, LAM, S)
    dz = sol[:n].astype(LD)
    want, mag = dz @ W_ @ dz, np.abs(dz) @ Wm @ np.abs(dz)
    assert abs(LD(wq) - want) <= C_ORACLE * (N + m + 4) * U * mag, (what, wq, float(want))


def _assert_nan(sol, wq, what):
    assert np.all(np.isnan(sol)) and np.isnan(wq), what


def _kkt_setup_case(shape, seed=0, P=None, q=None):
    n, ki, ke = shape
    prob, P, q, slack = qcqp_case(n, ki, ke, seed=seed, P=P, q=q)
    cf = closed_form(prob, P, q)
    rng = np.random.default_rng(1000 + shape_M(shape))
    X, LAM, S = oracle_inputs(n, ki + ke, B_KKT, seed=shape_M(shape))
    sigma, dw, dc, rhs = _kkt_params(cf, X, LAM, S, slack, rng)
    return prob, cf, slack, X, LAM, S, sigma, dw, dc, rhs


@pytest.mark.gpu
@pytest.mark.parametrize("shape", KKT_SHAPES, ids=shape_id)
def test_gpu_kkt_quasi_definite_edges(shape):
    """Quasi-definite systems (LDL' without pivoting is stable on them) at every block edge: the assembled K against
    the closed form, the inertia against eigenvalues, the backward error, scipy's solution and dz'Wdz.  All starts in
    one call, one start alone and a reversed subset give bit-identical rows."""
    prob, cf, slack, X, LAM, S, sigma, dw, dc, rhs = _kkt_setup_case(shape)
    run = KktRun(prob, slack, X, LAM, S)
    try:
        allst = np.arange(B_KKT)
        sol, inert, wq = run.solve(allst, sigma, dw, dc, rhs)
        Kd = [run.ev.kkt_matrix(b) for b in allst]
        for sub in (np.array([5]), allst[::-2]):
            s2, i2, w2 = run.solve(sub, sigma, dw, dc, rhs)
            assert np.array_equal(s2, sol[sub]) and np.array_equal(i2, inert[sub]), sub
            assert np.array_equal(w2, wq[sub], equal_nan=True), sub
    finally:
        run.close()
    for b in allst:
        _check_quasi_definite(cf, X[b], LAM[b], S[b], slack, Kd[b], sol[b], inert[b], wq[b], sigma[b], dw[b], dc[b],
                              rhs[b], "%s start %d" % (shape_id(shape), b))


def _indefinite_P0(n, neg, rng):
    Q, _ = np.linalg.qr(rng.standard_normal((n, n)))
    e = rng.uniform(1.0, 3.0, n)
    e[:neg] *= -1
    return (Q * e) @ Q.T


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(1, 0, 0), (30, 3, 2), (127, 1, 0)], ids=shape_id)
def test_gpu_kkt_indefinite(shape):
    """P0 with m + 1 negative eigenvalues, lam = 0, small Sigma and dw = 0: W has more negative directions than A
    has rows, so no K can have inertia (N, m, 0) (Haynsworth).  The device must say so and return NaN."""
    n, ki, ke = shape
    m = ki + ke
    rng = np.random.default_rng(77)
    P, q, _ = W.qcqp_data(n, m, seed=5)
    P[0] = _indefinite_P0(n, min(n, m + 1), rng)
    prob, P, q, slack = qcqp_case(n, ki, ke, P=P, q=q)
    X, _, S = oracle_inputs(n, m, B_KKT, seed=3)
    LAM = np.zeros((B_KKT, m))
    N, M = n + ki, n + ki + m
    sigma = np.full((B_KKT, N), 1e-3)
    dw, dc, rhs = np.zeros(B_KKT), np.full(B_KKT, 1e-2), rng.standard_normal((B_KKT, M))
    run = KktRun(prob, slack, X, LAM, S)
    try:
        sol, inert, wq = run.solve(np.arange(B_KKT), sigma, dw, dc, rhs)
    finally:
        run.close()
    for b in range(B_KKT):
        assert tuple(inert[b]) != (N, m, 0) and int(inert[b].sum()) == M and np.all(inert[b] >= 0), inert[b]
        _assert_nan(sol[b], wq[b], "start %d" % b)


DEGENERATE_SHAPE = (30, 3, 2)
BAD = 3


def _degenerate_case(kind):
    n, ki, ke = DEGENERATE_SHAPE
    P, q, _ = W.qcqp_data(n, ki + ke, seed=9)
    if kind == "singular":            # equality rows 0 and 1 identical: J has two equal rows
        P[2], q[2] = P[1].copy(), q[1].copy()
    if kind == "zero_pivot":
        P[0][0, 0] = 0.0
    return _kkt_setup_case(DEGENERATE_SHAPE, P=P, q=q)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["singular", "zero_pivot", "nan_x"])
def test_gpu_kkt_degenerate_start_leaves_the_others_alone(kind):
    """One start of eight made degenerate: two identical equality rows with dc = 0 (exactly singular), an exactly
    zero first pivot (P0[0,0] = 0, lam = 0, Sigma_0 = 0, dw = 0), or a NaN in x.  That start gets a zero pivot in its
    inertia and a NaN solution; every other start is bit for bit what it is when all eight are good."""
    prob, cf, slack, X, LAM, S, sigma, dw, dc, rhs = _degenerate_case(kind)
    n, ki, ke = DEGENERATE_SHAPE
    allst = np.arange(B_KKT)
    run = KktRun(prob, slack, X, LAM, S)
    try:
        good = run.solve(allst, sigma, dw, dc, rhs)
        Kd = run.ev.kkt_matrix(0)
        X2, LAM2, sigma2, dw2, dc2 = X.copy(), LAM.copy(), sigma.copy(), dw.copy(), dc.copy()
        if kind == "singular":
            dc2[BAD] = 0.0
        elif kind == "zero_pivot":
            LAM2[BAD] = 0.0
            sigma2[BAD, 0] = 0.0
            dw2[BAD] = 0.0
        else:
            X2[BAD, 7] = np.nan
        run.load(X2, LAM2, S)
        sol, inert, wq = run.solve(allst, sigma2, dw2, dc2, rhs)
        if kind == "zero_pivot":
            assert run.ev.kkt_matrix(BAD)[0, 0] == 0.0
    finally:
        run.close()
    _check_quasi_definite(cf, X[0], LAM[0], S[0], slack, Kd, good[0][0], good[1][0], good[2][0], sigma[0], dw[0],
                          dc[0], rhs[0], "%s good start 0" % kind)
    assert tuple(good[1][BAD]) == (n + ki, ki + ke, 0)
    assert inert[BAD][2] >= 1, inert[BAD]
    _assert_nan(sol[BAD], wq[BAD], kind)
    others = allst != BAD
    assert np.array_equal(sol[others], good[0][others])
    assert np.array_equal(inert[others], good[1][others])
    assert np.array_equal(wq[others], good[2][others])


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(1, 0, 0), (32, 0, 1), (62, 2, 3), (28, 2, 3), (127, 1, 0), (255, 0, 2)],
                         ids=shape_id)
def test_gpu_kkt_matches_numpy_at_edges(shape):
    """The same-algorithm check of test_lockstep_ipm.py (exact scatter, equal inertia, the NumPy LDL' solution) at
    block edges, with wide Sigma and indefinite W."""
    n, ki, ke = shape
    prob, _, _, _ = qcqp_case(n, ki, ke)
    _device_vs_numpy(prob, B_KKT, np.array([7, 2, 5, 0]), seed=shape_M(shape))


@pytest.mark.gpu
def test_gpu_kkt_setup_refuses_what_does_not_fit():
    """sum x^2 with n = 4096, m = 0 (bounds only): 4096 starts need 4096 * 4096^2 * 8 = 550 GB of dense systems,
    more than any B200 has.  kkt_setup raises with the size in the message and keeps nothing, the handle still
    evaluates; a small batch of the same problem then sets up and solves its diagonal systems."""
    from dnlp_b200 import ir
    from dnlp_b200.multistart import BatchedOracles
    n = 4096
    x = ir.Variable(n)
    prob = ir.ProblemIR(ir.sum(ir.power(x, 2)), [], [x], lb=-np.ones(n), ub=np.ones(n), x0=np.zeros(n))
    ev = BatchedOracles(prob, 4096)
    try:
        with pytest.raises(RuntimeError, match=r"B\*\(N\+m\)\^2\*8 = 4096\*4096\^2\*8"):
            ev.kkt_setup(np.zeros(0, dtype=np.int32))
        ev.kkt_N = n
        with pytest.raises(RuntimeError, match="kkt_setup first"):
            ev.kkt_solve([0], np.ones((1, n)), [0.0], [0.0], np.ones((1, n)))
        X = np.random.default_rng(0).uniform(-1, 1, (4096, n))
        f = ev.eval(X, want=("f",))["f"]
        np.testing.assert_allclose(f, np.sum(X * X, axis=1), rtol=1e-13)
    finally:
        ev.close()
    ev = BatchedOracles(prob, 2)
    try:
        ev.kkt_setup(np.zeros(0, dtype=np.int32))
        rng = np.random.default_rng(1)
        S = np.array([1.0, 0.5])
        ev.upload(rng.uniform(-1, 1, (2, n)), np.zeros((2, 0)), S)
        ev.run_device(("hess",))
        sigma, rhs = rng.uniform(0.1, 1.0, (2, n)), rng.standard_normal((2, n))
        sol, inert, wq = ev.kkt_solve([1, 0], sigma[::-1], [1e-3, 0.0], [0.0, 0.0], rhs[::-1])
        for c, b in enumerate([1, 0]):
            d = 2 * S[b] + sigma[b] + (1e-3 if c == 0 else 0.0)
            assert tuple(inert[c]) == (n, 0, 0)
            np.testing.assert_allclose(sol[c], rhs[b] / d, rtol=4 * U, atol=0)
    finally:
        ev.close()


# ---- GPU tier: oracle dispatch ---------------------------------------------------------------------------------------
def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _eval_once(prob, tape, B, X, LAM, S, env, monkeypatch, rows=None):
    """Outputs (rows ``rows`` only) of a fresh handle created under the environment ``env``, and the kernel name of
    every instruction.  Without ``env`` the handle evaluates twice: the second evaluation replays the captured graph."""
    from dnlp_b200.multistart import BatchedOracles
    with monkeypatch.context() as mp:
        for k, v in env.items():
            mp.setenv(k, v)
        ev = BatchedOracles(prob, B, tape=tape)
    take = (lambda o: {k: v[rows] for k, v in o.items()}) if rows is not None else (lambda o: o)
    try:
        outs = [take(ev.eval(X, LAM, S))]
        names = [ev.instr_kernel(i) for i in range(len(tape.instrs))]
        if not env:
            outs.append(take(ev.eval(X, LAM, S)))
    finally:
        ev.close()
    return outs, names


def _roles(tape):
    out = {}
    for i, ins in enumerate(tape.instrs):
        out.setdefault("gemm" if ins.kind == T.K_GEMV else _ROLE.get(ins.dst_space, "v"), []).append(i)
    return out


_seen_variants = set()


@pytest.mark.gpu
@pytest.mark.parametrize("case", DISPATCH, ids=dispatch_id)
def test_gpu_dispatch_edges(case, monkeypatch):
    """Every output of every start (every 37th at n = 512) within C_ORACLE * terms * u * magnitude of the closed form;
    the kernel variant of every instruction as the table says (on a 148-SM B200); bit-identical results from a
    second evaluation (graph replay) and from a handle without graphs; the m16n8k8 DMMA within the same bound."""
    from dnlp_b200.compiler import compile_problem
    n, k, B, want = case
    prob, P, q, _ = qcqp_case(n, k, 0)
    tape = compile_problem(prob)
    cf = closed_form(prob, P, q)
    X, LAM, S = oracle_inputs(n, k, B, seed=B + n)
    rows = np.arange(0, B, 37) if n >= 512 else np.arange(B)
    ref = cf.oracles(X[rows], LAM[rows], S[rows])

    def check(out, what):
        for name, (v, mag) in ref.items():
            if v.size:
                within_bound(out[name], v, mag, ClosedForm.TERMS[name](n, k), "%s %s %s" % (dispatch_id(case), what, name))

    outs, names = _eval_once(prob, tape, B, X, LAM, S, {}, monkeypatch, rows)
    check(outs[0], "graph")
    for name in outs[0]:
        assert np.array_equal(outs[0][name], outs[1][name]), ("replay", name)
    roles = _roles(tape)
    assert all(names[i] for ids in roles.values() for i in ids), names
    _seen_variants.update(names)
    if _sm_count() == 148:
        for role, kname in want.items():
            assert [names[i] for i in roles[role]] == [kname] * len(roles[role]), (role, [names[i] for i in roles[role]])
        for role in ("grad", "jac"):
            assert all(names[i] == "bpoly_kernel<0>" for i in roles.get(role, [])), role
    nog, _ = _eval_once(prob, tape, B, X, LAM, S, {"DNLP_BATCH_NO_GRAPHS": "1"}, monkeypatch, rows)
    for name in outs[0]:
        assert np.array_equal(outs[0][name], nog[0][name]), ("no graphs", name)
    k8, k8names = _eval_once(prob, tape, B, X, LAM, S, {"DNLP_DMMA_K8": "1"}, monkeypatch, rows)
    assert all(k8names[i] == "bgemm_dmma_kernel<1>" for i in roles["gemm"])
    check(k8[0], "m16n8k8")


@pytest.mark.gpu
def test_gpu_dispatch_covers_every_variant(monkeypatch):
    """The dispatch table reaches every variant it names (on a 148-SM B200); cases not run yet in this session are
    evaluated here."""
    from dnlp_b200.compiler import compile_problem
    if _sm_count() != 148:
        pytest.skip("the dispatch table is for a 148-SM B200")
    seen = set(_seen_variants)
    if not REQUIRED_VARIANTS <= seen:
        for n, k, B, _ in DISPATCH:
            if n >= 512:
                continue
            prob, _, _, _ = qcqp_case(n, k, 0)
            tape = compile_problem(prob)
            X, LAM, S = oracle_inputs(n, k, B, seed=1)
            _, names = _eval_once(prob, tape, B, X, LAM, S, {"DNLP_BATCH_NO_GRAPHS": "1"}, monkeypatch)
            seen.update(names)
    print("batched kernel variants seen:", ", ".join(sorted(seen)))
    assert REQUIRED_VARIANTS <= seen, sorted(REQUIRED_VARIANTS - seen)
