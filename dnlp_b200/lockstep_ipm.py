"""Lock-step primal-dual interior-point method: B starts of one smooth problem with variable bounds and inequality rows.

This is the serial barrier solver of the test-suite's IPOPT stand-in (tests/cyipopt_standin.py, ``_BarrierSolver.run``,
exact-Hessian branch) written over (B, .) arrays: slacks for the inequality rows, a monotone barrier update, the
fraction-to-the-boundary rule, inertia correction and l1-merit backtracking.  Every per-start scalar of the serial
method (mu, nu, dw_last, dw_min, the stall counter, the status, the iteration count) is a (B,) array; a start that has
stopped keeps its point and takes no further part.

One outer iteration:
  1. one batched evaluation of f, grad f, g and J at every start (copied to the host: J is small);
  2. the Hessian of the Lagrangian at (X, lambda, 1), left where the KKT backend wants it;
  3. the inertia-correction loop: the backend assembles, factors and solves the KKT systems of the starts whose
     inertia is still wrong, with a larger dw each round;
  4. lock-step backtracking: every round evaluates f and g at the trial points of the starts still searching; the
     others pass their current point and ignore the result.

The KKT backend is a constructor argument.  ``DeviceKKT`` keeps the Hessian and Jacobian in HBM and factors the
systems there (csrc/dnlp_batch_kkt.cuh, LDL' without pivoting); the test-suite passes a NumPy implementation of the
same factorisation.

``hessian_approximation="limited-memory"`` is the stand-in's quasi-Newton branch: W is a dense damped-BFGS matrix per
start, W_0 = I, updated after every accepted step (except the one that ends a start on the stall rule) with
s = x_new - x_old and y = (grad f + J'lam)(x_new) - (grad f + J'lam)(x_old), both with the new lam.  The update runs
at the top of the next outer iteration on the starts accepted in the previous one that are still active, from that
iteration's f / grad f / g / J evaluation (no extra evaluation); step 2 then evaluates only J, the Hessian is never
asked for.  With ``DeviceKKT(ev, quasi_newton=True)`` the matrices live in HBM and the update runs there
(csrc/dnlp_batch_qn.cuh).  Not covered: IPOPT's compact L-BFGS and the ``intermediate`` callback.
"""
import time

import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

INF = 1e19            # IPOPT's nlp_lower/upper_bound_inf

STATUS_MSG = {0: b"Algorithm terminated successfully at a locally optimal point",
              -1: b"Maximum number of iterations exceeded",
              3: b"Search direction becomes too small",
              -3: b"could not regularise the KKT system",
              -13: b"Invalid number detected"}


class DeviceKKT:
    """KKT backend on ``BatchedOracles``: the Hessian and Jacobian never leave HBM; the B dense systems are assembled,
    factored and solved there (``BatchedOracles.kkt_solve``).  With ``quasi_newton`` the Hessian is replaced by one
    damped-BFGS matrix per start, kept and updated in HBM (``BatchedOracles.qn_update``)."""

    def __init__(self, ev, quasi_newton=False):
        self.ev = ev
        self.quasi_newton = bool(quasi_newton)
        self.device_ms = 0.0          # CUDA-event time of assembly + factorisation + solve (+ QN update), summed
        self.qn_ms = 0.0              # CUDA-event time of the quasi-Newton updates alone
        self.qn_calls = self.qn_starts = 0

    def setup(self, slack_rows):
        self.ev.kkt_setup(slack_rows, quasi_newton=self.quasi_newton)

    def load(self, X, LAM):
        """The Jacobian and (exact mode) the Hessian of the Lagrangian (sigma = 1) of every start at (X, LAM), on the
        device."""
        self.ev.upload(X, LAM, np.ones(X.shape[0]))
        self.ev.run_device(("jac",) if self.quasi_newton else ("jac", "hess"))

    def update(self, starts, S, Y):
        applied = self.ev.qn_update(starts, S, Y)
        self.qn_ms += self.ev.qn_ms
        self.device_ms += self.ev.qn_ms
        self.qn_calls += 1
        self.qn_starts += len(starts)
        return applied

    def solve(self, starts, sigma, dw, dc, rhs):
        out = self.ev.kkt_solve(starts, sigma, dw, dc, rhs)
        self.device_ms += self.ev.kkt_ms
        return out


def _bounds(v, size, fill):
    return np.full(size, fill) if v is None else np.array(v, dtype=np.float64).reshape(size)


HESSIAN_APPROXIMATIONS = ("exact", "limited-memory")


def check_hessian_approximation(value):
    if value not in HESSIAN_APPROXIMATIONS:
        raise ValueError("hessian_approximation must be 'exact' or 'limited-memory', not %r" % (value,))
    return value == "limited-memory"


def lockstep_ipm(ev, kkt, X0, lb=None, ub=None, cl=None, cu=None, tol=1e-8, max_iter=500, mu_init=0.1, progress=None,
                 hessian_approximation="exact"):
    """Solve min f(x) s.t. cl <= g(x) <= cu, lb <= x <= ub from every row of ``X0`` (B, n) in lock step.

    ``ev``: batched evaluator (``BatchedOracles`` or anything with ``eval(X, LAM, SIGMA, want) -> {name: (B, len)}``,
    ``jacobianstructure()``, ``n``, ``m``); ``kkt``: KKT backend (``DeviceKKT(ev)`` or one with the same
    ``setup`` / ``load`` / ``solve``).  Bounds beyond 1e19 in magnitude are absent, as for IPOPT.
    ``hessian_approximation``: "exact" or "limited-memory" (damped BFGS per start, see the module docstring); the
    latter needs a backend built for it (``quasi_newton = True``, with ``update(starts, S, Y)``).

    Returns per start: ``x``, ``g``, ``f``, ``lam`` (constraint multipliers, IPOPT's mult_g), ``zL``, ``zU`` (bound
    multipliers), ``status`` (0 solved, -1 iteration limit, 3 step too small, -3 KKT system could not be regularised,
    -13 invalid number) and ``iterations``; plus ``timings``: per outer iteration the wall seconds spent in evaluations
    (``eval_s``), in the KKT backend (``kkt_s``) and in total (``total_s``).  ``progress(it, timing, n_active)``, when
    given, is called after every outer iteration (long batches run for minutes)."""
    qn = check_hessian_approximation(hessian_approximation)
    if bool(getattr(kkt, "quasi_newton", False)) != qn:
        raise ValueError("hessian_approximation=%r needs a KKT backend with quasi_newton=%s"
                         % (hessian_approximation, qn))
    X0 = np.array(X0, dtype=np.float64, ndmin=2)
    B, n = X0.shape
    m = int(ev.m)
    lb, ub = _bounds(lb, n, -2e19), _bounds(ub, n, 2e19)
    cl, cu = _bounds(cl, m, -2e19), _bounds(cu, m, 2e19)
    ineq = np.flatnonzero(cl != cu)
    ns = ineq.size
    N = n + ns
    Lb, Ub = np.concatenate([lb, cl[ineq]]), np.concatenate([ub, cu[ineq]])
    hasL, hasU = Lb > -INF, Ub < INF
    L, U = np.where(hasL, Lb, -np.inf), np.where(hasU, Ub, np.inf)
    rhs_eq = np.where(cl == cu, cl, 0.0)
    jr, jc = (np.asarray(a, dtype=np.int64) for a in ev.jacobianstructure())
    lin = jr * n + jc
    jac_unique = np.unique(lin).size == lin.size
    Jsum = None if jac_unique else sp.csr_matrix((np.ones(lin.size), (lin, np.arange(lin.size))), shape=(m * n, lin.size))
    Psel = sp.csr_matrix((np.ones(ns), (ineq, np.arange(ns))), shape=(m, ns))
    kkt.setup(ineq)

    def dense_jac(vals):
        if jac_unique:
            J = np.zeros((B, m * n))
            J[:, lin] = vals
        else:
            J = np.ascontiguousarray((Jsum @ vals.T).T)
        return J.reshape(B, m, n)

    def h(G, S):                       # g - cl on equality rows, g - s on the others
        out = G - rhs_eq
        out[:, ineq] -= S
        return out

    def push_inside(V):                # IPOPT's initial-point projection (bound_push = bound_frac = 1e-2)
        pl = np.minimum(1e-2 * np.maximum(1.0, np.abs(np.where(hasL, L, 0.0))), 1e-2 * (U - L))
        pu = np.minimum(1e-2 * np.maximum(1.0, np.abs(np.where(hasU, U, 0.0))), 1e-2 * (U - L))
        V = np.where(hasL, np.maximum(V, L + np.where(np.isfinite(pl), pl, 1e-2)), V)
        return np.where(hasU, np.minimum(V, U - np.where(np.isfinite(pu), pu, 1e-2)), V)

    def barrier(Z, mu):
        dl, du = Z[:, hasL] - L[hasL], U[hasU] - Z[:, hasU]
        bad = (dl <= 0).any(axis=1) | (du <= 0).any(axis=1)
        val = -mu * (np.log(dl).sum(axis=1) + np.log(du).sum(axis=1))
        return np.where(bad, np.inf, val)

    def amax(a):
        return np.abs(a).max(axis=1, initial=0.0)

    def lam_times_A(J, LAM):           # A' lam, A = [J, -P]
        return np.concatenate([np.matmul(LAM[:, None, :], J)[:, 0, :], -LAM[:, ineq]], axis=1)

    olderr = np.seterr(all="ignore")
    try:
        X = push_inside(np.concatenate([X0, np.zeros((B, ns))], axis=1))[:, :n]
        G = ev.eval(X, want=("g",))["g"] if m else np.zeros((B, 0))
        Z = push_inside(np.concatenate([X, G[:, ineq]], axis=1))
        X = Z[:, :n].copy()
        zL = np.tile(np.where(hasL, 1.0, 0.0), (B, 1))
        zU = np.tile(np.where(hasU, 1.0, 0.0), (B, 1))
        mu = np.full(B, float(mu_init))
        r0 = ev.eval(X, want=("grad", "jac") if m else ("grad",))
        lam = np.zeros((B, m))
        if m:                          # least-squares multiplier estimate, start by start as the serial solver does
            gz0 = np.concatenate([r0["grad"], np.zeros((B, ns))], axis=1)
            for b in range(B):
                try:
                    A = sp.hstack([sp.csr_matrix((r0["jac"][b], (jr, jc)), shape=(m, n)), -Psel], format="csr")
                    lb_ = spla.lsqr(A.T.tocsr(), -(gz0[b] - zL[b] + zU[b]), atol=1e-12, btol=1e-12)[0]
                    if np.all(np.isfinite(lb_)) and np.abs(lb_).max() <= 1e3:
                        lam[b] = lb_
                except Exception:
                    pass
        dw_last, dw_min, nu = np.zeros(B), np.zeros(B), np.ones(B)
        stalled = np.zeros(B, dtype=np.int64)
        status = np.full(B, -1, dtype=np.int64)
        iters = np.zeros(B, dtype=np.int64)
        active = np.ones(B, dtype=bool)
        f = np.zeros(B)
        qn_from = None                 # (accepted, x, grad f, J) of the previous iteration, for the BFGS update
        timings = []
        for it in range(max_iter + 1):
            t0 = time.perf_counter()
            res = ev.eval(X, want=("f", "grad", "g", "jac") if m else ("f", "grad"))
            t_eval = time.perf_counter() - t0
            t_kkt = 0.0
            f_new = np.asarray(res["f"], dtype=np.float64).reshape(B)
            f = np.where(active, f_new, f)
            if m:
                G = np.where(active[:, None], res["g"], G)
            J = dense_jac(res["jac"]) if m else np.zeros((B, 0, n))
            gz = np.concatenate([res["grad"], np.zeros((B, ns))], axis=1)
            ATlam = lam_times_A(J, lam)
            hv = h(G, Z[:, n:])
            dL, dU = np.where(hasL, Z - L, 1.0), np.where(hasU, U - Z, 1.0)
            rd = gz + ATlam - zL + zU
            sd = np.maximum(100.0, (np.abs(lam).sum(axis=1) + zL.sum(axis=1) + zU.sum(axis=1)) / max(m + 2 * N, 1)) / 100.0

            def err(mu_):
                comp = np.maximum(amax(np.where(hasL, dL * zL - mu_[:, None], 0.0)),
                                  amax(np.where(hasU, dU * zU - mu_[:, None], 0.0)))
                return np.maximum(np.maximum(amax(rd) / sd, amax(hv)), comp / sd)
            bad = active & ~(np.isfinite(f) & np.isfinite(rd).all(axis=1) & np.isfinite(hv).all(axis=1))
            status[bad], iters[bad], active[bad] = -13, it, False
            conv = active & (err(np.zeros(B)) <= tol)
            status[conv], iters[conv], active[conv] = 0, it, False
            if it == max_iter:
                iters[active] = it
                active[:] = False
            if not active.any():
                timings.append({"eval_s": t_eval, "kkt_s": 0.0, "total_s": time.perf_counter() - t0})
                break
            t_qn = 0.0
            if qn_from is not None:        # damped BFGS with the previous iteration's step, at the new lam
                t1 = time.perf_counter()
                acc_prev, X_old, grad_old, J_old = qn_from
                idx = np.flatnonzero(acc_prev & active)
                if idx.size:
                    Yn = res["grad"][idx] + np.matmul(lam[idx, None, :], J[idx])[:, 0, :]
                    Yo = grad_old[idx] + np.matmul(lam[idx, None, :], J_old[idx])[:, 0, :]
                    kkt.update(idx, X[idx] - X_old[idx], Yn - Yo)
                t_qn = time.perf_counter() - t1
            while True:                # monotone barrier update
                upd = active & (mu > tol / 10.0) & (err(mu) <= 10.0 * mu)
                if not upd.any():
                    break
                mu = np.where(upd, np.maximum(tol / 10.0, np.minimum(0.2 * mu, mu ** 1.5)), mu)
                nu = np.where(upd, 1.0, nu)
            t1 = time.perf_counter()
            kkt.load(X, lam)
            t_eval += time.perf_counter() - t1
            Sigma = np.where(hasL, zL / dL, 0.0) + np.where(hasU, zU / dU, 0.0)
            gphi = gz - np.where(hasL, mu[:, None] / dL, 0.0) + np.where(hasU, mu[:, None] / dU, 0.0)
            rhs = -np.concatenate([gphi + ATlam, hv], axis=1)
            # inertia correction: dw is raised per start until K has the inertia (N, m, 0) of a descent step
            t1 = time.perf_counter()
            dc = 1e-9 * np.maximum(mu, 1e-12) ** 0.25
            dw = dw_min.copy()
            sol = np.full((B, N + m), np.nan)
            wq = np.zeros(B)
            pend = active.copy()
            for attempt in range(60):
                idx = np.flatnonzero(pend)
                if idx.size == 0:
                    break
                s, inert, w = kkt.solve(idx, Sigma[idx], dw[idx], dc[idx], rhs[idx])
                ok = (inert[:, 0] == N) & (inert[:, 1] == m) & (inert[:, 2] == 0) & np.isfinite(s).all(axis=1)
                sol[idx[ok]], wq[idx[ok]] = s[ok], w[ok]
                pend[idx[ok]] = False
                rej = idx[~ok]
                d, d0 = dw[rej], dw_last[rej]
                dw[rej] = np.where(d == 0.0, np.maximum(d0 / 3.0, 1e-4),
                                   d * np.where((d0 == 0.0) & (attempt < 3), 100.0, 8.0))
                pend[rej[dw[rej] > 1e40]] = False
            t_kkt = time.perf_counter() - t1 + t_qn
            solved = active & np.isfinite(sol).all(axis=1)
            failed = active & ~solved
            status[failed], iters[failed], active[failed] = -3, it, False
            dw_last = np.where(solved, dw, dw_last)
            dz, dlam = sol[:, :N], sol[:, N:]
            dzL = np.where(hasL, mu[:, None] / dL - zL - zL / dL * dz, 0.0)
            dzU = np.where(hasU, mu[:, None] / dU - zU + zU / dU * dz, 0.0)
            tau = np.maximum(0.99, 1.0 - mu)

            def max_step(v, dv, mask):
                neg = mask & (dv < 0)
                return np.minimum(1.0, np.where(neg, -tau[:, None] * v / dv, np.inf).min(axis=1))
            a_max = np.minimum(max_step(dL, dz, hasL), max_step(dU, -dz, hasU))
            alpha_du = np.minimum(max_step(zL, dzL, hasL), max_step(zU, dzU, hasU))
            # l1 merit function with backtracking, all searching starts in lock step
            h1 = np.abs(hv).sum(axis=1)
            lin_ = (gphi * dz).sum(axis=1)
            quad = wq + (Sigma * dz * dz).sum(axis=1)
            nu = np.where(solved & (h1 > 0), np.maximum(nu, (lin_ + 0.5 * np.maximum(quad, 0.0)) / (0.9 * h1) + 1e-8), nu)
            phi0 = f + barrier(Z, mu) + nu * h1
            D = lin_ - nu * h1
            alpha = np.where(solved, a_max, 0.0)
            ls = np.zeros(B, dtype=np.int64)
            accepted = np.zeros(B, dtype=bool)
            Zacc, facc, Gacc = Z.copy(), f.copy(), G.copy()
            search = solved.copy()
            while search.any():
                Zt = np.where(search[:, None], Z + alpha[:, None] * dz, Z)
                t1 = time.perf_counter()
                rt = ev.eval(Zt[:, :n], want=("f", "g") if m else ("f",))
                t_eval += time.perf_counter() - t1
                ft = np.asarray(rt["f"], dtype=np.float64).reshape(B)
                gt = rt["g"] if m else np.zeros((B, 0))
                phit = ft + barrier(Zt, mu) + nu * np.abs(h(gt, Zt[:, n:])).sum(axis=1)
                ls += search
                ok = search & np.isfinite(phit) & \
                    (phit <= phi0 + 1e-8 * alpha * np.minimum(D, 0.0) + 10 * np.finfo(float).eps * np.abs(phi0))
                Zacc[ok], facc[ok], Gacc[ok] = Zt[ok], ft[ok], gt[ok]
                accepted |= ok
                search &= ~ok
                alpha = np.where(search, alpha * 0.5, alpha)
                search &= ls < 40
            rejected = solved & ~accepted     # try again with a more conservative direction
            dw_min = np.where(rejected, np.maximum(dw_last * 100.0, 1e-2), dw_min)
            small = rejected & (dw_min > 1e12)
            status[small], iters[small], active[small] = 3, it, False
            dw_min = np.where(accepted, 0.0, dw_min)
            step = alpha * amax(dz) < 1e-9 * (1.0 + amax(Z))
            stalled = np.where(accepted, np.where(step, stalled + 1, 0), stalled)
            stop = accepted & (stalled >= 30)  # the l1 merit line search has no filter / SOC
            status[stop], iters[stop], active[stop] = 3, it, False
            acc = accepted & ~stop
            if qn:
                qn_from = (acc, X, res["grad"], J)
            Z = np.where(acc[:, None], Zacc, Z)
            X = Z[:, :n].copy()
            f = np.where(acc, facc, f)
            G = np.where(acc[:, None], Gacc, G)
            lam = np.where(acc[:, None], lam + alpha[:, None] * dlam, lam)
            zLn, zUn = zL + alpha_du[:, None] * dzL, zU + alpha_du[:, None] * dzU
            # keep the bound multipliers within a factor of the primal estimate mu / (z - L)   (IPOPT eq. 16)
            dLn, dUn = np.where(hasL, Z - L, 1.0), np.where(hasU, U - Z, 1.0)
            zLn = np.where(hasL, np.clip(zLn, mu[:, None] / (1e10 * dLn), 1e10 * mu[:, None] / dLn), 0.0)
            zUn = np.where(hasU, np.clip(zUn, mu[:, None] / (1e10 * dUn), 1e10 * mu[:, None] / dUn), 0.0)
            zL, zU = np.where(acc[:, None], zLn, zL), np.where(acc[:, None], zUn, zU)
            timings.append({"eval_s": t_eval, "kkt_s": t_kkt, "total_s": time.perf_counter() - t0})
            if progress is not None:
                progress(it, timings[-1], int(active.sum()))
    finally:
        np.seterr(**olderr)
    return {"x": X, "g": G, "f": f, "lam": lam, "zL": zL[:, :n].copy(), "zU": zU[:, :n].copy(), "status": status,
            "iterations": iters, "timings": timings}
