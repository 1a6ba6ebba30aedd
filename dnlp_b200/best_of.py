"""Batched ``best_of``: every start of a multi-start solve advances in lock step on ONE compiled tape.

The reference's ``prob.solve(nlp=True, best_of=N)`` (cvxpy/problems/problem.py:1249-1275) is a serial loop:
re-sample the variables (``set_random_NLP_initial_point``, problem.py:1643-1693), re-apply the whole
reduction chain, run one IPOPT solve, keep the best objective, and hand every objective back in
``extra_stats['all_objs_from_best_of']`` (ipopt_nlpif.py:87-89).  ``install()`` already makes that loop
compile once (dnlp_b200/compile_cache.py); here the N solves themselves are batched:

``lockstep_newton_kkt``  a primal-dual Newton iteration on the KKT system of an equality-constrained smooth
    problem, for B starts at once.  Per iteration ONE ``BatchedOracles.eval`` produces f, grad, g, J and
    Hess L of every start (csrc/dnlp_batch.cu); the B dense KKT systems are solved as one batched LAPACK
    call on the host.  It touches the oracle only through the callback outputs and structures, like the
    test-suite's serial stand-in for IPOPT (tests/kkt_newton.py), and takes exactly its iterates.
    It is NOT an interior-point method: problems with a finite variable bound or an inequality row go to
    ``lockstep_ipm`` (dnlp_b200/lockstep_ipm.py) instead, whose B KKT systems are factored on the GPU.

``solve_best_of``  the reference's loop with the solves batched: N initial points from the reference's own
    sampler, one compile, one lock-step solve, ``all_objs_from_best_of`` and the best start unpacked through
    the reference's own invert chain.
"""
import numpy as np


def _dense_batch(rows, cols, vals, shape):
    """(B, nnz) triplet values on a fixed pattern -> (B, r, c) dense (duplicates add)."""
    B = vals.shape[0]
    out = np.zeros((B,) + shape)
    np.add.at(out, (slice(None), rows, cols), vals)
    return out


def lockstep_newton_kkt(ev, X0, tol=1e-12, max_iter=60):
    """``ev``: batched evaluator (``BatchedOracles`` or anything with ``eval(X, LAM, SIG) -> {name: (B, len)}``,
    ``jacobianstructure()``, ``hessianstructure()``, ``n``, ``m``).  Returns a dict with per-start
    ``x``, ``lam``, ``f``, ``iterations`` and ``converged``."""
    X = np.array(X0, dtype=np.float64)
    B, n = X.shape
    m = int(ev.m)
    jr, jc = (np.asarray(a, dtype=np.int64) for a in ev.jacobianstructure())
    hr, hc = (np.asarray(a, dtype=np.int64) for a in ev.hessianstructure())
    LAM = np.zeros((B, m))
    SIG = np.ones(B)
    iters = np.zeros(B, dtype=np.int64)
    done = np.zeros(B, dtype=bool)
    res = ev.eval(X, LAM, SIG)
    if m:       # least-squares multiplier estimate per start (IPOPT's least_square_init_duals, ipopt_nlpif.py:160)
        J0 = _dense_batch(jr, jc, res["jac"], (m, n))
        for b in range(B):
            LAM[b] = np.linalg.lstsq(J0[b].T, -res["grad"][b], rcond=None)[0]
    for it in range(max_iter + 1):
        res = ev.eval(X, LAM, SIG)
        G = res["grad"]
        Cv = res["g"] if m else np.zeros((B, 0))
        J = _dense_batch(jr, jc, res["jac"], (m, n)) if m else np.zeros((B, 0, n))
        H = _dense_batch(hr, hc, res["hess"], (n, n))
        H = H + np.transpose(np.tril(H, -1), (0, 2, 1))              # the structure is the lower triangle
        R = np.concatenate([G + np.einsum("bmn,bm->bn", J, LAM), Cv], axis=1)
        newly = ~done & (np.abs(R).max(axis=1) < tol)
        iters[newly] = it
        done |= newly
        if done.all() or it == max_iter:
            break
        K = np.zeros((B, n + m, n + m))
        K[:, :n, :n] = H
        K[:, :n, n:] = np.transpose(J, (0, 2, 1))
        K[:, n:, :n] = J
        act = ~done
        step = np.zeros((B, n + m))
        step[act] = np.linalg.solve(K[act], -R[act][..., None])[..., 0]
        X = X + step[:, :n]
        LAM = LAM + step[:, n:]
    iters[~done] = max_iter
    res = ev.eval(X, LAM, SIG)
    return {"x": X, "lam": LAM, "f": np.asarray(res["f"], dtype=np.float64).reshape(B), "iterations": iters,
            "converged": done}


def _equality_only(problem_ir):
    """No finite variable bound and no inequality row: the problem the Newton-KKT iteration handles."""
    finite = [v is not None and np.any(np.isfinite(v)) for v in (problem_ir.lb, problem_ir.ub)]
    cl, cu = problem_ir.cl, problem_ir.cu
    two_sided = problem_ir.m > 0 and (cl is None or cu is None or np.any(np.asarray(cl) != np.asarray(cu)))
    return not any(finite) and not two_sided


def best_of_lockstep(problem_ir, X0, device=0, evaluator=None, kkt=None, tol=None, max_iter=None):
    """All starts ``X0`` (B, n) of one smooth problem in lock step on the GPU; ``evaluator`` replaces
    ``BatchedOracles`` (CPU tests).  Equality-constrained problems without bounds take ``lockstep_newton_kkt``
    (defaults tol 1e-12, 60 iterations), every other problem ``lockstep_ipm`` (tol 1e-8, 500 iterations) with the KKT
    backend ``kkt`` (default: ``DeviceKKT`` on the evaluator).  Adds ``all_objs`` and ``best`` (index of the smallest
    objective among the converged starts) to the solver's result."""
    own = evaluator is None
    if own:
        from .multistart import BatchedOracles
        evaluator = BatchedOracles(problem_ir, len(X0), device=device)
    try:
        if _equality_only(problem_ir):
            out = lockstep_newton_kkt(evaluator, X0, tol=1e-12 if tol is None else tol,
                                      max_iter=60 if max_iter is None else max_iter)
        else:
            from .lockstep_ipm import DeviceKKT, lockstep_ipm
            out = lockstep_ipm(evaluator, DeviceKKT(evaluator) if kkt is None else kkt, X0, lb=problem_ir.lb,
                               ub=problem_ir.ub, cl=problem_ir.cl, cu=problem_ir.cu, tol=1e-8 if tol is None else tol,
                               max_iter=500 if max_iter is None else max_iter)
            out["converged"] = out["status"] == 0
    finally:
        if own:
            evaluator.close()
    f = np.where(out["converged"], out["f"], np.inf)
    out["all_objs"] = out["f"].copy()
    out["best"] = int(np.argmin(f))
    return out


def _pick(smooth_objs, maximize, faithful):
    """Index of the start the loop keeps.  ``smooth_objs``: objective of the smooth MINIMISATION problem per start."""
    if maximize and faithful:              # the reference compares the un-flipped objective with `<`
        return int(np.argmin(-smooth_objs))
    return int(np.argmin(smooth_objs))


def solve_best_of(prob, best_of, solver="lockstep", device=0, evaluator_factory=None, faithful=True, kkt_factory=None,
                  **solver_opts):
    """The reference's ``best_of`` loop (problem.py:1249-1275) with one compile and batched solves.
    ``prob`` is a cvxpy Problem of the installed reference; returns ``prob.value`` and leaves variable values,
    ``prob.solver_stats.extra_stats['all_objs_from_best_of']`` exactly where the reference's loop leaves them.
    ``solver``: "lockstep" (all starts at once on the GPU: the Newton-KKT iteration for equality-constrained problems
    without bounds, the lock-step interior-point method for every other problem) or "ipopt" (per-start
    ``solve_via_data`` on the shared resident oracle; needs cyipopt).  ``evaluator_factory(problem_ir, B)`` and
    ``kkt_factory(evaluator)`` replace ``BatchedOracles`` and the device KKT backend (CPU tests).

    ``faithful`` (default): the reference's loop ranks the starts by ``self.objective.value`` with ``<`` whatever the
    sense (problem.py:1262-1268), so for a Maximize problem it keeps the start with the SMALLEST objective, and it
    then reports ``all_objs_from_best_of`` negated (problem.py:1270-1272).  Reproduced as is, so that switching
    changes no result; ``faithful=False`` keeps the best start in the problem's own sense and reports the objective
    values with their own sign."""
    import cvxpy as cp
    from cvxpy.reductions.cvx_attr2constr import CvxAttr2Constr
    from cvxpy.reductions.dnlp2smooth.dnlp2smooth import Dnlp2Smooth
    from cvxpy.reductions.flip_objective import FlipObjective
    from cvxpy.reductions.solvers.nlp_solvers.ipopt_nlpif import IPOPT
    from cvxpy.reductions.solvers.solving_chain import SolvingChain

    from .frontend_cvxpy import data_to_ir
    if (not isinstance(best_of, int)) or best_of < 1:
        raise ValueError("best_of must be a positive integer.")
    if not prob.is_dnlp():
        raise cp.error.DNLPError("The problem you specified is not DNLP.")
    maximize = type(prob.objective) == cp.Maximize
    chain = SolvingChain(reductions=([FlipObjective()] if maximize else []) +
                         [CvxAttr2Constr(reduce_bounds=False), Dnlp2Smooth(), IPOPT()])
    starts, data, inverse_data = [], None, None
    for run in range(best_of):
        prob.set_random_NLP_initial_point(run)                     # the reference's own sampler and rng stream
        data, inverse_data = chain.apply(problem=prob)
        starts.append(np.array(data["x0"], dtype=np.float64, copy=True))
    if solver == "ipopt":
        sols = []
        for x0 in starts:
            d = dict(data, x0=x0)
            sols.append(chain.solver.solve_via_data(d, False, False, solver_opts=solver_opts))
        objs = np.array([s["obj_val"] for s in sols])
        best = _pick(objs, maximize, faithful)
        best_solution = sols[best]
    else:
        pir = data_to_ir(data)
        ev = evaluator_factory(pir, best_of) if evaluator_factory is not None else None
        kkt = kkt_factory(ev) if (kkt_factory is not None and ev is not None) else None
        out = best_of_lockstep(pir, np.stack(starts), device=device, evaluator=ev, kkt=kkt, **solver_opts)
        objs = out["all_objs"]
        best = _pick(np.asarray(objs), maximize, faithful)
        if "status" in out:            # the interior-point driver: IPOPT's status codes and bound multipliers
            best_solution = {"status": int(out["status"][best]), "x": out["x"][best], "obj_val": float(objs[best]),
                             "mult_g": out["lam"][best], "mult_x_L": out["zL"][best], "mult_x_U": out["zU"][best],
                             "iterations": int(out["iterations"][best])}
        else:
            best_solution = {"status": 0 if out["converged"][best] else -1, "x": out["x"][best],
                             "obj_val": float(objs[best]), "mult_g": out["lam"][best],
                             "iterations": int(out["iterations"][best])}
    true_objs = -np.asarray(objs) if maximize else np.asarray(objs)      # self.objective.value at every start's solution
    all_objs = -true_objs if (maximize and faithful) else true_objs
    best_solution["all_objs_from_best_of"] = all_objs
    prob.unpack_results(best_solution, chain, inverse_data)
    return prob.value
