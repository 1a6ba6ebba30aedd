"""Batched multi-start oracle: the same smooth problem evaluated at B start points in lock step.

The reference's ``best_of=N`` loop (cvxpy/problems/problem.py:1249-1275, 1643-1693) re-samples the
variables, re-applies the whole reduction chain and solves one start after the other.  Here the
problem is compiled once and all B points go through one set of kernel launches; start points are
independent, so a multi-GPU run gives each rank its own slice of the batch with no collective.

Arrays are (B, len): row b belongs to start b.  Structures are those of the single-start oracle.
"""
import ctypes as C

import numpy as np

from . import _cabi
from .compiler import compile_problem

_f64p = _cabi.c_f64p
_PROGS = ("f", "grad", "g", "jac", "hess")


def _ptr(a):
    return None if a is None else a.ctypes.data_as(_f64p)


class BatchedOracles:
    def __init__(self, problem_ir, batch, device=0, tape=None):
        self.problem = problem_ir
        self.tape = tape if tape is not None else compile_problem(problem_ir)
        self.batch = int(batch)
        self.dev = _cabi.DeviceBatch(self.tape, self.batch, device)
        self.n, self.m = self.tape.n, self.tape.m
        self.nnz_jac, self.nnz_hess = int(self.tape.jac_rows.size), int(self.tape.hess_rows.size)
        self._len = {"f": 1, "grad": self.n, "g": self.m, "jac": self.nnz_jac, "hess": self.nnz_hess}

    def close(self):
        self.dev.close()

    def jacobianstructure(self):
        return self.tape.jac_rows, self.tape.jac_cols

    def hessianstructure(self):
        return self.tape.hess_rows, self.tape.hess_cols

    def _check_in(self, X, LAM, SIGMA):
        X = np.ascontiguousarray(X, dtype=np.float64)
        if X.shape != (self.batch, self.n):
            raise ValueError("X must have shape (%d, %d)" % (self.batch, self.n))
        if LAM is not None:
            LAM = np.ascontiguousarray(LAM, dtype=np.float64).reshape(self.batch, self.m)
        if SIGMA is not None:
            SIGMA = np.ascontiguousarray(np.broadcast_to(np.asarray(SIGMA, dtype=np.float64), (self.batch,)))
        return X, LAM, SIGMA

    def eval(self, X, LAM=None, SIGMA=None, want=_PROGS):
        """Evaluate the requested quantities at every start; returns {name: (B, len) array}."""
        X, LAM, SIGMA = self._check_in(X, LAM, SIGMA)
        if "hess" in want and (SIGMA is None or (self.m and LAM is None)):
            raise ValueError("hessian needs LAM and SIGMA")
        outs = {k: np.empty((self.batch, self._len[k])) for k in want}
        args = [_ptr(outs.get(k)) for k in _PROGS]
        self.dev.check(self.dev._L.dnlp_batch_eval(self.dev.h, _ptr(X), _ptr(LAM), _ptr(SIGMA), *args))
        if "f" in outs:
            outs["f"] = outs["f"].reshape(self.batch)
        return outs

    # ---- device-resident measurement hooks (bench.py) ---------------------------------------------
    def upload(self, X, LAM, SIGMA):
        X, LAM, SIGMA = self._check_in(X, LAM, SIGMA)
        self.dev.check(self.dev._L.dnlp_batch_upload(self.dev.h, _ptr(X), _ptr(LAM), _ptr(SIGMA)))

    def run_device(self, programs=_PROGS, iters=1):
        mask = 0
        for p in programs:
            mask |= 1 << _cabi.PROG_IDS[p]
        ms = C.c_float(0)
        self.dev.check(self.dev._L.dnlp_batch_run_device(self.dev.h, mask, int(iters), C.byref(ms)))
        return float(ms.value)

    def read_output(self, name):
        """The device output ``name`` as a (B, len) array, as the last ``run_device`` step left it."""
        out = np.empty((self.batch, self._len[name]))
        space = {"f": 1, "grad": 2, "g": 3, "jac": 4, "hess": 5}[name]
        self.dev.check(self.dev._L.dnlp_batch_read_output(self.dev.h, space, _ptr(out)))
        return out

    def profile_instrs(self, program="all", iters=3):
        out = np.zeros(max(len(self.tape.instrs), 1), dtype=np.float32)
        self.dev.check(self.dev._L.dnlp_batch_profile_instrs(self.dev.h, _cabi.PROG_IDS[program], int(iters),
                                                            out.ctypes.data_as(_cabi.c_f32p)))
        return out[:len(self.tape.instrs)]

    def profile_gemm_groups(self, iters=5):
        """[(ms, TFLOP/s)] of every grouped DMMA GEMM launch (independent dense maps of one shape as one grid)."""
        ms = np.zeros(8, dtype=np.float32)
        fl = np.zeros(8, dtype=np.float64)
        n = self.dev._L.dnlp_batch_profile_groups(self.dev.h, int(iters), ms.ctypes.data_as(_cabi.c_f32p),
                                                  fl.ctypes.data_as(_cabi.c_f64p), 8)
        if n < 0:
            raise RuntimeError("dnlp_batch_profile_groups failed")
        return [(float(ms[i]), float(fl[i] / (ms[i] * 1e-3) / 1e12) if ms[i] > 0 else 0.0) for i in range(n)]

    def kernel_launches(self):
        return int(self.dev._L.dnlp_batch_kernel_launches(self.dev.h))

    def instr_kernel(self, instr):
        """Name of the kernel variant that ran instruction ``instr`` (template arguments included, e.g.
        ``bsmallk_kernel<9, 2>``); "" for an instruction no evaluation has launched yet."""
        return self.dev._L.dnlp_batch_instr_kernel(self.dev.h, int(instr)).decode()

    # ---- batched KKT systems (dnlp_b200/lockstep_ipm.py; include/dnlp_b200.h dnlp_batch_kkt_*) ---------------
    def kkt_setup(self, slack_rows, quasi_newton=False):
        """Scatter maps of K = [[W + diag(Sigma) + dw I, A'], [A, -dc I]], A = [J, -P], for the slack rows
        ``slack_rows`` (the inequality rows, in slack order), and B dense systems in HBM.  W is the HESS output, or
        with ``quasi_newton`` one damped-BFGS matrix per start kept in HBM (set to I here, see ``qn_update``)."""
        sr = np.ascontiguousarray(slack_rows, dtype=np.int32)
        names = ("jac_rows", "jac_cols") if quasi_newton else ("jac_rows", "jac_cols", "hess_rows", "hess_cols")
        pats = [np.ascontiguousarray(getattr(self.tape, a), dtype=np.int32) for a in names]
        setup = self.dev._L.dnlp_batch_kkt_setup_qn if quasi_newton else self.dev._L.dnlp_batch_kkt_setup
        self.dev.check(setup(self.dev.h, int(sr.size), sr.ctypes.data_as(_cabi.c_i32p),
                             *[a.ctypes.data_as(_cabi.c_i32p) for a in pats]))
        self.kkt_N = self.n + int(sr.size)
        self.kkt_ms = 0.0
        self.qn_ms = 0.0

    def qn_update(self, starts, S, Y):
        """Damped BFGS update of the quasi-Newton matrices of the start ids ``starts`` with the steps ``S`` and the
        gradient changes ``Y`` (count, n) (the update of the test-suite's stand-in, include/dnlp_b200.h).  Returns
        ``applied`` (count,) bool: False where s'Ws > 0 fails and W is left as it was.  ``qn_ms`` keeps the
        CUDA-event time of the call's kernels."""
        st = np.ascontiguousarray(starts, dtype=np.int32).reshape(-1)
        cnt = st.size
        S = np.ascontiguousarray(S, dtype=np.float64).reshape(cnt, self.n)
        Y = np.ascontiguousarray(Y, dtype=np.float64).reshape(cnt, self.n)
        applied = np.zeros(cnt, dtype=np.int32)
        ms = C.c_float(0)
        self.dev.check(self.dev._L.dnlp_batch_qn_update(self.dev.h, int(cnt), st.ctypes.data_as(_cabi.c_i32p),
                                                        _ptr(S), _ptr(Y), applied.ctypes.data_as(_cabi.c_i32p),
                                                        C.byref(ms)))
        self.qn_ms = float(ms.value)
        return applied.astype(bool)

    def qn_matrix(self, start):
        """The quasi-Newton matrix of start ``start``, (n, n)."""
        out = np.empty((self.n, self.n))
        self.dev.check(self.dev._L.dnlp_batch_qn_matrix(self.dev.h, int(start), _ptr(out)))
        return out

    def kkt_solve(self, starts, sigma, dw, dc, rhs):
        """Assemble, factor (LDL', no pivoting) and solve the systems of the start ids ``starts`` from the JAC and
        HESS outputs the last device run left in HBM.  ``sigma`` (count, N), ``dw`` / ``dc`` (count,), ``rhs``
        (count, N + m).  Returns ``(sol, inertia, wquad)``: (count, N + m), (count, 3) int (n+, n-, n0) and
        dz' W dz; a row whose inertia is not (N, m, 0) or whose refined solution fails the residual test is NaN.
        ``kkt_ms`` keeps the CUDA-event time of the call's assembly + factorisation + solve."""
        N, M = self.kkt_N, self.kkt_N + self.m
        st = np.ascontiguousarray(starts, dtype=np.int32).reshape(-1)
        cnt = st.size
        sig = np.ascontiguousarray(sigma, dtype=np.float64).reshape(cnt, N)
        dw = np.ascontiguousarray(dw, dtype=np.float64).reshape(cnt)
        dc = np.ascontiguousarray(dc, dtype=np.float64).reshape(cnt)
        rhs = np.ascontiguousarray(rhs, dtype=np.float64).reshape(cnt, M)
        sol = np.empty((cnt, M))
        inertia = np.empty((cnt, 3), dtype=np.int32)
        wq = np.empty(cnt)
        ms = C.c_float(0)
        self.dev.check(self.dev._L.dnlp_batch_kkt_solve(
            self.dev.h, int(cnt), st.ctypes.data_as(_cabi.c_i32p), _ptr(sig), _ptr(dw), _ptr(dc), _ptr(rhs),
            _ptr(sol), inertia.ctypes.data_as(_cabi.c_i32p), _ptr(wq), C.byref(ms)))
        self.kkt_ms = float(ms.value)
        return sol, inertia, wq

    def kkt_matrix(self, start):
        """The assembled K of start ``start`` as the last ``kkt_solve`` left it, (N + m, N + m)."""
        M = self.kkt_N + self.m
        out = np.empty((M, M))
        self.dev.check(self.dev._L.dnlp_batch_kkt_matrix(self.dev.h, int(start), _ptr(out)))
        return out
