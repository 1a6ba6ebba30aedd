"""The BASELINE configs as test cases: problem builders shared by the medium-golden and full-size tests."""
import hashlib
import os

import numpy as np

from dnlp_b200 import workloads as W

MEDIUM_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "medium")


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.int32).tobytes()).hexdigest()


def build(config, size="medium"):
    """ProblemIR of a BASELINE config at the medium-fixture size or at the full BASELINE size."""
    full = size == "full"
    if config == "c2":
        return W.eigen_qcqp(8192 if full else 1024)
    if config == "c3":
        m, n = (2_000_000, 4096) if full else (20000, 1024)
        At, x0 = W.logistic_data(m, n, 16)
        return W.logistic_regression(At, x0)
    if config == "c4":
        P, q, _ = W.qcqp_data(512, 8)
        return W.qcqp(P, q)
    if config == "c5":
        N = 10_000_000 if full else 100000
        A, x0 = W.microbench_data(N, N // 2, 10)
        return W.microbench(A, x0)
    raise KeyError(config)


def c4_starts(B=4096):
    _, _, rng = W.qcqp_data(512, 8)
    return rng.uniform(-1, 1, (B, 512))            # the stream SURVEY 8(d) C4 and bench.py use


class MediumGolden:
    def __init__(self, config):
        z = np.load(os.path.join(MEDIUM_DIR, config + "_medium.npz"), allow_pickle=False)
        self.z = z
        self.n, self.m = int(z["n"]), int(z["m"])
        self.nnz_jac, self.nnz_hess = int(z["nnz_jac"]), int(z["nnz_hess"])
        self.x0 = z["x0"]
        self.points = [{k: z["%s_%d" % (k, i)] for k in ("x", "lam", "sigma", "f", "grad", "g", "jac", "hess")}
                       for i in range(int(z["npoints"]))]
        self.starts = z["starts"] if "starts" in z.files else None

    def check_structure(self, jr, jc, hr, hc):
        assert jr.dtype == np.int32 and jc.dtype == np.int32 and hr.dtype == np.int32 and hc.dtype == np.int32
        assert (len(jr), len(hr)) == (self.nnz_jac, self.nnz_hess)
        for name, arr in (("jac_rows", jr), ("jac_cols", jc), ("hess_rows", hr), ("hess_cols", hc)):
            assert digest(arr) == str(self.z[name + "_sha256"]), "%s differs from the reference's" % name


def bench_dump_expected(workload, scale, max_entries):
    """What ``bench.py --dump-outputs`` must write for ``workload`` at ``scale`` (c4: DNLP_C4_BATCH starts): the CPU
    oracle port at the bench's seeded inputs, sampled as the bench samples an output longer than ``max_entries``."""
    import bench
    from oracle.dnlp_oracle import RefOracles
    if workload == "c4":
        s = bench.sizes_of("c4", scale)
        P, q, rng = W.qcqp_data(s["n"], s["k"])
        prob = W.qcqp(P, q)
        B = int(os.environ["DNLP_C4_BATCH"])
        X = rng.uniform(-1, 1, (B, s["n"]))
        LAM = np.random.default_rng(17).standard_normal((B, s["k"]))
        points = [(X[b], LAM[b], 1.0) for b in range(B)]
    else:
        prob = bench.build_workload(workload, scale)
        points = [bench.eval_point(prob, 0)]
    ref = RefOracles(prob)
    ref.jacobianstructure(), ref.hessianstructure()
    vals = {p: [] for p in bench.PROGS}
    with np.errstate(all="ignore"):
        for x, lam, sigma in points:
            for p, v in zip(bench.PROGS, (ref.objective(x), ref.gradient(x), ref.constraints(x), ref.jacobian(x),
                                          ref.hessian(x, lam, sigma))):
                vals[p].append(np.array(v, dtype=np.float64).ravel())
    out = {}
    for p, v in vals.items():
        a = np.concatenate(v)
        if a.size > max_entries:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, max_entries, replace=False))]
        out[p] = a
    return out
