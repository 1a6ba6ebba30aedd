"""Lock-step interior-point best_of at the C4 shape: where the time of one outer iteration goes.

    python tools/lockstep_ipm_bench.py [--n 512] [--k 8] [--B 4096] [--numpy-B 4]

The problem and the starts are bench.py's C4 (workloads.qcqp_data(n, k), X0 = rng.uniform(-1, 1, (B, n)) on the same
rng stream).  The driver runs on BatchedOracles with the device KKT backend; per outer iteration it reports the wall
time of the oracle evaluations (the f / grad / g / J evaluation, the Jacobian + Hessian programs and every line-search
round), of the KKT backend (the CUDA-event time of assembly + factorisation + solve is given separately) and of the
host logic (the rest).  Then the first --numpy-B starts run again with the NumPy backend of the test-suite (the same
LDL' without pivoting, start by start on the host) for --numpy-iters outer iterations, to put both on one axis.  The GPU's name and power limit are read in
the same run.  The last line is one JSON object with every number.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gpu_identity():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [s.strip() for s in out.split(",")[:2]]
        return name, power
    except Exception:
        import torch
        return torch.cuda.get_device_name(0), "unknown"


def split(out, device_ms=None):
    T = out["timings"]
    it = len(T)
    ev = sum(t["eval_s"] for t in T) * 1e3
    kk = sum(t["kkt_s"] for t in T) * 1e3
    tot = sum(t["total_s"] for t in T) * 1e3
    r = {"outer_iterations": it, "per_iter_ms": {"oracle_evals": ev / it, "kkt_backend": kk / it,
                                                 "host_logic": (tot - ev - kk) / it, "total": tot / it}}
    if device_ms is not None:
        r["per_iter_ms"]["kkt_device_events"] = device_ms / it
    st, cnt = np.unique(out["status"], return_counts=True)
    r["status_histogram"] = {int(s): int(c) for s, c in zip(st, cnt)}
    its = out["iterations"]
    r["iterations"] = {"min": int(its.min()), "median": float(np.median(its)), "max": int(its.max())}
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=512)
    ap.add_argument("--k", type=int, default=8)
    ap.add_argument("--B", type=int, default=4096)
    ap.add_argument("--numpy-B", type=int, default=2)
    ap.add_argument("--numpy-iters", type=int, default=10, help="outer iterations of the NumPy-backend run")
    ap.add_argument("--max-iter", type=int, default=500)
    ap.add_argument("--verbose", action="store_true", help="one line per outer iteration")
    a = ap.parse_args()
    from dnlp_b200 import workloads as W
    from dnlp_b200.lockstep_ipm import DeviceKKT, lockstep_ipm
    from dnlp_b200.multistart import BatchedOracles
    name, power = gpu_identity()
    P, q, rng = W.qcqp_data(a.n, a.k)
    prob = W.qcqp(P, q)
    X0 = rng.uniform(-1, 1, (a.B, a.n))
    bnds = dict(lb=prob.lb, ub=prob.ub, cl=prob.cl, cu=prob.cu)
    result = {"gpu": name, "power_limit": power, "n": a.n, "k": a.k, "B": a.B, "M": a.n + 2 * a.k}
    ev = BatchedOracles(prob, a.B)
    try:
        kkt = DeviceKKT(ev)
        t0 = time.perf_counter()
        def show(it, t, n_active):
            print("  iteration %d: %d starts active, %.1f ms (evals %.1f, KKT %.1f)"
                  % (it, n_active, 1e3 * t["total_s"], 1e3 * t["eval_s"], 1e3 * t["kkt_s"]), flush=True)
        out = lockstep_ipm(ev, kkt, X0, max_iter=a.max_iter, progress=show if a.verbose else None, **bnds)
        result["device"] = split(out, kkt.device_ms)
        result["device"]["wall_s"] = time.perf_counter() - t0
    finally:
        ev.close()
    print("GPU: %s, power limit %s" % (name, power))
    d = result["device"]
    print("device backend, B=%d, N+m=%d: %d outer iterations in %.1f s; per iteration: oracle evals %.2f ms, KKT %.2f ms "
          "(CUDA events %.2f ms), host logic %.2f ms" % (a.B, result["M"], d["outer_iterations"], d["wall_s"],
                                                        d["per_iter_ms"]["oracle_evals"], d["per_iter_ms"]["kkt_backend"],
                                                        d["per_iter_ms"]["kkt_device_events"], d["per_iter_ms"]["host_logic"]))
    print("  status histogram %s, iterations %s" % (d["status_histogram"], d["iterations"]))
    if a.numpy_B > 0:
        from test_lockstep_ipm import NumpyKKT
        ev = BatchedOracles(prob, a.numpy_B)
        try:
            t0 = time.perf_counter()
            out = lockstep_ipm(ev, NumpyKKT(ev), X0[:a.numpy_B], max_iter=min(a.max_iter, a.numpy_iters), **bnds)
            result["numpy"] = split(out)
            result["numpy"]["wall_s"] = time.perf_counter() - t0
            result["numpy"]["B"] = a.numpy_B
        finally:
            ev.close()
        d = result["numpy"]
        print("NumPy backend, B=%d: %d outer iterations in %.1f s; per iteration: oracle evals %.2f ms, KKT %.2f ms, "
              "host logic %.2f ms" % (a.numpy_B, d["outer_iterations"], d["wall_s"], d["per_iter_ms"]["oracle_evals"],
                                      d["per_iter_ms"]["kkt_backend"], d["per_iter_ms"]["host_logic"]))
        print("  status histogram %s" % d["status_histogram"])
    print(json.dumps(result))


if __name__ == "__main__":
    main()
