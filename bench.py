#!/usr/bin/env python
"""Benchmark of the NLP oracle hot path: oracle evals/s for the set (f, grad f, g, J, Hess L).

    python bench.py --gpus N --steps K --warmup W [--workload all|c1|c2|c3|c4|c5] [--impl reference]
                    [--dump-outputs DIR]

Headline workload (every N): BASELINE config 3, the sparse logistic-type regression m = 2 M, n = 4096 -
the configuration the metric is quoted on "at 1/2/4/8 B200": one GPU evaluates it whole, N > 1 GPUs
evaluate it ROW-SHARDED (strong scaling; dnlp_b200/sharded.py + csrc/dnlp_shard.cu: local tapes, one-shot
all-reduce of the shared entries over NVLink peer memory).  `configs` carries the other BASELINE configs
as sub-results: c2 (dense eigen-QCQP, one GPU), c5 (10 M-node DAG + 50 M-nnz Jacobian, one GPU) and c4
(4096-start multi-start batch, starts split over the N ranks, no collective).

One STEP = `evals_per_step` evaluations of all five quantities, every cache invalidated before each
evaluation; `evals_per_step` is chosen so that one step lasts about 50 ms, and K timed steps are run.

--dump-outputs DIR writes what the device-resident path computed in its last timed step (the five
outputs of every workload run, DIR/<workload>_<output>.npy, float64), so that two builds can be
compared output for output: the inputs are seeded and the same for the same arguments.

  value     device-side throughput: (x, lambda, sigma) resident in HBM, CUDA events on the oracle's own
            stream, max over ranks.  N > 1: the exchange of shared entries is inside the timed region.
  e2e       the same set through the public drop-in object (the five cyipopt callbacks, HOST buffers in
            and out, H2D / D2H inside the timed region, a new x and a new lambda every evaluation).
  roofline  the dominant kernel: SURVEY.md 8(d)'s algorithmic bytes of the quantity it computes / its
            CUDA-event duration, against the measured HBM copy bandwidth (MEASURED_PEAKS.json);
            `hbm_frac_whole_eval` = 8(d)'s bytes of the whole evaluation / device time per evaluation.
  cpu_baseline / --impl reference
            the UNMODIFIED reference (oracle/_ref: cvxgrp/DNLP's own chain and Oracles) on bounded
            samples of the same workload, on this box's host cores, extrapolated to the full size with
            the per-triplet cost fitted on two sample sizes (stated in `sample`).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

PROGS = ("f", "grad", "g", "jac", "hess")
METRIC = "oracle evals/s (f, grad f, g, J, Hess L)"
# MEASURED_PEAKS.json has no fp64 figure; cuBLAS DGEMM 4096^3 on this pool's B200 (tools/cublas_dgemm_ref.py,
# profiles/r01_cublas_dgemm.txt) reached 35.4 TFLOP/s, 27.3 at the C4 shape [512x512]x[512x4096].
FP64_TENSOR_PEAK = 35.4
FP64_TENSOR_PEAK_SRC = "measured: cuBLAS DGEMM 4096^3 on this pool (profiles/r01_cublas_dgemm.txt); nominal 40"
TARGET_STEP_S = 0.05          # one timed step of the device leg should last about this long
HBM_SPEC_GBS = 8000.0            # the nominal figure north_star quotes next to the measured copy bandwidth
TARGET_E2E_STEP_S = 0.03      # one timed step of the e2e leg
DUMP_MAX_ENTRIES = 1 << 18    # --dump-outputs: entries kept per output (5 workloads x 5 outputs x 2 MB < 64 MB)


# ------------------------------------------------------------------ workloads
def sizes_of(name, scale=1.0):
    if name == "c1":
        return {"n": 3}
    if name == "c2":
        return {"n": max(8, int(round(8192 * scale)))}
    if name == "c3":
        return {"m": max(64, int(2_000_000 * scale)), "n": max(16, int(4096 * (scale ** 0.5))), "k": 16}
    if name == "c4":
        return {"n": max(16, int(512 * scale)), "k": 8, "B": max(1, int(4096 * scale))}
    if name == "c5":
        N = max(64, int(10_000_000 * scale) // 8 * 8)
        return {"N": N, "m": max(8, N // 2), "k": 10}
    raise SystemExit("unknown workload %r" % name)


def describe_workload(name, scale=1.0):
    s = sizes_of(name, scale)
    if name == "c1":
        return "c1: README toy eigen-QCQP n=3"
    if name == "c2":
        return ("c2: eigen-QCQP maximize quad_form(x,A) s.t. sum_squares(x)==1, dense A n=%d, single start" % s["n"])
    if name == "c3":
        return ("c3: sparse logistic-type regression m=%d n=%d, 16 nnz/row (lifted smooth form)" % (s["m"], s["n"]))
    if name == "c4":
        return ("c4: multi-start batch of %d random starts of a nonconvex QCQP n=%d, %d quadratic constraints; "
                "one eval = one start's full set" % (s["B"], s["n"], s["k"]))
    if name == "c5":
        return "c5: %d-node elementwise DAG + %d-nnz CSR constraint Jacobian" % (s["N"], s["m"] * s["k"])
    return name


def build_workload(name, scale=1.0):
    """ProblemIR of a single-GPU workload."""
    from dnlp_b200 import workloads as W
    s = sizes_of(name, scale)
    if name in ("c1", "c2"):
        return W.eigen_qcqp(s["n"])
    if name == "c3":
        At, x0 = W.logistic_data(s["m"], s["n"], s["k"])
        return W.logistic_regression(At, x0)
    if name == "c5":
        A, x0 = W.microbench_data(s["N"], s["m"], s["k"])
        return W.microbench(A, x0)
    raise SystemExit("unknown workload %r" % name)


def survey_bytes(name, s):
    """SURVEY.md section 8(d): algorithmic bytes of one evaluation, per quantity."""
    if name in ("c1", "c2"):
        n = s["n"]
        nnzh = n * (n + 1) // 2
        return {"f+grad": 8 * n * n + 16 * n, "g": 8 * n, "J": 16 * n, "H": 16 * nnzh}
    if name == "c3":
        m, n = s["m"], s["n"]
        nnz = m * s["k"]
        return {"g": 12 * nnz + 4 * m + 8 * m + 8 * m, "f+grad": 16 * m, "H": 16 * m, "J": 16 * n}
    if name == "c5":
        N, m = s["N"], s["m"]
        nnz = m * s["k"]
        return {"g": 12 * nnz + 4 * (m + 1) + 8 * N + 8 * m, "J": 20 * nnz + 8 * N,
                "H": 12 * nnz + 8 * m + 8 * N + 8 * N, "f+grad": 16 * N}
    return {}


def eval_point(prob, seed):
    rng = np.random.default_rng(1000 + seed)
    x = np.asarray(prob.x0, dtype=np.float64) * (1.0 + 0.01 * rng.standard_normal(prob.n))
    lam = rng.standard_normal(prob.m)
    return x, lam, 1.0


# (main sample scale, second sample scale) of the reference arm per workload
REF_SAMPLES = {"c2": (0.125, 0.0625), "c3": (0.1, 0.05), "c5": (0.01, 0.005)}


def reference_sample_note(name):
    sc = REF_SAMPLES.get(name)
    if sc is None:
        return "full size"
    return ("reference arm: the unmodified reference at %g and %g of the full size, extrapolated with the fitted "
            "per-triplet cost" % sc)


def config_of(name, world, scale=1.0):
    """The `config` object: a pure function of (workload, N) so that both arms print the same one."""
    if name == "c3" and world > 1:
        par = ("row-sharded x%d: rows of A~ (with their lifted variables, constraint rows and Jacobian / Hessian "
               "slots) block-distributed, x replicated; shared entries all-reduced over NVLink peer memory" % world)
    elif name == "c4":
        par = "starts split over %d GPU(s), no collective" % world
    else:
        par = "single GPU" if world == 1 else "single GPU per problem (replicas only)"
    return {"workload": describe_workload(name, scale), "parallelism": par,
            "l2": "working set fits L2; no flush" if name == "c1" else "inputs larger than L2 (126 MB); no flush needed",
            "reference_sample": reference_sample_note(name)}


# ------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self._stop = index, [], threading.Event()
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                if out.returncode == 0 and out.stdout.strip():
                    self.rows.append([c.strip() for c in out.stdout.strip().split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self.t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for i, nm in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": int(self.rows[0][1]) if self.rows[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


# ------------------------------------------------------------------ the reference on host cores
def full_work(name):
    """Triplet work units of the FULL workload (Jacobian + 2 x Hessian entries + n + m), analytically."""
    s = sizes_of(name)
    if name == "c2":
        n = s["n"]
        return n + 2 * (n * (n + 1) // 2) + n + 1
    if name == "c3":
        m, n = s["m"], s["n"]
        return (s["k"] * m + m + 4 * n) + 2 * (m + 3 * n) + (m + 3 * n) + (m + 2 * n)
    if name == "c5":
        N, m = s["N"], s["m"]
        return s["k"] * m + 2 * N + N + m
    return None


def reference_evals_per_s(name, steps, warmup, budget_s):
    """The unmodified reference (oracle/_ref) on samples of `name`; returns (value for the FULL workload,
    measured seconds per step of the main sample, info dict)."""
    from oracle import ref_driver as R
    if not R.available():
        return port_evals_per_s(name, budget_s)
    if name == "c4":
        prob, desc = R.build("c4", 1.0)
        T = R.TimedReference(prob)
        for _ in range(max(1, warmup)):
            T.step()
        ts = [T.step() for _ in range(max(3, steps))]
        per = float(np.mean(ts))
        return 1.0 / per, per, {"kind": "reference", "steps_run": len(ts),
                                "sample": "one start of the same QCQP (%s), %d full evals, %.4f s/eval; starts are independent, "
                                "so the reference's serial best_of loop evaluates them one by one" % (desc, len(ts), per)}
    if name == "c1":
        T = R.TimedReference(R.build("c1", 1.0)[0])
        ts = [T.step() for _ in range(max(3, steps) + warmup)][warmup:]
        per = float(np.mean(ts))
        return 1.0 / per, per, {"kind": "reference", "sample": "full size (n=3), %d evals" % len(ts), "steps_run": len(ts)}
    sc_main, sc_2nd = REF_SAMPLES[name]
    prob, desc = R.build(name, sc_main)
    T = R.TimedReference(prob)
    t_used, ts = 0.0, []
    for _ in range(warmup):
        t_used += T.step()
    for _ in range(steps):
        dt = T.step()
        ts.append(dt)
        t_used += dt
        if t_used > budget_s and len(ts) >= 3:
            break
    per_main = float(np.mean(ts))
    prob2, desc2 = R.build(name, sc_2nd)
    T2 = R.TimedReference(prob2)
    T2.step()
    per_2nd = float(np.mean([T2.step() for _ in range(3)]))
    # t = a + b * work fitted on the two sizes; a < 0 (super-linear growth) falls back to pure scaling
    b = (per_main - per_2nd) / max(T.work - T2.work, 1)
    a = per_main - b * T.work
    wf = full_work(name)
    pred = a + b * wf if (a >= 0 and b > 0) else per_main * wf / T.work
    info = {"kind": "reference",
            "sample": "%s: %s, %d evals, %.4f s/eval (work %d triplets); %s: %.4f s/eval (work %d); fitted %.3f us/triplet "
                      "+ %.4f s -> %.2f s/eval at the full size (work %d); structure passes %.1f s not counted"
                      % (name, desc, len(ts), per_main, T.work, desc2, per_2nd, T2.work, b * 1e6, max(a, 0.0), pred, wf,
                         T.structure_s),
            "seconds_per_eval_main_sample": per_main, "seconds_per_eval_second_sample": per_2nd,
            "extrapolated_seconds_per_eval_full": pred, "steps_run": len(ts)}
    return 1.0 / pred, per_main, info


def port_evals_per_s(name, budget_s):
    """Fallback when oracle/_ref did not travel: the CPU oracle port (oracle/dnlp_oracle.py) on a sample."""
    from oracle.dnlp_oracle import RefOracles
    scale = {"c1": 1.0, "c2": 0.125, "c3": 0.01, "c5": 0.01, "c4": 1.0}[name]
    if name == "c4":
        from dnlp_b200 import workloads as W
        P, q, _ = W.qcqp_data(512, 8)
        prob = W.qcqp(P, q)
    else:
        prob = build_workload(name, scale)
    o = RefOracles(prob)
    jr, _ = o.jacobianstructure()
    hr, _ = o.hessianstructure()
    x, lam, sigma = eval_point(prob, 0)
    reps, t_total = 0, 0.0
    with np.errstate(all="ignore"):
        while reps < 3 or (t_total < budget_s and reps < 50):
            t0 = time.perf_counter()
            o.objective(x), o.gradient(x), o.constraints(x), o.jacobian(x), o.hessian(x, lam, sigma)
            t_total += time.perf_counter() - t0
            reps += 1
    per = t_total / reps
    work = len(jr) + 2 * len(hr) + prob.n + prob.m
    wf = full_work(name) or work
    pred = per * wf / work
    return 1.0 / pred, per, {"kind": "port", "steps_run": reps,
                             "sample": "oracle/_ref absent: CPU oracle PORT at scale %g, %d evals, %.4f s/eval, scaled x%.1f "
                             "by triplet count" % (scale, reps, per, wf / work)}


# ------------------------------------------------------------------ measurement helpers
class Group:
    """Process-group plumbing of the bench: the package's own stdlib rendezvous (no torch)."""

    def __init__(self, rank, world, local_rank):
        from dnlp_b200 import _cabi
        from dnlp_b200.comm import SocketStore
        self.rank, self.world, self.local_rank = rank, world, local_rank
        self.store = SocketStore(rank, world) if world > 1 else None
        self._cabi = _cabi

    def barrier(self):
        self._cabi.device_synchronize(self.local_rank)
        if self.store is not None:
            self.store.allgather(b"")
        self._cabi.device_synchronize(self.local_rank)

    def max(self, values):
        v = np.asarray(values, dtype=np.float64)
        if self.store is None:
            return v
        from dnlp_b200.comm import allreduce_max
        return allreduce_max(self.store, v)

    def sum(self, values):
        v = np.asarray(values, dtype=np.float64)
        if self.store is None:
            return v
        from dnlp_b200.comm import allreduce_sum
        return allreduce_sum(self.store, v)

    def close(self):
        if self.store is not None:
            self.store.close()


def timed_device(run, grp, steps, warmup, clock_index):
    """run(n) -> ms of n back-to-back device-resident evaluations.  Returns (ms of the K timed steps (max over
    ranks), evals_per_step, clocks)."""
    run(3)
    probe = max(float(grp.max([run(8) / 8.0])[0]), 1e-4)                 # ms per evaluation
    E = max(1, int(math.ceil(TARGET_STEP_S * 1e3 / probe)))
    nwarm = max(warmup, 3) * E
    run(nwarm if nwarm * probe < 2000 else max(3, int(2000 / probe)))
    grp.barrier()
    with ClockSampler(clock_index) as clk:
        ms = run(steps * E)
        grp.barrier()
    ms = float(grp.max([ms])[0])
    return ms, E, clk.summary()


def timed_e2e(five, grp, steps):
    """five(i) = one evaluation through the public callbacks.  Returns (seconds of the K timed steps, evals/step)."""
    for i in range(2):
        five(i)
    grp.barrier()
    t0 = time.perf_counter()
    five(2), five(3)
    probe = float(grp.max([(time.perf_counter() - t0) / 2.0])[0])
    E = max(1, int(math.ceil(TARGET_E2E_STEP_S / max(probe, 1e-6))))
    grp.barrier()
    t0 = time.perf_counter()
    for i in range(steps * E):
        five(i)
    dt = time.perf_counter() - t0
    grp.barrier()
    return float(grp.max([dt])[0]), E


def parity_excess(got, want, rtol=1e-10, atol_rel=1e-12):
    """max over entries of |got - want| / (rtol * |want| + atol_rel * max|want|): <= 1 means "equal within the
    test-suite's tolerance" (rel 1e-10; entries that cancel to ~0 are judged against the vector's own scale)."""
    a, b = np.asarray(got, np.float64).ravel(), np.asarray(want, np.float64).ravel()
    if a.size == 0:
        return 0.0
    scale = float(np.max(np.abs(b))) if b.size else 0.0
    return float(np.max(np.abs(a - b) / (rtol * np.abs(b) + atol_rel * max(scale, 1e-300) + 1e-300)))


def dump_outputs(dump_dir, workload, read):
    """--dump-outputs: read(p) is output p of the last timed step; written as DIR/<workload>_<p>.npy (float64).  An output
    longer than DUMP_MAX_ENTRIES is sampled at seeded positions that depend only on its length, so two builds of the same
    workload keep the same entries."""
    os.makedirs(dump_dir, exist_ok=True)
    for p in PROGS:
        a = np.asarray(read(p), dtype=np.float64).ravel()
        if a.size > DUMP_MAX_ENTRIES:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ENTRIES, replace=False))]
        np.save(os.path.join(dump_dir, "%s_%s.npy" % (workload, p)), a)


def load_traffic(workload, kname):
    for fn in ("r02_ncu_traffic.json", "r01_ncu_traffic.json"):
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", fn)))
            t = tj.get(workload, {}).get(kname, {}).get("dram_bytes_per_launch_max")
            if t:
                return t, "profiles/%s (ncu --set full, dram read+write per launch)" % fn
        except Exception:
            pass
    return None, None


def roofline_of(o, name, sizes, hbm_peak, peak_src):
    """Dominant kernel of the union program: CUDA events around every instruction."""
    tape = o.tape
    per = o.profile_instrs("all", iters=3)
    if os.environ.get("DNLP_BENCH_PROFILE"):
        names = {1: "elem", 2: "poly", 3: "gemv", 4: "scale"}
        for i in tape.programs["all"]:
            ii = tape.instrs[i]
            nb = ii.nbytes_algorithmic()
            sys.stderr.write("[%s instr %3d] %-5s dst=%d rows=%-9d terms=%-9d %8.4f ms %8.1f GB/s  %s\n" % (
                name, i, names.get(ii.kind, "?"), ii.dst_space, ii.count, 0 if ii.coef is None else ii.coef.size,
                per[i], nb / max(per[i], 1e-9) / 1e6, o.instr_kernel(i)))
    top = int(np.argmax(per))
    ins = tape.instrs[top]
    kname = o.instr_kernel(top)
    sb = survey_bytes(name, sizes)
    nterms = 0 if ins.coef is None else int(ins.coef.size)
    nnz = sizes.get("m", 0) * sizes.get("k", 0)
    quantity = None
    if ins.kind == 3:
        quantity = "f+grad"
    elif ins.kind == 4 and ins.dst_space == 5:
        quantity = "H"
    elif getattr(ins, "fused_jac", None) is not None:
        quantity = "g+J"
    elif ins.kind == 2 and ins.dst_space == 3 and nterms >= nnz > 0:
        quantity = "g"
    elif ins.kind == 2 and ins.dst_space == 4 and nterms >= nnz > 0:
        quantity = "J"
    elif ins.kind == 2 and ins.dst_space == 5 and nterms >= nnz > 0:
        quantity = "H"
    if quantity == "g+J" and "g" in sb:
        alg, src = sb["g"] + sb["J"], "SURVEY 8(d): quantities g + J of this config (one fused kernel)"
    elif quantity and quantity in sb:
        alg, src = sb[quantity], "SURVEY 8(d): quantity '%s' of this config" % quantity
    else:
        alg, src = ins.nbytes_algorithmic(), "tape-derived (streams + one pass over the gathered slots)"
    achieved = alg / (per[top] * 1e-3) / 1e9 if per[top] > 0 else 0.0
    traffic, tsrc = load_traffic(name, kname)
    return {"bound": "hbm", "kernel": "%s (instr %d, %d rows, %d terms)" % (kname, top, ins.count, nterms),
            "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
            "frac_of_8tbs_spec": achieved / HBM_SPEC_GBS, "traffic": traffic,
            "traffic_source": tsrc, "algorithmic_bytes": int(alg), "algorithmic_bytes_source": src,
            "ms": float(per[top]), "peak_source": peak_src, "share_of_step": float(per[top] / max(per.sum(), 1e-12))}


# ------------------------------------------------------------------ single-GPU tape workloads (c1, c2, c3, c5)
def bench_single(name, args, grp, hbm_peak, peak_src):
    """One GPU evaluates the whole problem.  Returns the result dict."""
    from dnlp_b200.oracles import GpuOracles
    sizes = sizes_of(name, args.scale)
    t0 = time.time()
    prob = build_workload(name, args.scale)
    tape, tape_file = None, None
    if os.environ.get("DNLP_TAPE_CACHE"):
        import pickle
        tape_file = os.path.join(os.environ["DNLP_TAPE_CACHE"], "tape_%s_%g.pkl" % (name, args.scale))
        if os.path.exists(tape_file):
            tape = pickle.load(open(tape_file, "rb"))
    o = GpuOracles(prob, device=grp.local_rank, tape=tape)
    compile_s = time.time() - t0
    if tape_file and tape is None:
        import pickle
        pickle.dump(o.tape, open(tape_file, "wb"), protocol=4)
    sys.stderr.write("[bench] %s: built + compiled in %.1f s, n=%d m=%d nnzJ=%d nnzH=%d, %d instructions\n"
                     % (describe_workload(name, args.scale), compile_s, prob.n, prob.m, o.nnz_jac, o.nnz_hess,
                        len(o.tape.instrs)))
    x, lam, sigma = eval_point(prob, 0)
    o.upload_point(x, lam, sigma)
    l0 = o.kernel_launches()
    solo = Group(0, 1, grp.local_rank)
    ms, E, clocks = timed_device(lambda n: o.run_device(PROGS, n), solo, args.steps, args.warmup, grp.local_rank)
    launches = o.kernel_launches() - l0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, name, o.read_output)
    per_eval_ms = ms / (args.steps * E)
    sys.stderr.write("[bench] %s device: %.4f ms/eval (%d evals per step)\n" % (name, per_eval_ms, E))
    sb = survey_bytes(name, sizes)
    total_8d = int(sum(sb.values()))
    res = {"value": args.steps * E / (ms * 1e-3), "unit": "evals/s", "ms_per_step": ms / args.steps, "evals_per_step": E,
           "ms_per_eval": per_eval_ms, "config": config_of(name, 1, args.scale), "clocks": clocks,
           "gpu_launches": int(launches), "compile_s": round(compile_s, 2), "nnz_jac": o.nnz_jac, "nnz_hess": o.nnz_hess,
           "algorithmic_bytes_per_eval": total_8d, "algorithmic_bytes_per_quantity": sb,
           "algorithmic_bytes_source": "SURVEY.md 8(d)",
           "hbm_gbs_whole_eval": total_8d / (per_eval_ms * 1e-3) / 1e9,
           "hbm_frac_whole_eval": total_8d / (per_eval_ms * 1e-3) / 1e9 / hbm_peak,
           "hbm_frac_whole_eval_of_8tbs_spec": total_8d / (per_eval_ms * 1e-3) / 1e9 / HBM_SPEC_GBS}
    if not args.device_only:
        rng = np.random.default_rng(7)
        npts = 4
        xs = [x * (1.0 + 1e-3 * rng.standard_normal(prob.n)) for _ in range(npts)]
        lams = [lam * (1.0 + 1e-3 * rng.standard_normal(prob.m)) for _ in range(npts)]

        def five(i, sg=sigma):
            xi, li = xs[i % npts], lams[i % npts]
            o.objective(xi), o.gradient(xi), o.constraints(xi), o.jacobian(xi), o.hessian(xi, li, sg)
        dt, E2 = timed_e2e(five, solo, args.steps)
        full = {"grad": prob.n, "g": prob.m, "jac": o.nnz_jac, "hess": o.nnz_hess}
        d2h = 8 * (1 + sum(o._dyn[k][0].size if k in o._dyn else v for k, v in full.items()))
        res["e2e"] = {"value": args.steps * E2 / dt, "unit": "evals/s", "evals_per_step": E2,
                      "h2d_bytes_per_step": int(E2 * (prob.n * 8 + (prob.m + 1) * 8)), "d2h_bytes_per_step": int(E2 * d2h),
                      "api": "GpuOracles.objective/gradient/constraints/jacobian/hessian (5 callbacks, host buffers)",
                      "inputs": "new x and new lambda every evaluation, sigma = 1.0 (IPOPT's calling pattern)",
                      "d2h_bytes_per_eval_without_elision": int(8 * (1 + prob.n + prob.m + o.nnz_jac + o.nnz_hess))}
        if name == "c2":
            # worst case for the sigma-keyed Hessian entries: the objective factor changes every evaluation
            five(0, 0.5)
            t0 = time.perf_counter()
            for i in range(6):
                five(i, 1.0 if i % 2 else 0.5)
            res["e2e"]["sigma_changing_every_eval_value"] = 6 / (time.perf_counter() - t0)
        cb_iters = 5
        o.upload_point(x, lam, sigma)
        res["per_callback"] = {"device_ms_nothing_cached": {p: o.run_device((p,), cb_iters) / cb_iters for p in PROGS}}
    res["roofline"] = roofline_of(o, name, sizes, hbm_peak, peak_src)
    o.close()
    return res


# ------------------------------------------------------------------ C3 row-sharded over N GPUs
def bench_c3_sharded(args, grp, hbm_peak, peak_src):
    from dnlp_b200 import workloads as W
    from dnlp_b200.oracles import GpuOracles
    from dnlp_b200.sharded import GlobalStructure, RowShardedOracles, shard_logistic_regression
    s = sizes_of("c3", args.scale)
    rank, world = grp.rank, grp.world
    t0 = time.time()
    At, x_init = W.logistic_data(s["m"], s["n"], s["k"])
    glob = W.logistic_regression(At, x_init)
    local, layout = shard_logistic_regression(At, x_init, rank, world)
    gs = GlobalStructure.from_problem(glob)
    o = RowShardedOracles(local, layout, gs, store=grp.store, device=grp.local_rank, workers="try")
    if o.has_worker_loop:
        o.set_worker_loop(False)                  # parity check and device-resident loop: every rank calls (SPMD)
    setup_s = time.time() - t0
    x, lam, sigma = eval_point(glob, 0)
    # ---- inline parity: the sharded result against the single-GPU oracle of the global problem -------------
    ref = GpuOracles(glob, device=grp.local_rank) if rank == 0 else None
    grp.barrier()
    got = {"f": o.objective(x), "grad": o.gradient(x), "g": o.constraints(x), "jac": o.jacobian(x),
           "hess": o.hessian(x, lam, sigma)}
    parity = {"checked": True, "against": "single-GPU GpuOracles of the global problem, same point, all five outputs"}
    if rank == 0:
        want = {"f": ref.objective(x), "grad": ref.gradient(x), "g": ref.constraints(x), "jac": ref.jacobian(x),
                "hess": ref.hessian(x, lam, sigma)}
        worst, worst_rel = 0.0, 0.0
        for k in got:
            worst = max(worst, parity_excess(got[k], want[k]))
            a, b = np.asarray(got[k], np.float64).ravel(), np.asarray(want[k], np.float64).ravel()
            worst_rel = max(worst_rel, float(np.max(np.abs(a - b)) / max(float(np.max(np.abs(b))), 1e-300)) if a.size else 0.0)
        parity["tolerance"] = "|got - want| <= 1e-10 |want| + 1e-12 max|want| per output (tests/golden_util.py)"
        parity["max_error_over_tolerance"] = worst
        parity["max_abs_err_over_output_scale"] = worst_rel
        parity["ok"] = bool(worst <= 1.0)
        ref.close()
    ok = bool(grp.sum([1.0 if (rank != 0 or parity["ok"]) else 0.0])[0] == world)
    if not ok:
        if rank == 0:
            emit(json.dumps({"metric": METRIC, "value": None, "error": "sharded result differs from the single-GPU result",
                              "parity": parity}))
        o.close()
        return None
    # ---- device-resident: local tapes + exchange of the shared entries ---------------------------------------
    xl, ll = x[layout.var_map], lam[layout.con_map]
    o.local.upload_point(xl, ll, sigma)
    l0 = o.local.kernel_launches()
    ms, E, clocks = timed_device(lambda n: o.run_device(PROGS, n), grp, args.steps, args.warmup, grp.local_rank)
    launches = o.local.kernel_launches() - l0
    per_eval_ms = ms / (args.steps * E)
    if rank == 0:
        sys.stderr.write("[bench] c3 row-sharded x%d: setup %.1f s, device %.4f ms/eval (%d evals per step)\n"
                         % (world, setup_s, per_eval_ms, E))
    e2e = None
    if not args.device_only:
        rng = np.random.default_rng(7)            # the same stream on every rank: the same global points
        npts = 4
        xs = [x * (1.0 + 1e-3 * rng.standard_normal(glob.n)) for _ in range(npts)]
        lams = [lam * (1.0 + 1e-3 * rng.standard_normal(glob.m)) for _ in range(npts)]

        def five(i):
            xi, li = xs[i % npts], lams[i % npts]
            o.objective(xi), o.gradient(xi), o.constraints(xi), o.jacobian(xi), o.hessian(xi, li, sigma)
        dt_spmd, E_spmd = timed_e2e(five, grp, args.steps)
        # the drop-in shape: ONE solver process (rank 0) issues the callbacks, the other ranks follow in serve()
        grp.barrier()
        one_solver = o.has_worker_loop
        if one_solver:
            o.set_worker_loop(True)
        if not one_solver:
            dt, E2 = 0.0, 0
        elif rank == 0:
            for i in range(2):
                five(i)
            t0 = time.perf_counter()
            five(2), five(3)
            probe = (time.perf_counter() - t0) / 2.0
            E2 = max(1, int(math.ceil(TARGET_E2E_STEP_S / max(probe, 1e-6))))
            t0 = time.perf_counter()
            for i in range(args.steps * E2):
                five(i)
            dt = time.perf_counter() - t0
            o.release_workers()
        else:
            o.serve()
            dt, E2 = 0.0, 0
        if one_solver:
            o.set_worker_loop(False)
        grp.barrier()
        dt, E2 = float(grp.max([dt])[0]), int(grp.max([E2])[0])
        h2d = float(grp.sum([8.0 * (layout.var_map.size + layout.con_map.size + 1)])[0])
        e2e = {"value": args.steps * E_spmd / dt_spmd, "unit": "evals/s", "evals_per_step": E_spmd,
               "mode": "every rank issues the five callbacks with its own host copies of x / lambda (SPMD, as the C4 "
                       "ranks do with their slices of the starts)",
               "one_solver_value": (args.steps * E2 / dt) if one_solver else None,
               "one_solver_evals_per_step": E2,
               "one_solver_note": "worker loop: rank 0 ALONE issues the callbacks (what one IPOPT process would do), "
                                  "posting x / lambda through shared host memory; the other ranks follow in "
                                  "RowShardedOracles.serve().  The root then reads all of x once per callback instead "
                                  "of its slice, which is the difference to `value`",
               "h2d_bytes_per_step": int(E_spmd * h2d),
               "d2h_bytes_per_step": int(E_spmd * 8 * (1 + glob.n + glob.m + gs.dynamic["jac"].size + gs.hess_rows.size)),
               "api": "RowShardedOracles five callbacks, host buffers; " + (
                   "outputs %s: every GPU copies the runs it owns over its own PCIe link into one host array shared by "
                   "the ranks (every rank returns the full output); the rest is stored into the root's device array over "
                   "NVLink and leaves the root in one D2H" % sorted(o._dev.shared) if o._dev.shared else
                   "owned entries are stored into the root's global array over NVLink, one D2H per callback leaves the root")}
    sb = survey_bytes("c3", s)
    total_8d = int(sum(sb.values()))
    local_sizes = dict(s, m=layout.con_map.size - (2 * s["n"] if rank == 0 else 0))
    roof = roofline_of(o.local, "c3", local_sizes, hbm_peak, peak_src) if rank == 0 else None
    res = None
    if rank == 0:
        res = {"value": args.steps * E / (ms * 1e-3), "unit": "evals/s", "ms_per_step": ms / args.steps, "evals_per_step": E,
               "ms_per_eval": per_eval_ms, "config": config_of("c3", world, args.scale), "clocks": clocks,
               "gpu_launches": int(launches), "setup_s": round(setup_s, 2), "parity": parity,
               "algorithmic_bytes_per_eval": total_8d, "algorithmic_bytes_source": "SURVEY.md 8(d)",
               "hbm_gbs_whole_eval": total_8d / (per_eval_ms * 1e-3) / 1e9,
               "hbm_frac_whole_eval": total_8d / (per_eval_ms * 1e-3) / 1e9 / (hbm_peak * world),
               "hbm_frac_whole_eval_of_8tbs_spec": total_8d / (per_eval_ms * 1e-3) / 1e9 / (HBM_SPEC_GBS * world),
               "hbm_frac_note": "against %d x the per-GPU measured peak" % world,
               "roofline": dict(roof, note="rank 0's local tape (its rows)"),
               "exchange": {"shared_entries": "f (1 double); everything else is owned by one rank",
                            "route": os.environ.get("DNLP_SHARD_ALLREDUCE", "auto")}}
        if e2e:
            res["e2e"] = e2e
    o.close()
    return res


# ------------------------------------------------------------------ C4: batched multi-start QCQP
def bench_multistart(args, grp, hbm_peak, peak_src):
    """4096 random starts of a nonconvex QCQP (n=512, 8 quadratic constraints); the batch is split
    evenly over the ranks (no collective).  One evaluation = one start's (f, grad, g, J, Hess L)."""
    from dnlp_b200 import workloads as W
    from dnlp_b200.multistart import BatchedOracles
    from dnlp_b200.oracles import GpuOracles
    rank, world = grp.rank, grp.world
    s = sizes_of("c4", args.scale)
    n, k = s["n"], s["k"]
    Btot = int(os.environ.get("DNLP_C4_BATCH", max(world, s["B"])))
    P, q, rng = W.qcqp_data(n, k)
    prob = W.qcqp(P, q)
    X = rng.uniform(-1, 1, (Btot, n))                       # the same rng stream as SURVEY 8(d) C4
    b0, b1 = (Btot * rank) // world, (Btot * (rank + 1)) // world
    B = b1 - b0
    LAM = np.random.default_rng(17).standard_normal((Btot, k))[b0:b1]
    SIG = np.ones(B)
    o = BatchedOracles(prob, B, device=grp.local_rank)
    # inline parity: first and last start of this rank's slice against the single-start oracle on this GPU
    single = GpuOracles(prob, device=grp.local_rank)
    res0 = o.eval(X[b0:b1], LAM, SIG)
    worst = 0.0
    for j in sorted({0, B - 1}):
        want = {"f": single.objective(X[b0 + j]), "grad": single.gradient(X[b0 + j]), "g": single.constraints(X[b0 + j]),
                "jac": single.jacobian(X[b0 + j]), "hess": single.hessian(X[b0 + j], LAM[j], 1.0)}
        for kk, w in want.items():
            worst = max(worst, parity_excess(res0[kk][j], w))
    single.close()
    del res0
    worst = float(grp.max([worst])[0])
    parity = {"checked": True, "against": "single-start GpuOracles at the first and last start of every rank's slice",
              "tolerance": "|got - want| <= 1e-10 |want| + 1e-12 max|want| per output (tests/golden_util.py)",
              "max_error_over_tolerance": worst, "ok": bool(worst <= 1.0)}
    o.upload(X[b0:b1], LAM, SIG)
    l0 = o.kernel_launches()
    ms, E, clocks = timed_device(lambda m_: o.run_device(PROGS, m_), grp, args.steps, args.warmup, grp.local_rank)
    launches = o.kernel_launches() - l0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, "c4", o.read_output)
    e2e = None
    if not args.device_only:
        o.eval(X[b0:b1], LAM, SIG)
        grp.barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            o.eval(X[b0:b1], LAM, SIG)
        dt = float(grp.max([time.perf_counter() - t0])[0])
        e2e = {"value": Btot * args.steps / dt, "unit": "evals/s", "api": "BatchedOracles.eval (host arrays in/out)",
               "h2d_bytes_per_step": int(8 * Btot * (n + k + 1)),
               "d2h_bytes_per_step": int(8 * Btot * (1 + n + k + o.nnz_jac + o.nnz_hess)), "steps": args.steps}
    res = None
    if rank == 0:
        per = o.profile_instrs("all", iters=2)
        if os.environ.get("DNLP_BENCH_PROFILE"):
            for i in o.tape.programs["all"]:
                ii = o.tape.instrs[i]
                sys.stderr.write("[binstr %3d] kind=%d dst=%d rows=%-8d terms=%-9d %8.4f ms\n" % (
                    i, ii.kind, ii.dst_space, ii.count, 0 if ii.coef is None else ii.coef.size, per[i]))
        gemm_ids = [i for i in o.tape.programs["all"] if o.tape.instrs[i].kind == 3]
        gemm_fl = float(sum(2.0 * o.tape.instrs[i].count * o.tape.instrs[i].ncols * B for i in gemm_ids))
        other_ms = float(sum(per[i] for i in o.tape.programs["all"] if i not in gemm_ids))
        step_ms = ms / (args.steps * E)
        groups = o.profile_gemm_groups(iters=5)
        gemm_ms_grouped = groups[0][0] if groups else max(step_ms - other_ms, 1e-9)
        hess_bytes = 8.0 * o.nnz_hess * B
        t_min = gemm_fl / (FP64_TENSOR_PEAK * 1e12) + hess_bytes / (hbm_peak * 1e9)
        top = int(np.argmax(per))
        ins = o.tape.instrs[top]
        if ins.kind == 3:
            roof = {"bound": "tensor", "kernel": "bgemm_dmma_kernel (grouped launch of %d maps [%dx%d]x[%dx%d])"
                    % (len(gemm_ids), ins.count, ins.ncols, ins.ncols, B),
                    "achieved": gemm_fl / (gemm_ms_grouped * 1e-3) / 1e12, "peak": FP64_TENSOR_PEAK, "unit": "TFLOP/s",
                    "frac": gemm_fl / (gemm_ms_grouped * 1e-3) / 1e12 / FP64_TENSOR_PEAK, "traffic": None,
                    "peak_source": FP64_TENSOR_PEAK_SRC, "ms": gemm_ms_grouped}
        else:
            nb = hess_bytes if ins.dst_space == 5 else ins.nbytes_algorithmic()
            roof = {"bound": "hbm", "kernel": "batched Hessian fill bsmallk_kernel (instr %d, %d rows x %d starts)"
                    % (top, ins.count, B),
                    "achieved": nb / (per[top] * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                    "frac": nb / (per[top] * 1e-3) / 1e9 / hbm_peak,
                    "frac_of_8tbs_spec": nb / (per[top] * 1e-3) / 1e9 / HBM_SPEC_GBS, "traffic": None, "peak_source": peak_src,
                    "algorithmic_bytes": int(nb), "algorithmic_bytes_source": "SURVEY 8(d) C4: 8 * nnzH * B output bytes",
                    "ms": float(per[top])}
        roof["share_of_step"] = float(per[top] / max(per.sum(), 1e-12))
        res = {"value": Btot * args.steps * E / (ms * 1e-3), "unit": "evals/s", "ms_per_step": ms / args.steps,
               "evals_per_step": E * Btot, "batches_per_step": E, "ms_per_batch": step_ms,
               "config": dict(config_of("c4", world, args.scale), starts_per_gpu=B), "clocks": clocks, "parity": parity,
               "gpu_launches": int(launches), "roofline": roof,
               "dmma": {"gemm_tflops_grouped_launch": gemm_fl / (gemm_ms_grouped * 1e-3) / 1e12,
                        "gemm_ms_grouped_launch": gemm_ms_grouped,
                        "gemm_tflops_individual_launches":
                            gemm_fl / max(float(sum(per[i] for i in gemm_ids)) * 1e-3, 1e-12) / 1e12,
                        "note": "the k+1 independent maps run as ONE grouped grid inside the step, timed on its own with "
                                "CUDA events (dnlp_batch_profile_groups)",
                        "peak_measured_tflops": FP64_TENSOR_PEAK, "peak_source": FP64_TENSOR_PEAK_SRC,
                        "cublas_same_shape_tflops": 27.3},
               "roofline_whole_batch": {"t_min_ms": t_min * 1e3, "frac": t_min * 1e3 / step_ms,
                                        "model": "GEMM flops / FP64 tensor peak + Hessian output bytes / HBM peak"}}
        if e2e:
            res["e2e"] = e2e
    o.close()
    return res


# ------------------------------------------------------------------ main
_RESULT_OUT = None


def emit(text):
    """The one JSON line, on the process's ORIGINAL stdout (see main: fd 1 itself is pointed at stderr)."""
    out = _RESULT_OUT if _RESULT_OUT is not None else sys.stdout
    out.write(text + "\n")
    out.flush()


def main():
    # stdout carries exactly one JSON line.  Libraries write banners straight to fd 1 (NCCL prints its version there
    # when the box sets NCCL_DEBUG=VERSION, and NCCL_DEBUG_FILE is not honoured at that level): keep a private handle
    # on the real stdout for the result and send everything else that lands on fd 1 to stderr.
    global _RESULT_OUT
    sys.stdout.flush()
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default=os.environ.get("DNLP_BENCH_WORKLOAD", "all"))
    ap.add_argument("--scale", type=float, default=float(os.environ.get("DNLP_BENCH_SCALE", "1.0")))
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--device-only", action="store_true",
                    help="profiling aid: only the device-resident step loop and the per-instruction timing")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed device step as DIR/<workload>_<output>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and (world > 1 or args.impl != "ours"):
        ap.error("--dump-outputs needs --impl ours in one process (WORLD_SIZE=1)")
    headline = "c3" if args.workload == "all" else args.workload
    subs = [w for w in os.environ.get("DNLP_BENCH_SUBS", "c4,c2,c5").split(",") if w] if args.workload == "all" else []

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"

    if args.impl == "reference":
        if rank != 0:
            return
        t_start = time.time()
        v, per, info = reference_evals_per_s(headline, args.steps, args.warmup, budget_s=150.0)
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "evals/s", "n_gpus": args.gpus,
                "steps": info.get("steps_run", args.steps), "warmup": args.warmup, "ms_per_step": per * 1e3,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config_of(headline, world, args.scale),
                "value_is": ("evals/s of the FULL workload, extrapolated from the sample steps actually run (ms_per_step is "
                             "the measured time of one sample step)") if headline in REF_SAMPLES else "measured at full size",
                "cpu_baseline": {"value": v, "unit": "evals/s", "cores": os.cpu_count(), "kind": info["kind"],
                                 "sample": info["sample"],
                                 "threads_note": "the reference is single-threaded Python; NumPy / BLAS may use the other "
                                                 "cores in dense products"},
                "e2e": {"value": v, "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "wall_s": round(time.time() - t_start, 1)}
        emit(json.dumps(line, default=float))
        return

    grp = Group(rank, world, local_rank)
    if headline == "c3" and world > 1:
        main_res = bench_c3_sharded(args, grp, hbm_peak, peak_src)
    elif headline == "c4":
        main_res = bench_multistart(args, grp, hbm_peak, peak_src)
    else:
        # a problem that does not shard (c1, c2, c5; c3 on one GPU): rank 0 measures, the others idle
        main_res = bench_single(headline, args, grp, hbm_peak, peak_src) if rank == 0 else None
    grp.barrier()
    sub_res = {}
    for w in subs:
        try:
            if w == "c4":
                r = bench_multistart(args, grp, hbm_peak, peak_src)
            elif world == 1:
                r = bench_single(w, args, grp, hbm_peak, peak_src)
            else:
                r = {"skipped": "%s does not shard (replicas only): see the N=1 line" % w} if rank == 0 else None
        except Exception as e:        # a sub-result must never take the headline down
            r = {"error": "%s: %s" % (type(e).__name__, e)} if rank == 0 else None
        grp.barrier()
        if rank == 0 and r is not None:
            sub_res[w] = r
    if rank == 0 and main_res is not None:
        line = {"metric": METRIC, "value": main_res["value"], "unit": "evals/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": main_res["ms_per_step"], "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic"}
        for k, v in main_res.items():
            if k not in ("value", "unit", "ms_per_step"):
                line[k] = v
        if args.device_only:
            line["e2e"] = None
            line["note"] = "--device-only profiling run: e2e legs skipped, not a bench line"
        if not args.no_cpu_baseline and not args.device_only:
            try:
                v, per, info = reference_evals_per_s(headline, steps=4, warmup=1, budget_s=25.0)
                line["cpu_baseline"] = {"value": v, "unit": "evals/s", "cores": os.cpu_count(), "kind": info["kind"],
                                        "sample": info["sample"]}
            except Exception as e:
                line["cpu_baseline"] = {"value": None, "error": "%s: %s" % (type(e).__name__, e)}
        line["ipopt_iters_per_s"] = None
        line["ipopt_iters_per_s_reason"] = ("cyipopt / libipopt are not installed in this image or on the GPU box and cannot "
                                            "be installed offline; tests/test_solver_in_the_loop.py runs the solver-level "
                                            "check as soon as `import cyipopt` succeeds")
        if sub_res:
            line["configs"] = sub_res
        emit(json.dumps(line, default=float))
    grp.barrier()
    grp.close()


if __name__ == "__main__":
    main()
