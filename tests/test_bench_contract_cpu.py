"""bench.py's single-GPU leg in the CPU tier: the workload builders, the timing / sizing control flow and the JSON line
(contract keys of the driver: metric, value, unit, e2e with byte counts, roofline with algorithmic bytes and fractions,
gpu_launches, clocks) with the tape executed by the interpreter-backed stand-in (tests/host_logic_device.py: fixed fake
timings, so the NUMBERS mean nothing here - the shape of the line and the SURVEY 8(d) byte accounting are under test)."""
import argparse
import os
import sys

import numpy as np
import pytest

import host_logic_device

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


@pytest.mark.parametrize("workload,scale", [("c3", 0.002), ("c5", 0.001), ("c2", 0.02), ("c1", 1.0)])
def test_single_gpu_bench_line(workload, scale, monkeypatch):
    import bench
    from dnlp_b200 import _cabi
    host_logic_device.install(monkeypatch)
    monkeypatch.setattr(_cabi, "device_synchronize", lambda *a: None)
    monkeypatch.setattr(bench, "TARGET_E2E_STEP_S", 0.05 / 3)
    args = argparse.Namespace(gpus=1, steps=3, warmup=3, workload=workload, scale=scale, impl="ours", no_cpu_baseline=True,
                              device_only=False, dump_outputs=None)
    grp = bench.Group(0, 1, 0)
    res = bench.bench_single(workload, args, grp, 6545.0, "test")
    for key in ("value", "unit", "ms_per_step", "evals_per_step", "ms_per_eval", "config", "clocks", "gpu_launches", "e2e",
                "roofline", "algorithmic_bytes_per_eval", "hbm_frac_whole_eval", "hbm_frac_whole_eval_of_8tbs_spec"):
        assert key in res, key
    assert res["unit"] == "evals/s" and res["value"] > 0 and res["gpu_launches"] > 0
    assert "workload" in res["config"] and "model" not in res["config"]
    e2e = res["e2e"]
    assert e2e["unit"] == "evals/s" and e2e["value"] > 0
    assert e2e["h2d_bytes_per_step"] > 0 and e2e["d2h_bytes_per_step"] > 0
    roof = res["roofline"]
    for key in ("bound", "achieved", "peak", "unit", "frac", "frac_of_8tbs_spec", "traffic", "algorithmic_bytes"):
        assert key in roof, key
    assert roof["bound"] == "hbm" and roof["peak"] == 6545.0
    assert np.isclose(roof["frac"], roof["achieved"] / 6545.0) and np.isclose(roof["frac_of_8tbs_spec"], roof["achieved"] / 8000.0)
    # SURVEY 8(d) byte accounting of the whole evaluation
    sizes = bench.sizes_of(workload, scale)
    assert res["algorithmic_bytes_per_eval"] == int(sum(bench.survey_bytes(workload, sizes).values()))


def test_multistart_bench_line_and_batched_oracles(monkeypatch):
    """C4 leg (starts split over the ranks, here one rank) and ``BatchedOracles`` itself: every start of the batch
    must equal the single-start oracle port; argument checks of the batched surface."""
    import bench
    from dnlp_b200 import _cabi
    from dnlp_b200 import workloads as W
    from dnlp_b200.multistart import BatchedOracles
    from golden_util import assert_close
    from oracle.dnlp_oracle import RefOracles
    host_logic_device.install(monkeypatch)
    monkeypatch.setattr(_cabi, "device_synchronize", lambda *a: None)
    monkeypatch.setattr(bench, "TARGET_E2E_STEP_S", 0.05 / 3)
    monkeypatch.setenv("DNLP_C4_BATCH", "6")
    args = argparse.Namespace(gpus=1, steps=3, warmup=3, workload="c4", scale=0.05, impl="ours", no_cpu_baseline=True,
                              device_only=False, dump_outputs=None)
    res = bench.bench_multistart(args, bench.Group(0, 1, 0), 6545.0, "test")
    for key in ("value", "unit", "ms_per_step", "config", "gpu_launches", "e2e", "roofline"):
        assert key in res, key
    assert res["e2e"]["h2d_bytes_per_step"] > 0 and res["e2e"]["d2h_bytes_per_step"] > 0
    # BatchedOracles against the single-start port
    P, q, rng = W.qcqp_data(12, 3)
    prob = W.qcqp(P, q)
    B = 5
    X, LAM, SIG = rng.uniform(-1, 1, (B, prob.n)), rng.standard_normal((B, prob.m)), rng.uniform(0.5, 1.5, B)
    bo = BatchedOracles(prob, B)
    out = bo.eval(X, LAM, SIG)
    ref = RefOracles(prob)
    np.testing.assert_array_equal(bo.jacobianstructure()[0], ref.jacobianstructure()[0])
    np.testing.assert_array_equal(bo.hessianstructure()[1], ref.hessianstructure()[1])
    assert out["f"].shape == (B,) and out["hess"].shape == (B, bo.nnz_hess)
    for b in range(B):
        assert_close(out["f"][b], ref.objective(X[b]), "f")
        assert_close(out["grad"][b], ref.gradient(X[b]), "grad")
        assert_close(out["g"][b], ref.constraints(X[b]), "g")
        assert_close(out["jac"][b], ref.jacobian(X[b]), "jac")
        assert_close(out["hess"][b], ref.hessian(X[b], LAM[b], SIG[b]), "hess")
    assert set(bo.eval(X, want=("f", "g"))) == {"f", "g"}
    with pytest.raises(ValueError):
        bo.eval(X[:-1], LAM, SIG)
    with pytest.raises(ValueError):
        bo.eval(X, want=("hess",))
    bo.close()


def _device_args(workload, scale, steps, dump=None):
    return argparse.Namespace(gpus=1, steps=steps, warmup=3, workload=workload, scale=scale, impl="ours", no_cpu_baseline=True,
                              device_only=True, dump_outputs=dump)


def test_steps_sets_the_number_of_timed_steps(monkeypatch):
    """--steps K times K steps of one size (the stand-in reports 0.05 ms per evaluation): twice the steps, the same
    step, twice the evaluations in the timed window.  The batched e2e leg runs K steps as well."""
    import bench
    from dnlp_b200 import _cabi
    host_logic_device.install(monkeypatch)
    monkeypatch.setattr(_cabi, "device_synchronize", lambda *a: None)
    res = {k: bench.bench_single("c1", _device_args("c1", 1.0, k), bench.Group(0, 1, 0), 6545.0, "test") for k in (3, 6)}
    assert res[3]["evals_per_step"] == res[6]["evals_per_step"] == round(bench.TARGET_STEP_S * 1e3 / 0.05)
    for k, r in res.items():
        assert r["ms_per_step"] == pytest.approx(0.05 * r["evals_per_step"])
        assert r["value"] == pytest.approx(k * r["evals_per_step"] / (k * r["ms_per_step"] * 1e-3))
    monkeypatch.setenv("DNLP_C4_BATCH", "3")
    args = argparse.Namespace(gpus=1, steps=4, warmup=3, workload="c4", scale=0.05, impl="ours", no_cpu_baseline=True,
                              device_only=False, dump_outputs=None)
    assert bench.bench_multistart(args, bench.Group(0, 1, 0), 6545.0, "test")["e2e"]["steps"] == 4


@pytest.mark.parametrize("workload,scale", [("c3", 0.002), ("c4", 0.05)])
def test_dump_outputs_are_the_last_timed_step(workload, scale, tmp_path, monkeypatch):
    """--dump-outputs writes the five outputs of the device-resident path at the bench's own seeded inputs, float64;
    an output longer than DUMP_MAX_ENTRIES is sampled at seeded positions that depend only on its length."""
    import bench
    from dnlp_b200 import _cabi
    from golden_util import assert_close
    from workload_cases import bench_dump_expected
    host_logic_device.install(monkeypatch)
    monkeypatch.setattr(_cabi, "device_synchronize", lambda *a: None)
    monkeypatch.setattr(bench, "DUMP_MAX_ENTRIES", 64)
    monkeypatch.setenv("DNLP_C4_BATCH", "3")
    run = bench.bench_multistart if workload == "c4" else (lambda a, *r: bench.bench_single(workload, a, *r))
    run(_device_args(workload, scale, 2, dump=str(tmp_path)), bench.Group(0, 1, 0), 6545.0, "test")
    want = bench_dump_expected(workload, scale, 64)
    assert sorted(os.listdir(tmp_path)) == sorted("%s_%s.npy" % (workload, p) for p in bench.PROGS)
    for p in bench.PROGS:
        got = np.load(tmp_path / ("%s_%s.npy" % (workload, p)))
        assert got.dtype == np.float64 and got.size <= 64
        assert_close(got, want[p], p, atol=1e-9 if p == "g" else 1e-12)
