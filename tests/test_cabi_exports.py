"""The C-ABI library loads and exports every symbol include/dnlp_b200.h declares (no compute)."""
import ctypes
import os
import re

from dnlp_b200 import _cabi, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "dnlp_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(dnlp_[a-z_0-9]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    build.build()
    lib = ctypes.CDLL(_cabi.LIB_PATH)
    names = declared_symbols()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), "missing export %s" % n
    assert sorted(_cabi.EXPORTS) == names


def test_no_silent_cpu_fallback():
    """Without a CUDA device creating an oracle must raise, never compute on the host."""
    import numpy as np
    import pytest
    from dnlp_b200 import ir
    from dnlp_b200.oracles import GpuOracles
    if _cabi.device_count() > 0:
        pytest.skip("CUDA device present")
    x = ir.Variable(3)
    prob = ir.ProblemIR(ir.sum(ir.exp(x)), [], x0=np.zeros(3))
    with pytest.raises(RuntimeError):
        GpuOracles(prob)


def test_null_handle_is_an_error_not_a_crash():
    """ADVICE r1: after close() the Python side passes NULL; every entry point must return non-zero
    (the wrapper then raises "oracle closed") instead of dereferencing it."""
    import ctypes as C
    import numpy as np
    build.build()
    L = _cabi.lib()
    x = np.zeros(4)
    out = np.zeros(4)
    p = x.ctypes.data_as(_cabi.c_f64p)
    q = out.ctypes.data_as(_cabi.c_f64p)
    assert L.dnlp_eval_f(None, p, q) != 0
    assert L.dnlp_eval_grad(None, p, q) != 0
    assert L.dnlp_eval_g(None, p, q) != 0
    assert L.dnlp_eval_jac(None, p, q) != 0
    assert L.dnlp_eval_hess(None, p, p, 1.0, q) != 0
    assert L.dnlp_eval_all(None, p, p, 1.0, q, q, q, q, q) != 0
    assert L.dnlp_run(None, 0, p, p, 1.0) != 0
    assert L.dnlp_upload_point(None, p, p, 1.0) != 0
    assert L.dnlp_batch_upload(None, p, p, p) != 0
    assert L.dnlp_kernel_launches(None) == -1
    assert L.dnlp_batch_kernel_launches(None) == -1
    assert L.dnlp_instr_kernel(None, 0) == b""
    assert L.dnlp_batch_instr_kernel(None, 0) == b""
    assert b"NULL" in L.dnlp_last_error(None)
    # the sharded oracle's host-side entry points (shared-host delivery, worker loop) as well
    import ctypes as C
    i64 = np.zeros(1, dtype=np.int64)
    p64 = i64.ctypes.data_as(_cabi.c_i64p)
    out, out2 = _cabi.c_f64p(), _cabi.c_f64p()
    prog, flags, sig = C.c_int32(0), C.c_int32(0), C.c_double(0.0)
    assert L.dnlp_shard_eval(None, 0, p, p, 1.0, q) != 0
    assert L.dnlp_shard_share_control(None, b"/dnlp_test_none", 0) != 0
    assert L.dnlp_shard_share_output(None, 2, b"/dnlp_test_none", 0, 1, p64, p64, p64, C.byref(out)) != 0
    assert L.dnlp_shard_share_inputs(None, b"/dnlp_test_x", b"/dnlp_test_l", 0, 1, 1, C.byref(out), C.byref(out2)) != 0
    assert L.dnlp_shard_post_command(None, 0, p, p, 1.0, 0, C.byref(flags)) != 0
    assert L.dnlp_shard_wait_command(None, 0.0, C.byref(prog), C.byref(sig), C.byref(flags)) != 0
    assert L.dnlp_shard_share_reset(None) != 0
    assert L.dnlp_shard_share_release(None, 0) != 0
    assert L.dnlp_shard_share_unlink(b"/dnlp_test_segment_that_does_not_exist") != 0
    assert b"NULL" in L.dnlp_shard_last_error(None)

    class _Dead(_cabi.DeviceTape):
        def __init__(self):
            self.h, self._L = None, L
    import pytest
    with pytest.raises(RuntimeError, match="oracle closed"):
        _Dead().check(L.dnlp_eval_f(None, p, q))


def test_duals_longer_than_m_are_accepted():
    """ADVICE r1: the reference slices duals[offset:offset+size] (nlp_solver.py:405-411); Knitro passes
    constraint and variable-bound multipliers in one vector (knitro_nlpif.py:284-291)."""
    import numpy as np
    import pytest
    from dnlp_b200.oracles import GpuOracles
    o = GpuOracles.__new__(GpuOracles)
    o.m = 3
    o._lam = np.zeros(3)
    lam = o._stage_lam(np.arange(8.0))
    assert lam.size == 3 and lam.flags.c_contiguous and np.array_equal(lam, [0.0, 1.0, 2.0])
    with pytest.raises(ValueError):
        o._stage_lam(np.zeros(2))
    o.dev = None
    o._handles = []


def test_int32_index_range_is_checked():
    """ADVICE r1: slots / positions are int32 on the device; a tape beyond that range must raise."""
    import numpy as np
    import pytest
    from dnlp_b200 import tape as T

    class _Big:
        size = 2 ** 31
    t = T.Tape(4, 0)
    t.jac_rows = t.jac_cols = np.zeros(0, np.int32)
    t.hess_rows = t.hess_cols = _Big()
    with pytest.raises(OverflowError):
        _cabi.make_tape_desc(t)
    t.hess_rows = t.hess_cols = np.zeros(0, np.int32)
    t.nslots = 2 ** 31 + 5
    with pytest.raises(OverflowError):
        _cabi.make_tape_desc(t)
