"""TEST INFRASTRUCTURE (CPU tier only): a stand-in for ``dnlp_b200._cabi.DeviceTape`` that executes the compiled tape
with the NumPy tape interpreter (tests/tape_interp.py) behind the SAME C entry-point names and ctypes arguments the
real library takes.  It exists so that the host logic of ``GpuOracles`` - constant-entry elision and the compact
dynamic transfers, the sigma-keyed Hessian entries, reused output buffers and return types, parameter re-arming,
argument checks - runs in ``-m "not gpu"`` too.  The product never imports this module: without the CUDA library or a
device, creating an oracle raises (dnlp_b200/_cabi.py)."""
import numpy as np

from tape_interp import TapeInterp

_SPACE_OF_PROG = {0: 1, 1: 2, 2: 3, 3: 4, 4: 5}
_NAME = {1: "f", 2: "grad", 3: "g", 4: "jac", 5: "hess"}


def _arr(ptr, count):
    return None if not ptr else np.ctypeslib.as_array(ptr, shape=(max(int(count), 1),))[:int(count)]


class _InterpLib:
    """The entry points ``GpuOracles`` calls, one instance per oracle (the handle argument is ignored)."""

    def __init__(self, tape):
        self.tape, self.it = tape, TapeInterp(tape)
        self.n, self.m = tape.n, tape.m
        self.len = {1: 1, 2: tape.n, 3: tape.m, 4: int(tape.jac_rows.size), 5: int(tape.hess_rows.size)}
        self.dyn, self.lam, self.sigma, self.calls = {}, np.zeros(tape.m), 1.0, []
        self.error = b""

    def _eval(self, space, x, lam=None, sigma=None):
        if lam is not None:
            self.lam, self.sigma = np.array(lam[:self.m], copy=True), float(sigma)
        self.calls.append(_NAME[space])
        with np.errstate(all="ignore"):
            if space == 5:
                return np.asarray(self.it.eval("hess", x, self.lam, self.sigma), dtype=np.float64).reshape(-1)
            return np.asarray(self.it.eval(_NAME[space], x), dtype=np.float64).reshape(-1)

    def _deliver(self, space, x, out, lam=None, sigma=None):
        if out is not None:
            _arr(out, self.len[space])[:] = self._eval(space, _arr(x, self.n), None if lam is None else _arr(lam, self.m), sigma)
        return 0

    def dnlp_eval_f(self, h, x, out):
        return self._deliver(1, x, out)

    def dnlp_eval_grad(self, h, x, out):
        return self._deliver(2, x, out)

    def dnlp_eval_g(self, h, x, out):
        return self._deliver(3, x, out)

    def dnlp_eval_jac(self, h, x, out):
        return self._deliver(4, x, out)

    def dnlp_eval_hess(self, h, x, lam, sigma, out):
        return self._deliver(5, x, out, lam, sigma)

    def dnlp_eval_all(self, h, x, lam, sigma, f, grad, g, jac, hess):
        for space, out in ((1, f), (2, grad), (3, g), (4, jac)):
            self._deliver(space, x, out)
        return self._deliver(5, x, hess, lam, sigma)

    def dnlp_set_dynamic(self, h, space, pos, count):
        self.dyn[int(space)] = np.array(np.ctypeslib.as_array(pos, shape=(max(int(count), 1),))[:int(count)], dtype=np.int64)
        return 0

    def dnlp_eval_dyn(self, h, prog, x, lam, sigma, compact):
        space = _SPACE_OF_PROG[int(prog)]
        if space not in self.dyn:
            self.error = b"no dynamic positions registered for this output"
            return 1
        full = self._eval(space, _arr(x, self.n), None if not lam else _arr(lam, self.m), sigma)
        pos = self.dyn[space]
        _arr(compact, pos.size)[:] = full[pos]
        return 0

    def dnlp_set_params(self, h, values, count):
        if int(count) != self.tape.n_params:
            self.error = b"wrong number of parameter values"
            return 1
        self.it.set_params(np.array(_arr(values, count), copy=True))
        return 0

    def dnlp_last_error(self, h):
        return self.error

    # ---- measurement hooks of bench.py: no device, so no timings - fixed figures that keep the control flow going ----
    def dnlp_upload_point(self, h, x, lam, sigma):
        self.x = np.array(_arr(x, self.n), copy=True)
        self.lam = np.zeros(self.m) if not lam else np.array(_arr(lam, self.m), copy=True)
        self.sigma, self.launches = float(sigma), getattr(self, "launches", 0)
        return 0

    def dnlp_run_device(self, h, mask, iters, ms_out):
        self.launches = getattr(self, "launches", 0) + int(iters) * len(self.tape.programs["all"])
        ms_out._obj.value = 0.05 * int(iters)
        return 0

    def dnlp_profile_instrs(self, h, prog, iters, out):
        k = max(len(self.tape.instrs), 1)
        np.ctypeslib.as_array(out, shape=(k,))[:] = 0.01
        return 0

    def dnlp_kernel_launches(self, h):
        return getattr(self, "launches", 0)

    def dnlp_instr_kernel(self, h, instr):
        return b"tape_interpreter"

    def dnlp_read_output(self, h, space, out):
        # what dnlp_run_device left on the device: the outputs at the uploaded point
        _arr(out, self.len[int(space)])[:] = self._eval(int(space), self.x)
        return 0

    def dnlp_set_graphs(self, h, on):
        return 0

    dnlp_set_parallel = dnlp_set_windows = dnlp_set_cache = dnlp_set_graphs


class InterpDeviceTape:
    """Drop-in for ``_cabi.DeviceTape`` in CPU tests: ``monkeypatch.setattr(_cabi, "DeviceTape", InterpDeviceTape)``."""

    def __init__(self, tape, device=0):
        self.tape, self.h, self._L = tape, 1, _InterpLib(tape)
        self.bound = None

    def check(self, rc):
        if rc != 0:
            raise RuntimeError("dnlp_b200: %s" % self._L.dnlp_last_error(self.h).decode())

    def set_params(self, values):
        self.check(self._L.dnlp_set_params(self.h, values.ctypes.data_as(__import__("dnlp_b200")._cabi.c_f64p), int(values.size)))

    def bind_outputs(self, f, grad, g, jac, eager):
        self.bound = (f, grad, g, jac, bool(eager))       # eager delivery is a device feature: the arrays are only recorded

    def close(self):
        self.h = None


class _InterpBatchLib:
    """Batched entry points (``BatchedOracles``): every start through the interpreter, one after the other."""

    def __init__(self, tape, batch):
        self.tape, self.B, self.it = tape, int(batch), TapeInterp(tape)
        self.n, self.m = tape.n, tape.m
        self.len = {"f": 1, "grad": tape.n, "g": tape.m, "jac": int(tape.jac_rows.size), "hess": int(tape.hess_rows.size)}
        self.launches, self.error = 0, b""

    def _mat(self, ptr, cols):
        return None if not ptr else np.ctypeslib.as_array(ptr, shape=(self.B * max(int(cols), 1),))[:self.B * int(cols)].reshape(self.B, int(cols))

    def _inputs(self, X, LAM, SIGMA):
        return (self._mat(X, self.n), self._mat(LAM, self.m) if self.m else None,
                None if not SIGMA else np.ctypeslib.as_array(SIGMA, shape=(self.B,)))

    def dnlp_batch_eval(self, h, X, LAM, SIGMA, f, grad, g, jac, hess):
        outs = {k: self._mat(p, self.len[k]) for k, p in (("f", f), ("grad", grad), ("g", g), ("jac", jac), ("hess", hess))}
        return self._fill(*self._inputs(X, LAM, SIGMA), outs)

    def _fill(self, X, LAM, SIG, outs):
        with np.errstate(all="ignore"):
            for b in range(self.B):
                for k, out in outs.items():
                    if out is None or self.len[k] == 0:
                        continue
                    if k == "hess":
                        lam = LAM[b] if LAM is not None else np.zeros(0)
                        out[b] = np.asarray(self.it.eval("hess", X[b], lam, float(SIG[b]))).reshape(-1)
                    else:
                        out[b] = np.asarray(self.it.eval(k, X[b])).reshape(-1)
        return 0

    def dnlp_batch_upload(self, h, X, LAM, SIGMA):
        self.uploaded = [None if a is None else np.array(a, copy=True) for a in self._inputs(X, LAM, SIGMA)]
        return 0

    def dnlp_batch_read_output(self, h, space, out):
        # what dnlp_batch_run_device left on the device: the outputs at the uploaded points
        name = _NAME[int(space)]
        return self._fill(*self.uploaded, {name: self._mat(out, self.len[name])})

    def dnlp_batch_run_device(self, h, mask, iters, ms_out):
        self.launches += int(iters) * len(self.tape.programs["all"])
        ms_out._obj.value = 0.05 * int(iters)
        return 0

    def dnlp_batch_profile_instrs(self, h, prog, iters, out):
        np.ctypeslib.as_array(out, shape=(max(len(self.tape.instrs), 1),))[:] = 0.01
        return 0

    def dnlp_batch_profile_groups(self, h, iters, ms, flops, cap):
        np.ctypeslib.as_array(ms, shape=(int(cap),))[0] = 0.02
        np.ctypeslib.as_array(flops, shape=(int(cap),))[0] = 1e9
        return 1

    def dnlp_batch_kernel_launches(self, h):
        return self.launches

    def dnlp_batch_last_error(self, h):
        return self.error


class InterpDeviceBatch:
    """Drop-in for ``_cabi.DeviceBatch`` in CPU tests."""

    def __init__(self, tape, batch, device=0):
        self.tape, self.batch, self.h, self._L = tape, int(batch), 1, _InterpBatchLib(tape, batch)

    def check(self, rc):
        if rc != 0:
            raise RuntimeError("dnlp_b200: %s" % self._L.dnlp_batch_last_error(self.h).decode())

    def close(self):
        self.h = None


def install(monkeypatch):
    """Route ``GpuOracles`` to the interpreter-backed stand-in for the duration of a test."""
    import types

    from dnlp_b200 import _cabi
    monkeypatch.setattr(_cabi, "DeviceTape", InterpDeviceTape)
    monkeypatch.setattr(_cabi, "DeviceBatch", InterpDeviceBatch)
    monkeypatch.setattr(_cabi, "pinned_empty", lambda k: (np.empty(int(k)), types.SimpleNamespace(free=lambda: None)))
