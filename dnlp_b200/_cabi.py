"""ctypes binding of libdnlp_b200.so (the C-ABI declared in include/dnlp_b200.h).

There is no CPU fallback: if the shared library is missing, cannot be loaded, or no CUDA
device is visible, creating an oracle raises.
"""
import ctypes as C
import os

import numpy as np

from . import tape as T

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libdnlp_b200.so")

PROG_IDS = {"f": 0, "grad": 1, "g": 2, "jac": 3, "hess": 4, "all": 5}
NPROG = 6

c_i64p = C.POINTER(C.c_int64)
c_i32p = C.POINTER(C.c_int32)
c_f64p = C.POINTER(C.c_double)
c_f32p = C.POINTER(C.c_float)


class InstrDesc(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("dst_space", C.c_int32), ("dst_off", C.c_int64), ("count", C.c_int64),
        ("fcode", C.c_int32), ("a_stride", C.c_int32), ("b_stride", C.c_int32), ("accumulate", C.c_int32),
        ("param", C.c_double), ("a_off", C.c_int64), ("b_off", C.c_int64),
        ("ptr", c_i64p), ("coef", c_f64p), ("f1", c_i32p), ("f2", c_i32p), ("pos", c_i32p),
        ("nterms", C.c_int64), ("row_len", C.c_int32), ("uses_lam", C.c_int32),
        ("level", C.c_int32), ("dep_mask", C.c_int32),
        ("Q", c_f64p), ("ncols", C.c_int64), ("x_off", C.c_int64), ("alpha", C.c_double),
        ("s_slot", C.c_int64),
        ("deps", c_i32p), ("n_deps", C.c_int64),
        ("dst_stride", C.c_int32), ("reserved0", C.c_int32), ("post_scale", C.c_double), ("qpos", c_i32p),
    ]


class TapeDesc(C.Structure):
    _fields_ = [
        ("n", C.c_int64), ("m", C.c_int64), ("nslots", C.c_int64), ("nnz_jac", C.c_int64), ("nnz_hess", C.c_int64),
        ("n_instr", C.c_int32), ("instrs", C.POINTER(InstrDesc)),
        ("prog", c_i32p * NPROG), ("prog_len", C.c_int32 * NPROG),
        ("f_const", C.c_double), ("grad_const", c_f64p), ("g_const", c_f64p),
        ("jac_const", c_f64p), ("hess_const", c_f64p),
        ("n_params", C.c_int64), ("params", c_f64p),
    ]


EXPORTS = [
    "dnlp_device_count", "dnlp_version", "dnlp_device_synchronize", "dnlp_create", "dnlp_destroy", "dnlp_last_error",
    "dnlp_eval_f", "dnlp_eval_grad", "dnlp_eval_g", "dnlp_eval_jac", "dnlp_eval_hess", "dnlp_eval_all",
    "dnlp_host_alloc", "dnlp_host_free", "dnlp_upload_point", "dnlp_run_device", "dnlp_profile_instrs",
    "dnlp_read_output", "dnlp_kernel_launches", "dnlp_set_cache", "dnlp_set_graphs", "dnlp_set_parallel", "dnlp_set_windows", "dnlp_set_dynamic", "dnlp_eval_dyn", "dnlp_bind_outputs", "dnlp_set_params", "dnlp_instr_kernel", "dnlp_run", "dnlp_output_ptr",
    "dnlp_batch_create", "dnlp_batch_destroy", "dnlp_batch_last_error", "dnlp_batch_eval", "dnlp_batch_upload",
    "dnlp_batch_run_device", "dnlp_batch_read_output", "dnlp_batch_profile_instrs", "dnlp_batch_kernel_launches", "dnlp_batch_profile_groups",
    "dnlp_batch_kkt_setup", "dnlp_batch_kkt_solve", "dnlp_batch_kkt_matrix",
    "dnlp_comm_unique_id", "dnlp_comm_create", "dnlp_comm_destroy", "dnlp_comm_last_error", "dnlp_comm_has_nccl",
    "dnlp_comm_ipc_handle", "dnlp_comm_open_peers", "dnlp_comm_allreduce_host",
    "dnlp_shard_create", "dnlp_shard_destroy", "dnlp_shard_last_error", "dnlp_shard_set_output",
    "dnlp_shard_root_handles", "dnlp_shard_open_root", "dnlp_shard_eval", "dnlp_shard_run_device", "dnlp_shard_set_layout",
    "dnlp_shard_share_control", "dnlp_shard_share_output", "dnlp_shard_share_unlink", "dnlp_shard_share_release", "dnlp_shard_share_reset",
    "dnlp_shard_share_inputs", "dnlp_shard_post_command", "dnlp_shard_wait_command",
]

_lib = None


def lib():
    """Load the CUDA library (raises if it has not been built: no silent fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "dnlp_b200: %s is missing - build it with `python -m dnlp_b200.build` "
            "(there is no CPU fallback for the oracle)" % LIB_PATH)
    # Several ranks share the host cores: the staging helpers size their OpenMP teams to cores / LOCAL_WORLD_SIZE - 1
    # (csrc/dnlp_cabi.cu stage_threads), so libgomp's default wait policy (spin briefly, then sleep) is kept: with
    # OMP_WAIT_POLICY=passive every parallel region paid a thread wake-up (C3 on 2 GPUs: 3.2 ms per evaluation
    # instead of 2.2, profiles/r02_e2e_breakdown_sharded.txt).
    L = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    L.dnlp_device_count.restype = C.c_int
    L.dnlp_version.restype = C.c_char_p
    L.dnlp_device_synchronize.argtypes = [C.c_int]
    L.dnlp_create.argtypes = [C.POINTER(TapeDesc), C.c_int, C.POINTER(vp)]
    L.dnlp_destroy.argtypes = [vp]
    L.dnlp_destroy.restype = None
    L.dnlp_last_error.argtypes = [vp]
    L.dnlp_last_error.restype = C.c_char_p
    L.dnlp_eval_f.argtypes = [vp, c_f64p, c_f64p]
    L.dnlp_eval_grad.argtypes = [vp, c_f64p, c_f64p]
    L.dnlp_eval_g.argtypes = [vp, c_f64p, c_f64p]
    L.dnlp_eval_jac.argtypes = [vp, c_f64p, c_f64p]
    L.dnlp_eval_hess.argtypes = [vp, c_f64p, c_f64p, C.c_double, c_f64p]
    L.dnlp_eval_all.argtypes = [vp, c_f64p, c_f64p, C.c_double] + [c_f64p] * 5
    L.dnlp_host_alloc.argtypes = [C.c_int64]
    L.dnlp_host_alloc.restype = vp
    L.dnlp_host_free.argtypes = [vp]
    L.dnlp_host_free.restype = None
    L.dnlp_upload_point.argtypes = [vp, c_f64p, c_f64p, C.c_double]
    L.dnlp_run_device.argtypes = [vp, C.c_int32, C.c_int32, c_f32p]
    L.dnlp_profile_instrs.argtypes = [vp, C.c_int32, C.c_int32, c_f32p]
    L.dnlp_read_output.argtypes = [vp, C.c_int32, c_f64p]
    L.dnlp_kernel_launches.argtypes = [vp]
    L.dnlp_kernel_launches.restype = C.c_int64
    L.dnlp_set_cache.argtypes = [vp, C.c_int32]
    L.dnlp_set_graphs.argtypes = [vp, C.c_int32]
    L.dnlp_set_parallel.argtypes = [vp, C.c_int32]
    L.dnlp_set_windows.argtypes = [vp, C.c_int32]
    L.dnlp_run.argtypes = [vp, C.c_int32, c_f64p, c_f64p, C.c_double]
    L.dnlp_output_ptr.argtypes = [vp, C.c_int32]
    L.dnlp_output_ptr.restype = vp
    L.dnlp_instr_kernel.argtypes = [vp, C.c_int32]
    L.dnlp_instr_kernel.restype = C.c_char_p
    L.dnlp_set_params.argtypes = [vp, c_f64p, C.c_int64]
    L.dnlp_bind_outputs.argtypes = [vp, c_f64p, c_f64p, c_f64p, c_f64p, C.c_int32]
    L.dnlp_set_dynamic.argtypes = [vp, C.c_int32, c_i32p, C.c_int64]
    L.dnlp_eval_dyn.argtypes = [vp, C.c_int32, c_f64p, c_f64p, C.c_double, c_f64p]
    L.dnlp_batch_create.argtypes = [C.POINTER(TapeDesc), C.c_int, C.c_int32, C.POINTER(vp)]
    L.dnlp_batch_destroy.argtypes = [vp]
    L.dnlp_batch_destroy.restype = None
    L.dnlp_batch_last_error.argtypes = [vp]
    L.dnlp_batch_last_error.restype = C.c_char_p
    L.dnlp_batch_eval.argtypes = [vp] + [c_f64p] * 8
    L.dnlp_batch_upload.argtypes = [vp, c_f64p, c_f64p, c_f64p]
    L.dnlp_batch_run_device.argtypes = [vp, C.c_int32, C.c_int32, c_f32p]
    L.dnlp_batch_read_output.argtypes = [vp, C.c_int32, c_f64p]
    L.dnlp_batch_profile_instrs.argtypes = [vp, C.c_int32, C.c_int32, c_f32p]
    L.dnlp_batch_profile_groups.argtypes = [vp, C.c_int32, c_f32p, c_f64p, C.c_int32]
    L.dnlp_batch_kernel_launches.argtypes = [vp]
    L.dnlp_batch_kernel_launches.restype = C.c_int64
    L.dnlp_batch_kkt_setup.argtypes = [vp, C.c_int64] + [c_i32p] * 5
    L.dnlp_batch_kkt_solve.argtypes = [vp, C.c_int32, c_i32p] + [c_f64p] * 5 + [c_i32p, c_f64p, c_f32p]
    L.dnlp_batch_kkt_matrix.argtypes = [vp, C.c_int32, c_f64p]
    cp = C.c_char_p
    L.dnlp_comm_unique_id.argtypes = [cp]
    L.dnlp_comm_create.argtypes = [cp, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]
    L.dnlp_comm_destroy.argtypes = [vp]
    L.dnlp_comm_destroy.restype = None
    L.dnlp_comm_last_error.argtypes = [vp]
    L.dnlp_comm_last_error.restype = C.c_char_p
    L.dnlp_comm_has_nccl.argtypes = [vp]
    L.dnlp_comm_ipc_handle.argtypes = [vp, cp]
    L.dnlp_comm_open_peers.argtypes = [vp, cp]
    L.dnlp_comm_allreduce_host.argtypes = [vp, c_f64p, C.c_int64]
    L.dnlp_shard_create.argtypes = [vp, vp, C.c_int, C.POINTER(vp)]
    L.dnlp_shard_destroy.argtypes = [vp]
    L.dnlp_shard_destroy.restype = None
    L.dnlp_shard_last_error.argtypes = [vp]
    L.dnlp_shard_last_error.restype = C.c_char_p
    L.dnlp_shard_set_output.argtypes = [vp, C.c_int32, C.c_int64, c_i32p, c_i32p, C.c_int64, c_i32p, c_i32p,
                                        C.c_int64, c_f64p, C.c_int64, c_i32p]
    L.dnlp_shard_root_handles.argtypes = [vp, cp]
    L.dnlp_shard_open_root.argtypes = [vp, cp]
    L.dnlp_shard_set_layout.argtypes = [vp, C.c_int32, c_i64p, c_i64p, C.c_int32, c_i64p, c_i64p]
    L.dnlp_shard_eval.argtypes = [vp, C.c_int32, c_f64p, c_f64p, C.c_double, c_f64p]
    L.dnlp_shard_run_device.argtypes = [vp, C.c_int32, C.c_int32, c_f32p]
    L.dnlp_shard_share_control.argtypes = [vp, C.c_char_p, C.c_int32]
    L.dnlp_shard_share_output.argtypes = [vp, C.c_int32, C.c_char_p, C.c_int32, C.c_int64, c_i64p, c_i64p, c_i64p,
                                          C.POINTER(c_f64p)]
    L.dnlp_shard_share_unlink.argtypes = [C.c_char_p]
    L.dnlp_shard_share_release.argtypes = [C.c_void_p, C.c_int64]
    L.dnlp_shard_share_reset.argtypes = [vp]
    L.dnlp_shard_share_inputs.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_int32, C.c_int64, C.c_int64,
                                          C.POINTER(c_f64p), C.POINTER(c_f64p)]
    L.dnlp_shard_post_command.argtypes = [vp, C.c_int32, c_f64p, c_f64p, C.c_double, C.c_int32, C.POINTER(C.c_int32)]
    L.dnlp_shard_wait_command.argtypes = [vp, C.c_double, C.POINTER(C.c_int32), C.POINTER(C.c_double),
                                          C.POINTER(C.c_int32)]
    _lib = L
    return L


def device_count():
    return int(lib().dnlp_device_count())


def device_synchronize(device=0):
    if lib().dnlp_device_synchronize(int(device)) != 0:
        raise RuntimeError("dnlp_b200: cudaDeviceSynchronize failed on device %d" % device)


def _p(arr, typ):
    return None if arr is None else arr.ctypes.data_as(typ)


def f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def pinned_empty(count):
    """float64 NumPy array backed by cudaMallocHost memory.

    The pinned block is released when the LAST view of it disappears (the handle rides on the
    ctypes buffer every view keeps as its base), so arrays handed to a solver stay valid even after
    the oracle that produced them was closed."""
    L = lib()
    nbytes = max(int(count), 1) * 8
    ptr = L.dnlp_host_alloc(nbytes)
    if not ptr:
        raise MemoryError("cudaMallocHost(%d) failed" % nbytes)
    buf = (C.c_double * max(int(count), 1)).from_address(ptr)
    handle = _PinnedHandle(ptr)
    buf._dnlp_handle = handle
    arr = np.frombuffer(buf, dtype=np.float64, count=int(count))
    return arr, handle


def shared_view(addr, count):
    """float64 NumPy array over a shared-host output array (dnlp_shard_share_output); the mapping is unpinned and
    unmapped when the LAST view disappears, so arrays handed to a solver outlive the shard handle."""
    buf = (C.c_double * max(int(count), 1)).from_address(addr)
    buf._dnlp_handle = _SharedHandle(addr, int(count))
    return np.frombuffer(buf, dtype=np.float64, count=int(count))


class _SharedHandle:
    def __init__(self, addr, count):
        self.addr, self.count = addr, count

    def __del__(self):
        try:
            if self.addr:
                lib().dnlp_shard_share_release(self.addr, self.count)
                self.addr = None
        except Exception:
            pass


class _PinnedHandle:
    def __init__(self, ptr):
        self.ptr = ptr

    def free(self):
        """Kept for API compatibility: release happens when the last array view is collected."""

    def __del__(self):
        try:
            if self.ptr:
                lib().dnlp_host_free(self.ptr)
                self.ptr = None
        except Exception:
            pass


def make_tape_desc(tape):
    """Tape -> (TapeDesc, keepalive list).  Host arrays referenced by the descriptor must stay alive
    until dnlp_create / dnlp_batch_create has copied them to the device."""
    keep = []
    n_instr = len(tape.instrs)
    # slot indices, scatter positions and pattern indices are int32 on the device
    i32max = int(np.iinfo(np.int32).max)
    for what, v in (("value slots", tape.nslots), ("Jacobian entries", tape.jac_rows.size),
                    ("Hessian entries", tape.hess_rows.size)):
        if int(v) > i32max:
            raise OverflowError("dnlp_b200: %d %s exceed the int32 index range of the device tape" % (int(v), what))
    arr = (InstrDesc * max(n_instr, 1))()
    for i, ins in enumerate(tape.instrs):
        d = arr[i]
        d.kind, d.dst_space, d.dst_off, d.count = ins.kind, ins.dst_space, int(ins.dst_off), int(ins.count)
        d.fcode, d.a_stride, d.b_stride = int(ins.fcode), int(ins.a_stride), int(ins.b_stride)
        d.accumulate = int(bool(ins.accumulate))
        d.param, d.a_off, d.b_off = float(ins.param), int(ins.a_off), int(ins.b_off)
        d.uses_lam = int(bool(ins.uses_lam))
        d.level = int(ins.level)
        d.dep_mask = int(ins.dep_mask)
        d.alpha, d.ncols, d.x_off, d.s_slot = float(ins.alpha), int(ins.ncols), int(ins.x_off), int(ins.s_slot)
        d.dst_stride, d.post_scale = int(ins.dst_stride), float(ins.post_scale)
        if ins.kind == T.K_SPMVJ:
            qpos = np.ascontiguousarray(ins.qpos, dtype=np.int32)
            keep.append(qpos)
            d.qpos = _p(qpos, c_i32p)
        if ins.kind in (T.K_POLY, T.K_SPMVJ):
            lens = np.diff(ins.ptr)
            uniform = lens.size > 0 and bool(np.all(lens == lens[0])) and lens[0] >= 1
            coef = f64(ins.coef)
            f1 = np.ascontiguousarray(ins.f1, dtype=np.int32)
            has_f2 = bool(np.any(ins.f2 >= 0))
            f2 = np.ascontiguousarray(ins.f2, dtype=np.int32) if has_f2 else None
            ptr = None if uniform else np.ascontiguousarray(ins.ptr, dtype=np.int64)
            keep += [coef, f1, f2, ptr]
            d.ptr, d.coef, d.f1, d.f2 = _p(ptr, c_i64p), _p(coef, c_f64p), _p(f1, c_i32p), _p(f2, c_i32p)
            d.nterms = int(coef.size)
            d.row_len = int(lens[0]) if uniform else 0
        elif ins.kind == T.K_GEMV:
            Q = f64(ins.Q)
            keep.append(Q)
            d.Q = _p(Q, c_f64p)
        elif ins.kind == T.K_SCALE:
            coef = f64(ins.coef)
            keep.append(coef)
            d.coef = _p(coef, c_f64p)
        if len(ins.deps):
            deps = np.ascontiguousarray(sorted(ins.deps), dtype=np.int32)
            keep.append(deps)
            d.deps, d.n_deps = _p(deps, c_i32p), int(deps.size)
        if ins.pos is not None:
            pos = np.ascontiguousarray(ins.pos, dtype=np.int32)
            keep.append(pos)
            d.pos = _p(pos, c_i32p)
    td = TapeDesc()
    td.n, td.m, td.nslots = tape.n, tape.m, tape.nslots
    td.nnz_jac, td.nnz_hess = int(tape.jac_rows.size), int(tape.hess_rows.size)
    td.n_instr, td.instrs = n_instr, arr
    for name, pid in PROG_IDS.items():
        p = np.ascontiguousarray(tape.programs.get(name, []), dtype=np.int32)
        keep.append(p)
        td.prog[pid] = _p(p, c_i32p) if p.size else None
        td.prog_len[pid] = int(p.size)
    consts = [f64(tape.grad_const), f64(tape.g_const), f64(tape.jac_const), f64(tape.hess_const)]
    keep += consts
    td.f_const = float(tape.f_const)
    td.grad_const, td.g_const, td.jac_const, td.hess_const = [_p(c, c_f64p) if c.size else None for c in consts]
    pv = f64(getattr(tape, "param_values", np.zeros(0)))
    keep.append(pv)
    td.n_params = int(getattr(tape, "n_params", 0))
    if pv.size != td.n_params:
        raise ValueError("tape has %d parameter slots but %d values" % (td.n_params, pv.size))
    td.params = _p(pv, c_f64p) if pv.size else None
    keep += [arr, td]
    return td, keep


def _require_device(L):
    if L.dnlp_device_count() <= 0:
        raise RuntimeError("dnlp_b200: no CUDA device visible (the oracle has no CPU fallback)")


class DeviceTape:
    """Uploads a compiled ``Tape`` and owns the ``dnlp_oracle`` handle."""

    def __init__(self, tape, device=0):
        L = lib()
        _require_device(L)
        self.tape = tape
        td, keep = make_tape_desc(tape)
        h = C.c_void_p()
        if L.dnlp_create(C.byref(td), int(device), C.byref(h)) != 0:
            raise RuntimeError("dnlp_create failed: %s" % L.dnlp_last_error(None).decode())
        self.h = h
        self._L = L

    def check(self, rc):
        if rc != 0:
            if not self.h:
                raise RuntimeError("dnlp_b200: oracle closed")
            raise RuntimeError("dnlp_b200: %s" % self._L.dnlp_last_error(self.h).decode())

    def set_params(self, values):
        self.check(self._L.dnlp_set_params(self.h, values.ctypes.data_as(c_f64p), int(values.size)))

    def bind_outputs(self, f, grad, g, jac, eager):
        """Name the host arrays the x-only callbacks deliver into (dnlp_bind_outputs)."""
        p = lambda a: a.ctypes.data_as(c_f64p)      # noqa: E731
        self.check(self._L.dnlp_bind_outputs(self.h, p(f), p(grad), p(g), p(jac), int(bool(eager))))

    def close(self):
        if getattr(self, "h", None):
            self._L.dnlp_destroy(self.h)
            self.h = None       # later calls pass NULL, which every entry point rejects (rc != 0)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DeviceBatch:
    """Batched (multi-start) counterpart of ``DeviceTape``: owns a ``dnlp_batch`` handle."""

    def __init__(self, tape, batch, device=0):
        L = lib()
        _require_device(L)
        self.tape, self.batch = tape, int(batch)
        td, keep = make_tape_desc(tape)
        h = C.c_void_p()
        if L.dnlp_batch_create(C.byref(td), int(device), int(batch), C.byref(h)) != 0:
            raise RuntimeError("dnlp_batch_create failed: %s" % L.dnlp_batch_last_error(None).decode())
        self.h = h
        self._L = L

    def check(self, rc):
        if rc != 0:
            if not self.h:
                raise RuntimeError("dnlp_b200: oracle closed")
            raise RuntimeError("dnlp_b200: %s" % self._L.dnlp_batch_last_error(self.h).decode())

    def close(self):
        if getattr(self, "h", None):
            self._L.dnlp_batch_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
