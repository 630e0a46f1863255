"""ctypes binding of csrc/libcadnip_b200.so -- the stand-in for the Julia ``ccall``
shim (INTEGRATION.md shows the Julia side).  Fails loudly: if the library is not
built, or no sm_100 device is present, every numerical call raises; there is no
CPU path.
"""
from __future__ import annotations

import ctypes as C
import os
import weakref
import shutil
import subprocess
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

from .circuit import MNASpec, MODES
from .lowering import LoweredCircuit

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(_CSRC, "libcadnip_b200.so")
_SOURCES = ["api.cu", "kernels.cu", "symbolic.cpp", "specialize.cpp"]
_HEADERS = ["kernels.h", "cb200_internal.h", "lane_kernels.cuh", "warp_kernels.cuh", "group_kernels.inc", "specialize.h",
            os.path.join("..", "..", "include", "cadnip_b200.h")]
GEN_DIR = os.path.join(_HERE, "_gen")
# Kernels compiled at run time (circuit-specialised kernels, kernel sets that GEN_DIR does not hold yet) are
# cached here.  A caller that must leave the tree untouched points it at a directory of its own.
RUN_CACHE_DIR = GEN_DIR

OK, EINVAL, ENOMEM, ECUDA, ENODEVICE, ESTATE, ESINGULAR = 0, -1, -2, -3, -4, -5, -6
LANE_OK, LANE_MAXITER, LANE_SINGULAR, LANE_NONFINITE, LANE_DTMIN = 0, 1, 2, 3, 4
METHOD_BE, METHOD_TRAP, METHOD_GEAR2, METHOD_BDF = 0, 1, 2, 3
# "IDA" / "FBDF" / "QNDF" / "bdf": the variable-order (1..5) variable-step BDF controller (adaptive mode only)
METHODS = {"be": 0, "implicit_euler": 0, "ImplicitEuler": 0, "trap": 1, "trapezoid": 1,
           "Trapezoid": 1, "gear2": 2, "bdf2": 2, "bdf": 3, "IDA": 3, "ida": 3, "FBDF": 3, "QNDF": 3}


class CB200Error(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"cb200 error {code}: {msg}")
        self.code = code


class Spec(C.Structure):
    _fields_ = [("temp", C.c_double), ("mode", C.c_int32), ("_pad", C.c_int32),
                ("gmin", C.c_double), ("gshunt", C.c_double), ("srcFact", C.c_double),
                ("tnom", C.c_double), ("abstol", C.c_double), ("reltol", C.c_double),
                ("vntol", C.c_double), ("iabstol", C.c_double)]


class Desc(C.Structure):
    _fields_ = [("n_nodes", C.c_int32), ("n_currents", C.c_int32), ("n_charges", C.c_int32),
                ("n_limits", C.c_int32),
                ("nG", C.c_int64), ("nC", C.c_int64), ("nb", C.c_int64),
                ("G_I", C.POINTER(C.c_int64)), ("G_J", C.POINTER(C.c_int64)),
                ("C_I", C.POINTER(C.c_int64)), ("C_J", C.POINTER(C.c_int64)),
                ("b_I", C.POINTER(C.c_int64)),
                ("n_devices", C.c_int32), ("n_uniform", C.c_int32),
                ("dev_kind", C.POINTER(C.c_int32)), ("dev_flags", C.POINTER(C.c_int32)),
                ("dev_node_ptr", C.POINTER(C.c_int32)), ("dev_nodes", C.POINTER(C.c_int32)),
                ("dev_param_ptr", C.POINTER(C.c_int32)), ("dev_params", C.POINTER(C.c_int32)),
                ("dev_gbase", C.POINTER(C.c_int64)), ("dev_cbase", C.POINTER(C.c_int64)),
                ("dev_bbase", C.POINTER(C.c_int64)),
                ("uniform", C.POINTER(C.c_double)),
                ("limit_init_ref", C.POINTER(C.c_int32)),
                ("n_lane_cols", C.c_int32), ("_pad", C.c_int32),
                ("dev_state_ptr", C.POINTER(C.c_int32))]


class DcOpts(C.Structure):
    _fields_ = [("abstol", C.c_double), ("maxiters", C.c_int32), ("use_stepping", C.c_int32)]


class TranOpts(C.Structure):
    _fields_ = [("method", C.c_int32), ("adaptive", C.c_int32),
                ("dt", C.c_double), ("abstol", C.c_double), ("reltol", C.c_double),
                ("lte_abstol", C.c_double), ("dtmin", C.c_double), ("dtmax", C.c_double),
                ("max_nl_iters", C.c_int32), ("save_every", C.c_int32),
                ("max_points", C.c_int32), ("init", C.c_int32),
                ("init_abstol", C.c_double), ("init_maxiters", C.c_int32), ("flags", C.c_int32),
                ("uic_steps", C.c_int32), ("_pad", C.c_int32), ("uic_dt", C.c_double),
                ("vntol", C.c_double), ("iabstol", C.c_double), ("chgtol", C.c_double)]


class Stats(C.Structure):
    _fields_ = [("kernel_ms", C.c_double), ("tran_kernel_ms", C.c_double), ("dc_kernel_ms", C.c_double),
                ("h2d_ms", C.c_double), ("d2h_ms", C.c_double),
                ("launches", C.c_int64), ("newton_iters", C.c_int64),
                ("steps_accepted", C.c_int64), ("steps_rejected", C.c_int64),
                ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64), ("device_evals", C.c_int64),
                ("dc_stepping_lanes", C.c_int64)]


def nvcc_path() -> Optional[str]:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    return None


def _stale() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    for f in _SOURCES + _HEADERS:
        fp = os.path.join(_CSRC, f)
        if os.path.exists(fp) and os.path.getmtime(fp) > t:
            return True
    return False


def build_library(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/ for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    if not force and not _stale():
        return LIB_PATH
    nvcc = nvcc_path()
    if nvcc is None:
        raise RuntimeError("nvcc not found: cannot build libcadnip_b200.so")
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
           "-Xcompiler", "-fPIC", "-shared", "-o", LIB_PATH] + _SOURCES + ["-ldl"]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    r = subprocess.run(cmd, cwd=_CSRC, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout)
    if verbose:
        print(r.stdout)
    return LIB_PATH


_lib = None


def lib():
    """Load libcadnip_b200.so.  The library must already be built (``build_library``
    / ``__graft_entry__.build``); a missing library is an error, never a fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CB200Error(ENODEVICE, f"{LIB_PATH} is not built (run __graft_entry__.build()); "
                         "the product has no CPU path")
    L = C.CDLL(LIB_PATH)
    vp, dp = C.c_void_p, C.POINTER(C.c_double)
    ip, lp = C.POINTER(C.c_int32), C.POINTER(C.c_int64)
    L.cb200_abi_version.restype = C.c_int
    L.cb200_last_error.restype = C.c_char_p
    L.cb200_last_error.argtypes = [vp]
    L.cb200_create.restype = C.c_int
    L.cb200_create.argtypes = [C.POINTER(Desc), C.c_int32, C.POINTER(vp)]
    L.cb200_destroy.restype = None
    L.cb200_destroy.argtypes = [vp]
    L.cb200_get_pattern.restype = C.c_int
    L.cb200_get_pattern.argtypes = [vp, lp, lp, lp, lp]
    L.cb200_get_maps.restype = C.c_int
    L.cb200_get_maps.argtypes = [vp, lp, lp, lp, lp]
    L.cb200_set_lanes.restype = C.c_int
    L.cb200_set_lanes.argtypes = [vp, C.c_int64, C.c_int32, dp]
    L.cb200_analyze.restype = C.c_int
    L.cb200_analyze.argtypes = [vp, C.POINTER(Spec), C.c_double]
    L.cb200_get_pivot_order.restype = C.c_int
    L.cb200_get_pivot_order.argtypes = [vp, lp, lp, lp]
    L.cb200_specialize.restype = C.c_int
    L.cb200_specialize.argtypes = [vp, C.POINTER(Spec), C.c_int32, C.c_double, C.c_char_p, C.c_char_p, C.c_int32]
    L.cb200_is_specialized.restype = C.c_int
    L.cb200_is_specialized.argtypes = [vp]
    L.cb200_weak_pivot_lanes.restype = C.c_int
    L.cb200_weak_pivot_lanes.argtypes = [vp, ip, lp]
    L.cb200_lane_mapping.restype = C.c_int
    L.cb200_lane_mapping.argtypes = [vp]
    L.cb200_host_lu_check.restype = C.c_int
    L.cb200_host_lu_check.argtypes = [C.POINTER(Desc), dp, dp, dp, dp, lp, lp, ip]
    L.cb200_host_lu_check_static.restype = C.c_int
    L.cb200_host_lu_check_static.argtypes = [C.POINTER(Desc), dp, dp, dp, dp, dp, dp, ip]
    L.cb200_load_va_models.restype = C.c_int
    L.cb200_load_va_models.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_char_p]
    L.cb200_emit_source.restype = C.c_int64
    L.cb200_emit_source.argtypes = [C.POINTER(Desc), dp, dp, C.c_int32, C.c_int64, C.c_int32, C.c_char_p, C.c_int64]
    L.cb200_eval.restype = C.c_int
    L.cb200_eval.argtypes = [vp, C.POINTER(Spec), C.c_double, C.c_int32, dp, dp, dp, dp, dp]
    L.cb200_dc.restype = C.c_int
    L.cb200_dc.argtypes = [vp, C.POINTER(Spec), C.POINTER(DcOpts), dp, dp, ip, ip]
    L.cb200_tran.restype = C.c_int
    L.cb200_tran.argtypes = [vp, C.POINTER(Spec), C.c_double, C.c_double, C.POINTER(TranOpts),
                             lp, C.c_int32, dp, C.POINTER(vp)]
    L.cb200_tran_fetch.restype = C.c_int
    L.cb200_tran_fetch.argtypes = [vp, C.POINTER(Spec), C.c_double, C.c_double, C.POINTER(TranOpts),
                                   lp, C.c_int32, dp, C.c_int32, dp, dp, ip, ip, ip]
    L.cb200_tran_fetch_ld.restype = C.c_int
    L.cb200_tran_fetch_ld.argtypes = [vp, C.POINTER(Spec), C.c_double, C.c_double, C.POINTER(TranOpts),
                                      lp, C.c_int32, dp, C.c_int32, dp, dp, C.c_int64, ip, ip, ip]
    L.cb200_wave_fetch_ld.restype = C.c_int
    L.cb200_wave_fetch_ld.argtypes = [vp, dp, dp, C.c_int64, C.c_int64, ip, ip, ip]
    L.cb200_measure_fp64_peak.restype = C.c_int
    L.cb200_measure_fp64_peak.argtypes = [C.c_int32, dp, dp]
    L.cb200_flop_model.restype = C.c_int
    L.cb200_flop_model.argtypes = [vp, lp]
    L.cb200_set_tstops.restype = C.c_int
    L.cb200_set_tstops.argtypes = [vp, dp, C.c_int32]
    L.cb200_wave_info.restype = C.c_int
    L.cb200_wave_info.argtypes = [vp, lp, lp, ip, ip]
    L.cb200_wave_fetch.restype = C.c_int
    L.cb200_wave_fetch.argtypes = [vp, dp, dp, ip, ip, ip]
    L.cb200_wave_final_state.restype = C.c_int
    L.cb200_wave_final_state.argtypes = [vp, dp]
    L.cb200_wave_free.restype = None
    L.cb200_wave_free.argtypes = [vp]
    L.cb200_get_stats.restype = C.c_int
    L.cb200_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.cb200_debug_exp.restype = C.c_int
    L.cb200_debug_exp.argtypes = [dp, dp, C.c_int32]
    if L.cb200_abi_version() != 2:
        raise CB200Error(EINVAL, "libcadnip_b200.so ABI version mismatch")
    _lib = L
    return L


EXPORTED_SYMBOLS = [
    "cb200_abi_version", "cb200_last_error", "cb200_create", "cb200_destroy", "cb200_get_pattern",
    "cb200_get_maps", "cb200_set_lanes", "cb200_analyze", "cb200_get_pivot_order", "cb200_eval",
    "cb200_specialize", "cb200_is_specialized", "cb200_weak_pivot_lanes", "cb200_lane_mapping", "cb200_host_lu_check", "cb200_host_lu_check_static", "cb200_emit_source", "cb200_load_va_models",
    "cb200_dc", "cb200_tran", "cb200_tran_fetch", "cb200_tran_fetch_ld", "cb200_set_tstops", "cb200_wave_info",
    "cb200_wave_fetch", "cb200_wave_fetch_ld", "cb200_wave_final_state",
    "cb200_wave_free", "cb200_get_stats", "cb200_debug_exp", "cb200_measure_fp64_peak", "cb200_flop_model"]


def va_models_cached(models) -> bool:
    """Is the kernel set of these models already built (in-tree cache)?  PSP103's takes ~45 minutes of
    ptxas, sp_bsim4v8's ~20: callers that cannot wait check first."""
    L = lib()
    L.cb200_va_models_cached.restype = C.c_int
    L.cb200_va_models_cached.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p]
    text = models if isinstance(models, str) else None
    if text is None:
        from . import verilog_a
        text = verilog_a.cuda_header(models)
    return bool(L.cb200_va_models_cached(text.encode(), _CSRC.encode(), GEN_DIR.encode()))


def prebuild_va_models(models) -> None:
    """Build the kernel set for a circuit's Verilog-A models into the in-tree cache
    (no GPU needed; what Handle.load_va_models would otherwise build on first use).
    models: the emitted header text (LoweredCircuit.va_cuda_header) or a list of models."""
    from . import verilog_a as _va
    text = models if isinstance(models, str) else _va.cuda_header(list(models))
    rc = lib().cb200_load_va_models(None, text.encode(), _CSRC.encode(), GEN_DIR.encode())
    if rc != OK:
        raise CB200Error(rc, (lib().cb200_last_error(None) or b"").decode())


def _dp(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))


def _lp(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_int64))


def _ip(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_int32))


def _check_f64(a: np.ndarray, shape, what: str) -> np.ndarray:
    """A caller-supplied float64 buffer the C side reads or writes ``prod(shape)`` doubles of:
    wrong dtype, shape or layout is an error here, never a heap overrun there."""
    if not isinstance(a, np.ndarray) or a.dtype != np.float64:
        raise ValueError(f"{what}: expected a float64 numpy array, got {getattr(a, 'dtype', type(a))}")
    if tuple(a.shape) != tuple(shape):
        raise ValueError(f"{what}: shape {tuple(a.shape)}, expected {tuple(shape)}")
    if not a.flags["C_CONTIGUOUS"]:
        raise ValueError(f"{what}: must be C-contiguous")
    return a


def _lane_block(a: np.ndarray, lead_shape, P: int, what: str, writable: bool = True) -> int:
    """``a`` is [*lead_shape][P] float64 whose last axis is contiguous and whose leading axes are
    packed over rows of ``ld >= P`` doubles (a column block of a wider array).  Returns ld."""
    if not isinstance(a, np.ndarray) or a.dtype != np.float64:
        raise ValueError(f"{what}: expected a float64 numpy array, got {getattr(a, 'dtype', type(a))}")
    if tuple(a.shape) != tuple(lead_shape) + (P,):
        raise ValueError(f"{what}: shape {tuple(a.shape)}, expected {tuple(lead_shape) + (P,)}")
    if writable and not a.flags["WRITEABLE"]:
        raise ValueError(f"{what}: must be writable")
    if a.size == 0:
        return P
    st = a.strides
    if P > 1 and st[-1] != 8:
        raise ValueError(f"{what}: the lane axis must be contiguous")
    rows = int(np.prod(lead_shape)) if lead_shape else 1
    if rows <= 1:
        return P
    ld = None
    for ax in range(len(lead_shape) - 1, -1, -1):        # innermost leading axis with extent > 1 sets ld
        if lead_shape[ax] > 1:
            ld = st[ax] // 8
            break
    if ld is None or ld < P or ld * 8 != st[ax]:
        raise ValueError(f"{what}: rows must be at least P doubles apart")
    expect = ld * 8
    for ax in range(len(lead_shape) - 1, -1, -1):        # every leading axis packed over rows of ld
        if lead_shape[ax] > 1 and st[ax] != expect:
            raise ValueError(f"{what}: leading axes must be packed (strides {st})")
        expect *= lead_shape[ax]
    return int(ld)


def measure_fp64_peak(device: int = 0):
    """(TFLOP/s, kernel ms) of the register-only FP64 FMA microbenchmark on ``device``."""
    tf, ms = C.c_double(), C.c_double()
    rc = lib().cb200_measure_fp64_peak(int(device), C.byref(tf), C.byref(ms))
    if rc != OK:
        raise CB200Error(rc, (lib().cb200_last_error(None) or b"").decode())
    return tf.value, ms.value


def make_spec(spec: MNASpec, mode: Optional[str] = None) -> Spec:
    m = MODES[mode or spec.mode]
    return Spec(spec.temp, m, 0, spec.gmin, spec.gshunt, spec.srcFact, spec.tnom, spec.abstol,
                spec.reltol, spec.vntol, spec.iabstol)


def make_desc(lc: LoweredCircuit):
    """Returns (Desc, keepalive list)."""
    keep = []

    def arr(a, dt):
        a = np.ascontiguousarray(a, dtype=dt)
        keep.append(a)
        return a

    G_I, G_J = arr(lc.G_I, np.int64), arr(lc.G_J, np.int64)
    C_I, C_J = arr(lc.C_I, np.int64), arr(lc.C_J, np.int64)
    b_I = arr(lc.b_I, np.int64)
    d = Desc(lc.n_nodes, lc.n_currents, lc.n_charges, lc.n_limits,
             len(G_I), len(C_I), len(b_I),
             _lp(G_I), _lp(G_J), _lp(C_I), _lp(C_J), _lp(b_I),
             len(lc.dev_kind), len(lc.uniform),
             _ip(arr(lc.dev_kind, np.int32)), _ip(arr(lc.dev_flags, np.int32)),
             _ip(arr(lc.dev_node_ptr, np.int32)), _ip(arr(lc.dev_nodes, np.int32)),
             _ip(arr(lc.dev_param_ptr, np.int32)), _ip(arr(lc.dev_params, np.int32)),
             _lp(arr(lc.dev_gbase, np.int64)), _lp(arr(lc.dev_cbase, np.int64)),
             _lp(arr(lc.dev_bbase, np.int64)),
             _dp(arr(lc.uniform, np.float64)), _ip(arr(lc.limit_init_ref, np.int32)),
             lc.n_lane_cols, 0,
             _ip(arr(getattr(lc, "dev_state_ptr", None) if getattr(lc, "dev_state_ptr", None) is not None
                     else np.zeros(len(lc.dev_kind) + 1), np.int32)))
    return d, keep


def emit_source(lc: LoweredCircuit, absJ_dc: np.ndarray, absJ_tr: np.ndarray, P: int = 65536,
                num_sms: int = 148, method="be") -> str:
    """Generated CUDA source of the circuit-specialised kernels (host only, no device)."""
    L = lib()
    desc, keep = make_desc(lc)
    a0 = np.ascontiguousarray(absJ_dc, dtype=np.float64)
    a1 = np.ascontiguousarray(absJ_tr, dtype=np.float64)
    m = METHODS[method] if isinstance(method, str) else int(method)
    n = L.cb200_emit_source(C.byref(desc), _dp(a0), _dp(a1), m, P, num_sms, None, 0)
    if n < 0:
        raise CB200Error(int(n), (L.cb200_last_error(None) or b"").decode())
    buf = C.create_string_buffer(n + 1)
    L.cb200_emit_source(C.byref(desc), _dp(a0), _dp(a1), m, P, num_sms, buf, n + 1)
    return buf.value.decode()


def host_lu_check_static(lc: LoweredCircuit, absJ: np.ndarray, J_nz: np.ndarray, rhs: np.ndarray,
                         absJmin: Optional[np.ndarray] = None):
    """cb200_host_lu_check_static: pivot order from ``absJ`` / ``absJmin`` (largest / smallest magnitude
    over probe states), numeric factor + solves on ``J_nz``."""
    L = lib()
    desc, keep = make_desc(lc)
    info = np.zeros(6, dtype=np.int32)
    a = np.ascontiguousarray(absJ, dtype=np.float64)
    J = np.ascontiguousarray(J_nz, dtype=np.float64)
    r = np.ascontiguousarray(rhs, dtype=np.float64)
    xs, xl = np.zeros(len(r)), np.zeros(len(r))
    amin = None if absJmin is None else np.ascontiguousarray(absJmin, dtype=np.float64)
    rc = L.cb200_host_lu_check_static(C.byref(desc), _dp(a), _dp(amin), _dp(J), _dp(r), _dp(xs), _dp(xl), _ip(info))
    if rc != OK:
        raise CB200Error(rc, (L.cb200_last_error(None) or b"").decode())
    return xs, xl, dict(n=int(info[0]), nnz=int(info[1]), nlu=int(info[2]), factor_levels=int(info[3]))


def host_lu_check(lc: LoweredCircuit, J_nz: Optional[np.ndarray] = None, rhs: Optional[np.ndarray] = None):
    """cb200_host_lu_check (host only, no device).  Without J_nz: (colptr, rowval) of the pattern,
    1-based.  With J_nz / rhs: (x_serial, x_level, info) -- the serial static-pivot schedule and the
    level schedule of the lane-per-warp kernels executed on the host for that matrix."""
    L = lib()
    desc, keep = make_desc(lc)
    info = np.zeros(6, dtype=np.int32)
    rc = L.cb200_host_lu_check(C.byref(desc), None, None, None, None, None, None, _ip(info))
    if rc != OK:
        raise CB200Error(rc, (L.cb200_last_error(None) or b"").decode())
    n, nnz = int(info[0]), int(info[1])
    colptr, rowval = np.zeros(n + 1, dtype=np.int64), np.zeros(nnz, dtype=np.int64)
    if J_nz is None:
        L.cb200_host_lu_check(C.byref(desc), None, None, None, None, _lp(colptr), _lp(rowval), _ip(info))
        return colptr, rowval
    J = np.ascontiguousarray(J_nz, dtype=np.float64)
    r = np.ascontiguousarray(rhs, dtype=np.float64)
    assert J.shape == (nnz,) and r.shape == (n,)
    xs, xl = np.zeros(n), np.zeros(n)
    rc = L.cb200_host_lu_check(C.byref(desc), _dp(J), _dp(r), _dp(xs), _dp(xl), None, None, _ip(info))
    if rc != OK:
        raise CB200Error(rc, (L.cb200_last_error(None) or b"").decode())
    return xs, xl, dict(n=n, nnz=nnz, nlu=int(info[2]), factor_levels=int(info[3]),
                        forward_levels=int(info[4]), backward_levels=int(info[5]))


class Wave:
    """Owns a cb200_wave: the waveforms of a transient sweep, resident in HBM."""

    def __init__(self, handle: "Handle", ptr):
        self._h, self._p = handle, ptr
        T, P, ns, ad = C.c_int64(), C.c_int64(), C.c_int32(), C.c_int32()
        handle._check(lib().cb200_wave_info(ptr, C.byref(T), C.byref(P), C.byref(ns), C.byref(ad)))
        self.T, self.P, self.n_save, self.adaptive = T.value, P.value, ns.value, bool(ad.value)
        handle._waves.add(self)

    def _live(self):
        if not self._p:
            raise CB200Error(ESTATE, "the wave was freed, or its handle was closed")
        return self._p

    def fetch(self, out_u: Optional[np.ndarray] = None, out_t: Optional[np.ndarray] = None):
        """D2H copy.  Returns dict(t, u[save][T][P], count, status, newton_iters).  ``out_u``
        ([save][T][P]) and, for adaptive waves, ``out_t`` ([T][P]) may be column blocks of wider
        arrays (multi-GPU gather); dtype, shape and layout are checked."""
        L = lib()
        p = self._live()
        if out_u is None:
            out_u = np.empty((self.n_save, self.T, self.P), dtype=np.float64)
        u_ld = _lane_block(out_u, (self.n_save, self.T), self.P, "Wave.fetch(out_u)")
        if self.adaptive:
            t = np.empty((self.T, self.P), dtype=np.float64) if out_t is None else out_t
            t_ld = _lane_block(t, (self.T,), self.P, "Wave.fetch(out_t)")
        else:
            t, t_ld = np.empty((self.T,), dtype=np.float64), self.P
        count = np.empty(self.P, np.int32)
        status = np.empty(self.P, np.int32)
        iters = np.empty(self.P, np.int32)
        self._h._check(L.cb200_wave_fetch_ld(p, _dp(t), _dp(out_u) if out_u.size else None, u_ld, t_ld,
                                             _ip(count), _ip(status), _ip(iters)))
        return dict(t=t, u=out_u, count=count, status=status, newton_iters=iters)

    def final_state(self) -> np.ndarray:
        x = np.empty((self._h.n, self.P), dtype=np.float64)
        self._h._check(lib().cb200_wave_final_state(self._live(), _dp(x)))
        return x

    def free(self):
        if self._p:
            lib().cb200_wave_free(self._p)
            self._p = None
        if self._h is not None:
            self._h._waves.discard(self)

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Handle:
    """Owns a cb200_handle (one per GPU)."""

    def __init__(self, lc: LoweredCircuit, device: int = 0):
        L = lib()
        self.lc = lc
        self.n = lc.n
        desc, keep = make_desc(lc)
        ptr = C.c_void_p()
        rc = L.cb200_create(C.byref(desc), device, C.byref(ptr))
        if rc != OK:
            raise CB200Error(rc, (L.cb200_last_error(None) or b"").decode())
        self._p = ptr
        self.P = 0
        self._waves = weakref.WeakSet()      # waves must not outlive the handle (their stream is its)
        if getattr(lc, "va_cuda_header", ""):
            self.load_va_models(lc.va_cuda_header)

    def load_va_models(self, cuda_header: str):
        """Rebuild (cached) and load the kernel set with the circuit's Verilog-A models."""
        cache = GEN_DIR if va_models_cached(cuda_header) else RUN_CACHE_DIR
        self._check(lib().cb200_load_va_models(self._p, cuda_header.encode(), _CSRC.encode(), cache.encode()))

    def _check(self, rc: int):
        if rc != OK:
            raise CB200Error(rc, (lib().cb200_last_error(self._p) or b"").decode())

    def close(self):
        if getattr(self, "_p", None):
            for w in list(self._waves):      # outstanding waves become unusable, not dangling
                w.free()
            lib().cb200_destroy(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- structure ---------------------------------------------------------- #
    def pattern(self):
        L = lib()
        n, nnz = C.c_int64(), C.c_int64()
        self._check(L.cb200_get_pattern(self._p, C.byref(n), C.byref(nnz), None, None))
        colptr = np.zeros(n.value + 1, np.int64)
        rowval = np.zeros(nnz.value, np.int64)
        self._check(L.cb200_get_pattern(self._p, None, None, _lp(colptr), _lp(rowval)))
        return colptr, rowval

    def maps(self):
        lc = self.lc
        g = np.zeros(len(lc.G_I), np.int64); c = np.zeros(len(lc.C_I), np.int64)
        b = np.zeros(len(lc.b_I), np.int64); d = np.zeros(lc.n_nodes, np.int64)
        self._check(lib().cb200_get_maps(self._p, _lp(g), _lp(c), _lp(b), _lp(d)))
        return dict(G_coo_to_idx=g, C_coo_to_idx=c, b_resolved=b, G_diag_idx=d)

    def set_lanes(self, soa: np.ndarray, P: int):
        soa = np.ascontiguousarray(soa, dtype=np.float64)
        if soa.shape != (self.lc.n_lane_cols, P):
            raise ValueError(f"lane SoA has shape {soa.shape}, expected {(self.lc.n_lane_cols, P)}")
        self._check(lib().cb200_set_lanes(self._p, P, self.lc.n_lane_cols, _dp(soa) if soa.size else None))
        self.P = P

    def analyze(self, spec: MNASpec, gamma: float, mode: Optional[str] = None):
        s = make_spec(spec, mode)
        self._check(lib().cb200_analyze(self._p, C.byref(s), float(gamma)))

    def specialize(self, spec: MNASpec, method, dt: float, compile_only: bool = False, limit: bool = False,
                   fixed_only: bool = False):
        """Generate + compile (cached in RUN_CACHE_DIR) + load kernels specialised
        for this circuit; later dc/tran calls use them.  limit: include the CB200_TRAN_LIMIT
        path (otherwise transients that ask for it run on the table-driven kernels)."""
        s = make_spec(spec, "tran")
        m = METHODS[method] if isinstance(method, str) else int(method)
        self._check(lib().cb200_specialize(self._p, C.byref(s), m, float(dt), _CSRC.encode(),
                                           RUN_CACHE_DIR.encode(), (1 if compile_only else 0) | (2 if limit else 0) | (4 if fixed_only else 0)))

    def is_specialized(self) -> bool:
        return bool(lib().cb200_is_specialized(self._p))

    def weak_pivot_lanes(self) -> np.ndarray:
        """bool[P]: lanes on which a refactor of the last dc / tran met a weak pivot under the
        static order (cb200_weak_pivot_lanes)."""
        f = np.zeros(self.P, np.int32)
        self._check(lib().cb200_weak_pivot_lanes(self._p, _ip(f), None))
        return f != 0

    def lane_mapping(self) -> str:
        """Mapping of the table-driven kernels for this circuit (cb200_lane_mapping)."""
        return {0: "thread/smem", 1: "thread/hbm", 2: "warp", 3: "block"}[lib().cb200_lane_mapping(self._p)]

    def pivot_order(self):
        r = np.zeros(self.n, np.int64); c = np.zeros(self.n, np.int64); nlu = C.c_int64()
        self._check(lib().cb200_get_pivot_order(self._p, _lp(r), _lp(c), C.byref(nlu)))
        return r, c, nlu.value

    # -- analyses ----------------------------------------------------------- #
    def eval(self, spec: MNASpec, x: Optional[np.ndarray] = None, t: float = 0.0,
             initjct: bool = False, mode: Optional[str] = None):
        """fast_rebuild! for every lane: returns G_nz[nnz][P], C_nz[nnz][P], b[n][P], limit_w."""
        colptr, rowval = self.pattern()
        nnz, P, n = len(rowval), self.P, self.n
        G = np.empty((nnz, P)); Cm = np.empty((nnz, P)); b = np.empty((n, P))
        lw = np.empty((max(self.lc.n_limits, 1), P))
        xx = None if x is None else np.ascontiguousarray(x, dtype=np.float64)
        if xx is not None and xx.shape != (n, P):
            raise ValueError(f"x has shape {xx.shape}, expected {(n, P)}")
        s = make_spec(spec, mode)
        self._check(lib().cb200_eval(self._p, C.byref(s), float(t), int(initjct), _dp(xx), _dp(G),
                                     _dp(Cm), _dp(b), _dp(lw)))
        return G, Cm, b, lw[:self.lc.n_limits]

    def dc(self, spec: MNASpec, u0: Optional[np.ndarray] = None, abstol: float = 1e-10,
           maxiters: int = 100, use_stepping: bool = True, mode: Optional[str] = "dcop"):
        n, P = self.n, self.P
        x = np.empty((n, P)); st = np.empty(P, np.int32); it = np.empty(P, np.int32)
        uu = None if u0 is None else _check_f64(np.ascontiguousarray(u0, dtype=np.float64), (n, P), "dc(u0)")
        s = make_spec(spec, mode)
        o = DcOpts(abstol, maxiters, int(use_stepping))
        self._check(lib().cb200_dc(self._p, C.byref(s), C.byref(o), _dp(uu), _dp(x), _ip(st), _ip(it)))
        return x, st, it

    def tran(self, spec: MNASpec, t0: float, t1: float, opts: TranOpts, save_idx: Sequence[int],
             u0: Optional[np.ndarray] = None) -> Wave:
        save = np.ascontiguousarray(save_idx, dtype=np.int64)
        uu = None if u0 is None else _check_f64(np.ascontiguousarray(u0, dtype=np.float64), (self.n, self.P), "tran(u0)")
        s = make_spec(spec, "tran")
        ptr = C.c_void_p()
        self._check(lib().cb200_tran(self._p, C.byref(s), float(t0), float(t1), C.byref(opts),
                                     _lp(save), len(save), _dp(uu), C.byref(ptr)))
        return Wave(self, ptr)

    def tran_fetch(self, spec: MNASpec, t0: float, t1: float, opts: TranOpts, save_idx: Sequence[int],
                   out_u: np.ndarray, u0: Optional[np.ndarray] = None, n_segments: int = 4):
        """Fixed-step tran! with the waveform delivered into ``out_u`` ([save][T][P], ideally
        pinned), the D2H copy of each time segment overlapping the next segment's compute."""
        save = np.ascontiguousarray(save_idx, dtype=np.int64)
        uu = None if u0 is None else _check_f64(np.ascontiguousarray(u0, dtype=np.float64), (self.n, self.P), "tran_fetch(u0)")
        s = make_spec(spec, "tran")
        if opts.adaptive:
            raise ValueError("tran_fetch is the fixed-step path; use tran(...).fetch(out_u) for adaptive runs")
        T = fixed_step_points(t0, t1, opts.dt, opts.save_every)     # what the C side will write
        u_ld = _lane_block(out_u, (len(save), T), self.P, "tran_fetch(out_u)")
        t = np.empty(T, dtype=np.float64)
        count = np.empty(self.P, np.int32); status = np.empty(self.P, np.int32)
        iters = np.empty(self.P, np.int32)
        self._check(lib().cb200_tran_fetch_ld(self._p, C.byref(s), float(t0), float(t1), C.byref(opts),
                                              _lp(save), len(save), _dp(uu), int(n_segments), _dp(t),
                                              _dp(out_u) if out_u.size else None, u_ld, _ip(count), _ip(status),
                                              _ip(iters)))
        return dict(t=t, u=out_u, count=count, status=status, newton_iters=iters)

    def flop_model(self) -> dict:
        """Static flop counts of one Newton iteration's linear algebra (cb200_flop_model)."""
        o = np.zeros(8, np.int64)
        self._check(lib().cb200_flop_model(self._p, _lp(o)))
        return dict(assemble_dc=int(o[0]), assemble_tran=int(o[1]), factor_dc=int(o[2]), factor_tran=int(o[3]),
                    solve_dc=int(o[4]), solve_tran=int(o[5]), update=int(o[6]), nonlinear_devices=int(o[7]))

    def set_tstops(self, tstops: Sequence[float]):
        t = np.ascontiguousarray(tstops, dtype=np.float64)
        self._check(lib().cb200_set_tstops(self._p, _dp(t) if t.size else None, int(t.size)))

    def stats(self) -> dict:
        s = Stats()
        self._check(lib().cb200_get_stats(self._p, C.byref(s)))
        return {k: getattr(s, k) for k, _ in Stats._fields_}


def fixed_step_points(t0: float, t1: float, dt: float, save_every: int = 1) -> int:
    """Saved points per lane of a fixed-step run: the same arithmetic as tran_impl (api.cu)."""
    nsteps = int(np.floor((float(t1) - float(t0)) / float(dt) + 0.5))        # llround for positives
    se = save_every if save_every > 0 else 1
    return 1 + nsteps // se + (1 if nsteps % se else 0)


def debug_exp(x: np.ndarray) -> np.ndarray:
    """The device kernels' junction exp evaluated on the GPU (accuracy tests)."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.empty_like(x)
    rc = lib().cb200_debug_exp(_dp(x), _dp(y), int(x.size))
    if rc != OK:
        raise CB200Error(rc, (lib().cb200_last_error(None) or b"").decode())
    return y


def make_tran_opts(method="be", adaptive=False, dt=0.0, abstol=1e-10, reltol=1e-8, lte_abstol=1e-10,
                   dtmin=0.0, dtmax=0.0, max_nl_iters=10, save_every=1, max_points=0, init=0,
                   init_abstol=1e-9, init_maxiters=500, limit=False, uic_steps=10, uic_dt=1e-12,
                   class_abstol=None) -> TranOpts:
    """limit: CB200_TRAN_LIMIT -- PCNR corrector inside the transient Newton loop.
    init: 0 CedarTranOp, 1 u0 as given, 2 CedarUICOp warm-up (uic_steps BE steps of uic_dt).
    class_abstol: (vntol, iabstol, chgtol) -- CB200_TRAN_CLASS_ABSTOL, state_abstol (build.jl:276-283)."""
    m = METHODS[method] if isinstance(method, str) else int(method)
    v, i, q = class_abstol or (0.0, 0.0, 0.0)
    return TranOpts(m, int(adaptive), dt, abstol, reltol, lte_abstol, dtmin, dtmax, max_nl_iters,
                    save_every, max_points, init, init_abstol, init_maxiters,
                    (1 if limit else 0) | (4 if class_abstol else 0), int(uic_steps), 0, float(uic_dt),
                    float(v), float(i), float(q))
