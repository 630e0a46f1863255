"""ctypes binding of the CPU oracle (oracle/libcadnip_oracle.so).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and the
cpu_baseline / --impl reference legs of bench.py.  The product package never
imports this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libcadnip_oracle.so")
# cache of the compiled Verilog-A model code; a caller that must leave the tree untouched points it elsewhere
GEN_DIR = os.path.join(_HERE, "_gen")


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "cadnip_oracle.c")
    hdr = os.path.join(_HERE, "cadnip_oracle.h")
    stale = (not os.path.exists(_LIB_PATH)
             or (os.path.exists(src) and os.path.getmtime(_LIB_PATH) < max(os.path.getmtime(src), os.path.getmtime(hdr))))
    if force or stale:
        subprocess.run(["make", "-C", _HERE, "-B", "libcadnip_oracle.so"], check=True,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    return _LIB_PATH


class Spec(C.Structure):
    _fields_ = [("temp", C.c_double), ("mode", C.c_int32), ("_pad", C.c_int32),
                ("gmin", C.c_double), ("gshunt", C.c_double), ("srcFact", C.c_double),
                ("tnom", C.c_double), ("abstol", C.c_double), ("reltol", C.c_double),
                ("vntol", C.c_double), ("iabstol", C.c_double)]


class Netlist(C.Structure):
    _fields_ = [("n_dev", C.c_int32), ("n_nodes", C.c_int32),
                ("kind", C.POINTER(C.c_int32)), ("flags", C.POINTER(C.c_int32)),
                ("node_ptr", C.POINTER(C.c_int32)), ("nodes", C.POINTER(C.c_int32)),
                ("par_ptr", C.POINTER(C.c_int32)), ("par", C.POINTER(C.c_double))]


class TranOpts(C.Structure):
    _fields_ = [("method", C.c_int32), ("adaptive", C.c_int32),
                ("dt", C.c_double), ("abstol", C.c_double), ("reltol", C.c_double),
                ("lte_abstol", C.c_double), ("dtmin", C.c_double), ("dtmax", C.c_double),
                ("max_nl_iters", C.c_int32), ("save_every", C.c_int32),
                ("max_points", C.c_int32), ("init", C.c_int32),
                ("init_abstol", C.c_double), ("init_maxiters", C.c_int32), ("flags", C.c_int32),
                ("uic_steps", C.c_int32), ("_pad", C.c_int32), ("uic_dt", C.c_double),
                ("vntol", C.c_double), ("iabstol", C.c_double), ("chgtol", C.c_double)]


_MODES = {"dcop": 0, "tran": 1, "tranop": 2, "ac": 3}
_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB_PATH)
        L = _lib
        dp, ip, lp = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_int64)
        L.ora_pwl_at_time.restype = C.c_double
        L.ora_pwl_at_time.argtypes = [dp, dp, C.c_int, C.c_double]
        L.ora_pulse_at_time.restype = C.c_double
        L.ora_pulse_at_time.argtypes = [C.c_double] * 8
        L.ora_sin_wave.restype = C.c_double
        L.ora_sin_wave.argtypes = [C.c_double] * 7
        L.ora_sind.restype = C.c_double
        L.ora_sind.argtypes = [C.c_double]
        L.ora_pnjlim.restype = C.c_double
        L.ora_pnjlim.argtypes = [C.c_double] * 4 + [C.POINTER(C.c_int)]
        L.ora_diode_iv.restype = None
        L.ora_diode_iv.argtypes = [C.c_double] * 3 + [dp, dp]
        L.ora_diode_vcrit.restype = C.c_double
        L.ora_diode_vcrit.argtypes = [C.c_double] * 3
        L.ora_sparse_coo.restype = C.c_int64
        L.ora_sparse_coo.argtypes = [C.c_int64, C.c_int64, lp, lp, dp, lp, lp, dp, lp]
        L.ora_expand_breakpoints.restype = C.c_int64
        L.ora_expand_breakpoints.argtypes = [C.c_int, dp, C.c_int, C.c_double, C.c_double, dp, C.c_int64]
        L.ora_detect_structure.restype = C.c_void_p
        L.ora_detect_structure.argtypes = [C.POINTER(Netlist), C.POINTER(Spec)]
        L.ora_build.restype = C.c_void_p
        L.ora_build.argtypes = [C.POINTER(Netlist), C.POINTER(Spec), C.c_double, dp, C.c_int64]
        L.ora_ctx_free.argtypes = [C.c_void_p]
        L.ora_ctx_sizes.argtypes = [C.c_void_p] + [lp] * 7
        L.ora_ctx_coo.argtypes = [C.c_void_p, lp, lp, dp, lp, lp, dp, lp, dp, dp]
        L.ora_compile_structure.restype = C.c_void_p
        L.ora_compile_structure.argtypes = [C.POINTER(Netlist), C.POINTER(Spec), C.c_void_p]
        L.ora_structure_free.argtypes = [C.c_void_p]
        L.ora_structure_sizes.argtypes = [C.c_void_p, lp, lp]
        L.ora_structure_arrays.argtypes = [C.c_void_p, lp, lp, lp, lp, lp, lp, dp, dp]
        L.ora_create_workspace.restype = C.c_void_p
        L.ora_create_workspace.argtypes = [C.c_void_p]
        L.ora_workspace_free.argtypes = [C.c_void_p]
        L.ora_fast_rebuild.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Spec), dp, C.c_double,
                                       C.c_int, dp, dp, dp, dp]
        L.ora_dc_pcnr_newton.restype = C.c_int
        L.ora_dc_pcnr_newton.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Spec), dp, C.c_double,
                                         C.c_int, C.POINTER(C.c_int)]
        L.ora_dc_solve_with_fallbacks.restype = C.c_int
        L.ora_dc_solve_with_fallbacks.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Spec), dp,
                                                  C.c_double, C.c_int, C.c_int, C.POINTER(C.c_int)]
        L.ora_solve_dc.restype = C.c_int
        L.ora_solve_dc.argtypes = [C.POINTER(Netlist), C.POINTER(Spec), dp, C.c_int64, C.c_double,
                                   C.c_int, dp, C.c_int64, lp, C.POINTER(C.c_int)]
        L.ora_tran.restype = C.c_int
        L.ora_tran.argtypes = [C.POINTER(Netlist), C.POINTER(Spec), C.c_double, C.c_double,
                               C.POINTER(TranOpts), lp, C.c_int, dp, dp, dp, C.c_int64, lp, lp, lp, dp]
        L.ora_sweep_dc.restype = C.c_int
        L.ora_sweep_dc.argtypes = [C.POINTER(Netlist), dp, C.c_int64, C.c_int64, C.POINTER(Spec),
                                   C.c_double, C.c_int, C.c_int, dp, C.c_int64, ip, ip, C.c_int]
        L.ora_sweep_tran.restype = C.c_int
        L.ora_sweep_tran.argtypes = [C.POINTER(Netlist), dp, C.c_int64, C.c_int64, C.POINTER(Spec),
                                     C.c_double, C.c_double, C.POINTER(TranOpts), lp, C.c_int,
                                     dp, dp, C.c_int64, ip, ip, lp, C.c_int]
        L.ora_num_threads.restype = C.c_int
        L.ora_set_va_table.restype = None
        L.ora_set_va_table.argtypes = [C.c_void_p]
    return _lib


def _dp(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))


def _lp(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_int64))


def _ip(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_int32))


def make_spec(spec=None, **over) -> Spec:
    """Accepts anything with MNASpec's fields (duck-typed), or keyword overrides."""
    d = dict(temp=27.0, mode="tran", gmin=1e-12, gshunt=0.0, srcFact=1.0, tnom=27.0,
             abstol=1e-12, reltol=1e-3, vntol=1e-6, iabstol=1e-12)
    if spec is not None:
        for k in d:
            d[k] = getattr(spec, k)
    d.update(over)
    mode = d["mode"]
    return Spec(d["temp"], _MODES[mode] if isinstance(mode, str) else int(mode), 0, d["gmin"],
                d["gshunt"], d["srcFact"], d["tnom"], d["abstol"], d["reltol"], d["vntol"],
                d["iabstol"])


def make_tran_opts(method=0, adaptive=0, dt=0.0, abstol=1e-10, reltol=1e-8, lte_abstol=1e-10,
                   dtmin=0.0, dtmax=0.0, max_nl_iters=10, save_every=1, max_points=0, init=0,
                   init_abstol=1e-9, init_maxiters=500, limit=False, uic_steps=10, uic_dt=1e-12,
                   class_abstol=None) -> TranOpts:
    """init: 0 CedarTranOp, 1 u0 given as is, 2 CedarUICOp warm-up (uic_steps BE steps of uic_dt).
    class_abstol: (vntol, iabstol, chgtol) of state_abstol (build.jl:276-283) for the LTE test."""
    v, i, q = class_abstol or (0.0, 0.0, 0.0)
    return TranOpts(method, adaptive, dt, abstol, reltol, lte_abstol, dtmin, dtmax, max_nl_iters,
                    save_every, max_points, init, init_abstol, init_maxiters,
                    (1 if limit else 0) | (4 if class_abstol else 0), uic_steps, 0, uic_dt, v, i, q)


class OracleNetlist:
    """Holds the numpy arrays alive behind an ora_netlist for one lane (or a lane
    matrix, for the sweep drivers)."""

    def __init__(self, tables: dict, lane: int = 0):
        self.kind = np.ascontiguousarray(tables["kind"], dtype=np.int32)
        self.flags = np.ascontiguousarray(tables["flags"], dtype=np.int32)
        self.node_ptr = np.ascontiguousarray(tables["node_ptr"], dtype=np.int32)
        self.nodes = np.ascontiguousarray(tables["nodes"], dtype=np.int32)
        self.par_ptr = np.ascontiguousarray(tables["par_ptr"], dtype=np.int32)
        self.par_lanes = np.ascontiguousarray(tables["par"], dtype=np.float64)   # [P][npar]
        self.n_nodes = int(tables["n_nodes"])
        self.P, self.npar = self.par_lanes.shape
        self.lane = lane
        self.c = self._make(lane)

    def _make(self, lane: int) -> Netlist:
        row = self.par_lanes[lane]
        return Netlist(len(self.kind), self.n_nodes, _ip(self.kind), _ip(self.flags),
                       _ip(self.node_ptr), _ip(self.nodes), _ip(self.par_ptr),
                       row.ctypes.data_as(C.POINTER(C.c_double)))

    def for_lane(self, lane: int) -> "OracleNetlist":
        o = OracleNetlist.__new__(OracleNetlist)
        o.__dict__.update(self.__dict__)
        o.lane = lane
        o.c = self._make(lane)
        return o


class Structure:
    """detect_structure + compile_structure + workspace for one lane."""

    def __init__(self, nl: OracleNetlist, spec: Spec):
        L = lib()
        self.nl, self.spec = nl, spec
        self.ctx = L.ora_detect_structure(C.byref(nl.c), C.byref(spec))
        sz = [C.c_int64() for _ in range(7)]
        L.ora_ctx_sizes(self.ctx, *[C.byref(s) for s in sz])
        (self.n_nodes, self.n_currents, self.n_charges, self.n_limits,
         self.nG, self.nC, self.nb) = [s.value for s in sz]
        self.cs = L.ora_compile_structure(C.byref(nl.c), C.byref(spec), self.ctx)
        n, nnz = C.c_int64(), C.c_int64()
        L.ora_structure_sizes(self.cs, C.byref(n), C.byref(nnz))
        self.n, self.nnz = n.value, nnz.value
        self.ws = L.ora_create_workspace(self.cs)

    def coo(self):
        L = lib()
        G_I = np.zeros(self.nG, np.int64); G_J = np.zeros(self.nG, np.int64); G_V = np.zeros(self.nG)
        C_I = np.zeros(self.nC, np.int64); C_J = np.zeros(self.nC, np.int64); C_V = np.zeros(self.nC)
        b_I = np.zeros(self.nb, np.int64); b_V = np.zeros(self.nb)
        li = np.zeros(self.n_limits)
        L.ora_ctx_coo(self.ctx, _lp(G_I), _lp(G_J), _dp(G_V), _lp(C_I), _lp(C_J), _dp(C_V),
                      _lp(b_I), _dp(b_V), _dp(li))
        return dict(G_I=G_I, G_J=G_J, G_V=G_V, C_I=C_I, C_J=C_J, C_V=C_V, b_I=b_I, b_V=b_V,
                    limit_init=li)

    def arrays(self):
        L = lib()
        colptr = np.zeros(self.n + 1, np.int64); rowval = np.zeros(self.nnz, np.int64)
        gmap = np.zeros(self.nG, np.int64); cmap = np.zeros(self.nC, np.int64)
        brow = np.zeros(self.nb, np.int64); diag = np.zeros(self.n_nodes, np.int64)
        g0 = np.zeros(self.nnz); c0 = np.zeros(self.nnz)
        L.ora_structure_arrays(self.cs, _lp(colptr), _lp(rowval), _lp(gmap), _lp(cmap), _lp(brow),
                               _lp(diag), _dp(g0), _dp(c0))
        return dict(colptr=colptr, rowval=rowval, G_coo_to_idx=gmap, C_coo_to_idx=cmap,
                    b_resolved=brow, G_diag_idx=diag, G_nz0=g0, C_nz0=c0)

    def rebuild(self, u: Optional[np.ndarray], t: float = 0.0, initjct: bool = False, spec=None):
        L = lib()
        G = np.zeros(self.nnz); Cm = np.zeros(self.nnz); b = np.zeros(self.n)
        lw = np.zeros(self.n_limits)
        uu = np.zeros(self.n) if u is None else np.ascontiguousarray(u, dtype=np.float64)
        L.ora_fast_rebuild(self.ws, self.cs, C.byref(spec or self.spec), _dp(uu), t, int(initjct),
                           _dp(G), _dp(Cm), _dp(b), _dp(lw))
        return G, Cm, b, lw

    def dense(self, nz: np.ndarray) -> np.ndarray:
        a = self.arrays()
        M = np.zeros((self.n, self.n))
        for j in range(self.n):
            for idx in range(a["colptr"][j], a["colptr"][j + 1]):
                M[a["rowval"][idx - 1] - 1, j] = nz[idx - 1]
        return M

    def pcnr(self, u0=None, abstol=1e-10, maxiters=100, spec=None):
        L = lib()
        u = np.zeros(self.n) if u0 is None else np.array(u0, dtype=np.float64)
        it = C.c_int()
        ok = L.ora_dc_pcnr_newton(self.ws, self.cs, C.byref(spec or self.spec), _dp(u), abstol,
                                  maxiters, C.byref(it))
        return u, bool(ok), it.value

    def dc(self, u0=None, abstol=1e-10, maxiters=100, use_stepping=True, spec=None):
        L = lib()
        u = np.zeros(self.n) if u0 is None else np.array(u0, dtype=np.float64)
        it = C.c_int()
        ok = L.ora_dc_solve_with_fallbacks(self.ws, self.cs, C.byref(spec or self.spec), _dp(u),
                                           abstol, maxiters, int(use_stepping), C.byref(it))
        return u, bool(ok), it.value

    def close(self):
        L = lib()
        if self.ws:
            L.ora_workspace_free(self.ws); self.ws = None
        if self.cs:
            L.ora_structure_free(self.cs); self.cs = None
        if self.ctx:
            L.ora_ctx_free(self.ctx); self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def solve_dc(nl: OracleNetlist, spec: Spec, u0=None, abstol=1e-10, maxiters=100, cap=4096):
    L = lib()
    x = np.zeros(cap)
    n = C.c_int64(); it = C.c_int()
    u0a = None if u0 is None else np.ascontiguousarray(u0, dtype=np.float64)
    ok = L.ora_solve_dc(C.byref(nl.c), C.byref(spec), _dp(u0a), 0 if u0a is None else len(u0a),
                        abstol, maxiters, _dp(x), cap, C.byref(n), C.byref(it))
    return x[:n.value].copy(), ok == 1, it.value


def tran(nl: OracleNetlist, spec: Spec, t0: float, t1: float, opts: TranOpts,
         save_idx: Sequence[int], u0=None, cap_T: Optional[int] = None):
    L = lib()
    save = np.ascontiguousarray(save_idx, dtype=np.int64)
    if cap_T is None:
        if opts.adaptive:
            cap_T = max(int(opts.max_points), 16)
        else:
            cap_T = int(round((t1 - t0) / opts.dt)) // max(opts.save_every, 1) + 3
    ot = np.zeros(cap_T); ou = np.zeros((cap_T, len(save)))
    T = C.c_int64(); it = C.c_int64(); rej = C.c_int64()
    xf = np.zeros(8192)
    u0a = None if u0 is None else np.ascontiguousarray(u0, dtype=np.float64)
    st = L.ora_tran(C.byref(nl.c), C.byref(spec), t0, t1, C.byref(opts), _lp(save), len(save),
                    _dp(u0a), _dp(ot), _dp(ou), cap_T, C.byref(T), C.byref(it), C.byref(rej), _dp(xf))
    Tn = min(T.value, cap_T)
    return dict(t=ot[:Tn].copy(), u=ou[:Tn].copy(), status=st, newton_iters=it.value,
                rejected=rej.value, T=T.value, x_final=xf)


def sweep_dc(nl: OracleNetlist, spec: Spec, n: int, abstol=1e-10, maxiters=100,
             continuation=False, nthreads=0):
    L = lib()
    P = nl.P
    x = np.zeros((P, n)); st = np.zeros(P, np.int32); it = np.zeros(P, np.int32)
    L.ora_sweep_dc(C.byref(nl.c), _dp(nl.par_lanes), P, nl.npar, C.byref(spec), abstol, maxiters,
                   int(continuation), _dp(x), n, _ip(st), _ip(it), nthreads)
    return x, st, it


def sweep_tran(nl: OracleNetlist, spec: Spec, t0, t1, opts: TranOpts, save_idx, nthreads=0,
               lanes: Optional[slice] = None):
    L = lib()
    par = nl.par_lanes if lanes is None else np.ascontiguousarray(nl.par_lanes[lanes])
    P = par.shape[0]
    save = np.ascontiguousarray(save_idx, dtype=np.int64)
    if opts.adaptive:
        cap_T = max(int(opts.max_points), 16)
        ot = np.zeros((P, cap_T))
    else:
        cap_T = int(round((t1 - t0) / opts.dt)) // max(opts.save_every, 1) + 3
        ot = np.zeros(cap_T)
    ou = np.zeros((P, cap_T, len(save)))
    Tn = np.zeros(P, np.int32); st = np.zeros(P, np.int32); it = np.zeros(P, np.int64)
    L.ora_sweep_tran(C.byref(nl.c), _dp(par), P, nl.npar, C.byref(spec), t0, t1, C.byref(opts),
                     _lp(save), len(save), _dp(ot), _dp(ou), cap_T, _ip(Tn), _ip(st), _lp(it),
                     nthreads)
    return dict(t=ot, u=ou, T=Tn, status=st, newton_iters=it)


_va_libs = []


def load_va_models(models, count_ops: bool = False) -> None:
    """Compile the C the product's emitter generated for these Verilog-A modules
    (gcc, cached under GEN_DIR) and register it with the oracle.  The model index
    is the position in ``models`` (== dev_flags of the lowered circuit).
    count_ops: build the op-counting variant (verilog_a.instrument_ops) -- `va_op_counts()` then
    returns the flops / transcendentals the model code EXECUTED since `va_op_reset()`; counting
    runs must be single-threaded (the counter is a plain global)."""
    import hashlib
    import sys
    global _va_count_lib
    if isinstance(models, str):                  # LoweredCircuit.va_c_source
        src = models
    else:
        sys.path.insert(0, os.path.dirname(_HERE))
        import cadnip_b200.verilog_a as va
        src = va.c_source(models)
    if count_ops:
        sys.path.insert(0, os.path.dirname(_HERE))
        import cadnip_b200.verilog_a as va
        src = va.instrument_ops(src)
    os.makedirs(GEN_DIR, exist_ok=True)
    h = hashlib.sha256(src.encode()).hexdigest()[:16]
    so = os.path.join(GEN_DIR, f"va_{h}.so")
    if not os.path.exists(so):
        cfile = os.path.join(GEN_DIR, f"va_{h}.c")
        with open(cfile, "w") as f:
            f.write(src)
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
        subprocess.run([cc, "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-o", so + ".tmp", cfile, "-lm"],
                       check=True)
        os.replace(so + ".tmp", so)
    L = C.CDLL(so)
    _va_libs.append(L)
    _va_count_lib = L if count_ops else None
    lib().ora_set_va_table(C.cast(L.ora_va_table, C.c_void_p))


_va_count_lib = None


def va_op_reset() -> None:
    ops = (C.c_longlong * 3).in_dll(_va_count_lib, "ora_va_ops")
    ops[0] = ops[1] = ops[2] = 0


def va_op_counts():
    """(flops, transcendentals, model calls) executed by the instrumented model code since
    va_op_reset()."""
    ops = (C.c_longlong * 3).in_dll(_va_count_lib, "ora_va_ops")
    return int(ops[0]), int(ops[1]), int(ops[2])


_detect_keep = None


def set_detect_override(seq) -> None:
    """Replay a recorded voltage-dependent-charge detection outcome (LoweredCircuit.va_detect_seq)
    instead of probing; None restores the probe."""
    global _detect_keep
    L = lib()
    L.ora_set_detect_override.argtypes = [C.POINTER(C.c_int32), C.c_int64]
    L.ora_set_detect_override.restype = None
    if seq is None:
        _detect_keep = None
        L.ora_set_detect_override(None, 0)
        return
    _detect_keep = np.ascontiguousarray(seq, dtype=np.int32)
    L.ora_set_detect_override(_detect_keep.ctypes.data_as(C.POINTER(C.c_int32)), len(_detect_keep))


def last_dc_tier() -> int:
    """Tier of _dc_solve_with_fallbacks that produced this thread's last DC result (-1: none)."""
    return int(lib().ora_last_dc_tier())


def set_linear_solver(kind: int) -> None:
    """0: dense partial-pivot LU (the checker, default); 1: fixed-pattern sparse LU (timed baseline)."""
    lib().ora_set_linear_solver(int(kind))


def num_threads() -> int:
    return lib().ora_num_threads()
