"""CPU tests of the host logic: sweep iterator algebra (test/sweep.jl:49-180), the
recording MNAContext (test/mna/core.jl:53-233), lowering, the C-ABI surface, and the
multi-GPU sharding plumbing under gloo (world_size 2)."""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

import cadnip_b200 as cb
import circuits
from cadnip_b200 import (MNAContext, ZERO_VECTOR, get_node, stamp_G, stamp_C, stamp_b, stamp,
                         Resistor, VoltageSource, Sweep, ProductSweep, TandemSweep, SerialSweep,
                         CircuitSweep, sweepvars, split_axes, sweepify)
from cadnip_b200 import backend, distributed

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- MNAContext ------------------------------------------------------------
def test_context_basics_and_stamping_primitives():
    ctx = MNAContext()
    assert get_node(ctx, "gnd") == 0 and get_node(ctx, "0") == 0 and get_node(ctx, "gnd!") == 0
    n1 = get_node(ctx, "n1"); n2 = get_node(ctx, "n2")
    assert (n1, n2) == (1, 2) and get_node(ctx, "n1") == 1 and get_node(ctx, 7) == 7
    stamp_G(ctx, n1, n1, 1.0); stamp_G(ctx, n1, n2, -1.0); stamp_G(ctx, n2, n1, -1.0); stamp_G(ctx, n2, n2, 1.0)
    assert ctx.G_I == [1, 1, 2, 2] and ctx.G_J == [1, 2, 1, 2] and ctx.G_V == [1.0, -1.0, -1.0, 1.0]
    stamp_C(ctx, n1, n1, 1e-6)
    assert len(ctx.C_V) == 1
    stamp_b(ctx, n1, 5.0); stamp_b(ctx, n1, 3.0)
    assert ctx.b_I == [1, 1] and sum(ctx.b_V) == 8.0
    stamp_G(ctx, 0, n1, 1.0); stamp_G(ctx, n1, 0, 1.0); stamp_b(ctx, 0, 5.0)   # ground: ignored, not counted
    assert len(ctx.G_V) == 4 and len(ctx.b_V) == 2
    i1 = cb.alloc_current(ctx, "I_", "V1")
    l1 = cb.alloc_limit(ctx, "vdlim", "D1", 1, 2, init=0.66)
    n3 = cb.alloc_internal_node(ctx, "a_int", "D1")
    assert n3 == 3 and ctx.node_names[-1] == "D1_a_int" and ctx.internal_node_flags[2]
    # deferred resolution: indices move when nodes are added later (context.jl:577-581)
    assert cb.resolve_index(ctx, i1) == 4 and cb.resolve_index(ctx, l1) == 5
    assert ctx.limit_names == ["D1_vdlim"] and ctx.limit_init == [0.66] and cb.system_size(ctx) == 5
    assert ctx.get_current_idx("I_V1") == cb.CurrentIndex(1)
    cb.reset_for_restamping(ctx)
    assert ctx.n_limits == 0 and ctx.n_nodes == 0 and not ctx.G_I


def test_zero_vector_and_sources_reject_closures():
    assert ZERO_VECTOR[5] == 0.0 and len(ZERO_VECTOR) == 0
    with pytest.raises(TypeError):
        VoltageSource(0.0, tran=lambda t: t)


# ---- sweeps (test/sweep.jl:49-180) ------------------------------------------
def test_sweep_iterators():
    s = Sweep(R1=np.arange(0.1, 1.01, 0.1))
    assert len(s) == 10 and s.sweepvars() == {"R1"}
    assert Sweep("R1", [1, 2]) == Sweep(("R1", [1, 2])) == Sweep(R1=[1, 2])
    with pytest.raises(ValueError):
        Sweep(a=[1], b=[2])
    ps = ProductSweep(R1=[1, 2, 3, 4], R2=[10, 20, 30])
    pts = list(ps)
    assert len(ps) == 12 and ps.size() == (4, 3)
    assert pts[0] == (("R1", 1), ("R2", 10)) and pts[1] == (("R1", 2), ("R2", 10)) and pts[4] == (("R1", 1), ("R2", 20))
    ts = TandemSweep(R1=[1, 2, 3], R2=[4, 5, 6])
    assert list(ts)[1] == (("R1", 2), ("R2", 5)) and len(ts) == 3
    with pytest.raises(ValueError):
        TandemSweep(R1=[1, 2], R2=[1])
    ss = SerialSweep(R1=[1, 2], R2=[7])
    assert list(ss) == [(("R1", 1), ("R2", None)), (("R1", 2), ("R2", None)), (("R1", None), ("R2", 7))]
    nested = ProductSweep(Sweep(A=[1, 2]), TandemSweep(B=[1, 2, 3], C=[4, 5, 6]))
    assert len(nested) == 6 and list(nested)[3] == (("A", 2), ("B", 2), ("C", 5))
    assert sweepvars(nested) == {"A", "B", "C"}
    assert ProductSweep(R1=[1, 2]) == Sweep(R1=[1, 2])
    outer, inner = split_axes(ProductSweep(A=range(1, 11), B=range(1, 9), C=range(1, 7), D=range(1, 5)), ["A", "C"])
    assert outer.sweepvars() == {"B", "D"} and len(outer) == 32
    assert inner.sweepvars() == {"A", "C"} and len(inner) == 60
    assert len(sweepify([dict(r1=range(1, 11), r2=range(1, 11)), dict(r3=range(1, 11))])) == 110
    assert cb.find_param_ranges(ps)["R2"] == (10.0, 30.0, 3)


def test_columns_match_iteration_order():
    sweeps = [ProductSweep(R1=[1.0, 2.0, 3.0], R2=[10.0, 20.0], R3=[5.0, 6.0]),
              ProductSweep(Sweep(A=[1.0, 2.0]), TandemSweep(B=[1.0, 2.0, 3.0], C=[4.0, 5.0, 6.0])),
              SerialSweep(Sweep(A=[1.0, 2.0]), ProductSweep(A=[3.0], B=[8.0, 9.0]))]
    for sw in sweeps:
        vals, isset = sw.columns()
        for lane, pt in enumerate(sw):
            for k, v in pt:
                if v is None:
                    assert not isset[k][lane]
                else:
                    assert isset[k][lane] and vals[k][lane] == v


def test_circuit_sweep_and_alter():
    cs = CircuitSweep(circuits.divider, ProductSweep(R1=[100.0, 200.0], R2=[100.0, 200.0, 300.0]))
    assert len(cs) == 6 and cs.size() == (2, 3) and cs.sweepvars() == {"R1", "R2"}
    first = next(iter(cs))
    assert first.params.R1 == 100.0 and first.params.R2 == 100.0
    last = list(cs)[-1]
    assert last.params.R1 == 200.0 and last.params.R2 == 300.0
    c = cb.MNACircuit(circuits.divider, R1=1.0, R2=2.0)
    c2 = cb.alter(c, R1=5.0, R2=None, **{"inner.params.R3": 7.0})
    assert c2.params.R1 == 5.0 and c2.params.R2 == 2.0 and c2.params.inner.params.R3 == 7.0 and c.params.R1 == 1.0
    # with_mode(circuit, mode) resets the spec to defaults except temp (solve.jl:1976-1979)
    c3 = cb.with_mode(cb.MNACircuit(circuits.divider, spec=cb.MNASpec(temp=50.0, gmin=1e-9), R1=1.0, R2=1.0), "dcop")
    assert c3.spec.mode == "dcop" and c3.spec.temp == 50.0 and c3.spec.gmin == 1e-12
    assert cb.with_mode(cb.MNASpec(gmin=1e-9), "dcop").gmin == 1e-9
    # serial sweep leaves unset variables at the circuit default
    cs2 = CircuitSweep(circuits.divider, SerialSweep(R1=[1.0, 2.0], R2=[9.0]), R1=100.0, R2=200.0)
    p, P = cs2.lane_params()
    assert list(p.R1) == [1.0, 2.0, 1.0] or list(p.R1) == [1.0, 2.0, 100.0]
    assert list(p.R2)[2] == 9.0


# ---- lowering ---------------------------------------------------------------
def test_lowering_clipper_c2_shape():
    """SURVEY 8d C2: n = 4 (2 nodes + I_V1 + 1 limit), nnz = 8 with the stated entries."""
    from cadnip_b200.workloads import clipper_sweep
    cs = clipper_sweep(4, 3)
    params, P = cs.lane_params()
    lc = cb.lower(cs.builder, params, cb.MNASpec(), P=P)
    assert P == 12 and lc.n == 4 and lc.unknown_names() == ["in", "out", "I_V1", "D1_vdlim"]
    coords = sorted(set(zip(list(lc.G_I) + list(lc.C_I), list(lc.G_J) + list(lc.C_J))))
    assert coords == sorted([(1, 1), (1, 2), (2, 1), (2, 2), (1, 3), (3, 1), (4, 2), (4, 4)])
    assert lc.n_lane_cols == 2 and lc.lane_soa.shape == (2, 12)
    # R is the fastest axis
    assert lc.lane_soa[0, 0] != lc.lane_soa[0, 1] and lc.lane_soa[1, 0] == lc.lane_soa[1, 1]
    t = lc.netlist_tables()
    assert t["par"].shape[0] == 12 and list(t["kind"]) == [4, 1, 10, 2]
    # the diode's vcrit is uniform here (Is, Vt, n are not swept)
    assert lc.limit_init_ref[0] >= 0


def test_structural_boundary_is_rejected():
    def bad(params, spec, t=0.0, x=ZERO_VECTOR, ctx=None):
        ctx = MNAContext()
        a = get_node(ctx, "a")
        stamp(VoltageSource(1.0), ctx, a, 0)
        if params.rs > 0:                       # branches on a swept value
            stamp(Resistor(params.rs), ctx, a, 0)
        return ctx
    cs = CircuitSweep(bad, Sweep(rs=[0.0, 1.0]))
    params, P = cs.lane_params()
    with pytest.raises(cb.StructuralSweepError):
        cb.lower(cs.builder, params, cb.MNASpec(), P=P)


# ---- C ABI ------------------------------------------------------------------
def test_c_abi_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "cadnip_b200.h")).read()
    declared = sorted(set(re.findall(r"\b(cb200_[a-z0-9_]+)\s*\(", hdr)))
    assert declared == sorted(backend.EXPORTED_SYMBOLS)
    backend.build_library()
    L = C.CDLL(backend.LIB_PATH)
    for sym in declared:
        assert hasattr(L, sym), sym
    assert backend.lib().cb200_abi_version() == 2


def test_no_cpu_fallback_without_device():
    """Without a CUDA device the product must fail loudly, never fall back."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lc = cb.lower_circuit(cb.MNACircuit(circuits.rectifier(True)))
    with pytest.raises(backend.CB200Error) as e:
        backend.Handle(lc)
    assert e.value.code == backend.ENODEVICE
    with pytest.raises(backend.CB200Error):
        cb.dc(cb.MNACircuit(circuits.rectifier(True)))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "cadnip.jl_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cpp", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "cadnip_oracle" not in src and "oracle/" not in src, f


# ---- sharding under gloo -----------------------------------------------------
def test_shard_slices_cover_sweep():
    for P in (0, 1, 7, 8, 65536, 100000):
        for world in (1, 2, 3, 8):
            sl = [distributed.shard_slice(P, r, world) for r in range(world)]
            got = [i for s in sl for i in range(s.start, s.stop)]
            assert got == list(range(P))


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        P = 11

        def run_local(sl):
            lanes = np.arange(sl.start, sl.stop, dtype=np.float64)
            return np.stack([lanes, lanes * 10.0])          # [save][lane]

        full = distributed.run_sharded(P, run_local, lane_axis=-1)
        q.put((rank, None if full is None else full.tolist()))
    finally:
        dist.destroy_process_group()


def test_gather_world_size_2_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    assert res[1] is None
    full = np.array(res[0])
    assert full.shape == (2, 11)
    assert np.array_equal(full[0], np.arange(11.0)) and np.array_equal(full[1], np.arange(11.0) * 10)


# ---- the emitter (host only) -------------------------------------------------
def test_emitter_generates_compilable_source(tmp_path):
    """cb200_emit_source -> nvcc (sm_100a cross-compile, no GPU needed)."""
    import subprocess
    import cadnip_oracle as ora
    from cadnip_b200.workloads import clipper_builder

    def builder(params, spec, t=0.0, x=cb.ZERO_VECTOR, ctx=None):
        # the C2 clipper plus a PWL-driven branch: the PWL table walk must not index the
        # parameter tables (and through them the register workspace) dynamically
        ctx = clipper_builder(params, spec, t, x=x, ctx=ctx)
        aux = cb.get_node(ctx, "aux")
        cb.stamp(cb.VoltageSource(0.0, tran=cb.PWLWave([0.0, 1e-4, 2e-4, 5e-4], [0.0, 1.0, 1.0, 0.0]), name="V2"),
                 ctx, aux, 0)
        cb.stamp(cb.Resistor(params.R, name="R2"), ctx, aux, cb.get_node(ctx, "out"))
        return ctx
    cs = cb.CircuitSweep(builder, cb.ProductSweep(R=[1e2, 1e3, 1e4, 1e5], C=[1e-10, 1e-9, 1e-8]))
    params, P = cs.lane_params()
    lc = cb.lower(cs.builder, params, cb.MNASpec(mode="tran"), P=P)
    S = ora.Structure(ora.OracleNetlist(lc.netlist_tables()), ora.make_spec(mode="tran"))
    G, Cm, _, _ = S.rebuild(np.zeros(lc.n), initjct=True)       # nominal magnitudes for the pivot choice
    src = backend.emit_source(lc, np.abs(G), np.abs(G + 1e6 * Cm), P=65536)
    assert "cb200_spec_tran_fixed_kernel" in src and "eval_device<1>(pg, w, 2," in src
    assert "__device__ constexpr int k_SProg_dev_node[]" in src      # tables at namespace scope, not on the stack
    assert "__launch_bounds__(kBlock, kMinBlocks)" in src and "constexpr int kMinBlocks = 7;" in src
    # one time loop (tran_fixed_body of lane_kernels.cuh, with the bypass as a program trait) and one fixed-step kernel
    assert "static constexpr bool kBypass = true;" in src and "tran_fixed_body(pg, lu, w, p, sp, a);" in src
    assert "spec_tran_fixed_body" not in src and "pair" not in src
    cu = tmp_path / "spec.cu"
    cu.write_text(src)
    nvcc = backend.nvcc_path()
    if nvcc is None:
        pytest.skip("nvcc not available")
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler",
                        "-fPIC", "-shared", "-Xptxas", "-v", "-I", os.path.join(ROOT, "cadnip.jl_b200", "csrc"),
                        "-o", str(tmp_path / "spec.so"), str(cu)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    # the lane state must live in registers: no local-memory frame beyond libm's slow path
    frames = [int(x) for x in re.findall(r"(\d+) bytes stack frame", r.stderr)]
    assert max(frames) <= 64, frames


def _random_matrix_on_pattern(colptr, rowval, rng):
    """Random values on a CSC pattern (1-based), made safely non-singular: strong diagonal where the
    pattern has one, O(1) couplings elsewhere (MNA source rows have a structurally zero diagonal)."""
    n = len(colptr) - 1
    A = np.zeros((n, n))
    J = rng.uniform(-1.0, 1.0, len(rowval))
    for j in range(n):
        for q in range(colptr[j] - 1, colptr[j + 1] - 1):
            i = rowval[q] - 1
            if i == j:
                J[q] = rng.uniform(4.0, 8.0) * n ** 0.5
            A[i, j] = J[q]
    return J, A


def test_level_schedule_equals_serial_schedule_on_host():
    """The level-scheduled refactor / solves of the lane-per-warp kernels (symbolic.cpp:
    build_level_schedule) run on the host next to the serial static-pivot schedule: identical bits,
    and both solve the system.  Covers the gf180 flip-flop (n = 145) and small circuits."""
    import test_gpu_parity as tg
    rng = np.random.default_rng(20261018)
    cases = [("dff", cb.LoweredCircuit.load(os.path.join(os.path.dirname(__file__), "golden", "va_mos1_dff.json.gz")))]
    for name, cs in tg.SWEEPS:
        params, P = cs.lane_params()
        cases.append((name, cb.lower(cs.builder, params, cb.MNASpec(mode="tran"), P=P)))
    for name, lc in cases:
        colptr, rowval = backend.host_lu_check(lc)
        assert colptr[0] == 1 and colptr[-1] == len(rowval) + 1
        for trial in range(3):
            J, A = _random_matrix_on_pattern(colptr, rowval, rng)
            if abs(np.linalg.det(A / np.abs(A).max())) < 1e-200 or np.linalg.cond(A) > 1e10:
                continue
            rhs = rng.uniform(-1.0, 1.0, len(colptr) - 1)
            xs, xl, info = backend.host_lu_check(lc, J, rhs)
            assert np.array_equal(xs, xl), (name, trial)
            ref = np.linalg.solve(A, rhs)
            assert np.allclose(xs, ref, rtol=1e-8, atol=1e-10 * np.abs(ref).max()), (name, trial)
            assert 1 <= info["factor_levels"] <= info["n"] and info["nlu"] >= info["nnz"]
            if name == "dff":
                assert info["n"] == 145 and info["factor_levels"] < 40      # 145 pivots, a few levels


# ---- round-2 host logic -------------------------------------------------------
def test_lowered_circuit_json_round_trip(tmp_path):
    """LoweredCircuit.save / load (gzip'd JSON, the fixture format): every table bit-exact,
    breakpoints usable by expand_breakpoints."""
    from cadnip_b200.workloads import clipper_sweep, inverter_sweep
    for cs in (clipper_sweep(3, 2), inverter_sweep(2, 2, 2)):
        params, P = cs.lane_params()
        lc = cb.lower(cs.builder, params, cb.MNASpec(mode="tran"), P=P)
        path = str(tmp_path / "lc.json.gz")
        lc.save(path)
        l2 = cb.LoweredCircuit.load(path)
        for k in cb.LoweredCircuit._ARRAYS:
            a, b = getattr(lc, k), getattr(l2, k)
            assert (a is None and b is None) or (a.dtype == b.dtype and np.array_equal(a, b)), k
        assert np.array_equal(lc.lane_soa, l2.lane_soa) and l2.lane_soa.dtype == np.float64
        assert lc.node_names == l2.node_names and lc.dev_user_nodes == l2.dev_user_nodes
        assert cb.expand_breakpoints(lc.breakpoints, (0.0, 1.0)) == cb.expand_breakpoints(l2.breakpoints, (0.0, 1.0))
        with pytest.raises(ValueError):
            cb.LoweredCircuit.from_dict({"format": "something else"})


def test_caller_buffers_are_validated():
    """backend._check_f64 / _lane_block (ADVICE r1): wrong dtype, shape or layout raises before
    anything reaches the C side; a column block of a wider array yields its leading dimension."""
    x = np.zeros((2, 5, 7))
    assert backend._lane_block(x, (2, 5), 7, "x") == 7
    assert backend._lane_block(x[..., 2:5], (2, 5), 3, "x") == 7
    assert backend._lane_block(x[:, :1, 2:5], (2, 1), 3, "x") == 35
    for bad, lead, P in ((x.astype(np.float32), (2, 5), 7), (x[:, ::2, 2:5], (2, 3), 3), (x[..., ::2], (2, 5), 4),
                         (x, (2, 4), 7), (x.T, (7, 5), 2)):
        with pytest.raises(ValueError):
            backend._lane_block(bad, lead, P, "x")
    with pytest.raises(ValueError):
        backend._check_f64(np.zeros((3, 4), dtype=np.float32), (3, 4), "u0")
    with pytest.raises(ValueError):
        backend._check_f64(np.zeros((3, 5)), (3, 4), "u0")
    assert backend.fixed_step_points(0.0, 2e-3, 1e-6, 10) == 201
    assert backend.fixed_step_points(0.0, 1.003e-3, 1e-6, 10) == 102
    assert backend.fixed_step_points(0.0, 4e-7, 1e-10, 1) == 4001


def _shared_buffer_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        P, T = 11, 3
        buf = distributed.SharedSweepBuffer((2, T, P), pin=False)
        sl = distributed.shard_slice(P, rank, world)
        blk = buf.lane_block(sl)
        ld = backend._lane_block(blk, (2, T), sl.stop - sl.start, "block")
        lanes = np.arange(sl.start, sl.stop, dtype=np.float64)
        for s in range(2):
            for t in range(T):
                blk[s, t, :] = lanes + 100.0 * t + 1000.0 * s      # what cb200_tran_fetch_ld writes
        dist.barrier()
        full = buf.array.copy() if rank == 0 else None
        buf.close()
        q.put((rank, ld, None if full is None else full.tolist()))
    finally:
        dist.destroy_process_group()


def test_shared_sweep_buffer_world_size_2_gloo():
    """The end-of-run gather of a sharded sweep: both ranks write their lane blocks into ONE
    shared host array; rank 0 reads the full [save][T][P] result."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_shared_buffer_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = {r: (ld, full) for r, ld, full in (q.get(timeout=120) for _ in range(2))}
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    assert res[0][0] == 11 and res[1][0] == 11
    full = np.array(res[0][1])
    want = np.arange(11.0)[None, None, :] + 100.0 * np.arange(3.0)[None, :, None] + 1000.0 * np.arange(2.0)[:, None, None]
    assert np.array_equal(full, want)


def test_emitter_op_counts():
    """verilog_a.count_ops_static / instrument_ops on a small inline module: known counts."""
    from cadnip_b200 import verilog_a
    assert verilog_a._line_ops("const double t3 = t1 * t2 + 1.5e-3 * V0;") == (3, 0)
    assert verilog_a._line_ops("const double t4 = CB_EXP(t3) / (t1 - 2.0);") == (1, 2)
    assert verilog_a._line_ops("Ieq += -dI0 * V0;") == (2, 0)
    assert verilog_a._line_ops("const double t5 = -t4;") == (0, 0)
    assert verilog_a._line_ops("const double t6 = (t5 >= -80.0 && t5 <= 80.0) ? t4 : 0.0;") == (0, 0)
    m = cb.va("""module res(a, b); inout a, b; electrical a, b; parameter real r = 1e3;
                 analog begin if (r > 0) I(a, b) <+ V(a, b) / r; else I(a, b) <+ V(a, b) * 1e12; end endmodule""")
    src = verilog_a.c_source([m.default])
    st = verilog_a.count_ops_static(src)
    assert len(st) == 1 and list(st.values())[0][0] > 0
    inst = verilog_a.instrument_ops(src)
    assert "ora_va_ops[2] += 1;" in inst and inst.count("VA_OPS(") >= 2


def test_state_abstol_layout_and_oracle_class_tolerances():
    """state_abstol (src/mna/build.jl:276-283): vntol on nodes AND limit unknowns, iabstol on branch
    currents, chgtol on charge states; the oracle's adaptive controller honours it (flags bit 2)."""
    import cadnip_oracle as ora
    import circuits
    lc = cb.lower_circuit(cb.MNACircuit(circuits.rectifier(True)))
    tol = cb.state_abstol(lc, vntol=1e-6, iabstol=1e-12, chgtol=1e-14)
    assert (lc.n_nodes, lc.n_currents, lc.n_charges, lc.n_limits) == (2, 1, 0, 1)
    assert tol.tolist() == [1e-6, 1e-6, 1e-12, 1e-6]
    lc = cb.lower_circuit(cb.MNACircuit(circuits.mos_amp, vg=1.0, rd=2e3))
    nl = ora.OracleNetlist(lc.netlist_tables())
    counts = {}
    for name, kw in (("scalar", dict(lte_abstol=1e-6)), ("class", dict(class_abstol=(1e-6, 1e-12, 1e-14)))):
        o = ora.make_tran_opts(method=1, adaptive=1, dt=1e-11, reltol=1e-5, max_points=20000, **kw)
        r = ora.tran(nl, ora.make_spec(mode="tran"), 0.0, 3e-8, o, [lc.index_of("d")])
        assert r["status"] == 0
        counts[name] = r["T"]
    assert counts["class"] > counts["scalar"]
    with pytest.raises(ValueError):
        cb.tran(cb.MNACircuit(circuits.mos_amp, vg=1.0, rd=2e3), (0.0, 1e-9), abstol=dict(vtol=1e-6))


def _resistor_mesh(nx, ny, n_src=6, seed=5):
    """nx x ny resistor mesh with a few voltage sources, current-controlled sources and capacitors:
    the large-circuit symbolic path (analyze_lu_sparse: n > 1536)."""
    from cadnip_b200 import MNAContext, ZERO_VECTOR, get_node, stamp, Resistor, Capacitor, VoltageSource, VCCS, CCCS
    rng = np.random.default_rng(seed)

    def build(params, spec, t=0.0, x=ZERO_VECTOR, ctx=None):
        ctx = MNAContext() if ctx is None else ctx
        node = [[get_node(ctx, f"n{i}_{j}") for j in range(ny)] for i in range(nx)]
        srcs = []
        for k in range(n_src):
            i, j = int(rng.integers(nx)), int(rng.integers(ny))
            srcs.append(stamp(VoltageSource(1.0 + k, name=f"V{k}"), ctx, node[i][j], 0))
        for i in range(nx):
            for j in range(ny):
                if i + 1 < nx:
                    stamp(Resistor(float(rng.uniform(100, 1e4))), ctx, node[i][j], node[i + 1][j])
                if j + 1 < ny:
                    stamp(Resistor(float(rng.uniform(100, 1e4))), ctx, node[i][j], node[i][j + 1])
                if (i * ny + j) % 7 == 0:
                    stamp(Capacitor(1e-12), ctx, node[i][j], 0)
                if (i * ny + j) % 97 == 5:
                    a, b = int(rng.integers(nx)), int(rng.integers(ny))
                    stamp(VCCS(1e-4, name=f"G{i}_{j}"), ctx, node[i][j], 0, node[a][b], 0)
        stamp(CCCS(0.5, name="F1"), ctx, node[nx // 2][ny // 2], 0, srcs[0])
        stamp(Resistor(1e3), ctx, node[0][0], 0)
        return ctx
    return build


def test_sparse_symbolic_analysis_large_circuit():
    """analyze_lu_sparse (csrc/symbolic.cpp): matching for the zero-diagonal source rows, Markowitz
    ordering + symbolic fill on sparse rows, level schedule -- on a 3 600-node mesh (n > 1536 takes the
    sparse path); the serial and the level schedule agree bitwise and solve A x = b as scipy does."""
    import time
    import scipy.sparse as sp
    import scipy.sparse.linalg as spla
    from cadnip_b200 import backend
    rng = np.random.default_rng(11)
    lc = cb.lower_circuit(cb.MNACircuit(_resistor_mesh(60, 60)))
    assert lc.n > 3600
    colptr, rowval = backend.host_lu_check(lc)
    n, nnz = len(colptr) - 1, len(rowval)
    # values with the structure of an MNA Jacobian: negative node-to-node couplings, diagonals that
    # dominate their row (conductances add up), unit incidence entries on the source rows / columns
    cols = np.repeat(np.arange(n), np.diff(colptr))
    rws = rowval - 1
    node_blk = (rws < lc.n_nodes) & (cols < lc.n_nodes)
    J = np.where(node_blk, -rng.uniform(0.5, 2.0, nnz), 1.0)
    diag = rws == cols
    J[diag] = 0.0
    rowsum = np.zeros(n)
    np.add.at(rowsum, rws[node_blk], np.abs(J[node_blk]))
    J[diag] = rowsum[rws[diag]] + 0.25
    A = sp.csc_matrix((J, rowval - 1, colptr - 1), shape=(n, n))
    rhs = rng.uniform(-1.0, 1.0, n)
    t0 = time.perf_counter()
    xs, xl, info = backend.host_lu_check(lc, J, rhs)
    dt = time.perf_counter() - t0
    ref = spla.spsolve(A, rhs)
    assert np.array_equal(xs, xl)
    assert np.allclose(xs, ref, rtol=1e-9, atol=1e-11 * np.abs(ref).max())
    # a planar mesh under a fill-reducing order: the factor stays within a small multiple of the pattern
    assert info["nlu"] < 12 * info["nnz"] and info["factor_levels"] < info["n"] // 4
    print(f"n {n} nnz {nnz} nlu {info['nlu']} levels {info['factor_levels']} analysis+solve {dt:.2f} s")


def test_julia_shim_matches_header():
    """julia/CadnipB200.jl (the ccall binding a Cadnip.jl maintainer adds; cannot run here -- no Julia
    in the image) mirrors the C structs field by field: names, order and sizes must equal the ctypes
    structures the tests drive the library with, and every symbol it calls must be exported."""
    import ctypes as C
    import re
    from cadnip_b200 import backend
    src = open(os.path.join(ROOT, "julia", "CadnipB200.jl")).read()
    size = {"Int32": 4, "Int64": 8, "Cdouble": 8}
    for jname, ct in (("Spec", backend.Spec), ("DcOpts", backend.DcOpts), ("TranOpts", backend.TranOpts),
                      ("Desc", backend.Desc)):
        body = re.search(rf"^struct {jname}\b[^\n]*\n(.*?)^end", src, re.S | re.M).group(1)
        fields = re.findall(r"(\w+)::((?:Ptr\{\w+\})|\w+)", body)
        want = [(n, C.sizeof(t)) for n, t in ct._fields_]
        got = [(n, 8 if t.startswith("Ptr") else size[t]) for n, t in fields]
        assert [g[1] for g in got] == [w[1] for w in want], (jname, got, want)
        assert [g[0].lower() for g in got] == [w[0].lower() for w in want], (jname, got, want)
        assert sum(g[1] for g in got) == C.sizeof(ct), jname          # no implicit padding on either side
    for sym in set(re.findall(r"\(:(cb200_\w+), LIB\[\]\)", src)):
        assert sym in backend.EXPORTED_SYMBOLS, sym


def test_terminal_currents_operating_point_info():
    """``terminal_currents`` (src/mna/context.jl:1251-1270): device terminal currents at the DC point,
    names ``i_<device>_<terminal>``; KCL closes at every node."""
    import cadnip_oracle as ora
    from cadnip_b200.analysis import terminal_currents
    lc = cb.lower_circuit(cb.MNACircuit(circuits.rectifier(True)))
    x, ok, it = ora.solve_dc(ora.OracleNetlist(lc.netlist_tables()), ora.make_spec(mode="dcop"))
    assert ok
    tc = terminal_currents(lc, x)
    vout = x[lc.index_of("out") - 1]
    assert tc["i_R_p"] == pytest.approx((5.0 - vout) / 1000.0, rel=1e-12) and tc["i_R_n"] == -tc["i_R_p"]
    assert tc["i_D1_p"] == pytest.approx(tc["i_R_p"], rel=1e-6)            # series loop: same current
    assert tc["i_D1_p"] == pytest.approx(1e-14 * (math.exp(vout / 0.026) - 1.0), rel=1e-9)
    assert -x[lc.index_of("I_V1") - 1] == pytest.approx(tc["i_R_p"], rel=1e-9)
    lc = cb.lower_circuit(cb.MNACircuit(circuits.mos_amp, vg=1.5, rd=2e3))
    x, ok, it = ora.solve_dc(ora.OracleNetlist(lc.netlist_tables()), ora.make_spec(mode="dcop"))
    tc = terminal_currents(lc, x)
    vd = x[lc.index_of("d") - 1]
    assert tc["i_M1_d"] == pytest.approx((3.3 - vd) / 2e3 + tc["i_DC1_p"], rel=1e-6)   # KCL at the drain node
    assert tc["i_M1_g"] == 0.0 and tc["i_M1_s"] == -tc["i_M1_d"]
