"""The reference's VADistiller models (sp_mos1, sp_diode: $limit / PCNR, node collapse,
$param_given, analog functions, charge detection) through the emitter.  Circuits come from
the committed fixtures (tests/golden/va_*.json.gz, made by tests/golden/make_va_fixtures.py from
the reference's .va files); known answers are the reference's own (test/params.jl,
test/sweep.jl, test/mna/oscillator_test.jl)."""
import math
import os
import subprocess

import numpy as np
import pytest

import cadnip_b200 as cb
import cadnip_oracle as ora

HERE = os.path.dirname(os.path.abspath(__file__))
HAVE_REF = os.path.isdir("/root/reference/models/VADistillerModels.jl/va")
needs_ref = pytest.mark.skipif(not HAVE_REF, reason="reference tree not mounted")

FIXTURE_NAMES = ["mos1_corner", "diode_chain", "diode_rs_cap", "mos1_inverter", "mos1_c3", "mos1_dff", "mos1_ring",
                 "mos1_ring_caps", "bjt_ce", "jfet2_cs", "vdmos_cs", "inductor_rl", "mos1_c6288_slice", "psp_ring"]


GPU_FIXTURES = ["mos1_corner", "diode_chain", "mos1_inverter", "diode_rs_cap", "mos1_ring", "mos1_c3", "mos1_dff"]   # used by -m gpu tests


def fixture(name):
    return cb.LoweredCircuit.load(os.path.join(HERE, "golden", f"va_{name}.json.gz"))


def oracle_of(lc):
    ora.load_va_models(lc.va_c_source)
    return ora.OracleNetlist(lc.netlist_tables())


# ---- emitter over the reference's model files ---------------------------------------
@needs_ref
@pytest.mark.parametrize("name", ["resistor", "capacitor", "inductor", "diode", "bjt", "mos1", "mos2", "mos3", "mos6",
                                  "mos9", "jfet1", "jfet2", "mes1", "vdmos"])
def test_vadistiller_model_emits_compilable_c(name, tmp_path):
    from cadnip_b200 import verilog_a
    import va_circuits
    m = verilog_a.load_va(va_circuits.VA_DIR + name + ".va")
    v = m.default
    assert v.nodes[:len(m.ports)] == m.ports
    src = verilog_a.c_source([v])
    c = tmp_path / "m.c"
    c.write_text(src)
    subprocess.run(["gcc", "-O0", "-fsyntax-only", "-Wall", "-Werror=implicit-function-declaration", str(c)],
                   check=True)
    assert f"va_stamp_{v.cname}" in verilog_a.cuda_header([v])


def test_new_vadistiller_models_known_answers():
    """sp_inductor / sp_bjt / sp_jfet2 / sp_vdmos -- the models that need potential contributions with
    branch currents (internal-to-internal and to-ground shorts, named branches: bjt.va:739-753,
    :1009-1013; jfet2.va:653-663; vdmos.va:105, :855-868, :1431; inductor.va:61, :272) -- in the
    reference's own test circuits (test/mna/vadistiller_integration.jl:240-259, :390-416, :498-519,
    :694-711) with the reference's expected ranges."""
    want = {"inductor_rl": ("mid", -0.01, 0.01), "bjt_ce": ("collector", 0.0, 5.0),
            "jfet2_cs": ("drain", 0.0, 10.0), "vdmos_cs": ("drain", 0.0, 10.0)}
    for name, (node, lo, hi) in want.items():
        lc = fixture(name)
        xo, sto, ito = ora.sweep_dc(oracle_of(lc), ora.make_spec(mode="dcop"), lc.n)
        v = xo[:, lc.index_of(node) - 1]
        assert (sto == 0).all() and np.all(np.isfinite(xo)), name
        assert np.all((v > lo) & (v < hi)) or name == "vdmos_cs", (name, v)
    lc = fixture("bjt_ce")
    # 8 nodes (4 user + c_int, sub_con, xf1, xf2: the other three internals alias their port), 2 source
    # currents + 4 branch currents of the executed shorts, 3 $limit unknowns (bjt.va:1040-1042)
    assert (lc.n_nodes, lc.n_currents, lc.n_charges, lc.n_limits) == (8, 6, 0, 3)
    xo, _, _ = ora.sweep_dc(oracle_of(lc), ora.make_spec(mode="dcop"), lc.n)
    vc = xo[:, lc.index_of("collector") - 1].reshape(2, 3)          # [bf][vb]
    assert np.all(np.diff(vc, axis=1) < 0) and np.all(vc[1] < vc[0])   # more base drive / more gain: lower collector
    assert np.allclose(xo[:, lc.index_of("Q1_sp_bjt_c_int") - 1], xo[:, lc.index_of("collector") - 1], atol=1e-12)
    lc = fixture("vdmos_cs")
    vd = ora.sweep_dc(oracle_of(lc), ora.make_spec(mode="dcop"), lc.n)[0][:, lc.index_of("drain") - 1]
    assert vd[0] == pytest.approx(10.0, abs=1e-6) and 0.0 < vd[2] < 1.0 and np.all(np.diff(vd) < 0)   # off below vto = 2 V


@needs_ref
def test_sp_bsim4v8_and_bsim3v3_known_answers():
    """The two large VADistiller MOSFETs through the emitter and the oracle: string parameter
    (`version`), named noise branches with current probes, 9 $limit branches, internal-to-internal
    shorts (bsim4v8.va:98-100, :163, :4539-4574, :5992-6000, :9836-9845).  Known answer of the reference:
    0.9 < V(drain) < 1.0 for l = 100 nm, w = 1 um, 1 k load on 1 V, gate at 0.5 V
    (test/mna/vadistiller_integration.jl:758-775); sp_bsim3v3: 0 < V(drain) < 1.8 (:718-741)."""
    from cadnip_b200 import verilog_a
    import va_circuits
    from cadnip_b200 import MNAContext, ZERO_VECTOR, get_node, stamp, VoltageSource, Resistor
    for fname, vdd_v, vg_v, lo, hi in (("bsim4v8", 1.0, 0.5, 0.9, 1.0), ("bsim3v3", 1.8, 1.0, 0.0, 1.8)):
        m = verilog_a.load_va(va_circuits.VA_DIR + fname + ".va")

        def build(params, spec, t=0.0, x=ZERO_VECTOR, ctx=None):
            ctx = MNAContext() if ctx is None else ctx
            vdd = get_node(ctx, "vdd"); d = get_node(ctx, "drain"); g = get_node(ctx, "gate")
            stamp(VoltageSource(vdd_v, name="Vdd"), ctx, vdd, 0)
            stamp(VoltageSource(vg_v, name="Vg"), ctx, g, 0)
            stamp(Resistor(1000.0, name="Rd"), ctx, vdd, d)
            stamp(m(l=100e-9, w=1e-6, name="M1"), ctx, d, g, 0, 0)
            return ctx
        lc = cb.lower_circuit(cb.MNACircuit(build))
        nl = oracle_of(lc)
        coo = ora.Structure(nl, ora.make_spec(mode="dcop")).coo()
        assert np.array_equal(coo["G_I"], lc.G_I) and np.array_equal(coo["G_J"], lc.G_J)      # host == oracle builder
        assert np.array_equal(coo["C_I"], lc.C_I) and np.array_equal(coo["b_I"], lc.b_I)
        x, ok, it = ora.solve_dc(nl, ora.make_spec(mode="dcop"))
        assert ok and lo < x[lc.index_of("drain") - 1] < hi, (fname, x[lc.index_of("drain") - 1])
        if fname == "bsim4v8":
            assert lc.n_limits == 9 and m.mod["sparams"] == {"version": "4.8.3"}
            assert x[lc.index_of("drain") - 1] == pytest.approx(0.9066, abs=2e-4)


@needs_ref
def test_psp103_preprocessor_and_known_answer():
    """PSP103 (models/PSPModels.jl/va/psp103.va) is written in the Verilog-A macro language: `include of
    seven files, 150 function-like `define macros, multi-line bodies.  Through the preprocessor and the
    emitter it must reproduce the reference's own test (test/mna/psp103_integration.jl:40-63: NMOS W =
    10u, L = 1u, default card, Vds 1.2 V, Vgs 0.6 V -> 100 uA < |Id| < 1 mA) and its published structure:
    8 internal nodes per FET (:163) and -- c6288, doc/c6288_bottleneck_findings.md:75-84 -- 7 branch
    currents and 5 charge states per FET (70 818 / 10 112, 50 560 / 10 112)."""
    from cadnip_b200 import verilog_a
    from cadnip_b200 import MNAContext, ZERO_VECTOR, get_node, stamp, VoltageSource
    from cadnip_b200.workloads import PSP_DIR
    m = verilog_a.load_va(PSP_DIR + "psp103.va")
    assert m.name == "PSP103VA" and m.ports == ["D", "G", "S", "B"]
    assert m.internal == ["NOI", "GP", "SI", "DI", "BP", "BI", "BS", "BD"]
    assert len(m.param_names) > 700

    def build(params, spec, t=0.0, x=ZERO_VECTOR, ctx=None):
        ctx = MNAContext() if ctx is None else ctx
        d = get_node(ctx, "d"); g = get_node(ctx, "g")
        stamp(m(TYPE=1, W=10e-6, L=1e-6, name="M1"), ctx, d, g, 0, 0)
        stamp(VoltageSource(1.2, name="vds"), ctx, d, 0)
        stamp(VoltageSource(0.6, name="vgs"), ctx, g, 0)
        return ctx
    lc = cb.lower_circuit(cb.MNACircuit(build))
    assert (lc.n_nodes, lc.n_currents, lc.n_charges, lc.n_limits) == (2 + 8, 2 + 7, 5, 0)
    nl = oracle_of(lc)
    coo = ora.Structure(nl, ora.make_spec(mode="dcop")).coo()
    assert np.array_equal(coo["G_I"], lc.G_I) and np.array_equal(coo["G_J"], lc.G_J)
    assert np.array_equal(coo["C_I"], lc.C_I) and np.array_equal(coo["b_I"], lc.b_I)
    x, ok, it = ora.solve_dc(nl, ora.make_spec(mode="dcop"))
    assert ok
    assert x[lc.index_of("d") - 1] == pytest.approx(1.2, abs=1e-6) and x[lc.index_of("g") - 1] == pytest.approx(0.6, abs=1e-6)
    assert 100e-6 < abs(x[lc.index_of("I_vds") - 1]) < 1e-3


def test_psp103_ring_oscillator_known_behaviour():
    """The 9-stage PSP103 ring of benchmarks/vacask/ring/cedarsim (the fixture: two supply voltages):
    the metastable DC point sits near Vdd / 2 and the 10 uA kick starts a rail-to-rail oscillation."""
    lc = fixture("psp_ring")
    assert lc.n == 370 and lc.n_limits == 0                 # the reference reports 371 unknowns for this deck
    nl = oracle_of(lc)
    xo, sto, ito = ora.sweep_dc(nl, ora.make_spec(mode="tranop"), lc.n)
    assert (sto == 0).all()
    v3 = xo[:, lc.index_of("3") - 1] / np.array([1.1, 1.2])
    assert np.all((v3 > 0.5) & (v3 < 0.6))                   # the p-channel is the stronger device
    ora.set_linear_solver(1)
    try:
        o = ora.make_tran_opts(method=1, dt=5e-11)
        ro = ora.sweep_tran(nl, ora.make_spec(mode="tran"), 0.0, 2e-8, o, [lc.index_of("5")])
    finally:
        ora.set_linear_solver(0)
    assert (ro["status"] == 0).all()
    u = ro["u"][1, :, 0]
    assert u.min() < 0.1 and u.max() > 1.1
    assert 3 <= int(np.sum((u[1:] > 0.6) & (u[:-1] <= 0.6))) <= 8
    # the reference's benchmark settings (benchmarks/vacask/ring/cedarsim/runme.jl:47-67: reltol 1e-2, abstol 1e-4,
    # dtmax 0.05 ns) on the variable-order BDF controller, the reference's own solver family (IDA): the adaptive
    # run completes and oscillates.  (The trapezoidal controller does not get through this circuit: the rule's
    # undamped ringing on the charge-state constraints keeps the error estimate from shrinking with h.)
    ora.set_linear_solver(1)
    try:
        o = ora.make_tran_opts(method=3, adaptive=1, dt=1e-12, reltol=1e-2, lte_abstol=1e-4, dtmax=0.05e-9, max_points=20000)
        rb = ora.sweep_tran(nl, ora.make_spec(mode="tran"), 0.0, 3e-8, o, [lc.index_of("5")])
    finally:
        ora.set_linear_solver(0)
    assert (rb["status"] == 0).all()
    T = int(rb["T"][1])
    ub = rb["u"][1, :T, 0]
    assert rb["t"][1, T - 1] == 3e-8 and ub.min() < 0.1 and ub.max() > 1.1


@needs_ref
def test_sp_mos1_structure():
    from cadnip_b200 import verilog_a
    import va_circuits
    m = verilog_a.load_va(va_circuits.VA_DIR + "mos1.va")
    v = m.default
    assert v.nodes == ["d", "g", "s", "b", "d_int", "s_int"]
    # one limit unknown per unique $limit probe branch, 8 call sites (mos1.va:919-922, :976-979)
    assert v.lim_branches == [("g", "s_int"), ("d_int", "s_int"), ("b", "s_int"), ("b", "d_int")]
    assert len(v.sites) == 8
    # node-to-ground contributions first, then the three noise branches (mos1.va:1164-1221)
    assert v.branches[:6] == [(n, None) for n in ("d", "g", "s", "b", "d_int", "s_int")]
    assert v.branches[6:] == [("d_int", "d"), ("s_int", "s"), ("d_int", "s_int")]
    assert v.reactive == [False, True, False, True, True, True, False, False, False]
    assert set(m.collapses) == {"d_int", "s_int"}           # V(d_int,d) <+ 0 / V(s_int,s) <+ 0
    inst = m(type=1, vto=0.7, kp=1e-4, w=1e-6, l=1e-6)
    assert inst.collapsed(cb.MNASpec()) == {"d_int": "d", "s_int": "s"}
    assert m(type=1, rd=10.0).collapsed(cb.MNASpec()) == {"s_int": "s"}
    assert m(VTO=0.7).given == frozenset({"vto"}) and m(vt0=0.7).given == frozenset({"vto"})   # aliasparam
    # set-up / evaluation split: parameter and temperature preprocessing (mos1.va:560-900) runs once
    # per kernel and hands its results to the per-iteration code through private state slots
    var = m.variant(inst.given, None)
    setup, evaln, n_state = var._sections(split=True)     # optional (verilog_a.SPLIT_SETUP), off by default
    assert 40 < n_state < 200
    assert sum(ln.count("VA_ST(") for ln in setup) == n_state == sum(ln.count("VA_LD(") for ln in evaln)
    assert not any("V0" in ln or "vold" in ln or "limw" in ln for ln in setup)      # nothing bias-dependent
    assert sum(ln.count("log(") for ln in setup) >= 5 and sum(ln.count("CB_EXP(") for ln in setup) >= 3


@needs_ref
@pytest.mark.parametrize("name", FIXTURE_NAMES)
def test_fixtures_are_current(name):
    import va_circuits
    lc = va_circuits.lower_fixture(name)
    fx = fixture(name)
    assert lc.va_cuda_header == fx.va_cuda_header and lc.va_c_source == fx.va_c_source
    assert np.array_equal(lc.G_I, fx.G_I) and np.array_equal(lc.dev_nodes, fx.dev_nodes)
    assert np.array_equal(lc.lane_soa, fx.lane_soa) and np.array_equal(lc.uniform, fx.uniform)


# ---- host structure == oracle structure -----------------------------------------------
@pytest.mark.parametrize("name", FIXTURE_NAMES)
def test_host_coo_matches_oracle_builder(name):
    """The oracle runs the emitted C as the builder (it allocates its own internal nodes,
    limit and charge unknowns, evaluates the collapse conditions and detects
    voltage-dependent charges over 5 passes); the host derives the same from the stamp plan."""
    lc = fixture(name)
    nl = oracle_of(lc)
    S = ora.Structure(nl, ora.make_spec(mode="tran"))
    assert (S.n, S.n_nodes, S.n_charges, S.n_limits) == (lc.n, lc.n_nodes, lc.n_charges, lc.n_limits)
    coo = S.coo()
    for k in ("G_I", "G_J", "C_I", "C_J", "b_I"):
        assert np.array_equal(coo[k], getattr(lc, k)), k


def test_sp_mos1_unknown_count():
    lc = fixture("mos1_inverter")
    assert lc.dev_state_ptr[0] == 0 and np.all(np.diff(lc.dev_state_ptr) >= 0)
    # 4 nodes + 3 source currents + 2 x 4 limit unknowns; zero device caps -> no charge states
    assert (lc.n_nodes, lc.n_currents, lc.n_charges, lc.n_limits) == (4, 3, 0, 8)
    assert lc.limit_names[:4] == ["MP_sp_mos1_lim_g_s_int", "MP_sp_mos1_lim_d_int_s_int",
                                  "MP_sp_mos1_lim_b_s_int", "MP_sp_mos1_lim_b_d_int"]
    assert fixture("mos1_ring_caps").n_charges > 0


# ---- known answers ------------------------------------------------------------------------
def test_mos1_square_law_known_answer():
    """test/params.jl:686-712: V(drain) = 5 - 10e3 * 1/2 kp 20 (1.2 - vto)^2, atol 1e-6."""
    lc = fixture("mos1_corner")
    nl = oracle_of(lc)
    x, st, it = ora.sweep_dc(nl, ora.make_spec(mode="dcop"), lc.n)
    assert (st == 0).all() and it.max() <= 10
    vd = x[:, lc.index_of("drain") - 1].reshape(2, 3)
    for j, kp in enumerate((100e-6, 50e-6)):
        for i, vto in enumerate((0.6, 0.7, 0.9)):
            assert vd[j, i] == pytest.approx(5 - 10e3 * 0.5 * kp * 20 * (1.2 - vto) ** 2, abs=1e-6)


def test_sp_diode_chain_sweep_known_answer():
    """test/sweep.jl:334-353: 40 points converge, n1 monotone in the supply, clamped near 3 x 0.7 V."""
    lc = fixture("diode_chain")
    nl = oracle_of(lc)
    x, st, it = ora.sweep_dc(nl, ora.make_spec(mode="dcop"), lc.n)
    assert (st == 0).all()
    n1 = x[:, lc.index_of("n1") - 1]
    assert np.all(np.diff(n1) > 0) and 1.5 < n1[-1] < 2.5
    # Shockley law at the solved point: I = Is (exp(V/(n kT/q)) - 1) + gmin V per junction
    i = -x[:, lc.index_of("I_v1") - 1]
    vt = 1.38064852e-23 / 1.6021766208e-19 * 300.15
    v3 = x[:, lc.index_of("n3") - 1]
    assert np.allclose(i, 1e-14 * np.expm1(v3 / vt) + 1e-12 * v3, rtol=1e-6, atol=1e-15)
    # limit unknowns settle on their probe voltages (PCNR fixed point)
    assert np.allclose(x[:, lc.index_of("d3_sp_diode_lim_a_int_c") - 1], v3, atol=1e-9)


def _ring_u0(lc):
    u0 = np.zeros(lc.n)
    u0[lc.index_of("vdd") - 1] = 3.3
    u0[lc.index_of("out1") - 1] = 3.3                     # asymmetric start (UIC)
    return u0


@pytest.mark.parametrize("name", ["mos1_ring", "mos1_ring_caps"])
def test_ring_oscillator_known_answer(name):
    """test/mna/oscillator_test.jl:73-160: swing > 2 V on 3.3 V, rails reached, period 0.5-50 ns."""
    lc = fixture(name)
    nl = oracle_of(lc)
    save = [lc.index_of(n) for n in ("out1", "out2", "in1")]
    o = ora.make_tran_opts(method=1, dt=5e-12, init=1)
    r = ora.tran(nl, ora.make_spec(mode="tran"), 0.0, 20e-9, o, save, u0=_ring_u0(lc))
    assert r["status"] == 0
    t, u = r["t"], r["u"]
    late = t > 10e-9
    for k in range(3):
        v = u[late, k]
        assert v.max() - v.min() > 2.0 and v.max() > 2.5 and v.min() < 0.8
    v = u[late, 0]
    mid = 0.5 * (v.max() + v.min())
    crossings = np.count_nonzero(np.diff((v > mid).astype(int)))
    period = 2 * (t[late][-1] - t[late][0]) / crossings
    assert 0.05e-9 < period < 50e-9


def test_transient_limiting_rescues_fast_edges():
    """C3 corner lanes (SURVEY 8d): with a 1 fF load the output flips inside one 0.1 ns step and
    the first Newton iterate forward-biases a bulk junction; the plain iteration (limit rows as
    ordinary unknowns, the reference's transient formulation) crawls down the exponential and
    misses 10 solves, CB200_TRAN_LIMIT redoes those steps with the models' $limit damping."""
    lc = fixture("mos1_c3")
    nl = oracle_of(lc)
    save = [lc.index_of("q")]
    plain = ora.sweep_tran(nl, ora.make_spec(mode="tran"), 0.0, 1.3e-7,
                           ora.make_tran_opts(method=0, dt=1e-10, save_every=10), save)
    lim = ora.sweep_tran(nl, ora.make_spec(mode="tran"), 0.0, 1.3e-7,
                         ora.make_tran_opts(method=0, dt=1e-10, save_every=10, limit=True), save)
    assert (plain["status"] == 1).any() and (lim["status"] == 0).all()
    ok = plain["status"] == 0
    assert np.allclose(plain["u"][ok], lim["u"][ok], rtol=0, atol=1e-6)      # same converged steps
    vdd = lc.param_value(int(lc.dev_params[lc.dev_param_ptr[lc.dev_names.index("VVDD")]]))
    assert np.all(lim["u"][:, -1, 0] < 0.05 * vdd)                              # input high -> output low


def test_dff_known_behaviour():
    """SURVEY 8d C4 (gf180 D flip-flop, 30 FETs; sp_mos1 fallback card): n = 18 nodes + 7 source
    currents + 30 x 4 limit unknowns; the DC operating point latches Q high with D low and CLKN high,
    and the first falling clock edge (t = 51 ns) transfers D = 0 to Q."""
    lc = fixture("mos1_dff")
    assert (lc.n_nodes, lc.n_currents, lc.n_charges, lc.n_limits) == (18, 7, 0, 120)
    nl = oracle_of(lc)
    x, st, it = ora.sweep_dc(nl, ora.make_spec(mode="tranop"), lc.n)
    assert (st == 0).all()
    for name, level in (("Q_neg", 0.0), ("cki", 5.0), ("ncki", 0.0)):
        assert np.allclose(x[:, lc.index_of(name) - 1], level, atol=1e-3)
    o = ora.make_tran_opts(method=1, adaptive=1, dt=1e-12, reltol=1e-3, lte_abstol=1e-5, max_points=4000, limit=True)
    r = ora.tran(nl, ora.make_spec(mode="tran"), 0.0, 1.2e-7, o, [lc.index_of("Q"), lc.index_of("CLKN")])
    assert r["status"] == 0 and 100 < len(r["t"]) < 4000
    q = np.interp([40e-9, 110e-9], r["t"], r["u"][:, 0])
    assert q[0] > 4.9 and q[1] < 0.1


# ---- emitted derivatives against finite differences ------------------------------------------
@pytest.mark.parametrize("name", ["mos1_inverter", "diode_rs_cap", "mos1_ring_caps"])
def test_emitted_jacobian_matches_finite_differences(name):
    """F(u) = G(u) u - b(u) is the sum of branch currents; with the limit unknowns on their
    probe voltages (no limiting active) dF/du must equal the stamped G."""
    lc = fixture(name)
    nl = oracle_of(lc)
    S = ora.Structure(nl, ora.make_spec(mode="tran"))
    rng = np.random.default_rng(7)
    n = S.n
    for trial in range(3):
        u = np.zeros(n)
        u[:lc.n_nodes] = rng.uniform(0.2, 2.5, lc.n_nodes)

        def settle(u):
            # put every limit unknown on its probe voltage: x_lim = V_p - V_n
            for k, (p, q) in enumerate(lc_limit_branches(lc)):
                u[n - lc.n_limits + k] = (u[p - 1] if p else 0.0) - (u[q - 1] if q else 0.0)
            return u

        def F(u):
            G, C, b, _ = S.rebuild(settle(u.copy()))
            return S.dense(G) @ settle(u.copy()) - b
        u = settle(u)
        G, C, b, _ = S.rebuild(u)
        Gd = S.dense(G)
        for j in range(lc.n_nodes):
            h = 1e-6
            up, um = u.copy(), u.copy()
            up[j] += h; um[j] -= h
            dF = (F(up) - F(um)) / (2 * h)
            # total derivative along "limit unknowns follow their probes": G[:, j] + G[:, lim] dlim/du_j
            col = Gd[:, j].copy()
            for k, (p, q) in enumerate(lc_limit_branches(lc)):
                s = (1.0 if p == j + 1 else 0.0) - (1.0 if q == j + 1 else 0.0)
                col += Gd[:, n - lc.n_limits + k] * s
            rows = [i for i in range(lc.n_nodes)]
            # central differences on currents of size |G|max * |u|: absolute floor ~1e-8 of that
            scale = np.abs(Gd[:lc.n_nodes, :lc.n_nodes]).max() + 1e-12
            assert np.allclose(dF[rows], col[rows], rtol=1e-5, atol=1e-8 * scale), (name, trial, j)


class _VoldIsVnew(dict):
    """vold of every $limit probe = its present voltage: the models' limiters return vnew unchanged."""
    def __init__(self, V):
        super().__init__()
        self.V = V

    def __bool__(self):
        return True

    def get(self, key, default=0.0):
        a, b = key
        return self.V[a] - (self.V[b] if b is not None else 0.0)


INTERP_CASES = [("resistor", dict(resistance=2e3), [1.0, 0.2]),
                ("capacitor", dict(capacitance=1e-12), [1.0, 0.2]),
                ("inductor", dict(inductance=1e-3), [1.0, 0.2]),
                ("diode", {}, [0.65, 0.05]),
                ("bjt", dict(bf=100.0, **{"is": 1e-15}), [2.0, 0.68, 0.02, 0.0]),
                ("mos1", dict(w=1e-6, l=1e-6, vto=0.7, kp=100e-6), [1.5, 1.2, 0.1, 0.0]),
                ("mos2", dict(w=1e-6, l=1e-6, vto=0.7, kp=100e-6), [1.5, 1.2, 0.1, 0.0]),
                # nsub given: with the default card MOS3alpha = 0 and the model's sqrt(kappa * alpha * ...) has a
                # 0 * inf derivative under ANY forward-mode AD (the reference's ForwardDiff duals included;
                # ngspice's hand-written partials avoid it) -- see DESIGN.md s. 4b
                ("mos3", dict(w=1e-6, l=1e-6, vto=0.7, kp=100e-6, nsub=1e15), [1.5, 1.2, 0.1, 0.0]),
                ("mos6", dict(w=1e-6, l=1e-6), [1.5, 1.2, 0.1, 0.0]),
                ("mos9", dict(w=1e-6, l=1e-6, vto=0.7, kp=100e-6, nsub=1e15), [1.5, 1.2, 0.1, 0.0]),
                ("jfet1", {}, [3.0, -0.4, 0.1]),
                ("jfet2", {}, [3.0, -0.4, 0.1]),
                ("mes1", {}, [2.0, -0.3, 0.1]),
                ("vdmos", dict(vto=2.0, kp=0.5), [4.0, 3.0, 0.1, 0.0, 0.0]),
                ("bsim3v3", dict(l=1e-6, w=1e-6), [1.5, 1.2, 0.1, 0.0]),
                ("bsim4v8", dict(l=100e-9, w=1e-6), [0.8, 0.7, 0.05, 0.0])]


@needs_ref
@pytest.mark.parametrize("name,kw,bias", INTERP_CASES, ids=[c[0] for c in INTERP_CASES])
def test_emitted_model_matches_interpreter(name, kw, bias):
    """An emitter-INDEPENDENT check of every VADistiller model: the emitted C (parser -> emit-time
    differentiation -> code generator, run through the oracle's rebuild) against `_Interp`, the host's
    tree-walking interpreter of the same parsed module, which shares neither the code generator nor the
    differentiation.  One instance with every port on a voltage source, internal nodes at random voltages,
    limit unknowns on their probe voltages: the KCL rows of G u - b must equal the interpreter's branch
    currents, and the stamped G must equal central differences OF THE INTERPRETER."""
    from cadnip_b200 import verilog_a
    import va_circuits
    _check_against_interpreter(verilog_a.load_va(va_circuits.VA_DIR + name + ".va"), kw, bias)


INLINE_INTERP_CASES = [("VADDiode", [0.65, 0.05]), ("VADDiodeRs", [0.65, 0.05]), ("ChainDiodeRs", [0.7, 0.0]),
                       ("SimpleMOS", [1.5, 1.2, 0.1]), ("CapMOS", [1.5, 1.2, 0.1]), ("PMOS", [0.1, 0.2, 1.5]),
                       ("JunctionCap", [-0.5, 0.0])]


@pytest.mark.parametrize("name,bias", INLINE_INTERP_CASES, ids=[c[0] for c in INLINE_INTERP_CASES])
def test_inline_model_matches_interpreter(name, bias):
    """The same emitter-independent check on the Verilog-A modules written out in tests/test_va.py, so that it
    runs wherever the repository does."""
    import test_va
    _check_against_interpreter(getattr(test_va, name), {}, bias)


def _check_against_interpreter(m, kw, bias):
    from cadnip_b200 import MNAContext, ZERO_VECTOR, stamp, VoltageSource
    held = {}

    def builder(params, spec, t=0.0, x=ZERO_VECTOR, ctx=None):
        ctx = MNAContext() if ctx is None else ctx
        for k, v in enumerate(bias):
            stamp(VoltageSource(v, name=f"V{k}"), ctx, f"p{k}", 0)
        held["inst"] = m(name="X1", **kw)
        stamp(held["inst"], ctx, *[f"p{k}" for k in range(len(bias))])
        return ctx
    spec = cb.MNASpec(mode="tran")
    lc = cb.lower_circuit(cb.MNACircuit(builder, spec=spec))
    inst = held["inst"]
    S = ora.Structure(oracle_of(lc), ora.make_spec(mode="tran"))
    n = S.n
    rng = np.random.default_rng(11)
    collapsed = inst.collapsed(spec)
    cnode = {p: lc.index_of(f"p{k}") for k, p in enumerate(m.ports)}
    for node in m.internal:
        cnode[node] = cnode[collapsed[node]] if node in collapsed else lc.index_of(f"X1_{m.name}_{node}")
    u = np.zeros(n)
    for k, v in enumerate(bias):
        u[cnode[m.ports[k]] - 1] = v
    for node in m.internal:
        if node not in collapsed:
            u[cnode[node] - 1] = rng.uniform(min(bias), max(bias))
    lim = lc_limit_branches(lc)

    def settle(u):
        for k, (p, q) in enumerate(lim):
            u[n - lc.n_limits + k] = (u[p - 1] if p else 0.0) - (u[q - 1] if q else 0.0)
        return u

    def interp(u):
        V = {node: u[cnode[node] - 1] for node in m.nodes}
        it = inst._interp(spec)
        it.run(V, _VoldIsVnew(V))
        out = np.zeros(lc.n_nodes)
        for (p, q), i in it.I.items():
            if p in cnode:
                out[cnode[p] - 1] += i
            if q in cnode:
                out[cnode[q] - 1] -= i
        return out
    u = settle(u)
    G, C, b, _ = S.rebuild(u)
    Gd = S.dense(G)
    I_emit = (Gd @ u - b)[:lc.n_nodes]
    I_int = interp(u)
    assert np.all(np.isfinite(I_emit)) and np.all(np.isfinite(Gd))
    scale = max(float(np.abs(I_int).max()), 1e-30)
    assert np.max(np.abs(I_emit - I_int)) <= 1e-9 * scale, (m.name, I_emit, I_int)
    gs = float(np.abs(Gd[:lc.n_nodes, :lc.n_nodes]).max()) + 1e-30
    for j in range(lc.n_nodes):
        h = 1e-6
        up, um = u.copy(), u.copy()
        up[j] += h; um[j] -= h
        dI = (interp(settle(up)) - interp(settle(um))) / (2 * h)
        col = Gd[:lc.n_nodes, j].copy()
        for k, (p, q) in enumerate(lim):                     # limit unknowns follow their probes
            col += Gd[:lc.n_nodes, n - lc.n_limits + k] * ((1.0 if p == j + 1 else 0.0) - (1.0 if q == j + 1 else 0.0))
        assert np.max(np.abs(dI - col)) <= 1e-6 * gs, (m.name, j, float(np.max(np.abs(dI - col)) / gs))


def lc_limit_branches(lc):
    """(p, n) circuit nodes of each limit unknown, from its tracking row G[l,l]=1, G[l,p]=-1, G[l,n]=+1."""
    lim0 = lc.n - lc.n_limits
    out = [[0, 0] for _ in range(lc.n_limits)]
    seen = [0] * lc.n_limits
    for i, j in zip(lc.G_I, lc.G_J):
        if i > lim0 and j <= lc.n_nodes and seen[i - lim0 - 1] < 2:
            k = i - lim0 - 1
            out[k][seen[k]] = int(j)
            seen[k] += 1
    return [tuple(x) for x in out]


# ---- GPU parity ------------------------------------------------------------------------------
def _close(a, b, rtol=1e-9, atol=1e-12):
    return bool(np.all(np.abs(a - b) <= atol + rtol * np.maximum(np.abs(a), np.abs(b))))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mos1_corner", "diode_chain", "mos1_inverter", "bjt_ce", "jfet2_cs", "vdmos_cs",
                                  "inductor_rl", "bsim4_stage"])
def test_gpu_va_models_dc(name):
    lc = fixture(name)
    from cadnip_b200 import backend
    if name == "bsim4_stage" and not backend.va_models_cached(lc.va_cuda_header):
        pytest.skip("the sp_bsim4v8 kernel set is not in the in-tree cache (nvcc needs ~20 minutes for it)")
    nl = oracle_of(lc)
    comp = cb.CompiledSweep(lc, cb.MNASpec(mode="tran"))
    try:
        x, st, it = comp.dc()
    finally:
        comp.close()
    xo, sto, ito = ora.sweep_dc(nl, ora.make_spec(mode="dcop"), lc.n)
    assert np.array_equal(st, sto) and (st == 0).all()
    assert _close(x.T, xo), float(np.max(np.abs(x.T - xo)))          # north_star: 1e-9 rel / 1e-12 abs
    assert np.array_equal(it, ito)


@pytest.mark.gpu
@pytest.mark.parametrize("name,tspan,dt,method,spec", [
    ("mos1_inverter", (0.0, 10e-9), 1e-11, "trap", False),
    ("mos1_inverter", (0.0, 10e-9), 1e-11, "be", True),
    ("diode_rs_cap", (0.0, 10e-9), 1e-11, "trap", True),
    ("bjt_ce", (0.0, 2e-6), 1e-8, "be", False),
    ("bjt_ce", (0.0, 2e-6), 1e-8, "trap", True),
    ("vdmos_cs", (0.0, 1e-7), 1e-9, "be", False),
    ("inductor_rl", (0.0, 1e-5), 1e-7, "trap", False),
])
def test_gpu_va_models_transient(name, tspan, dt, method, spec):
    lc = fixture(name)
    nl = oracle_of(lc)
    save = list(range(1, lc.n + 1))
    comp = cb.CompiledSweep(lc, cb.MNASpec(mode="tran"))
    try:
        wave = comp.tran(tspan, dt, method=method, save_idxs=save, specialize=spec)
        r = wave.fetch(); wave.free()
        assert comp.handle.is_specialized() == spec
    finally:
        comp.close()
    o = ora.make_tran_opts(method={"be": 0, "trap": 1, "gear2": 2}[method], dt=dt)
    ro = ora.sweep_tran(nl, ora.make_spec(mode="tran"), tspan[0], tspan[1], o, save)
    gpu = np.transpose(r["u"], (2, 1, 0))
    ref = ro["u"][:, :gpu.shape[1], :]
    assert np.array_equal(r["status"], ro["status"]) and (r["status"] == 0).all()
    assert _close(gpu, ref), float(np.max(np.abs(gpu - ref)))
    if name == "bjt_ce":
        # the collector node carries mA currents: the residual norm sits at the rounding floor of the
        # 1e-10 A test on some steps, where GPU (static pivots) and oracle (partial pivoting) differ by
        # an iteration -- waveforms agree to 1e-9 above; counts to a few per cent
        assert np.all(np.abs(r["newton_iters"] - ro["newton_iters"]) <= 0.05 * ro["newton_iters"])
    else:
        assert np.array_equal(r["newton_iters"], ro["newton_iters"])
    if name == "mos1_inverter":
        q = gpu[:, :, lc.index_of("q") - 1]
        vdd = gpu[:, 0, lc.index_of("vdd") - 1]
        assert np.all(q.max(axis=1) > 0.95 * vdd)                          # it inverts ...
        assert np.all(q[:4].min(axis=1) < 0.05 * vdd[:4])                  # ... fully, with the 1 fF load


@pytest.mark.gpu
def test_gpu_global_workspace_path_with_ragged_lane_count(monkeypatch):
    """Lane state in HBM ([slot][lane], the layout for circuits too large for shared memory) with a
    lane count that is not a multiple of the block: every thread must own its workspace column."""
    monkeypatch.setenv("CB200_FORCE_GLOBAL_WS", "1")
    lc = fixture("mos1_inverter")                      # 8 lanes, blocks of 64
    nl = oracle_of(lc)
    save = list(range(1, lc.n + 1))
    comp = cb.CompiledSweep(lc, cb.MNASpec(mode="tran"))
    try:
        x, st, it = comp.dc()
        wave = comp.tran((0.0, 4e-9), 1e-11, method="trap", save_idxs=save)
        r = wave.fetch(); wave.free()
    finally:
        comp.close()
    xo, sto, ito = ora.sweep_dc(nl, ora.make_spec(mode="dcop"), lc.n)
    assert np.array_equal(st, sto) and _close(x.T, xo) and np.array_equal(it, ito)
    ro = ora.sweep_tran(nl, ora.make_spec(mode="tran"), 0.0, 4e-9, ora.make_tran_opts(method=1, dt=1e-11), save)
    gpu = np.transpose(r["u"], (2, 1, 0))
    assert (r["status"] == 0).all() and np.array_equal(r["newton_iters"], ro["newton_iters"])
    assert _close(gpu, ro["u"][:, :gpu.shape[1], :])


@pytest.mark.gpu
def test_gpu_va_c3_corner_lanes_with_transient_limiting():
    lc = fixture("mos1_c3")
    nl = oracle_of(lc)
    save = [lc.index_of("q"), lc.index_of("d")]
    comp = cb.CompiledSweep(lc, cb.MNASpec(mode="tran"))
    try:
        wave = comp.tran((0.0, 1.3e-7), 1e-10, method="be", save_idxs=save, save_every=10, limit=True)
        r = wave.fetch(); wave.free()
    finally:
        comp.close()
    ro = ora.sweep_tran(nl, ora.make_spec(mode="tran"), 0.0, 1.3e-7,
                        ora.make_tran_opts(method=0, dt=1e-10, save_every=10, limit=True), save)
    gpu = np.transpose(r["u"], (2, 1, 0))
    assert np.array_equal(r["status"], ro["status"]) and (r["status"] == 0).all()
    assert _close(gpu, ro["u"][:, :gpu.shape[1], :]), float(np.max(np.abs(gpu - ro["u"][:, :gpu.shape[1], :])))
    assert np.array_equal(r["newton_iters"], ro["newton_iters"])


@pytest.mark.gpu
def test_gpu_bypass_equals_plain_kernel(monkeypatch):
    """Two builds of the specialised fixed-step kernel on the C3 corner lanes must agree bit for bit --
    waveforms, statuses, Newton counts, segmented or not -- and match the oracle: the plain time loop
    (CB200_NO_BYPASS=1) and the default one with the quiescent-step bypass (steps whose first residual would be
    bitwise the one that just converged are not executed: lane_kernels.cuh, tran_fixed_body)."""
    lc = fixture("mos1_c3")
    nl = oracle_of(lc)
    save = [lc.index_of("q"), lc.index_of("d")]
    out = {}
    for build in ("plain", "bypass"):
        if build == "plain":
            monkeypatch.setenv("CB200_NO_BYPASS", "1")
        else:
            monkeypatch.delenv("CB200_NO_BYPASS", raising=False)
        comp = cb.CompiledSweep(lc, cb.MNASpec(mode="tran"))
        try:
            comp.specialize(1e-10, "be", limit=True, fixed_only=True)
            assert comp.handle.is_specialized()
            wave = comp.tran((0.0, 1.3e-7), 1e-10, method="be", save_idxs=save, save_every=10, limit=True)
            r = wave.fetch(); wave.free()
            host = np.full_like(r["u"], np.nan)
            r3 = comp.tran_fetch((0.0, 1.3e-7), 1e-10, host, method="be", save_idxs=save, save_every=10, limit=True,
                                 n_segments=3)
            out[build] = (r["u"], r["status"], r["newton_iters"], r3["u"], r3["newton_iters"], comp.handle.stats())
        finally:
            comp.close()
    for a, b in zip(out["plain"][:5], out["bypass"][:5]):
        assert np.array_equal(a, b, equal_nan=True)
    assert out["bypass"][5]["device_evals"] == out["plain"][5]["device_evals"]
    assert np.array_equal(out["bypass"][0], out["bypass"][3])   # segmented = single launch with the bypass
    ro = ora.sweep_tran(nl, ora.make_spec(mode="tran"), 0.0, 1.3e-7,
                        ora.make_tran_opts(method=0, dt=1e-10, save_every=10, limit=True), save)
    gpu = np.transpose(out["bypass"][0], (2, 1, 0))
    assert (out["bypass"][1] == 0).all() and _close(gpu, ro["u"][:, :gpu.shape[1], :])
    assert np.array_equal(out["bypass"][2], ro["newton_iters"])
    print("kernel ms: plain loop", out["plain"][5]["tran_kernel_ms"], "with bypass", out["bypass"][5]["tran_kernel_ms"])


@pytest.mark.gpu
def test_gpu_va_dff_adaptive():
    """C4 on the table-driven kernels (n = 145, ~5000 workspace doubles per lane: the lane-per-warp
    mapping, workspace row in HBM / L2) against the oracle, adaptive mode at the north_star
    tolerance: reltol 1e-6, time-point counts reported and equal, waveforms within reltol on the
    lanes' own (identical) time grids."""
    lc = fixture("mos1_dff")
    nl = oracle_of(lc)
    save = [lc.index_of("Q"), lc.index_of("Q_neg"), lc.index_of("net0")]
    reltol, lte_abstol, cap = 1e-6, 1e-9, 8000
    comp = cb.CompiledSweep(lc, cb.MNASpec(mode="tran"))
    try:
        x, st, it = comp.dc()
        wave = comp.tran_adaptive((0.0, 1.2e-7), dt0=1e-12, method="trap", save_idxs=save, reltol=reltol,
                                  lte_abstol=lte_abstol, max_points=cap, limit=True)
        r = wave.fetch(); wave.free()
    finally:
        comp.close()
    xo, sto, ito = ora.sweep_dc(nl, ora.make_spec(mode="dcop"), lc.n)
    assert np.array_equal(st, sto) and (st == 0).all() and _close(x.T, xo)
    # 120 pnjlim / fetlim decisions per PCNR iteration: on this circuit the iteration COUNT depends on the
    # rounding of the linear solve -- the oracle itself needs [38 36 30 34] iterations with its dense
    # partial-pivot LU and [37 36 36 34] with its fixed-pattern sparse LU, landing on the same point.  The GPU
    # (static pivots) must reproduce one of the two per lane, and exactly where they agree.
    ora.set_linear_solver(1)
    try:
        _, _, ito2 = ora.sweep_dc(nl, ora.make_spec(mode="dcop"), lc.n)
    finally:
        ora.set_linear_solver(0)
    assert np.all((it == ito) | (it == ito2)), (it, ito, ito2)
    o = ora.make_tran_opts(method=1, adaptive=1, dt=1e-12, reltol=reltol, lte_abstol=lte_abstol, max_points=cap,
                           limit=True)
    # The same sensitivity carries into the adaptive transient: a Newton solve that needs 10 iterations with one
    # LU rounding and 11 (= a rejected step) with the other changes the time grid from there on.  The oracle's own
    # two linear solvers give [2441 2378 2376 2340] and [2420 2377 2376 2340] points, identical grids for the
    # first ~1600 points and waveforms within 2e-10 V of each other over the whole span.  So per lane: the GPU
    # grid must coincide with one of the oracle's over a long common prefix (same controller, same decisions),
    # agree there within reltol, have a point count inside the oracle's own spread (2 %), and agree over the
    # whole span (oracle interpolated onto the GPU grid) within 10 reltol.
    ros = []
    for solver in (0, 1):
        ora.set_linear_solver(solver)
        try:
            ros.append(ora.sweep_tran(nl, ora.make_spec(mode="tran"), 0.0, 1.2e-7, o, save))
        finally:
            ora.set_linear_solver(0)
    assert (r["status"] == 0).all() and all(np.array_equal(r["status"], ro["status"]) for ro in ros)
    print("time points per lane: gpu", r["count"].tolist(), "oracle", [ro["T"].tolist() for ro in ros])
    scale = lte_abstol / reltol
    worst = worst_span = 0.0
    for p in range(lc.P):
        ng = int(r["count"][p])
        tg = r["t"][:ng, p]
        best = None
        for ro in ros:
            no = int(ro["T"][p])
            m = min(ng, no)
            same = np.isclose(tg[:m], ro["t"][p, :m], rtol=1e-9, atol=0.0)
            prefix = m if same.all() else int(np.argmin(same))
            if best is None or prefix > best[0]:
                best = (prefix, no, ro)
        prefix, no, ro = best
        assert abs(ng - no) <= 0.02 * no, (p, ng, no)
        assert prefix >= min(ng, no) // 2, (p, prefix, ng, no)
        for k in range(len(save)):
            a, b = r["u"][k, :prefix, p], ro["u"][p, :prefix, k]
            worst = max(worst, float(np.max(np.abs(a - b) / (scale + np.maximum(np.abs(a), np.abs(b))))))
            a = r["u"][k, :ng, p]
            b = np.interp(tg, ro["t"][p, :no], ro["u"][p, :no, k])
            worst_span = max(worst_span, float(np.max(np.abs(a - b) / (scale + np.maximum(np.abs(a), np.abs(b))))))
    print("max scaled waveform difference: common prefix", worst, "whole span (interpolated)", worst_span)
    assert worst <= reltol and worst_span <= 10 * reltol


@pytest.mark.gpu
def test_gpu_va_dff_lane_per_warp_equals_lane_per_thread(monkeypatch):
    """The flip-flop (n = 145, 30 FETs) runs on the lane-per-warp kernels with the level-scheduled
    refactor / solves; they must reproduce the serial lane-per-thread schedule bit for bit
    (DC state, PCNR iteration counts, adaptive time grid, waveforms)."""
    lc = fixture("mos1_dff")
    save = [lc.index_of("Q"), lc.index_of("Q_neg"), lc.index_of("net0")]

    def run():
        comp = cb.CompiledSweep(lc, cb.MNASpec(mode="tran"))
        try:
            mapping = comp.handle.lane_mapping()
            x, st, it = comp.dc()
            wave = comp.tran_adaptive((0.0, 4e-8), dt0=1e-12, method="trap", save_idxs=save, reltol=1e-3,
                                      lte_abstol=1e-5, max_points=4000, limit=True)
            r = wave.fetch(); wave.free()
            wave = comp.tran((0.0, 2e-9), 1e-11, method="trap", save_idxs=save, limit=True)
            rf = wave.fetch(); wave.free()
        finally:
            comp.close()
        T = int(r["count"].max())
        valid = np.arange(T)[:, None] < r["count"][None, :]
        return mapping, [x, st, it, r["count"], r["status"], r["newton_iters"], np.where(valid, r["t"][:T], 0.0),
                         np.where(valid[None], r["u"][:, :T], 0.0), rf["u"], rf["newton_iters"], rf["status"]]

    m_warp, got = run()
    assert m_warp == "warp"
    monkeypatch.setenv("CB200_LANE_PER_THREAD", "1")
    m_thr, ref = run()
    assert m_thr == "thread/hbm"
    for a, b in zip(ref, got):
        assert np.array_equal(np.asarray(a), np.asarray(b), equal_nan=True)


@pytest.mark.gpu
def test_gpu_va_ring_oscillator():
    lc = fixture("mos1_ring")
    nl = oracle_of(lc)
    save = [lc.index_of(n) for n in ("out1", "out2", "in1")]
    u0 = np.repeat(_ring_u0(lc)[:, None], lc.P, axis=1)
    comp = cb.CompiledSweep(lc, cb.MNASpec(mode="tran"))
    try:
        wave = comp.tran((0.0, 5e-9), 5e-12, method="trap", save_idxs=save, u0=u0)
        r = wave.fetch(); wave.free()
    finally:
        comp.close()
    o = ora.make_tran_opts(method=1, dt=5e-12, init=1)
    gpu = np.transpose(r["u"], (2, 1, 0))
    ref = np.stack([ora.tran(nl.for_lane(p), ora.make_spec(mode="tran"), 0.0, 5e-9, o, save,
                             u0=u0[:, p].copy())["u"][:gpu.shape[1]] for p in range(lc.P)])
    assert (r["status"] == 0).all()
    # a perturbation of 1e-13 of the start stays 1e-13 over this window (no amplification), so the
    # fixed-step bar applies to the oscillator as to every other circuit
    print("ring: max |gpu - oracle|", float(np.max(np.abs(gpu - ref))))
    assert _close(gpu, ref), float(np.max(np.abs(gpu - ref)))
    assert gpu[:, :, 0].max() - gpu[:, :, 0].min() > 2.0


# ---- large circuits: sparse symbolic analysis + one lane on a warp (C5, fallback tier) ----------
@pytest.mark.gpu
def test_gpu_c6288_slice_matches_oracle():
    """The first 70 gates (420 FETs) of the c6288 multiplier deck (benchmarks/vacask/c6288/cedarsim) on
    sp_mos1 cards: n = 1957 > 1536, so the pivot order comes from analyze_lu_sparse and the lane runs
    on the level-scheduled kernels.  DC (PCNR, 1680 limit unknowns) and 40 BE steps against the oracle
    (its fixed-pattern sparse LU: the dense checker is O(n^3) here)."""
    lc = fixture("mos1_c6288_slice")
    assert lc.n == 1957 and lc.n_limits == 1680
    nl = oracle_of(lc)
    save = list(range(1, lc.n_nodes + 1))
    comp = cb.CompiledSweep(lc, cb.MNASpec(mode="tran"))
    try:
        assert comp.handle.lane_mapping() == "warp"
        x, st, it = comp.dc()
        wave = comp.tran((0.0, 4e-10), 1e-11, method="be", save_idxs=save)
        r = wave.fetch(); wave.free()
    finally:
        comp.close()
    ora.set_linear_solver(1)
    try:
        xo, sto, ito = ora.sweep_dc(nl, ora.make_spec(mode="dcop"), lc.n)
        o = ora.make_tran_opts(method=0, dt=1e-11)
        ro = ora.sweep_tran(nl, ora.make_spec(mode="tran"), 0.0, 4e-10, o, save)
    finally:
        ora.set_linear_solver(0)
    assert np.array_equal(st, sto) and (st == 0).all() and np.array_equal(it, ito)
    assert _close(x.T, xo), float(np.max(np.abs(x.T - xo)))
    gpu = np.transpose(r["u"], (2, 1, 0))
    ref = ro["u"][:, :gpu.shape[1], :]
    assert np.array_equal(r["status"], ro["status"]) and (r["status"] == 0).all()
    assert _close(gpu, ref), float(np.max(np.abs(gpu - ref)))
    assert np.array_equal(r["newton_iters"], ro["newton_iters"])


@pytest.mark.gpu
def test_gpu_psp103_ring_matches_oracle():
    """PSP103 on the GPU: the ring's operating point (CedarTranOp) at 1e-9 relative / 1e-12 absolute and the first
    5 ns of its trapezoidal transient against the oracle (bar: see below), Newton counts within 2 %."""
    from cadnip_b200 import backend
    lc = fixture("psp_ring")
    if not backend.va_models_cached(lc.va_cuda_header):
        pytest.skip("the PSP103 kernel set is not in the in-tree cache (ptxas needs more than two hours for it)")
    nl = oracle_of(lc)
    save = [lc.index_of(str(k)) for k in range(1, 10)]
    comp = cb.CompiledSweep(lc, cb.MNASpec(mode="tran"))
    try:
        assert comp.handle.lane_mapping() == "warp"
        wave = comp.tran((0.0, 5e-9), 5e-11, method="trap", save_idxs=save)
        r = wave.fetch(); wave.free()
        st = comp.handle.stats()
    finally:
        comp.close()
    o = ora.make_tran_opts(method=1, dt=5e-11)
    ro = ora.sweep_tran(nl, ora.make_spec(mode="tran"), 0.0, 5e-9, o, save)
    gpu = np.transpose(r["u"], (2, 1, 0))
    ref = ro["u"][:, :gpu.shape[1], :]
    assert np.array_equal(r["status"], ro["status"]) and (r["status"] == 0).all()
    print("psp ring: max |gpu - oracle|", float(np.max(np.abs(gpu - ref))), "newton iters", r["newton_iters"].tolist(),
          ro["newton_iters"].tolist(), f"kernel {st['tran_kernel_ms']:.1f} ms")
    # The ring leaves a METASTABLE operating point: the start-up amplifies what the two sides bring along.  Measured
    # in the oracle alone: a 1e-13 relative perturbation of the start state is 1.1e-9 V after these 5 ns, 1e-12 is
    # 1.3e-8 V (x 1e4); the two operating points agree to the Newton tolerance (~1e-11 relative), which arrives as
    # 1.6e-7 V (measured on a B200).  So the bar here is 1e4 x the fixed-step bar (1e-6 V absolute, 1e-5 relative), not the fixed-step bar itself.
    assert np.all(np.abs(gpu - ref) <= 1e-6 + 1e-5 * np.maximum(np.abs(gpu), np.abs(ref))), float(np.max(np.abs(gpu - ref)))
    assert _close(gpu[:, 0, :], ref[:, 0, :])                # the operating point itself: the usual bar
    assert np.all(np.abs(r["newton_iters"] - ro["newton_iters"]) <= 0.02 * ro["newton_iters"])


@pytest.mark.gpu
def test_gpu_c6288_full_transient_residual():
    """The whole multiplier on sp_mos1 cards: 10 112 FETs, n = 45 604 (5 122 nodes, 34 source currents,
    40 448 limit unknowns), nnz 158 870 -- one lane on the 512 threads of a block, pivot order from the
    sparse analysis.  The oracle's LUs do not reach this size, so the GPU's result is checked through the
    oracle's OWN rebuild: after CedarUICOp (the reference's DC chain fails on this fallback-tier circuit
    exactly as it does when restated with SciPy on the host: undamped Newton overshoots the junction
    exponentials) and 20 backward-Euler steps, the last step must satisfy the reference's convergence
    criterion || C du + G u - b ||_2 < abstol (solve.jl:552) at the GPU's states."""
    lc = fixture("mos1_c6288")
    assert (lc.n, lc.n_nodes, lc.n_limits) == (45604, 5122, 40448)
    nl = oracle_of(lc)
    h = 1e-12
    comp = cb.CompiledSweep(lc, cb.MNASpec(mode="tran"))
    try:
        assert comp.handle.lane_mapping() == "block"          # one lane on the 512 threads of a block
        wave = comp.tran((0.0, 20 * h), h, method="be", save_idxs=list(range(1, lc.n + 1)), limit=True,
                         initializealg=cb.CedarUICOp(warmup_steps=10, dt=1e-13))
        r = wave.fetch(); wave.free()
        tstats = comp.handle.stats()
    finally:
        comp.close()
    assert (r["status"] == 0).all(), r["status"]
    u1, u0 = r["u"][:, -1, 0], r["u"][:, -2, 0]
    S = ora.Structure(nl, ora.make_spec(mode="tran"))
    G, C, b, lw = S.rebuild(u1, t=20 * h)
    a = S.arrays()
    cols = np.repeat(np.arange(lc.n), np.diff(a["colptr"]))
    F = np.zeros(lc.n)
    np.add.at(F, a["rowval"] - 1, G * u1[cols] + C * ((u1 - u0) / h)[cols])
    F -= b
    assert np.linalg.norm(F) < 1e-9, np.linalg.norm(F)
    print(f"c6288 (sp_mos1): 20 BE steps, {int(r['newton_iters'][0])} Newton iterations, "
          f"kernel {tstats['tran_kernel_ms']:.1f} ms")


# ---- C3 at BASELINE size (last on purpose: the longest single test) ------------------------------
@pytest.mark.gpu
def test_full_size_properties_c3():
    """BASELINE config C3 at full size -- the 50 x 50 x 40 grid, 100 000 lanes x 4000 BE steps on the specialised
    kernels, exactly what bench.py measures -- against the oracle on 24 SEEDED lanes of the grid (1e-9 / 1e-12 on
    every saved point, equal Newton counts), plus what must hold for every lane whatever its parameters."""
    from cadnip_b200 import workloads
    lc = workloads.load_workload("mos1_c3")
    lc.lane_soa, lc.P = workloads.c3_lanes(lc)
    assert lc.P == 100000
    save = [lc.index_of("q")]
    comp = cb.CompiledSweep(lc, cb.MNASpec(mode="tran"))
    try:
        comp.specialize(1e-10, "be", limit=True, fixed_only=True)
        wave = comp.tran((0.0, 4e-7), 1e-10, method="be", save_idxs=save, save_every=10, limit=True)
        r = wave.fetch(); wave.free()
        st = comp.handle.stats()
    finally:
        comp.close()
    u = r["u"][0]                                           # [T][P]
    assert u.shape == (401, 100000) and (r["status"] == 0).all() and np.all(np.isfinite(u))
    # the bypass skipped work, never results: executed lane-steps are counted, every point is there
    assert 0 < st["steps_accepted"] <= 4000 * 100000
    assert np.all(r["newton_iters"] > 0)
    rng = np.random.default_rng(20261019)
    lanes = np.sort(rng.choice(100000, 24, replace=False))
    sub = dict(lc.netlist_tables()); sub["par"] = np.ascontiguousarray(sub["par"][lanes])
    ora.load_va_models(lc.va_c_source)
    ro = ora.sweep_tran(ora.OracleNetlist(sub), ora.make_spec(mode="tran"), 0.0, 4e-7,
                        ora.make_tran_opts(method=0, dt=1e-10, save_every=10, limit=True), save)
    a, b = ro["u"][:, :401, 0], u[:, lanes].T
    assert (ro["status"] == 0).all()
    assert _close(a, b), float(np.max(np.abs(a - b)))
    assert np.array_equal(r["newton_iters"][lanes], ro["newton_iters"])
    print("C3 full size: 24 seeded lanes max |gpu - oracle|", float(np.max(np.abs(a - b))),
          "executed lane-steps", int(st["steps_accepted"]), "of", 4000 * 100000, "kernel ms", st["tran_kernel_ms"])
