#!/usr/bin/env python
"""bench.py -- headline measurement of the batched MNA Newton/transient hot path.

Default workload = the north_star target (BASELINE.json configs[2], SURVEY.md 8d C3): the CMOS
inverter CircuitSweep, 100 000 parameter points (50 W_n x 50 Vdd x 40 C_L), sp_mos1 Verilog-A
FETs through the emitter, DC operating point (CedarTranOp / PCNR) + fixed-step backward-Euler
transient, 4000 steps of 0.1 ns.  One "step" of this benchmark = one full pass of that sweep.
With --gpus N the ONE sweep is partitioned: rank g solves lanes [g*ceil(P/N), (g+1)*ceil(P/N))
(sweep order, src/sweeps.jl:272), no collective on the hot path, and the final waveforms of all
ranks are gathered into one host array [save][T][P] (strong scaling).
Metric: transient sweep points per second (lanes completed / time); Newton iterations per second
reported alongside.  Other BASELINE configs: --workload c1 | c2 | c4.

    python bench.py --gpus N --steps K --warmup W            # B200 arm
    python bench.py --impl reference ...                     # CPU oracle arm
    python bench.py --dump-outputs DIR ...                   # also write the last timed step's results

The run writes nothing into the source tree: kernels and model code it compiles go to a temporary
directory (kernel sets that __graft_entry__.build() prebuilt are read from the tree).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np

N_R, N_C = 256, 256
N_SEGMENTS = int(os.environ.get("CB200_SEGMENTS", "8"))
# integrator of the adaptive workloads (c4, ring, c5): "trap" (LTE-controlled trapezoid, default) or "bdf" (the
# variable-order BDF controller of the IDA family, DESIGN.md s. 5)
ADAPTIVE_METHOD = os.environ.get("CB200_ADAPTIVE_METHOD", "")       # "" = the workload's own choice
assert ADAPTIVE_METHOD in ("", "trap", "bdf")
METRIC = "transient_sweep_points_per_sec"
UNIT = "points/s"
# parity gate of the same-run spot check against the oracle (north_star, fixed step)
RTOL, ATOL = 1e-9, 1e-12
WORKLOADS = {
    "c1": dict(tspan=(0.0, 4e-7), dt=1e-10, save_every=10, save="q", steps=4000, limit=True, fixture="mos1_c3",
               lanes=1,
               text="C1 CMOS inverter, SINGLE point (W_n = 0.36 um, Vdd = 1.8 V, C_L = 1 fF; deck of "
                    "benchmarks/benchmark_common.jl:82-106 with sp_mos1 cards): DC op + fixed-step BE 4000 x 0.1ns; also "
                    "the time of one residual+Jacobian evaluation on the device"),
    "c2": dict(tspan=(0.0, 2e-3), dt=1e-6, save_every=10, save="out", steps=2000, limit=False,
               text="C2 RC/diode clipper CircuitSweep: 65536 points (256 R x 256 C, log grids), DC op "
                    "(CedarTranOp/PCNR) + fixed-step BE 2000 x 1us; V(out) saved every 10th step"),
    "c3": dict(tspan=(0.0, 4e-7), dt=1e-10, save_every=10, save="q", steps=4000, limit=True, fixture="mos1_c3",
               text="C3 CMOS inverter CircuitSweep (sp_mos1 Verilog-A model through the emitter): 100000 points "
                    "(50 W_n x 50 Vdd x 40 C_L), DC op (CedarTranOp/PCNR) + fixed-step BE 4000 x 0.1ns "
                    "(CB200_TRAN_LIMIT: steps that miss 10 Newton solves are redone with $limit damping); "
                    "V(q) saved every 10th step"),
    "c4": dict(tspan=(0.0, 6e-7), dt=1e-12, save_every=1, save="Q", steps=0, limit=True, adaptive=True,
               reltol=float(os.environ.get("CB200_C4_RELTOL", "1e-3")), lte_abstol=1e-5,
               max_points=int(os.environ.get("CB200_C4_MAXPOINTS", "2048")), probe_per_core=2,
               fixture="mos1_dff",
               text="C4 gf180 D flip-flop corner/Monte-Carlo CircuitSweep (30 FETs; PDK cards absent -> FALLBACK tier: "
                    "sp_mos1 Verilog-A model, synthetic 5 V card, 5 fF parasitic per net): 16384 points (4 corners x "
                    "4096 draws), DC op (PCNR + fallbacks) + adaptive trapezoidal/LTE transient (0, 6e-7); "
                    "table-driven kernels, one lane per warp"),
    "ring": dict(tspan=(0.0, float(os.environ.get("CB200_RING_TSTOP", "1e-6"))), dt=1e-12, save_every=1, save="1", steps=0,
                 limit=False, adaptive=True, method="bdf", oscillator=True, reltol=1e-2, lte_abstol=1e-4, dtmax=0.05e-9, cpu_tstop=2e-8,
                 max_points=int(os.environ.get("CB200_RING_MAXPOINTS", "49152")), probe_per_core=1, fixture="psp_ring",
                 lanes=int(os.environ.get("CB200_RING_LANES", "1024")),
                 text="9-stage PSP103 ring oscillator (benchmarks/vacask/ring/cedarsim: 18 PSP103VA FETs with the deck's "
                      "psp103n / psp103p cards through the emitter, n = 370), swept over the supply voltage (1.0 .. 1.4 V); "
                      "CedarTranOp + adaptive variable-order BDF transient (0, 1e-6), reltol 1e-2, abstol 1e-4, dtmax 0.05 ns "
                      "(the reference's benchmark settings, runme.jl:47-67); table-driven kernels, one lane per warp"),
    "c5": dict(tspan=(0.0, 2e-9), dt=1e-12, save_every=1, save="p0", steps=0, limit=True, adaptive=True,
               reltol=float(os.environ.get("CB200_C5_RELTOL", "1e-5")), lte_abstol=1e-6,
               max_points=int(os.environ.get("CB200_C5_MAXPOINTS", "4096")), fixture="mos1_c6288", lanes=1, init="uic",
               text="C5 ISCAS c6288 16x16 multiplier (benchmarks/vacask/c6288/cedarsim: 10112 FETs, 32 pulse drivers), "
                    "single large circuit on 1 GPU; FALLBACK tier: sp_mos1 cards (vto +-0.4 V, kp 200u/100u, 1 fF per net) instead "
                    "of PSP103 (which emits and lowers -- workloads.psp_c6288, n = 212228 -- but whose 10112-instance kernel "
                    "set is not built here), n = 45604, nnz 158870; CedarUICOp "
                    "(the reference's DC chain fails on this fallback-tier circuit: undamped Newton overshoots the junction "
                    "exponentials -- restated with SciPy on the host it fails the same way) + adaptive trapezoidal/LTE "
                    "transient (0, 2e-9), lte abstol 1e-6; sparse symbolic analysis (threshold Markowitz on sparse rows), "
                    "level-scheduled LU, one lane on the 512 threads of a block"),
}
W = WORKLOADS["c3"]
TSPAN, DT, SAVE_EVERY, WORKLOAD = W["tspan"], W["dt"], W["save_every"], W["text"]


def select_workload(name):
    global W, TSPAN, DT, SAVE_EVERY, WORKLOAD
    W = WORKLOADS[name]
    TSPAN, DT, SAVE_EVERY, WORKLOAD = W["tspan"], W["dt"], W["save_every"], W["text"]
    global ADAPTIVE_METHOD
    if not ADAPTIVE_METHOD:
        # the PSP103 ring rings under the trapezoidal rule (the LTE estimate stops shrinking with h at
        # t = 11 ns and the controller walks h down to dtmin, in the oracle as on the device); the
        # variable-order BDF controller -- the reference's own solver family -- integrates it
        ADAPTIVE_METHOD = W.get("method", "trap")
    if W.get("adaptive"):
        WORKLOAD += f"; reltol {W['reltol']:g}"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--lanes", type=int, default=0, help="debug: override lane count")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the results of the B200 arm")
    return args


class ClockSampler:
    """nvidia-smi clocks line sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(smax)) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_sweep(args):
    """(lowered circuit with the FULL sweep's lane columns, P).  VA circuits: .va source -> emitter ->
    lower where the reference tree is mounted, else the committed lowered circuit (workloads.load_workload)."""
    import cadnip_b200 as cb
    from cadnip_b200 import workloads
    if args.workload == "c4":
        lc = workloads.load_workload(W["fixture"])
        lc.lane_soa, lc.P = workloads.c4_lanes(lc, args.lanes)
        return cb, lc, lc.P
    if args.workload == "c5":
        lc = workloads.load_fixture(W["fixture"]) if os.path.exists(workloads.fixture_path(W["fixture"])) \
            else workloads.load_workload(W["fixture"])
        return cb, lc, lc.P
    if args.workload == "ring":
        lc = workloads.load_fixture(W["fixture"]) if os.path.exists(workloads.fixture_path(W["fixture"])) \
            else workloads.load_workload(W["fixture"])
        P = args.lanes or W["lanes"]
        assert lc.lane_soa.shape[0] == 1, "the ring fixture sweeps the supply voltage only"
        lc.lane_soa, lc.P = np.ascontiguousarray(np.linspace(1.0, 1.4, P)[None, :]), P
        return cb, lc, P
    if args.workload in ("c3", "c1"):
        lc = workloads.load_workload(W["fixture"])
        if args.workload == "c1":
            lc.lane_soa, lc.P = workloads.c3_lanes(lc, shape=(50, 50, 40))
            lc.lane_soa, lc.P = np.ascontiguousarray(lc.lane_soa[:, :1]), 1
        else:
            lc.lane_soa, lc.P = workloads.c3_lanes(lc, args.lanes)
        return cb, lc, lc.P
    side = max(1, int(round(args.lanes ** 0.5))) if args.lanes else 0
    cs = workloads.clipper_sweep(side or N_R, side or N_C)
    params, P = cs.lane_params()
    lc = cb.lower(cs.builder, params, cb.MNASpec(mode="tran"), P=P)
    return cb, lc, P


def host_threads() -> int:
    """All host threads this process may use (torchrun exports OMP_NUM_THREADS=1; the
    oracle's thread count is set explicitly instead)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def oracle_opts():
    import cadnip_oracle as ora
    if W.get("adaptive"):
        return ora.make_tran_opts(method=3 if ADAPTIVE_METHOD == "bdf" else 1, adaptive=1, dt=DT, reltol=W["reltol"], lte_abstol=W["lte_abstol"],
                                  max_points=W["max_points"], limit=W["limit"], dtmax=W.get("dtmax", 0.0))
    return ora.make_tran_opts(method=0, dt=DT, save_every=SAVE_EVERY, limit=W["limit"])


def cpu_oracle_rate(lc, sample_lanes, nthreads=0):
    """Times the CPU oracle (kind 'port') on a strided sample of the same sweep."""
    import cadnip_oracle as ora
    nthreads = nthreads or host_threads()
    if lc.va_c_source:
        ora.load_va_models(lc.va_c_source)
    sub = dict(lc.netlist_tables()); sub["par"] = np.ascontiguousarray(sub["par"][sample_lanes])
    nls = ora.OracleNetlist(sub)
    # "cpu_tstop": the oracle integrates only the first part of the transient (a periodic steady
    # state: every part costs the same) and the rate is scaled to the whole span
    tstop = W.get("cpu_tstop", TSPAN[1])
    frac = (tstop - TSPAN[0]) / (TSPAN[1] - TSPAN[0])
    # the TIMED leg uses the oracle's fixed-pattern sparse LU (what KLU does for the reference); its dense
    # partial-pivot LU stays the checker of the parity tests and of the spot check below
    # (for n < 64 the dense elimination is the faster of the two and is kept: an honest baseline)
    ora.set_linear_solver(1 if lc.n >= 64 else 0)
    try:
        t0 = time.perf_counter()
        r = ora.sweep_tran(nls, ora.make_spec(mode="tran"), TSPAN[0], tstop, oracle_opts(), [lc.index_of(W["save"])],
                           nthreads=nthreads)
        dt = time.perf_counter() - t0
    finally:
        ora.set_linear_solver(0)
    return len(sample_lanes) * frac / dt, int(r["newton_iters"].sum()), dt


def model_op_counts(lc, lanes):
    """FP64 operations ONE call of the emitted model code executes, averaged over the full transient
    of the given lanes: the oracle's C with verilog_a.instrument_ops counters (single thread).
    Returns (flops, transcendentals, calls) or None for circuits without Verilog-A devices."""
    if not lc.va_c_source:
        return None
    import cadnip_oracle as ora
    ora.load_va_models(lc.va_c_source, count_ops=True)
    sub = dict(lc.netlist_tables()); sub["par"] = np.ascontiguousarray(sub["par"][lanes])
    ora.va_op_reset()
    ora.sweep_tran(ora.OracleNetlist(sub), ora.make_spec(mode="tran"), TSPAN[0], TSPAN[1], oracle_opts(),
                   [lc.index_of(W["save"])], nthreads=1)
    f, t, calls = ora.va_op_counts()
    ora.load_va_models(lc.va_c_source)              # back to the uninstrumented build
    return f, t, calls


# static estimates for the native devices (lane_kernels.cuh: eval_device), flops incl. one exp as 1
NATIVE_EVAL_FLOPS = {10: 27, 11: 45, 12: 25}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path.  The reference is
    Julia and cannot run here (DESIGN.md), so this is the oracle port, all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb, lc, P = build_sweep(args)
    cores = host_threads()
    # calibrate a bounded sample: ~4 s of wall per step
    probe = np.linspace(0, P - 1, min(P, W.get("probe_per_core", 64) * cores), dtype=np.int64)
    rate, _, _ = cpu_oracle_rate(lc, probe)
    n_sample = int(min(P, max(len(probe), rate * 4.0)))
    lanes = np.linspace(0, P - 1, n_sample, dtype=np.int64)
    for _ in range(min(args.warmup, 1)):
        cpu_oracle_rate(lc, lanes)
    t0 = time.perf_counter()
    iters = 0
    for _ in range(args.steps):
        _, it, _ = cpu_oracle_rate(lc, lanes)
        iters += it
    wall = time.perf_counter() - t0
    value = n_sample * args.steps / wall
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "newton_iters_per_sec": iters / wall,
            "config": {"workload": WORKLOAD, "lanes_per_step": n_sample, "lanes_total": P},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{n_sample} of {P} lanes (strided over the sweep), full "
                                       f"{'adaptive' if W.get('adaptive') else str(W['steps']) + '-step'} transient each, "
                                       "OpenMP over lanes"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


DUMP_BYTES = 64_000_000


def dump_outputs(path, u, t, st, adaptive):
    """--dump-outputs: what the sweep's caller receives from the last timed step, as <path>/<name>.npy in float64.
    u [save][T][P] waveforms and t ([T], or [T][P] when adaptive) come for a fixed, seeded sample of lanes
    (lanes.npy) sized so that all files stay within DUMP_BYTES; status, newton_iters and count (saved points)
    come for every lane.  Adaptive waveforms are zero past a lane's count."""
    os.makedirs(path, exist_ok=True)
    n_save, T, P = u.shape
    budget = DUMP_BYTES - 4096 - 8 * 3 * P - (0 if adaptive else 8 * T)          # 4096: the .npy headers
    k = int(min(P, budget // (8 * (T * (n_save + adaptive) + 1))))
    lanes = np.arange(P) if k == P else np.sort(np.random.default_rng(0).choice(P, k, replace=False))
    valid = np.arange(T)[:, None] < st[2, lanes][None, :]
    out = {"lanes": lanes, "status": st[0], "newton_iters": st[1], "count": st[2],
           "u": np.where(valid[None], u[:, :, lanes], 0.0),
           "t": np.where(valid, t[:, lanes], 0.0) if adaptive else t}
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))


def run_b200(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 arm has no CPU fallback")
    torch.cuda.set_device(local_rank)
    # stdout carries exactly one JSON line: whatever libraries print there while the run is in
    # progress (NCCL's version banner at the first collective) is sent to stderr instead
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    from cadnip_b200 import backend, distributed
    numa = distributed.pin_to_gpu_numa_node(local_rank) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    cb, lc, P = build_sweep(args)
    if args.workload == "c5":
        # a single large circuit does not shard (SURVEY 8e: "1 GPU, replicas only"); the CPU oracle's
        # linear solvers (dense O(n^3), dense-bookkeeping sparse analysis) do not reach n = 45604
        if world > 1:
            raise SystemExit("bench.py: C5 is a single large circuit on 1 GPU (replicas only); run with --gpus 1")
        args.no_cpu_baseline = True
    # strong scaling: the ONE sweep is block-partitioned over the ranks in sweep order
    sl = distributed.shard_slice(P, rank, world)
    Pl = sl.stop - sl.start
    if Pl <= 0:
        raise SystemExit(f"bench.py: rank {rank} of {world} has no lanes (P = {P})")
    comp = cb.CompiledSweep(lc, cb.MNASpec(mode="tran"), device=local_rank, lanes=sl)
    save = [lc.index_of(W["save"])]
    adaptive = bool(W.get("adaptive"))
    T = W["max_points"] if adaptive else backend.fixed_step_points(TSPAN[0], TSPAN[1], DT, SAVE_EVERY)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    # destination of the end-of-run gather: ONE host array [save][T][P] for the whole sweep, shared
    # by the ranks of the node and page-locked in each; rank g's GPU writes columns sl directly
    out_full = distributed.SharedSweepBuffer((len(save), T, P))
    t_full = distributed.SharedSweepBuffer((T, P)) if adaptive else None
    st_full = distributed.SharedSweepBuffer((3, P), dtype=np.int32, pin=False)     # status, newton iters, count
    out_np = out_full.lane_block(sl)
    pinned_in = torch.from_numpy(np.ascontiguousarray(comp._soa)).pin_memory()
    comp._soa = pinned_in.numpy()
    peak_tf, peak_ms = backend.measure_fp64_peak(local_rank)

    # 30 inlined model instances are beyond a straight-line kernel: C4 runs table-driven
    use_spec = os.environ.get("CB200_NO_SPECIALIZE", "0") != "1" and not adaptive
    if use_spec:
        comp.specialize(DT, "be", limit=W["limit"], fixed_only=True)        # emitter: circuit-specialised kernels (nvcc)

    def tran_resident():
        if adaptive:
            return comp.tran_adaptive(TSPAN, dt0=DT, method=ADAPTIVE_METHOD, save_idxs=save, reltol=W["reltol"],
                                      lte_abstol=W["lte_abstol"], max_points=W["max_points"], limit=W["limit"],
                                      dtmax=W.get("dtmax", 0.0),
                                      initializealg=cb.CedarUICOp(10, 1e-13) if W.get("init") == "uic" else None)
        return comp.tran(TSPAN, DT, method="be", save_idxs=save, save_every=SAVE_EVERY, limit=W["limit"])

    def step_resident():
        wave = tran_resident()
        return wave, comp.handle.stats()

    def step_e2e():
        comp.upload_lanes()                                   # H2D from pinned memory
        h2d = comp.handle.stats()["h2d_bytes"]
        if adaptive:                                          # ragged waveforms: one D2H after the run
            wave = tran_resident()
            st = comp.handle.stats()
            r = wave.fetch(out_np, t_full.lane_block(sl)); wave.free()
            d2h = int(out_np.size * 8 + T * Pl * 8 + 12 * Pl)
        else:
            # tran! into pinned host memory: D2H of each time segment overlaps the next one's compute
            r = comp.tran_fetch(TSPAN, DT, out_np, method="be", save_idxs=save, save_every=SAVE_EVERY,
                                n_segments=N_SEGMENTS, limit=W["limit"])
            st = comp.handle.stats()
            d2h = st["d2h_bytes"]
        st_full.array[0, sl] = r["status"]; st_full.array[1, sl] = r["newton_iters"]; st_full.array[2, sl] = r["count"]
        return st, r, h2d, d2h

    # ---- warm-up -----------------------------------------------------------
    sampler = ClockSampler(local_rank)
    sampler.start()                      # started early: nvidia-smi start-up must not land in the timed region
    iters_local = None
    for _ in range(max(args.warmup, 3)):
        wave, st = step_resident()
        if iters_local is None:
            r = wave.fetch()
            first_u = r["u"][0].copy()                    # [T][Pl] saved waveform of the first pass
            first_t, first_count = (r["t"].copy(), r["count"].copy()) if adaptive else (None, None)
            iters_local = int(r["newton_iters"].astype(np.int64).sum())
            evals_local = int(st["device_evals"])
            exec_local = int(st["steps_accepted"])          # fixed step: lane-steps the kernel executed
            bad = int((r["status"] != 0).sum())
            if bad:
                raise SystemExit(f"bench.py: {bad} lanes did not converge")
        wave.free()
        flush.zero_()
    step_e2e()

    # ---- timed: inputs resident in HBM --------------------------------------
    time.sleep(0.3)                      # samples cover warm-up and both timed regions (same load)
    barrier()
    t0 = time.perf_counter()
    kern_ms = tran_ms = 0.0
    launches = 0
    last_wave = None
    for i in range(args.steps):
        wave, st = step_resident()
        kern_ms += st["kernel_ms"]; tran_ms += st["tran_kernel_ms"]; launches += st["launches"]
        if args.dump_outputs and i == args.steps - 1:
            last_wave = wave                 # fetched after the timed region
        else:
            wave.free()
        flush.zero_()
    barrier()
    wall = time.perf_counter() - t0
    if last_wave is not None:                # every rank's block of the sweep into the shared host arrays
        r = last_wave.fetch(out_np, t_full.lane_block(sl) if adaptive else None)
        last_wave.free()
        st_full.array[0, sl] = r["status"]; st_full.array[1, sl] = r["newton_iters"]; st_full.array[2, sl] = r["count"]
        barrier()
        if rank == 0:
            dump_outputs(args.dump_outputs, out_full.array, t_full.array if adaptive else r["t"], st_full.array,
                         adaptive)
    # ---- timed: end to end through the C ABI with host buffers; ends when every rank's block of
    # the full-sweep waveform array is in host memory (the final gather) -------
    barrier()
    t1 = time.perf_counter()
    for _ in range(args.steps):
        st, r, h2d, d2h = step_e2e()
        flush.zero_()
    barrier()
    wall_e2e = time.perf_counter() - t1
    clocks = sampler.stop()

    tot = torch.tensor([float(iters_local), float(evals_local), float(h2d), float(d2h), float(launches), float(exec_local)],
                       dtype=torch.float64, device="cuda")
    if world > 1:
        tt = torch.tensor([wall, wall_e2e, tran_ms, kern_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        wall, wall_e2e, tran_ms, kern_ms = [float(x) for x in tt]
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    iters_per_step, evals_per_step, h2d_all, d2h_all, launches_all, executed_steps = [int(x) for x in tot.tolist()]
    value = P * args.steps / wall
    e2e = P * args.steps / wall_e2e
    gathered_ok = True
    if rank == 0:                        # the gathered result: every lane's status and waveform are here
        gathered_ok = bool((st_full.array[0] == 0).all()) and bool(np.isfinite(out_full.array[0, -1]).all())

    # ---- roofline of the dominant kernel (the time-loop kernel) ---------------
    rowp, colp, nnz_lu = comp.handle.pivot_order()
    colptr, rowval = comp.handle.pattern()
    nnz_j, n = len(rowval), lc.n
    b_iter = 8 * (nnz_j + 2 * nnz_lu + 4 * n)                 # SURVEY 8d: bytes / Newton iteration / lane
    out_bytes = 8 * len(save) * T * P
    par_bytes = 8 * lc.n_lane_cols * P
    alg_bytes = iters_per_step * b_iter + out_bytes + par_bytes          # whole sweep, all ranks
    tran_s = (tran_ms / args.steps) * 1e-3                               # max over ranks
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_achieved = alg_bytes / world / tran_s / 1e9 if tran_s > 0 else 0.0   # per GPU
    traffic = fp64_ncu = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if world == 1 and not args.lanes:
            ent = tj.get({"c2": "tran_fixed_kernel", "c3": "c3_spec_tran_fixed_kernel",
                          "c4": "c4_tran_adaptive_warp_kernel"}.get(args.workload, ""))
            traffic = ent
    except Exception:
        pass
    mapping = comp.handle.lane_mapping()
    kernel_name = ("cb200_spec_tran_fixed_kernel (circuit-specialised, lane state in registers)" if comp.handle.is_specialized()
                   else (("tran_adaptive" if adaptive else "tran_fixed") +
                         {"warp": "_warp_kernel (table-driven, one lane per warp, workspace row in HBM/L2)",
                          "block": "_block_kernel (table-driven, one lane per block of 512 threads, workspace row in HBM/L2)",
                          "thread/hbm": "_kernel<global> (table-driven, one lane per thread, lane state in HBM)",
                          "thread/smem": "_kernel<smem> (table-driven, one lane per thread)"}[mapping]))
    hbm_obj = {"achieved": hbm_achieved, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_achieved / hbm_peak,
               "algorithmic_bytes_per_launch_per_gpu": alg_bytes // world, "bytes_per_newton_iter_per_lane": b_iter,
               "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s"}
    if comp.handle.is_specialized() or mapping == "thread/smem":
        # FP64 roofline (SURVEY 8d): the fused kernel keeps the lane state on chip, so the FP64 pipe
        # is the bound.  Executed flops = device-model evaluation passes x the flops one pass
        # executes (emitter op counter, run in the oracle over the sampled lanes' transients) +
        # the static counts of assembly / refactor / solves (cb200_flop_model).
        fm = comp.handle.flop_model()
        nsteps_total = W["steps"] * P
        if rank == 0:
            chk_lanes = np.linspace(0, P - 1, min(P, 8), dtype=np.int64)
            oc = model_op_counts(lc, chk_lanes)
        else:
            oc = None
        if lc.va_c_source:
            oc_t = torch.tensor(list(oc) if oc else [0.0, 0.0, 1.0], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.broadcast(oc_t, src=0)
            f_call, t_call = float(oc_t[0] / oc_t[2]), float(oc_t[1] / oc_t[2])
            n_va = int((lc.dev_kind == 13).sum())
            f_eval = n_va * (f_call + t_call)
            eval_note = (f"emitted model code: {f_call:.0f} flops + {t_call:.0f} div/sqrt/exp/log/pow (each counted as ONE "
                         f"flop) per call, executed-path count from the op-counting build of the emitted C over the "
                         f"sampled lanes' transients; {n_va} calls per evaluation pass")
        else:
            f_eval = float(sum(NATIVE_EVAL_FLOPS.get(int(k), 0) for k in lc.dev_kind))
            eval_note = "native device models: static estimate per evaluation pass (exp counted as one flop)"
        # assemblies executed: one per EXECUTED lane-step + one per Newton solve.  The specialised kernel's
        # quiescent-step bypass does not execute steps whose first residual would be bitwise the one that just
        # converged; the lane-steps it did execute are counted on the device (cb200_stats.steps_accepted)
        bypass = comp.handle.is_specialized() and not adaptive and os.environ.get("CB200_NO_BYPASS") is None
        assemblies = iters_per_step + (executed_steps if bypass else nsteps_total)
        flops = (evals_per_step * f_eval + assemblies * fm["assemble_tran"] +
                 iters_per_step * (fm["factor_tran"] + fm["solve_tran"] + fm["update"]))
        achieved = flops / world / tran_s / 1e12 if tran_s > 0 else 0.0
        roof = {"bound": "fp64", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": achieved / peak_tf if peak_tf else None, "traffic": traffic, "kernel": kernel_name,
                "flops_per_launch_per_gpu": int(flops // world),
                "device_eval_passes_per_launch": evals_per_step, "flops_per_eval_pass": f_eval,
                "assemblies_counted": int(assemblies), "quiescent_step_bypass": bool(bypass),
                "lane_steps_executed": int(executed_steps), "lane_steps_total": int(nsteps_total),
                "linear_algebra_flops_per_iter": fm,
                "peak_source": f"measured in this run: cb200_measure_fp64_peak, register-only FMA kernel, 8 chains/thread, "
                               f"64 warps/SM, {peak_ms:.2f} ms (2 flops per FMA)",
                "note": eval_note + "; evaluation passes counted on the device (cb200_stats.device_evals): a step "
                        "whose first residual re-uses the stamps of the previous step's converged check executes none"
                        + ("; quiescent-step bypass on: a backward-Euler step whose sources are bitwise unchanged after a "
                           "step that converged without a solve is not executed (bit-identical results); executed lane-steps "
                           "counted on the device" if bypass else ""),
                "hbm_algorithmic": hbm_obj}
    else:
        roof = {"bound": "hbm", **hbm_obj, "traffic": traffic, "kernel": kernel_name,
                "note": ("lane state is a [lane][slot] row in global memory shared by the 32 threads of the lane's "
                         "warp; `traffic` = ncu dram bytes of one full launch" if mapping == "warp" else
                         "lane state is a [slot] row in global memory shared by the 512 threads of the lane's block"
                         if mapping == "block" else
                         "lane state in HBM ([slot][thread] workspace)")}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": 1e3 * wall / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "newton_iters_per_sec": iters_per_step * args.steps / wall,
            "newton_iters_per_step": iters_per_step,
            "config": {"workload": WORKLOAD, "lanes_total": P, "lanes_per_gpu": -(-P // world),
                       "parallelism": (f"the one {P}-lane sweep block-partitioned over {world} GPUs in sweep order "
                                       f"(rank g: lanes [g*{-(-P // world)}, (g+1)*{-(-P // world)})), structure replicated, "
                                       "no hot-path collective; every rank's waveform block lands in ONE shared "
                                       "page-locked host array [save][T][P] (final gather)") if world > 1 else "1 GPU",
                       "method": (f"adaptive {'variable-order BDF (1..5, IDA family)' if ADAPTIVE_METHOD == 'bdf' else 'trapezoidal + LTE'}, reltol {W['reltol']:g}, <= {W['max_points']} points/lane"
                                  if adaptive else f"BE fixed dt={DT:g}, {W['steps']} steps"),
                       "numa_cpus": numa,
                       "l2": "256 MiB device memset between steps (inside the timed region)"},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d_all, "d2h_bytes_per_step": d2h_all,
                    "ms_per_step": 1e3 * wall_e2e / args.steps, "gathered_all_lanes_ok": gathered_ok,
                    "path": ("cb200_set_lanes (pinned H2D) + cb200_tran_fetch_ld (" + str(N_SEGMENTS) + " time segments, each "
                             "D2H'd into this rank's column block of the shared host array while the next computes)")
                            if not adaptive else
                            "cb200_set_lanes (pinned H2D) + cb200_tran + cb200_wave_fetch_ld into the shared host array"},
            "gpu_launches": launches_all,
            "kernel_ms_per_step": kern_ms / args.steps, "tran_kernel_ms_per_step": tran_ms / args.steps,
            "roofline": roof, "clocks": clocks}
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            import cadnip_oracle as ora
            cores = host_threads()
            probe = np.linspace(0, P - 1, min(P, W.get("probe_per_core", 64) * cores), dtype=np.int64)
            rate, _, _ = cpu_oracle_rate(lc, probe)
            n_sample = int(min(P, max(len(probe), rate * 12.0)))
            lanes = np.linspace(0, P - 1, n_sample, dtype=np.int64)
            rate, it, secs = cpu_oracle_rate(lc, lanes)
            # spot check of the measured pass against the oracle (8 lanes spread over the sweep)
            chk = np.linspace(0, P - 1, min(P, 8), dtype=np.int64)
            sub = dict(lc.netlist_tables()); sub["par"] = np.ascontiguousarray(sub["par"][chk])
            chk_tstop = W.get("cpu_tstop", TSPAN[1])        # ring: the first 20 ns (5 periods) of the microsecond
            ro = ora.sweep_tran(ora.OracleNetlist(sub), ora.make_spec(mode="tran"), TSPAN[0], chk_tstop, oracle_opts(),
                                [lc.index_of(W["save"])])
            if adaptive:                                  # ragged time axes: same grid expected, compare point by point
                diff, tdiff, same_counts = 0.0, 0.0, True
                for q, lane in enumerate(chk):
                    ng, no = int(first_count[lane]), int(ro["T"][q])
                    same_counts &= (ng == no)
                    m = min(ng, no)
                    if chk_tstop < TSPAN[1]:
                        m = max(1, no - 2)          # the oracle's last step is cut to its shorter span
                    if W.get("oscillator"):
                        # a free-running oscillator started from a metastable point amplifies the 1e-11 the two
                        # operating points differ by (x 1e4 per 5 ns, tests/test_va_models.py): the pointwise gate
                        # covers the common prefix of the two time grids (identical controller decisions)
                        same = np.isclose(first_t[:m, lane], ro["t"][q, :m], rtol=1e-9, atol=0.0)
                        m = m if same.all() else max(1, int(np.argmin(same)))
                        prefix_pts = m if q == 0 else min(prefix_pts, m)
                    tdiff = max(tdiff, float(np.max(np.abs(first_t[:m, lane] - ro["t"][q, :m]))))
                    a, b = first_u[:m, lane], ro["u"][q, :m, 0]
                    diff = max(diff, float(np.max(np.abs(a - b) / (ATOL / W["reltol"] + np.maximum(np.abs(a), np.abs(b))))))
                line["parity"] = {"lanes_checked": len(chk), "max_rel_diff_vs_oracle": diff, "max_time_diff": tdiff,
                                  "timepoints_gpu": [int(first_count[l]) for l in chk],
                                  "timepoints_oracle": [int(c) for c in ro["T"]],
                                  "gate": f"same controller on both sides: relative difference <= reltol = {W['reltol']:g}"}
                if W.get("oscillator"):
                    line["parity"]["gate"] += f" on the common prefix of the time grids (>= {prefix_pts} points per lane)"
                    same_counts = True
                if not diff <= W["reltol"]:
                    raise SystemExit(f"bench.py: GPU waveform differs from the oracle by {diff} (relative)")
            else:
                a, b = ro["u"][:, :first_u.shape[0], 0], first_u[:, chk].T
                err = np.abs(a - b) - (ATOL + RTOL * np.maximum(np.abs(a), np.abs(b)))
                diff = float(np.max(np.abs(a - b)))
                line["parity"] = {"lanes_checked": len(chk), "max_abs_diff_vs_oracle": diff,
                                  "gate": f"|gpu - oracle| <= {ATOL:g} + {RTOL:g} * max(|gpu|, |oracle|) on every saved point"}
                if not float(np.max(err)) <= 0.0:
                    raise SystemExit(f"bench.py: GPU waveform differs from the oracle by {diff}")
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                                    "newton_iters_per_sec": it / secs,
                                    "linear_solver": ("fixed-pattern sparse LU (oracle linear solver 1)" if lc.n >= 64 else
                                                      "dense LU with partial pivoting (n < 64: faster than the sparse one)"),
                                    "sample": f"{n_sample} of {P} lanes (strided over the sweep), " +
                                              (f"the first {W['cpu_tstop']:g} s of the {TSPAN[1]:g} s transient (periodic steady state; "
                                               f"rate scaled to the full span), " if "cpu_tstop" in W else "full ") +
                                              f"{'adaptive' if adaptive else str(W['steps']) + '-step'} transient each, "
                                              f"OpenMP over lanes, {secs:.1f} s"}
        if args.workload == "c1" and world == 1:
            line["c1"] = c1_eval_times(cb, backend)
        if args.workload == "ring":
            us_iter_lane = 1e6 * wall / args.steps / max(iters_per_step, 1)
            line["ring"] = {"n": lc.n, "lanes": P, "newton_iters_per_lane": iters_per_step / P,
                            "timepoints_per_lane": float(np.mean(first_count)),
                            "us_per_newton_iter_amortised": us_iter_lane,
                            "us_per_newton_iter_one_lane_latency": us_iter_lane * P,
                            "reference_published": {"cadnip_us_per_iter": 1376.0, "vacask_us_per_iter": 27.8,
                                                    "cadnip_points": 43968, "cadnip_newton_iters": 242293, "cadnip_wall_s": 333.5,
                                                    "source": "doc/ring_oscillator_investigation.md:297-313 (dev box, 1 thread)"},
                            "note": "amortised = wall / (Newton iterations of ALL lanes): the throughput figure of a sweep; "
                                    "one-lane latency = wall / iterations of ONE lane (every lane advances concurrently)"}
        if args.workload == "c5":
            ms_iter = 1e3 * wall / args.steps / max(iters_per_step, 1)
            line["c5"] = {"n": lc.n, "nnz_J": nnz_j, "nnz_LU": int(nnz_lu), "timepoints": int(first_count[0]),
                          "newton_iters": iters_per_step, "ms_per_newton_iter": ms_iter,
                          "reference_published": {"per_newton_iter_s": {"rebuild": 0.480, "residual": 0.657, "jacobian": 1.017,
                                                                         "klu_factor_solve": 2.72},
                                                  "n": 212228, "nnz_J": 2452148, "model": "PSP103",
                                                  "timepoints_reltol_1e-5": 118,
                                                  "source": "doc/c6288_bottleneck_findings.md:87-91,111-118; "
                                                            "benchmarks/vacask/c6288/cedarsim/runme.jl:60-66"},
                          "note": "same topology, different device model (sp_mos1 fallback) and therefore a 4.7x smaller "
                                  "system: the per-iteration times are not like for like"}
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port",
                                    "sample": "not run: the oracle's linear solvers do not reach n = 45604; the DC point is "
                                              "checked through the oracle's own rebuild (tests/test_va_models.py)"}
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
    comp.close()
    out_full.close(); st_full.close()
    if t_full is not None:
        t_full.close()
    if world > 1:
        dist.destroy_process_group()


def c1_eval_times(cb, backend):
    """What the legacy bench measured (benchmarks/benchmark_common.jl:130-181): the time of one
    residual / Jacobian evaluation.  Here fast_rebuild! (device evaluation K1 + assembly K2) over
    many copies of the single point; G, C and b come out of the same pass."""
    from cadnip_b200 import workloads
    lc = workloads.load_workload("mos1_c3")
    soa, _ = workloads.c3_lanes(lc, shape=(50, 50, 40))
    out = {}
    for Pn in (1, 65536):
        lc.lane_soa, lc.P = np.ascontiguousarray(np.repeat(soa[:, :1], Pn, axis=1)), Pn
        comp = cb.CompiledSweep(lc, cb.MNASpec(mode="tran"), device=0)
        try:
            x = np.zeros((lc.n, Pn))
            best = 1e30
            for _ in range(5):
                comp.handle.eval(comp.spec, x, 0.0)
                best = min(best, comp.handle.stats()["kernel_ms"])
        finally:
            comp.close()
        out[f"rebuild_ns_per_evaluation_P{Pn}"] = best * 1e6 / Pn
    out["note"] = ("one fast_rebuild! = residual AND Jacobian data (G, C, b) in one pass; P1 = latency of a single "
                   "evaluation (3 launches), P65536 = throughput per evaluation when batched")
    return out


def main():
    args = parse()
    select_workload(args.workload)
    import cadnip_oracle as ora
    from cadnip_b200 import backend
    with tempfile.TemporaryDirectory(prefix="cadnip_b200_bench_") as cache:
        backend.RUN_CACHE_DIR = os.path.join(cache, "kernels")
        ora.GEN_DIR = os.path.join(cache, "oracle")
        if args.impl == "reference":
            run_reference(args)
        else:
            run_b200(args)


if __name__ == "__main__":
    main()
