// lane_kernels.cuh -- sm_100a device code of the batched MNA Newton / transient hot path.
//
// Mapping (DESIGN.md): one sweep lane per thread.  A lane's whole Newton state --
// iterate, history, stamp values, the sparse LU factor -- is private to its thread:
//   * generic kernels: a column of shared memory, ws[slot * blockDim.x + threadIdx.x]
//     (fp64, conflict-free: a warp touches 32 consecutive 8-byte words), or of a
//     global [slot][lane] array when the circuit is too large for shared memory
//     (coalesced: lane is the fastest index);
//   * specialised kernels (generated per circuit by specialize.cpp): a register
//     array whose indices are all compile-time constants.
// Lanes never communicate: no barriers, no atomics.
//
// Every kernel is a template over a program type PG and an LU-schedule type LU:
//   * DynProg / DynLu read the device table, segment lists and elimination schedule
//     from read-only global arrays at warp-uniform addresses (one compiled kernel
//     serves every circuit);
//   * a generated StaticProg / StaticLu exposes the same accessors as constexpr
//     functions, so after unrolling every index is an immediate and the kernel is
//     straight-line code for that circuit.
//
// The device-evaluation functions restate the stamp! methods of
// src/mna/devices.jl; they write each stamp VALUE to the slot the reference's
// DirectStampContext would have visited at that program position
// (src/mna/value_only.jl:395-478).  Assembly then sums every matrix entry's segment
// of stamp slots left to right, i.e. in program order: the same floating-point
// summation order as the reference's `nzval[map[pos]] += v`, without atomics.
#pragma once
#include <cfloat>
#include <cmath>
#include <cstdint>

#include <cuda_runtime.h>

#include "../../include/cadnip_b200.h"
#include "kernels.h"

namespace cb200 {

// ---------------------------------------------------------------------------
// dynamic (table-driven) program / LU accessors
// ---------------------------------------------------------------------------
struct DynProg {
    static constexpr bool kStatic = false;
    static constexpr int kUnroll = 1;
    static constexpr int kMethod = -1;      // integration method chosen at run time
    static constexpr bool kTranLimit = true; // CB200_TRAN_LIMIT supported (specialised kernels: opt-in)
    static constexpr bool kBypass = false;   // quiescent-step bypass of tran_fixed_body (generated programs only)
    const Program &p;
    __device__ __forceinline__ explicit DynProg(const Program &pp) : p(pp) {}
    __device__ __forceinline__ int n() const { return p.n; }
    __device__ __forceinline__ int n_limits() const { return p.n_limits; }
    __device__ __forceinline__ int nnz() const { return p.nnz; }
    __device__ __forceinline__ int n_dev() const { return p.n_dev; }
    __device__ __forceinline__ int n_src() const { return p.n_src; }
    __device__ __forceinline__ int n_nl() const { return p.n_nl; }
    __device__ __forceinline__ int n_lane_cols() const { return p.n_lane_cols; }
    __device__ __forceinline__ int src_list(int q) const { return __ldg(p.src_list + q); }
    __device__ __forceinline__ int nl_list(int q) const { return __ldg(p.nl_list + q); }
    __device__ __forceinline__ bool src_uniform(int q) const { return __ldg(p.src_uniform + q) != 0; }
    __device__ __forceinline__ int dev_kind(int d) const { return __ldg(p.dev_kind + d); }
    __device__ __forceinline__ int dev_flags(int d) const { return __ldg(p.dev_flags + d); }
    __device__ __forceinline__ int dev_node_ptr(int d) const { return __ldg(p.dev_node_ptr + d); }
    __device__ __forceinline__ int dev_node(int i) const { return __ldg(p.dev_nodes + i); }
    __device__ __forceinline__ int dev_param_ptr(int d) const { return __ldg(p.dev_param_ptr + d); }
    __device__ __forceinline__ int dev_param(int i) const { return __ldg(p.dev_params + i); }
    __device__ __forceinline__ int dev_gbase(int d) const { return __ldg(p.dev_gbase + d); }
    __device__ __forceinline__ int dev_cbase(int d) const { return __ldg(p.dev_cbase + d); }
    __device__ __forceinline__ int dev_bbase(int d) const { return __ldg(p.dev_bbase + d); }
    __device__ __forceinline__ int dev_sbase(int d) const { return __ldg(p.dev_sbase + d); }
    __device__ __forceinline__ double uniform(int r) const { return __ldg(p.uniform + r); }
    __device__ __forceinline__ int limit_init_ref(int k) const { return __ldg(p.limit_init_ref + k); }
    __device__ __forceinline__ int gseg_ptr(int s) const { return __ldg(p.gseg_ptr + s); }
    __device__ __forceinline__ int gseg_idx(int q) const { return __ldg(p.gseg_idx + q); }
    __device__ __forceinline__ int cseg_ptr(int s) const { return __ldg(p.cseg_ptr + s); }
    __device__ __forceinline__ int cseg_idx(int q) const { return __ldg(p.cseg_idx + q); }
    __device__ __forceinline__ int bseg_ptr(int r) const { return __ldg(p.bseg_ptr + r); }
    __device__ __forceinline__ int bseg_idx(int q) const { return __ldg(p.bseg_idx + q); }
    __device__ __forceinline__ int colptr(int j) const { return __ldg(p.colptr + j); }
    __device__ __forceinline__ int rowval(int s) const { return __ldg(p.rowval + s); }
    __device__ __forceinline__ bool nz_is_node_diag(int s) const { return __ldg(p.nz_is_node_diag + s) != 0; }
    __device__ __forceinline__ int off_u() const { return p.off_u; }
    __device__ __forceinline__ int off_un() const { return p.off_un; }
    __device__ __forceinline__ int off_dterm() const { return p.off_dterm; }
    __device__ __forceinline__ int off_F() const { return p.off_F; }
    __device__ __forceinline__ int off_wv() const { return p.off_wv; }
    __device__ __forceinline__ int off_SG() const { return p.off_SG; }
    __device__ __forceinline__ int off_SC() const { return p.off_SC; }
    __device__ __forceinline__ int off_SB() const { return p.off_SB; }
    __device__ __forceinline__ int off_LU() const { return p.off_LU; }
    __device__ __forceinline__ int off_limw() const { return p.off_limw; }
    __device__ __forceinline__ int off_lp() const { return p.off_lp; }
    __device__ __forceinline__ int off_DS() const { return p.off_DS; }
    __device__ __forceinline__ int off_srcc() const { return p.off_srcc; }
    __device__ __forceinline__ int off_h1() const { return p.off_h1; }
    __device__ __forceinline__ int off_h2() const { return p.off_h2; }
    __device__ __forceinline__ int off_phi() const { return p.off_phi; }
    // lane-per-warp kernels only (warp_kernels.cuh)
    __device__ __forceinline__ int rowptr(int r) const { return __ldg(p.rowptr + r); }
    __device__ __forceinline__ int row_nz(int q) const { return __ldg(p.row_nz + q); }
    __device__ __forceinline__ int nz_col(int s) const { return __ldg(p.nz_col + s); }
    __device__ __forceinline__ int off_GS() const { return p.off_GS; }
    __device__ __forceinline__ int off_CS() const { return p.off_CS; }
    __device__ __forceinline__ int off_DI() const { return p.off_DI; }
};

struct DynLu {
    const LuProgram &l;
    __device__ __forceinline__ explicit DynLu(const LuProgram &ll) : l(ll) {}
    __device__ __forceinline__ int n() const { return l.n; }
    __device__ __forceinline__ int n_fill() const { return l.n_fill; }
    __device__ __forceinline__ int rowperm(int k) const { return __ldg(l.rowperm + k); }
    __device__ __forceinline__ int colperm(int k) const { return __ldg(l.colperm + k); }
    __device__ __forceinline__ int diag_slot(int k) const { return __ldg(l.diag_slot + k); }
    __device__ __forceinline__ int Lptr(int k) const { return __ldg(l.Lptr + k); }
    __device__ __forceinline__ int L_slot(int e) const { return __ldg(l.L_slot + e); }
    __device__ __forceinline__ int L_row(int e) const { return __ldg(l.L_row + e); }
    __device__ __forceinline__ int Uptr(int k) const { return __ldg(l.Uptr + k); }
    __device__ __forceinline__ int U_slot(int q) const { return __ldg(l.U_slot + q); }
    __device__ __forceinline__ int U_col(int q) const { return __ldg(l.U_col + q); }
    __device__ __forceinline__ int tgt_ptr(int k) const { return __ldg(l.tgt_ptr + k); }
    __device__ __forceinline__ int tgt(int q) const { return __ldg(l.tgt + q); }
    __device__ __forceinline__ int jmap(int s) const { return __ldg(l.jmap + s); }
    __device__ __forceinline__ int fill_slot(int q) const { return __ldg(l.fill_slots + q); }
};

// ---------------------------------------------------------------------------
// lane workspace accessors
// ---------------------------------------------------------------------------
template <typename IdxT>
struct LaneWs {
    double *ws;
    IdxT stride;
    bool weak = false;              // a refactor of this lane met a weak pivot (weak_pivot())
    __device__ __forceinline__ double &operator()(int slot) const { return ws[(IdxT)slot * stride]; }
};

template <int N>
struct RegWs {                      // specialised kernels: constant indices -> registers
    double r[N > 0 ? N : 1];
    bool weak = false;
    __device__ __forceinline__ double &operator()(int slot) { return r[slot]; }
};

// Static-pivot safeguard (SURVEY H2).  The pivot order is chosen once on the host from sample
// lanes; a lane whose values differ may meet a pivot that is tiny against its column -- not zero,
// so the solve goes on, but with element growth 1/ratio.  A multiplier |l| = |a_ik / pivot| beyond
// 1e8 (what partial pivoting would never produce: |l| <= 1, KLU's threshold: <= 1e3) marks the lane;
// the mark is advisory -- the kernel carries on -- and the host re-solves marked lanes with a pivot
// order chosen from their own values (cb200_weak_pivot_lanes).  Integer test on the high word: no
// FP64 issue slot; NaN / Inf multipliers are marked too.
__device__ __forceinline__ bool weak_pivot(double l)
{
    return (__double2hiint(l) & 0x7fffffff) > 0x4197d783;        // |l| > ~1e8
}

#define CB_UNROLL _Pragma("unroll (PG::kUnroll)")

template <typename PG, typename W>
__device__ __forceinline__ double param(const PG &pg, W &w, int pbase, int i)
{
    const int r = pg.dev_param(pbase + i);
    return r >= 0 ? pg.uniform(r) : w(pg.off_lp() + ~r);
}

// u[idx] with a run-time index (saved-output gather).  A register workspace must
// never be indexed dynamically, so the static variant selects over constant slots.
template <typename PG, typename W>
__device__ __forceinline__ double read_u(const PG &pg, W &w, int idx)
{
    if constexpr (PG::kStatic) {
        double v = 0.0;
        CB_UNROLL
        for (int i = 0; i < pg.n(); i++) {
            // read first, select after: a guarded read lets the optimiser substitute the
            // run-time idx for the constant i and demote the register array to local memory
            const double ui = w(pg.off_u() + i);
            v = (idx == i) ? ui : v;
        }
        return v;
    } else {
        return w(pg.off_u() + idx);
    }
}

template <typename PG, typename W>
__device__ __forceinline__ double xval(const PG &pg, W &w, int idx)
{
    // V_k = node_k == 0 ? 0.0 : x[node_k]   (devices.jl:1373)
    return idx == 0 ? 0.0 : w(pg.off_u() + idx - 1);
}

// ---------------------------------------------------------------------------
// waveforms (src/mna/devices.jl:30-216)
// ---------------------------------------------------------------------------
__device__ __forceinline__ double d_mod(double x, double y)   // Julia mod, y > 0
{
    double r = fmod(x, y);
    if (r != 0.0 && ((r < 0.0) != (y < 0.0))) r += y;
    return r;
}

// Base.sind restated: exact reduction mod 360, octant folding.
__device__ __forceinline__ double d_sind(double x)
{
    const double d2r = 0.017453292519943295;
    if (isnan(x) || isinf(x)) return NAN;
    const double rx = copysign(fmod(x, 360.0), x);
    const double arx = fabs(rx);
    if (rx == 0.0) return rx;
    else if (arx < 45.0) return sin(rx * d2r);
    else if (arx <= 135.0) return copysign(cos((90.0 - arx) * d2r), rx);
    else if (arx == 180.0) return copysign(0.0, rx);
    else if (arx < 225.0) return sin(((180.0 - arx) * (rx < 0 ? -1.0 : 1.0)) * d2r);
    else if (arx <= 315.0) return -copysign(cos((270.0 - arx) * d2r), rx);
    else return sin((rx - copysign(360.0, rx)) * d2r);
}

// pulse_at_time  devices.jl:85-103
__device__ __forceinline__ double d_pulse(double v1, double v2, double td, double tr, double tf,
                                          double pw, double per, double t)
{
    if (t < td) return v1;
    const double phase = per > 0 ? d_mod(t - td, per) : (t - td);
    if (phase < tr) return tr > 0 ? v1 + (v2 - v1) * (phase / tr) : v2;
    else if (phase < tr + pw) return v2;
    else if (phase < tr + pw + tf) return tf > 0 ? v2 + (v1 - v2) * ((phase - tr - pw) / tf) : v1;
    else return v1;
}

// get_source_value (devices.jl:352-360) over PWLWave / PulseWave / SinWave.
// params: [0] = dc, [1..] = wave parameters.
template <typename PG, typename W>
__device__ __forceinline__ double source_value(const PG &pg, W &w, int wave, int pb, int npar,
                                               double t, int mode)
{
    if (wave == CB200_WAVE_NONE) return param(pg, w, pb, 0);
    if (mode == CB200_MODE_DCOP || mode == CB200_MODE_AC) return param(pg, w, pb, 0);
    if (wave == CB200_WAVE_SIN) {          // SinWave  devices.jl:168-174
        const double vo = param(pg, w, pb, 1), va = param(pg, w, pb, 2), fr = param(pg, w, pb, 3);
        const double td = param(pg, w, pb, 4), th = param(pg, w, pb, 5), ph = param(pg, w, pb, 6);
        if (t < td) return vo + va * d_sind(ph);
        return vo + va * exp(-th * (t - td)) * d_sind(360 * fr * (t - td) + ph);
    }
    if (wave == CB200_WAVE_PULSE) {
        return d_pulse(param(pg, w, pb, 1), param(pg, w, pb, 2), param(pg, w, pb, 3),
                       param(pg, w, pb, 4), param(pg, w, pb, 5), param(pg, w, pb, 6),
                       param(pg, w, pb, 7), t);
    }
    // PWL: pwl_at_time devices.jl:47-71 with find_t_in_ts :30-36.  Written as a
    // branch-free scan so that it unrolls for a static program.
    // Every parameter is READ FIRST and selected after: a read guarded by `k == i` lets the
    // optimiser substitute the run-time i for the constant k, i.e. index the parameter tables --
    // and through them the register workspace -- dynamically, which demotes the whole lane state
    // of a specialised kernel to local memory.
    const int np = (npar - 1) / 2;
    int i = 1;                              // 1-based searchsortedfirst
    CB_UNROLL
    for (int k = 1; k <= np; k++) {
        const double tk = param(pg, w, pb, 1 + 2 * (k - 1));
        i = (tk < t) ? k + 1 : i;
    }
    double result = 0.0;
    bool found = false;
    // step past an exact hit
    bool hit = false;
    CB_UNROLL
    for (int k = 1; k <= np; k++) {
        const double tk = param(pg, w, pb, 1 + 2 * (k - 1));
        hit = (k == i && tk == t) ? true : hit;
    }
    if (hit) i++;
    const double y_first = param(pg, w, pb, 2), y_last = param(pg, w, pb, 2 + 2 * (np - 1));
    if (i <= 1) { result = y_first; found = true; }
    if (!found && i > np) { result = y_last; found = true; }
    if (!found) {
        double t0 = 0, y0 = 0, t1 = 0, y1 = 0;
        CB_UNROLL
        for (int k = 2; k <= np; k++) {
            const double a0 = param(pg, w, pb, 1 + 2 * (k - 2)), b0 = param(pg, w, pb, 2 + 2 * (k - 2));
            const double a1 = param(pg, w, pb, 1 + 2 * (k - 1)), b1 = param(pg, w, pb, 2 + 2 * (k - 1));
            const bool sel = (k == i);
            t0 = sel ? a0 : t0; y0 = sel ? b0 : y0;
            t1 = sel ? a1 : t1; y1 = sel ? b1 : y1;
        }
        if (y0 == y1) result = y1;
        else if (t1 == t0) result = (y0 + y1) / 2;
        else {
            const double slope = (y1 - y0) / (t1 - t0);
            result = y0 + (t - t0) * slope;
        }
    }
    return result;
}

// ---------------------------------------------------------------------------
// exp for the junction models.  Same algorithm as any libm exp (k = rint(x/ln2),
// Cody-Waite reduction, polynomial, scale by 2^k; <= 1 ulp), but the coefficients sit
// in constant memory so that every FMA takes its coefficient as a constant-bank
// operand: libdevice's exp spends more issue slots materialising its fp64 immediates
// (UMOV + IMAD.MOV pairs) than on arithmetic, and this kernel is issue-bound.
// ---------------------------------------------------------------------------
__constant__ double cb200_exp_coef[14] = {
    1.0, 1.0, 0.5, 1.6666666666666666e-01, 4.1666666666666664e-02, 8.3333333333333332e-03,
    1.3888888888888889e-03, 1.9841269841269841e-04, 2.4801587301587302e-05, 2.7557319223985893e-06,
    2.7557319223985888e-07, 2.5052108385441720e-08, 2.0876756987868100e-09, 1.6059043836821613e-10};

__device__ __forceinline__ double d_exp(double x)
{
    if (!(fabs(x) < 700.0)) return exp(x);                 // overflow / underflow / NaN: library path
    const double magic = 6755399441055744.0;               // 1.5 * 2^52: rounds to nearest integer
    const double t = fma(x, 1.4426950408889634, magic);
    const double k = t - magic;
    double r = fma(k, -6.93147180369123816490e-01, x);     // ln2 high part (exact product for |k| < 2^11)
    r = fma(k, -1.90821492927058770002e-10, r);            // ln2 low part
    double p = cb200_exp_coef[13];
#pragma unroll
    for (int i = 12; i >= 0; i--) p = fma(p, r, cb200_exp_coef[i]);
    const int ki = __double2loint(t);                      // low word of the magic sum = k
    return __hiloint2double(__double2hiint(p) + (ki << 20), __double2loint(p));
}

// ---------------------------------------------------------------------------
// limiting primitives (src/mna/devices.jl:1169-1258, :1333-1345)
// ---------------------------------------------------------------------------
__device__ __forceinline__ double d_pnjlim(double vnew, double vold, double vt, double vcrit)
{
    if (vnew > vcrit && fabs(vnew - vold) > vt + vt) {
        if (vold > 0.0) {
            const double arg = (vnew - vold) / vt;
            if (arg > 0.0) return vold + vt * (2.0 + log(arg - 2.0));
            return vold - vt * (2.0 + log(2.0 - arg));
        }
        return vt * log(vnew / vt);
    } else if (vnew < 0.0) {
        const double arg = vold > 0.0 ? -vold - 1.0 : 2.0 * vold - 1.0;
        if (vnew < arg) return arg;
    }
    return vnew;
}

__device__ __forceinline__ void d_diode_iv(double Is, double nVt, double v, double &I0, double &Gd)
{
    const double xarg = v / nVt;
    if (xarg > 80.0) {
        const double e80 = exp(80.0);
        I0 = Is * (e80 * (1.0 + (xarg - 80.0)) - 1.0);
        Gd = Is / nVt * e80;
    } else {
        const double expterm = d_exp(xarg);
        I0 = Is * (expterm - 1.0);
        Gd = Is / nVt * expterm;
    }
}

// diode_junction_cap  devices.jl:1505-1516
__device__ __forceinline__ double d_junction_cap(double V, double Cj0, double Vj, double m)
{
    const double Vmax = 0.9 * Vj;
    if (V < Vmax) return Cj0 / pow(1 - V / Vj, m);
    const double C_at_max = Cj0 / pow(1 - Vmax / Vj, m);
    const double dC_dV = Cj0 * m / Vj / pow(1 - Vmax / Vj, m + 1);
    return C_at_max + dC_dV * (V - Vmax);
}

// ---------------------------------------------------------------------------
// Verilog-A modules: the emitter (cadnip_b200/verilog_a.py) writes one va_stamp_<module>
// function per module plus va_dispatch; kernels that serve circuits with VA devices
// are compiled with -DCB200_VA_HEADER="...".
// ---------------------------------------------------------------------------
#ifdef CB200_VA_HEADER
#include CB200_VA_HEADER
#endif
// A nonlinear device whose stamps depend on the time ($abstime in a Verilog-A module) as well as on
// the iterate: the time loops then re-evaluate at the start of every step (see `fresh` below).
#ifdef CB200_VA_TIME_DEP
constexpr bool kNlTimeDep = true;
#else
constexpr bool kNlTimeDep = false;
#endif
#ifndef CB200_VA_HEADER
template <int PASS, typename PG, typename W>
__device__ __forceinline__ void va_dispatch(const PG &, W &, int, int, double, int, bool) {}
#endif

// ---------------------------------------------------------------------------
// device evaluation: one stamp! call.
//   PASS 0 writes every stamp (once per kernel);
//   PASS 1 writes the stamps that depend on the iterate x (every Newton iteration);
//   PASS 2 writes the stamps that depend on time only (once per time step).
// Slot positions advance identically in every pass.
// ---------------------------------------------------------------------------
#define ST_G(i, j, v) do { if ((i) != 0 && (j) != 0) { if (PASS == 0) w(g) = (v); g++; } } while (0)
#define DY_G(i, j, v) do { if ((i) != 0 && (j) != 0) { w(g) = (v); g++; } } while (0)
#define ST_C(i, j, v) do { if ((i) != 0 && (j) != 0) { if (PASS == 0) w(c) = (v); c++; } } while (0)
#define DY_C(i, j, v) do { if ((i) != 0 && (j) != 0) { w(c) = (v); c++; } } while (0)
#define DY_B(i, v)    do { if ((i) != 0) { w(b) = (v); b++; } } while (0)

template <int PASS, typename PG, typename W>
__device__ __forceinline__ void eval_device(const PG &pg, W &w, int d, double t, int mode,
                                            bool initjct)
{
    const int kind = pg.dev_kind(d), flags = pg.dev_flags(d);
    const int nb = pg.dev_node_ptr(d);
    const int pb = pg.dev_param_ptr(d);
    const int npar = pg.dev_param_ptr(d + 1) - pb;
    int g = pg.off_SG() + pg.dev_gbase(d);
    int c = pg.off_SC() + pg.dev_cbase(d);
    int b = pg.off_SB() + pg.dev_bbase(d);
    (void)npar; (void)c; (void)b; (void)flags; (void)g;

    switch (kind) {
    case CB200_DEV_RESISTOR: {                       // devices.jl:498-510
        const int pp = pg.dev_node(nb), nn = pg.dev_node(nb + 1);
        const double G = 1.0 / param(pg, w, pb, 0);
        ST_G(pp, pp, G); ST_G(pp, nn, -G); ST_G(nn, pp, -G); ST_G(nn, nn, G);
    } break;
    case CB200_DEV_CAPACITOR: {                      // devices.jl:531-534
        const int pp = pg.dev_node(nb), nn = pg.dev_node(nb + 1);
        const double C = param(pg, w, pb, 0);
        ST_C(pp, pp, C); ST_C(pp, nn, -C); ST_C(nn, pp, -C); ST_C(nn, nn, C);
    } break;
    case CB200_DEV_INDUCTOR: {                       // devices.jl:569-586
        const int pp = pg.dev_node(nb), nn = pg.dev_node(nb + 1), I = pg.dev_node(nb + 2);
        ST_G(pp, I, 1.0); ST_G(nn, I, -1.0); ST_G(I, pp, 1.0); ST_G(I, nn, -1.0);
        ST_C(I, I, -param(pg, w, pb, 0));
    } break;
    case CB200_DEV_VSOURCE: {                        // devices.jl:643-663
        const int pp = pg.dev_node(nb), nn = pg.dev_node(nb + 1), I = pg.dev_node(nb + 2);
        ST_G(pp, I, 1.0); ST_G(nn, I, -1.0); ST_G(I, pp, 1.0); ST_G(I, nn, -1.0);
        if (PASS != 1) DY_B(I, source_value(pg, w, flags, pb, npar, t, mode));
    } break;
    case CB200_DEV_ISOURCE: {                        // devices.jl:719-737
        const int pp = pg.dev_node(nb), nn = pg.dev_node(nb + 1);
        if (PASS != 1) {
            const double i = source_value(pg, w, flags, pb, npar, t, mode);
            DY_B(pp, i); DY_B(nn, -i);
        }
    } break;
    case CB200_DEV_VCVS: {                           // devices.jl:760-775
        const int op = pg.dev_node(nb), on = pg.dev_node(nb + 1), ip = pg.dev_node(nb + 2);
        const int in = pg.dev_node(nb + 3), I = pg.dev_node(nb + 4);
        const double A = param(pg, w, pb, 0);
        ST_G(op, I, 1.0); ST_G(on, I, -1.0); ST_G(I, op, 1.0); ST_G(I, on, -1.0);
        ST_G(I, ip, -A); ST_G(I, in, A);
    } break;
    case CB200_DEV_VCCS: {                           // devices.jl:797-808
        const int op = pg.dev_node(nb), on = pg.dev_node(nb + 1), ip = pg.dev_node(nb + 2);
        const int in = pg.dev_node(nb + 3);
        const double gm = param(pg, w, pb, 0);
        ST_G(op, ip, -gm); ST_G(op, in, gm); ST_G(on, ip, gm); ST_G(on, in, -gm);
    } break;
    case CB200_DEV_CCVS: {
        const double rm = param(pg, w, pb, 0);
        if (flags == 0) {                            // devices.jl:824-849
            const int op = pg.dev_node(nb), on = pg.dev_node(nb + 1), ip = pg.dev_node(nb + 2);
            const int in = pg.dev_node(nb + 3), Iin = pg.dev_node(nb + 4), Iout = pg.dev_node(nb + 5);
            ST_G(ip, Iin, 1.0); ST_G(in, Iin, -1.0); ST_G(Iin, ip, 1.0); ST_G(Iin, in, -1.0);
            ST_G(op, Iout, 1.0); ST_G(on, Iout, -1.0); ST_G(Iout, op, 1.0); ST_G(Iout, on, -1.0);
            ST_G(Iout, Iin, -rm);
        } else {                                     // devices.jl:898-913
            const int op = pg.dev_node(nb), on = pg.dev_node(nb + 1), Iin = pg.dev_node(nb + 2);
            const int Iout = pg.dev_node(nb + 3);
            ST_G(op, Iout, 1.0); ST_G(on, Iout, -1.0); ST_G(Iout, op, 1.0); ST_G(Iout, on, -1.0);
            ST_G(Iout, Iin, -rm);
        }
    } break;
    case CB200_DEV_CCCS: {
        const double A = param(pg, w, pb, 0);
        if (flags == 0) {                            // devices.jl:865-881
            const int op = pg.dev_node(nb), on = pg.dev_node(nb + 1), ip = pg.dev_node(nb + 2);
            const int in = pg.dev_node(nb + 3), Iin = pg.dev_node(nb + 4);
            ST_G(ip, Iin, 1.0); ST_G(in, Iin, -1.0); ST_G(Iin, ip, 1.0); ST_G(Iin, in, -1.0);
            ST_G(op, Iin, -A); ST_G(on, Iin, A);
        } else {                                     // devices.jl:924-931
            const int op = pg.dev_node(nb), on = pg.dev_node(nb + 1), Iin = pg.dev_node(nb + 2);
            ST_G(op, Iin, -A); ST_G(on, Iin, A);
        }
    } break;
    case CB200_DEV_DIODE: {                          // devices.jl:1370-1428
        const int pp = pg.dev_node(nb), nn = pg.dev_node(nb + 1);
        if (flags & 1) {
            const int lim = pg.dev_node(nb + 2);
            ST_G(lim, lim, 1.0); ST_G(lim, pp, -1.0); ST_G(lim, nn, 1.0);
            if (PASS != 2) {
                const double V0 = xval(pg, w, pp) - xval(pg, w, nn);
                const double Is = param(pg, w, pb, 0), Vt = param(pg, w, pb, 1), nf = param(pg, w, pb, 2);
                const double nVt = nf * Vt;
                // limit!  devices.jl:1209-1234
                const double vcrit = param(pg, w, pb, 3);
                const double vold = w(pg.off_u() + lim - 1);
                const double wv = initjct ? (V0 - V0 + vcrit) : d_pnjlim(V0, vold, nVt, vcrit);
                w(pg.off_limw() + (lim - 1 - (pg.n() - pg.n_limits()))) = wv;     // record_limit_w!
                double I0, Gd;
                d_diode_iv(Is, nVt, wv, I0, Gd);
                // stamp_limited_companion!  devices.jl:1251-1258
                DY_G(pp, pp, Gd); DY_G(pp, nn, -Gd); DY_G(nn, pp, -Gd); DY_G(nn, nn, Gd);
                const double Ieq = I0 - Gd * wv;
                DY_B(pp, -Ieq); DY_B(nn, Ieq);
            }
        } else if (PASS != 2) {
            const double V0 = xval(pg, w, pp) - xval(pg, w, nn);
            const double Is = param(pg, w, pb, 0), Vt = param(pg, w, pb, 1), nf = param(pg, w, pb, 2);
            const double nVt = nf * Vt;
            const double expterm = d_exp(V0 / nVt);
            const double I0 = Is * (expterm - 1.0);
            const double Gd = Is / nVt * expterm;
            const double Ieq = I0 - Gd * V0;
            DY_G(pp, pp, Gd); DY_G(pp, nn, -Gd); DY_G(nn, pp, -Gd); DY_G(nn, nn, Gd);
            DY_B(pp, -Ieq); DY_B(nn, Ieq);
        }
    } break;
    case CB200_DEV_DIODECAP: {                       // devices.jl:1558-1602
        if (PASS != 2) {
            const int pp = pg.dev_node(nb), nn = pg.dev_node(nb + 1);
            const double V0 = xval(pg, w, pp) - xval(pg, w, nn);
            const double Is = param(pg, w, pb, 0), Vt = param(pg, w, pb, 1), nf = param(pg, w, pb, 2);
            const double nVt = nf * Vt;
            const double expterm = d_exp(V0 / nVt);
            const double I0 = Is * (expterm - 1.0);
            const double G = Is / nVt * expterm;
            const double Ieq = I0 - G * V0;
            DY_G(pp, pp, G); DY_G(pp, nn, -G); DY_G(nn, pp, -G); DY_G(nn, nn, G);
            DY_B(pp, -Ieq); DY_B(nn, Ieq);
            const double Cj = d_junction_cap(V0, param(pg, w, pb, 3), param(pg, w, pb, 4), param(pg, w, pb, 5));
            DY_C(pp, pp, Cj); DY_C(pp, nn, -Cj); DY_C(nn, pp, -Cj); DY_C(nn, nn, Cj);
        }
    } break;
    case CB200_DEV_SIMPLEMOS: {                      // devices.jl:1667-1749
        const int dd = pg.dev_node(nb), gg = pg.dev_node(nb + 1), ss = pg.dev_node(nb + 2);
        if (PASS != 2) {
            const double Vd = xval(pg, w, dd), Vg = xval(pg, w, gg), Vs = xval(pg, w, ss);
            const double Vgs = Vg - Vs, Vds = Vd - Vs;
            const double Vth = param(pg, w, pb, 0), K = param(pg, w, pb, 1), lambda = param(pg, w, pb, 2);
            double Ids, gm, gds;
            if (Vgs <= Vth) { Ids = 0.0; gm = 0.0; gds = 0.0; }
            else if (Vds <= Vgs - Vth) {
                Ids = K * ((Vgs - Vth) * Vds - Vds * Vds / 2);
                gm = K * Vds;
                gds = K * (Vgs - Vth - Vds);
            } else {
                Ids = K / 2 * ((Vgs - Vth) * (Vgs - Vth)) * (1 + lambda * Vds);
                gm = K * (Vgs - Vth) * (1 + lambda * Vds);
                gds = K / 2 * ((Vgs - Vth) * (Vgs - Vth)) * lambda;
            }
            const double Ieq = Ids - gm * Vgs - gds * Vds;
            DY_G(dd, dd, gds); DY_G(dd, gg, gm); DY_G(dd, ss, -(gds + gm));
            DY_G(ss, dd, -gds); DY_G(ss, gg, -gm); DY_G(ss, ss, gds + gm);
            DY_B(dd, -Ieq); DY_B(ss, Ieq);
        }
        if (PASS == 0) {
            const double Cgd = param(pg, w, pb, 3), Cgs = param(pg, w, pb, 4);
            ST_C(gg, gg, Cgs); ST_C(gg, ss, -Cgs); ST_C(ss, gg, -Cgs); ST_C(ss, ss, Cgs);
            ST_C(gg, gg, Cgd); ST_C(gg, dd, -Cgd); ST_C(dd, gg, -Cgd); ST_C(dd, dd, Cgd);
        }
    } break;
    case CB200_DEV_VA:                               // emitted Verilog-A module, flags = model index
        va_dispatch<PASS>(pg, w, d, flags, t, mode, initjct);
        break;
    default: break;
    }
}

// A static (generated) program supplies eval_all / eval_nonlinear / eval_sources and
// its LU type supplies assemble / factor_and_solve / apply_update as straight-line
// code (one statement per stamp, per matrix entry, per elimination update) emitted by
// specialize.cpp in exactly the order of the loops below.
template <typename PG, typename W>
__device__ __forceinline__ void eval_all(const PG &pg, W &w, double t, int mode, bool initjct)
{
    if constexpr (PG::kStatic) {
        PG::eval_all(w, t, mode, initjct);
        PG::accumulate(w);          // G(u), C(u) entry sums: what the static assemble() reads
    } else {
        for (int d = 0; d < pg.n_dev(); d++) eval_device<0>(pg, w, d, t, mode, initjct);
    }
}

// devices whose stamps depend on the iterate (every Newton iteration)
template <typename PG, typename W>
__device__ __forceinline__ void eval_nonlinear(const PG &pg, W &w, double t, int mode, bool initjct)
{
    if constexpr (PG::kStatic) {
        PG::eval_nonlinear(w, t, mode, initjct);
        PG::accumulate(w);
    } else {
        for (int q = 0; q < pg.n_nl(); q++) eval_device<1>(pg, w, pg.nl_list(q), t, mode, initjct);
    }
}

// value of independent source d at time t, and its b stamps (devices.jl:643-737)
template <typename PG, typename W>
__device__ __forceinline__ double device_source_value(const PG &pg, W &w, int d, double t, int mode)
{
    const int pb = pg.dev_param_ptr(d);
    return source_value(pg, w, pg.dev_flags(d), pb, pg.dev_param_ptr(d + 1) - pb, t, mode);
}

template <typename PG, typename W>
__device__ __forceinline__ void device_source_stamp(const PG &pg, W &w, int d, double v)
{
    const int nb = pg.dev_node_ptr(d);
    int b = pg.off_SB() + pg.dev_bbase(d);
    if (pg.dev_kind(d) == CB200_DEV_VSOURCE) {
        w(b) = v;                                  // stamp_b!(ctx, I_idx, v): I is never ground
    } else {
        const int pp = pg.dev_node(nb), nn = pg.dev_node(nb + 1);
        if (pp != 0) { w(b) = v; b++; }
        if (nn != 0) { w(b) = -v; b++; }
    }
}

// One source, fixed-step mode.  When every parameter of the source is uniform over the
// sweep, its value at step k is the same in all lanes: each lane of the warp then
// evaluates ONE of the next 32 time points (t_{k+lane}) and the values are handed out
// by warp shuffle, one per step -- the waveform (fmod/sin/exp ...) costs 1/32 of an
// evaluation per step instead of one.  Bit-identical to evaluating in place: the same
// instructions run on the same inputs, in another lane.
template <typename PG, typename W>
__device__ __forceinline__ void source_step_one(const PG &pg, W &w, int q, int d, bool uniform,
                                                int64_t k, bool first, double t0, double h, int mode)
{
    double v;
    if (uniform) {
        const int j = (int)((k - 1) & 31);
        if (j == 0 || first)      // lane L holds the value of step (k - j) + L
            w(pg.off_srcc() + q) = device_source_value(pg, w, d, t0 + (double)((k - j) + (threadIdx.x & 31)) * h, mode);
        v = __shfl_sync(0xffffffffu, w(pg.off_srcc() + q), j);
    } else {
        v = device_source_value(pg, w, d, t0 + (double)k * h, mode);
    }
    device_source_stamp(pg, w, d, v);
}

template <typename PG, typename W>
__device__ __forceinline__ void eval_sources_step(const PG &pg, W &w, int64_t k, bool first, double t0,
                                                  double h, int mode)
{
    if constexpr (PG::kStatic) {
        PG::eval_sources_step(w, k, first, t0, h, mode);
    } else {
        for (int q = 0; q < pg.n_src(); q++)
            source_step_one(pg, w, q, pg.src_list(q), pg.src_uniform(q), k, first, t0, h, mode);
    }
}

// sources: stamps depend on time only (once per time step)
template <typename PG, typename W>
__device__ __forceinline__ void eval_sources(const PG &pg, W &w, double t, int mode)
{
    if constexpr (PG::kStatic) {
        PG::eval_sources(w, t, mode);
    } else {
        for (int q = 0; q < pg.n_src(); q++) eval_device<2>(pg, w, pg.src_list(q), t, mode, false);
    }
}

// ---------------------------------------------------------------------------
// assembly (deterministic segmented reduction) fused with the residual
//   F = C*du + G*u - b      (fast_residual!, precompile.jl:546-557; DC: F = G*u - b)
// and the Jacobian scatter  J = G + gamma*C  (fast_jacobian!, :568-585) straight into
// the LU workspace.  Also applies srcFact / gshunt (fast_rebuild!, :517-534).
// Returns ||F||_2^2; bad is set when F has a non-finite entry.
// ---------------------------------------------------------------------------
template <bool TRAN, typename PG, typename LU, typename W>
__device__ __forceinline__ double assemble(const PG &pg, const LU &lu, W &w, double gamma,
                                           double gshunt, double srcFact, bool &bad)
{
    if constexpr (PG::kStatic) return LU::template assemble<TRAN>(w, gamma, gshunt, srcFact, bad);
    for (int r = 0; r < pg.n(); r++) w(pg.off_F() + r) = 0.0;
    for (int q = 0; q < lu.n_fill(); q++) w(pg.off_LU() + lu.fill_slot(q)) = 0.0;
    for (int j = 0; j < pg.n(); j++) {
        const double uj = w(pg.off_u() + j);
        double duj = 0.0;
        if (TRAN) duj = gamma * (uj - w(pg.off_un() + j)) + w(pg.off_dterm() + j);
        const int s1 = pg.colptr(j + 1);
            for (int s = pg.colptr(j); s < s1; s++) {
            double gsum = 0.0;
            const int g1 = pg.gseg_ptr(s + 1);
                    for (int q = pg.gseg_ptr(s); q < g1; q++) gsum += w(pg.off_SG() + pg.gseg_idx(q));
            if (gshunt != 0.0 && pg.nz_is_node_diag(s)) gsum += gshunt;
            double jv = gsum;
            const int r = pg.rowval(s);
            double f = w(pg.off_F() + r);
            if (TRAN) {
                double csum = 0.0;
                const int c1 = pg.cseg_ptr(s + 1);
                            for (int q = pg.cseg_ptr(s); q < c1; q++) csum += w(pg.off_SC() + pg.cseg_idx(q));
                f += csum * duj;
                jv += gamma * csum;
            }
            f += gsum * uj;
            w(pg.off_F() + r) = f;
            w(pg.off_LU() + lu.jmap(s)) = jv;
        }
    }
    double nrm2 = 0.0;
    bad = false;
    for (int r = 0; r < pg.n(); r++) {
        double bsum = 0.0;
        const int b1 = pg.bseg_ptr(r + 1);
            for (int q = pg.bseg_ptr(r); q < b1; q++) bsum += w(pg.off_SB() + pg.bseg_idx(q));
        if (srcFact < 1.0) bsum *= srcFact;
        const double f = w(pg.off_F() + r) - bsum;
        w(pg.off_F() + r) = f;
        nrm2 += f * f;
    }
    bad = !isfinite(nrm2);     // a NaN / Inf entry of F poisons the sum (all(isfinite, F), solve.jl:632)
    return nrm2;
}

// ---------------------------------------------------------------------------
// numeric refactor on the fixed pattern with the host's static pivot order, then
// the triangular solves.  delta (in pivot coordinates) ends up in the wv slots.
// Returns false when a pivot vanished or the solution is non-finite.
// ---------------------------------------------------------------------------
template <typename PG, typename LU, typename W>
__device__ __forceinline__ bool factor_and_solve(const PG &pg, const LU &lu, W &w, bool &singular)
{
    if constexpr (PG::kStatic) return LU::factor_and_solve(w, singular);
    singular = false;
    for (int k = 0; k < lu.n(); k++) {
        const int ds = pg.off_LU() + lu.diag_slot(k);
        const double dgl = w(ds);
        if (!(fabs(dgl) >= DBL_MIN) || !isfinite(dgl)) singular = true;
        const double inv = 1.0 / dgl;
        w(ds) = inv;
        const int l0 = lu.Lptr(k), l1 = lu.Lptr(k + 1);
        const int u0 = lu.Uptr(k), u1 = lu.Uptr(k + 1);
        const int t0 = lu.tgt_ptr(k);
            for (int e = l0; e < l1; e++) {
            const int ls = pg.off_LU() + lu.L_slot(e);
            const double l = w(ls) * inv;
            w(ls) = l;
            w.weak |= weak_pivot(l);
                    for (int q = u0; q < u1; q++) {
                const int ts = pg.off_LU() + lu.tgt(t0 + (e - l0) * (u1 - u0) + (q - u0));
                w(ts) = w(ts) - l * w(pg.off_LU() + lu.U_slot(q));
            }
        }
    }
    // forward: z = L^-1 P F
    for (int k = 0; k < lu.n(); k++) w(pg.off_wv() + k) = w(pg.off_F() + lu.rowperm(k));
    for (int k = 0; k < lu.n(); k++) {
        const double zk = w(pg.off_wv() + k);
        const int l1 = lu.Lptr(k + 1);
            for (int e = lu.Lptr(k); e < l1; e++) {
            const int i = pg.off_wv() + lu.L_row(e);
            w(i) = w(i) - w(pg.off_LU() + lu.L_slot(e)) * zk;
        }
    }
    // backward: y = U^-1 z
    bool finite = true;
    for (int kk = 0; kk < lu.n(); kk++) {
        const int k = lu.n() - 1 - kk;
        double acc = w(pg.off_wv() + k);
        const int u1 = lu.Uptr(k + 1);
            for (int q = lu.Uptr(k); q < u1; q++)
            acc -= w(pg.off_LU() + lu.U_slot(q)) * w(pg.off_wv() + lu.U_col(q));
        acc *= w(pg.off_LU() + lu.diag_slot(k));
        w(pg.off_wv() + k) = acc;
        finite &= isfinite(acc);
    }
    return finite && !singular;
}

// u[colperm[k]] -= delta[k]
template <typename PG, typename LU, typename W>
__device__ __forceinline__ void apply_update(const PG &pg, const LU &lu, W &w)
{
    if constexpr (PG::kStatic) { LU::apply_update(w); return; }
    for (int k = 0; k < lu.n(); k++) {
        const int j = pg.off_u() + lu.colperm(k);
        w(j) = w(j) - w(pg.off_wv() + k);
    }
}

template <typename PG, typename W>
__device__ __forceinline__ void load_lane_params(const PG &pg, W &w, const double *lanes, int64_t P,
                                                 int64_t lane)
{
    CB_UNROLL
    for (int c = 0; c < pg.n_lane_cols(); c++) w(pg.off_lp() + c) = lanes[(int64_t)c * P + lane];
}

// ---------------------------------------------------------------------------
// DC body: _dc_pcnr_newton (solve.jl:599-698) and the plain-Newton restatement of
// _dc_newton_compiled (solve.jl:542-578), one lane per thread, masked lanes.
// ---------------------------------------------------------------------------
template <typename PG, typename LU, typename W>
__device__ __forceinline__ void dc_body(const PG &pg, const LU &lu, W &w, const Program &p,
                                        const SpecArgs &sp, const DcArgs &a)
{
    const int64_t lane0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool in_range = lane0 < p.P;
    const int64_t lane = in_range ? lane0 : p.P - 1;      // clamp: compute, never commit
    const bool act = in_range && (a.active == nullptr || a.active[lane]);

    load_lane_params(pg, w, p.lanes, p.P, lane);
    bool cold = true;
    CB_UNROLL
    for (int i = 0; i < pg.n(); i++) {
        const double v = a.u[(int64_t)i * p.P + lane];
        w(pg.off_u() + i) = v;
        cold &= (v == 0.0);
    }
    const double gshunt = a.gshunt_lane ? a.gshunt_lane[lane] : sp.gshunt;
    const double srcFact = a.srcfact_lane ? a.srcfact_lane[lane] : sp.srcFact;
    const int lim0 = pg.n() - pg.n_limits();
    const bool pcnr = (a.algorithm == 0);
    const double abstol2 = a.abstol * a.abstol;     // ||F||_2 < abstol  <=>  ||F||_2^2 < abstol^2
    bool initjct = false;
    if (pcnr && cold) {                                   // solve.jl:622-627
        CB_UNROLL
        for (int k = 0; k < pg.n_limits(); k++) {
            const int r = pg.limit_init_ref(k);
            w(pg.off_u() + lim0 + k) = r >= 0 ? pg.uniform(r) : w(pg.off_lp() + ~r);
        }
        initjct = true;
    }
    eval_all(pg, w, a.t, sp.mode, false);                 // static stamps + sources (t fixed)

    bool done = !act;
    bool settling = false;
    int status = CB200_LANE_MAXITER, solves = 0, iter = 0;
    bool conv = false;
    while (true) {
        if (__all_sync(0xffffffffu, done)) break;
        if (!settling) iter++;
        // loop bound: PCNR `for iter in 1:maxiters`; Newton: maxiters solves then a final test
        const int bound = pcnr ? a.maxiters : a.maxiters + 1;
        if (!done && iter > bound) { done = true; status = CB200_LANE_MAXITER; }
        eval_nonlinear(pg, w, a.t, sp.mode, initjct);
        initjct = false;
        bool bad;
        const double nrm2 = assemble<false>(pg, lu, w, 0.0, gshunt, srcFact, bad);
        if (done) continue;
        if (bad) { done = true; status = CB200_LANE_NONFINITE; continue; }
        if (nrm2 < abstol2) {
            if (!pcnr || settling) { done = true; conv = true; status = CB200_LANE_OK; continue; }
            // settle the limit slots and re-verify (solve.jl:640-663)
            CB_UNROLL
            for (int k = 0; k < pg.n_limits(); k++) w(pg.off_u() + lim0 + k) = w(pg.off_limw() + k);
            settling = true;
            continue;
        }
        settling = false;
        if (!pcnr && iter > a.maxiters) { done = true; status = CB200_LANE_MAXITER; continue; }
        bool singular;
        const bool ok = factor_and_solve(pg, lu, w, singular);
        if (!ok) { done = true; status = singular ? CB200_LANE_SINGULAR : CB200_LANE_NONFINITE; continue; }
        apply_update(pg, lu, w);
        solves++;
        if (pcnr) {                                         // CORRECT  solve.jl:686-689
            CB_UNROLL
            for (int k = 0; k < pg.n_limits(); k++) w(pg.off_u() + lim0 + k) = w(pg.off_limw() + k);
        }
    }
    if (act) {
        CB_UNROLL
        for (int i = 0; i < pg.n(); i++) a.u[(int64_t)i * p.P + lane] = w(pg.off_u() + i);
        a.status[lane] = status;
        if (a.weak && w.weak) a.weak[lane] = 1;
        a.iters[lane] += solves;
        a.converged[lane] = conv ? 1 : 0;
    }
}

// ---------------------------------------------------------------------------
// DC continuation on the device: _gshunt_stepping (solve.jl:720-783) then _source_stepping
// (:805-850) for the lanes tiers 0-1 left unconverged (DcArgs.algorithm == 2).  The per-lane
// controller below is the reference's loop turned inside out: the kernel runs ONE flat loop of
// Newton iterations (_dc_newton_compiled: at most maxiters solves, then a final test) and the
// controller is told the outcome of every inner solve; it answers with the next (gshunt,
// srcFact) and whether the lane restarts from its saved state.  No state leaves the device
// between continuation steps.
// ---------------------------------------------------------------------------
struct StepCtl {
    int phase;                 // 0 gshunt ramp, 1 final solve at the exact target, 2 source ramp, 3 finished
    double cur, factor, target, thr;
    double sf, sf_conv, raise;
    int steps;                 // inner solves of the current ramp (max 20 / 50)
    bool conv;
    __device__ __forceinline__ void begin(double target_gshunt)
    {
        phase = 0; cur = 1e-3; factor = 10.0; target = target_gshunt;
        thr = target > 1e-12 ? target : 1e-12;
        sf = 0.0; sf_conv = 0.0; raise = 0.1; steps = 0; conv = false;
    }
    __device__ __forceinline__ double gshunt() const { return phase == 0 ? cur : target; }
    __device__ __forceinline__ double srcfact(double spec_srcfact) const { return phase == 2 ? sf : spec_srcfact; }
    // outcome of one inner solve; returns what the lane state must become: 0 keep u (and save it),
    // 1 restore the saved state, 2 restart from zeros (source stepping begins), 3 keep (finished)
    __device__ __forceinline__ int result(bool ok)
    {
        if (phase == 0) {
            steps++;
            if (ok) {
                if (cur <= thr) {
                    if (cur != target) { phase = 1; return 0; }
                    conv = true; phase = 3; return 3;
                }
                cur /= factor;
                if (cur < thr) cur = thr;
                if (steps >= 20) { start_source(); return 2; }
                return 0;
            }
            if (factor <= 1.5 || steps >= 20) { start_source(); return 2; }
            factor = sqrt(factor);
            return 1;
        }
        if (phase == 1) {
            if (ok) { conv = true; phase = 3; return 3; }
            start_source();
            return 2;
        }
        steps++;
        if (ok) {
            sf_conv = sf;
            if (sf >= 1.0) { conv = true; phase = 3; return 3; }
            sf = sf + raise < 1.0 ? sf + raise : 1.0;
            if (steps >= 50) { phase = 3; return 3; }
            return 0;
        }
        if (sf - sf_conv < 1e-6 || steps >= 50) { phase = 3; return 1; }
        raise /= 2.0;
        sf = sf_conv + raise;
        return 1;
    }
    __device__ __forceinline__ void start_source() { phase = 2; sf = 0.0; sf_conv = 0.0; raise = 0.1; steps = 0; }
};

template <typename PG, typename LU, typename W>
__device__ __forceinline__ void dc_stepping_body(const PG &pg, const LU &lu, W &w, const Program &p,
                                                 const SpecArgs &sp, const DcArgs &a)
{
    const int64_t lane0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool in_range = lane0 < p.P;
    const int64_t lane = in_range ? lane0 : p.P - 1;
    const bool act = in_range && (a.active == nullptr || a.active[lane]);

    load_lane_params(pg, w, p.lanes, p.P, lane);
    for (int i = 0; i < pg.n(); i++) { w(pg.off_u() + i) = 0.0; w(pg.off_h1() + i) = 0.0; }   // both tiers start from zeros
    eval_all(pg, w, a.t, sp.mode, false);
    StepCtl ctl;
    ctl.begin(sp.gshunt);
    if (a.algorithm == 3) ctl.start_source();
    const double abstol2 = a.abstol * a.abstol;
    int iter = 0, solves = 0;
    bool fin = !act;
    while (true) {
        if (__all_sync(0xffffffffu, fin)) break;
        eval_nonlinear(pg, w, a.t, sp.mode, false);
        bool bad;
        const double nrm2 = assemble<false>(pg, lu, w, 0.0, ctl.gshunt(), ctl.srcfact(sp.srcFact), bad);
        if (fin) continue;
        int res = -1;                                       // -1: the inner solve goes on
        if (bad) res = 0;
        else if (nrm2 < abstol2) res = 1;
        else if (iter == a.maxiters) res = 0;
        else {
            bool singular;
            if (!factor_and_solve(pg, lu, w, singular)) res = 0;
            else { apply_update(pg, lu, w); solves++; iter++; }
        }
        if (res < 0) continue;
        iter = 0;
        const int act_on = ctl.result(res == 1);
        if (act_on == 0) { for (int i = 0; i < pg.n(); i++) w(pg.off_h1() + i) = w(pg.off_u() + i); }
        else if (act_on == 1) { for (int i = 0; i < pg.n(); i++) w(pg.off_u() + i) = w(pg.off_h1() + i); }
        else if (act_on == 2) { for (int i = 0; i < pg.n(); i++) { w(pg.off_u() + i) = 0.0; w(pg.off_h1() + i) = 0.0; } }
        if (ctl.phase == 3) fin = true;
    }
    if (act) {
        for (int i = 0; i < pg.n(); i++) a.u[(int64_t)i * p.P + lane] = w(pg.off_u() + i);
        a.status[lane] = ctl.conv ? CB200_LANE_OK : CB200_LANE_MAXITER;
        if (a.weak && w.weak) a.weak[lane] = 1;
        a.iters[lane] += solves;
        a.converged[lane] = ctl.conv ? 1 : 0;
    }
}

// ---------------------------------------------------------------------------
// Newton iteration of one implicit step (both transient bodies), from the predictor in u: rebuild,
// F, stop when ||F||_2 < abstol, otherwise solve J delta = F and update; at most max_nl solves.
// Masked: a lane that is done (`done` on entry: a lane that has finished its time loop) keeps its
// state but still takes part in the warp's evaluations, solves and votes.
// `limit` (CB200_TRAN_LIMIT): a step the plain iteration does not finish in max_nl solves is redone
// from u_n with the PCNR corrector after every solve (4*max_nl solves allowed); lim_on reports it.
// Returns the CB200_LANE_* status of the step.  Counts solves and evaluation passes; `fresh`: see
// tran_fixed_body.
// ---------------------------------------------------------------------------
template <typename PG, typename LU, typename W>
__device__ __forceinline__ int newton_step(const PG &pg, const LU &lu, W &w, const SpecArgs &sp, bool done,
                                           double t, double gamma, double abstol2, int max_nl, int limit,
                                           int &solves, int &evals, bool &fresh, bool &lim_on)
{
    int st = CB200_LANE_OK;
    lim_on = false;
    int it0 = 0;
    for (int it = 0;; it++) {
        // lanes that are fresh recompute identical values when another lane of the warp is not
        if (__any_sync(0xffffffffu, kNlTimeDep || !fresh)) { eval_nonlinear(pg, w, t, CB200_MODE_TRAN, false); evals++; }
        fresh = true;
        bool bad;
        const double nrm2 = assemble<true>(pg, lu, w, gamma, sp.gshunt, sp.srcFact, bad);
        bool restart = false;
        if (!done) {
            if (bad) { done = true; st = CB200_LANE_NONFINITE; }
            else if (nrm2 < abstol2) { done = true; }
            else if (it - it0 >= (lim_on ? 4 * max_nl : max_nl)) {
                if (PG::kTranLimit && limit && !lim_on) { lim_on = true; it0 = it + 1; restart = true; }
                else { done = true; st = CB200_LANE_MAXITER; }
            }
        }
        if (__all_sync(0xffffffffu, done)) break;
        bool singular;
        const bool ok = factor_and_solve(pg, lu, w, singular);
        if (!done) {
            if (restart) {                             // redo the step from u_n, limiting on
                CB_UNROLL
                for (int i = 0; i < pg.n(); i++) w(pg.off_u() + i) = w(pg.off_un() + i);
                fresh = false;
            } else if (!ok) { done = true; st = singular ? CB200_LANE_SINGULAR : CB200_LANE_NONFINITE; }
            else {
                apply_update(pg, lu, w);
                fresh = false;
                solves++;
                if (lim_on) {                          // PCNR corrector, solve.jl:686-689
                    const int lim0 = pg.n() - pg.n_limits();
                    CB_UNROLL
                    for (int q = 0; q < pg.n_limits(); q++) w(pg.off_u() + lim0 + q) = w(pg.off_limw() + q);
                }
            }
        }
    }
    return st;
}

// ---------------------------------------------------------------------------
// fixed-step transient body: the whole time loop of a lane on the device.
//   du = gamma*(u - u_n) + dterm
//   BE:    gamma = 1/h,      dterm = 0
//   trap:  gamma = 2/h,      dterm = -du_n                      (first step BE)
//   Gear2: gamma = 3/(2h),   dterm = -(u_n - u_{n-1})/(2h)      (first step BE)
// Newton per step from u = u_n (newton_step).  t_k = t0 + k*h.
// ---------------------------------------------------------------------------
template <typename PG, typename LU, typename W>
__device__ __forceinline__ void tran_fixed_body(const PG &pg, const LU &lu, W &w, const Program &p,
                                                const SpecArgs &sp, const TranArgs &a)
{
    const int64_t lane0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool act = lane0 < p.P;
    const int64_t lane = act ? lane0 : p.P - 1;

    // The time loop may be cut into segments [k_begin, k_end] (one launch each) so that the
    // copy of a finished segment's waveform to the host overlaps the next segment's compute;
    // a resumed segment reloads the integrator history (u_n, dterm) the previous one stored.
    const bool resume = a.k_begin > 1;
    load_lane_params(pg, w, p.lanes, p.P, lane);
    CB_UNROLL
    for (int i = 0; i < pg.n(); i++) {
        w(pg.off_u() + i) = a.u[(int64_t)i * p.P + lane];
        w(pg.off_dterm() + i) = resume ? a.hist[(int64_t)(pg.n() + i) * p.P + lane] : 0.0;
        w(pg.off_un() + i) = resume ? a.hist[(int64_t)i * p.P + lane] : 0.0;
    }
    eval_all(pg, w, a.t0, CB200_MODE_TRAN, false);

    int status = a.status[lane], solves = 0;       // keeps an InitialFailure from the DC init
    int evals = 0;                                 // device-model evaluation passes this thread executed
    int64_t tp = a.tp_begin;
    if (!resume) {
        if (act)
            for (int q = 0; q < a.n_save; q++)
                a.out[((int64_t)q * a.T + tp) * p.P + lane] = read_u(pg, w, __ldg(a.save_idx + q));
        tp++;
    }
    const double h = a.h;
    const double abstol2 = a.abstol * a.abstol;
    // a specialised kernel is generated for one integration method: branches on it fold
    const int amethod = PG::kMethod >= 0 ? PG::kMethod : a.method;
    // `fresh`: the stamp slots of the nonlinear devices hold their values AT the current iterate.
    // A step that converged ends with an evaluation at its final u, and the next step starts its
    // Newton iteration from that same u: G(u), C(u) and the companion currents are functions of
    // u alone, so the first residual of a step re-assembles them with the new source values and
    // history terms instead of evaluating every device model again for identical values.
    bool fresh = false;
    // Quiescent-step bypass (PG::kBypass, backward Euler; a generated program knows its source stamp slots at
    // compile time).  `quiet`: the previous step of this lane converged at its first residual -- no solve, so
    // u == u_n, d == 0 and the stamps are those of u.  If in addition every source stamp of the new step is
    // bitwise what it was, the new step's first residual F = G u - b is bit for bit the one that just passed
    // the test: the step would assemble the same numbers, find them converged and change nothing.  When that
    // holds for all 32 lanes of the warp the step is not executed (its saved point is written from the
    // unchanged u).  Identical waveforms, statuses and Newton counts by construction; a lane that could not
    // skip alone executes the step as usual.
    bool quiet = false;
    int nexec = 0;                                 // steps this lane executed (not bypassed)
    for (int64_t k = a.k_begin; k <= a.k_end; k++) {
        const double t = a.t0 + (double)k * h;
        const int method = (k == 1) ? CB200_METHOD_BE : amethod;
        const double gamma = method == CB200_METHOD_BE ? 1.0 / h
                           : method == CB200_METHOD_TRAP ? 2.0 / h : 3.0 / (2.0 * h);
        if constexpr (PG::kBypass) {
            double src_old[PG::kSrcSlots > 0 ? PG::kSrcSlots : 1];
            PG::src_snapshot(w, src_old);
            eval_sources_step(pg, w, k, k == a.k_begin, a.t0, h, CB200_MODE_TRAN);
            if (PG::kMethod == CB200_METHOD_BE && !kNlTimeDep) {
                if (__all_sync(0xffffffffu, PG::src_same(w, src_old, quiet && k != a.k_begin))) {
                    if (k % a.save_every == 0 || k == a.nsteps) {
                        if (act)
                            for (int q = 0; q < a.n_save; q++)
                                a.out[((int64_t)q * a.T + tp) * p.P + lane] = read_u(pg, w, __ldg(a.save_idx + q));
                        tp++;
                    }
                    continue;
                }
            }
            nexec++;
        }
        // history terms; un <- u
        CB_UNROLL
        for (int i = 0; i < pg.n(); i++) {
            const double ui = w(pg.off_u() + i);
            if (method == CB200_METHOD_GEAR2) w(pg.off_dterm() + i) = -(ui - w(pg.off_un() + i)) / (2.0 * h);
            else if (method == CB200_METHOD_BE) w(pg.off_dterm() + i) = 0.0;
            /* trap: dterm already holds -du_n */
            w(pg.off_un() + i) = ui;
        }
        // with the bypass the sources were evaluated above, where it tests them; both orders give the same
        // results, and here the table-driven kernels keep the register allocation they were measured with
        if constexpr (!PG::kBypass) eval_sources_step(pg, w, k, k == a.k_begin, a.t0, h, CB200_MODE_TRAN);
        const int solves0 = solves;
        bool lim_on;
        const int st = newton_step(pg, lu, w, sp, false, t, gamma, abstol2, a.max_nl, a.limit, solves, evals, fresh,
                                   lim_on);
        quiet = st == CB200_LANE_OK && solves == solves0 && !lim_on;
        if (st != CB200_LANE_OK && status == CB200_LANE_OK) status = st;
        if (st != CB200_LANE_OK) fresh = false;           // the last evaluation was not at the state kept
        if (st == CB200_LANE_NONFINITE || st == CB200_LANE_SINGULAR) {  // dead lane: hold last state
            CB_UNROLL
            for (int i = 0; i < pg.n(); i++) w(pg.off_u() + i) = w(pg.off_un() + i);
        }
        if (amethod == CB200_METHOD_TRAP) {               // dterm <- -du_{n+1}
            CB_UNROLL
            for (int i = 0; i < pg.n(); i++)
                w(pg.off_dterm() + i) = -(gamma * (w(pg.off_u() + i) - w(pg.off_un() + i)) + w(pg.off_dterm() + i));
        }
        if (k % a.save_every == 0 || k == a.nsteps) {
            if (act)
                for (int q = 0; q < a.n_save; q++)
                    a.out[((int64_t)q * a.T + tp) * p.P + lane] = read_u(pg, w, __ldg(a.save_idx + q));
            tp++;
        }
    }
    if (act) {
        CB_UNROLL
        for (int i = 0; i < pg.n(); i++) {
            a.u[(int64_t)i * p.P + lane] = w(pg.off_u() + i);
            if (a.hist != nullptr) {                     // history for a resumed segment
                a.hist[(int64_t)i * p.P + lane] = w(pg.off_un() + i);
                a.hist[(int64_t)(pg.n() + i) * p.P + lane] = w(pg.off_dterm() + i);
            }
        }
        a.status[lane] = status;
        if (a.weak && w.weak) a.weak[lane] = 1;
        a.iters[lane] += solves;
        if (a.evals != nullptr) a.evals[lane] += evals;
        if constexpr (PG::kBypass) PG::count_steps(nexec);
    }
}

// ---------------------------------------------------------------------------
// adaptive transient body: trapezoidal (or BE) integration with LTE step control, one
// private time axis per lane, masked lanes.  Stand-in for the reference's third-party
// variable-step integrators (IDA / OrdinaryDiffEq; sweeps.jl:599-601, :650, :664):
//  - tstops (source breakpoints, solve.jl:1847-1918) are hit exactly and restart the
//    integrator (BE step, fresh history);
//  - error estimate = scaled corrector-minus-predictor difference, linear predictor
//    while only two points are known (order 1), quadratic afterwards (order 2);
//  - weighted RMS norm with lte_abstol + reltol*max(|u|, |u_n|); accept when <= 1;
//  - h_new = h * clamp(0.9 * err^(-1/(p+1)), 0.2, 2); Newton failure: h /= 4;
//    h < dtmin ends the lane with CB200_LANE_DTMIN.
// The same statement is the oracle's (oracle/cadnip_oracle.c: ora__tran_adaptive).
// ---------------------------------------------------------------------------
// absolute tolerance of unknown i in the LTE test: state_abstol (build.jl:276-283)
__device__ __forceinline__ double lte_atol(const AdaptArgs &a, int i)
{
    return i < a.cls_i0 ? a.tol_v : i < a.cls_q0 ? a.tol_i : i < a.cls_l0 ? a.tol_q : a.tol_v;
}

// ---------------------------------------------------------------------------
// Variable-order, variable-step BDF (orders 1..5), fixed-leading-coefficient form: the integrator
// family of the reference's default Sundials.IDA (sweeps.jl:599-601).  Scalar state of one lane;
// the modified divided differences phi[0..5] live in the lane workspace (off_phi + j n).
// Restated from the published algorithm (Brenan / Campbell / Petzold ch. 5; SUNDIALS, ACM TOMS 31):
// coefficient recurrences, error estimates at orders k-2 .. k+1, order / step selection, failure
// rules.  Statement for statement the oracle's (oracle/cadnip_oracle.c: ora_bdf, tran_bdf).
// ---------------------------------------------------------------------------
constexpr int kBdfMaxOrd = 5;
struct Bdf {
    int kk, kused, knew, ns, phase, nef;
    double hused, cj, ck;
    double est, terk, terkm1, erkm1, erkp1;                // of the last error test
    double psi[kBdfMaxOrd + 1], alpha[kBdfMaxOrd + 1], beta[kBdfMaxOrd + 1];
    double sigma[kBdfMaxOrd + 1], gam[kBdfMaxOrd + 1];

    __device__ __forceinline__ void restart(double hh)
    {
        kk = 1; kused = 0; knew = 1; ns = 0; phase = 0; nef = 0; hused = 0.0; cj = 1.0 / hh; ck = 1.0;
        est = terk = terkm1 = erkm1 = erkp1 = 0.0;
        for (int i = 0; i <= kBdfMaxOrd; i++) { psi[i] = hh; alpha[i] = beta[i] = sigma[i] = gam[i] = 0.0; }
    }
    // IDASetCoeffs
    __device__ __forceinline__ void set_coeffs(double hh)
    {
        if (hh != hused || kk != kused) ns = 0;
        ns = ns + 1 < kused + 2 ? ns + 1 : kused + 2;
        if (kk + 1 >= ns) {
            beta[0] = 1.0; alpha[0] = 1.0; gam[0] = 0.0; sigma[0] = 1.0;
            double temp1 = hh;
            for (int i = 1; i <= kk; i++) {
                const double temp2 = psi[i - 1];
                psi[i - 1] = temp1;
                beta[i] = beta[i - 1] * psi[i - 1] / temp2;
                temp1 = temp2 + hh;
                alpha[i] = hh / temp1;
                sigma[i] = (double)i * sigma[i - 1] * alpha[i];
                gam[i] = gam[i - 1] + alpha[i - 1] / hh;
            }
            psi[kk] = temp1;
        }
        double alphas = 0.0, alpha0 = 0.0;
        for (int i = 0; i < kk; i++) { alphas -= 1.0 / (double)(i + 1); alpha0 -= alpha[i]; }
        cj = -alphas / hh;
        ck = fabs(alpha[kk] + alphas - alpha0);
        if (ck < alpha[kk]) ck = alpha[kk];
    }
    // IDARestore (the phi are un-scaled by the caller)
    __device__ __forceinline__ void restore(double hh)
    {
        for (int j = 1; j <= kk; j++) psi[j - 1] = psi[j] - hh;
    }
    // IDATestError from the four sums of squares: |ee|, |ee + phi[k]|, |ee + phi[k] + phi[k-1]|, |ee - phi[k+1]|
    // (each already divided by the weights); true = the step fails the error test
    __device__ __forceinline__ bool test(double a0, double a1, double a2, double ap, int n)
    {
        const double enorm = sqrt(a0 / (double)n);
        const double erk = sigma[kk] * enorm;
        terk = (double)(kk + 1) * erk;
        est = erk; knew = kk;
        terkm1 = 0.0; erkm1 = 0.0;
        if (kk > 1) {
            erkm1 = sigma[kk - 1] * sqrt(a1 / (double)n);
            terkm1 = (double)kk * erkm1;
            if (kk > 2) {
                const double erkm2 = sigma[kk - 2] * sqrt(a2 / (double)n);
                const double terkm2 = (double)(kk - 1) * erkm2;
                if (fmax(terkm1, terkm2) <= terk) { knew = kk - 1; est = erkm1; }
            } else if (terkm1 <= 0.5 * terk) { knew = kk - 1; est = erkm1; }
        }
        erkp1 = sqrt(ap / (double)n) / (double)(kk + 2);
        return ck * enorm > 1.0;
    }
    // IDAHandleNFlag after an error-test failure: new order and step
    __device__ __forceinline__ double after_error_fail(double hh)
    {
        nef++;
        if (nef == 1) {
            kk = knew;
            double rr = 0.9 * pow(2.0 * est + 0.0001, -1.0 / (double)(kk + 1));
            rr = fmax(0.25, fmin(0.9, rr));
            return hh * rr;
        }
        if (nef == 2) { kk = knew; return hh * 0.25; }
        kk = 1;
        return hh * 0.25;
    }
    // IDACompleteStep (scalar part): order of the next step and its size; `kdone` = order just used
    __device__ __forceinline__ double complete(double hh)
    {
        const int kdone = kk;
        const int kdiff = kdone - kused;
        kused = kdone; hused = hh; nef = 0;
        if (knew == kdone - 1 || kdone == kBdfMaxOrd) phase = 1;
        if (phase == 0) { kk = kdone + 1; return 2.0 * hh; }
        int action;                                        // -1 lower, 0 maintain, +1 raise
        if (knew == kdone - 1) action = -1;
        else if (kdone == kBdfMaxOrd) action = 0;
        else if (kdone + 1 >= ns || kdiff == 1) action = 0;
        else {
            const double terkp1 = (double)(kdone + 2) * erkp1;
            if (kdone == 1) action = terkp1 >= 0.5 * terk ? 0 : 1;
            else if (terkm1 <= fmin(terk, terkp1)) action = -1;
            else if (terkp1 >= terk) action = 0;
            else action = 1;
        }
        double e = est;
        if (action == 1) { kk = kdone + 1; e = erkp1; }
        else if (action == -1) { kk = kdone - 1; e = erkm1; }
        double hnew = hh;
        double rr = pow(2.0 * e + 0.0001, -1.0 / (double)(kk + 1));
        if (rr >= 2.0) hnew = 2.0 * hh;
        else if (rr <= 1.0) { rr = fmax(0.5, fmin(0.9, rr)); hnew = hh * rr; }
        return hnew;
    }
};

// one attempt begins: scale phi[ns..kk] by beta, predict (IDAPredict): un <- sum phi, dterm <- sum gam phi, u <- un
template <typename PG, typename W>
__device__ __forceinline__ void bdf_predict(const PG &pg, W &w, const Bdf &B)
{
    const int n = pg.n();
    #pragma unroll
    for (int j = 1; j <= kBdfMaxOrd; j++) {
        if (j >= B.ns && j <= B.kk) {
            const double bj = B.beta[j];
            CB_UNROLL
            for (int i = 0; i < n; i++) w(pg.off_phi() + j * n + i) *= bj;
        }
    }
    CB_UNROLL
    for (int i = 0; i < n; i++) {
        double yy = w(pg.off_phi() + i), yp = 0.0;
        #pragma unroll
        for (int j = 1; j <= kBdfMaxOrd; j++) {
            if (j <= B.kk) { const double f = w(pg.off_phi() + j * n + i); yy += f; yp = fma(B.gam[j], f, yp); }
        }
        w(pg.off_un() + i) = yy; w(pg.off_dterm() + i) = yp; w(pg.off_u() + i) = yy;
    }
}

// a failed attempt (Newton or error test): IDARestore; u <- phi[0] (the last accepted point)
// `reseed`: the first step after a (re)start failed its error test -- phi[1] = h y' was seeded with y' = 0; the
// failed solution gives the secant slope, phi[1] <- y_failed - y_0 (see the oracle, tran_bdf)
template <typename PG, typename W>
__device__ __forceinline__ void bdf_undo(const PG &pg, W &w, Bdf &B, double hh, bool reseed)
{
    const int n = pg.n();
    B.restore(hh);
    if (reseed) B.psi[0] = hh;                             // the step the reseeded phi[1] belongs to
    #pragma unroll
    for (int j = 1; j <= kBdfMaxOrd; j++) {
        if (j >= B.ns && j <= B.kk) {
            const double bj = B.beta[j];
            CB_UNROLL
            for (int i = 0; i < n; i++) w(pg.off_phi() + j * n + i) /= bj;
        }
    }
    CB_UNROLL
    for (int i = 0; i < n; i++) {
        const double y0 = w(pg.off_phi() + i);
        if (reseed) w(pg.off_phi() + n + i) = w(pg.off_u() + i) - y0;
        w(pg.off_u() + i) = y0;
    }
}

// phi[j] by run-time order with compile-time slot arithmetic (a specialised kernel's workspace is a register file)
template <typename PG, typename W>
__device__ __forceinline__ double bdf_phi(const PG &pg, W &w, int j, int i)
{
    const int n = pg.n();
    double v = 0.0;
    #pragma unroll
    for (int q = 0; q <= kBdfMaxOrd; q++) if (q == j) v = w(pg.off_phi() + q * n + i);
    return v;
}

template <typename PG, typename W>
__device__ __forceinline__ bool bdf_error_test(const PG &pg, W &w, const AdaptArgs &a, Bdf &B)
{
    const int n = pg.n(), kk = B.kk;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, ap = 0.0;
    CB_UNROLL
    for (int i = 0; i < n; i++) {
        const double ui = w(pg.off_u() + i), yi = w(pg.off_un() + i);
        const double tol = lte_atol(a, i) + a.reltol * fmax(fabs(ui), fabs(yi));
        const double ee = ui - yi;
        double e = ee / tol;
        a0 += e * e;
        if (kk > 1) {
            double d = ee + bdf_phi(pg, w, kk, i);
            e = d / tol; a1 += e * e;
            if (kk > 2) { d += bdf_phi(pg, w, kk - 1, i); e = d / tol; a2 += e * e; }
        }
        if (kk < kBdfMaxOrd) { e = (ee - bdf_phi(pg, w, kk + 1, i)) / tol; ap += e * e; }
    }
    return B.test(a0, a1, a2, ap, n);
}

// accepted step of order kdone: phi[kdone+1] = ee, phi[kdone] += ee, running sums downwards
template <typename PG, typename W>
__device__ __forceinline__ void bdf_advance(const PG &pg, W &w, int kdone)
{
    const int n = pg.n();
    CB_UNROLL
    for (int i = 0; i < n; i++) {
        const double ee = w(pg.off_u() + i) - w(pg.off_un() + i);
        double acc = ee;
        #pragma unroll
        for (int j = kBdfMaxOrd; j >= 0; j--) {
            if (j == kdone + 1) w(pg.off_phi() + j * n + i) = ee;
            else if (j <= kdone) { acc += w(pg.off_phi() + j * n + i); w(pg.off_phi() + j * n + i) = acc; }
        }
    }
}

template <typename PG, typename LU, typename W>
__device__ __forceinline__ void tran_adaptive_body(const PG &pg, const LU &lu, W &w, const Program &p,
                                                   const SpecArgs &sp, const AdaptArgs &a)
{
    const int64_t lane0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool act = lane0 < p.P;
    const int64_t lane = act ? lane0 : p.P - 1;

    load_lane_params(pg, w, p.lanes, p.P, lane);
    CB_UNROLL
    for (int i = 0; i < pg.n(); i++) {
        w(pg.off_u() + i) = a.u[(int64_t)i * p.P + lane];
        w(pg.off_dterm() + i) = 0.0;
        w(pg.off_un() + i) = 0.0;
        w(pg.off_h1() + i) = 0.0;
        w(pg.off_h2() + i) = 0.0;
    }
    eval_all(pg, w, a.t0, CB200_MODE_TRAN, false);

    int status = a.status[lane], solves = 0, rej = 0, T = 0, evals = 0;
    bool fresh = false;                                    // see tran_fixed_body
    if (act) {
        a.out_t[(int64_t)T * p.P + lane] = a.t0;
        for (int q = 0; q < a.n_save; q++)
            a.out[((int64_t)q * a.max_points + T) * p.P + lane] = read_u(pg, w, __ldg(a.save_idx + q));
    }
    T++;
    const int amethod = PG::kMethod >= 0 ? PG::kMethod : a.method;
    const bool bdf = amethod == CB200_METHOD_BDF;
    const double abstol2 = a.abstol * a.abstol;
    double t = a.t0, h = a.h0, h1 = 0.0, h2 = 0.0;
    int nhist = 0, istop = 0;
    bool finished = !(t < a.t1);
    Bdf B;
    if (bdf) B.restart(h);
    while (true) {
        if (__all_sync(0xffffffffu, finished)) break;
        // ---- choose the step
        while (istop < a.n_tstops && __ldg(a.tstops + istop) <= fma(4.440892098500626e-16, fabs(t), t)) istop++;   // 4 eps(t), either sign of t
        double tnext = istop < a.n_tstops ? __ldg(a.tstops + istop) : a.t1;
        if (tnext > a.t1) tnext = a.t1;
        double hh = h;
        bool hit = false;
        if (t + hh >= tnext - 1e-3 * hh) { hh = tnext - t; hit = true; }
        const double tn = hit ? tnext : t + hh;
        const bool be = (nhist == 0 || amethod == CB200_METHOD_BE);
        double gamma = be ? 1.0 / hh : 2.0 / hh;
        if (bdf) {
            if (!finished) {
                if (nhist == 0) {                          // (re)start: order 1, phi[0] = y, phi[1] = h y' = 0
                    B.restart(hh);
                    CB_UNROLL
                    for (int i = 0; i < pg.n(); i++) {
                        w(pg.off_phi() + i) = w(pg.off_u() + i);
                        #pragma unroll
                        for (int j = 1; j <= kBdfMaxOrd; j++) w(pg.off_phi() + j * pg.n() + i) = 0.0;
                    }
                    nhist = 1;
                }
                B.set_coeffs(hh);
                bdf_predict(pg, w, B);
                fresh = false;                             // the predictor is not the point last evaluated
            }
            gamma = B.cj;
        } else if (!finished) {
            CB_UNROLL
            for (int i = 0; i < pg.n(); i++) {
                w(pg.off_un() + i) = w(pg.off_u() + i);
                if (be) w(pg.off_dterm() + i) = 0.0;       // trap: dterm holds -du_n
            }
        }
        eval_sources(pg, w, tn, CB200_MODE_TRAN);
        // ---- Newton on the implicit step
        bool lim_on;
        const int st = newton_step(pg, lu, w, sp, finished, tn, gamma, abstol2, a.max_nl, a.limit, solves, evals, fresh,
                                   lim_on);
        if (finished) continue;
        if (bdf) {
            bool fail = st != CB200_LANE_OK;
            if (fail) {                                       // Newton failed: quarter the step
                bdf_undo(pg, w, B, hh, false);
                fresh = false;
                rej++;
                h = hh / 4.0;
                if (h < a.dtmin) {
                    if (status == CB200_LANE_OK) status = (st == CB200_LANE_MAXITER) ? CB200_LANE_DTMIN : st;
                    finished = true;
                }
                continue;
            }
            if (bdf_error_test(pg, w, a, B)) {                // IDATestError failed
                bdf_undo(pg, w, B, hh, B.kused == 0 && B.nef == 0);
                fresh = false;
                rej++;
                h = B.after_error_fail(hh);
                if (h < a.dtmin || B.nef >= 20) { if (status == CB200_LANE_OK) status = CB200_LANE_DTMIN; finished = true; }
                continue;
            }
            const int kdone = B.kk;
            const double hnew = B.complete(hh);
            bdf_advance(pg, w, kdone);
            t = tn;
            if (act && T < a.max_points) {
                a.out_t[(int64_t)T * p.P + lane] = t;
                for (int q = 0; q < a.n_save; q++)
                    a.out[((int64_t)q * a.max_points + T) * p.P + lane] = read_u(pg, w, __ldg(a.save_idx + q));
            }
            T++;
            h = hnew > a.dtmax ? a.dtmax : hnew;
            if (hit && tn < a.t1) nhist = 0;                  // restart after a breakpoint
            if (!(t < a.t1)) finished = true;
            else if (T >= a.max_points) { if (status == CB200_LANE_OK) status = CB200_LANE_MAXITER; finished = true; }
            continue;
        }
        if (st != CB200_LANE_OK) {                            // Newton failed: shrink and retry
            CB_UNROLL
            for (int i = 0; i < pg.n(); i++) w(pg.off_u() + i) = w(pg.off_un() + i);
            fresh = false;
            rej++;
            h = hh / 4.0;
            if (h < a.dtmin) {
                if (status == CB200_LANE_OK) status = (st == CB200_LANE_MAXITER) ? CB200_LANE_DTMIN : st;
                finished = true;
            }
            continue;
        }
        // ---- local truncation error estimate
        double err = 0.0;
        int pord = 1;
        if (nhist >= 1) {
            double acc = 0.0;
            if (be || nhist == 1) {
                const double r = hh / h1, c = hh / (2.0 * hh + h1);
                CB_UNROLL
                for (int i = 0; i < pg.n(); i++) {
                    const double ui = w(pg.off_u() + i), uni = w(pg.off_un() + i);
                    const double up = uni + r * (uni - w(pg.off_h1() + i));
                    const double tol = lte_atol(a, i) + a.reltol * fmax(fabs(ui), fabs(uni));
                    const double e = c * (ui - up) / tol;
                    acc += e * e;
                }
            } else {
                pord = 2;
                const double ta = -(h1 + h2), tb = -h1, tc = 0.0, tx = hh;
                const double la = (tx - tb) * (tx - tc) / ((ta - tb) * (ta - tc));
                const double lb = (tx - ta) * (tx - tc) / ((tb - ta) * (tb - tc));
                const double lc = (tx - ta) * (tx - tb) / ((tc - ta) * (tc - tb));
                const double c = hh * hh / (hh * hh + 2.0 * (hh + h1) * (hh + h1 + h2));
                CB_UNROLL
                for (int i = 0; i < pg.n(); i++) {
                    const double ui = w(pg.off_u() + i), uni = w(pg.off_un() + i);
                    const double up = la * w(pg.off_h2() + i) + lb * w(pg.off_h1() + i) + lc * uni;
                    const double tol = lte_atol(a, i) + a.reltol * fmax(fabs(ui), fabs(uni));
                    const double e = c * (ui - up) / tol;
                    acc += e * e;
                }
            }
            err = sqrt(acc / (double)pg.n());
        }
        if (err > 1.0) {                                      // reject
            CB_UNROLL
            for (int i = 0; i < pg.n(); i++) w(pg.off_u() + i) = w(pg.off_un() + i);
            fresh = false;
            rej++;
            double f = 0.9 * pow(err, -1.0 / (pord + 1));
            if (f < 0.2) f = 0.2;
            h = hh * f;
            if (h < a.dtmin) { if (status == CB200_LANE_OK) status = CB200_LANE_DTMIN; finished = true; }
            continue;
        }
        // ---- accept
        CB_UNROLL
        for (int i = 0; i < pg.n(); i++) {
            const double ui = w(pg.off_u() + i), uni = w(pg.off_un() + i);
            w(pg.off_dterm() + i) = -(gamma * (ui - uni) + w(pg.off_dterm() + i));   // -du_{n+1}
            w(pg.off_h2() + i) = w(pg.off_h1() + i);
            w(pg.off_h1() + i) = uni;
        }
        h2 = h1; h1 = hh;
        t = tn;
        nhist++;
        if (act && T < a.max_points) {
            a.out_t[(int64_t)T * p.P + lane] = t;
            for (int q = 0; q < a.n_save; q++)
                a.out[((int64_t)q * a.max_points + T) * p.P + lane] = read_u(pg, w, __ldg(a.save_idx + q));
        }
        T++;
        double f = err > 0.0 ? 0.9 * pow(err, -1.0 / (pord + 1)) : 2.0;
        if (f > 2.0) f = 2.0;
        if (f < 0.2) f = 0.2;
        h = hh * f;
        if (h > a.dtmax) h = a.dtmax;
        // restart after a breakpoint: the first step after it is accepted without an error estimate (no
        // history), so it is no longer than the initial step the caller asked for
        if (hit && tn < a.t1) { nhist = 0; h = fmin(h, a.h0); }
        if (!(t < a.t1)) finished = true;
        else if (T >= a.max_points) { if (status == CB200_LANE_OK) status = CB200_LANE_MAXITER; finished = true; }
    }
    if (act) {
        CB_UNROLL
        for (int i = 0; i < pg.n(); i++) a.u[(int64_t)i * p.P + lane] = w(pg.off_u() + i);
        a.status[lane] = status;
        if (a.weak && w.weak) a.weak[lane] = 1;
        a.iters[lane] += solves;
        a.rejected[lane] = rej;
        a.count[lane] = T < a.max_points ? T : a.max_points;
        if (a.evals != nullptr) a.evals[lane] += evals;
    }
}

}  // namespace cb200
