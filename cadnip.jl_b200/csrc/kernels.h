// kernels.h -- device-visible program descriptors and kernel launchers.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace cb200 {

// Everything the device needs to re-run the "builder" for a lane: the device table
// recorded next to each stamp! call, the segment lists of the assembly, the CSC
// coordinates, and the layout of a lane's workspace.  All pointers are device
// pointers to read-only int32 / fp64 arrays that are uniform across lanes.
struct Program {
    int n, n_nodes, n_limits, nnz, nG, nC, nb, n_dev, n_src, n_nl, n_lane_cols;
    int64_t P;                      // lanes on this device
    const int *dev_kind, *dev_flags, *dev_node_ptr, *dev_nodes, *dev_param_ptr, *dev_params;
    const int *dev_gbase, *dev_cbase, *dev_bbase;
    const int *dev_sbase;           // first private state slot of each device (relative to off_DS)
    const int *src_list;            // devices whose stamps depend on t only (sources)
    const int *nl_list;             // devices whose stamps depend on the iterate x
    const unsigned char *src_uniform;  // [n_src] 1: every parameter of the source is uniform
    const double *uniform;          // uniform parameter pool
    const double *lanes;            // per-lane parameter SoA [col][P]
    const int *limit_init_ref;      // [n_limits]
    const int *gseg_ptr, *gseg_idx, *cseg_ptr, *cseg_idx, *bseg_ptr, *bseg_idx;
    const int *colptr, *rowval;
    const unsigned char *nz_is_node_diag;
    // lane workspace: slot offsets (in doubles); element (slot) of a lane lives at
    // ws[slot * stride + lane_in_block]  (shared) or ws[slot * P + lane] (global).
    int off_u, off_un, off_dterm, off_F, off_wv, off_SG, off_SC, off_SB, off_LU, off_limw, off_lp;
    int off_DS;                     // private device state (Verilog-A set-up values)
    int off_srcc;                   // [n_src] warp-cooperative source value cache
    int off_h1, off_h2;             // adaptive history (u_{n-1}, u_{n-2})
    int off_phi;                    // variable-order BDF: modified divided differences phi[0..5], 6 n slots
    int n_slots;
    // lane-per-warp kernels (warp_kernels.cuh): CSR view of the pattern (row -> nz indices in
    // column order, nz -> column) and three more workspace arrays behind the n_slots above:
    // per-entry G and C sums [nnz] each, reciprocal pivots [n].  A lane's workspace is the
    // contiguous row ws[lane * n_slots_w + slot].
    const int *rowptr, *row_nz, *nz_col;
    int off_GS, off_CS, off_DI;
    int n_slots_w;
};

// Static-pivot LU schedule (see LuSchedule in cb200_internal.h).
struct LuProgram {
    int n, nlu, n_fill;
    const int *rowperm, *colperm, *diag_slot;
    const int *Lptr, *L_slot, *L_row, *Uptr, *U_slot, *U_col, *tgt_ptr, *tgt, *jmap, *fill_slots;
    // level schedule of the same factorisation (lane-per-warp kernels; LevelSchedule in
    // cb200_internal.h): per level the pivots, the L entries to scale and the update targets
    int n_lev, n_fwd, n_bwd;
    int n_sc, n_bent, n_tg, n_upd;      // record counts of sc / fent, bent, tg, upd
    const int *piv_ptr, *sc_ptr, *tg_ptr;
    const int2 *piv, *sc;
    const int4 *tg, *upd;
    const int *flev_ptr;
    const int4 *frow;
    const int2 *fent;
    const int *blev_ptr;
    const int4 *brow;
    const int2 *bent;
};

struct SpecArgs {
    int mode;
    double temp, gmin, gshunt, srcFact;
};

// ---- evaluation only (K1 instance x lane device evaluation, K2 segmented assembly)
struct EvalArgs {
    double t;
    int initjct;
    double *ws;             // global workspace [n_slots][P]; x already in the off_u slots
    double *G_nz, *C_nz, *b;  // outputs [nnz][P], [nnz][P], [n][P] (may be null)
    double *limw;           // [n_limits][P] or null
};
cudaError_t launch_eval(const Program &p, const SpecArgs &s, const EvalArgs &a, cudaStream_t st,
                        int64_t *launches);

// ---- DC: PCNR / plain Newton per lane (src/mna/solve.jl:542-698)
struct DcArgs {
    int algorithm;          // 0: PCNR (_dc_pcnr_newton), 1: plain Newton (_dc_newton_compiled),
                            // 2: gshunt stepping then source stepping (solve.jl:720-850), 3: source stepping only
    double abstol;
    int maxiters;
    double t;
    double *u;              // [n][P] in: start, out: solution
    const unsigned char *active;   // [P] or null = all lanes
    const double *gshunt_lane;     // [P] or null -> spec.gshunt
    const double *srcfact_lane;    // [P] or null -> spec.srcFact
    int *status;            // [P] CB200_LANE_*
    int *iters;             // [P] (+= linear solves)
    unsigned char *converged;  // [P]
    int *weak;              // [P] or null: set to 1 when a refactor of the lane met a weak pivot (see weak_pivot())
    double *ws_global;      // used when the lane workspace does not fit in shared memory
    int gather_ch;          // set by the launcher: doubles of the shared-memory gather buffer of a lane-per-warp / -block lane
};
cudaError_t launch_dc(const Program &p, const LuProgram &lu, const SpecArgs &s, const DcArgs &a,
                      int block, size_t smem_limit, cudaStream_t st, int64_t *launches);

// ---- transient, fixed step (BE / trap / Gear-2), whole time loop on the device
struct TranArgs {
    int method;             // CB200_METHOD_*
    double t0, h;
    int64_t nsteps;         // total steps of the run (final point is always saved)
    int64_t k_begin, k_end; // steps this launch performs (1-based, inclusive)
    int64_t tp_begin;       // first output point this launch writes
    double *hist;           // [2n][P] integrator history (u_n, dterm) carried between segments, or null
    double abstol;
    int max_nl;
    int limit;              // CB200_TRAN_LIMIT: PCNR corrector after every transient Newton solve
    int save_every;
    int n_save;
    const int *save_idx;    // device, 0-based unknown indices
    int64_t T;              // saved points per lane
    double *u;              // [n][P] in: u(t0); out: u(t1)
    double *out;            // [n_save][T][P]
    int *status;            // [P]
    int *iters;             // [P]
    int *evals;             // [P] or null: += device-model evaluation passes executed for the lane
    int *weak;              // [P] or null (see DcArgs)
    double *ws_global;
    int gather_ch;
};
cudaError_t launch_tran_fixed(const Program &p, const LuProgram &lu, const SpecArgs &s,
                              const TranArgs &a, int block, size_t smem_limit, cudaStream_t st,
                              int64_t *launches);

// ---- transient, adaptive (trap + LTE), per-lane time axis
struct AdaptArgs {
    int method;
    double t0, t1, h0, dtmin, dtmax;
    double abstol, reltol, lte_abstol;
    // absolute LTE tolerance per class of unknown [nodes | currents | charges | limits]
    // (state_abstol, build.jl:276-283); all three = lte_abstol unless CB200_TRAN_CLASS_ABSTOL
    double tol_v, tol_i, tol_q;
    int cls_i0, cls_q0, cls_l0;      // first current / charge / limit unknown (0-based)
    int max_nl;
    int limit;
    int n_save;
    const int *save_idx;
    int max_points;
    const double *tstops;   // device, sorted
    int n_tstops;
    double *u;              // [n][P]
    double *out_t;          // [max_points][P]
    double *out;            // [n_save][max_points][P]
    int *count;             // [P]
    int *status, *iters, *rejected;
    int *evals;             // [P] or null (see TranArgs)
    int *weak;              // [P] or null (see DcArgs)
    double *ws_global;
    int gather_ch;
};
cudaError_t launch_tran_adaptive(const Program &p, const LuProgram &lu, const SpecArgs &s,
                                 const AdaptArgs &a, int block, size_t smem_limit,
                                 cudaStream_t st, int64_t *launches);

cudaError_t launch_debug_exp(const double *x, double *y, int n, cudaStream_t st);

// pick lanes-per-block so the lane workspace fits in shared memory (0 = use global)
int choose_block(int n_slots, size_t smem_limit, int preferred);
// true: the circuit runs on the lane-per-warp kernels (workspace [lane][n_slots_w] in HBM / L2)
bool use_warp_kernels(int n_slots, size_t smem_limit, int preferred);
// true: ... on the lane-per-BLOCK kernels (large circuits on few lanes)
bool use_block_kernels(const Program &p, size_t smem_limit, int preferred);

}  // namespace cb200

// C entry points of a kernel set (kernels.cu; see KernelSet in specialize.h)
extern "C" {
int cb200_k_abi(void);
cudaError_t cb200_k_eval(const cb200::Program *, const cb200::SpecArgs *, const cb200::EvalArgs *,
                         cudaStream_t, int64_t *);
cudaError_t cb200_k_dc(const cb200::Program *, const cb200::LuProgram *, const cb200::SpecArgs *,
                       const cb200::DcArgs *, int, size_t, cudaStream_t, int64_t *);
cudaError_t cb200_k_tran_fixed(const cb200::Program *, const cb200::LuProgram *, const cb200::SpecArgs *,
                               const cb200::TranArgs *, int, size_t, cudaStream_t, int64_t *);
cudaError_t cb200_k_tran_adaptive(const cb200::Program *, const cb200::LuProgram *,
                                  const cb200::SpecArgs *, const cb200::AdaptArgs *, int, size_t,
                                  cudaStream_t, int64_t *);
}
