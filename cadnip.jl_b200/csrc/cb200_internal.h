// cb200_internal.h -- host-side structures shared by symbolic.cpp / api.cu / kernels.cu.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/cadnip_b200.h"

namespace cb200 {

// CSC pattern + stamp maps: the CompiledStructure of src/mna/precompile.jl:88-160,
// 0-based internally (getters convert to Julia's 1-based Int).
struct Structure {
    int n = 0, n_nodes = 0, n_currents = 0, n_charges = 0, n_limits = 0;
    int64_t nnz = 0, nG = 0, nC = 0, nb = 0;
    std::vector<int> colptr, rowval;         // unified G|C pattern
    std::vector<int> G_map, C_map;           // COO k -> nz slot
    std::vector<int> b_rows;                 // b stamp k -> row (-1 = dropped)
    std::vector<int> diag_nz;                // [n_nodes] nz slot of (i,i) or -1
    // segment lists for the deterministic, atomics-free assembly: nz slot s sums the
    // stamp values gseg_idx[gseg_ptr[s] .. gseg_ptr[s+1]) left to right, i.e. in COO
    // (program) order -- the summation order of `nzval[idx] += v` in the reference
    // (src/mna/value_only.jl:395-421).
    std::vector<int> gseg_ptr, gseg_idx, cseg_ptr, cseg_idx, bseg_ptr, bseg_idx;
    std::vector<int> nz_row, nz_col;         // coordinates of every nz slot
    std::vector<uint8_t> nz_is_node_diag;    // gshunt target (precompile.jl:524-534)
};

// Build pattern and maps from resolved 1-based COO.  Returns "" or an error.
std::string build_structure(const cb200_desc &d, Structure &out);

// Host copy of the device table of a checked description (api.cu: read_circuit), and the device
// lists derived from it.
struct Circuit {
    std::vector<int> dev_kind, dev_flags, dev_node_ptr, dev_nodes, dev_param_ptr, dev_params;
    std::vector<int> dev_gbase, dev_cbase, dev_bbase, dev_sbase, limit_init_ref;
    std::vector<double> uniform;
    int n_lane_cols = 0;
    std::vector<int> src_list;               // devices whose stamps depend on t only (sources)
    std::vector<unsigned char> src_uniform;  // [src] 1: every parameter of the source is uniform
    std::vector<int> nl_list;                // devices whose stamps depend on the iterate
    bool has_va = false;
};

// Static-pivot sparse LU schedule (the symbolic phase that replaces KLU analyze).
struct LuSchedule {
    int n = 0;
    int64_t nlu = 0;                         // number of stored factor entries
    std::vector<int> rowperm, colperm;       // pivot k eliminates row rowperm[k], col colperm[k]
    std::vector<int> diag_slot;              // [n]
    std::vector<int> Lptr, L_slot, L_row;    // column k of L (below-diagonal), rows in pivot coords
    std::vector<int> Uptr, U_slot, U_col;    // row k of U (right of diagonal), cols in pivot coords
    std::vector<int> tgt_ptr, tgt;           // for pivot k: tgt[tgt_ptr[k] + e*nU + q]
    std::vector<int> jmap;                   // nz slot -> lu slot
    std::vector<int> fill_slots;             // lu slots with no nz source (zeroed per factor)
    int64_t flops = 0;                       // multiply-subtract count of one refactor
    double gamma = 0.0;
    bool valid = false;
};

// absJ: nominal magnitude of every pattern entry (max over probes; 0 = numerically
// absent at the probes).  Threshold Markowitz on the magnitudes, then symbolic fill.
// absJmin (optional): the SMALLEST magnitude of every entry over the probes; the sparse analysis
// (n > 1536) admits a pivot on its smallest value against its column's largest.
std::string analyze_lu(const Structure &s, const std::vector<double> &absJ, double threshold,
                       LuSchedule &out, const std::vector<double> *absJmin = nullptr);

// Level schedule of the same factorisation for the lane-per-warp kernels (warp_kernels.cuh):
// the elimination DAG cut into levels whose operations are independent, so that the 32 threads
// of a lane's warp work in parallel between two __syncwarp()s.  Every target entry still receives
// its updates in ascending pivot order and every row of the triangular solves its terms in
// ascending (L) / stored (U) order: the floating-point results equal the serial schedule's bit
// for bit.  Arrays of int2 / int4 records are stored flattened.
struct LevelSchedule {
    int n_lev = 0, n_fwd = 0, n_bwd = 0;
    std::vector<int> piv_ptr, sc_ptr, tg_ptr;   // [n_lev + 1] ranges of the three per-level lists
    std::vector<int> piv;                       // int2 {pivot k, diag slot}
    std::vector<int> sc;                        // int2 {L slot, pivot k}: L[slot] *= 1/pivot
    std::vector<int> tg;                        // int4 {target slot, upd begin, upd end, 0}
    std::vector<int> upd;                       // int4 {L slot, U slot, pivot k, 0}
    std::vector<int> flev_ptr;                  // [n_fwd + 1]
    std::vector<int> frow;                      // int4 {row i, rowperm[i], ent begin, ent end}
    std::vector<int> fent;                      // int2 {L slot, column k}
    std::vector<int> blev_ptr;                  // [n_bwd + 1]
    std::vector<int> brow;                      // int4 {row k, ent begin, ent end, 0}
    std::vector<int> bent;                      // int2 {U slot, column}
};
void build_level_schedule(const LuSchedule &S, LevelSchedule &out);
// test hook: run the serial and the level schedule on the host (J in pattern order)
void host_lu_solve(const LuSchedule &S, const LevelSchedule &V, const std::vector<double> &J,
                   const std::vector<double> &rhs, std::vector<double> &x_serial, std::vector<double> &x_level);

}  // namespace cb200
