// warp_kernels.cuh -- the batched MNA Newton / transient hot path for MEDIUM circuits:
// one sweep lane per WARP.
//
// lane_kernels.cuh gives every lane one thread.  That is the right mapping while the lane state
// fits in registers / shared memory and the sweep has >> 148 * 2048 lanes; a circuit such as
// the gf180 D flip-flop (30 Verilog-A FETs, n = 145, ~5000 workspace doubles, 16 384 lanes) then
// runs 110 threads per SM, each walking its own 40 KB column of HBM -- pure latency.  Here the 32
// threads of a warp share ONE lane:
//   * device evaluation: thread i evaluates device instance i, i + 32, ... (30 FETs = one round);
//   * assembly: thread per matrix entry sums its stamp segment in program order, then thread per
//     row forms F = C*du + G*u - b over the row's entries in column order;
//   * LU refactor on the host's static pivot order, cut into LEVELS of independent pivots: per
//     level one thread per pivot (reciprocal), one per L entry (scaling), one per target entry
//     (its updates in ascending pivot order), two __syncwarp per level;
//   * triangular solves by rows, one thread per row of a level, one __syncwarp per level;
//   * norms are summed by every thread over ALL rows in index order.
// Every floating-point operation is performed with the same operands in the same order as in
// lane_kernels.cuh (only WHICH thread performs it changes), so the two mappings agree bit for bit;
// tests/test_gpu_parity.py asserts identical waveforms and Newton iteration counts.
// The lane's workspace is a contiguous row ws[lane][slot] of a global array: consecutive slots
// are consecutive addresses, a warp's accesses coalesce, and the resident working set
// (16 warps/SM * 148 SMs * 40 KB = 95 MB) lives in the 126 MB L2.  The arrays on the
// DEPENDENT chains of the refactor and the triangular solves -- the LU factor, the residual /
// solution vector, the work vector and the reciprocal pivots -- stay in that row (struct Hot
// points at them): measured on C4, a copy in shared memory lost to the L1 it takes from the
// lane rows (DESIGN.md s. 4c).
#pragma once
#include "lane_kernels.cuh"

namespace cb200 {

#define CB_FULL 0xffffffffu

// The read-only tables the warp kernels walk on every Newton iteration (segment lists, CSR view,
// level schedule: 43 KB for the flip-flop).  Every data access of the assembly and of the
// refactor is index -> data, so an index that misses the L1 (the lane rows and the model body's
// spills compete for it) puts an L2 round trip on the dependent chain.  Staging the tables in
// shared memory once per block was measured on C4 and loses (2.00 s vs 1.34 s): the shared memory
// it takes from the L1 costs more than the guaranteed index hits save -- so WTab points at the
// global arrays (stage_tables, kernels.cu).  The struct itself lives in shared memory.
struct WTab {
    const int *gseg_ptr, *gseg_idx, *cseg_ptr, *cseg_idx, *bseg_ptr, *bseg_idx, *rowptr, *row_nz, *nz_col;
    const int *jmap, *fill_slots, *colperm;
    const int *piv_ptr, *sc_ptr, *tg_ptr, *flev_ptr, *blev_ptr;
    const int2 *piv, *sc, *fent, *bent;
    const int4 *tg, *upd, *frow, *brow;
};

struct Hot {
    double *F, *wv, *DI, *LU;   // latency-critical arrays of the lane, in its workspace row
    double *buf;      // shared-memory gather buffer of the segmented assembly, ch doubles
    int ch;
    const WTab *tb;   // in shared memory
};

__device__ __forceinline__ int wtid() { return threadIdx.x & 31; }

// ---- the group bodies, once per group shape (see group_kernels.inc) ----
namespace wg32 {
#define G_SIZE 32
#define G_TID ((int)(threadIdx.x & 31))
#define G_SYNC() __syncwarp()
#define G_ALL(x) __all_sync(CB_FULL, (x))
#define G_ANY(x) __any_sync(CB_FULL, (x))
#include "group_kernels.inc"
#undef G_SIZE
#undef G_TID
#undef G_SYNC
#undef G_ALL
#undef G_ANY
}  // namespace wg32

namespace wgblk {
#define G_SIZE ((int)blockDim.x)
#define G_TID ((int)threadIdx.x)
#define G_SYNC() __syncthreads()
#define G_ALL(x) (__syncthreads_and((x)) != 0)
#define G_ANY(x) (__syncthreads_or((x)) != 0)
#include "group_kernels.inc"
#undef G_SIZE
#undef G_TID
#undef G_SYNC
#undef G_ALL
#undef G_ANY
}  // namespace wgblk

}  // namespace cb200
