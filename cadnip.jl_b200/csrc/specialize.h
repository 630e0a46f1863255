// specialize.h -- circuit-specialised kernel generation (see specialize.cpp).
#pragma once
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "cb200_internal.h"
#include "kernels.h"

namespace cb200 {

constexpr int kSpecAbi = 9;

struct SpecInput {
    const Structure *st;
    const Program *prog;              // workspace offsets / n_slots
    const std::vector<int> *dev_kind, *dev_flags, *dev_node_ptr, *dev_nodes, *dev_param_ptr,
        *dev_params, *dev_gbase, *dev_cbase, *dev_bbase, *dev_sbase, *src_list, *nl_list, *limit_init_ref;
    const std::vector<double> *uniform;
    const std::vector<unsigned char> *src_uniform;
    int method;                       // CB200_METHOD_* compiled into the transient kernel
    std::string va_header_path;       // emitted Verilog-A models ("" = none)
    bool with_adaptive = true;        // also generate the adaptive transient kernel (a third of the compile time)
    bool tran_limit = false;          // compile the CB200_TRAN_LIMIT restart path into the transient kernels
    const LuSchedule *lu_dc, *lu_tr;
    int n_lane_cols;
    int block, min_blocks;            // __launch_bounds__ of the generated kernels
};

typedef cudaError_t (*spec_dc_fn)(const Program *, const SpecArgs *, const DcArgs *, cudaStream_t);
typedef cudaError_t (*spec_tran_fn)(const Program *, const SpecArgs *, const TranArgs *, cudaStream_t);
typedef cudaError_t (*spec_adapt_fn)(const Program *, const SpecArgs *, const AdaptArgs *, cudaStream_t);
typedef cudaError_t (*spec_counters_fn)(unsigned long long *, cudaStream_t);

struct SpecModule {
    void *dl = nullptr;
    spec_dc_fn dc = nullptr;
    spec_tran_fn tran_fixed = nullptr;
    spec_adapt_fn tran_adaptive = nullptr;
    spec_counters_fn take_counters = nullptr;   // lane-steps executed by the fixed-step kernels (bypass), or null
    int block = 0;
    std::string path;
};

// A kernel set: the table-driven kernels of kernels.cu, either the library's built-in
// copy or a variant rebuilt with Verilog-A device models (-DCB200_VA_HEADER=...).
typedef cudaError_t (*k_eval_fn)(const Program *, const SpecArgs *, const EvalArgs *, cudaStream_t, int64_t *);
typedef cudaError_t (*k_dc_fn)(const Program *, const LuProgram *, const SpecArgs *, const DcArgs *, int,
                               size_t, cudaStream_t, int64_t *);
typedef cudaError_t (*k_tran_fn)(const Program *, const LuProgram *, const SpecArgs *, const TranArgs *, int,
                                 size_t, cudaStream_t, int64_t *);
typedef cudaError_t (*k_adapt_fn)(const Program *, const LuProgram *, const SpecArgs *, const AdaptArgs *, int,
                                  size_t, cudaStream_t, int64_t *);
struct KernelSet {
    void *dl = nullptr;
    k_eval_fn eval = nullptr;
    k_dc_fn dc = nullptr;
    k_tran_fn tran_fixed = nullptr;
    k_adapt_fn tran_adaptive = nullptr;
    std::string va_header_path;       // "" for the built-in set
};
// Writes the emitted Verilog-A header into cache_dir, rebuilds kernels.cu against it
// (nvcc, cached by content hash) and loads the result.  Returns "" on success.
bool va_kernel_set_cached(const std::string &va_header_text, const std::string &csrc_dir, const std::string &cache_dir);
std::string build_va_kernel_set(const std::string &va_header_text, const std::string &csrc_dir,
                                const std::string &cache_dir, KernelSet &out);
void unload_kernel_set(KernelSet &k);

std::string generate_spec_source(const SpecInput &in);
// Returns "" on success.  The shared object is cached under cache_dir, keyed by a hash
// of the generated source and of the headers it includes.
std::string build_and_load_spec(const std::string &src, const std::string &csrc_dir,
                                const std::string &cache_dir, bool compile_only, SpecModule &out);
void unload_spec(SpecModule &m);

}  // namespace cb200
