// specialize.cpp -- the emitter: lowers ONE circuit (device table, stamp segments,
// CSC pattern, static-pivot LU schedules, uniform parameter values) to sm_100a CUDA
// source in which every index is a compile-time constant, compiles it with nvcc
// into a small shared object and loads it.  The generated translation unit only
// instantiates the templates of lane_kernels.cuh with a constexpr program type, so
// the specialised and the table-driven kernels share one implementation of every
// device model, of the assembly and of the LU (and therefore one arithmetic).
#include <dlfcn.h>
#include <sys/stat.h>
#include <unistd.h>

#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <sstream>

#include "specialize.h"

namespace cb200 {

// Tables live at namespace scope (`__device__ constexpr`): an access with a constant index
// folds to the literal, one with a run-time index is a read-only global load.  A function-local
// `constexpr T t[]` would be copied to the STACK for any run-time index -- and the stores that
// rebuild it stay in the kernel even when every such access is later optimised away.
static std::ostringstream *g_data = nullptr;     // namespace-scope table definitions of the file being generated
static std::string g_prefix;                     // struct the accessors belong to (table names must be unique)

static void emit_int_table(std::ostringstream &o, const char *name, const std::vector<int> &v)
{
    std::ostringstream &d = *g_data;
    d << "__device__ constexpr int k_" << g_prefix << "_" << name << "[] = {";
    if (v.empty()) d << "0";
    for (size_t i = 0; i < v.size(); i++) d << (i ? "," : "") << v[i];
    d << "};\n";
    o << "    __device__ static constexpr int " << name << "(int i) { return k_" << g_prefix << "_" << name
      << "[i]; }\n";
}

static void emit_const(std::ostringstream &o, const char *name, long long v)
{
    o << "    __device__ static constexpr int " << name << "() { return " << v << "; }\n";
}

static std::string hexdouble(double v)
{
    char buf[64];
    if (v != v) return "(0.0/0.0)";
    if (v == 1.0 / 0.0) return "(1.0/0.0)";
    if (v == -1.0 / 0.0) return "(-1.0/0.0)";
    snprintf(buf, sizeof buf, "%a", v);
    return buf;
}

// ---- straight-line code: one statement per stamp / matrix entry / elimination update,
// in exactly the order of the loops of lane_kernels.cuh (assemble, factor_and_solve,
// apply_update), so both variants perform the same floating-point operations.
// Per-entry sums of the stamp segments, G and C separately: G(u) and C(u) as CSC values.  They
// depend on the iterate only (sources and linear devices stamp constants into G / C), so the time
// loop keeps them from the converged check of one step to the first residual of the next
// (tran_fixed_body: `fresh`).  Emitted into SProg; called after every device evaluation.
static void emit_accumulate(std::ostringstream &o, const Structure &st, const Program &p)
{
    o << "    template <typename W>\n    __device__ static __forceinline__ void accumulate(W &w)\n    {\n";
    for (int s = 0; s < (int)st.nnz; s++) {
        if (st.gseg_ptr[s] < st.gseg_ptr[s + 1]) {
            o << "        {\n            double gsum = 0.0;\n";
            for (int q = st.gseg_ptr[s]; q < st.gseg_ptr[s + 1]; q++)
                o << "            gsum += w(" << p.off_SG + st.gseg_idx[q] << ");\n";
            o << "            w(" << p.off_GS + s << ") = gsum;\n        }\n";
        }
        if (st.cseg_ptr[s] < st.cseg_ptr[s + 1]) {
            o << "        {\n            double csum = 0.0;\n";
            for (int q = st.cseg_ptr[s]; q < st.cseg_ptr[s + 1]; q++)
                o << "            csum += w(" << p.off_SC + st.cseg_idx[q] << ");\n";
            o << "            w(" << p.off_CS + s << ") = csum;\n        }\n";
        }
    }
    o << "    }\n";
}

static void emit_assemble(std::ostringstream &o, const Structure &st, const Program &p,
                          const LuSchedule &S)
{
    o << "    template <bool TRAN, typename W>\n"
         "    __device__ static __forceinline__ double assemble(W &w, double gamma, double gshunt,\n"
         "                                                      double srcFact, bool &bad)\n    {\n";
    for (int r = 0; r < st.n; r++) o << "        double F" << r << " = 0.0;\n";
    for (int s : S.fill_slots) o << "        w(" << p.off_LU + s << ") = 0.0;\n";
    for (int j = 0; j < st.n; j++) {
        if (st.colptr[j] == st.colptr[j + 1]) continue;
        o << "        {   // column " << j << "\n";
        o << "            const double uj = w(" << p.off_u + j << ");\n";
        o << "            double duj = 0.0;\n";
        o << "            if (TRAN) duj = gamma * (uj - w(" << p.off_un + j << ")) + w(" << p.off_dterm + j << ");\n";
        o << "            (void)duj;\n";
        for (int s = st.colptr[j]; s < st.colptr[j + 1]; s++) {
            const int r = st.rowval[s];
            const bool has_g = st.gseg_ptr[s] < st.gseg_ptr[s + 1];
            const bool has_c = st.cseg_ptr[s] < st.cseg_ptr[s + 1];
            o << "            {   // (" << r << "," << j << ")\n";
            if (has_g) o << "                double gsum = w(" << p.off_GS + s << ");\n";
            else o << "                double gsum = 0.0;\n";
            if (st.nz_is_node_diag[s]) o << "                if (gshunt != 0.0) gsum += gshunt;\n";
            o << "                double jv = gsum;\n";
            if (has_c) {
                o << "                if (TRAN) {\n                    const double csum = w(" << p.off_CS + s << ");\n";
                o << "                    F" << r << " += csum * duj;\n                    jv += gamma * csum;\n                }\n";
            }
            if (has_g || st.nz_is_node_diag[s]) o << "                F" << r << " += gsum * uj;\n";
            o << "                w(" << p.off_LU + S.jmap[s] << ") = jv;\n            }\n";
        }
        o << "        }\n";
    }
    o << "        double nrm2 = 0.0;\n";
    for (int r = 0; r < st.n; r++) {
        o << "        {\n            double bsum = 0.0;\n";
        for (int q = st.bseg_ptr[r]; q < st.bseg_ptr[r + 1]; q++)
            o << "            bsum += w(" << p.off_SB + st.bseg_idx[q] << ");\n";
        if (st.bseg_ptr[r] < st.bseg_ptr[r + 1]) o << "            if (srcFact < 1.0) bsum *= srcFact;\n";
        o << "            const double f = F" << r << " - bsum;\n";
        o << "            w(" << p.off_F + r << ") = f;\n            nrm2 += f * f;\n        }\n";
    }
    o << "        bad = !isfinite(nrm2);\n        return nrm2;\n    }\n";
}

static void emit_factor_solve(std::ostringstream &o, const Program &p, const LuSchedule &S)
{
    const int LU = p.off_LU, WV = p.off_wv;
    o << "    template <typename W>\n"
         "    __device__ static __forceinline__ bool factor_and_solve(W &w, bool &singular)\n    {\n"
         "        singular = false;\n";
    for (int k = 0; k < S.n; k++) {
        const int ds = LU + S.diag_slot[k];
        const int l0 = S.Lptr[k], l1 = S.Lptr[k + 1], u0 = S.Uptr[k], u1 = S.Uptr[k + 1];
        o << "        {   // pivot " << k << "\n";
        o << "            const double dgl = w(" << ds << ");\n";
        o << "            if (!(fabs(dgl) >= DBL_MIN) || !isfinite(dgl)) singular = true;\n";
        o << "            const double inv = 1.0 / dgl;\n            w(" << ds << ") = inv;\n";
        int tq = S.tgt_ptr[k];
        for (int e = l0; e < l1; e++) {
            const int ls = LU + S.L_slot[e];
            o << "            {\n                const double l = w(" << ls << ") * inv;\n                w(" << ls << ") = l;\n"
                 "                w.weak |= weak_pivot(l);\n";
            for (int q = u0; q < u1; q++, tq++) {
                const int ts = LU + S.tgt[tq];
                o << "                w(" << ts << ") = w(" << ts << ") - l * w(" << LU + S.U_slot[q] << ");\n";
            }
            o << "            }\n";
        }
        o << "        }\n";
    }
    for (int k = 0; k < S.n; k++) o << "        w(" << WV + k << ") = w(" << p.off_F + S.rowperm[k] << ");\n";
    for (int k = 0; k < S.n; k++) {
        if (S.Lptr[k] == S.Lptr[k + 1]) continue;
        o << "        {\n            const double zk = w(" << WV + k << ");\n";
        for (int e = S.Lptr[k]; e < S.Lptr[k + 1]; e++) {
            const int i = WV + S.L_row[e];
            o << "            w(" << i << ") = w(" << i << ") - w(" << LU + S.L_slot[e] << ") * zk;\n";
        }
        o << "        }\n";
    }
    o << "        bool finite = true;\n";
    for (int k = S.n - 1; k >= 0; k--) {
        o << "        {\n            double acc = w(" << WV + k << ");\n";
        for (int q = S.Uptr[k]; q < S.Uptr[k + 1]; q++)
            o << "            acc -= w(" << LU + S.U_slot[q] << ") * w(" << WV + S.U_col[q] << ");\n";
        o << "            acc *= w(" << LU + S.diag_slot[k] << ");\n            w(" << WV + k << ") = acc;\n"
             "            finite &= isfinite(acc);\n        }\n";
    }
    o << "        return finite && !singular;\n    }\n";
    o << "    template <typename W>\n    __device__ static __forceinline__ void apply_update(W &w)\n    {\n";
    for (int k = 0; k < S.n; k++) {
        const int j = p.off_u + S.colperm[k];
        o << "        w(" << j << ") = w(" << j << ") - w(" << WV + k << ");\n";
    }
    o << "    }\n";
}

static void emit_lu(std::ostringstream &o, const char *sname, const Structure &st, const Program &p,
                    const LuSchedule &S)
{
    g_prefix = sname;
    o << "struct " << sname << " {\n";
    emit_assemble(o, st, p, S);
    emit_factor_solve(o, p, S);
    emit_const(o, "n", S.n);
    emit_const(o, "n_fill", (long long)S.fill_slots.size());
    emit_int_table(o, "rowperm", S.rowperm);
    emit_int_table(o, "colperm", S.colperm);
    emit_int_table(o, "diag_slot", S.diag_slot);
    emit_int_table(o, "Lptr", S.Lptr);
    emit_int_table(o, "L_slot", S.L_slot);
    emit_int_table(o, "L_row", S.L_row);
    emit_int_table(o, "Uptr", S.Uptr);
    emit_int_table(o, "U_slot", S.U_slot);
    emit_int_table(o, "U_col", S.U_col);
    emit_int_table(o, "tgt_ptr", S.tgt_ptr);
    emit_int_table(o, "tgt", S.tgt);
    emit_int_table(o, "jmap", S.jmap);
    emit_int_table(o, "fill_slot", S.fill_slots);
    o << "};\n";
}

// What the quiescent-step bypass of tran_fixed_body needs of one circuit: the b stamp slots of its sources
// (a snapshot before the step's source evaluation, and the bitwise comparison after it), and the hook that
// adds a thread's executed steps to cb200_spec_nexec.
static void emit_bypass(std::ostringstream &o, const SpecInput &in)
{
    const Program &p = *in.prog;
    std::ostringstream so, ss;
    int q = 0;
    for (int d : *in.src_list)
        for (int b = (*in.dev_bbase)[d]; b < (*in.dev_bbase)[d + 1]; b++, q++) {
            so << "        old[" << q << "] = w(" << p.off_SB + b << ");\n";
            ss << "        same = same && (w(" << p.off_SB + b << ") == old[" << q << "]);\n";
        }
    o << "    static constexpr int kSrcSlots = " << q << ";\n";
    o << "    template <typename W>\n    __device__ static __forceinline__ void src_snapshot(W &w, double *old)\n    {\n"
      << so.str() << "    }\n";
    o << "    template <typename W>\n    __device__ static __forceinline__ bool src_same(W &w, const double *old, bool same)\n    {\n"
      << ss.str() << "        return same;\n    }\n";
    o << "    __device__ static __forceinline__ void count_steps(int nexec)\n    {\n"
         "        atomicAdd(&cb200_spec_nexec, (unsigned long long)nexec);\n    }\n";
}

std::string generate_spec_source(const SpecInput &in)
{
    const Structure &st = *in.st;
    const Program &p = *in.prog;
    std::ostringstream head, data, o;
    g_data = &data;
    g_prefix = "SProg";
    head << "// generated by cadnip-b200 (specialize.cpp) -- circuit-specialised kernels; do not edit\n";
    if (!in.va_header_path.empty())
        head << "#define CB200_VA_FN __forceinline__\n#define CB200_VA_HEADER \"" << in.va_header_path << "\"\n";
    head << "#include \"lane_kernels.cuh\"\n";
    head << "namespace {\nusing namespace cb200;\n";
    // CB200_NO_BYPASS=1 generates the fixed-step kernel without the quiescent-step bypass of tran_fixed_body
    const bool bypass = getenv("CB200_NO_BYPASS") == nullptr;
    if (bypass) o << "__device__ unsigned long long cb200_spec_nexec;   // lane-steps executed (not bypassed) since last read\n";
    o << "struct SProg {\n";
    o << "    static constexpr bool kStatic = true;\n    static constexpr int kUnroll = 4096;\n";
    o << "    static constexpr int kMethod = " << in.method << ";\n";
    o << "    static constexpr bool kTranLimit = " << (in.tran_limit ? "true" : "false") << ";\n";
    o << "    static constexpr bool kBypass = " << (bypass ? "true" : "false") << ";\n";
    if (bypass) emit_bypass(o, in);
    emit_const(o, "n", st.n);
    emit_const(o, "n_limits", st.n_limits);
    emit_const(o, "nnz", st.nnz);
    emit_const(o, "n_dev", (long long)in.dev_kind->size());
    emit_const(o, "n_src", (long long)in.src_list->size());
    emit_const(o, "n_nl", (long long)in.nl_list->size());
    emit_const(o, "n_lane_cols", in.n_lane_cols);
    emit_int_table(o, "src_list", *in.src_list);
    emit_int_table(o, "nl_list", *in.nl_list);
    emit_int_table(o, "dev_kind", *in.dev_kind);
    emit_int_table(o, "dev_flags", *in.dev_flags);
    emit_int_table(o, "dev_node_ptr", *in.dev_node_ptr);
    emit_int_table(o, "dev_node", *in.dev_nodes);
    emit_int_table(o, "dev_param_ptr", *in.dev_param_ptr);
    emit_int_table(o, "dev_param", *in.dev_params);
    emit_int_table(o, "dev_gbase", *in.dev_gbase);
    emit_int_table(o, "dev_cbase", *in.dev_cbase);
    emit_int_table(o, "dev_bbase", *in.dev_bbase);
    emit_int_table(o, "dev_sbase", *in.dev_sbase);
    data << "__device__ constexpr double k_SProg_uniform[] = {";
    if (in.uniform->empty()) data << "0.0";
    for (size_t i = 0; i < in.uniform->size(); i++) data << (i ? "," : "") << hexdouble((*in.uniform)[i]);
    data << "};\n";
    o << "    __device__ static constexpr double uniform(int i) { return k_SProg_uniform[i]; }\n";
    emit_int_table(o, "limit_init_ref", *in.limit_init_ref);
    emit_int_table(o, "gseg_ptr", st.gseg_ptr);
    emit_int_table(o, "gseg_idx", st.gseg_idx);
    emit_int_table(o, "cseg_ptr", st.cseg_ptr);
    emit_int_table(o, "cseg_idx", st.cseg_idx);
    emit_int_table(o, "bseg_ptr", st.bseg_ptr);
    emit_int_table(o, "bseg_idx", st.bseg_idx);
    emit_int_table(o, "colptr", st.colptr);
    emit_int_table(o, "rowval", st.rowval);
    {
        std::vector<int> nd(st.nz_is_node_diag.begin(), st.nz_is_node_diag.end());
        data << "__device__ constexpr int k_SProg_nz_is_node_diag[] = {";
        if (nd.empty()) data << "0";
        for (size_t i = 0; i < nd.size(); i++) data << (i ? "," : "") << nd[i];
        data << "};\n";
        o << "    __device__ static constexpr bool nz_is_node_diag(int i) { return k_SProg_nz_is_node_diag[i] != 0; }\n";
    }
    emit_const(o, "off_u", p.off_u); emit_const(o, "off_un", p.off_un);
    emit_const(o, "off_dterm", p.off_dterm); emit_const(o, "off_F", p.off_F);
    emit_const(o, "off_wv", p.off_wv); emit_const(o, "off_SG", p.off_SG);
    emit_const(o, "off_SC", p.off_SC); emit_const(o, "off_SB", p.off_SB);
    emit_const(o, "off_LU", p.off_LU); emit_const(o, "off_limw", p.off_limw);
    emit_const(o, "off_lp", p.off_lp); emit_const(o, "off_srcc", p.off_srcc);
    emit_const(o, "off_DS", p.off_DS);
    emit_const(o, "off_h1", p.off_h1);
    emit_const(o, "off_h2", p.off_h2);
    emit_const(o, "off_phi", p.off_phi);
    emit_const(o, "off_GS", p.off_GS);
    emit_const(o, "off_CS", p.off_CS);
    emit_accumulate(o, st, p);
    // straight-line device evaluation lists (eval_all / eval_nonlinear / eval_sources)
    o << "    template <typename W>\n    __device__ static __forceinline__ void eval_all(W &w, double t, int mode, bool initjct)\n    {\n        SProg pg;\n";
    for (size_t d = 0; d < in.dev_kind->size(); d++)
        o << "        eval_device<0>(pg, w, " << d << ", t, mode, initjct);\n";
    o << "    }\n";
    o << "    template <typename W>\n    __device__ static __forceinline__ void eval_nonlinear(W &w, double t, int mode, bool initjct)\n    {\n        SProg pg;\n";
    for (int d : *in.nl_list) o << "        eval_device<1>(pg, w, " << d << ", t, mode, initjct);\n";
    o << "    }\n";
    o << "    template <typename W>\n    __device__ static __forceinline__ void eval_sources(W &w, double t, int mode)\n    {\n        SProg pg;\n";
    for (int d : *in.src_list) o << "        eval_device<2>(pg, w, " << d << ", t, mode, false);\n";
    o << "    }\n";
    o << "    template <typename W>\n    __device__ static __forceinline__ void eval_sources_step(W &w, int64_t k, bool first, double t0, double h, int mode)\n    {\n        SProg pg;\n";
    for (size_t q = 0; q < in.src_list->size(); q++)
        o << "        source_step_one(pg, w, " << q << ", " << (*in.src_list)[q] << ", "
          << ((*in.src_uniform)[q] ? "true" : "false") << ", k, first, t0, h, mode);\n";
    o << "    }\n";
    o << "};\n";
    emit_lu(o, "SLuDc", st, p, *in.lu_dc);
    emit_lu(o, "SLuTr", st, p, *in.lu_tr);
    o << "constexpr int kSlots = " << p.n_slots_w << ";\n";
    o << "constexpr int kBlock = " << in.block << ";\nconstexpr int kMinBlocks = " << in.min_blocks << ";\n";
    o << "__global__ void __launch_bounds__(kBlock, kMinBlocks) cb200_spec_dc_kernel(Program p, SpecArgs sp, DcArgs a)\n"
         "{\n    SProg pg; SLuDc lu; RegWs<kSlots> w;\n    dc_body(pg, lu, w, p, sp, a);\n}\n";
    o << "__global__ void __launch_bounds__(kBlock, kMinBlocks) cb200_spec_tran_fixed_kernel(Program p, SpecArgs sp, TranArgs a)\n"
         "{\n    SProg pg; SLuTr lu; RegWs<kSlots> w;\n    tran_fixed_body(pg, lu, w, p, sp, a);\n}\n";
    if (in.with_adaptive)
        o << "__global__ void __launch_bounds__(kBlock, kMinBlocks) cb200_spec_tran_adaptive_kernel(Program p, SpecArgs sp, AdaptArgs a)\n"
             "{\n    SProg pg; SLuTr lu; RegWs<kSlots> w;\n    tran_adaptive_body(pg, lu, w, p, sp, a);\n}\n";
    o << "}  // namespace\n";
    o << "extern \"C\" int cb200_spec_abi(void) { return " << kSpecAbi << "; }\n";
    o << "extern \"C\" int cb200_spec_block(void) { return kBlock; }\n";
    o << "extern \"C\" cudaError_t cb200_spec_dc(const cb200::Program *p, const cb200::SpecArgs *s,\n"
         "                                     const cb200::DcArgs *a, cudaStream_t st)\n{\n"
         "    const unsigned grid = (unsigned)((p->P + kBlock - 1) / kBlock);\n"
         "    cb200_spec_dc_kernel<<<grid, kBlock, 0, st>>>(*p, *s, *a);\n    return cudaGetLastError();\n}\n";
    o << "extern \"C\" cudaError_t cb200_spec_tran_fixed(const cb200::Program *p, const cb200::SpecArgs *s,\n"
         "                                             const cb200::TranArgs *a, cudaStream_t st)\n{\n"
         "    const unsigned grid = (unsigned)((p->P + kBlock - 1) / kBlock);\n"
         "    cb200_spec_tran_fixed_kernel<<<grid, kBlock, 0, st>>>(*p, *s, *a);\n    return cudaGetLastError();\n}\n";
    if (bypass)
        o << "// lane-steps the fixed-step kernels executed since the last call (then reset): the bypass makes it less than\n"
             "// steps x lanes, and the FP64 roofline counts one assembly per EXECUTED step\n"
             "extern \"C\" cudaError_t cb200_spec_take_counters(unsigned long long *executed, cudaStream_t st)\n{\n"
             "    unsigned long long v = 0, zero = 0;\n"
             "    cudaError_t e = cudaMemcpyFromSymbolAsync(&v, cb200_spec_nexec, sizeof v, 0, cudaMemcpyDeviceToHost, st);\n"
             "    if (e == cudaSuccess) e = cudaMemcpyToSymbolAsync(cb200_spec_nexec, &zero, sizeof zero, 0, cudaMemcpyHostToDevice, st);\n"
             "    if (e == cudaSuccess) e = cudaStreamSynchronize(st);\n"
             "    if (executed) *executed = v;\n    return e;\n}\n";
    if (in.with_adaptive)
    o << "extern \"C\" cudaError_t cb200_spec_tran_adaptive(const cb200::Program *p, const cb200::SpecArgs *s,\n"
         "                                                const cb200::AdaptArgs *a, cudaStream_t st)\n{\n"
         "    const unsigned grid = (unsigned)((p->P + kBlock - 1) / kBlock);\n"
         "    cb200_spec_tran_adaptive_kernel<<<grid, kBlock, 0, st>>>(*p, *s, *a);\n    return cudaGetLastError();\n}\n";
    g_data = nullptr;
    return head.str() + data.str() + o.str();
}

static uint64_t fnv1a(uint64_t h, const std::string &s)
{
    for (unsigned char c : s) { h ^= c; h *= 1099511628211ULL; }
    return h;
}

static std::string slurp(const std::string &path)
{
    std::ifstream f(path, std::ios::binary);
    std::ostringstream ss;
    ss << f.rdbuf();
    return ss.str();
}

static bool exists(const std::string &p)
{
    struct stat sb;
    return stat(p.c_str(), &sb) == 0;
}

static std::string find_nvcc()
{
    const char *env = getenv("CB200_NVCC");
    if (env && exists(env)) return env;
    if (exists("/usr/local/cuda/bin/nvcc")) return "/usr/local/cuda/bin/nvcc";
    return "nvcc";
}

// Generated modules stay mapped until the process exits: a handle that is done with one merely
// forgets it.  (dlopen of a path that is already loaded returns the same mapping, so reloading is
// free; and a driver that lists the shared objects of the process after the run sees every kernel
// module that executed, not only libcadnip_b200.so.)
static void *open_module(const std::string &path)
{
    return dlopen(path.c_str(), RTLD_NOW | RTLD_LOCAL | RTLD_NODELETE);
}

void unload_kernel_set(KernelSet &k)
{
    k = KernelSet();
}

// Cache key of a kernel set: the emitted header, the sources it is rebuilt from, and CB200_NVCC_FLAGS
// (extra compiler flags, e.g. -Xptxas -O1).
static std::string va_kernel_set_keys(const std::string &va_header_text, const std::string &csrc_dir,
                                      std::string &hdr_hex, std::string &so_hex, std::string &extra)
{
    uint64_t h = 1469598103934665603ULL;
    h = fnv1a(h, va_header_text);
    char hex[32];
    snprintf(hex, sizeof hex, "%016llx", (unsigned long long)h);
    hdr_hex = hex;
    uint64_t hk = h;
    for (const char *f : {"/kernels.cu", "/lane_kernels.cuh", "/warp_kernels.cuh", "/group_kernels.inc", "/kernels.h", "/../../include/cadnip_b200.h"}) {
        std::string body = slurp(csrc_dir + f);
        if (body.empty()) return "va models: cannot read " + csrc_dir + f;
        hk = fnv1a(hk, body);
    }
    const char *extra_env = getenv("CB200_NVCC_FLAGS");
    extra = extra_env ? extra_env : "";
    // Giant models (PSP103: 9 MB of emitted CUDA, sp_bsim4v8: 14 MB): ptxas at its default -O3 needs hours
    // and tens of GB on functions of 1e5 statements (measured: > 80 minutes for PSP103, not finished), so
    // their kernel sets are assembled at -O1.  Part of the cache key like any other flag.
    if (va_header_text.size() > (size_t)(4 << 20) && extra.find("-Xptxas") == std::string::npos) extra += " -Xptxas -O1";
    hk = fnv1a(hk, extra);
    snprintf(hex, sizeof hex, "%016llx", (unsigned long long)hk);
    so_hex = hex;
    return "";
}

bool va_kernel_set_cached(const std::string &va_header_text, const std::string &csrc_dir, const std::string &cache_dir)
{
    std::string hdr_hex, so_hex, extra;
    if (!va_kernel_set_keys(va_header_text, csrc_dir, hdr_hex, so_hex, extra).empty()) return false;
    return exists(cache_dir + "/kern_" + so_hex + ".so");
}

std::string build_va_kernel_set(const std::string &va_header_text, const std::string &csrc_dir,
                                const std::string &cache_dir, KernelSet &out)
{
    std::string hdr_hex, so_hex, extra;
    std::string ke = va_kernel_set_keys(va_header_text, csrc_dir, hdr_hex, so_hex, extra);
    if (!ke.empty()) return ke;
    mkdir(cache_dir.c_str(), 0755);
    const std::string hdr = cache_dir + "/va_" + hdr_hex + ".cuh";
    if (!exists(hdr)) {
        const std::string tmp = hdr + ".tmp" + std::to_string((long)getpid());
        { std::ofstream f(tmp); f << va_header_text; if (!f) return "va models: cannot write " + tmp; }
        if (rename(tmp.c_str(), hdr.c_str()) != 0) return "va models: cannot move " + tmp;
    }
    const char *hex = so_hex.c_str();
    const std::string so = cache_dir + "/kern_" + hex + ".so", log = cache_dir + "/kern_" + hex + ".log";
    if (!exists(so)) {
        const std::string tmp = cache_dir + "/kern_" + hex + ".tmp" + std::to_string((long)getpid()) + ".so";
        // giant models: ptxas works on the kernels in parallel (measured on sp_bsim4v8: 14.5 -> 10 min; the serial
        // front end is the rest).  Not part of the cache key: it does not change what is compiled.
        const std::string par = va_header_text.size() > (size_t)(4 << 20) ? " -split-compile 0" : "";
        std::string cmd = find_nvcc() + " -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 "
                          "-Xcompiler -fPIC -shared " + extra + par + " -DCB200_VA_HEADER='\"" + hdr + "\"' -I\"" + csrc_dir +
                          "\" -o \"" + tmp + "\" \"" + csrc_dir + "/kernels.cu\" > \"" + log + "\" 2>&1";
        if (system(cmd.c_str()) != 0) {
            std::string l = slurp(log);
            if (l.size() > 3000) l = l.substr(l.size() - 3000);
            return "va models: nvcc failed (" + cmd + "):\n" + l;
        }
        if (rename(tmp.c_str(), so.c_str()) != 0) return "va models: cannot move " + tmp;
    }
    void *dl = open_module(so);
    if (!dl) return std::string("va models: dlopen failed: ") + dlerror();
    out.eval = (k_eval_fn)dlsym(dl, "cb200_k_eval");
    out.dc = (k_dc_fn)dlsym(dl, "cb200_k_dc");
    out.tran_fixed = (k_tran_fn)dlsym(dl, "cb200_k_tran_fixed");
    out.tran_adaptive = (k_adapt_fn)dlsym(dl, "cb200_k_tran_adaptive");
    if (!out.eval || !out.dc || !out.tran_fixed || !out.tran_adaptive) {
        out = KernelSet();
        return "va models: " + so + " does not export the kernel entry points";
    }
    out.dl = dl;
    out.va_header_path = hdr;
    return "";
}

void unload_spec(SpecModule &m)
{
    m = SpecModule();
}

std::string build_and_load_spec(const std::string &src, const std::string &csrc_dir,
                                const std::string &cache_dir, bool compile_only, SpecModule &out)
{
    uint64_t h = 1469598103934665603ULL;
    h = fnv1a(h, src);
    for (const char *f : {"/lane_kernels.cuh", "/kernels.h", "/../../include/cadnip_b200.h"}) {
        std::string body = slurp(csrc_dir + f);
        if (body.empty()) return "specialize: cannot read " + csrc_dir + f;
        h = fnv1a(h, body);
    }
    char hex[32];
    snprintf(hex, sizeof hex, "%016llx", (unsigned long long)h);
    mkdir(cache_dir.c_str(), 0755);
    const std::string base = cache_dir + "/spec_" + hex;
    const std::string so = base + ".so", cu = base + ".cu", log = base + ".log";
    if (!exists(so)) {
        {
            std::ofstream f(cu);
            f << src;
            if (!f) return "specialize: cannot write " + cu;
        }
        const std::string tmp = base + ".tmp" + std::to_string((long)getpid()) + ".so";
        std::string cmd = find_nvcc() + " -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 "
                          "-Xcompiler -fPIC -shared -Xptxas -v -I\"" + csrc_dir + "\" -o \"" + tmp + "\" \"" + cu +
                          "\" > \"" + log + "\" 2>&1";
        int rc = system(cmd.c_str());
        if (rc != 0) {
            std::string l = slurp(log);
            if (l.size() > 2000) l = l.substr(l.size() - 2000);
            return "specialize: nvcc failed (" + cmd + "):\n" + l;
        }
        if (rename(tmp.c_str(), so.c_str()) != 0) return "specialize: cannot move " + tmp;
    }
    out.path = so;
    if (compile_only) return "";
    void *dl = open_module(so);
    if (!dl) return std::string("specialize: dlopen failed: ") + dlerror();
    typedef int (*int_fn)(void);
    int_fn abi = (int_fn)dlsym(dl, "cb200_spec_abi");
    int_fn blk = (int_fn)dlsym(dl, "cb200_spec_block");
    out.dc = (spec_dc_fn)dlsym(dl, "cb200_spec_dc");
    out.tran_fixed = (spec_tran_fn)dlsym(dl, "cb200_spec_tran_fixed");
    out.tran_adaptive = (spec_adapt_fn)dlsym(dl, "cb200_spec_tran_adaptive");
    out.take_counters = (spec_counters_fn)dlsym(dl, "cb200_spec_take_counters");      // optional
    if (!abi || !blk || !out.dc || !out.tran_fixed || abi() != kSpecAbi) {       // tran_adaptive is optional
        out = SpecModule();
        return "specialize: " + so + " does not export the expected entry points";
    }
    out.dl = dl;
    out.block = blk();
    return "";
}

}  // namespace cb200
