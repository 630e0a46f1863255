// api.cu -- C ABI of libcadnip_b200.so (include/cadnip_b200.h).
//
// Host side of the B200 path: owns the device copies of the circuit program, the
// lane-parameter SoA and the lane state, runs the host symbolic phase, launches
// the kernels on the handle's own stream and times them with CUDA events.  There
// is no CPU fallback: every numerical entry point fails with CB200_ENODEVICE when
// no CUDA device is usable.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "cb200_internal.h"
#include "kernels.h"
#include "specialize.h"

using namespace cb200;

static thread_local std::string g_last_error;

namespace {

// Cache of device allocations shared by a handle and the waves it produced: the
// waveform buffers of a sweep are large (O(100 MB)) and cudaMalloc / cudaFree of that
// size cost milliseconds and serialise against every other driver call, so buffers
// are recycled by exact size instead of being returned to the driver.
struct BufPool {
    int device = 0;
    std::mutex mu;
    std::multimap<size_t, void *> free_;
    size_t cached_bytes = 0;
    // cap of the cache: 1 GiB unless CB200_POOL_MAX_MB says otherwise (a second handle on the same
    // GPU must not be starved by buffers this one only keeps for reuse)
    size_t kMaxCached = (size_t)1 << 30;
    BufPool()
    {
        if (const char *e = getenv("CB200_POOL_MAX_MB")) kMaxCached = (size_t)std::max(0, atoi(e)) << 20;
    }
    cudaError_t get(size_t bytes, void **out)
    {
        {
            std::lock_guard<std::mutex> g(mu);
            auto it = free_.find(bytes);
            if (it != free_.end()) {
                *out = it->second;
                cached_bytes -= bytes;
                free_.erase(it);
                return cudaSuccess;
            }
        }
        cudaError_t e = cudaMalloc(out, bytes);
        if (e != cudaSuccess) {              // out of memory: drop EVERY pool's cache and retry once
            trim_all_pools();
            cudaGetLastError();
            e = cudaMalloc(out, bytes);
        }
        return e;
    }
    static void trim_all_pools();
    void put(void *p, size_t bytes)
    {
        std::lock_guard<std::mutex> g(mu);
        free_.emplace(bytes, p);
        cached_bytes += bytes;
        while (cached_bytes > kMaxCached && !free_.empty()) {
            auto it = --free_.end();
            cudaFree(it->second);
            cached_bytes -= it->first;
            free_.erase(it);
        }
    }
    void trim(size_t keep)
    {
        std::lock_guard<std::mutex> g(mu);
        while (cached_bytes > keep && !free_.empty()) {
            auto it = --free_.end();
            cudaFree(it->second);
            cached_bytes -= it->first;
            free_.erase(it);
        }
    }
    ~BufPool()
    {
        cudaSetDevice(device);
        for (auto &kv : free_) cudaFree(kv.second);
    }
};

// live pools of the process (weak: a pool dies with its handle and its last wave)
static std::mutex g_pools_mu;
static std::vector<std::weak_ptr<BufPool>> g_pools;

void BufPool::trim_all_pools()
{
    std::vector<std::shared_ptr<BufPool>> live;
    {
        std::lock_guard<std::mutex> g(g_pools_mu);
        for (auto it = g_pools.begin(); it != g_pools.end();) {
            if (auto sp = it->lock()) { live.push_back(sp); ++it; }
            else it = g_pools.erase(it);
        }
    }
    int cur = 0;
    cudaGetDevice(&cur);
    for (auto &p : live) { cudaSetDevice(p->device); p->trim(0); }
    cudaSetDevice(cur);
}

template <typename T>
struct DevBuf {
    T *p = nullptr;
    size_t n = 0;
    std::shared_ptr<BufPool> pool;           // optional
    cudaError_t alloc(size_t count)
    {
        release();
        n = count;
        if (count == 0) return cudaSuccess;
        if (pool) return pool->get(count * sizeof(T), (void **)&p);
        return cudaMalloc((void **)&p, count * sizeof(T));
    }
    cudaError_t upload(const std::vector<T> &v, cudaStream_t st)
    {
        cudaError_t e = alloc(v.size());
        if (e != cudaSuccess || v.empty()) return e;
        return cudaMemcpyAsync(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, st);
    }
    void release()
    {
        if (p) {
            if (pool) pool->put(p, n * sizeof(T));
            else cudaFree(p);
        }
        p = nullptr; n = 0;
    }
    ~DevBuf() { release(); }
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
};

struct DevLu {
    LuSchedule host;
    DevBuf<int> rowperm, colperm, diag_slot, Lptr, L_slot, L_row, Uptr, U_slot, U_col, tgt_ptr, tgt,
        jmap, fill_slots;
    LevelSchedule lvl;
    DevBuf<int> piv_ptr, sc_ptr, tg_ptr, piv, sc, tg, upd, flev_ptr, frow, fent, blev_ptr, brow, bent;
    LuProgram prog{};
};

}  // namespace

struct cb200_handle {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::string err;
    Structure st;
    // host copies of the description
    std::vector<int> dev_kind, dev_flags, dev_node_ptr, dev_nodes, dev_param_ptr, dev_params;
    std::vector<int> dev_gbase, dev_cbase, dev_bbase, dev_sbase, src_list, nl_list, limit_init_ref;
    std::vector<unsigned char> src_uniform;
    std::vector<double> uniform;
    int n_lane_cols = 0;
    // lanes
    int64_t P = 0;
    std::vector<double> lanes_host;
    // device copies
    DevBuf<int> d_dev_kind, d_dev_flags, d_dev_node_ptr, d_dev_nodes, d_dev_param_ptr, d_dev_params;
    DevBuf<int> d_dev_gbase, d_dev_cbase, d_dev_bbase, d_dev_sbase, d_src_list, d_nl_list, d_limit_init_ref;
    DevBuf<int> d_gseg_ptr, d_gseg_idx, d_cseg_ptr, d_cseg_idx, d_bseg_ptr, d_bseg_idx;
    DevBuf<int> d_colptr, d_rowval, d_rowptr, d_row_nz, d_nz_col;
    DevBuf<unsigned char> d_node_diag, d_src_uniform;
    DevBuf<double> d_uniform, d_lanes;
    DevBuf<double> d_state;        // [n][P]
    DevBuf<double> d_ws_global;    // [n_slots][P] (eval path / shared-memory overflow)
    DevBuf<int> d_status, d_iters;
    DevBuf<int> d_weak;            // [P] weak-pivot marks of the last cb200_dc / cb200_tran (lane_kernels.cuh: weak_pivot)
    DevBuf<unsigned char> d_conv, d_active;
    DevBuf<double> d_gshunt_lane, d_srcfact_lane;
    DevBuf<int> d_save, d_rejected, d_evals;
    DevBuf<double> d_hist;         // [2n][P] integrator history between time segments
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t seg_ev[16] = {};
    std::vector<double> tstops;    // sorted breakpoints for adaptive stepping
    DevBuf<double> d_tstops;
    std::shared_ptr<BufPool> pool;  // recycled waveform buffers (shared with live waves)
    Program prog{};
    DevLu lu[2];                   // 0: DC (gamma = 0), 1: transient
    int lu_gen[2] = {0, 0};        // bumped by every (re-)analysis
    KernelSet k;                   // table-driven kernels: built-in, or rebuilt with VA models
    bool has_va = false;
    SpecModule spec;               // circuit-specialised kernels (optional)
    int spec_gen[2] = {-1, -1};    // schedule generations the module was generated from
    int spec_method = -1;          // integration method baked into the transient kernel
    bool spec_limit = false;       // transient kernels were generated with the CB200_TRAN_LIMIT path
    int num_sms = 148;
    size_t smem_limit = 0;
    int block_pref = 64;
    cb200_stats stats{};
    std::vector<cb200_wave *> waves;   // live waves: orphaned (buffers released) by cb200_destroy
};

struct cb200_wave {
    cb200_handle *h = nullptr;     // null once the handle was destroyed: every accessor then fails with CB200_ESTATE
    int64_t T = 0, P = 0;
    int n_save = 0, adaptive = 0, n = 0;
    double t0 = 0, dt = 0;
    int save_every = 1;
    int64_t nsteps = 0;
    DevBuf<double> d_out, d_t, d_final;
    DevBuf<int> d_count, d_status, d_iters;
};

#define CUDA_TRY(h, expr)                                                              \
    do {                                                                               \
        cudaError_t _e = (expr);                                                       \
        if (_e != cudaSuccess) {                                                       \
            (h)->err = std::string(#expr) + ": " + cudaGetErrorString(_e);             \
            g_last_error = (h)->err;                                                   \
            return CB200_ECUDA;                                                        \
        }                                                                              \
    } while (0)

static int fail(cb200_handle *h, int code, const std::string &msg)
{
    if (h) h->err = msg;
    g_last_error = msg;
    return code;
}

static std::vector<int> to_int(const int32_t *p, size_t n) { return std::vector<int>(p, p + n); }
static std::vector<int> to_int64(const int64_t *p, size_t n)
{
    std::vector<int> v(n);
    for (size_t i = 0; i < n; i++) v[i] = (int)p[i];
    return v;
}

static SpecArgs spec_args(const cb200_spec *s)
{
    SpecArgs a;
    a.mode = s->mode; a.temp = s->temp; a.gmin = s->gmin; a.gshunt = s->gshunt; a.srcFact = s->srcFact;
    return a;
}

// workspace slot layout of one lane
static void layout_workspace(cb200_handle *h)
{
    Program &p = h->prog;
    int o = 0;
    const int n = h->st.n;
    p.off_u = o; o += n;
    p.off_un = o; o += n;
    p.off_dterm = o; o += n;
    p.off_F = o; o += n;
    p.off_wv = o; o += n;
    p.off_SG = o; o += (int)h->st.nG;
    p.off_SC = o; o += (int)h->st.nC;
    p.off_SB = o; o += (int)h->st.nb;
    p.off_limw = o; o += h->st.n_limits;
    p.off_lp = o; o += h->n_lane_cols;
    p.off_DS = o; o += h->dev_sbase.empty() ? 0 : h->dev_sbase.back();
    p.off_srcc = o; o += (int)h->src_list.size();
    p.off_h1 = o; o += n;
    p.off_h2 = o; o += n;
    p.off_phi = o; o += 6 * n;
    p.off_LU = o;                       // LU last: its size depends on the schedule
    int64_t nlu = std::max(h->lu[0].host.nlu, h->lu[1].host.nlu);
    if (nlu == 0) nlu = h->st.nnz;
    o += (int)nlu;
    p.n_slots = o;
    // lane-per-warp kernels: per-entry sums and reciprocal pivots behind the common layout;
    // a lane's row is padded to a whole number of 128-byte lines
    p.off_GS = o; o += (int)h->st.nnz;
    p.off_CS = o; o += (int)h->st.nnz;
    p.off_DI = o; o += n;
    p.n_slots_w = (o + 15) / 16 * 16;
}

// the lane workspace lives in global memory (lane-per-warp kernels, or shared-memory overflow)
static bool needs_global_ws(const cb200_handle *h)
{
    return use_warp_kernels(h->prog.n_slots, h->smem_limit, h->block_pref) ||
           choose_block(h->prog.n_slots, h->smem_limit, h->block_pref) == 0;
}

// devices whose stamps depend on time only (evaluated once per time step) ...
static bool is_source_kind(int kind) { return kind == CB200_DEV_VSOURCE || kind == CB200_DEV_ISOURCE; }
// ... and on the iterate (evaluated every Newton iteration)
static bool is_nonlinear_kind(int kind)
{
    return kind == CB200_DEV_DIODE || kind == CB200_DEV_DIODECAP || kind == CB200_DEV_SIMPLEMOS ||
           kind == CB200_DEV_VA;
}

extern "C" int cb200_abi_version(void) { return CB200_ABI_VERSION; }

extern "C" const char *cb200_last_error(const cb200_handle *h)
{
    return h ? h->err.c_str() : g_last_error.c_str();
}

extern "C" int cb200_create(const cb200_desc *d, int32_t device, cb200_handle **out)
{
    if (!d || !out) return fail(nullptr, CB200_EINVAL, "cb200_create: null argument");
    *out = nullptr;
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0 || device < 0 || device >= ndev)
        return fail(nullptr, CB200_ENODEVICE,
                    std::string("cb200_create: no usable CUDA device (there is no CPU fallback): ") +
                        (ce != cudaSuccess ? cudaGetErrorString(ce) : "device ordinal out of range"));
    cb200_handle *h = new cb200_handle();
    h->device = device;
    h->k.eval = cb200_k_eval; h->k.dc = cb200_k_dc;
    h->k.tran_fixed = cb200_k_tran_fixed; h->k.tran_adaptive = cb200_k_tran_adaptive;
    h->pool = std::make_shared<BufPool>();
    h->pool->device = device;
    {
        std::lock_guard<std::mutex> g(g_pools_mu);
        g_pools.push_back(h->pool);
    }
    ce = cudaSetDevice(device);
    if (ce != cudaSuccess) { delete h; return fail(nullptr, CB200_ECUDA, cudaGetErrorString(ce)); }
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    if (prop.major < 10) {
        std::string m = "cb200_create: device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor) +
                        "; this library is built for sm_100a only";
        delete h;
        return fail(nullptr, CB200_ENODEVICE, m);
    }
    h->smem_limit = prop.sharedMemPerBlockOptin;
    h->num_sms = prop.multiProcessorCount;
    std::string e = build_structure(*d, h->st);
    if (!e.empty()) { delete h; return fail(nullptr, CB200_EINVAL, e); }

    const int nd = d->n_devices;
    for (int i = 0; i < nd; i++)
        if (d->dev_kind[i] < 1 || d->dev_kind[i] > CB200_DEV_KIND_MAX) {
            delete h;
            return fail(nullptr, CB200_EINVAL, "cb200_create: unknown device kind");
        }
    h->dev_kind = to_int(d->dev_kind, nd);
    for (int kd : h->dev_kind) h->has_va |= (kd == CB200_DEV_VA);
    h->dev_flags = to_int(d->dev_flags, nd);
    h->dev_node_ptr = to_int(d->dev_node_ptr, nd + 1);
    h->dev_nodes = to_int(d->dev_nodes, nd ? d->dev_node_ptr[nd] : 0);
    h->dev_param_ptr = to_int(d->dev_param_ptr, nd + 1);
    h->dev_params = to_int(d->dev_params, nd ? d->dev_param_ptr[nd] : 0);
    h->dev_gbase = to_int64(d->dev_gbase, nd + 1);
    h->dev_cbase = to_int64(d->dev_cbase, nd + 1);
    h->dev_bbase = to_int64(d->dev_bbase, nd + 1);
    h->dev_sbase = d->dev_state_ptr ? to_int(d->dev_state_ptr, nd + 1) : std::vector<int>(nd + 1, 0);
    h->uniform.assign(d->uniform, d->uniform + d->n_uniform);
    h->limit_init_ref = to_int(d->limit_init_ref, d->n_limits);
    h->n_lane_cols = d->n_lane_cols;
    for (int r : h->dev_params)
        if (r >= d->n_uniform || (r < 0 && ~r >= d->n_lane_cols)) {
            delete h;
            return fail(nullptr, CB200_EINVAL, "cb200_create: parameter reference out of range");
        }
    for (int v : h->dev_nodes)
        if (v < 0 || v > h->st.n) {
            delete h;
            return fail(nullptr, CB200_EINVAL, "cb200_create: device node index out of range");
        }
    for (int i = 0; i < nd; i++) {
        if (is_source_kind(h->dev_kind[i])) {
            h->src_list.push_back(i);
            bool uni = true;
            for (int q = h->dev_param_ptr[i]; q < h->dev_param_ptr[i + 1]; q++) uni &= h->dev_params[q] >= 0;
            h->src_uniform.push_back(uni ? 1 : 0);
        }
        if (is_nonlinear_kind(h->dev_kind[i])) h->nl_list.push_back(i);
    }

    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&h->ev0) != cudaSuccess || cudaEventCreate(&h->ev1) != cudaSuccess) {
        delete h;
        return fail(nullptr, CB200_ECUDA, "cb200_create: stream/event creation failed");
    }
    cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking);
    for (auto &e : h->seg_ev) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    cudaStream_t s = h->stream;
    const Structure &st = h->st;
    std::vector<unsigned char> nd8(st.nz_is_node_diag.begin(), st.nz_is_node_diag.end());
    // CSR view of the CSC pattern for the row-parallel residual of the lane-per-warp kernels:
    // a counting sort over columns in ascending order leaves every row's entries column-sorted
    std::vector<int> rowptr(st.n + 1, 0), row_nz(st.nnz), nz_col(st.nnz);
    for (int64_t q = 0; q < st.nnz; q++) rowptr[st.rowval[q] + 1]++;
    for (int r = 0; r < st.n; r++) rowptr[r + 1] += rowptr[r];
    {
        std::vector<int> fillp(rowptr.begin(), rowptr.end() - 1);
        for (int j = 0; j < st.n; j++)
            for (int q = st.colptr[j]; q < st.colptr[j + 1]; q++) {
                nz_col[q] = j;
                row_nz[fillp[st.rowval[q]]++] = q;
            }
    }
    bool ok = h->d_dev_kind.upload(h->dev_kind, s) == cudaSuccess &&
              h->d_dev_flags.upload(h->dev_flags, s) == cudaSuccess &&
              h->d_dev_node_ptr.upload(h->dev_node_ptr, s) == cudaSuccess &&
              h->d_dev_nodes.upload(h->dev_nodes, s) == cudaSuccess &&
              h->d_dev_param_ptr.upload(h->dev_param_ptr, s) == cudaSuccess &&
              h->d_dev_params.upload(h->dev_params, s) == cudaSuccess &&
              h->d_dev_gbase.upload(h->dev_gbase, s) == cudaSuccess &&
              h->d_dev_cbase.upload(h->dev_cbase, s) == cudaSuccess &&
              h->d_dev_bbase.upload(h->dev_bbase, s) == cudaSuccess &&
              h->d_dev_sbase.upload(h->dev_sbase, s) == cudaSuccess &&
              h->d_src_list.upload(h->src_list, s) == cudaSuccess &&
              h->d_nl_list.upload(h->nl_list, s) == cudaSuccess &&
              h->d_src_uniform.upload(h->src_uniform, s) == cudaSuccess &&
              h->d_limit_init_ref.upload(h->limit_init_ref, s) == cudaSuccess &&
              h->d_uniform.upload(h->uniform, s) == cudaSuccess &&
              h->d_gseg_ptr.upload(st.gseg_ptr, s) == cudaSuccess &&
              h->d_gseg_idx.upload(st.gseg_idx, s) == cudaSuccess &&
              h->d_cseg_ptr.upload(st.cseg_ptr, s) == cudaSuccess &&
              h->d_cseg_idx.upload(st.cseg_idx, s) == cudaSuccess &&
              h->d_bseg_ptr.upload(st.bseg_ptr, s) == cudaSuccess &&
              h->d_bseg_idx.upload(st.bseg_idx, s) == cudaSuccess &&
              h->d_colptr.upload(st.colptr, s) == cudaSuccess &&
              h->d_rowval.upload(st.rowval, s) == cudaSuccess &&
              h->d_rowptr.upload(rowptr, s) == cudaSuccess &&
              h->d_row_nz.upload(row_nz, s) == cudaSuccess &&
              h->d_nz_col.upload(nz_col, s) == cudaSuccess &&
              h->d_node_diag.upload(nd8, s) == cudaSuccess;
    if (!ok || cudaStreamSynchronize(s) != cudaSuccess) {
        std::string m = std::string("cb200_create: upload failed: ") + cudaGetErrorString(cudaGetLastError());
        cb200_destroy(h);
        return fail(nullptr, CB200_ECUDA, m);
    }
    Program &p = h->prog;
    p.n = st.n; p.n_nodes = st.n_nodes; p.n_limits = st.n_limits; p.nnz = (int)st.nnz;
    p.nG = (int)st.nG; p.nC = (int)st.nC; p.nb = (int)st.nb; p.n_dev = nd;
    p.n_src = (int)h->src_list.size(); p.n_nl = (int)h->nl_list.size();
    p.n_lane_cols = h->n_lane_cols; p.P = 0;
    p.dev_kind = h->d_dev_kind.p; p.dev_flags = h->d_dev_flags.p;
    p.dev_node_ptr = h->d_dev_node_ptr.p; p.dev_nodes = h->d_dev_nodes.p;
    p.dev_param_ptr = h->d_dev_param_ptr.p; p.dev_params = h->d_dev_params.p;
    p.dev_gbase = h->d_dev_gbase.p; p.dev_cbase = h->d_dev_cbase.p; p.dev_bbase = h->d_dev_bbase.p;
    p.dev_sbase = h->d_dev_sbase.p;
    p.src_list = h->d_src_list.p; p.nl_list = h->d_nl_list.p; p.src_uniform = h->d_src_uniform.p;
    p.uniform = h->d_uniform.p; p.lanes = nullptr;
    p.limit_init_ref = h->d_limit_init_ref.p;
    p.gseg_ptr = h->d_gseg_ptr.p; p.gseg_idx = h->d_gseg_idx.p;
    p.cseg_ptr = h->d_cseg_ptr.p; p.cseg_idx = h->d_cseg_idx.p;
    p.bseg_ptr = h->d_bseg_ptr.p; p.bseg_idx = h->d_bseg_idx.p;
    p.colptr = h->d_colptr.p; p.rowval = h->d_rowval.p; p.nz_is_node_diag = h->d_node_diag.p;
    p.rowptr = h->d_rowptr.p; p.row_nz = h->d_row_nz.p; p.nz_col = h->d_nz_col.p;
    layout_workspace(h);
    *out = h;
    return CB200_OK;
}

extern "C" void cb200_destroy(cb200_handle *h)
{
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->stream) cudaStreamDestroy(h->stream);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    for (auto &e : h->seg_ev) if (e) cudaEventDestroy(e);
    for (cb200_wave *w : h->waves) {     // waves the caller still holds: free their device memory now
        w->d_out.release(); w->d_t.release(); w->d_final.release();
        w->d_count.release(); w->d_status.release(); w->d_iters.release();
        w->h = nullptr;
    }
    h->waves.clear();
    unload_spec(h->spec);
    if (h->k.dl) unload_kernel_set(h->k);
    delete h;
}

extern "C" int cb200_get_pattern(const cb200_handle *h, int64_t *n, int64_t *nnz, int64_t *colptr,
                                 int64_t *rowval)
{
    if (!h) return CB200_EINVAL;
    if (n) *n = h->st.n;
    if (nnz) *nnz = h->st.nnz;
    if (colptr) for (int j = 0; j <= h->st.n; j++) colptr[j] = h->st.colptr[j] + 1;
    if (rowval) for (int64_t q = 0; q < h->st.nnz; q++) rowval[q] = h->st.rowval[q] + 1;
    return CB200_OK;
}

extern "C" int cb200_get_maps(const cb200_handle *h, int64_t *G_map, int64_t *C_map, int64_t *b_rows,
                              int64_t *G_diag)
{
    if (!h) return CB200_EINVAL;
    if (G_map) for (int64_t k = 0; k < h->st.nG; k++) G_map[k] = h->st.G_map[k] + 1;
    if (C_map) for (int64_t k = 0; k < h->st.nC; k++) C_map[k] = h->st.C_map[k] + 1;
    if (b_rows) for (int64_t k = 0; k < h->st.nb; k++) b_rows[k] = h->st.b_rows[k] + 1;
    if (G_diag) for (int i = 0; i < h->st.n_nodes; i++) G_diag[i] = h->st.diag_nz[i] + 1;   // 0 = absent
    return CB200_OK;
}

static int ensure_lane_buffers(cb200_handle *h)
{
    const int64_t P = h->P;
    const int n = h->st.n;
    if (h->d_state.n != (size_t)n * P) CUDA_TRY(h, h->d_state.alloc((size_t)n * P));
    if (h->d_status.n != (size_t)P) {
        CUDA_TRY(h, h->d_status.alloc(P));
        CUDA_TRY(h, h->d_iters.alloc(P));
        CUDA_TRY(h, h->d_weak.alloc(P));
        CUDA_TRY(h, h->d_conv.alloc(P));
        CUDA_TRY(h, h->d_active.alloc(P));
        CUDA_TRY(h, h->d_gshunt_lane.alloc(P));
        CUDA_TRY(h, h->d_srcfact_lane.alloc(P));
    }
    return CB200_OK;
}

static int ensure_global_ws(cb200_handle *h)
{
    // lane-per-thread kernels: [n_slots][P padded to the block (64)]; lane-per-warp: [P][n_slots_w]
    const size_t need = (size_t)std::max(h->prog.n_slots, h->prog.n_slots_w) * ((h->P + 63) / 64 * 64);
    if (h->d_ws_global.n < need) CUDA_TRY(h, h->d_ws_global.alloc(need));
    return CB200_OK;
}

extern "C" int cb200_set_lanes(cb200_handle *h, int64_t P, int32_t n_cols, const double *soa)
{
    if (!h || P <= 0) return fail(h, CB200_EINVAL, "cb200_set_lanes: bad arguments");
    if (n_cols != h->n_lane_cols) return fail(h, CB200_EINVAL, "cb200_set_lanes: column count differs from the description");
    if (n_cols > 0 && !soa) return fail(h, CB200_EINVAL, "cb200_set_lanes: null SoA");
    cudaSetDevice(h->device);
    // New parameter values: the static pivot order was chosen from magnitudes probed on the OLD
    // lanes, so both schedules are re-analysed on next use (re-sending identical values, e.g. a
    // per-step H2D refresh, keeps them -- and the kernels specialised for them).
    const size_t cnt = (size_t)n_cols * P;
    if (P != h->P || h->lanes_host.size() != cnt ||
        (cnt > 0 && memcmp(h->lanes_host.data(), soa, cnt * sizeof(double)) != 0)) {
        h->lu[0].host.valid = false;
        h->lu[1].host.valid = false;
    }
    h->P = P;
    h->prog.P = P;
    h->lanes_host.assign(soa, soa + cnt);
    if (n_cols > 0) {
        if (h->d_lanes.n != (size_t)n_cols * P) CUDA_TRY(h, h->d_lanes.alloc((size_t)n_cols * P));
        CUDA_TRY(h, cudaEventRecord(h->ev0, h->stream));
        CUDA_TRY(h, cudaMemcpyAsync(h->d_lanes.p, soa, (size_t)n_cols * P * sizeof(double),
                                    cudaMemcpyHostToDevice, h->stream));
        CUDA_TRY(h, cudaEventRecord(h->ev1, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        float ms = 0; cudaEventElapsedTime(&ms, h->ev0, h->ev1);
        h->stats.h2d_ms = ms;
        h->stats.h2d_bytes = (int64_t)n_cols * P * sizeof(double);
    }
    h->prog.lanes = h->d_lanes.p;
    return ensure_lane_buffers(h);
}

static int upload_lu(cb200_handle *h, DevLu &L)
{
    cudaStream_t s = h->stream;
    const LuSchedule &S = L.host;
    CUDA_TRY(h, L.rowperm.upload(S.rowperm, s)); CUDA_TRY(h, L.colperm.upload(S.colperm, s));
    CUDA_TRY(h, L.diag_slot.upload(S.diag_slot, s));
    CUDA_TRY(h, L.Lptr.upload(S.Lptr, s)); CUDA_TRY(h, L.L_slot.upload(S.L_slot, s));
    CUDA_TRY(h, L.L_row.upload(S.L_row, s));
    CUDA_TRY(h, L.Uptr.upload(S.Uptr, s)); CUDA_TRY(h, L.U_slot.upload(S.U_slot, s));
    CUDA_TRY(h, L.U_col.upload(S.U_col, s));
    CUDA_TRY(h, L.tgt_ptr.upload(S.tgt_ptr, s)); CUDA_TRY(h, L.tgt.upload(S.tgt, s));
    CUDA_TRY(h, L.jmap.upload(S.jmap, s)); CUDA_TRY(h, L.fill_slots.upload(S.fill_slots, s));
    build_level_schedule(S, L.lvl);
    const LevelSchedule &V = L.lvl;
    CUDA_TRY(h, L.piv_ptr.upload(V.piv_ptr, s)); CUDA_TRY(h, L.sc_ptr.upload(V.sc_ptr, s));
    CUDA_TRY(h, L.tg_ptr.upload(V.tg_ptr, s)); CUDA_TRY(h, L.piv.upload(V.piv, s));
    CUDA_TRY(h, L.sc.upload(V.sc, s)); CUDA_TRY(h, L.tg.upload(V.tg, s)); CUDA_TRY(h, L.upd.upload(V.upd, s));
    CUDA_TRY(h, L.flev_ptr.upload(V.flev_ptr, s)); CUDA_TRY(h, L.frow.upload(V.frow, s));
    CUDA_TRY(h, L.fent.upload(V.fent, s)); CUDA_TRY(h, L.blev_ptr.upload(V.blev_ptr, s));
    CUDA_TRY(h, L.brow.upload(V.brow, s)); CUDA_TRY(h, L.bent.upload(V.bent, s));
    CUDA_TRY(h, cudaStreamSynchronize(s));
    LuProgram &q = L.prog;
    q.n = S.n; q.nlu = (int)S.nlu; q.n_fill = (int)S.fill_slots.size();
    q.rowperm = L.rowperm.p; q.colperm = L.colperm.p; q.diag_slot = L.diag_slot.p;
    q.Lptr = L.Lptr.p; q.L_slot = L.L_slot.p; q.L_row = L.L_row.p;
    q.Uptr = L.Uptr.p; q.U_slot = L.U_slot.p; q.U_col = L.U_col.p;
    q.tgt_ptr = L.tgt_ptr.p; q.tgt = L.tgt.p; q.jmap = L.jmap.p; q.fill_slots = L.fill_slots.p;
    q.n_lev = V.n_lev; q.n_fwd = V.n_fwd; q.n_bwd = V.n_bwd;
    q.n_sc = (int)(V.sc.size() / 2); q.n_bent = (int)(V.bent.size() / 2);
    q.n_tg = (int)(V.tg.size() / 4); q.n_upd = (int)(V.upd.size() / 4);
    q.piv_ptr = L.piv_ptr.p; q.sc_ptr = L.sc_ptr.p; q.tg_ptr = L.tg_ptr.p;
    q.piv = (const int2 *)L.piv.p; q.sc = (const int2 *)L.sc.p;
    q.tg = (const int4 *)L.tg.p; q.upd = (const int4 *)L.upd.p;
    q.flev_ptr = L.flev_ptr.p; q.frow = (const int4 *)L.frow.p; q.fent = (const int2 *)L.fent.p;
    q.blev_ptr = L.blev_ptr.p; q.brow = (const int4 *)L.brow.p; q.bent = (const int2 *)L.bent.p;
    return CB200_OK;
}

static int require_models(cb200_handle *h)
{
    if (h->has_va && h->k.va_header_path.empty())
        return fail(h, CB200_ESTATE, "the circuit contains Verilog-A devices: call cb200_load_va_models first");
    return CB200_OK;
}

// Evaluate G, C at state x for a compact set of sample lanes; returns |G + gamma*C|
// maxima per pattern entry.  Runs the K1/K2 evaluation kernels on a temporary
// program whose lane SoA holds only the samples.
static int probe_magnitudes(cb200_handle *h, const cb200_spec *spec, double gamma,
                            std::vector<double> &absJ, std::vector<double> *absJmin = nullptr)
{
    const int64_t P = h->P;
    const int n = h->st.n;
    const int64_t nnz = h->st.nnz;
    const int ns = (int)std::min<int64_t>(P, 16);
    std::vector<int64_t> sample(ns);
    for (int i = 0; i < ns; i++) sample[i] = ns == 1 ? 0 : (int64_t)((double)i * (double)(P - 1) / (double)(ns - 1));
    std::vector<double> soa((size_t)h->n_lane_cols * ns);
    for (int c = 0; c < h->n_lane_cols; c++)
        for (int i = 0; i < ns; i++) soa[(size_t)c * ns + i] = h->lanes_host[(size_t)c * P + sample[i]];
    DevBuf<double> d_soa, d_ws, d_G, d_C;
    CUDA_TRY(h, d_soa.upload(soa, h->stream));
    Program p = h->prog;
    p.P = ns; p.lanes = d_soa.p;
    CUDA_TRY(h, d_ws.alloc((size_t)p.n_slots * ns));
    CUDA_TRY(h, d_G.alloc((size_t)nnz * ns));
    CUDA_TRY(h, d_C.alloc((size_t)nnz * ns));
    absJ.assign(nnz, 0.0);
    if (absJmin) absJmin->assign(nnz, 1.0 / 0.0);
    std::vector<double> hG((size_t)nnz * ns), hC((size_t)nnz * ns), ws_host((size_t)p.n_slots * ns, 0.0);
    // probe states: ZERO_VECTOR with the PCNR seeds (initjct), ZERO_VECTOR, and two
    // deterministic pseudo-random states in [-1, 1] (cf. solve.jl:992-1015).
    uint64_t rng = 0xDEADBEEFULL;
    auto rnd = [&rng]() {
        rng ^= rng >> 12; rng ^= rng << 25; rng ^= rng >> 27;
        return (double)((rng * 2685821657736338717ULL) >> 11) / 9007199254740992.0;
    };
    for (int probe = 0; probe < 4; probe++) {
        std::fill(ws_host.begin(), ws_host.end(), 0.0);
        if (probe >= 2)
            for (int i = 0; i < n; i++)
                for (int l = 0; l < ns; l++) ws_host[(size_t)(p.off_u + i) * ns + l] = (rnd() - 0.5) * 2.0;
        CUDA_TRY(h, cudaMemcpyAsync(d_ws.p, ws_host.data(), ws_host.size() * sizeof(double),
                                    cudaMemcpyHostToDevice, h->stream));
        EvalArgs a{};
        a.t = 0.0; a.initjct = (probe == 0); a.ws = d_ws.p; a.G_nz = d_G.p; a.C_nz = d_C.p;
        SpecArgs sa = spec_args(spec);
        CUDA_TRY(h, h->k.eval(&p, &sa, &a, h->stream, &h->stats.launches));
        CUDA_TRY(h, cudaMemcpyAsync(hG.data(), d_G.p, hG.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaMemcpyAsync(hC.data(), d_C.p, hC.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        for (int64_t q = 0; q < nnz; q++)
            for (int l = 0; l < ns; l++) {
                double v = std::fabs(hG[(size_t)q * ns + l] + gamma * hC[(size_t)q * ns + l]);
                if (std::isfinite(v) && v > absJ[q]) absJ[q] = v;
                if (absJmin && !(v >= (*absJmin)[q])) (*absJmin)[q] = std::isfinite(v) ? v : 0.0;
            }
    }
    return CB200_OK;
}

extern "C" int cb200_analyze(cb200_handle *h, const cb200_spec *spec, double gamma)
{
    if (!h || !spec) return fail(h, CB200_EINVAL, "cb200_analyze: null argument");
    if (h->P <= 0) return fail(h, CB200_ESTATE, "cb200_analyze: call cb200_set_lanes first");
    if (require_models(h) != CB200_OK) return CB200_ESTATE;
    cudaSetDevice(h->device);
    const int which = gamma == 0.0 ? 0 : 1;
    std::vector<double> absJ, absJmin;
    int rc = probe_magnitudes(h, spec, gamma, absJ, &absJmin);
    if (rc != CB200_OK) return rc;
    DevLu &L = h->lu[which];
    std::string e = analyze_lu(h->st, absJ, 1e-3, L.host, &absJmin);
    if (!e.empty()) return fail(h, CB200_ESINGULAR, e);
    L.host.gamma = gamma;
    rc = upload_lu(h, L);
    if (rc != CB200_OK) return rc;
    h->lu_gen[which]++;
    layout_workspace(h);
    return CB200_OK;
}

static int ensure_lu(cb200_handle *h, const cb200_spec *spec, int which, double gamma)
{
    if (h->lu[which].host.valid && (which == 0 || h->lu[which].host.gamma == gamma)) return CB200_OK;
    return cb200_analyze(h, spec, gamma);
}

extern "C" int cb200_get_pivot_order(const cb200_handle *h, int64_t *rowperm, int64_t *colperm,
                                     int64_t *nnz_lu)
{
    if (!h) return CB200_EINVAL;
    const LuSchedule &S = h->lu[1].host.valid ? h->lu[1].host : h->lu[0].host;
    if (!S.valid) return CB200_ESTATE;
    for (int k = 0; k < S.n; k++) {
        if (rowperm) rowperm[k] = S.rowperm[k] + 1;
        if (colperm) colperm[k] = S.colperm[k] + 1;
    }
    if (nnz_lu) *nnz_lu = S.nlu;
    return CB200_OK;
}

extern "C" int cb200_eval(cb200_handle *h, const cb200_spec *spec, double t, int32_t initjct,
                          const double *x, double *G_nz, double *C_nz, double *b, double *limw)
{
    if (!h || !spec) return fail(h, CB200_EINVAL, "cb200_eval: null argument");
    if (h->P <= 0) return fail(h, CB200_ESTATE, "cb200_eval: call cb200_set_lanes first");
    if (require_models(h) != CB200_OK) return CB200_ESTATE;
    cudaSetDevice(h->device);
    const int64_t P = h->P;
    const int n = h->st.n;
    const int64_t nnz = h->st.nnz;
    h->stats = cb200_stats{};
    int rc = ensure_global_ws(h);
    if (rc != CB200_OK) return rc;
    cudaStream_t s = h->stream;
    CUDA_TRY(h, cudaMemsetAsync(h->d_ws_global.p, 0, (size_t)h->prog.n_slots * P * sizeof(double), s));
    if (x) CUDA_TRY(h, cudaMemcpyAsync(h->d_ws_global.p + (size_t)h->prog.off_u * P, x,
                                       (size_t)n * P * sizeof(double), cudaMemcpyHostToDevice, s));
    DevBuf<double> dG, dC, db, dl;
    CUDA_TRY(h, dG.alloc((size_t)nnz * P)); CUDA_TRY(h, dC.alloc((size_t)nnz * P));
    CUDA_TRY(h, db.alloc((size_t)n * P)); CUDA_TRY(h, dl.alloc((size_t)std::max(1, h->st.n_limits) * P));
    EvalArgs a{};
    a.t = t; a.initjct = initjct; a.ws = h->d_ws_global.p;
    a.G_nz = dG.p; a.C_nz = dC.p; a.b = db.p; a.limw = dl.p;
    CUDA_TRY(h, cudaEventRecord(h->ev0, s));
    {
        SpecArgs sa = spec_args(spec);
        CUDA_TRY(h, h->k.eval(&h->prog, &sa, &a, s, &h->stats.launches));
    }
    CUDA_TRY(h, cudaEventRecord(h->ev1, s));
    if (G_nz) CUDA_TRY(h, cudaMemcpyAsync(G_nz, dG.p, (size_t)nnz * P * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (C_nz) CUDA_TRY(h, cudaMemcpyAsync(C_nz, dC.p, (size_t)nnz * P * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (b) CUDA_TRY(h, cudaMemcpyAsync(b, db.p, (size_t)n * P * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (limw && h->st.n_limits > 0)
        CUDA_TRY(h, cudaMemcpyAsync(limw, dl.p, (size_t)h->st.n_limits * P * sizeof(double), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(h, cudaStreamSynchronize(s));
    float ms = 0; cudaEventElapsedTime(&ms, h->ev0, h->ev1);
    h->stats.kernel_ms = ms;
    return CB200_OK;
}

// the specialised module is usable only for the LU schedules it was generated from
static bool spec_usable(const cb200_handle *h)
{
    return h->spec.dl != nullptr && h->spec_gen[0] == h->lu_gen[0] && h->spec_gen[1] == h->lu_gen[1];
}

// ---------------------------------------------------------------------------
// DC on the device: _dc_solve_with_fallbacks (solve.jl:871-929) over all lanes.
// State stays in h->d_state; per-lane tier bookkeeping on the host.
// ---------------------------------------------------------------------------
struct DcRun {
    cb200_handle *h;
    SpecArgs sa;
    double t;
    double abstol;
    int maxiters;
    float kernel_ms = 0;
};

static int dc_launch(DcRun &r, int algorithm, const unsigned char *d_active, const double *d_gshunt,
                     const double *d_srcfact)
{
    cb200_handle *h = r.h;
    DcArgs a{};
    a.algorithm = algorithm; a.abstol = r.abstol; a.maxiters = r.maxiters; a.t = r.t;
    a.u = h->d_state.p; a.active = d_active; a.gshunt_lane = d_gshunt; a.srcfact_lane = d_srcfact;
    a.status = h->d_status.p; a.iters = h->d_iters.p; a.converged = h->d_conv.p; a.weak = h->d_weak.p;
    a.ws_global = nullptr;
    if (needs_global_ws(h)) {
        int rc = ensure_global_ws(h);
        if (rc != CB200_OK) return rc;
        a.ws_global = h->d_ws_global.p;
    }
    CUDA_TRY(h, cudaEventRecord(h->ev0, h->stream));
    if (spec_usable(h)) {
        h->stats.launches += 1;
        CUDA_TRY(h, h->spec.dc(&h->prog, &r.sa, &a, h->stream));
    } else {
        CUDA_TRY(h, h->k.dc(&h->prog, &h->lu[0].prog, &r.sa, &a, h->block_pref, h->smem_limit, h->stream,
                            &h->stats.launches));
    }
    CUDA_TRY(h, cudaEventRecord(h->ev1, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    float ms = 0; cudaEventElapsedTime(&ms, h->ev0, h->ev1);
    r.kernel_ms += ms;
    return CB200_OK;
}

// Runs the fallback chain on the device state.  d_state must hold u0 for every lane;
// u0_host is the same start on the host (null = zeros), needed only to restart the
// lanes tier 0 leaves unconverged.
static int dc_chain(cb200_handle *h, const cb200_spec *spec, double t, double abstol, int maxiters,
                    int use_stepping, const double *u0_host, std::vector<unsigned char> &conv_out,
                    std::vector<int> &status_out)
{
    const int64_t P = h->P;
    const int n = h->st.n;
    int rc = ensure_lu(h, spec, 0, 0.0);
    if (rc != CB200_OK) return rc;
    DcRun r{h, spec_args(spec), t, abstol, maxiters};
    cudaStream_t s = h->stream;
    CUDA_TRY(h, cudaMemsetAsync(h->d_iters.p, 0, P * sizeof(int), s));
    CUDA_TRY(h, cudaMemsetAsync(h->d_conv.p, 0, P, s));
    std::vector<unsigned char> conv(P, 0), active(P, 1);
    std::vector<int> status(P, CB200_LANE_OK);

    auto fetch = [&]() -> int {
        CUDA_TRY(h, cudaMemcpyAsync(conv.data(), h->d_conv.p, P, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(h, cudaMemcpyAsync(status.data(), h->d_status.p, P * sizeof(int), cudaMemcpyDeviceToHost, s));
        CUDA_TRY(h, cudaStreamSynchronize(s));
        return CB200_OK;
    };
    auto all_conv = [&]() { return std::all_of(conv.begin(), conv.end(), [](unsigned char c) { return c != 0; }); };

    const bool has_limits = h->st.n_limits > 0;
    // use_stepping 2 / 3: test hooks that enter the chain at tier 2 / tier 3 (cb200_dc_opts)
    const bool direct = use_stepping < 2;
    if (!direct) CUDA_TRY(h, cudaMemsetAsync(h->d_status.p, 0, P * sizeof(int), s));
    if (direct && has_limits) {
        rc = dc_launch(r, 0, nullptr, nullptr, nullptr);                  // tier 0: PCNR
        if (rc != CB200_OK) return rc;
        if ((rc = fetch()) != CB200_OK) return rc;
    }
    if (direct && (!has_limits || !all_conv())) {
        // tier 1: plain Newton from u0 on the lanes PCNR left unconverged
        if (has_limits) {
            std::vector<double> cur((size_t)n * P);
            CUDA_TRY(h, cudaMemcpyAsync(cur.data(), h->d_state.p, cur.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
            CUDA_TRY(h, cudaStreamSynchronize(s));
            for (int64_t l = 0; l < P; l++) {
                active[l] = conv[l] ? 0 : 1;
                if (active[l])
                    for (int i = 0; i < n; i++) cur[(size_t)i * P + l] = u0_host ? u0_host[(size_t)i * P + l] : 0.0;
            }
            CUDA_TRY(h, cudaMemcpyAsync(h->d_state.p, cur.data(), cur.size() * sizeof(double), cudaMemcpyHostToDevice, s));
            CUDA_TRY(h, cudaMemcpyAsync(h->d_active.p, active.data(), P, cudaMemcpyHostToDevice, s));
        }
        rc = dc_launch(r, 1, has_limits ? h->d_active.p : nullptr, nullptr, nullptr);
        if (rc != CB200_OK) return rc;
        if ((rc = fetch()) != CB200_OK) return rc;
    }
    if (use_stepping && !all_conv()) {
        // tiers 2 and 3 on the device: _gshunt_stepping (solve.jl:720-783), then _source_stepping
        // (:805-850), each from zeros, one launch for all lanes that are still unconverged -- the
        // per-lane continuation state never leaves the GPU (lane_kernels.cuh: dc_stepping_body).
        // Always the table-driven kernels: a rare path is not worth a third specialised kernel.
        std::vector<unsigned char> todo(P);
        std::vector<int> status01 = status;
        for (int64_t l = 0; l < P; l++) todo[l] = conv[l] ? 0 : 1;
        CUDA_TRY(h, cudaMemcpyAsync(h->d_active.p, todo.data(), P, cudaMemcpyHostToDevice, s));
        {
            DcArgs a{};
            a.algorithm = use_stepping == 3 ? 3 : 2; a.abstol = r.abstol; a.maxiters = r.maxiters; a.t = r.t;
            a.u = h->d_state.p; a.active = h->d_active.p;
            a.status = h->d_status.p; a.iters = h->d_iters.p; a.converged = h->d_conv.p; a.weak = h->d_weak.p;
            if (needs_global_ws(h)) {
                if ((rc = ensure_global_ws(h)) != CB200_OK) return rc;
                a.ws_global = h->d_ws_global.p;
            }
            CUDA_TRY(h, cudaEventRecord(h->ev0, s));
            CUDA_TRY(h, h->k.dc(&h->prog, &h->lu[0].prog, &r.sa, &a, h->block_pref, h->smem_limit, s, &h->stats.launches));
            CUDA_TRY(h, cudaEventRecord(h->ev1, s));
            CUDA_TRY(h, cudaStreamSynchronize(s));
            float ms = 0; cudaEventElapsedTime(&ms, h->ev0, h->ev1);
            r.kernel_ms += ms;
        }
        if ((rc = fetch()) != CB200_OK) return rc;
        h->stats.dc_stepping_lanes = 0;
        for (int64_t l = 0; l < P; l++) {
            if (!todo[l]) continue;
            h->stats.dc_stepping_lanes++;
            // a lane the continuation could not rescue keeps the status of its direct attempt
            if (!conv[l] && status01[l] != CB200_LANE_OK) status[l] = status01[l];
        }
    }
    h->stats.kernel_ms += r.kernel_ms;
    h->stats.dc_kernel_ms += r.kernel_ms;
    conv_out = conv;
    status_out = status;
    for (int64_t l = 0; l < P; l++) if (conv_out[l]) status_out[l] = CB200_LANE_OK;
    return CB200_OK;
}

extern "C" int cb200_dc(cb200_handle *h, const cb200_spec *spec, const cb200_dc_opts *opts,
                        const double *u0, double *x_out, int32_t *status, int32_t *iters)
{
    if (!h || !spec || !opts) return fail(h, CB200_EINVAL, "cb200_dc: null argument");
    if (h->P <= 0) return fail(h, CB200_ESTATE, "cb200_dc: call cb200_set_lanes first");
    cudaSetDevice(h->device);
    const int64_t P = h->P;
    const int n = h->st.n;
    h->stats = cb200_stats{};
    cudaStream_t s = h->stream;
    if (n == 0) { for (int64_t l = 0; l < P; l++) { if (status) status[l] = 0; if (iters) iters[l] = 0; } return CB200_OK; }
    CUDA_TRY(h, cudaMemsetAsync(h->d_weak.p, 0, P * sizeof(int), s));
    if (u0) {
        CUDA_TRY(h, cudaMemcpyAsync(h->d_state.p, u0, (size_t)n * P * sizeof(double), cudaMemcpyHostToDevice, s));
        h->stats.h2d_bytes += (int64_t)n * P * sizeof(double);
    } else {
        CUDA_TRY(h, cudaMemsetAsync(h->d_state.p, 0, (size_t)n * P * sizeof(double), s));
    }
    std::vector<unsigned char> conv;
    std::vector<int> st;
    int rc = dc_chain(h, spec, 0.0, opts->abstol, opts->maxiters, opts->use_stepping, u0, conv, st);
    if (rc != CB200_OK) return rc;
    if (x_out) {
        CUDA_TRY(h, cudaMemcpyAsync(x_out, h->d_state.p, (size_t)n * P * sizeof(double), cudaMemcpyDeviceToHost, s));
        h->stats.d2h_bytes += (int64_t)n * P * sizeof(double);
    }
    std::vector<int> it(P);
    CUDA_TRY(h, cudaMemcpyAsync(it.data(), h->d_iters.p, P * sizeof(int), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(h, cudaStreamSynchronize(s));
    int64_t tot = 0;
    for (int64_t l = 0; l < P; l++) {
        if (status) status[l] = st[l];
        if (iters) iters[l] = it[l];
        tot += it[l];
    }
    h->stats.newton_iters = tot;
    return CB200_OK;
}

// ---------------------------------------------------------------------------
// transient
// ---------------------------------------------------------------------------
static const int kMaxSegments = 16;

static int tran_impl(cb200_handle *h, const cb200_spec *spec, double t0, double t1,
                     const cb200_tran_opts *o, const int64_t *save_idx, int32_t n_save,
                     const double *u0, double *host_u, int64_t host_ld, int n_segments, cb200_wave **out)
{
    if (!h || !spec || !o || !out) return fail(h, CB200_EINVAL, "cb200_tran: null argument");
    *out = nullptr;
    if (h->P <= 0) return fail(h, CB200_ESTATE, "cb200_tran: call cb200_set_lanes first");
    if (!(t1 > t0) || !(o->dt > 0.0)) return fail(h, CB200_EINVAL, "cb200_tran: need t1 > t0 and dt > 0");
    if (n_save < 0 || (n_save > 0 && !save_idx)) return fail(h, CB200_EINVAL, "cb200_tran: bad save list");
    if (o->method < CB200_METHOD_BE || o->method > CB200_METHOD_BDF) return fail(h, CB200_EINVAL, "cb200_tran: unknown method");
    if (o->method == CB200_METHOD_BDF && !o->adaptive)
        return fail(h, CB200_EINVAL, "cb200_tran: CB200_METHOD_BDF is a variable-step method (adaptive = 1)");
    cudaSetDevice(h->device);
    const int64_t P = h->P;
    const int n = h->st.n;
    for (int q = 0; q < n_save; q++)
        if (save_idx[q] < 1 || save_idx[q] > n) return fail(h, CB200_EINVAL, "cb200_tran: save index out of range");
    h->stats = cb200_stats{};
    cudaStream_t s = h->stream;

    CUDA_TRY(h, cudaMemsetAsync(h->d_weak.p, 0, P * sizeof(int), s));
    // initialisation: CedarTranOp (dcop.jl:160-203) or caller-provided state
    std::vector<unsigned char> conv(P, 1);
    std::vector<int> st0(P, CB200_LANE_OK);
    if (o->init == 0) {
        CUDA_TRY(h, cudaMemsetAsync(h->d_state.p, 0, (size_t)n * P * sizeof(double), s));
        cb200_spec sdc = *spec;
        sdc.mode = CB200_MODE_TRANOP;
        int rc = dc_chain(h, &sdc, t0, o->init_abstol, o->init_maxiters, 1, nullptr, conv, st0);
        if (rc != CB200_OK) return rc;
    } else {
        if (!u0 && o->init == 1) return fail(h, CB200_EINVAL, "cb200_tran: init=1 needs u0");
        if (u0) {
            CUDA_TRY(h, cudaMemcpyAsync(h->d_state.p, u0, (size_t)n * P * sizeof(double), cudaMemcpyHostToDevice, s));
            h->stats.h2d_bytes += (int64_t)n * P * sizeof(double);
        } else {
            CUDA_TRY(h, cudaMemsetAsync(h->d_state.p, 0, (size_t)n * P * sizeof(double), s));
        }
        CUDA_TRY(h, cudaMemsetAsync(h->d_iters.p, 0, P * sizeof(int), s));
    }
    const double gamma_nom = (o->method == CB200_METHOD_BE || o->method == CB200_METHOD_BDF ? 1.0 : o->method == CB200_METHOD_TRAP ? 2.0 : 1.5) / o->dt;
    int rc = ensure_lu(h, spec, 1, gamma_nom);
    if (rc != CB200_OK) return rc;

    bool used_spec = false;            // the fixed-step launches went to the circuit-specialised kernels
    cb200_wave *w = new cb200_wave();
    w->h = h; w->P = P; w->n_save = n_save; w->n = n; w->adaptive = o->adaptive; w->t0 = t0; w->dt = o->dt;
    w->d_out.pool = w->d_t.pool = w->d_final.pool = h->pool;
    w->d_count.pool = w->d_status.pool = w->d_iters.pool = h->pool;
    std::vector<int> save0(n_save);
    for (int q = 0; q < n_save; q++) save0[q] = (int)save_idx[q] - 1;
    DevBuf<int> &d_save = h->d_save;
    if (d_save.n != (size_t)n_save && d_save.alloc(n_save) != cudaSuccess) { delete w; return fail(h, CB200_ECUDA, "cb200_tran: allocation failed"); }
    if (n_save > 0 && cudaMemcpyAsync(d_save.p, save0.data(), n_save * sizeof(int), cudaMemcpyHostToDevice, s) != cudaSuccess) {
        delete w; return fail(h, CB200_ECUDA, "cb200_tran: upload failed");
    }
    // lanes whose initialisation failed keep that status (InitialFailure, dcop.jl:197-200)
    if (cudaMemcpyAsync(h->d_status.p, st0.data(), P * sizeof(int), cudaMemcpyHostToDevice, s) != cudaSuccess) {
        delete w; return fail(h, CB200_ECUDA, "cb200_tran: upload failed");
    }
    SpecArgs sa = spec_args(spec);
    sa.mode = CB200_MODE_TRAN;
    if ((h->d_evals.n != (size_t)P && h->d_evals.alloc(P) != cudaSuccess) ||
        cudaMemsetAsync(h->d_evals.p, 0, P * sizeof(int), s) != cudaSuccess) {
        delete w; return fail(h, CB200_ECUDA, "cb200_tran: allocation failed");
    }
    double *ws_global = nullptr;
    if (needs_global_ws(h)) {
        rc = ensure_global_ws(h);
        if (rc != CB200_OK) { delete w; return rc; }
        ws_global = h->d_ws_global.p;
    }
    cudaError_t ce = cudaSuccess;
    if (o->init == 2 && o->uic_steps > 0) {
        // CedarUICOp (dcop.jl:311-411): uic_steps backward-Euler steps of uic_dt from the start state
        // on the table-driven kernels (same pivot schedule), nothing saved; Newton failures are
        // marched through (force_dtmin=true), so the lane status is reset afterwards.
        DevBuf<double> scratch;
        scratch.pool = h->pool;
        if (scratch.alloc((size_t)2 * P) != cudaSuccess) { delete w; return fail(h, CB200_ENOMEM, "cb200_tran: allocation failed"); }
        TranArgs a{};
        a.method = CB200_METHOD_BE; a.t0 = t0; a.h = o->uic_dt > 0 ? o->uic_dt : 1e-12; a.nsteps = o->uic_steps;
        a.k_begin = 1; a.k_end = o->uic_steps; a.tp_begin = 0;
        a.abstol = o->abstol; a.max_nl = o->max_nl_iters; a.limit = o->flags & CB200_TRAN_LIMIT;
        a.save_every = o->uic_steps; a.n_save = 0; a.save_idx = d_save.p; a.T = 2;
        a.u = h->d_state.p; a.out = scratch.p; a.status = h->d_status.p; a.iters = h->d_iters.p;
        a.evals = h->d_evals.p; a.weak = h->d_weak.p; a.ws_global = ws_global;
        ce = h->k.tran_fixed(&h->prog, &h->lu[1].prog, &sa, &a, h->block_pref, h->smem_limit, s, &h->stats.launches);
        if (ce == cudaSuccess) ce = cudaMemsetAsync(h->d_status.p, 0, P * sizeof(int), s);
        if (ce != cudaSuccess) { delete w; return fail(h, CB200_ECUDA, std::string("cb200_tran: warm-up failed: ") + cudaGetErrorString(ce)); }
    }
    if (!o->adaptive) {
        const int64_t nsteps = (int64_t)std::llround((t1 - t0) / o->dt);
        const int se = o->save_every > 0 ? o->save_every : 1;
        const int64_t T = 1 + nsteps / se + ((nsteps % se) ? 1 : 0);
        w->T = T; w->nsteps = nsteps; w->save_every = se;
        if (w->d_out.alloc((size_t)std::max(1, n_save) * T * P) != cudaSuccess) {
            delete w; return fail(h, CB200_ENOMEM, "cb200_tran: waveform buffer allocation failed");
        }
        TranArgs a{};
        a.method = o->method; a.t0 = t0; a.h = o->dt; a.nsteps = nsteps; a.abstol = o->abstol;
        a.max_nl = o->max_nl_iters; a.limit = o->flags & CB200_TRAN_LIMIT; a.save_every = se; a.n_save = n_save; a.save_idx = d_save.p;
        a.T = T; a.u = h->d_state.p; a.out = w->d_out.p; a.status = h->d_status.p; a.iters = h->d_iters.p;
        a.evals = h->d_evals.p; a.weak = h->d_weak.p;
        a.ws_global = ws_global;
        // Time segments: one launch each.  With a host destination the D2H copy of a finished
        // segment runs on the copy stream while the next segment computes.
        int nseg = (host_u != nullptr && n_segments > 1) ? (int)std::min<int64_t>(n_segments, std::max<int64_t>(1, nsteps / 64)) : 1;
        if (nseg > kMaxSegments) nseg = kMaxSegments;
        if (nseg > 1) {
            if (h->d_hist.n != (size_t)2 * n * P && h->d_hist.alloc((size_t)2 * n * P) != cudaSuccess) {
                delete w; return fail(h, CB200_ENOMEM, "cb200_tran: history buffer allocation failed");
            }
            a.hist = h->d_hist.p;
        }
        const int64_t seg_len = (nsteps + nseg - 1) / nseg;
        cudaEventRecord(h->ev0, s);
        for (int g = 0; g < nseg && ce == cudaSuccess; g++) {
            a.k_begin = (int64_t)g * seg_len + 1;
            a.k_end = std::min<int64_t>(nsteps, (int64_t)(g + 1) * seg_len);
            if (a.k_begin > a.k_end) break;
            a.tp_begin = g == 0 ? 0 : 1 + (a.k_begin - 1) / se;
            if (spec_usable(h) && h->spec_method == o->method && (!a.limit || h->spec_limit)) {
                h->stats.launches += 1;
                if (!used_spec && h->spec.take_counters) h->spec.take_counters(nullptr, s);   // reset
                used_spec = true;
                ce = h->spec.tran_fixed(&h->prog, &sa, &a, s);
            } else {
                ce = h->k.tran_fixed(&h->prog, &h->lu[1].prog, &sa, &a, h->block_pref, h->smem_limit, s, &h->stats.launches);
            }
            if (host_u != nullptr && ce == cudaSuccess) {
                int64_t tp_end = 1 + a.k_end / se;                     // one past the last point written
                if (a.k_end == nsteps && nsteps % se != 0) tp_end += 1;
                cudaEventRecord(h->seg_ev[g], s);
                cudaStreamWaitEvent(h->copy_stream, h->seg_ev[g], 0);
                for (int q = 0; q < n_save; q++) {
                    // host rows may be wider than the device rows (host_ld >= P): this handle's lanes
                    // are then one column block of a waveform array that several GPUs fill
                    const size_t off = ((size_t)q * T + a.tp_begin) * P;
                    const size_t hoff = ((size_t)q * T + a.tp_begin) * (size_t)host_ld;
                    ce = cudaMemcpy2DAsync(host_u + hoff, (size_t)host_ld * sizeof(double), w->d_out.p + off,
                                           (size_t)P * sizeof(double), (size_t)P * sizeof(double),
                                           (size_t)(tp_end - a.tp_begin), cudaMemcpyDeviceToHost, h->copy_stream);
                    if (ce != cudaSuccess) break;
                }
                h->stats.d2h_bytes += (int64_t)n_save * (tp_end - a.tp_begin) * P * sizeof(double);
            }
        }
        cudaEventRecord(h->ev1, s);
        if (host_u != nullptr && ce == cudaSuccess) ce = cudaStreamSynchronize(h->copy_stream);
    } else {
        // LTE-controlled stepping, per-lane time axis; tstops come from cb200_set_tstops
        const int T = o->max_points > 1 ? o->max_points : 4096;
        w->T = T;
        const double span = t1 - t0;
        AdaptArgs a{};
        a.method = o->method == CB200_METHOD_BE ? CB200_METHOD_BE : o->method == CB200_METHOD_BDF ? CB200_METHOD_BDF : CB200_METHOD_TRAP;
        a.t0 = t0; a.t1 = t1;
        a.dtmax = o->dtmax > 0 ? o->dtmax : span / 50.0;
        a.dtmin = o->dtmin > 0 ? o->dtmin : span * 1e-12;
        a.h0 = std::min(o->dt, a.dtmax);
        a.abstol = o->abstol; a.reltol = o->reltol; a.lte_abstol = o->lte_abstol;
        const bool cls = (o->flags & CB200_TRAN_CLASS_ABSTOL) != 0;
        a.tol_v = cls ? o->vntol : o->lte_abstol; a.tol_i = cls ? o->iabstol : o->lte_abstol;
        a.tol_q = cls ? o->chgtol : o->lte_abstol;
        a.cls_i0 = h->st.n_nodes; a.cls_q0 = h->st.n_nodes + h->st.n_currents;
        a.cls_l0 = h->st.n_nodes + h->st.n_currents + h->st.n_charges;
        if (cls && !(a.tol_v > 0 && a.tol_i > 0 && a.tol_q > 0)) { delete w; return fail(h, CB200_EINVAL, "cb200_tran: CB200_TRAN_CLASS_ABSTOL needs vntol, iabstol, chgtol > 0"); }
        a.max_nl = o->max_nl_iters; a.limit = o->flags & CB200_TRAN_LIMIT;
        a.n_save = n_save; a.save_idx = d_save.p; a.max_points = T;
        if (w->d_out.alloc((size_t)std::max(1, n_save) * T * P) != cudaSuccess ||
            w->d_t.alloc((size_t)T * P) != cudaSuccess || w->d_count.alloc(P) != cudaSuccess ||
            (h->d_rejected.n != (size_t)P && h->d_rejected.alloc(P) != cudaSuccess)) {
            delete w; return fail(h, CB200_ENOMEM, "cb200_tran: waveform buffer allocation failed");
        }
        a.tstops = h->d_tstops.p; a.n_tstops = (int)h->tstops.size();
        a.u = h->d_state.p; a.out_t = w->d_t.p; a.out = w->d_out.p; a.count = w->d_count.p;
        a.status = h->d_status.p; a.iters = h->d_iters.p; a.rejected = h->d_rejected.p;
        a.evals = h->d_evals.p; a.weak = h->d_weak.p;
        a.ws_global = ws_global;
        cudaEventRecord(h->ev0, s);
        if (spec_usable(h) && h->spec.tran_adaptive && h->spec_method == a.method && (!a.limit || h->spec_limit)) {
            h->stats.launches += 1;
            ce = h->spec.tran_adaptive(&h->prog, &sa, &a, s);
        } else {
            ce = h->k.tran_adaptive(&h->prog, &h->lu[1].prog, &sa, &a, h->block_pref, h->smem_limit, s, &h->stats.launches);
        }
        cudaEventRecord(h->ev1, s);
        if (ce == cudaSuccess) {
            std::vector<int> cnt(P), rj(P);
            cudaMemcpyAsync(cnt.data(), w->d_count.p, P * sizeof(int), cudaMemcpyDeviceToHost, s);
            cudaMemcpyAsync(rj.data(), h->d_rejected.p, P * sizeof(int), cudaMemcpyDeviceToHost, s);
            ce = cudaStreamSynchronize(s);
            int64_t acc = 0, rejt = 0;
            for (int64_t l = 0; l < P; l++) { acc += cnt[l] - 1; rejt += rj[l]; }
            h->stats.steps_accepted = acc;
            h->stats.steps_rejected = rejt;
        }
    }
    if (ce == cudaSuccess) ce = cudaStreamSynchronize(s);
    if (ce != cudaSuccess) {
        delete w;
        return fail(h, CB200_ECUDA, std::string("cb200_tran: kernel failed: ") + cudaGetErrorString(ce));
    }
    float ms = 0; cudaEventElapsedTime(&ms, h->ev0, h->ev1);
    h->stats.kernel_ms += ms;
    h->stats.tran_kernel_ms = ms;
    // keep per-lane results with the wave so the handle can be reused
    w->d_status.alloc(P); w->d_iters.alloc(P); w->d_final.alloc((size_t)n * P);
    cudaMemcpyAsync(w->d_status.p, h->d_status.p, P * sizeof(int), cudaMemcpyDeviceToDevice, s);
    cudaMemcpyAsync(w->d_iters.p, h->d_iters.p, P * sizeof(int), cudaMemcpyDeviceToDevice, s);
    cudaMemcpyAsync(w->d_final.p, h->d_state.p, (size_t)n * P * sizeof(double), cudaMemcpyDeviceToDevice, s);
    ce = cudaStreamSynchronize(s);
    if (ce != cudaSuccess) { delete w; return fail(h, CB200_ECUDA, cudaGetErrorString(ce)); }
    if (!o->adaptive) h->stats.steps_accepted = w->nsteps * P;
    if (!o->adaptive && used_spec && h->spec.take_counters) {
        // specialised kernels skip quiescent steps bit-exactly (lane_kernels.cuh, tran_fixed_body): the
        // lane-steps actually executed
        unsigned long long nexec = 0;
        if (h->spec.take_counters(&nexec, s) == cudaSuccess) h->stats.steps_accepted = (int64_t)nexec;
    }
    {   // device-model evaluation passes executed (sum over lanes): the work the FP64 roofline counts
        std::vector<int> ev(P);
        cudaMemcpyAsync(ev.data(), h->d_evals.p, P * sizeof(int), cudaMemcpyDeviceToHost, s);
        cudaStreamSynchronize(s);
        int64_t tot = 0;
        for (int64_t l = 0; l < P; l++) tot += ev[l];
        h->stats.device_evals = tot;
    }
    h->waves.push_back(w);
    *out = w;
    return CB200_OK;
}

extern "C" int cb200_tran(cb200_handle *h, const cb200_spec *spec, double t0, double t1,
                          const cb200_tran_opts *o, const int64_t *save_idx, int32_t n_save,
                          const double *u0, cb200_wave **out)
{
    return tran_impl(h, spec, t0, t1, o, save_idx, n_save, u0, nullptr, 0, 1, out);
}

// tran! straight into host memory: the time loop is cut into n_segments launches and the
// waveform of each finished segment is copied out (copy stream) while the next computes.
static int wave_fetch_impl(cb200_wave *w, double *t, double *u, int64_t u_ld, int64_t t_ld, int32_t *count,
                           int32_t *status, int32_t *newton_iters);

extern "C" int cb200_tran_fetch_ld(cb200_handle *h, const cb200_spec *spec, double t0, double t1,
                                   const cb200_tran_opts *o, const int64_t *save_idx, int32_t n_save,
                                   const double *u0, int32_t n_segments, double *t_out, double *u_out,
                                   int64_t u_ld, int32_t *count, int32_t *status, int32_t *newton_iters)
{
    if (!o || !h) return fail(h, CB200_EINVAL, "cb200_tran_fetch: null argument");
    if (u_ld == 0) u_ld = h->P;
    if (u_ld < h->P) return fail(h, CB200_EINVAL, "cb200_tran_fetch: u_ld is smaller than the lane count");
    cb200_wave *w = nullptr;
    const bool pipelined = !o->adaptive && u_out != nullptr;
    int rc = tran_impl(h, spec, t0, t1, o, save_idx, n_save, u0, pipelined ? u_out : nullptr, u_ld,
                       n_segments, &w);
    if (rc != CB200_OK) return rc;
    const int64_t d2h = h->stats.d2h_bytes;
    rc = wave_fetch_impl(w, t_out, pipelined ? nullptr : u_out, u_ld, u_ld, count, status, newton_iters);
    h->stats.d2h_bytes += d2h;
    cb200_wave_free(w);
    return rc;
}

extern "C" int cb200_tran_fetch(cb200_handle *h, const cb200_spec *spec, double t0, double t1,
                                const cb200_tran_opts *o, const int64_t *save_idx, int32_t n_save,
                                const double *u0, int32_t n_segments, double *t_out, double *u_out,
                                int32_t *count, int32_t *status, int32_t *newton_iters)
{
    return cb200_tran_fetch_ld(h, spec, t0, t1, o, save_idx, n_save, u0, n_segments, t_out, u_out, 0,
                               count, status, newton_iters);
}

extern "C" int cb200_load_va_models(cb200_handle *h, const char *cuda_header, const char *csrc_dir,
                                    const char *cache_dir)
{
    if (!cuda_header || !csrc_dir || !cache_dir) return fail(h, CB200_EINVAL, "cb200_load_va_models: null argument");
    KernelSet ks;
    std::string e = build_va_kernel_set(cuda_header, csrc_dir, cache_dir, ks);
    if (!e.empty()) return fail(h, CB200_ECUDA, e);
    if (!h) { unload_kernel_set(ks); return CB200_OK; }      // cache warm-up only
    cudaSetDevice(h->device);
    if (h->k.dl) unload_kernel_set(h->k);
    h->k = ks;
    unload_spec(h->spec);                 // specialised kernels were generated without these models
    h->spec_gen[0] = h->spec_gen[1] = -1;
    return CB200_OK;
}

// 1 when the kernel set of this header is already in the cache (no nvcc run needed), else 0
extern "C" int cb200_va_models_cached(const char *cuda_header, const char *csrc_dir, const char *cache_dir)
{
    if (!cuda_header || !csrc_dir || !cache_dir) return 0;
    return va_kernel_set_cached(cuda_header, csrc_dir, cache_dir) ? 1 : 0;
}

extern "C" int cb200_set_tstops(cb200_handle *h, const double *tstops, int32_t n)
{
    if (!h || n < 0 || (n > 0 && !tstops)) return fail(h, CB200_EINVAL, "cb200_set_tstops: bad arguments");
    cudaSetDevice(h->device);
    h->tstops.assign(tstops, tstops + n);
    std::sort(h->tstops.begin(), h->tstops.end());
    CUDA_TRY(h, h->d_tstops.upload(h->tstops, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CB200_OK;
}

// ---------------------------------------------------------------------------
// circuit specialisation (the emitter)
// ---------------------------------------------------------------------------
// What the emitter reads of a handle's circuit, and the launch bounds of the generated kernels: 64 threads
// per block and enough resident blocks per SM for all P lanes in one wave, as far as registers allow.
static SpecInput spec_input(const cb200_handle &h, int method, int64_t P, int num_sms)
{
    SpecInput in{};
    in.st = &h.st; in.prog = &h.prog;
    in.dev_kind = &h.dev_kind; in.dev_flags = &h.dev_flags; in.dev_node_ptr = &h.dev_node_ptr;
    in.dev_nodes = &h.dev_nodes; in.dev_param_ptr = &h.dev_param_ptr; in.dev_params = &h.dev_params;
    in.dev_gbase = &h.dev_gbase; in.dev_cbase = &h.dev_cbase; in.dev_bbase = &h.dev_bbase; in.dev_sbase = &h.dev_sbase;
    in.src_list = &h.src_list; in.nl_list = &h.nl_list; in.limit_init_ref = &h.limit_init_ref;
    in.src_uniform = &h.src_uniform; in.method = method;
    in.va_header_path = h.k.va_header_path;
    in.uniform = &h.uniform; in.lu_dc = &h.lu[0].host; in.lu_tr = &h.lu[1].host;
    in.n_lane_cols = h.n_lane_cols;
    in.block = 64;
    const int64_t lanes_per_sm = (P + num_sms - 1) / num_sms;
    in.min_blocks = std::max(1, std::min((int)((lanes_per_sm + in.block - 1) / in.block), 1024 / in.block));
    // a lane state beyond the register file lives in local memory: measured on B200 (C3, sp_mos1
    // inverter, 432 slots) 4 resident blocks x 255 registers beat 11 x 93 by 1.6x
    if (h.prog.n_slots > 120) in.min_blocks = std::min(in.min_blocks, 4);
    return in;
}

extern "C" int cb200_specialize(cb200_handle *h, const cb200_spec *spec, int32_t method, double dt,
                                const char *csrc_dir, const char *cache_dir, int32_t flags)
{
    if (method < 0 || method > 3 || !(dt > 0.0)) return fail(h, CB200_EINVAL, "cb200_specialize: bad method / dt");
    const double gamma = (method == CB200_METHOD_BE || method == CB200_METHOD_BDF ? 1.0 : method == CB200_METHOD_TRAP ? 2.0 : 1.5) / dt;
    if (!h || !spec || !csrc_dir || !cache_dir) return fail(h, CB200_EINVAL, "cb200_specialize: null argument");
    if (h->P <= 0) return fail(h, CB200_ESTATE, "cb200_specialize: call cb200_set_lanes first");
    cudaSetDevice(h->device);
    cb200_spec sdc = *spec;
    int rc = ensure_lu(h, &sdc, 0, 0.0);
    if (rc != CB200_OK) return rc;
    rc = ensure_lu(h, spec, 1, gamma);
    if (rc != CB200_OK) return rc;
    const bool want_limit = (flags & CB200_SPEC_TRAN_LIMIT) != 0;
    const bool want_adaptive = (flags & CB200_SPEC_FIXED_ONLY) == 0;
    if (spec_usable(h) && h->spec_method == method && h->spec_limit == want_limit &&
        (!want_adaptive || h->spec.tran_adaptive)) return CB200_OK;
    SpecInput in = spec_input(*h, method, h->P, h->num_sms);
    in.tran_limit = want_limit;
    in.with_adaptive = want_adaptive;
    if (h->prog.n_slots > 4096) return fail(h, CB200_EINVAL, "cb200_specialize: circuit too large for a register-resident kernel");
    const std::string src = generate_spec_source(in);
    unload_spec(h->spec);
    std::string e = build_and_load_spec(src, csrc_dir, cache_dir, (flags & 1) != 0, h->spec);
    if (!e.empty()) return fail(h, CB200_ECUDA, e);
    h->spec_gen[0] = h->lu_gen[0];
    h->spec_gen[1] = h->lu_gen[1];
    h->spec_method = method;
    h->spec_limit = want_limit;
    return CB200_OK;
}

// Lanes on which a refactor of the last cb200_dc / cb200_tran* met a weak pivot under the static
// order (multiplier beyond 1e8; lane_kernels.cuh: weak_pivot).  Waits for the handle's stream.
extern "C" int cb200_weak_pivot_lanes(cb200_handle *h, int32_t *flags, int64_t *count)
{
    if (!h || (!flags && !count)) return fail(h, CB200_EINVAL, "cb200_weak_pivot_lanes: null argument");
    if (h->P <= 0) return fail(h, CB200_ESTATE, "cb200_weak_pivot_lanes: call cb200_set_lanes first");
    cudaSetDevice(h->device);
    std::vector<int> f((size_t)h->P);
    CUDA_TRY(h, cudaMemcpyAsync(f.data(), h->d_weak.p, (size_t)h->P * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    int64_t c = 0;
    for (int64_t l = 0; l < h->P; l++) { if (flags) flags[l] = f[l] != 0; c += f[l] != 0; }
    if (count) *count = c;
    return CB200_OK;
}

extern "C" int cb200_is_specialized(const cb200_handle *h) { return h && spec_usable(h) ? 1 : 0; }

// Host-only test hook (no device): pattern + static-pivot schedule + level schedule of a
// description, and both schedules executed on the host for one matrix.  info = {n, nnz, nlu,
// factor levels, forward levels, backward levels}.
static int host_lu_check_impl(const cb200_desc *d, const double *absJ, const double *absJmin, const double *J_nz,
                              const double *rhs, double *x_serial, double *x_level, int64_t *colptr, int64_t *rowval,
                              int32_t *info);

extern "C" int cb200_host_lu_check(const cb200_desc *d, const double *J_nz, const double *rhs,
                                   double *x_serial, double *x_level, int64_t *colptr, int64_t *rowval,
                                   int32_t *info)
{
    return host_lu_check_impl(d, nullptr, nullptr, J_nz, rhs, x_serial, x_level, colptr, rowval, info);
}

// The same with the pivot order chosen from OTHER magnitudes than the matrix that is factored: absJ
// plays the probed magnitudes of cb200_analyze, J_nz a Jacobian met later in the Newton loop.
extern "C" int cb200_host_lu_check_static(const cb200_desc *d, const double *absJ, const double *absJmin,
                                          const double *J_nz, const double *rhs, double *x_serial,
                                          double *x_level, int32_t *info)
{
    if (!absJ) { g_last_error = "cb200_host_lu_check_static: null argument"; return CB200_EINVAL; }
    return host_lu_check_impl(d, absJ, absJmin, J_nz, rhs, x_serial, x_level, nullptr, nullptr, info);
}

static int host_lu_check_impl(const cb200_desc *d, const double *absJ, const double *absJmin, const double *J_nz,
                              const double *rhs, double *x_serial, double *x_level, int64_t *colptr, int64_t *rowval,
                              int32_t *info)
{
    if (!d || !info) { g_last_error = "cb200_host_lu_check: null argument"; return CB200_EINVAL; }
    Structure st;
    std::string e = build_structure(*d, st);
    if (!e.empty()) { g_last_error = e; return CB200_EINVAL; }
    info[0] = st.n; info[1] = (int32_t)st.nnz; info[2] = info[3] = info[4] = info[5] = 0;
    if (colptr) for (int j = 0; j <= st.n; j++) colptr[j] = st.colptr[j] + 1;
    if (rowval) for (int64_t q = 0; q < st.nnz; q++) rowval[q] = st.rowval[q] + 1;
    if (!J_nz) return CB200_OK;
    if (!rhs || !x_serial || !x_level) { g_last_error = "cb200_host_lu_check: null argument"; return CB200_EINVAL; }
    std::vector<double> J(J_nz, J_nz + st.nnz), a(st.nnz), r(rhs, rhs + st.n), xs, xl;
    for (int64_t q = 0; q < st.nnz; q++) a[q] = absJ ? absJ[q] : std::fabs(J[q]);
    std::vector<double> amin;
    if (absJmin) amin.assign(absJmin, absJmin + st.nnz);
    LuSchedule S;
    e = analyze_lu(st, a, 1e-3, S, absJmin ? &amin : nullptr);
    if (!e.empty()) { g_last_error = e; return CB200_ESINGULAR; }
    LevelSchedule V;
    build_level_schedule(S, V);
    info[2] = (int32_t)S.nlu; info[3] = V.n_lev; info[4] = V.n_fwd; info[5] = V.n_bwd;
    host_lu_solve(S, V, J, r, xs, xl);
    std::copy(xs.begin(), xs.end(), x_serial);
    std::copy(xl.begin(), xl.end(), x_level);
    return CB200_OK;
}

extern "C" int cb200_lane_mapping(const cb200_handle *h)
{
    if (!h) return CB200_EINVAL;
    if (use_block_kernels(h->prog, h->smem_limit, h->block_pref)) return 3;
    if (use_warp_kernels(h->prog.n_slots, h->smem_limit, h->block_pref)) return 2;
    return choose_block(h->prog.n_slots, h->smem_limit, h->block_pref) == 0 ? 1 : 0;
}

// Host-only view of the emitter (no device needed): structure + LU analysis from
// caller-supplied nominal magnitudes |J| (DC and transient) -> generated CUDA source.
// Used to unit-test the emitter where no GPU is present; returns the source length.
extern "C" int64_t cb200_emit_source(const cb200_desc *d, const double *absJ_dc, const double *absJ_tr,
                                     int32_t method, int64_t P, int32_t num_sms, char *out, int64_t cap)
{
    if (!d || !absJ_dc || !absJ_tr) { g_last_error = "cb200_emit_source: null argument"; return CB200_EINVAL; }
    cb200_handle h;
    std::string e = build_structure(*d, h.st);
    if (!e.empty()) { g_last_error = e; return CB200_EINVAL; }
    const int nd = d->n_devices;
    h.dev_kind = to_int(d->dev_kind, nd); h.dev_flags = to_int(d->dev_flags, nd);
    h.dev_node_ptr = to_int(d->dev_node_ptr, nd + 1);
    h.dev_nodes = to_int(d->dev_nodes, nd ? d->dev_node_ptr[nd] : 0);
    h.dev_param_ptr = to_int(d->dev_param_ptr, nd + 1);
    h.dev_params = to_int(d->dev_params, nd ? d->dev_param_ptr[nd] : 0);
    h.dev_gbase = to_int64(d->dev_gbase, nd + 1); h.dev_cbase = to_int64(d->dev_cbase, nd + 1);
    h.dev_bbase = to_int64(d->dev_bbase, nd + 1);
    h.dev_sbase = d->dev_state_ptr ? to_int(d->dev_state_ptr, nd + 1) : std::vector<int>(nd + 1, 0);
    h.uniform.assign(d->uniform, d->uniform + d->n_uniform);
    h.limit_init_ref = to_int(d->limit_init_ref, d->n_limits);
    h.n_lane_cols = d->n_lane_cols;
    for (int i = 0; i < nd; i++) {
        if (is_source_kind(h.dev_kind[i])) {
            h.src_list.push_back(i);
            bool uni = true;
            for (int q = h.dev_param_ptr[i]; q < h.dev_param_ptr[i + 1]; q++) uni &= h.dev_params[q] >= 0;
            h.src_uniform.push_back(uni ? 1 : 0);
        }
        if (is_nonlinear_kind(h.dev_kind[i])) h.nl_list.push_back(i);
    }
    std::vector<double> a0(absJ_dc, absJ_dc + h.st.nnz), a1(absJ_tr, absJ_tr + h.st.nnz);
    e = analyze_lu(h.st, a0, 1e-3, h.lu[0].host);
    if (e.empty()) e = analyze_lu(h.st, a1, 1e-3, h.lu[1].host);
    if (!e.empty()) { g_last_error = e; return CB200_ESINGULAR; }
    layout_workspace(&h);
    const SpecInput in = spec_input(h, method, P, num_sms);
    const std::string src = generate_spec_source(in);
    if (out && cap > 0) {
        const int64_t m = std::min<int64_t>(cap - 1, (int64_t)src.size());
        memcpy(out, src.data(), m);
        out[m] = 0;
    }
    return (int64_t)src.size();
}

extern "C" int cb200_wave_info(const cb200_wave *w, int64_t *T, int64_t *P, int32_t *n_save,
                               int32_t *adaptive)
{
    if (!w) return CB200_EINVAL;
    if (!w->h) return fail(nullptr, CB200_ESTATE, "cb200_wave_info: the wave's handle was destroyed");
    if (T) *T = w->T;
    if (P) *P = w->P;
    if (n_save) *n_save = w->n_save;
    if (adaptive) *adaptive = w->adaptive;
    return CB200_OK;
}

extern "C" int cb200_wave_fetch(cb200_wave *w, double *t, double *u, int32_t *count, int32_t *status,
                                int32_t *newton_iters)
{
    return wave_fetch_impl(w, t, u, 0, 0, count, status, newton_iters);
}

extern "C" int cb200_wave_fetch_ld(cb200_wave *w, double *t, double *u, int64_t u_ld, int64_t t_ld,
                                   int32_t *count, int32_t *status, int32_t *newton_iters)
{
    return wave_fetch_impl(w, t, u, u_ld, t_ld, count, status, newton_iters);
}

static int wave_fetch_impl(cb200_wave *w, double *t, double *u, int64_t u_ld, int64_t t_ld, int32_t *count,
                           int32_t *status, int32_t *newton_iters)
{
    if (!w) return CB200_EINVAL;
    cb200_handle *h = w->h;
    if (!h) return fail(nullptr, CB200_ESTATE, "cb200_wave_fetch: the wave's handle was destroyed");
    if (u_ld == 0) u_ld = w->P;
    if (t_ld == 0) t_ld = w->P;
    if (u_ld < w->P || t_ld < w->P) return fail(h, CB200_EINVAL, "cb200_wave_fetch: leading dimension smaller than the lane count");
    cudaSetDevice(h->device);
    cudaStream_t s = h->stream;
    CUDA_TRY(h, cudaEventRecord(h->ev0, s));
    int64_t bytes = 0;
    if (u && w->n_save > 0) {
        CUDA_TRY(h, cudaMemcpy2DAsync(u, (size_t)u_ld * sizeof(double), w->d_out.p, (size_t)w->P * sizeof(double),
                                      (size_t)w->P * sizeof(double), (size_t)w->n_save * w->T, cudaMemcpyDeviceToHost, s));
        bytes += (int64_t)w->n_save * w->T * w->P * sizeof(double);
    }
    if (status) { CUDA_TRY(h, cudaMemcpyAsync(status, w->d_status.p, w->P * sizeof(int), cudaMemcpyDeviceToHost, s)); bytes += w->P * 4; }
    if (newton_iters) { CUDA_TRY(h, cudaMemcpyAsync(newton_iters, w->d_iters.p, w->P * sizeof(int), cudaMemcpyDeviceToHost, s)); bytes += w->P * 4; }
    if (w->adaptive) {
        if (t) {
            CUDA_TRY(h, cudaMemcpy2DAsync(t, (size_t)t_ld * sizeof(double), w->d_t.p, (size_t)w->P * sizeof(double),
                                          (size_t)w->P * sizeof(double), (size_t)w->T, cudaMemcpyDeviceToHost, s));
            bytes += (int64_t)w->T * w->P * sizeof(double);
        }
        if (count) CUDA_TRY(h, cudaMemcpyAsync(count, w->d_count.p, w->P * sizeof(int), cudaMemcpyDeviceToHost, s));
    }
    CUDA_TRY(h, cudaEventRecord(h->ev1, s));
    CUDA_TRY(h, cudaStreamSynchronize(s));
    float ms = 0; cudaEventElapsedTime(&ms, h->ev0, h->ev1);
    h->stats.d2h_ms = ms;
    h->stats.d2h_bytes = bytes;
    if (!w->adaptive) {
        if (t) {
            int64_t q = 0;
            t[q++] = w->t0;
            for (int64_t k = 1; k <= w->nsteps; k++)
                if (k % w->save_every == 0 || k == w->nsteps) t[q++] = w->t0 + (double)k * w->dt;
        }
        if (count) for (int64_t l = 0; l < w->P; l++) count[l] = (int32_t)w->T;
    }
    if (newton_iters) {
        int64_t tot = 0;
        for (int64_t l = 0; l < w->P; l++) tot += newton_iters[l];
        h->stats.newton_iters = tot;
    }
    return CB200_OK;
}

extern "C" int cb200_wave_final_state(cb200_wave *w, double *x_out)
{
    if (!w || !x_out) return CB200_EINVAL;
    cb200_handle *h = w->h;
    if (!h) return fail(nullptr, CB200_ESTATE, "cb200_wave_final_state: the wave's handle was destroyed");
    cudaSetDevice(h->device);
    CUDA_TRY(h, cudaMemcpyAsync(x_out, w->d_final.p, (size_t)w->n * w->P * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    return CB200_OK;
}

extern "C" void cb200_wave_free(cb200_wave *w)
{
    if (!w) return;
    if (w->h) {
        cudaSetDevice(w->h->device);
        auto &v = w->h->waves;
        v.erase(std::remove(v.begin(), v.end(), w), v.end());
    }
    delete w;
}

// Test hook: evaluates the device-side junction exp (lane_kernels.cuh: d_exp) on host data.
extern "C" int cb200_debug_exp(const double *x, double *y, int32_t n)
{
    if (!x || !y || n <= 0) return CB200_EINVAL;
    double *dx = nullptr, *dy = nullptr;
    if (cudaMalloc((void **)&dx, n * sizeof(double)) != cudaSuccess) return fail(nullptr, CB200_ENODEVICE, "cb200_debug_exp: no device");
    cudaMalloc((void **)&dy, n * sizeof(double));
    cudaMemcpy(dx, x, n * sizeof(double), cudaMemcpyHostToDevice);
    cudaError_t e = launch_debug_exp(dx, dy, n, 0);
    if (e == cudaSuccess) e = cudaMemcpy(y, dy, n * sizeof(double), cudaMemcpyDeviceToHost);
    cudaFree(dx); cudaFree(dy);
    return e == cudaSuccess ? CB200_OK : fail(nullptr, CB200_ECUDA, cudaGetErrorString(e));
}

// ---------------------------------------------------------------------------
// FP64 roofline support: a measured FMA peak and the static flop model of the
// per-iteration linear algebra (SURVEY 8d: "measure once with an FMA microbenchmark").
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) cb200_fp64_fma_kernel(double *out, int iters, double a, double b)
{
    // 8 independent dependent-FMA chains per thread, 64 resident warps per SM: the FP64 pipe is
    // the only limiter (no memory traffic, no other pipe in the loop)
    double x0 = threadIdx.x * 1e-3, x1 = x0 + 1.0, x2 = x0 + 2.0, x3 = x0 + 3.0;
    double x4 = x0 + 4.0, x5 = x0 + 5.0, x6 = x0 + 6.0, x7 = x0 + 7.0;
#pragma unroll 4
    for (int i = 0; i < iters; i++) {
        x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
        x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
    }
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
}

extern "C" int cb200_measure_fp64_peak(int32_t device, double *tflops, double *ms_out)
{
    if (!tflops) return fail(nullptr, CB200_EINVAL, "cb200_measure_fp64_peak: null argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev)
        return fail(nullptr, CB200_ENODEVICE, "cb200_measure_fp64_peak: no usable CUDA device");
    cudaSetDevice(device);
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 1 << 15;
    double *d = nullptr;
    if (cudaMalloc((void **)&d, (size_t)blocks * threads * sizeof(double)) != cudaSuccess)
        return fail(nullptr, CB200_ENOMEM, "cb200_measure_fp64_peak: allocation failed");
    cudaStream_t s;
    cudaEvent_t e0, e1;
    cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    float best = 1e30f;
    for (int rep = 0; rep < 6; rep++) {               // first launches warm the clocks up
        cudaEventRecord(e0, s);
        cb200_fp64_fma_kernel<<<blocks, threads, 0, s>>>(d, iters, 0.999999, 1e-9);
        cudaEventRecord(e1, s);
        cudaError_t ce = cudaStreamSynchronize(s);
        if (ce != cudaSuccess) {
            cudaFree(d);
            return fail(nullptr, CB200_ECUDA, std::string("cb200_measure_fp64_peak: ") + cudaGetErrorString(ce));
        }
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        if (rep >= 2 && ms < best) best = ms;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaStreamDestroy(s); cudaFree(d);
    const double flops = 2.0 * 8.0 * (double)iters * (double)blocks * (double)threads;
    *tflops = flops / ((double)best * 1e-3) / 1e12;
    if (ms_out) *ms_out = best;
    return CB200_OK;
}

// Static flop counts of ONE Newton iteration's linear algebra for this circuit (adds, multiplies
// and FMAs as 1 / 1 / 2; each reciprocal counted as ONE flop): out[0..1] assembly + residual
// (DC, transient), out[2..3] numeric refactor, out[4..5] both triangular solves, out[6] update,
// out[7] number of device rows evaluated per iteration (nonlinear devices).
extern "C" int cb200_flop_model(const cb200_handle *h, int64_t *out)
{
    if (!h || !out) return CB200_EINVAL;
    const Structure &st = h->st;
    int64_t asm_dc = 0, asm_tr = 3LL * st.n;          // du_j = gamma (u_j - un_j) + dterm_j
    for (int64_t s = 0; s < st.nnz; s++) {
        const int64_t ng = st.gseg_ptr[s + 1] - st.gseg_ptr[s], nc = st.cseg_ptr[s + 1] - st.cseg_ptr[s];
        asm_dc += ng + 2; asm_tr += ng + 2;           // segment sum, F += gsum * u_j
        if (nc > 0) asm_tr += nc + 4;                 // segment sum, F += csum * du_j, J += gamma * csum
    }
    for (int r = 0; r < st.n; r++) {
        const int64_t nb = st.bseg_ptr[r + 1] - st.bseg_ptr[r];
        asm_dc += nb + 3; asm_tr += nb + 3;           // segment sum, F -= b, ||F||^2 += F^2
    }
    out[0] = asm_dc; out[1] = asm_tr;
    for (int w = 0; w < 2; w++) {
        const LuSchedule &S = h->lu[w].host;
        int64_t fac = 0, sol = 0;
        if (S.valid) {
            fac = S.n + (int64_t)S.L_slot.size() + 2LL * (int64_t)S.tgt.size();
            sol = 2LL * (int64_t)S.L_slot.size() + 2LL * (int64_t)S.U_slot.size() + S.n;
        }
        out[2 + w] = fac; out[4 + w] = sol;
    }
    out[6] = st.n;
    out[7] = (int64_t)h->nl_list.size();
    return CB200_OK;
}

extern "C" int cb200_get_stats(const cb200_handle *h, cb200_stats *out)
{
    if (!h || !out) return CB200_EINVAL;
    *out = h->stats;
    return CB200_OK;
}
