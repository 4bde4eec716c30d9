// cpd_b200.cu -- host side of libcpd_b200.so: the C ABI declared in include/cpd_b200.h.
// One handle = one device + one stream; every EM iteration is a fixed sequence of launches on
// that stream (pack, pass 1, finalize 1, pass 2, finalize 2, moments [+ all-reduce] + M-step).
#include "cpd_b200.h"
#include "kernels.cuh"
#include "lowrank.cuh"
#include "gram_i8.cuh"

#include <cub/device/device_radix_sort.cuh>
#ifdef CPD_HOST_EMU
#include "emu_nccl.h"
#include "emu_solver.h"
#endif

#include <dlfcn.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

using namespace cpd;

// ---------------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(CPD_ERR_CUDA, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(e_)); \
    } while (0)
#define KCHECK() CU(cudaGetLastError())

extern "C" const char* cpd_last_error(void) { return g_err; }
extern "C" int cpd_version(void) { return 100; }
extern "C" int cpd_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

// ---------------------------------------------------------------------------------------------
// NCCL, bound at run time (libnccl.so.2 -- torch's bundled copy if it is already loaded)
// ---------------------------------------------------------------------------------------------
namespace {
typedef struct { char internal[128]; } nccl_uid;
typedef void* nccl_comm;
struct NcclApi {
    void* lib = nullptr;
    int (*GetUniqueId)(nccl_uid*) = nullptr;
    int (*CommInitRank)(nccl_comm*, int, nccl_uid, int) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, nccl_comm, cudaStream_t) = nullptr;
    int (*CommDestroy)(nccl_comm) = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
NcclApi g_nccl;
int load_nccl() {
    if (g_nccl.lib) return CPD_OK;
#ifdef CPD_HOST_EMU   // CPU test build (tests/emu): ranks are threads of one process, the collective is a rendezvous
    static_assert(sizeof(nccl_uid) == sizeof(emu::nccl_uid_t), "unique id layout");
    g_nccl.GetUniqueId = reinterpret_cast<int (*)(nccl_uid*)>(emu::ncclGetUniqueId);
    g_nccl.CommInitRank = reinterpret_cast<int (*)(nccl_comm*, int, nccl_uid, int)>(emu::ncclCommInitRank);
    g_nccl.AllReduce = emu::ncclAllReduce;
    g_nccl.CommDestroy = emu::ncclCommDestroy;
    g_nccl.GetErrorString = emu::ncclGetErrorString;
    g_nccl.lib = (void*)&g_nccl;
    return CPD_OK;
#endif
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    void* lib = nullptr;
    for (const char* nm : names) { lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL); if (lib) break; }
    if (!lib) return fail(CPD_ERR_NCCL, "cannot dlopen libnccl.so.2: %s", dlerror());
    g_nccl.GetUniqueId = (int (*)(nccl_uid*))dlsym(lib, "ncclGetUniqueId");
    g_nccl.CommInitRank = (int (*)(nccl_comm*, int, nccl_uid, int))dlsym(lib, "ncclCommInitRank");
    g_nccl.AllReduce = (int (*)(const void*, void*, size_t, int, int, nccl_comm, cudaStream_t))dlsym(lib, "ncclAllReduce");
    g_nccl.CommDestroy = (int (*)(nccl_comm))dlsym(lib, "ncclCommDestroy");
    g_nccl.GetErrorString = (const char* (*)(int))dlsym(lib, "ncclGetErrorString");
    if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllReduce || !g_nccl.CommDestroy)
        return fail(CPD_ERR_NCCL, "libnccl lacks an expected symbol");
    g_nccl.lib = lib;
    return CPD_OK;
}
constexpr int NCCL_DOUBLE = 8, NCCL_SUM = 0;

// cuSOLVER (dense LU of the non-rigid M-step only), bound at run time like NCCL
struct SolverApi {
    void* lib = nullptr;
    int (*Create)(void**) = nullptr;
    int (*Destroy)(void*) = nullptr;
    int (*SetStream)(void*, cudaStream_t) = nullptr;
    int (*CreateParams)(void**) = nullptr;
    int (*DestroyParams)(void*) = nullptr;
    int (*XgetrfBuf)(void*, void*, int64_t, int64_t, int, const void*, int64_t, int, size_t*, size_t*) = nullptr;
    int (*Xgetrf)(void*, void*, int64_t, int64_t, int, void*, int64_t, int64_t*, int, void*, size_t, void*, size_t, int*) = nullptr;
    int (*Xgetrs)(void*, void*, int, int64_t, int64_t, int, const void*, int64_t, const int64_t*, int, void*, int64_t, int*) = nullptr;
};
SolverApi g_sol;
int load_cusolver() {
    if (g_sol.lib) return CPD_OK;
#ifdef CPD_HOST_EMU   // CPU test build (tests/emu): documented-behaviour stand-ins instead of the real library
    g_sol.Create = emu::solverCreate; g_sol.Destroy = emu::solverDestroy; g_sol.SetStream = emu::solverSetStream;
    g_sol.CreateParams = emu::solverCreateParams; g_sol.DestroyParams = emu::solverDestroyParams;
    g_sol.XgetrfBuf = emu::solverXgetrfBuf; g_sol.Xgetrf = emu::solverXgetrf; g_sol.Xgetrs = emu::solverXgetrs;
    g_sol.lib = (void*)&g_sol;
    return CPD_OK;
#endif
    const char* names[] = {"libcusolver.so.11", "/usr/local/cuda/lib64/libcusolver.so.11", "libcusolver.so"};
    void* lib = nullptr;
    for (const char* nm : names) { lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL); if (lib) break; }
    if (!lib) return fail(CPD_ERR_CUDA, "cannot dlopen libcusolver.so.11: %s", dlerror());
#define SOLSYM(field, name) g_sol.field = (decltype(g_sol.field))dlsym(lib, name)
    SOLSYM(Create, "cusolverDnCreate");
    SOLSYM(Destroy, "cusolverDnDestroy");
    SOLSYM(SetStream, "cusolverDnSetStream");
    SOLSYM(CreateParams, "cusolverDnCreateParams");
    SOLSYM(DestroyParams, "cusolverDnDestroyParams");
    SOLSYM(XgetrfBuf, "cusolverDnXgetrf_bufferSize");
    SOLSYM(Xgetrf, "cusolverDnXgetrf");
    SOLSYM(Xgetrs, "cusolverDnXgetrs");
#undef SOLSYM
    if (!g_sol.Create || !g_sol.SetStream || !g_sol.CreateParams || !g_sol.XgetrfBuf || !g_sol.Xgetrf || !g_sol.Xgetrs)
        return fail(CPD_ERR_CUDA, "libcusolver lacks an expected symbol");
    g_sol.lib = lib;
    return CPD_OK;
}
constexpr int CUDA_R_64F_ = 1, CUBLAS_OP_T_ = 1;
}  // namespace
#define SOLV(call)                                                                          \
    do {                                                                                    \
        int r_ = (call);                                                                    \
        if (r_ != 0) return fail(CPD_ERR_CUDA, "%s failed with cusolverStatus %d", #call, r_); \
    } while (0)
#define NC(call)                                                                                                   \
    do {                                                                                                           \
        int r_ = (call);                                                                                           \
        if (r_ != 0)                                                                                               \
            return fail(CPD_ERR_NCCL, "%s failed: %s", #call, g_nccl.GetErrorString ? g_nccl.GetErrorString(r_) : "?"); \
    } while (0)

// ---------------------------------------------------------------------------------------------
// handle
// ---------------------------------------------------------------------------------------------
struct cpd_ctx {
    int device = 0, dim = 3, sm_count = 148, slots1 = 296, slots2 = 296;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    long long m = 0, mpad = 0, n = 0, npad = 0, n_global = 0;
    double *d_yc = nullptr, *d_ts = nullptr, *d_xc = nullptr, *d_raw = nullptr;
    size_t raw_cap = 0;
    float4 *d_srcP = nullptr, *d_srcJ = nullptr, *d_tgtP = nullptr, *d_tgtQ = nullptr;
    P1Part* d_part1 = nullptr;
    double* d_part2 = nullptr;
    size_t part1_cap = 0, part2_cap = 0;
    double *d_pt1 = nullptr, *d_p1 = nullptr, *d_pxc = nullptr, *d_px = nullptr;
    double *d_mom_src = nullptr, *d_mom_tgt = nullptr, *d_mom = nullptr, *d_sums = nullptr;
    size_t mom_src_cap = 0, mom_tgt_cap = 0, sums_cap = 0;
    DevState* d_state = nullptr;
    DevState h_state;
    double* h_pin = nullptr;   // 64 pinned doubles for small D2H reads
    double* d_frame = nullptr;          // [2][8]: what cloud_frame_kernel derives per cloud (sources, targets)
    double* h_stats = nullptr;          // [2][9] pinned: the clouds' statistics on their way to the host (ensure_stats)
    cudaEvent_t stats_ev = nullptr, copy_ev = nullptr;
    int stats_pending = 0;              // bit 0: sources, bit 1: targets
    long long stats_count[2] = {0, 0};
    bool origin_given = false;
    int it1 = 0, it2 = 0, j1 = 1, j2 = 1, g1 = 1, g2 = 1;   // i-tiles, max partial slots per tile, work items (= grid)
    // exact culling of far blocks (late iterations): stage bounding boxes, per-stage max offset
    float4 *d_sbox = nullptr, *d_tbox = nullptr, *d_ssub = nullptr, *d_tsub = nullptr;
    float *d_omax = nullptr, *d_omax_sub = nullptr;
    bool cull_on = true, cull_active = false;
    double extent = 0.0;              // largest bounding-box edge of the target shard (caller units)
    int4 *d_work1 = nullptr, *d_work2 = nullptr;
    int *d_slots1 = nullptr, *d_slots2 = nullptr;
    bool have_source = false, have_target = false, have_state = false, prepared = false;
    nccl_comm comm = nullptr;
    int world = 1, rank = 0;
    // Morton ordering (internal permutation; results leave in the caller's order)
    int *d_perm_src = nullptr, *d_perm_tgt = nullptr, *d_idx_tmp = nullptr;
    unsigned *d_codes = nullptr, *d_codes_out = nullptr;
    size_t sort_cap = 0, sort_tmp_cap = 0;
    void* d_sort_tmp = nullptr;
    double *d_outN = nullptr, *d_outM = nullptr;      // staging for un-permuted outputs / permuted inputs
    // non-rigid CPD (dense G)
    float* d_G = nullptr;
    double *d_W = nullptr, *d_A = nullptr, *d_B = nullptr, *d_ts2 = nullptr, *d_nrpart = nullptr;
    int64_t* d_ipiv = nullptr;
    int* d_info = nullptr;
    void *d_work = nullptr, *h_work = nullptr, *sol = nullptr, *sol_params = nullptr;
    size_t work_dev = 0, work_host = 0;
    long long nr_m = 0;
    double nr_lmd = 0.0;
    bool nr_ready = false;
    // weighted E-step (BCPD): per-source exponent offsets and the {log2 c, dead-column shift} pair for finalize 1
    float* d_la = nullptr;
    size_t la_cap = 0;
    double* d_log2c = nullptr;
    bool wgt_on = false;
    // correspondence priors of ConstrainedNonRigidCPD
    double *d_wgt = nullptr, *d_p1t = nullptr, *d_pxt = nullptr;
    long long prior_m = 0;
    double prior_alpha = 1.0;
    bool prior_on = false;
    // non-rigid CPD, rank-K G ~= Q Bc Q^T (lowrank.cuh)
    int lr_rank = 0;                      // > 0: cpd_nonrigid_step takes the low-rank M-step
    bool lr_w_stale = false;              // W of the low-rank path is formed on demand
    float lr_setup_ms[3] = {0.f, 0.f, 0.f};   // products / orthonormalisations / core of the last profiled set-up
    long long lr_m = 0;
    int lr_cap = 0;
    float4* d_lr_pts = nullptr;
    double *d_lr_Q = nullptr, *d_lr_X = nullptr, *d_lr_coef = nullptr, *d_lr_part = nullptr, *d_lr_Bc = nullptr, *d_lr_S = nullptr,
           *d_lr_R = nullptr, *d_lr_sys = nullptr, *d_lr_rhs = nullptr, *d_lr_c = nullptr, *d_lr_out = nullptr, *d_lr_panel = nullptr, *d_lr_Lt = nullptr;
    bool lr_spd = true;                   // symmetric positive definite K x K system on Qt = Q L (lr_spd_form); CPD_B200_LR_CORE=lu: LU of (c I + Bc S)
    size_t lr_part_cap = 0;               // doubles in d_lr_part (slice partials of lr_inner)
    unsigned char* d_gi_planes = nullptr;                      // exact int8-digit product: digit planes of X, FP64 chunk partials, column maxima
    double *d_gi_part = nullptr, *d_gi_colmax = nullptr;
    size_t gi_planes_cap = 0, gi_part_cap = 0, gi_colmax_cap = 0, gi_pairs_cap = 0;
    float4* d_gi_pairs = nullptr;                            // the scaled source points as packed pair records (generators' f32x2 maths)
    size_t lr_out_cap = 0;
    P2PMailbox* d_box = nullptr;          // this rank's mailbox (peers write into it)
    P2PInfo* d_p2p = nullptr;             // device copy of the peer table; non-null => fused P2P exchange
    void* peer_ptr[P2P_MAX] = {nullptr};  // mappings opened with cudaIpcOpenMemHandle
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, sev[7] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    bool profiling = false;
    int64_t launches = 0;
    // the fused EM iteration as a CUDA graph (cpd_em_step): one graph launch instead of 7-12 kernel launches per iteration
    DevState* h_state_ring = nullptr;     // pinned staging slots of upload_state
    cudaEvent_t state_ev[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    int state_slot = 0;
    bool graph_on = true;
    cudaGraphExec_t em_graph = nullptr;
    int em_graph_key = -1, em_graph_launches = 0, prepare_gen = 0;
    void* d_flush = nullptr;
    size_t flush_cap = 0;
    std::vector<cudaEvent_t> pool;
};

namespace {
constexpr int STATE_RING = 8;
template <typename T>
int dev_alloc(T** p, size_t count) {
    if (*p) { cudaFree(*p); *p = nullptr; }
    cudaError_t e = cudaMalloc((void**)p, std::max<size_t>(count, 1) * sizeof(T));
    if (e != cudaSuccess) return fail(CPD_ERR_CUDA, "cudaMalloc(%zu bytes) failed: %s", count * sizeof(T), cudaGetErrorString(e));
    return CPD_OK;
}
#define TRY(x) do { int r__ = (x); if (r__ != CPD_OK) return r__; } while (0)
// device buffer of a stateless entry point: freed on every exit path
template <typename T>
struct DevBuf {
    T* p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    int alloc(size_t count) { return dev_alloc(&p, count); }
};

inline unsigned blocks_for(long long n) { return (unsigned)((n + THREADS - 1) / THREADS); }

// Work list of one pass: every i-tile is cut into J contiguous stage ranges ("splits"), one CTA each; J is chosen to
// minimise the makespan  ceil(ntiles*J / slots) * (ceil(nstages/J) + pipeline fill)  over the resident CTA slots, and slots
// left over in a single-wave launch go to extra splits of the first tiles.  All tiles carry the same work, so this is within
// one stage of the optimum whatever N, M and the GPU count are.  (A finer "stream-K" cut that lets one CTA span two tiles was
// measured 15-19 % slower: the extra live state pushes the hot loops past 128 registers.)
struct WorkList {
    std::vector<int4> items;        // {tile, first unit, end unit, slot within the tile}; a unit is a sub-chunk of SUB j-records
    std::vector<int> tile_slots;    // partial slots used per tile
    int max_slots = 1;
};
// Cut ntiles x nunits of work into CTA work items for `slots` resident CTAs.  A tile costs `nunits` (the last one, whose warps
// beyond the end of the i-points leave the kernel at once, `last_cost` = live warps / warps per CTA of that).  Two candidates:
//   * one wave (ntiles <= slots): every tile starts with one item; the next cut always goes to the tile whose longest item is the most
//     expensive, until the slots are used up -- cuts land where the cost is, at the granularity of a sub-chunk (an item may begin
//     and end inside a TMA stage; the kernels load the whole stages and skip the sub-chunks outside the item);
//   * several waves: the same number of cuts j for every tile, j chosen by waves x (item length + item overhead).
// `overhead`: what an item costs before its first unit (offset seeding sweep, pipeline fill), in units: half a stage.
WorkList build_work(int ntiles, int nunits, int slots, double last_cost, double overhead) {
    const double OVERHEAD = overhead;
    WorkList w;
    nunits = std::max(1, nunits);
    auto cost_of = [&](int t) { return t == ntiles - 1 ? last_cost : 1.0; };
    auto span_of = [&](int t, int j) { return cost_of(t) * (double)((nunits + j - 1) / j) + OVERHEAD; };
    // several waves, uniform j
    int best_j = 1;
    double best = 1e300;
    for (int j = 1; j <= nunits; ++j) {
        const long long items = (long long)ntiles * j;
        const double waves = ceil((double)items / slots);
        const double span = waves * ((double)((nunits + j - 1) / j) + OVERHEAD);
        if (span < best - 1e-9) { best = span; best_j = j; }
        if (items > 8LL * slots) break;
    }
    w.tile_slots.assign(ntiles, best_j);
    if (ntiles <= slots) {
        // one wave, cuts by cost
        std::vector<int> cuts(ntiles, 1);
        int used = ntiles;
        while (used < slots) {
            int worst = -1;
            double wv = -1.0;
            for (int t = 0; t < ntiles; ++t) {
                const double v = span_of(t, cuts[t]);
                if (cuts[t] < nunits && v > wv) { wv = v; worst = t; }
            }
            if (worst < 0) break;
            ++cuts[worst];
            ++used;
        }
        double span = 0.0;
        for (int t = 0; t < ntiles; ++t) span = std::max(span, span_of(t, cuts[t]));
        if (span <= best + 1e-9) w.tile_slots = cuts;
    }
    for (int t = 0; t < ntiles; ++t) {
        const int j = w.tile_slots[t];
        for (int s = 0; s < j; ++s) {
            const int a = (int)((long long)nunits * s / j), b = (int)((long long)nunits * (s + 1) / j);
            w.items.push_back(make_int4(t, a, b, s));
        }
        w.max_slots = std::max(w.max_slots, j);
    }
    // longest (most expensive) first: the hardware hands CTAs out in order
    std::stable_sort(w.items.begin(), w.items.end(), [&](const int4& a, const int4& b) {
        return cost_of(a.x) * (a.z - a.y) > cost_of(b.x) * (b.z - b.y);
    });
    return w;
}

// Stream-ordered, no synchronise: the state goes through a small ring of pinned staging slots (a cudaMemcpyAsync from pageable
// memory would synchronise the stream first); a slot is re-used only after the copy that last read it has completed.
int ensure_stats(cpd_ctx* h);
int upload_state(cpd_ctx* h) {
    TRY(ensure_stats(h));
    if (!h->h_state_ring) {
        CU(cudaMallocHost((void**)&h->h_state_ring, STATE_RING * sizeof(DevState)));
        for (int k = 0; k < STATE_RING; ++k) CU(cudaEventCreateWithFlags(&h->state_ev[k], cudaEventDisableTiming));
    }
    const int k = h->state_slot;
    h->state_slot = (k + 1) % STATE_RING;
    CU(cudaEventSynchronize(h->state_ev[k]));                  // never recorded: returns at once
    h->h_state_ring[k] = h->h_state;
    CU(cudaMemcpyAsync(h->d_state, &h->h_state_ring[k], sizeof(DevState), cudaMemcpyHostToDevice, h->stream));
    CU(cudaEventRecord(h->state_ev[k], h->stream));
    return CPD_OK;
}

// copy a host cloud (count x dim doubles) into a device count x 3 array
int upload_cloud(cpd_ctx* h, const double* src, long long count, double* dst3) {
    if (h->dim == 3) {
        CU(cudaMemcpyAsync(dst3, src, (size_t)count * 3 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    } else {
        CU(cudaMemsetAsync(dst3, 0, (size_t)count * 3 * sizeof(double), h->stream));
        CU(cudaMemcpy2DAsync(dst3, 3 * sizeof(double), src, 2 * sizeof(double), 2 * sizeof(double), (size_t)count,
                             cudaMemcpyHostToDevice, h->stream));
    }
    return CPD_OK;
}
int download_cloud(cpd_ctx* h, const double* src3, long long count, double* dst) {
    if (h->dim == 3) {
        CU(cudaMemcpyAsync(dst, src3, (size_t)count * 3 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    } else {
        CU(cudaMemcpy2DAsync(dst, 2 * sizeof(double), src3, 3 * sizeof(double), 2 * sizeof(double), (size_t)count,
                             cudaMemcpyDeviceToHost, h->stream));
    }
    return CPD_OK;
}

// d_out[0] = sum |p|^2, d_out[1..3] = sum p   over a device count x 3 cloud; stays on the device (stream-ordered, no sync).
// `part`: blocks_for(count) * 4 doubles of scratch.
int cloud_sums_dev(cpd_ctx* h, const double* d_pts, long long count, double* part, double* d_out) {
    const unsigned nb = blocks_for(count);
    cloud_sums_kernel<<<nb, THREADS, 0, h->stream>>>(d_pts, count, part);
    reduce_cols_kernel<<<1, 4 * 32, 0, h->stream>>>(part, (int)nb, 4, d_out);
    KCHECK();
    h->launches += 2;
    return CPD_OK;
}

// A cloud's way into the library, one stream-ordered sequence without a host round trip: upload -> nine statistics (sums, minima,
// maxima) -> frame (cloud_frame_kernel: Morton box, origin; origin and count patched into the device state) -> Morton sort ->
// out[k] = raw[perm[k]] - origin.  The host copy of the statistics travels behind (pinned h_stats, stats_ev) and is read by
// ensure_stats() when the host first needs the centroid or the extent.  The call returns once the upload itself has been
// consumed (copy_ev), so the caller's buffer is free again, as before.
int ingest_cloud(cpd_ctx* h, const double* host_pts, long long count, int is_target, long long n_global, const double* origin,
                 int* d_perm, double* d_out) {
    if (h->raw_cap < (size_t)count * 3) { TRY(dev_alloc(&h->d_raw, (size_t)count * 3)); h->raw_cap = (size_t)count * 3; }
    const unsigned nb = blocks_for(count);
    if (h->sums_cap < (size_t)nb * 9 + 16) {
        TRY(dev_alloc(&h->d_sums, (size_t)nb * 9 + 16));
        h->sums_cap = (size_t)nb * 9 + 16;
    }
    if (h->sort_cap < (size_t)count) {
        TRY(dev_alloc(&h->d_codes, (size_t)count));
        TRY(dev_alloc(&h->d_codes_out, (size_t)count));
        TRY(dev_alloc(&h->d_idx_tmp, (size_t)count));
        h->sort_cap = (size_t)count;
    }
    size_t need = 0;
    CU(cub::DeviceRadixSort::SortPairs(nullptr, need, h->d_codes, h->d_codes_out, h->d_idx_tmp, d_perm, (int)count, 0, 30, h->stream));
    if (need > h->sort_tmp_cap) {
        if (h->d_sort_tmp) cudaFree(h->d_sort_tmp);
        h->d_sort_tmp = nullptr;
        CU(cudaMalloc(&h->d_sort_tmp, need));
        h->sort_tmp_cap = need;
    }
    TRY(upload_cloud(h, host_pts, count, h->d_raw));
    CU(cudaEventRecord(h->copy_ev, h->stream));
    double* frame = h->d_frame + 8 * is_target;
    stats_kernel<<<nb, THREADS, 0, h->stream>>>(h->d_raw, count, h->d_sums + 16);
    stats_fold_kernel<<<1, 288, 0, h->stream>>>(h->d_sums + 16, (int)nb, h->d_sums);
    cloud_frame_kernel<<<1, 32, 0, h->stream>>>(h->d_sums, count, is_target, n_global, origin != nullptr, origin ? origin[0] : 0.0,
                                                origin ? origin[1] : 0.0, origin ? origin[2] : 0.0, h->d_state, frame);
    CU(cudaMemcpyAsync(h->h_stats + 9 * is_target, h->d_sums, 9 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaEventRecord(h->stats_ev, h->stream));
    h->stats_pending |= 1 << is_target;
    h->stats_count[is_target] = count;
    morton_frame_kernel<<<nb, THREADS, 0, h->stream>>>(h->d_raw, count, frame, h->d_codes, h->d_idx_tmp);
    CU(cub::DeviceRadixSort::SortPairs(h->d_sort_tmp, need, h->d_codes, h->d_codes_out, h->d_idx_tmp, d_perm, (int)count, 0, 30,
                                       h->stream));
    gather3_frame_kernel<<<nb, THREADS, 0, h->stream>>>(h->d_raw, d_perm, count, frame, d_out);
    KCHECK();
    h->launches += 6;
    CU(cudaEventSynchronize(h->copy_ev));
    return CPD_OK;
}

// The host's copy of what cloud_frame_kernel derived on the device (centroid of the sources, frame origin and extent of the targets).
// Every entry point that reads h_state.cx / cy or h->extent, or uploads the host state, calls this first.
int ensure_stats(cpd_ctx* h) {
    if (!h->stats_pending) return CPD_OK;
    CU(cudaEventSynchronize(h->stats_ev));
    if (h->stats_pending & 1)
        for (int a = 0; a < 3; ++a) h->h_state.cy[a] = h->h_stats[a] / (double)h->stats_count[0];
    if (h->stats_pending & 2) {
        const double* t = h->h_stats + 9;
        if (!h->origin_given) for (int a = 0; a < 3; ++a) h->h_state.cx[a] = t[a] / (double)h->stats_count[1];
        h->extent = std::max(t[6] - t[3], std::max(t[7] - t[4], t[8] - t[5]));
    }
    h->stats_pending = 0;
    return CPD_OK;
}

int prepare(cpd_ctx* h) {
    TRY(ensure_stats(h));
    if (h->prepared) return CPD_OK;
    if (!h->have_source || !h->have_target) return fail(CPD_ERR_STATE, "source and target must both be set");
    h->it1 = (int)((h->n + ITILE1 - 1) / ITILE1);
    h->it2 = (int)((h->m + ITILE2 - 1) / ITILE2);
    // Pass 1 cuts at sub-chunks, and the warps of its last i-tile whose i-points are all padding leave the kernel at once.  What such
    // a tile then costs was measured (1/8 and 1/4 target shards of 100k: 2 and 4 of 8 warps alive; profiles/r2_plan_sweep.txt): the
    // best plans come from a cost of 0.6 of a full tile in BOTH cases -- not w / 8: the live warps get a larger share of the SM's
    // pipes, but a warp on its own is latency-bound (0.45 makes the tile's few long items set the time: +10 %; 1.0 wastes the early
    // exit: +2..4 %).  Pass 2 keeps whole stages as the unit (its kernel is the one closest to the register limit; cutting it at
    // sub-chunks cost 1.4 % at every size).
    const long long in_last = h->n - (long long)(h->it1 - 1) * ITILE1;
    const int live = (int)((in_last + 32 * RI1 - 1) / (32 * RI1));          // warps of the last tile that hold i-points
    double last_cost = live < THREADS / 32 ? std::max(0.6, live / (double)(THREADS / 32)) : 1.0;
    if (const char* e = getenv("CPD_B200_PLAN_LAST_COST")) { const double v = atof(e); if (v > 0.0 && v <= 1.0) last_cost = v; }   // tuning
    WorkList w1;
    if (const char* e = getenv("CPD_B200_PLAN_UNIT"); e && !strcmp(e, "stage")) {      // tuning: items of whole stages, as pass 2
        w1 = build_work(h->it1, (int)(h->mpad / P1_STAGE), h->slots1, last_cost, 0.5);
        for (int4& it : w1.items) { it.y *= P1_STAGE / SUB; it.z *= P1_STAGE / SUB; }
    } else {
        w1 = build_work(h->it1, (int)(h->mpad / SUB), h->slots1, last_cost, 0.5 * (P1_STAGE / SUB));
    }
    const WorkList w2 = build_work(h->it2, (int)(h->npad / P2_STAGE), h->slots2, 1.0, 0.5);
    h->j1 = w1.max_slots; h->g1 = (int)w1.items.size();
    h->j2 = w2.max_slots; h->g2 = (int)w2.items.size();
    TRY(dev_alloc(&h->d_work1, w1.items.size()));
    TRY(dev_alloc(&h->d_work2, w2.items.size()));
    TRY(dev_alloc(&h->d_slots1, w1.tile_slots.size()));
    TRY(dev_alloc(&h->d_slots2, w2.tile_slots.size()));
    // on the handle's (non-blocking) stream, which the consuming kernels run on; the vectors live until the synchronise below
    CU(cudaMemcpyAsync(h->d_work1, w1.items.data(), w1.items.size() * sizeof(int4), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_work2, w2.items.data(), w2.items.size() * sizeof(int4), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_slots1, w1.tile_slots.data(), w1.tile_slots.size() * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_slots2, w2.tile_slots.data(), w2.tile_slots.size() * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    TRY(dev_alloc(&h->d_sbox, (size_t)(h->mpad / P1_STAGE) * 2));
    TRY(dev_alloc(&h->d_tbox, (size_t)(h->npad / P2_STAGE) * 2));
    TRY(dev_alloc(&h->d_omax, (size_t)(h->npad / P2_STAGE)));
    TRY(dev_alloc(&h->d_ssub, (size_t)(h->mpad / SUB) * 2));
    TRY(dev_alloc(&h->d_tsub, (size_t)(h->npad / SUB) * 2));
    TRY(dev_alloc(&h->d_omax_sub, (size_t)(h->npad / SUB)));
    const size_t need1 = (size_t)h->j1 * h->n, need2 = (size_t)h->j2 * h->m * 4;
    if (need1 > h->part1_cap) { TRY(dev_alloc(&h->d_part1, need1)); h->part1_cap = need1; }
    if (need2 > h->part2_cap) { TRY(dev_alloc(&h->d_part2, need2)); h->part2_cap = need2; }
    const size_t ms = (size_t)blocks_for(h->m) * MOM_SRC, mt = (size_t)blocks_for(h->npad) * MOM_TGT;   // MOM_* >= RM_*
    if (ms > h->mom_src_cap) { TRY(dev_alloc(&h->d_mom_src, ms)); h->mom_src_cap = ms; }
    if (mt > h->mom_tgt_cap) { TRY(dev_alloc(&h->d_mom_tgt, mt)); h->mom_tgt_cap = mt; }
    h->prepared = true;
    h->prepare_gen += 1;                 // buffers / work lists changed: a captured EM graph is stale
    return CPD_OK;
}

int allreduce(cpd_ctx* h, double* buf, size_t count) {
    if (!h->comm) return CPD_OK;
    NC(g_nccl.AllReduce(buf, buf, count, NCCL_DOUBLE, NCCL_SUM, h->comm, h->stream));
    return CPD_OK;
}

inline void mark(cpd_ctx* h, int k) {
    if (h->profiling) cudaEventRecord(h->sev[k], h->stream);
}

// pack + pass 1 + finalize 1 + pass 2 + finalize 2; sigma2/w read from the given device scalars
int launch_estep(cpd_ctx* h, const double* d_sigma2, const double* d_w, const double* d_ts) {
    TRY(prepare(h));
    const long long cover = std::max(h->mpad, h->n);
    mark(h, 0);
    pack_kernel<<<blocks_for(cover), THREADS, 0, h->stream>>>(h->d_state, d_sigma2, h->d_yc, d_ts, h->d_xc, h->m, h->mpad,
                                                              h->n, h->d_srcP, h->d_srcJ, h->d_tgtP);
    mark(h, 1);
    const bool cull = h->cull_on && h->cull_active;
    const int nst1 = (int)(h->mpad / P1_STAGE);
    stage_bbox_kernel<<<(unsigned)nst1, THREADS, 0, h->stream>>>(h->d_srcP, (int)h->m, P1_STAGE, h->d_sbox);   // offset seeding (always)
    h->launches += 1;
    const int nsub1 = (int)(h->mpad / SUB), nsub2 = (int)(h->npad / SUB);
    if (cull) {
        stage_bbox_kernel<<<(unsigned)(h->npad / P2_STAGE), THREADS, 0, h->stream>>>(h->d_tgtP, (int)h->n, P2_STAGE, h->d_tbox);
        sub_bbox_kernel<<<(unsigned)((nsub1 + 7) / 8), THREADS, 0, h->stream>>>(h->d_srcP, (int)h->m, nsub1, h->d_ssub);
        sub_bbox_kernel<<<(unsigned)((nsub2 + 7) / 8), THREADS, 0, h->stream>>>(h->d_tgtP, (int)h->n, nsub2, h->d_tsub);
        h->launches += 3;
    }
    const bool wgt = h->wgt_on;
    if (wgt) {
        weight_patch_kernel<<<blocks_for(h->m), THREADS, 0, h->stream>>>(h->d_la, h->m, h->d_srcP, h->d_srcJ);
        h->launches += 1;
    }
#define CPD_PASS1(C, W) pass1_kernel<C, W><<<h->g1, THREADS, PASS1_SMEM, h->stream>>>(h->d_tgtP, (int)h->n, h->d_srcJ, h->d_work1, h->d_part1, h->d_sbox, nst1, (C) ? h->d_ssub : nullptr)
    if (cull) { if (wgt) CPD_PASS1(true, true); else CPD_PASS1(true, false); }
    else { if (wgt) CPD_PASS1(false, true); else CPD_PASS1(false, false); }
#undef CPD_PASS1
    mark(h, 2);
    finalize1_kernel<<<blocks_for(h->npad), THREADS, 0, h->stream>>>(h->d_state, d_sigma2, d_w, h->d_part1, h->d_slots1, (int)h->n,
                                                                     h->d_tgtP, h->d_tgtQ, h->npad, h->d_pt1, h->d_mom_tgt,
                                                                     wgt ? h->d_log2c : nullptr);
    mark(h, 3);
    if (cull) {
        stage_omax_kernel<<<(unsigned)(h->npad / P2_STAGE), THREADS, 0, h->stream>>>(h->d_tgtQ, h->d_omax);
        sub_omax_kernel<<<(unsigned)((nsub2 + 7) / 8), THREADS, 0, h->stream>>>(h->d_tgtQ, nsub2, h->d_omax_sub);
        h->launches += 2;
    }
#define CPD_PASS2(C, W) pass2_kernel<C, W><<<h->g2, THREADS, PASS2_SMEM, h->stream>>>(h->d_srcP, (int)h->m, h->d_tgtQ, h->d_work2, h->d_part2, (C) ? h->d_tbox : nullptr, (C) ? h->d_omax : nullptr, (C) ? h->d_tsub : nullptr, (C) ? h->d_omax_sub : nullptr)
    if (cull) { if (wgt) CPD_PASS2(true, true); else CPD_PASS2(true, false); }
    else { if (wgt) CPD_PASS2(false, true); else CPD_PASS2(false, false); }
#undef CPD_PASS2
    mark(h, 4);
    finalize2_kernel<<<blocks_for(h->m), THREADS, 0, h->stream>>>(h->d_state, d_sigma2, h->d_part2, h->d_slots2, (int)h->m, h->d_yc,
                                                                  d_ts, h->d_p1, h->d_pxc, h->d_mom_src);
    mark(h, 5);
    mark(h, 6);          // E-step-only callers end here; cpd_em_step / cpd_nonrigid_step record event 6 again after their M-step
    KCHECK();
    h->launches += 5;
    return CPD_OK;
}

int read_params(cpd_ctx* h, cpd_params* out) {
    static_assert(sizeof(DevState) <= 48 * sizeof(double), "DevState outgrew the pinned staging buffer");
    CU(cudaMemcpyAsync(h->h_pin, h->d_state, sizeof(DevState), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (reinterpret_cast<const DevState*>(h->h_pin)->err)
        return fail(CPD_ERR_STATE, "a peer rank did not deliver its moments within the P2P exchange timeout");
    const int d = h->dim;
    for (int i = 0; i < 9; ++i) out->lin[i] = 0.0;
    for (int i = 0; i < d; ++i)
        for (int j = 0; j < d; ++j) out->lin[i * d + j] = h->h_pin[3 * i + j];
    for (int i = 0; i < 3; ++i) out->t[i] = (i < d) ? h->h_pin[9 + i] : 0.0;
    out->scale = h->h_pin[12];
    out->sigma2 = h->h_pin[13];
    // a point reaches ~13.3 sigma (2^-127); culling can only pay once that is well inside the cloud
    TRY(ensure_stats(h));
    h->cull_active = h->extent > 0.0 && 13.3 * sqrt(out->sigma2) < 0.25 * h->extent;
    out->q = h->h_pin[14];
    out->n_p = h->h_pin[15];
    return CPD_OK;
}
}  // namespace

// Host-only view of the work list a pass would be launched with (no device needed): lets the CPU tests check that
// every (tile, unit) is covered exactly once and how well the resident CTA slots are filled.
extern "C" int cpd_plan_work(int ntiles, int nunits, int slots, double last_tile_cost, int* items /* 4 ints each, may be NULL */,
                             int capacity, int* n_items, int* max_slots) {
    if (ntiles < 1 || nunits < 1 || slots < 1 || !(last_tile_cost > 0.0 && last_tile_cost <= 1.0) || !n_items || !max_slots)
        return fail(CPD_ERR_ARG, "bad argument");
    const WorkList w = build_work(ntiles, nunits, slots, last_tile_cost, 0.5 * (P1_STAGE / SUB));     // pass 1's units
    *n_items = (int)w.items.size();
    *max_slots = w.max_slots;
    if (items) {
        if (capacity < (int)w.items.size()) return fail(CPD_ERR_ARG, "capacity %d < %d work items", capacity, (int)w.items.size());
        for (size_t i = 0; i < w.items.size(); ++i) {
            items[4 * i] = w.items[i].x; items[4 * i + 1] = w.items[i].y; items[4 * i + 2] = w.items[i].z; items[4 * i + 3] = w.items[i].w;
        }
    }
    return CPD_OK;
}

extern "C" int cpd_create(cpd_ctx** out, int device, int dim, void* stream) {
    if (!out) return fail(CPD_ERR_ARG, "out is NULL");
    if (dim != 2 && dim != 3) return fail(CPD_ERR_ARG, "dim must be 2 or 3, got %d", dim);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(CPD_ERR_CUDA, "no CUDA device: this library has no CPU path");
    }
    if (device < 0 || device >= ndev) return fail(CPD_ERR_ARG, "device %d out of range (%d visible)", device, ndev);
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail(CPD_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
    cpd_ctx* h = new cpd_ctx();
    h->device = device;
    h->dim = dim;
    h->sm_count = prop.multiProcessorCount;
    if (stream) { h->stream = (cudaStream_t)stream; h->own_stream = false; }
    else { CU(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)); h->own_stream = true; }
    CU(cudaFuncSetAttribute(pass1_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, PASS1_SMEM));
    CU(cudaFuncSetAttribute(pass2_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, PASS2_SMEM));
    CU(cudaFuncSetAttribute(pass1_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, PASS1_SMEM));
    CU(cudaFuncSetAttribute(pass2_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, PASS2_SMEM));
    CU(cudaFuncSetAttribute(pass1_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, PASS1_SMEM));
    CU(cudaFuncSetAttribute(pass2_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, PASS2_SMEM));
    CU(cudaFuncSetAttribute(pass1_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, PASS1_SMEM));
    CU(cudaFuncSetAttribute(pass2_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, PASS2_SMEM));
    int occ1 = 0, occ2 = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ1, pass1_kernel<false, false>, THREADS, PASS1_SMEM));
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ2, pass2_kernel<false, false>, THREADS, PASS2_SMEM));
    h->slots1 = h->sm_count * std::max(1, occ1);
    h->slots2 = h->sm_count * std::max(1, occ2);
    TRY(dev_alloc(&h->d_state, 1));
    TRY(dev_alloc(&h->d_mom, (size_t)MOM_PAD));
    CU(cudaMallocHost((void**)&h->h_pin, 64 * sizeof(double)));
    TRY(dev_alloc(&h->d_frame, 16));
    CU(cudaMallocHost((void**)&h->h_stats, 18 * sizeof(double)));
    CU(cudaEventCreateWithFlags(&h->stats_ev, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&h->copy_ev, cudaEventDisableTiming));
    CU(cudaEventCreate(&h->ev0));
    CU(cudaEventCreate(&h->ev1));
    for (int k = 0; k < 7; ++k) CU(cudaEventCreate(&h->sev[k]));
    { const char* e = getenv("CPD_B200_NO_CULL"); h->cull_on = !(e && e[0] == '1'); }
    { const char* e = getenv("CPD_B200_NO_GRAPH"); h->graph_on = !(e && e[0] == '1'); }
    memset(&h->h_state, 0, sizeof(DevState));
    h->h_state.dim = dim;
    h->h_state.scale = 1.0;
    h->h_state.lin[0] = h->h_state.lin[4] = h->h_state.lin[8] = 1.0;
    h->h_state.update_scale = 1;
    *out = h;
    return upload_state(h);          // the device state starts as a copy of the host's (cloud_frame_kernel patches single fields)
}

extern "C" void cpd_destroy(cpd_ctx* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    void* wl[] = {h->d_work1, h->d_work2, h->d_slots1, h->d_slots2, h->d_sbox, h->d_tbox, h->d_omax, h->d_ssub, h->d_tsub, h->d_omax_sub};
    for (void* p : wl) if (p) cudaFree(p);
    void* srt[] = {h->d_perm_src, h->d_perm_tgt, h->d_idx_tmp, h->d_codes, h->d_codes_out, h->d_sort_tmp, h->d_outN, h->d_outM};
    for (void* p : srt) if (p) cudaFree(p);
    void* nrp[] = {h->d_G, h->d_W, h->d_A, h->d_B, h->d_ts2, h->d_nrpart, h->d_ipiv, h->d_info, h->d_work};
    for (void* p : nrp) if (p) cudaFree(p);
    void* lrp[] = {h->d_lr_pts, h->d_lr_Q, h->d_lr_X, h->d_lr_coef, h->d_lr_part, h->d_lr_Bc, h->d_lr_S, h->d_lr_R, h->d_lr_sys, h->d_lr_rhs,
                   h->d_lr_c, h->d_lr_out, h->d_lr_panel, h->d_lr_Lt, h->d_gi_planes, h->d_gi_part, h->d_gi_colmax, h->d_gi_pairs, h->d_wgt, h->d_p1t, h->d_pxt, h->d_la, h->d_log2c};
    for (void* p : lrp) if (p) cudaFree(p);
    if (h->h_work) free(h->h_work);
    if (h->sol_params && g_sol.DestroyParams) g_sol.DestroyParams(h->sol_params);
    if (h->sol && g_sol.Destroy) g_sol.Destroy(h->sol);
    for (int r = 0; r < P2P_MAX; ++r) if (h->peer_ptr[r]) cudaIpcCloseMemHandle(h->peer_ptr[r]);
    if (h->d_box) cudaFree(h->d_box);
    if (h->d_p2p) cudaFree(h->d_p2p);
    void* ptrs[] = {h->d_yc, h->d_ts, h->d_xc, h->d_raw, h->d_srcP, h->d_srcJ, h->d_tgtP, h->d_tgtQ, h->d_part1, h->d_part2, h->d_pt1, h->d_p1,
                    h->d_pxc, h->d_px, h->d_mom_src, h->d_mom_tgt, h->d_mom, h->d_sums, h->d_state, h->d_flush};
    for (void* p : ptrs) if (p) cudaFree(p);
    if (h->h_pin) cudaFreeHost(h->h_pin);
    if (h->h_stats) cudaFreeHost(h->h_stats);
    if (h->d_frame) cudaFree(h->d_frame);
    if (h->stats_ev) cudaEventDestroy(h->stats_ev);
    if (h->copy_ev) cudaEventDestroy(h->copy_ev);
#ifndef CPD_HOST_EMU
    if (h->em_graph) cudaGraphExecDestroy(h->em_graph);
#endif
    if (h->h_state_ring) cudaFreeHost(h->h_state_ring);
    for (int k = 0; k < 8; ++k) if (h->state_ev[k]) cudaEventDestroy(h->state_ev[k]);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    for (int k = 0; k < 7; ++k) if (h->sev[k]) cudaEventDestroy(h->sev[k]);
    for (cudaEvent_t e : h->pool) if (e) cudaEventDestroy(e);
    if (h->own_stream) cudaStreamDestroy(h->stream);
    delete h;
}

extern "C" int cpd_set_source(cpd_ctx* h, const double* source, int64_t m) {
    if (!h || !source) return fail(CPD_ERR_ARG, "null argument");
    if (m < 1 || m > 0x7fffffffLL - 65536) return fail(CPD_ERR_ARG, "source count %lld out of range", (long long)m);
    CU(cudaSetDevice(h->device));
    if (m != h->m || !h->d_yc) {
        h->m = m;
        h->mpad = (m + P1_STAGE - 1) / P1_STAGE * P1_STAGE;
        TRY(dev_alloc(&h->d_yc, (size_t)m * 3));
        TRY(dev_alloc(&h->d_ts, (size_t)m * 3));
        TRY(dev_alloc(&h->d_srcP, (size_t)h->mpad));
        TRY(dev_alloc(&h->d_srcJ, (size_t)h->mpad * 2));
        TRY(dev_alloc(&h->d_p1, (size_t)m));
        TRY(dev_alloc(&h->d_pxc, (size_t)m * 3));
        TRY(dev_alloc(&h->d_px, (size_t)m * 3));
        TRY(dev_alloc(&h->d_perm_src, (size_t)m));
        TRY(dev_alloc(&h->d_outM, (size_t)m * 3));
        h->prepared = false;
        h->nr_ready = false;
    }
    TRY(ingest_cloud(h, source, m, 0, 0, nullptr, h->d_perm_src, h->d_yc));
    h->h_state.m = m;
    h->have_source = true;
    return CPD_OK;
}

extern "C" int cpd_set_target(cpd_ctx* h, const double* target, int64_t n_local, int64_t n_global, const double* frame_origin) {
    if (!h || !target) return fail(CPD_ERR_ARG, "null argument");
    if (n_local < 1 || n_local > 0x7fffffffLL - 65536) return fail(CPD_ERR_ARG, "target count %lld out of range", (long long)n_local);
    if (n_global < n_local) return fail(CPD_ERR_ARG, "n_global (%lld) < n_local (%lld)", (long long)n_global, (long long)n_local);
    if (!frame_origin && n_global != n_local) return fail(CPD_ERR_ARG, "a sharded target needs an explicit frame_origin");
    CU(cudaSetDevice(h->device));
    if (n_local != h->n || !h->d_xc) {
        h->n = n_local;
        h->npad = (n_local + P2_STAGE - 1) / P2_STAGE * P2_STAGE;
        TRY(dev_alloc(&h->d_xc, (size_t)n_local * 3));
        TRY(dev_alloc(&h->d_tgtP, (size_t)n_local));
        TRY(dev_alloc(&h->d_tgtQ, (size_t)h->npad * 3));
        TRY(dev_alloc(&h->d_pt1, (size_t)n_local));
        TRY(dev_alloc(&h->d_perm_tgt, (size_t)n_local));
        TRY(dev_alloc(&h->d_outN, (size_t)n_local));
        h->prepared = false;
    }
    h->n_global = n_global;
    double origin[3] = {0.0, 0.0, 0.0};
    if (frame_origin) for (int a = 0; a < h->dim; ++a) origin[a] = frame_origin[a];
    h->origin_given = frame_origin != nullptr;
    if (h->origin_given) for (int a = 0; a < 3; ++a) h->h_state.cx[a] = origin[a];
    TRY(ingest_cloud(h, target, n_local, 1, n_global, frame_origin ? origin : nullptr, h->d_perm_tgt, h->d_xc));
    h->h_state.n_global = n_global;
    h->have_target = true;
    return CPD_OK;
}

extern "C" int cpd_sigma2_init(cpd_ctx* h, double* sigma2) {
    if (!h || !sigma2) return fail(CPD_ERR_ARG, "null argument");
    if (!h->have_source || !h->have_target) return fail(CPD_ERR_STATE, "source and target must both be set");
    CU(cudaSetDevice(h->device));
    // target sums (summed over the ranks on the device), source sums, ONE read-back: a single host synchronisation
    double sx[4], sy[4];
    const size_t pn = (size_t)blocks_for(h->n) * 4, pm = (size_t)blocks_for(h->m) * 4;
    if (h->sums_cap < 16 + pn + pm) { TRY(dev_alloc(&h->d_sums, 16 + pn + pm)); h->sums_cap = 16 + pn + pm; }
    TRY(cloud_sums_dev(h, h->d_xc, h->n, h->d_sums + 16, h->d_sums));
    if (h->comm) TRY(allreduce(h, h->d_sums, 4));
    TRY(cloud_sums_dev(h, h->d_yc, h->m, h->d_sums + 16 + pn, h->d_sums + 4));
    CU(cudaMemcpyAsync(h->h_pin, h->d_sums, 8 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    TRY(ensure_stats(h));
    for (int k = 0; k < 4; ++k) { sx[k] = h->h_pin[k]; sy[k] = h->h_pin[4 + k]; }
    // move the source sums into the targets' frame: y' = y~ + (cy - cx)
    double dlt[3], d2 = 0.0, dsy = 0.0;
    for (int a = 0; a < 3; ++a) { dlt[a] = h->h_state.cy[a] - h->h_state.cx[a]; d2 += dlt[a] * dlt[a]; dsy += dlt[a] * sy[1 + a]; }
    const double M = (double)h->m, N = (double)h->n_global;
    const double syy = sy[0] + 2.0 * dsy + M * d2;
    double cross = 0.0;
    for (int a = 0; a < 3; ++a) cross += sx[1 + a] * (sy[1 + a] + M * dlt[a]);
    *sigma2 = (M * sx[0] + N * syy - 2.0 * cross) / (M * N * h->dim);
    return CPD_OK;
}

extern "C" int cpd_set_state(cpd_ctx* h, int tf_kind, int update_scale, double w, const cpd_params* init) {
    if (!h || !init) return fail(CPD_ERR_ARG, "null argument");
    if (tf_kind != CPD_TF_RIGID && tf_kind != CPD_TF_AFFINE) return fail(CPD_ERR_ARG, "tf_kind %d not supported by the fused EM loop", tf_kind);
    if (!(w >= 0.0 && w < 1.0)) return fail(CPD_ERR_ARG, "w must be in [0, 1), got %g", w);
    if (!(init->sigma2 > 0.0)) return fail(CPD_ERR_ARG, "sigma2 must be positive, got %g", init->sigma2);
    CU(cudaSetDevice(h->device));
    DevState& s = h->h_state;
    const int d = h->dim;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) s.lin[3 * i + j] = (i < d && j < d) ? init->lin[i * d + j] : (i == j ? 1.0 : 0.0);
    for (int i = 0; i < 3; ++i) s.t[i] = (i < d) ? init->t[i] : 0.0;
    s.scale = (tf_kind == CPD_TF_RIGID) ? init->scale : 1.0;
    s.sigma2 = init->sigma2;
    s.q = init->q;
    s.n_p = 0.0;
    s.w = w;
    s.tf_kind = tf_kind;
    s.update_scale = update_scale ? 1 : 0;
    s.dim = d;
    TRY(ensure_stats(h));
    h->cull_active = h->extent > 0.0 && 13.3 * sqrt(init->sigma2) < 0.25 * h->extent;
    h->have_state = true;
    return upload_state(h);
}

namespace {
// the launches of one fused EM iteration, in stream order (also what a graph capture records)
int em_step_launches(cpd_ctx* h) {
    TRY(launch_estep(h, &h->d_state->sigma2, &h->d_state->w, nullptr));
    const int nbs = (int)blocks_for(h->m), nbt = (int)blocks_for(h->npad);
    if (h->d_p2p) {
        moments_p2p_kernel<<<1, 256, 0, h->stream>>>(h->d_state, h->d_mom_src, nbs, RM_SRC, h->d_mom_tgt, nbt, RM_TGT, h->d_mom,
                                                     h->d_p2p);
        h->launches += 1;
    } else if (h->comm) {
        moments_kernel<0><<<1, 256, 0, h->stream>>>(h->d_state, h->d_mom_src, nbs, RM_SRC, h->d_mom_tgt, nbt, RM_TGT, h->d_mom);
        TRY(allreduce(h, h->d_mom, MOM_PAD));
        mstep_residual_kernel<<<1, 32, 0, h->stream>>>(h->d_state, h->d_mom);
        h->launches += 2;
    } else {
        moments_kernel<1><<<1, 256, 0, h->stream>>>(h->d_state, h->d_mom_src, nbs, RM_SRC, h->d_mom_tgt, nbt, RM_TGT, h->d_mom);
        h->launches += 1;
    }
    mark(h, 6);
    KCHECK();
    return CPD_OK;
}
}  // namespace

// One EM iteration (probreg/cpd.py:111-113).  The launch sequence is fixed per {culling on/off, buffer generation}, so it is
// captured once into a CUDA graph and replayed: one graph launch per iteration.  Not captured: profiling runs (events between
// the kernels) and the ncclAllReduce variant of the multi-rank exchange (CPD_B200_NO_P2P=1); CPD_B200_NO_GRAPH=1 turns it off.
extern "C" int cpd_em_step(cpd_ctx* h, cpd_params* out) {
    if (!h) return fail(CPD_ERR_ARG, "null handle");
    if (!h->have_state) return fail(CPD_ERR_STATE, "cpd_set_state has not been called");
    CU(cudaSetDevice(h->device));
#ifndef CPD_HOST_EMU
    const bool use_graph = h->graph_on && !h->profiling && !(h->comm && !h->d_p2p) && !h->wgt_on;
#else
    const bool use_graph = false;
#endif
    if (!use_graph) {
        TRY(em_step_launches(h));
    }
#ifndef CPD_HOST_EMU
    else {
        TRY(prepare(h));                                    // allocations and uploads happen outside the capture
        const int key = h->prepare_gen * 2 + ((h->cull_on && h->cull_active) ? 1 : 0);
        if (!h->em_graph || h->em_graph_key != key) {
            if (h->em_graph) { cudaGraphExecDestroy(h->em_graph); h->em_graph = nullptr; }
            const int64_t before = h->launches;
            cudaGraph_t g = nullptr;
            CU(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
            const int rc = em_step_launches(h);
            const cudaError_t ce = cudaStreamEndCapture(h->stream, &g);
            h->em_graph_launches = (int)(h->launches - before);
            h->launches = before;
            if (rc != CPD_OK) { if (g) cudaGraphDestroy(g); return rc; }
            if (ce != cudaSuccess) return fail(CPD_ERR_CUDA, "cudaStreamEndCapture failed: %s", cudaGetErrorString(ce));
            const cudaError_t ie = cudaGraphInstantiate(&h->em_graph, g, 0);
            cudaGraphDestroy(g);
            if (ie != cudaSuccess) { h->em_graph = nullptr; return fail(CPD_ERR_CUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ie)); }
            h->em_graph_key = key;
        }
        CU(cudaGraphLaunch(h->em_graph, h->stream));
        h->launches += h->em_graph_launches;                // kernels executed, whatever carried them to the device
    }
#endif
    if (out) return read_params(h, out);
    return CPD_OK;
}

extern "C" int cpd_em_run(cpd_ctx* h, int maxiter, double tol, cpd_params* out, int* iters_run, double* trace) {
    if (!h || !out) return fail(CPD_ERR_ARG, "null argument");
    if (!h->have_state) return fail(CPD_ERR_STATE, "cpd_set_state has not been called");
    double q = h->h_state.q;
    int it = 0;
    cpd_params cur;
    memset(&cur, 0, sizeof(cur));
    for (it = 0; it < maxiter; ++it) {
        TRY(cpd_em_step(h, &cur));
        if (trace) { trace[2 * it] = cur.sigma2; trace[2 * it + 1] = cur.q; }
        if (fabs(cur.q - q) < tol) { ++it; break; }          // cpd.py:117
        q = cur.q;
    }
    if (maxiter <= 0) TRY(read_params(h, &cur));
    *out = cur;
    if (iters_run) *iters_run = it;
    return CPD_OK;
}

extern "C" int cpd_estep(cpd_ctx* h, const double* t_source, double sigma2, double w, double* pt1, double* p1, double* px, double* n_p) {
    if (!h || !t_source) return fail(CPD_ERR_ARG, "null argument");
    if (!(sigma2 > 0.0)) return fail(CPD_ERR_ARG, "sigma2 must be positive, got %g", sigma2);
    if (!(w >= 0.0 && w < 1.0)) return fail(CPD_ERR_ARG, "w must be in [0, 1), got %g", w);
    if (!h->have_source || !h->have_target) return fail(CPD_ERR_STATE, "source and target must both be set");
    CU(cudaSetDevice(h->device));
    if (h->raw_cap < (size_t)h->m * 3) { TRY(dev_alloc(&h->d_raw, (size_t)h->m * 3)); h->raw_cap = (size_t)h->m * 3; }
    TRY(upload_cloud(h, t_source, h->m, h->d_raw));
    gather3_kernel<<<blocks_for(h->m), THREADS, 0, h->stream>>>(h->d_raw, h->d_perm_src, h->m, 0.0, 0.0, 0.0, h->d_ts);
    h->launches += 1;
    TRY(ensure_stats(h));
    h->cull_active = h->extent > 0.0 && 13.3 * sqrt(sigma2) < 0.25 * h->extent;
    h->h_pin[32] = sigma2;
    h->h_pin[33] = w;
    CU(cudaMemcpyAsync(&h->d_state->es_sigma2, h->h_pin + 32, 2 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    TRY(launch_estep(h, &h->d_state->es_sigma2, &h->d_state->es_w, h->d_ts));
    if (h->comm) {
        TRY(allreduce(h, h->d_p1, (size_t)h->m));
        TRY(allreduce(h, h->d_pxc, (size_t)h->m * 3));
    }
    return cpd_last_estep(h, pt1, p1, px, n_p);
}

// BayesianCoherentPointDrift.expectation_step (probreg/bcpd.py:53-72): the CPD E-step with a weight per source,
//   pmat_nm = exp(-|x_n - t_m|^2 / 2 sigma2) (2 pi sigma2)^(-D/2) * exp(-scale^2 / (2 sigma2) * sigma_mm * D) * (1 - w) * alpha_m,
//   den_n = w / N + sum_m pmat_nm,  P = pmat / den,  nu_d = sum_m P (n),  nu = sum_n P (m),  px = P x (m x D),  n_p = sum nu.
// The weights enter the exponent as la_m = -log2(weight_m) (FP64 here, minus their minimum so that la >= 0 and FP32 keeps
// them to ~1e-7 absolute); the constant w / N moves to the same units.  x_hat = px / nu is left to the caller (bcpd.py:70-71).
extern "C" int cpd_bcpd_estep(cpd_ctx* h, const double* t_source, double scale, const double* alpha, const double* sigma_diag,
                              double sigma2, double w, double* nu_d, double* nu, double* px, double* n_p) {
    if (!h || !t_source || !alpha || !sigma_diag) return fail(CPD_ERR_ARG, "null argument");
    if (!(sigma2 > 0.0)) return fail(CPD_ERR_ARG, "sigma2 must be positive, got %g", sigma2);
    if (!(w >= 0.0 && w < 1.0)) return fail(CPD_ERR_ARG, "w must be in [0, 1), got %g", w);
    if (!h->have_source || !h->have_target) return fail(CPD_ERR_STATE, "source and target must both be set");
    CU(cudaSetDevice(h->device));
    const long long m = h->m;
    std::vector<double> la((size_t)m);
    const double kf = scale * scale / (2.0 * sigma2) * (double)h->dim * LOG2E, l1w = -log2(1.0 - w);
    double la_min = INFINITY;
    for (long long i = 0; i < m; ++i) {
        if (!(alpha[i] >= 0.0) || !(sigma_diag[i] >= 0.0)) return fail(CPD_ERR_ARG, "alpha and diag(sigma_mat) must be non-negative");
        la[(size_t)i] = (alpha[i] > 0.0 ? -log2(alpha[i]) : INFINITY) + l1w + kf * sigma_diag[i];
        la_min = std::min(la_min, la[(size_t)i]);
    }
    if (!(la_min < INFINITY)) return fail(CPD_ERR_ARG, "every source has zero weight");
    for (long long i = 0; i < m; ++i) la[(size_t)i] = std::min(la[(size_t)i] - la_min, 1.0e30);      // +inf -> a weight of exactly 0
    if (h->la_cap < (size_t)m) { TRY(dev_alloc(&h->d_la, (size_t)m)); h->la_cap = (size_t)m; }
    if (!h->d_log2c) TRY(dev_alloc(&h->d_log2c, 2));
    const double half_d_log2 = 0.5 * (double)h->dim * log2(2.0 * 3.14159265358979323846 * sigma2);
    h->h_pin[34] = (w > 0.0) ? log2(w / (double)h->n_global) + la_min + half_d_log2 : -INFINITY;   // log2 of the constant, in kernel units
    // Dead columns (bcpd.py:64-65: den == 0 -> eps, so P = 0): a term of the reference's float64 sum is exactly 0 when
    // exp(-d2 / 2 sigma2) underflows (log2 < -1075) or when its product with the factors does.  In kernel units
    // (S' = sum_m 2^-(u + la')) the first is log2 S' < -1075 -- exact for equal weights, the dominant-term approximation
    // otherwise -- and the second log2 S' - la_min - (D/2) log2(2 pi sigma2) < -1075: the smaller of the two shifts decides.
    h->h_pin[35] = std::min(0.0, -la_min - half_d_log2);
    CU(cudaMemcpyAsync(h->d_log2c, h->h_pin + 34, 2 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->d_outM, la.data(), (size_t)m * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    gather_f32_kernel<<<blocks_for(m), THREADS, 0, h->stream>>>(h->d_outM, h->d_perm_src, m, h->d_la);
    KCHECK();
    CU(cudaStreamSynchronize(h->stream));          // `la` (pageable host memory) may go out of scope
    if (h->raw_cap < (size_t)m * 3) { TRY(dev_alloc(&h->d_raw, (size_t)m * 3)); h->raw_cap = (size_t)m * 3; }
    TRY(upload_cloud(h, t_source, m, h->d_raw));
    gather3_kernel<<<blocks_for(m), THREADS, 0, h->stream>>>(h->d_raw, h->d_perm_src, m, 0.0, 0.0, 0.0, h->d_ts);
    h->launches += 2;
    TRY(ensure_stats(h));
    h->cull_active = h->extent > 0.0 && 13.3 * sqrt(sigma2) < 0.25 * h->extent;
    h->h_pin[32] = sigma2;
    h->h_pin[33] = w;
    CU(cudaMemcpyAsync(&h->d_state->es_sigma2, h->h_pin + 32, 2 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    h->wgt_on = true;
    const int r = launch_estep(h, &h->d_state->es_sigma2, &h->d_state->es_w, h->d_ts);
    h->wgt_on = false;
    TRY(r);
    if (h->comm) {
        TRY(allreduce(h, h->d_p1, (size_t)m));
        TRY(allreduce(h, h->d_pxc, (size_t)m * 3));
    }
    return cpd_last_estep(h, nu_d, nu, px, n_p);
}

extern "C" int cpd_last_estep(cpd_ctx* h, double* pt1, double* p1, double* px, double* n_p) {
    if (!h) return fail(CPD_ERR_ARG, "null handle");
    if (!h->prepared) return fail(CPD_ERR_STATE, "no E-step has run on this handle");
    CU(cudaSetDevice(h->device));
    if (pt1) {
        scatter_kernel<<<blocks_for(h->n), THREADS, 0, h->stream>>>(h->d_pt1, h->d_perm_tgt, h->n, 1, h->d_outN);
        CU(cudaMemcpyAsync(pt1, h->d_outN, (size_t)h->n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        h->launches += 1;
    }
    if (p1) {
        scatter_kernel<<<blocks_for(h->m), THREADS, 0, h->stream>>>(h->d_p1, h->d_perm_src, h->m, 1, h->d_outM);
        CU(cudaMemcpyAsync(p1, h->d_outM, (size_t)h->m * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CU(cudaStreamSynchronize(h->stream));      // d_outM is reused for px below
        h->launches += 1;
    }
    if (px) {
        uncentre_px_kernel<<<blocks_for(h->m), THREADS, 0, h->stream>>>(h->d_state, h->d_p1, h->d_pxc, (int)h->m, h->d_px);
        scatter_kernel<<<blocks_for(h->m), THREADS, 0, h->stream>>>(h->d_px, h->d_perm_src, h->m, 3, h->d_outM);
        KCHECK();
        h->launches += 2;
        TRY(download_cloud(h, h->d_outM, h->m, px));
    }
    if (n_p) {
        // n_p = sum(p1) (cpd.py:88): block partials of the (possibly all-reduced) p1
        const unsigned nb = blocks_for(h->m);
        if (h->sums_cap < (size_t)nb * 4 + 4) { TRY(dev_alloc(&h->d_sums, (size_t)nb * 4 + 4)); h->sums_cap = (size_t)nb * 4 + 4; }
        src_moments_api_kernel<<<nb, THREADS, 0, h->stream>>>((int)h->m, h->d_yc, h->d_p1, h->d_pxc, h->d_mom_src);
        reduce_cols_kernel<<<1, MOM_SRC * 32, 0, h->stream>>>(h->d_mom_src, (int)nb, MOM_SRC, h->d_mom);
        KCHECK();
        h->launches += 2;
        CU(cudaMemcpyAsync(h->h_pin + 40, h->d_mom, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    }
    CU(cudaStreamSynchronize(h->stream));
    if (n_p) *n_p = h->h_pin[40];
    return CPD_OK;
}

extern "C" int cpd_mstep(cpd_ctx* h, int tf_kind, int update_scale, const double* pt1, const double* p1, const double* px, double n_p,
                         cpd_params* out) {
    (void)n_p;   // recomputed as sum(p1), which is what the reference passes (cpd.py:88)
    if (!h || !pt1 || !p1 || !px || !out) return fail(CPD_ERR_ARG, "null argument");
    if (tf_kind != CPD_TF_RIGID && tf_kind != CPD_TF_AFFINE) return fail(CPD_ERR_ARG, "tf_kind %d not supported", tf_kind);
    if (!h->have_source || !h->have_target) return fail(CPD_ERR_STATE, "source and target must both be set");
    CU(cudaSetDevice(h->device));
    TRY(prepare(h));
    h->h_state.tf_kind = tf_kind;
    h->h_state.update_scale = update_scale ? 1 : 0;
    // only the two selectors: the rest of the device state may be ahead of the host mirror
    CU(cudaMemcpyAsync(&h->d_state->tf_kind, &h->h_state.tf_kind, 2 * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    // caller's order -> internal (Morton) order
    CU(cudaMemcpyAsync(h->d_outN, pt1, (size_t)h->n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    gather1_kernel<<<blocks_for(h->n), THREADS, 0, h->stream>>>(h->d_outN, h->d_perm_tgt, h->n, h->d_pt1);
    CU(cudaMemcpyAsync(h->d_outM, p1, (size_t)h->m * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    gather1_kernel<<<blocks_for(h->m), THREADS, 0, h->stream>>>(h->d_outM, h->d_perm_src, h->m, h->d_p1);
    if (h->raw_cap < (size_t)h->m * 3) { TRY(dev_alloc(&h->d_raw, (size_t)h->m * 3)); h->raw_cap = (size_t)h->m * 3; }
    TRY(upload_cloud(h, px, h->m, h->d_raw));
    gather3_kernel<<<blocks_for(h->m), THREADS, 0, h->stream>>>(h->d_raw, h->d_perm_src, h->m, 0.0, 0.0, 0.0, h->d_px);
    h->launches += 3;
    const int nbs = (int)blocks_for(h->m), nbt = (int)blocks_for(h->n);
    centre_px_kernel<<<nbs, THREADS, 0, h->stream>>>(h->d_state, h->d_p1, h->d_px, (int)h->m, h->d_pxc);
    src_moments_api_kernel<<<nbs, THREADS, 0, h->stream>>>((int)h->m, h->d_yc, h->d_p1, h->d_pxc, h->d_mom_src);
    tgt_moments_api_kernel<<<nbt, THREADS, 0, h->stream>>>(h->d_pt1, h->d_xc, (int)h->n, h->d_mom_tgt);
    moments_kernel<0><<<1, 256, 0, h->stream>>>(h->d_state, h->d_mom_src, nbs, MOM_SRC, h->d_mom_tgt, nbt, MOM_TGT, h->d_mom);
    KCHECK();
    if (h->comm) TRY(allreduce(h, h->d_mom + MOM_SRC, MOM_TGT));   // p1/px are already global; pt1 is per shard
    mstep_api_kernel<<<1, 32, 0, h->stream>>>(h->d_state, h->d_mom);
    KCHECK();
    h->launches += 5;
    return read_params(h, out);
}

// The remaining entry points live in four .inl files of this same translation unit:
#include "host_nonrigid.inl"     // cpd_nonrigid_* (dense G, low-rank factors, priors)
#include "host_stateless.inl"    // cpd_rbf_kernel, cpd_imq_kernel, cpd_gauss_transform, cpd_squared_kernel_sum
#include "host_multi.inl"        // cpd_comm_*, cpd_p2p_*
#include "host_measure.inl"      // cpd_timer_*, cpd_event_*, cpd_stage_times, cpd_flush_l2, cpd_microbench
