// kao_engine.cu — kernels, device session and the C ABI (include/kao.h) of libkao.so.
//
// Replaces the reference's "emit the LP of README.md:139-185, run lp_solve, read the binaries
// back" step (/root/reference/README.md:135-136) with a GPU candidate search over the same model.
// There is no CPU fallback: every entry point fails with KAO_E_CUDA when no device is usable.
#include "kao_kernels.cuh"
#include "kao_host.hpp"
#include "kao_bound.hpp"
#include "../../include/kao.h"

#include <chrono>
#include <condition_variable>
#include <map>
#include <mutex>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

// The search kernels are instantiated in kao_inst.cu (one object per row width / counter depth /
// evaluation mode); here they are only declared.
#define KAO_DECL_FULL(W, NPH, R, O)                                             \
    extern template __global__ void KAO_ROUND_KERNEL(W, NPH, R, O);            \
    extern template __global__ void KAO_PERSISTENT_KERNEL(W, NPH, R, O, threads_for<W>(), false);
#define KAO_DECL_DELTA(W, NPH, R, O) extern template __global__ void KAO_PERSISTENT_KERNEL(W, NPH, R, O, kThreadsDelta, true);
KAO_FOR_CFGS_NARROW(KAO_DECL_FULL, 1, 5) KAO_FOR_CFGS_NARROW(KAO_DECL_FULL, 2, 5)
KAO_FOR_CFGS_WIDE(KAO_DECL_FULL, 4, 5) KAO_FOR_CFGS_WIDE(KAO_DECL_FULL, 8, 5)
KAO_FOR_CFGS_NARROW(KAO_DECL_DELTA, 1, 5) KAO_FOR_CFGS_NARROW(KAO_DECL_DELTA, 2, 5)
KAO_FOR_CFGS_WIDE(KAO_DECL_DELTA, 4, 5) KAO_FOR_CFGS_WIDE(KAO_DECL_DELTA, 8, 5)
// column-major evaluator (kao_device_t.cuh), every built schedule
#define KAO_DECL_T(S, POP, T)                                                  \
    extern template __global__ void KAO_PERSISTENT_KERNEL_T(1, 0, S, POP, T);  \
    extern template __global__ void KAO_PERSISTENT_KERNEL_T(1, 32, S, POP, T); \
    extern template __global__ void KAO_PERSISTENT_KERNEL_T(2, 0, S, POP, T);  \
    extern template __global__ void KAO_PERSISTENT_KERNEL_T(2, 32, S, POP, T);
KAO_FOR_SCHEDULES(KAO_DECL_T)


// Winner of a round becomes the base: re-materialise its patches from (seed, round, index), write
// the patched rows to the base in HBM, then rebuild the displaced list D.  One block.
template <int W>
__global__ void __launch_bounds__(1024, 1)
apply_winner_kernel(Params d, uint64_t seed, uint32_t round, uint32_t round_size,
                    const unsigned long long *key, int regen_only)
{
    __shared__ uint32_t s_prow[kMaxOps * W];
    __shared__ int s_scan[72];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (warp == 0 && !regen_only) {
        const unsigned long long k = *key;
        if (k != kKeyNone) {
            Gen<W> gen;
            uint32_t no_rows[kMaxOps][W];
            gen.bitsT = d.bitsT; gen.leader = d.leader; gen.cs = d.consts; gen.d = &d;
            gen.prow = s_prow; gen.lane = lane;
            gen.D = d.D; gen.DL = d.DL; gen.nD = d.nD[0]; gen.nL = d.nD[1];
            PatchSet ps;
            gen.run(seed, round, (uint32_t)(k & kIdxMask), round_size, ps, no_rows);
            __syncwarp();
            if (lane == 0) {
#pragma unroll
                for (int i = 0; i < kMaxOps; ++i) {
                    if (i < ps.n) {
                        for (int t = 0; t < W; ++t) d.bitsT[(size_t)t * d.Ppad + ps.p[i]] = s_prow[i * W + t];
                        d.leader[ps.p[i]] = (uint8_t)ps.ld[i];
                    }
                }
            }
        }
    }
    __threadfence_block();
    __syncthreads();
    rebuild_lists<1024>(d.bitsT, d.leader, d.homeT, d.P, d.Ppad, d.D, d.DL, d.nD, s_scan);
}

__global__ void fill_u64_kernel(unsigned long long *p, unsigned long long v, size_t n)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}

// Explicit population: one warp per candidate, rows read straight from HBM (coalesced 128-bit
// loads), same evaluator.  cand_bits [n][W][Ppad], cand_leader [n][Ppad].
template <int W, int NPH>
__global__ void __launch_bounds__(256)
eval_batch_kernel(Params d, const uint32_t *cand_bits, const uint8_t *cand_leader, int n,
                  long long *viol_out, long long *obj_out)
{
    const int lane = threadIdx.x & 31;
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (w >= n) return;
    PatchSet ps;
    ps.n = 0;
#pragma unroll
    for (int i = 0; i < kMaxOps; ++i) { ps.p[i] = -1; ps.ld[i] = 0xFF; }
    int viol, obj;
    eval_candidate<EvalCfg<W, NPH, 0, kObjEntries>, false>(d, cand_bits + (size_t)w * W * d.Ppad,
                                                               cand_leader + (size_t)w * d.Ppad, d.swT, d.consts, ps,
                                                               nullptr, lane, viol, obj);
    if (lane == 0) { viol_out[w] = viol; obj_out[w] = obj; }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(int code, const std::string &msg) { g_err = msg; return code; }
static bool schedule_exists(int sync, int pop, int threads);
#define CUDA_TRY(expr)                                                                       \
    do {                                                                                     \
        cudaError_t e_ = (expr);                                                             \
        if (e_ != cudaSuccess)                                                               \
            return fail(KAO_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));     \
    } while (0)

// Nothing may cross the C ABI but a return code (include/kao.h: "never throw"): every extern "C" body
// runs inside this guard.
template <class F> static int guarded(F &&f) noexcept
{
    try {
        return f();
    } catch (const std::bad_alloc &) {
        return fail(KAO_E_ARG, "out of host memory (argument too large?)");
    } catch (const std::exception &e) {
        return fail(KAO_E_CUDA, std::string("internal error: ") + e.what());
    } catch (...) {
        return fail(KAO_E_CUDA, "internal error");
    }
}

// Device buffers are recycled across handles: kao_solve creates and destroys a session per call,
// and cudaMalloc / cudaFree (which synchronises the device) would dominate short solves.
namespace {
struct DevPool {
    std::mutex mu;
    std::multimap<std::pair<int, size_t>, void *> free_;
    size_t held = 0;
    cudaError_t get(int dev, void **p, size_t n)
    {
        n = (n + 255) & ~size_t(255);
        {
            std::lock_guard<std::mutex> g(mu);
            auto it = free_.find({dev, n});
            if (it != free_.end()) { *p = it->second; free_.erase(it); held -= n; return cudaSuccess; }
        }
        return cudaMalloc(p, n);
    }
    void put(int dev, void *p, size_t n)
    {
        n = (n + 255) & ~size_t(255);
        std::lock_guard<std::mutex> g(mu);
        if (held + n > (size_t(1) << 30)) { cudaFree(p); return; }
        free_.insert({{dev, n}, p});
        held += n;
    }
};
DevPool g_pool;

// a temporary device buffer that is freed on every path out of the scope that owns it
template <class T> struct DevTmp {
    T *p = nullptr;
    cudaError_t alloc(size_t count) { return cudaMalloc(&p, count * sizeof(T)); }
    ~DevTmp() { if (p) cudaFree(p); }
};

// every wait inside a kernel (grid barrier, peer GPUs) gives up after this much wall time and the call
// returns KAO_E_CUDA instead of hanging the GPU; KAO_WAIT_TIMEOUT_MS overrides the 20 s default
unsigned long long wait_budget_ns()
{
    static const unsigned long long ns = [] {
        double ms = 20000.0;
        if (const char *e = std::getenv("KAO_WAIT_TIMEOUT_MS")) { const double v = std::atof(e); if (v >= 1.0) ms = v; }
        return (unsigned long long)(ms * 1e6);
    }();
    return ns;
}
}  // namespace

constexpr size_t kBarBytes = 32;   // d_bar: [0] grid barrier, [1] release, [2] abort, [3] rounds run, [4..7] early-stop carry (2 x u64)

struct kao_handle {
    std::vector<std::pair<void *, size_t>> owned;   // device buffers to hand back to the pool
    HostModel hm;               // layout, tables, host copy of problem data
    int device = 0;
    int sms = 0;
    Params prm{};
    SmemPlan plan{};
    int threads = 0, grid = 0;
    // column-major full evaluator (kao_set_evaluator): layout supported, selected (the default wherever it applies)
    bool trans_ok = false;
    int evaluator = KAO_EVAL_ROW_MAJOR;
    // schedule of the column-major evaluator (kao_set_schedule): barrier form, popcount compression per
    // stream, threads per CTA.  Same results whatever the schedule.
    int sch_sync = KAO_SCHEDULE_DEFAULT_SYNC, sch_pop = KAO_SCHEDULE_DEFAULT_POP, sch_threads = KAO_SCHEDULE_DEFAULT_THREADS;
    // device buffers
    uint32_t *d_bits = nullptr; uint8_t *d_leader = nullptr; uint32_t *d_sw = nullptr;
    uint32_t *d_dense = nullptr; uint32_t *d_planes = nullptr; uint8_t *d_zslot = nullptr; uint32_t *d_home = nullptr; uint16_t *d_D = nullptr; uint16_t *d_DL = nullptr; int *d_nD = nullptr;
    Consts *d_consts = nullptr; unsigned long long *d_key = nullptr; unsigned long long *d_keys = nullptr;
    size_t keys_cap = 0;
    long long *d_vo = nullptr;
    unsigned int *d_bar = nullptr;          // kBarBytes, see above
    // cross-GPU exchange (kao_p2p_*, kao_solve with n_gpus > 1)
    Mailbox *d_mail = nullptr;              // own mailbox (plain cudaMalloc: exported through CUDA IPC / used by peers directly)
    Mailbox *peer_mail[kMaxPeers] = {};
    Mailbox **d_mailptrs = nullptr;         // device copy of peer_mail for the kernel
    bool peer_opened[kMaxPeers] = {};       // mapped with cudaIpcOpenMemHandle (to be closed)
    bool mail_pooled = false;               // d_mail came from the buffer pool (kao_solve's gang), not from cudaMalloc
    int p2p_rank = 0, p2p_world = 1;
    uint64_t p2p_calls = 0;
    uint32_t patience = 0, last_rounds = 0;
    unsigned long long *d_lkeys = nullptr; size_t lkeys_cap = 0;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    uint64_t launches = 0;
};


template <class T> static cudaError_t dalloc(kao_handle *h, T **p, size_t bytes)
{
    void *v = nullptr;
    cudaError_t e = g_pool.get(h->device, &v, bytes);
    if (e == cudaSuccess) { *p = static_cast<T *>(v); h->owned.emplace_back(v, bytes); }
    return e;
}

struct RoundArgs {
    uint64_t seed; uint32_t round, round_size, lo, hi; unsigned long long *d_key, *d_all; cudaStream_t st;
};
struct PersistArgs {
    uint64_t seed; uint32_t first_round, rounds, round_size; unsigned long long *d_keys; unsigned int *d_bar; cudaStream_t st;
    P2P pp;
    unsigned long long *all_keys;
};

template <class Cfg> static cudaError_t set_smem_attr(kao_handle *h, const void *kern, bool *done)
{
    if (!done[h->device & 63]) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) return e;
        done[h->device & 63] = true;
    }
    return cudaSuccess;
}

struct LaunchRound {
    template <class Cfg> cudaError_t run(kao_handle *h, const RoundArgs &a) const
    {
        constexpr int T = threads_for<Cfg::W>();
        auto kern = search_round_kernel<Cfg, T>;
        static bool done[64] = {};
        cudaError_t e = set_smem_attr<Cfg>(h, reinterpret_cast<const void *>(kern), done);
        if (e != cudaSuccess) return e;
        const uint32_t n = a.hi - a.lo, warps = T / 32;
        uint32_t grid = (n + warps - 1) / warps;
        if (grid > (uint32_t)h->grid) grid = (uint32_t)h->grid;
        if (grid == 0) return cudaSuccess;
        kern<<<grid, T, h->plan.total, a.st>>>(h->prm, h->plan, a.seed, a.round, a.round_size, a.lo, a.hi, a.d_key, a.d_all);
        ++h->launches;
        return cudaGetLastError();
    }
};
template <bool kDelta> struct LaunchPersistent {
    template <class Cfg> cudaError_t run(kao_handle *h, const PersistArgs &a) const
    {
        {
            constexpr int T = kDelta ? kThreadsDelta : cfg_threads<Cfg>();
            auto kern = search_persistent_kernel<Cfg, T, kDelta>;
            static bool done[64] = {};
            cudaError_t e = set_smem_attr<Cfg>(h, reinterpret_cast<const void *>(kern), done);
            if (e != cudaSuccess) return e;
            Params prm = h->prm;
            // the column-major plan depends on the warps per CTA of the schedule (per-warp scratch)
            SmemPlan plan = Cfg::kTrans ? make_plan_t(Cfg::W, h->hm.Ppad, T, h->hm.P, h->hm.RF)
                            : (kDelta && Cfg::W > 2) ? make_plan_delta_wide(Cfg::W, h->hm.Ppad, T, h->hm.P, h->hm.RF) : h->plan;
            if (plan.total > 227u * 1024u) return cudaErrorInvalidConfiguration;
            uint64_t seed = a.seed; uint32_t fr = a.first_round, rounds = a.rounds, rs = a.round_size;
            unsigned long long *keys = a.d_keys, *all = a.all_keys; unsigned int *bar = a.d_bar;
            P2P pp = a.pp;
            void *args[] = {&prm, &plan, &seed, &fr, &rounds, &rs, &keys, &bar, &pp, &all};
            ++h->launches;
            // cooperative launch: all CTAs are guaranteed co-resident, which the grid barrier needs
            return cudaLaunchCooperativeKernel(reinterpret_cast<const void *>(kern), dim3(h->grid), dim3(T), args,
                                               plan.total, a.st);
        }
    }
};

template <int W, int NPH, int kRack, class F, class A>
static cudaError_t dispatch_obj(kao_handle *h, const F &f, const A &a)
{
    if constexpr (W <= 2) {
        if (h->prm.nplanes == 3) return f.template run<EvalCfg<W, NPH, kRack, 3>>(h, a);
    }
    return f.template run<EvalCfg<W, NPH, kRack, kObjEntries>>(h, a);
}
// Rack form of the evaluator (kao_device.cuh, row_rack_terms): "at most one replica per rack" with
// the field width fixed at compile time (8 / 16 slots / whole words), or general bounds.
template <int W, int NPH, class F, class A>
static cudaError_t dispatch_w(kao_handle *h, const F &f, const A &a)
{
    if (!h->hm.hi1) return dispatch_obj<W, NPH, 0>(h, f, a);
    if (h->hm.log2S == 3) return dispatch_obj<W, NPH, 3>(h, f, a);
    if (h->hm.log2S == 4) return dispatch_obj<W, NPH, 4>(h, f, a);
    return dispatch_obj<W, NPH, 5>(h, f, a);
}
template <class F, class A> static cudaError_t dispatch(kao_handle *h, const F &f, const A &a)
{
    switch (h->hm.W) {                                    // one counter depth: per-lane column counts up to 255
    case 1: return dispatch_w<1, 5>(h, f, a);
    case 2: return dispatch_w<2, 5>(h, f, a);
    case 4: return dispatch_w<4, 5>(h, f, a);
    default: return dispatch_w<8, 5>(h, f, a);
    }
}
// all rounds of a search in one cooperative launch, with the evaluator the session selected
static cudaError_t launch_persistent(kao_handle *h, const PersistArgs &pa, bool delta)
{
    if (delta) return dispatch(h, LaunchPersistent<true>{}, pa);
    if (h->evaluator == KAO_EVAL_COLUMN_MAJOR) {
        const bool nw32 = h->hm.Ppad == 1024;                   // 32 partition words per slot: compile-time offsets
#define KAO_RUN_T(S, POP, T)                                                                                   \
    if (h->sch_sync == S && h->sch_pop == POP && h->sch_threads == T) {                                        \
        if (h->hm.W == 1) return nw32 ? LaunchPersistent<false>{}.template run<EvalCfgT<1, 32, S, POP, T>>(h, pa) \
                                      : LaunchPersistent<false>{}.template run<EvalCfgT<1, 0, S, POP, T>>(h, pa); \
        return nw32 ? LaunchPersistent<false>{}.template run<EvalCfgT<2, 32, S, POP, T>>(h, pa)                 \
                    : LaunchPersistent<false>{}.template run<EvalCfgT<2, 0, S, POP, T>>(h, pa);                 \
    }
        KAO_FOR_SCHEDULES(KAO_RUN_T)
#undef KAO_RUN_T
        return cudaErrorInvalidValue;                           // kao_set_schedule only accepts built schedules
    }
    return dispatch(h, LaunchPersistent<false>{}, pa);
}
static cudaError_t launch_round(kao_handle *h, uint64_t seed, uint32_t round, uint32_t round_size,
                                uint32_t lo, uint32_t hi, unsigned long long *d_key,
                                unsigned long long *d_all, cudaStream_t st)
{
    return dispatch(h, LaunchRound{}, RoundArgs{seed, round, round_size, lo, hi, d_key, d_all, st});
}
static cudaError_t launch_apply(kao_handle *h, uint64_t seed, uint32_t round, uint32_t round_size,
                                const unsigned long long *d_key, int regen_only, cudaStream_t st)
{
    switch (h->hm.W) {
    case 1: apply_winner_kernel<1><<<1, 1024, 0, st>>>(h->prm, seed, round, round_size, d_key, regen_only); break;
    case 2: apply_winner_kernel<2><<<1, 1024, 0, st>>>(h->prm, seed, round, round_size, d_key, regen_only); break;
    case 4: apply_winner_kernel<4><<<1, 1024, 0, st>>>(h->prm, seed, round, round_size, d_key, regen_only); break;
    default: apply_winner_kernel<8><<<1, 1024, 0, st>>>(h->prm, seed, round, round_size, d_key, regen_only); break;
    }
    ++h->launches;
    return cudaGetLastError();
}

static int upload_base(kao_handle *h, const std::vector<uint32_t> &bitsT, const std::vector<uint8_t> &leader)
{
    CUDA_TRY(cudaMemcpy(h->d_bits, bitsT.data(), bitsT.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(h->d_leader, leader.data(), leader.size(), cudaMemcpyHostToDevice));
    CUDA_TRY(launch_apply(h, 0, 0, 2, h->d_key, /*regen_only=*/1, 0));
    CUDA_TRY(cudaDeviceSynchronize());
    return KAO_OK;
}

static int destroy_impl(kao_handle *h)
{
    if (!h) return KAO_OK;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();                   // nothing of this session may still be running on a recycled buffer
    for (auto &b : h->owned) g_pool.put(h->device, b.first, b.second);
    for (int r = 0; r < kMaxPeers; ++r)
        if (h->peer_opened[r]) cudaIpcCloseMemHandle(h->peer_mail[r]);
    if (h->d_mail && !h->mail_pooled) cudaFree(h->d_mail);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    delete h;
    return KAO_OK;
}

static int reset_impl(kao_handle *h)
{
    if (!h) return fail(KAO_E_ARG, "null handle");
    CUDA_TRY(cudaSetDevice(h->device));
    std::vector<uint32_t> bitsT; std::vector<uint8_t> leader;
    initial_base(h->hm, bitsT, leader);
    return upload_base(h, bitsT, leader);
}

static int create_impl(const kao_problem *pb, int32_t device, kao_handle *h)
{
    std::string why;
    if (!build_host_model(*pb, h->hm, why)) return fail(KAO_E_ARG, why);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
        return fail(KAO_E_CUDA, "no CUDA device: libkao has no CPU path");
    if (device < 0 || device >= ndev) return fail(KAO_E_ARG, "bad device ordinal");
    h->device = device;
    CUDA_TRY(cudaSetDevice(device));
    {   // cudaGetDeviceProperties costs tens of milliseconds per call; one attribute, cached per device
        static int sm_count[64] = {};
        if (!sm_count[device & 63])
            CUDA_TRY(cudaDeviceGetAttribute(&sm_count[device & 63], cudaDevAttrMultiProcessorCount, device));
        h->sms = sm_count[device & 63];
    }
    const HostModel &m = h->hm;
    const int W = m.W, Ppad = m.Ppad;
    h->threads = W <= 2 ? kThreads : kThreadsWide;
    h->plan = make_plan(W, Ppad, h->threads / 32, m.nplanes > 0 ? m.nplanes * W : 4, m.P, m.RF, m.nplanes > 0);
    if (h->plan.total > 227u * 1024u && m.nplanes > 0) {
        // mask planes + one-hot plane do not fit next to the base: score with packed entries / the dense table
        h->hm.nplanes = 0;
        h->plan = make_plan(W, Ppad, h->threads / 32, 4, m.P, m.RF, false);
    }
    if (h->plan.total > 227u * 1024u)
        return fail(KAO_E_ARG, "problem too large for the shared-memory resident search kernel");
    // column-major evaluator: 8-slot rack fields, C7 = "at most one replica per rack", an objective that fits
    // eight term planes (kao_host.hpp); its two transposed planes (2 * W words per partition) and the term planes
    // take the place of the objective table.  It is the default full evaluator wherever it applies.
    h->trans_ok = W <= 2 && m.hi1 && m.log2S == 3 && m.z_ok &&
                  column_major_fits(W, Ppad, 1024, m.P, m.RF);     // sized for the largest schedule (1024 threads)
    if (h->trans_ok) h->evaluator = KAO_EVAL_COLUMN_MAJOR;
    if (const char *env = std::getenv("KAO_EVALUATOR"))       // "row" forces the row-major evaluator (measurements)
        if (std::strcmp(env, "row") == 0) h->evaluator = KAO_EVAL_ROW_MAJOR;
    if (const char *env = std::getenv("KAO_SCHEDULE")) {      // "sync,pop(hex),threads": measurements only, ignored if not built
        int a = 0, c = 0; unsigned b = 0;
        if (std::sscanf(env, "%d,%x,%d", &a, &b, &c) == 3 && schedule_exists(a, (int)b, c)) {
            h->sch_sync = a; h->sch_pop = (int)b; h->sch_threads = c;
        }
    }
    h->grid = h->sms;
    CUDA_TRY(dalloc(h, &h->d_bits, (size_t)W * Ppad * 4));
    CUDA_TRY(dalloc(h, &h->d_leader, (size_t)Ppad));
    CUDA_TRY(dalloc(h, &h->d_sw, (size_t)4 * Ppad * 4));
    CUDA_TRY(dalloc(h, &h->d_home, (size_t)Ppad * 4));
    CUDA_TRY(dalloc(h, &h->d_D, (size_t)Ppad * 2));
    CUDA_TRY(dalloc(h, &h->d_DL, (size_t)Ppad * 2));
    CUDA_TRY(dalloc(h, &h->d_nD, 16));
    CUDA_TRY(dalloc(h, &h->d_consts, sizeof(Consts)));
    CUDA_TRY(dalloc(h, &h->d_key, 16));
    CUDA_TRY(dalloc(h, &h->d_bar, kBarBytes));
    CUDA_TRY(cudaMemset(h->d_nD, 0, 16));
    { const unsigned long long none[2] = {kKeyNone, kKeyNone}; CUDA_TRY(cudaMemcpy(h->d_key, none, 16, cudaMemcpyHostToDevice)); }
    if (m.dense) {
        CUDA_TRY(dalloc(h, &h->d_dense, m.dense_w.size() * 4));
        CUDA_TRY(cudaMemcpy(h->d_dense, m.dense_w.data(), m.dense_w.size() * 4, cudaMemcpyHostToDevice));
    }
    CUDA_TRY(cudaMemcpy(h->d_sw, m.swT.data(), m.swT.size() * 4, cudaMemcpyHostToDevice));
    if (m.nplanes > 0) {
        CUDA_TRY(dalloc(h, &h->d_planes, m.planesT.size() * 4));
        CUDA_TRY(cudaMemcpy(h->d_planes, m.planesT.data(), m.planesT.size() * 4, cudaMemcpyHostToDevice));
    }
    CUDA_TRY(cudaMemcpy(h->d_home, m.homeT.data(), m.homeT.size() * 4, cudaMemcpyHostToDevice));
    if (m.z_ok) {
        CUDA_TRY(dalloc(h, &h->d_zslot, m.zslot.size()));
        CUDA_TRY(cudaMemcpy(h->d_zslot, m.zslot.data(), m.zslot.size(), cudaMemcpyHostToDevice));
    }
    Consts cs;
    fill_consts(m, cs);
    CUDA_TRY(cudaMemcpy(h->d_consts, &cs, sizeof cs, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaEventCreate(&h->ev0));
    CUDA_TRY(cudaEventCreate(&h->ev1));
    Params &p = h->prm;
    p.P = m.P; p.Ppad = Ppad; p.B = m.B; p.R = m.R; p.RF = m.RF; p.NS = m.NS; p.log2S = m.log2S;
    set_rf_masks(p);
    p.ppr_lo = m.ppr_lo; p.ppr_hi = m.ppr_hi; p.dense = m.dense ? 1 : 0;
    p.key_obj_bits = m.key_obj_bits;
    p.nentries = m.nentries; p.nplanes = m.nplanes; p.plane_on_leader = m.plane_on_leader;
    for (int c = 0; c < 6; ++c) p.plane_value[c] = m.plane_value[c];
    p.planesT = h->d_planes;
    p.nz = m.z_ok ? m.nz : 0; p.z_on_leader = m.z_on_leader; p.zslot = h->d_zslot;
    for (int j = 0; j < 8; ++j) p.z_value[j] = m.z_value[j];
    p.bitsT = h->d_bits; p.leader = h->d_leader; p.swT = h->d_sw; p.dense_w = h->d_dense;
    p.homeT = h->d_home; p.D = h->d_D; p.DL = h->d_DL; p.nD = h->d_nD; p.consts = h->d_consts;
    return reset_impl(h);
}

static int create_handle(const kao_problem *pb, int32_t device, kao_handle **out)
{
    if (!pb || !out) return fail(KAO_E_ARG, "null argument");
    *out = nullptr;
    kao_handle *h = new kao_handle();
    const int rc = create_impl(pb, device, h);
    if (rc != KAO_OK) {
        const std::string keep = g_err;
        destroy_impl(h);
        g_err = keep;
        return rc;
    }
    *out = h;
    return KAO_OK;
}

static int set_base_impl(kao_handle *h, const int32_t *replicas)
{
    if (!h || !replicas) return fail(KAO_E_ARG, "null argument");
    CUDA_TRY(cudaSetDevice(h->device));
    std::vector<uint32_t> bitsT; std::vector<uint8_t> leader;
    encode_replicas(h->hm, replicas, bitsT, leader);
    return upload_base(h, bitsT, leader);
}

static int eval_on_device(kao_handle *h, const uint32_t *d_bits, const uint8_t *d_leader, int n,
                          long long *d_viol, long long *d_obj)
{
    const int blocks = (n * 32 + 255) / 256;
    switch (h->hm.W) {
    case 1: eval_batch_kernel<1, 5><<<blocks, 256>>>(h->prm, d_bits, d_leader, n, d_viol, d_obj); break;
    case 2: eval_batch_kernel<2, 5><<<blocks, 256>>>(h->prm, d_bits, d_leader, n, d_viol, d_obj); break;
    case 4: eval_batch_kernel<4, 5><<<blocks, 256>>>(h->prm, d_bits, d_leader, n, d_viol, d_obj); break;
    default: eval_batch_kernel<8, 5><<<blocks, 256>>>(h->prm, d_bits, d_leader, n, d_viol, d_obj); break;
    }
    ++h->launches;
    CUDA_TRY(cudaGetLastError());
    return KAO_OK;
}

static int get_base_impl(kao_handle *h, int32_t *replicas, int64_t *violation, int64_t *objective, int32_t *moves)
{
    if (!h) return fail(KAO_E_ARG, "null handle");
    CUDA_TRY(cudaSetDevice(h->device));
    const HostModel &m = h->hm;
    std::vector<uint32_t> bitsT((size_t)m.W * m.Ppad);
    std::vector<uint8_t> leader((size_t)m.Ppad);
    CUDA_TRY(cudaMemcpy(bitsT.data(), h->d_bits, bitsT.size() * 4, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(leader.data(), h->d_leader, leader.size(), cudaMemcpyDeviceToHost));
    std::vector<int32_t> reps((size_t)m.P * m.RF);
    decode_replicas(m, bitsT, leader, reps.data());
    if (replicas) std::memcpy(replicas, reps.data(), reps.size() * 4);
    if (moves) *moves = count_moves(m, reps.data());
    if (violation || objective) {
        if (!h->d_vo) CUDA_TRY(dalloc(h, &h->d_vo, 16));
        int rc = eval_on_device(h, h->d_bits, h->d_leader, 1, h->d_vo, h->d_vo + 1);
        long long vo[2] = {0, 0};
        if (rc == KAO_OK && cudaMemcpy(vo, h->d_vo, 16, cudaMemcpyDeviceToHost) != cudaSuccess) rc = KAO_E_CUDA;
        if (rc != KAO_OK) return rc;
        if (violation) *violation = vo[0];
        if (objective) *objective = vo[1];
    }
    return KAO_OK;
}

static bool check_round_args(uint32_t round_size) { return round_size >= 2 && round_size <= KAO_MAX_ROUND_SIZE; }
// delta evaluation keeps the base and the per-round tables in shared memory (rows wider than 64 slots: without the objective table)
static bool delta_fits(const kao_handle *h)
{
    if (h->hm.W <= 2) return true;                              // the session's own plan (validated at kao_create)
    return make_plan_delta_wide(h->hm.W, h->hm.Ppad, kThreadsDelta, h->hm.P, h->hm.RF).total <= 227u * 1024u;
}

static int reserve_keys(kao_handle *h, uint32_t rounds)
{
    if (h->keys_cap < rounds || !h->d_keys) {
        h->d_keys = nullptr;                   // the old buffer stays owned by the handle until destroy
        CUDA_TRY(dalloc(h, &h->d_keys, (size_t)(rounds > 0 ? rounds : 1) * 8));
        h->keys_cap = rounds;
    }
    if (rounds) {
        fill_u64_kernel<<<64, 256>>>(h->d_keys, kKeyNone, (size_t)rounds);
        CUDA_TRY(cudaGetLastError());
    }
    return KAO_OK;
}

static P2P solo_p2p(kao_handle *h, uint32_t idx_lo, uint32_t idx_hi)
{
    P2P pp{};
    pp.rank = 0; pp.world = 1; pp.idx_lo = idx_lo; pp.idx_hi = idx_hi;
    pp.abort = reinterpret_cast<int *>(h->d_bar + 2);
    pp.patience = h->patience; pp.rounds_run = h->d_bar + 3;
    pp.best_in = kKeyNone; pp.stall_in = 0;
    pp.carry = reinterpret_cast<unsigned long long *>(h->d_bar + 4);
    pp.timeout_ns = wait_budget_ns();
    return pp;
}

static int search_impl(kao_handle *h, uint64_t seed, uint32_t first_round, uint32_t rounds,
                       uint32_t round_size, uint64_t *round_keys, double *device_ms, bool delta)
{
    if (!h) return fail(KAO_E_ARG, "null handle");
    if (delta && !delta_fits(h)) return fail(KAO_E_ARG, "delta evaluation: the base and its per-round tables do not fit in shared memory");
    if (!check_round_args(round_size)) return fail(KAO_E_ARG, "round_size must be 2..2^24");
    if (rounds > KAO_MAX_ROUNDS) return fail(KAO_E_ARG, "rounds must not exceed KAO_MAX_ROUNDS (2^20) per call");
    CUDA_TRY(cudaSetDevice(h->device));
    h->last_rounds = 0;
    int rc = reserve_keys(h, rounds);
    if (rc != KAO_OK) return rc;
    CUDA_TRY(cudaMemsetAsync(h->d_bar, 0, kBarBytes, 0));
    CUDA_TRY(cudaEventRecord(h->ev0, 0));
    if (rounds) {
        // all rounds in one cooperative launch; the HBM base is kept current by CTA 0, the displaced
        // lists in HBM are rebuilt once at the end for the per-round entry points
        CUDA_TRY(launch_persistent(h, PersistArgs{seed, first_round, rounds, round_size, h->d_keys, h->d_bar, 0,
                                                  solo_p2p(h, 0, round_size), nullptr}, delta));
        CUDA_TRY(launch_apply(h, seed, first_round, round_size, h->d_keys, /*regen_only=*/1, 0));
    }
    CUDA_TRY(cudaEventRecord(h->ev1, 0));
    CUDA_TRY(cudaEventSynchronize(h->ev1));
    if (device_ms) {
        float ms = 0;
        CUDA_TRY(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
        *device_ms = ms;
    }
    if (rounds) {
        unsigned int st[4] = {0, 0, 0, 0};
        CUDA_TRY(cudaMemcpy(st, h->d_bar, 16, cudaMemcpyDeviceToHost));
        if (st[2]) return fail(KAO_E_CUDA, "search kernel timed out at a grid barrier");
        h->last_rounds = st[3];
    }
    if (round_keys && rounds)
        CUDA_TRY(cudaMemcpy(round_keys, h->d_keys, (size_t)rounds * 8, cudaMemcpyDeviceToHost));
    return KAO_OK;
}

static bool schedule_exists(int sync, int pop, int threads)
{
#define KAO_HAS_T(S, POP, T) if (sync == S && pop == POP && threads == T) return true;
    KAO_FOR_SCHEDULES(KAO_HAS_T)
#undef KAO_HAS_T
    return false;
}

static int candidate_keys_impl(kao_handle *h, uint64_t seed, uint32_t round, uint32_t round_size,
                               uint32_t idx_begin, uint32_t count, uint64_t *keys, bool delta)
{
    if (!h || !keys) return fail(KAO_E_ARG, "null argument");
    if (!check_round_args(round_size) || idx_begin > round_size || count > round_size - idx_begin)
        return fail(KAO_E_ARG, "bad index range");
    if (delta && !delta_fits(h)) return fail(KAO_E_ARG, "delta evaluation: the base and its per-round tables do not fit in shared memory");
    if (count == 0) return KAO_OK;
    CUDA_TRY(cudaSetDevice(h->device));
    DevTmp<unsigned long long> all;
    CUDA_TRY(all.alloc(count));
    { const unsigned long long none = kKeyNone; CUDA_TRY(cudaMemcpy(h->d_key, &none, 8, cudaMemcpyHostToDevice)); }
    if (delta || h->evaluator == KAO_EVAL_COLUMN_MAJOR) {
        // these evaluators live in the persistent kernel only: one round, key dump, base untouched
        CUDA_TRY(cudaMemset(h->d_bar, 0, kBarBytes));
        P2P pp = solo_p2p(h, idx_begin, idx_begin + count);
        pp.patience = 0;
        CUDA_TRY(launch_persistent(h, PersistArgs{seed, round, 1, round_size, h->d_key, h->d_bar, 0, pp, all.p}, delta));
    } else {
        CUDA_TRY(launch_round(h, seed, round, round_size, idx_begin, idx_begin + count, h->d_key, all.p, 0));
    }
    CUDA_TRY(cudaMemcpy(keys, all.p, (size_t)count * 8, cudaMemcpyDeviceToHost));
    return KAO_OK;
}

// ---- cross-GPU sharded search: the 8-byte minimum of every round travels through peer-writable mailboxes
static int ensure_mailbox(kao_handle *h)
{
    if (h->d_mail) return KAO_OK;
    CUDA_TRY(cudaSetDevice(h->device));
    CUDA_TRY(cudaMalloc(&h->d_mail, sizeof(Mailbox)));
    CUDA_TRY(cudaMemset(h->d_mail, 0xFF, sizeof(Mailbox)));        // kMailEmpty everywhere
    CUDA_TRY(cudaDeviceSynchronize());
    return KAO_OK;
}
static int publish_mailboxes(kao_handle *h, int rank, int world)
{
    if (!h->d_mailptrs) CUDA_TRY(dalloc(h, &h->d_mailptrs, sizeof(Mailbox *) * kMaxPeers));
    CUDA_TRY(cudaMemcpy(h->d_mailptrs, h->peer_mail, sizeof(Mailbox *) * kMaxPeers, cudaMemcpyHostToDevice));
    h->p2p_rank = rank; h->p2p_world = world; h->p2p_calls = 0;
    return KAO_OK;
}

static int p2p_export_impl(kao_handle *h, uint8_t *handle_out)
{
    if (!h || !handle_out) return fail(KAO_E_ARG, "null argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == KAO_IPC_HANDLE_BYTES, "ipc handle size");
    const int rc = ensure_mailbox(h);
    if (rc != KAO_OK) return rc;
    cudaIpcMemHandle_t ipc;
    CUDA_TRY(cudaIpcGetMemHandle(&ipc, h->d_mail));
    std::memcpy(handle_out, &ipc, sizeof ipc);
    return KAO_OK;
}

static int p2p_connect_impl(kao_handle *h, int32_t rank, int32_t world, const uint8_t *handles)
{
    if (!h || !handles) return fail(KAO_E_ARG, "null argument");
    if (world < 1 || world > kMaxPeers || rank < 0 || rank >= world) return fail(KAO_E_ARG, "bad rank / world");
    if (!h->d_mail) return fail(KAO_E_STATE, "call kao_p2p_export first");
    CUDA_TRY(cudaSetDevice(h->device));
    for (int r = 0; r < world; ++r) {
        if (r == rank) { h->peer_mail[r] = h->d_mail; continue; }
        cudaIpcMemHandle_t ipc;
        std::memcpy(&ipc, handles + (size_t)r * KAO_IPC_HANDLE_BYTES, sizeof ipc);
        void *p = nullptr;
        CUDA_TRY(cudaIpcOpenMemHandle(&p, ipc, cudaIpcMemLazyEnablePeerAccess));
        h->peer_mail[r] = static_cast<Mailbox *>(p);
        h->peer_opened[r] = true;
    }
    return publish_mailboxes(h, rank, world);
}

static int sharded_impl(kao_handle *h, uint64_t seed, uint32_t first_round, uint32_t rounds,
                        uint32_t round_size, uint64_t *round_keys, double *device_ms, bool delta)
{
    if (!h) return fail(KAO_E_ARG, "null handle");
    if (delta && !delta_fits(h)) return fail(KAO_E_ARG, "delta evaluation: the base and its per-round tables do not fit in shared memory");
    if (!check_round_args(round_size)) return fail(KAO_E_ARG, "round_size must be 2..2^24");
    if (rounds > KAO_MAX_ROUNDS) return fail(KAO_E_ARG, "rounds must not exceed KAO_MAX_ROUNDS (2^20) per call");
    if (h->p2p_world < 2 || !h->peer_mail[h->p2p_world - 1]) return fail(KAO_E_STATE, "kao_p2p_connect first");
    CUDA_TRY(cudaSetDevice(h->device));
    h->last_rounds = 0;
    int rc = reserve_keys(h, rounds);
    if (rc != KAO_OK) return rc;
    if (h->lkeys_cap < kMailRounds) {
        CUDA_TRY(dalloc(h, &h->d_lkeys, (size_t)kMailRounds * 8));
        h->lkeys_cap = kMailRounds;
    }
    const int world = h->p2p_world, rank = h->p2p_rank;
    // contiguous slice of every round for this rank (same split on every rank)
    const uint32_t base = round_size / world, extra = round_size % world;
    const uint32_t lo = rank * base + ((uint32_t)rank < extra ? rank : extra);
    const uint32_t hi = lo + base + ((uint32_t)rank < extra ? 1 : 0);
    unsigned long long best = kKeyNone;                             // early-stop state, carried from launch to launch
    uint32_t stall = 0;
    CUDA_TRY(cudaEventRecord(h->ev0, 0));
    for (uint32_t done = 0; done < rounds; done += kMailRounds) {
        const uint32_t n = rounds - done < kMailRounds ? rounds - done : kMailRounds;
        const int bank = (int)(h->p2p_calls & 1);
        ++h->p2p_calls;
        // the OTHER bank is reset now: no peer can reach the next launch before this rank has taken
        // part in every round of this one (docs/MODEL.md §7), so the reset cannot race with a writer
        CUDA_TRY(cudaMemsetAsync(&h->d_mail->slot[bank ^ 1][0][0], 0xFF, sizeof(h->d_mail->slot[0]), 0));
        fill_u64_kernel<<<32, 256>>>(h->d_lkeys, kKeyNone, (size_t)n);
        CUDA_TRY(cudaMemsetAsync(h->d_bar, 0, kBarBytes, 0));
        h->launches += 1;
        P2P pp = solo_p2p(h, lo, hi);
        pp.rank = rank; pp.world = world; pp.bank = bank;
        pp.mail = h->d_mailptrs;
        pp.lkeys = h->d_lkeys; pp.release = h->d_bar + 1;
        pp.best_in = best; pp.stall_in = stall;
        const PersistArgs pa{seed, first_round + done, n, round_size, h->d_keys + done, h->d_bar, 0, pp, nullptr};
        CUDA_TRY(launch_persistent(h, pa, delta));
        unsigned int st[8] = {};
        CUDA_TRY(cudaMemcpy(st, h->d_bar, kBarBytes, cudaMemcpyDeviceToHost));
        if (st[2]) return fail(KAO_E_CUDA, "sharded search timed out waiting for a peer GPU");
        h->last_rounds = done + st[3];
        std::memcpy(&best, st + 4, 8);
        { unsigned long long s64; std::memcpy(&s64, st + 6, 8); stall = (uint32_t)s64; }
        if (st[3] < n) break;                                   // early stop (every rank stops at the same round)
    }
    if (rounds) CUDA_TRY(launch_apply(h, seed, first_round, round_size, h->d_keys, /*regen_only=*/1, 0));
    CUDA_TRY(cudaEventRecord(h->ev1, 0));
    CUDA_TRY(cudaEventSynchronize(h->ev1));
    if (device_ms) {
        float ms = 0;
        CUDA_TRY(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
        *device_ms = ms;
    }
    if (round_keys && rounds)
        CUDA_TRY(cudaMemcpy(round_keys, h->d_keys, (size_t)rounds * 8, cudaMemcpyDeviceToHost));
    return KAO_OK;
}

static int profile_rounds_impl(kao_handle *h, uint64_t seed, uint32_t first_round, uint32_t rounds,
                               uint32_t round_size, double *search_ms, double *apply_ms)
{
    if (!h || !rounds || rounds > 4096) return fail(KAO_E_ARG, "bad argument (1..4096 rounds)");
    if (!check_round_args(round_size)) return fail(KAO_E_ARG, "bad round_size");
    CUDA_TRY(cudaSetDevice(h->device));
    struct Events {
        std::vector<cudaEvent_t> ev;
        ~Events() { for (auto &e : ev) if (e) cudaEventDestroy(e); }
    } evs;
    evs.ev.assign(3 * (size_t)rounds, nullptr);
    for (auto &e : evs.ev) CUDA_TRY(cudaEventCreate(&e));
    DevTmp<unsigned long long> k;
    CUDA_TRY(k.alloc(rounds));
    fill_u64_kernel<<<32, 256>>>(k.p, kKeyNone, (size_t)rounds);
    for (uint32_t t = 0; t < rounds; ++t) {
        CUDA_TRY(cudaEventRecord(evs.ev[3 * t], 0));
        CUDA_TRY(launch_round(h, seed, first_round + t, round_size, 0, round_size, k.p + t, nullptr, 0));
        CUDA_TRY(cudaEventRecord(evs.ev[3 * t + 1], 0));
        CUDA_TRY(launch_apply(h, seed, first_round + t, round_size, k.p + t, 0, 0));
        CUDA_TRY(cudaEventRecord(evs.ev[3 * t + 2], 0));
    }
    CUDA_TRY(cudaDeviceSynchronize());
    double s_ms = 0, a_ms = 0;
    for (uint32_t t = 0; t < rounds; ++t) {
        float a = 0, b = 0;
        CUDA_TRY(cudaEventElapsedTime(&a, evs.ev[3 * t], evs.ev[3 * t + 1]));
        CUDA_TRY(cudaEventElapsedTime(&b, evs.ev[3 * t + 1], evs.ev[3 * t + 2]));
        s_ms += a; a_ms += b;
    }
    if (search_ms) *search_ms = s_ms;
    if (apply_ms) *apply_ms = a_ms;
    return KAO_OK;
}

static int eval_impl(const kao_problem *pb, int32_t device, const int32_t *replicas, int32_t n,
                     int64_t *violation, int64_t *objective)
{
    if (!pb || !replicas || n < 0 || !violation || !objective) return fail(KAO_E_ARG, "bad argument");
    kao_handle *h = nullptr;
    int rc = create_handle(pb, device, &h);
    if (rc != KAO_OK) return rc;
    struct Closer { kao_handle *h; ~Closer() { const std::string keep = g_err; destroy_impl(h); g_err = keep; } } closer{h};
    const HostModel &m = h->hm;
    const size_t nb = (size_t)m.W * m.Ppad, nl = (size_t)m.Ppad;
    if (n == 0) return KAO_OK;
    std::vector<uint32_t> bits(nb * n), one;
    std::vector<uint8_t> lead(nl * n), onel;
    for (int i = 0; i < n; ++i) {
        encode_replicas(m, replicas + (size_t)i * m.P * m.RF, one, onel);
        std::memcpy(bits.data() + nb * i, one.data(), nb * 4);
        std::memcpy(lead.data() + nl * i, onel.data(), nl);
    }
    DevTmp<uint32_t> d_b; DevTmp<uint8_t> d_l; DevTmp<long long> d_v;
    CUDA_TRY(d_b.alloc(bits.size()));
    CUDA_TRY(d_l.alloc(lead.size()));
    CUDA_TRY(d_v.alloc((size_t)n * 2));
    CUDA_TRY(cudaMemcpy(d_b.p, bits.data(), bits.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_l.p, lead.data(), lead.size(), cudaMemcpyHostToDevice));
    rc = eval_on_device(h, d_b.p, d_l.p, n, d_v.p, d_v.p + n);
    if (rc != KAO_OK) return rc;
    static_assert(sizeof(long long) == sizeof(int64_t), "abi");
    CUDA_TRY(cudaMemcpy(violation, d_v.p, (size_t)n * 8, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(objective, d_v.p + n, (size_t)n * 8, cudaMemcpyDeviceToHost));
    return KAO_OK;
}

// ---- kao_solve: one GPU, or the rounds sharded over several GPUs of this process
static int pick_devices(const kao_options *opt, std::vector<int> &devs)
{
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
        return fail(KAO_E_CUDA, "no CUDA device: libkao has no CPU path");
    devs.clear();
    if (opt->device_mask) {
        for (int i = 0; i < 32; ++i)
            if (opt->device_mask >> i & 1u) devs.push_back(i);
        if (opt->n_gpus > 1 && opt->n_gpus != (int)devs.size()) return fail(KAO_E_ARG, "n_gpus does not match device_mask");
    } else {
        const int n = opt->n_gpus > 1 ? opt->n_gpus : 1;
        for (int i = 0; i < n; ++i) devs.push_back(opt->device + i);
    }
    if (devs.empty() || (int)devs.size() > KAO_MAX_GPUS) return fail(KAO_E_ARG, "1..KAO_MAX_GPUS devices");
    for (int d : devs)
        if (d < 0 || d >= ndev) return fail(KAO_E_ARG, "bad device ordinal (n_gpus / device_mask exceed the visible devices)");
    return KAO_OK;
}

// ---- several GPUs of this process: one host thread per GPU does everything for its device (create, connect,
// search, destroy), so that the per-call set-up cost does not grow with the number of GPUs
namespace {
struct Rendezvous {                                   // a reusable barrier that also spreads "somebody failed"
    std::mutex mu;
    std::condition_variable cv;
    int n, waiting = 0, generation = 0;
    bool failed = false;
    explicit Rendezvous(int parties) : n(parties) {}
    bool arrive(bool ok)                              // -> false once any party has arrived with ok == false
    {
        std::unique_lock<std::mutex> lk(mu);
        failed |= !ok;
        const int gen = generation;
        if (++waiting == n) { waiting = 0; ++generation; cv.notify_all(); }
        else cv.wait(lk, [&] { return gen != generation; });
        return !failed;
    }
};
std::mutex g_peer_mu;
bool g_peer_enabled[64][64] = {};
}  // namespace

static int enable_peers(int dev, const std::vector<int> &devs)
{
    CUDA_TRY(cudaSetDevice(dev));
    for (int other : devs) {
        if (other == dev) continue;
        {
            std::lock_guard<std::mutex> g(g_peer_mu);
            if (g_peer_enabled[dev & 63][other & 63]) continue;
        }
        int can = 0;
        CUDA_TRY(cudaDeviceCanAccessPeer(&can, dev, other));
        if (!can) return fail(KAO_E_CUDA, "the selected GPUs cannot access each other's memory (no peer access)");
        const cudaError_t e = cudaDeviceEnablePeerAccess(other, 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
        else if (e != cudaSuccess) return fail(KAO_E_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
        std::lock_guard<std::mutex> g(g_peer_mu);
        g_peer_enabled[dev & 63][other & 63] = true;
    }
    return KAO_OK;
}

struct GangResult {                                   // what rank 0 reports per restart
    int64_t viol = 0, obj = 0;
    int32_t moves = 0;
    uint32_t rounds = 0;
    double dev_ms = 0;
};

static int solve_gang(const kao_problem *pb, const kao_options *opt, kao_result *res, const std::vector<int> &devs,
                      uint32_t restarts, bool delta, std::vector<uint64_t> &keys, std::vector<int32_t> &reps,
                      uint32_t &rounds_run, double &dev_ms_total, HostModel &hm_out)
{
    const int world = (int)devs.size();
    std::vector<kao_handle *> hs(world, nullptr);
    std::vector<int> rcs(world, KAO_OK);
    std::vector<std::string> errs(world);
    std::vector<double> ms(world, 0.0);
    Rendezvous meet(world);
    bool have = false;
    static const bool trace = std::getenv("KAO_TRACE") != nullptr;       // stderr: where a multi-GPU solve spends its host time
    const auto t_start = std::chrono::steady_clock::now();
    auto worker = [&](int i) {
        int phase = 0;
        auto step = [&](int rc) {                     // record the first failure of this rank, then meet the others
            if (rc != KAO_OK && rcs[i] == KAO_OK) { rcs[i] = rc; errs[i] = g_err; }
            const auto t_a = std::chrono::steady_clock::now();
            const bool all_ok = meet.arrive(rc == KAO_OK);
            if (trace) {
                const auto t_b = std::chrono::steady_clock::now();
                std::fprintf(stderr, "[kao trace] gpu %d phase %d: reached at %.3f ms, waited %.3f ms for the others\n", devs[i], phase,
                             std::chrono::duration<double, std::milli>(t_a - t_start).count(),
                             std::chrono::duration<double, std::milli>(t_b - t_a).count());
            }
            ++phase;
            return all_ok;
        };
        kao_handle *h = nullptr;
        bool ok = step(guarded([&] { return create_handle(pb, devs[i], &h); }));
        hs[i] = h;
        if (ok) ok = step(guarded([&] {
            int rc = enable_peers(devs[i], devs);
            if (rc != KAO_OK) return rc;
            CUDA_TRY(dalloc(h, &h->d_mail, sizeof(Mailbox)));          // recycled: no cudaMalloc / cudaFree per solve
            h->mail_pooled = true;
            CUDA_TRY(cudaMemsetAsync(h->d_mail, 0xFF, sizeof(Mailbox), 0));   // kMailEmpty everywhere, before any peer can write
            CUDA_TRY(cudaStreamSynchronize(0));
            h->patience = opt->flags >> 16;                         // KAO_FLAG_PATIENCE(n)
            if (opt->flags & KAO_FLAG_ROW_MAJOR) h->evaluator = KAO_EVAL_ROW_MAJOR;
            return KAO_OK;
        }));
        if (ok) ok = step(guarded([&] {
            for (int j = 0; j < world; ++j) h->peer_mail[j] = hs[j]->d_mail;    // unified addressing: a peer's pointer is valid here
            return publish_mailboxes(h, i, world);
        }));
        for (uint32_t r = 0; ok && r < restarts; ++r) {
            const uint64_t seed = opt->seed + 0x9E3779B97F4A7C15ull * r;
            ok = step(guarded([&] {
                int rc = r ? reset_impl(h) : KAO_OK;
                if (rc == KAO_OK) rc = sharded_impl(h, seed, 0, opt->rounds, opt->round_size, i == 0 ? keys.data() : nullptr, &ms[i], delta);
                return rc;
            }));
            if (ok && i == 0) {                       // all ranks hold the same base: rank 0 reports it
                GangResult g;
                int rc = guarded([&] { return get_base_impl(h, reps.data(), &g.viol, &g.obj, &g.moves); });
                if (rc == KAO_OK) {
                    for (int j = 0; j < world; ++j) g.dev_ms = ms[j] > g.dev_ms ? ms[j] : g.dev_ms;
                    dev_ms_total += g.dev_ms;
                    rounds_run += h->last_rounds;
                    if (!have || g.viol < res->violation || (g.viol == res->violation && g.obj > res->objective)) {
                        std::memcpy(res->replicas, reps.data(), reps.size() * 4);
                        res->violation = g.viol; res->objective = g.obj; res->moves = g.moves;
                        res->key = h->last_rounds ? keys[h->last_rounds - 1] : kKeyNone;
                        have = true;
                    }
                } else { rcs[0] = rc; errs[0] = g_err; }
            }
            if (ok) ok = meet.arrive(i != 0 || rcs[0] == KAO_OK);   // nobody resets the base while rank 0 reads it
        }
        if (i == 0 && h) hm_out = h->hm;
        if (h) { const std::string keep = g_err; destroy_impl(h); g_err = keep; }
        if (trace)
            std::fprintf(stderr, "[kao trace] gpu %d destroyed at %.3f ms\n", devs[i],
                         std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count());
    };
    std::vector<std::thread> th;
    for (int i = 1; i < world; ++i) th.emplace_back(worker, i);
    worker(0);
    for (auto &t : th) t.join();
    for (int i = 0; i < world; ++i)
        if (rcs[i] != KAO_OK) return fail(rcs[i], "GPU " + std::to_string(devs[i]) + ": " + errs[i]);
    return KAO_OK;
}

// KAO_FLAG_SPREAD_RESTARTS: the restarts of one kao_solve side by side on the GPUs of the call — restart r runs on
// GPU r mod N as an ordinary single-GPU search (no exchange between the GPUs at all), one host thread per GPU; the
// best final assignment wins, ties go to the lowest restart index: exactly what one GPU returns for the same call.
static int solve_spread(const kao_problem *pb, const kao_options *opt, kao_result *res, const std::vector<int> &devs,
                        uint32_t restarts, bool delta, uint32_t &rounds_run, double &dev_ms_total, HostModel &hm_out)
{
    const int world = (int)devs.size();
    struct Best {
        bool have = false;
        int64_t viol = 0, obj = 0;
        int32_t moves = 0;
        uint32_t restart = 0, rounds = 0;
        uint64_t key = kKeyNone;
        double dev_ms = 0;
        std::vector<int32_t> reps;
        HostModel hm;
    };
    std::vector<Best> best(world);
    std::vector<int> rcs(world, KAO_OK);
    std::vector<std::string> errs(world);
    auto worker = [&](int i) {
        Best &b = best[i];
        rcs[i] = guarded([&]() -> int {
            kao_handle *h = nullptr;
            int rc = create_handle(pb, devs[i], &h);
            if (rc != KAO_OK) return rc;
            struct Closer { kao_handle *h; ~Closer() { const std::string keep = g_err; destroy_impl(h); g_err = keep; } } closer{h};
            h->patience = opt->flags >> 16;
            if (opt->flags & KAO_FLAG_ROW_MAJOR) h->evaluator = KAO_EVAL_ROW_MAJOR;
            b.hm = h->hm;
            std::vector<uint64_t> keys(opt->rounds ? opt->rounds : 1, kKeyNone);
            std::vector<int32_t> reps((size_t)pb->P * pb->RF);
            bool first = true;
            for (uint32_t r = (uint32_t)i; r < restarts; r += (uint32_t)world) {
                double dev_ms = 0;
                if (!first && (rc = reset_impl(h)) != KAO_OK) return rc;
                first = false;
                rc = search_impl(h, opt->seed + 0x9E3779B97F4A7C15ull * r, 0, opt->rounds, opt->round_size, keys.data(), &dev_ms, delta);
                if (rc != KAO_OK) return rc;
                int64_t viol = 0, obj = 0;
                int32_t moves = 0;
                rc = get_base_impl(h, reps.data(), &viol, &obj, &moves);
                if (rc != KAO_OK) return rc;
                b.dev_ms += dev_ms;
                b.rounds += h->last_rounds;
                if (!b.have || viol < b.viol || (viol == b.viol && obj > b.obj)) {
                    b.have = true; b.viol = viol; b.obj = obj; b.moves = moves; b.restart = r;
                    b.key = h->last_rounds ? keys[h->last_rounds - 1] : kKeyNone;
                    b.reps = reps;
                }
            }
            return KAO_OK;
        });
        if (rcs[i] != KAO_OK) errs[i] = g_err;
    };
    std::vector<std::thread> th;
    for (int i = 1; i < world; ++i) th.emplace_back(worker, i);
    worker(0);
    for (auto &t : th) t.join();
    for (int i = 0; i < world; ++i)
        if (rcs[i] != KAO_OK) return fail(rcs[i], "GPU " + std::to_string(devs[i]) + ": " + errs[i]);
    const Best *win = nullptr;
    for (const Best &b : best) {
        if (!b.have) continue;                        // more GPUs than restarts
        rounds_run += b.rounds;
        dev_ms_total = b.dev_ms > dev_ms_total ? b.dev_ms : dev_ms_total;
        if (!win || b.viol < win->viol || (b.viol == win->viol && (b.obj > win->obj || (b.obj == win->obj && b.restart < win->restart)))) win = &b;
    }
    if (!win) return fail(KAO_E_STATE, "no restart ran");
    std::memcpy(res->replicas, win->reps.data(), win->reps.size() * 4);
    res->violation = win->viol; res->objective = win->obj; res->moves = win->moves; res->key = win->key;
    hm_out = best[0].hm;
    return KAO_OK;
}

static int solve_impl(const kao_problem *pb, const kao_options *opt, kao_result *res)
{
    if (!pb || !opt || !res || !res->replicas) return fail(KAO_E_ARG, "null argument");
    if (opt->rounds > KAO_MAX_ROUNDS) return fail(KAO_E_ARG, "rounds must not exceed KAO_MAX_ROUNDS (2^20)");
    if (!check_round_args(opt->round_size)) return fail(KAO_E_ARG, "round_size must be 2..2^24");
    const auto t0 = std::chrono::steady_clock::now();
    std::vector<int> devs;
    int rc = pick_devices(opt, devs);
    if (rc != KAO_OK) return rc;
    const int world = (int)devs.size();
    // independent restarts (flags & 0xFF, 0 and 1 both mean a single search): each restarts from the
    // initial base with its own seed; the best final assignment wins (violation, then objective)
    const uint32_t restarts = (opt->flags & 0xFFu) ? (opt->flags & 0xFFu) : 1u;
    const bool delta = (opt->flags & KAO_FLAG_DELTA) != 0;
    uint32_t rounds_run = 0;
    std::vector<uint64_t> keys(opt->rounds ? opt->rounds : 1, kKeyNone);
    std::vector<int32_t> reps((size_t)pb->P * pb->RF);
    double dev_ms_total = 0;
    HostModel hm;
    static const bool trace = std::getenv("KAO_TRACE") != nullptr;
    auto stamp = [&](const char *what) {
        if (trace)
            std::fprintf(stderr, "[kao trace] kao_solve: %s at %.3f ms\n", what,
                         std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
    };
    if (world == 1) {
        kao_handle *h0 = nullptr;
        rc = create_handle(pb, devs[0], &h0);
        if (rc != KAO_OK) return rc;
        stamp("session created (model built, tables uploaded, initial base)");
        struct Closer { kao_handle *h; ~Closer() { const std::string keep = g_err; destroy_impl(h); g_err = keep; } } closer{h0};
        h0->patience = opt->flags >> 16;                         // KAO_FLAG_PATIENCE(n)
        // the column-major evaluator is the default where the layout allows it; the flag selects the other full evaluator (same keys)
        if (opt->flags & KAO_FLAG_ROW_MAJOR) h0->evaluator = KAO_EVAL_ROW_MAJOR;
        bool have = false;
        for (uint32_t r = 0; r < restarts; ++r) {
            double dev_ms = 0;
            if (r && (rc = reset_impl(h0)) != KAO_OK) return rc;
            rc = search_impl(h0, opt->seed + 0x9E3779B97F4A7C15ull * r, 0, opt->rounds, opt->round_size, keys.data(), &dev_ms, delta);
            if (rc != KAO_OK) return rc;
            stamp("search done");
            int64_t viol = 0, obj = 0;
            int32_t moves = 0;
            rc = get_base_impl(h0, reps.data(), &viol, &obj, &moves);
            if (rc != KAO_OK) return rc;
            stamp("result downloaded and evaluated");
            dev_ms_total += dev_ms;
            rounds_run += h0->last_rounds;
            if (!have || viol < res->violation || (viol == res->violation && obj > res->objective)) {
                std::memcpy(res->replicas, reps.data(), reps.size() * 4);
                res->violation = viol; res->objective = obj; res->moves = moves;
                res->key = h0->last_rounds ? keys[h0->last_rounds - 1] : kKeyNone;
                have = true;
            }
        }
        hm = h0->hm;
    } else if (opt->flags & KAO_FLAG_SPREAD_RESTARTS) {
        rc = solve_spread(pb, opt, res, devs, restarts, delta, rounds_run, dev_ms_total, hm);
        if (rc != KAO_OK) return rc;
    } else {
        rc = solve_gang(pb, opt, res, devs, restarts, delta, keys, reps, rounds_run, dev_ms_total, hm);
        if (rc != KAO_OK) return rc;
    }
    stamp("session destroyed");
    res->feasible = res->violation == 0;
    res->n_candidates = (uint64_t)rounds_run * opt->round_size;
    res->rounds_run = rounds_run;
    res->restarts = restarts;
    res->device_ms = dev_ms_total;
    res->objective_bound = objective_upper_bound(hm, *pb);
    if ((opt->flags & KAO_FLAG_BOUND) && res->feasible)
        res->objective_bound = objective_flow_bound(hm, *pb, res->replicas, res->objective_bound);
    res->optimal = res->feasible && res->objective == res->objective_bound;
    res->key_obj_bits = hm.key_obj_bits;
    res->n_gpus = world;
    res->reserved = 0;
    stamp("bound computed");
    res->total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (!res->feasible) { g_err = "no candidate satisfying C1..C7 was found"; return KAO_INFEASIBLE; }
    return KAO_OK;
}

// ------------------------------------------------------------------------------------------
// the C ABI (include/kao.h): thin, guarded entry points
// ------------------------------------------------------------------------------------------
extern "C" int kao_version(void) { return KAO_VERSION; }
extern "C" const char *kao_last_error(void) { return g_err.c_str(); }
extern "C" int kao_key_obj_bits(const kao_problem *pb)
{
    return guarded([&] {
        if (!pb) return fail(KAO_E_ARG, "null argument");
        HostModel m;
        std::string why;
        if (!build_host_model(*pb, m, why)) return fail(KAO_E_ARG, why);
        return m.key_obj_bits;
    });
}
extern "C" int kao_objective_bound(const kao_problem *pb, const int32_t *replicas, int64_t *bound)
{
    return guarded([&] {
        if (!pb || !bound) return fail(KAO_E_ARG, "null argument");
        HostModel m;
        std::string why;
        if (!build_host_model(*pb, m, why)) return fail(KAO_E_ARG, why);
        *bound = objective_upper_bound(m, *pb);
        if (replicas) *bound = objective_flow_bound(m, *pb, replicas, *bound);
        return KAO_OK;
    });
}
extern "C" int kao_create(const kao_problem *pb, int32_t device, kao_handle **out) { return guarded([&] { return create_handle(pb, device, out); }); }
extern "C" int kao_destroy(kao_handle *h) { return guarded([&] { return destroy_impl(h); }); }
extern "C" int kao_reset(kao_handle *h) { return guarded([&] { return reset_impl(h); }); }
extern "C" int kao_set_base(kao_handle *h, const int32_t *replicas) { return guarded([&] { return set_base_impl(h, replicas); }); }
extern "C" int kao_get_base(kao_handle *h, int32_t *replicas, int64_t *violation, int64_t *objective, int32_t *moves)
{
    return guarded([&] { return get_base_impl(h, replicas, violation, objective, moves); });
}
extern "C" int kao_round_launch(kao_handle *h, uint64_t seed, uint32_t round, uint32_t round_size,
                                uint32_t idx_lo, uint32_t idx_hi, uint64_t *d_key, void *stream)
{
    return guarded([&] {
        if (!h || !d_key) return fail(KAO_E_ARG, "null argument");
        if (!check_round_args(round_size) || idx_lo > idx_hi || idx_hi > round_size)
            return fail(KAO_E_ARG, "bad round_size / index range");
        CUDA_TRY(cudaSetDevice(h->device));
        CUDA_TRY(launch_round(h, seed, round, round_size, idx_lo, idx_hi,
                              reinterpret_cast<unsigned long long *>(d_key), nullptr, (cudaStream_t)stream));
        return KAO_OK;
    });
}
extern "C" int kao_round_apply(kao_handle *h, uint64_t seed, uint32_t round, uint32_t round_size,
                               const uint64_t *d_key, void *stream)
{
    return guarded([&] {
        if (!h || !d_key) return fail(KAO_E_ARG, "null argument");
        if (!check_round_args(round_size)) return fail(KAO_E_ARG, "bad round_size");
        CUDA_TRY(cudaSetDevice(h->device));
        CUDA_TRY(launch_apply(h, seed, round, round_size, reinterpret_cast<const unsigned long long *>(d_key), 0,
                              (cudaStream_t)stream));
        return KAO_OK;
    });
}
extern "C" int kao_set_evaluator(kao_handle *h, int32_t evaluator)
{
    return guarded([&] {
        if (!h) return fail(KAO_E_ARG, "null handle");
        if (evaluator != KAO_EVAL_ROW_MAJOR && evaluator != KAO_EVAL_COLUMN_MAJOR) return fail(KAO_E_ARG, "unknown evaluator");
        if (evaluator == KAO_EVAL_COLUMN_MAJOR && !h->trans_ok)
            return fail(KAO_E_ARG, "column-major evaluator: needs rows of up to 64 slots, racks of up to 8 brokers, at most one "
                                   "replica per rack (C7 0..1), three objective mask planes, and its planes in shared memory");
        h->evaluator = evaluator;
        return KAO_OK;
    });
}
extern "C" int kao_set_schedule(kao_handle *h, int32_t sync, int32_t pop, int32_t threads)
{
    return guarded([&] {
        if (!h) return fail(KAO_E_ARG, "null handle");
        if (!schedule_exists(sync, pop, threads)) return fail(KAO_E_ARG, "no such schedule (kao.h, kao_set_schedule)");
        h->sch_sync = sync; h->sch_pop = pop; h->sch_threads = threads;
        return KAO_OK;
    });
}
extern "C" int kao_get_evaluator(kao_handle *h, int32_t *evaluator, int32_t *sync, int32_t *pop, int32_t *threads)
{
    if (!h) return fail(KAO_E_ARG, "null handle");
    if (evaluator) *evaluator = h->evaluator;
    if (sync) *sync = h->sch_sync;
    if (pop) *pop = h->sch_pop;
    if (threads) *threads = h->sch_threads;
    return KAO_OK;
}
extern "C" int kao_set_patience(kao_handle *h, uint32_t rounds_without_improvement)
{
    if (!h) return fail(KAO_E_ARG, "null handle");
    h->patience = rounds_without_improvement;
    return KAO_OK;
}
extern "C" int kao_last_rounds(kao_handle *h, uint32_t *rounds_run)
{
    if (!h || !rounds_run) return fail(KAO_E_ARG, "null argument");
    *rounds_run = h->last_rounds;
    return KAO_OK;
}
extern "C" int kao_search(kao_handle *h, uint64_t seed, uint32_t first_round, uint32_t rounds,
                          uint32_t round_size, uint64_t *round_keys, double *device_ms)
{
    return guarded([&] { return search_impl(h, seed, first_round, rounds, round_size, round_keys, device_ms, false); });
}
// Same search, same keys, same trajectory — but every candidate is scored by DELTA evaluation
// (base totals + its <= 3 patched rows, one thread per candidate) instead of a full evaluation.
extern "C" int kao_search_delta(kao_handle *h, uint64_t seed, uint32_t first_round, uint32_t rounds,
                                uint32_t round_size, uint64_t *round_keys, double *device_ms)
{
    return guarded([&] { return search_impl(h, seed, first_round, rounds, round_size, round_keys, device_ms, true); });
}
extern "C" int kao_candidate_keys(kao_handle *h, uint64_t seed, uint32_t round, uint32_t round_size,
                                  uint32_t idx_begin, uint32_t count, uint64_t *keys)
{
    return guarded([&] { return candidate_keys_impl(h, seed, round, round_size, idx_begin, count, keys, false); });
}
extern "C" int kao_candidate_keys_delta(kao_handle *h, uint64_t seed, uint32_t round, uint32_t round_size,
                                        uint32_t idx_begin, uint32_t count, uint64_t *keys)
{
    return guarded([&] { return candidate_keys_impl(h, seed, round, round_size, idx_begin, count, keys, true); });
}
extern "C" int kao_p2p_export(kao_handle *h, uint8_t *handle_out) { return guarded([&] { return p2p_export_impl(h, handle_out); }); }
extern "C" int kao_p2p_connect(kao_handle *h, int32_t rank, int32_t world, const uint8_t *handles)
{
    return guarded([&] { return p2p_connect_impl(h, rank, world, handles); });
}
extern "C" int kao_search_sharded(kao_handle *h, uint64_t seed, uint32_t first_round, uint32_t rounds,
                                  uint32_t round_size, uint64_t *round_keys, double *device_ms)
{
    return guarded([&] { return sharded_impl(h, seed, first_round, rounds, round_size, round_keys, device_ms, false); });
}
extern "C" int kao_search_sharded_delta(kao_handle *h, uint64_t seed, uint32_t first_round, uint32_t rounds,
                                        uint32_t round_size, uint64_t *round_keys, double *device_ms)
{
    return guarded([&] { return sharded_impl(h, seed, first_round, rounds, round_size, round_keys, device_ms, true); });
}
extern "C" int kao_profile_rounds(kao_handle *h, uint64_t seed, uint32_t first_round, uint32_t rounds,
                                  uint32_t round_size, double *search_ms, double *apply_ms)
{
    return guarded([&] { return profile_rounds_impl(h, seed, first_round, rounds, round_size, search_ms, apply_ms); });
}
extern "C" int kao_stats(kao_handle *h, uint64_t *kernel_launches, int32_t *words_per_row,
                         int32_t *slots, int32_t *dense_weights)
{
    if (!h) return fail(KAO_E_ARG, "null handle");
    if (kernel_launches) *kernel_launches = h->launches;
    if (words_per_row) *words_per_row = h->hm.W;
    if (slots) *slots = h->hm.NS;
    if (dense_weights) *dense_weights = h->hm.dense ? 1 : 0;
    return KAO_OK;
}
extern "C" int kao_eval(const kao_problem *pb, int32_t device, const int32_t *replicas, int32_t n,
                        int64_t *violation, int64_t *objective)
{
    return guarded([&] { return eval_impl(pb, device, replicas, n, violation, objective); });
}
extern "C" int kao_solve(const kao_problem *pb, const kao_options *opt, kao_result *res)
{
    return guarded([&] { return solve_impl(pb, opt, res); });
}
