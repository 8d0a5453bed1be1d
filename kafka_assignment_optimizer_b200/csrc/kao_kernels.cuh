// kao_kernels.cuh — the search kernels (one search round; all rounds in one persistent cooperative
// launch, full or delta evaluation) and what they share with the host side: the shared-memory plan
// and the cross-GPU mailbox.  Included by kao_engine.cu (host side, C ABI; the kernels are only
// DECLARED there through explicit instantiation declarations) and by kao_inst.cu, which is compiled
// once per (row width, counter depth, evaluation mode) and holds the explicit instantiations — the
// translation units build in parallel and every one of them is compiled deterministically.
#pragma once
#include "kao_device.cuh"
#include "kao_device_t.cuh"
#include "kao_plan.hpp"

#include <cstdint>

using namespace kao;

// threads per CTA: row-major full evaluation (rows of up to 64 slots / wider rows), delta evaluation
constexpr int kThreads = 768;
constexpr int kThreadsWide = 256;
constexpr int kThreadsDelta = 512;
template <int W> constexpr int threads_for() { return W <= 2 ? kThreads : kThreadsWide; }
// threads per CTA of the full-evaluation kernels of a configuration (column-major schedules may choose)
template <class Cfg> constexpr int cfg_threads()
{
    if constexpr (Cfg::kTrans) return Cfg::kThreads ? Cfg::kThreads : threads_for<Cfg::W>();
    else return threads_for<Cfg::W>();
}

// ------------------------------------------------------------------------------------------
// PTX wrappers: mbarrier + TMA bulk copy (SASS: SYNCS / UBLKCP)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t ok = 0;
    while (!ok) {
        asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    }
}

// Leader one-hot plane of the shared-memory base (kao_device.cuh, has_oh_plane): row & (1 << leader),
// empty when the leader slot is not one of the row's replicas.  Stored right behind the bit-plane.
template <int W> __device__ __forceinline__ uint32_t oh_word(uint32_t x, uint32_t ld, int w)
{
    return ((int)(ld >> 5) == w) ? (x & (1u << (ld & 31u))) : 0u;
}
template <int W, int THREADS>
__device__ __forceinline__ void build_oh_plane(uint32_t *s_bits, const uint8_t *s_leader, int Ppad)
{
    for (int p = threadIdx.x; p < Ppad; p += THREADS) {
        const uint32_t ld = s_leader[p];
#pragma unroll
        for (int w = 0; w < W; ++w) s_bits[(size_t)(W + w) * Ppad + p] = oh_word<W>(s_bits[(size_t)w * Ppad + p], ld, w);
    }
    __syncthreads();
}

// Column-major evaluator (kao_device_t.cuh): the two transposed planes and the term planes of the objective
// are gathered once per launch from the staged row-major base (2 * W words per partition at off_sw, the term
// planes at off_z).
template <int W, int THREADS>
__device__ __forceinline__ void build_t_planes(const Params &d, uint32_t *T, uint32_t *Z, const uint32_t *s_bits, const uint8_t *s_leader)
{
    constexpr int NSL = 32 * W;
    const int nW = t_words(d.Ppad), total = kTPlanes * NSL * nW;
    for (int o = threadIdx.x; o < total; o += THREADS) {
        const int w = o % nW, s = (o / nW) % NSL, q = o / (nW * NSL);
        T[t_word(q, s, w, nW, NSL)] = t_gather<W>(q, s, w, s_bits, s_leader, d.Ppad);
    }
    for (int o = threadIdx.x; o < kZPlanes * nW; o += THREADS) Z[o] = z_gather<W>(d, o / nW, o % nW, s_bits, s_leader);
    for (int o = threadIdx.x; o < kAPlanes<W>() * nW; o += THREADS) Z[kZPlanes * nW + o] = a_gather<W>(o / nW, o % nW, s_bits, d.Ppad);
    __syncthreads();
}

// One search round (or a slice of it): every warp walks candidate indices idx_lo + gw, + stride ...,
// generates the candidate from the shared-memory base, evaluates it in full and keeps the minimum
// packed key; the block minimum goes to *out_key with one atomicMin.  all_keys (optional)
// receives every candidate's key (parity tests).
template <class Cfg, int THREADS>
__global__ void __launch_bounds__(THREADS, 1)
search_round_kernel(Params d, SmemPlan plan, uint64_t seed, uint32_t round, uint32_t round_size,
                    uint32_t idx_lo, uint32_t idx_hi, unsigned long long *out_key,
                    unsigned long long *all_keys)
{
    extern __shared__ __align__(128) uint8_t smem[];
    uint32_t *s_bits = reinterpret_cast<uint32_t *>(smem + plan.off_bits);
    uint32_t *s_sw = reinterpret_cast<uint32_t *>(smem + plan.off_sw);
    uint8_t *s_leader = smem + plan.off_leader;
    Consts *s_cs = reinterpret_cast<Consts *>(smem + plan.off_consts);
    uint32_t *s_prow = reinterpret_cast<uint32_t *>(smem + plan.off_prow);
    unsigned long long *s_red = reinterpret_cast<unsigned long long *>(smem + plan.off_red);
    uint64_t *s_bar = reinterpret_cast<uint64_t *>(smem + plan.off_bar);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int kWarps = THREADS / 32;
    constexpr int W = Cfg::W;
    const uint32_t *g_obj = Cfg::kObj > 0 ? d.planesT : d.swT;
    const uint32_t obj_words = Cfg::kObj > 0 ? (uint32_t)Cfg::kObj * W : (uint32_t)d.nentries;

    // stage base + tables: HBM/L2 -> shared memory with TMA bulk copies, one mbarrier
    if (tid == 0) mbar_init(s_bar, 1);
    __syncthreads();
    if (tid == 0) {
        const uint32_t nb = (uint32_t)W * d.Ppad * 4, ns = obj_words * d.Ppad * 4, nl = (uint32_t)d.Ppad;
        mbar_expect_tx(s_bar, nb + ns + nl + (uint32_t)sizeof(Consts));
        bulk_g2s(s_bits, d.bitsT, nb, s_bar);
        if (ns) bulk_g2s(s_sw, g_obj, ns, s_bar);
        bulk_g2s(s_leader, d.leader, nl, s_bar);
        bulk_g2s(s_cs, d.consts, (uint32_t)sizeof(Consts), s_bar);
    }
    mbar_wait(s_bar, 0);
    if constexpr (has_oh_plane<Cfg>()) build_oh_plane<W, THREADS>(s_bits, s_leader, d.Ppad);

    Gen<W> gen;
    uint32_t no_rows[kMaxOps][W];          // warp mode keeps patched rows in shared memory instead
    gen.bitsT = s_bits; gen.leader = s_leader; gen.cs = s_cs; gen.d = &d;
    gen.prow = s_prow + warp * kMaxOps * W; gen.lane = lane;
    gen.D = d.D; gen.DL = d.DL; gen.nD = d.nD[0]; gen.nL = d.nD[1];

    unsigned long long best = kKeyNone;
    const uint32_t stride = gridDim.x * kWarps;
    // every warp of the block runs the same number of iterations and meets at a barrier before each
    // evaluation: the warps of a scheduler then walk the same code together (instruction cache)
    const uint32_t first = idx_lo + blockIdx.x * kWarps;
    const uint32_t iters = first < idx_hi ? (idx_hi - first + stride - 1) / stride : 0;
    for (uint32_t it = 0; it < iters; ++it) {
        const uint32_t idx = first + warp + it * stride;
        const bool live = idx < idx_hi;
        PatchSet ps;
        ps.n = 0;
#pragma unroll
        for (int i = 0; i < kMaxOps; ++i) { ps.p[i] = -1; ps.ld[i] = 0xFF; }
        if (live) gen.run(seed, round, idx, round_size, ps, no_rows);
        __syncthreads();
        if (live) {
            int viol, obj;
            eval_candidate<Cfg, true>(d, s_bits, s_leader, s_sw, s_cs, ps, gen.prow, lane, viol, obj);
            const unsigned long long key = live ? pack_key(viol, obj, idx, d.key_obj_bits) : kKeyNone;
            if (all_keys && lane == 0) all_keys[idx - idx_lo] = key;
            best = key < best ? key : best;
        }
        __syncwarp();
    }
    if (lane == 0) s_red[warp] = best;
    __syncthreads();
    if (warp == 0) {
        unsigned long long v = lane < kWarps ? s_red[lane] : kKeyNone;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long w = __shfl_xor_sync(0xFFFFFFFFu, v, o);
            v = w < v ? w : v;
        }
        if (lane == 0 && v != kKeyNone) atomicMin(out_key, v);
    }
}

// Rebuilds the displaced lists of a base with the whole block (ballot compaction, ascending
// order).  cnt: 2 x 36 ints of shared scratch.  counts[0] = |D|, counts[1] = |DL|.
template <int THREADS>
__device__ __forceinline__ void rebuild_lists(const uint32_t *bitsT, const uint8_t *leader, const uint32_t *homeT,
                                              int P, int Ppad, uint16_t *D, uint16_t *DL, int *counts, int *cnt)
{
    constexpr int kWarps = THREADS / 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int *cD = cnt, *cL = cnt + 36;
    int baseD = 0, baseL = 0;
    for (int p0 = 0; p0 < P; p0 += THREADS) {
        const int p = p0 + tid;
        bool miss = false, ldis = false;
        if (p < P) {
            const uint32_t h4 = homeT[p];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int hs = (h4 >> (8 * i)) & 0xFF;
                if (hs != 0xFF) {
                    const bool has = (bitsT[(size_t)(hs >> 5) * Ppad + p] >> (hs & 31)) & 1u;
                    miss |= !has;
                    if (i == 0) ldis = has && ((int)leader[p] != hs);
                }
            }
        }
        const uint32_t mD = __ballot_sync(0xFFFFFFFFu, miss);
        const uint32_t mL = __ballot_sync(0xFFFFFFFFu, ldis);
        if (lane == 0) { cD[warp] = __popc(mD); cL[warp] = __popc(mL); }
        __syncthreads();
        if (warp == 0) {
            int c = lane < kWarps ? cD[lane] : 0, incl = c, cl = lane < kWarps ? cL[lane] : 0, incl2 = cl;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(0xFFFFFFFFu, incl, o);
                const int v2 = __shfl_up_sync(0xFFFFFFFFu, incl2, o);
                if (lane >= o) { incl += v; incl2 += v2; }
            }
            cD[lane] = incl - c;
            cL[lane] = incl2 - cl;
            if (lane == 31) { cD[32] = incl; cL[32] = incl2; }
        }
        __syncthreads();
        const uint32_t below = (1u << lane) - 1u;
        if (miss) D[baseD + cD[warp] + __popc(mD & below)] = (uint16_t)p;
        if (ldis) DL[baseL + cL[warp] + __popc(mL & below)] = (uint16_t)p;
        baseD += cD[32];
        baseL += cL[32];
        __syncthreads();
    }
    if (tid == 0) { counts[0] = baseD; counts[1] = baseL; }
    __syncthreads();
}

// Cross-GPU exchange state of the persistent kernel (docs/MODEL.md §7): every rank owns a mailbox in
// its HBM that all peers can write (mapped through CUDA IPC between processes, or directly with peer
// access inside one process).  Per round every rank stores its 8-byte key into ITS slot of every
// mailbox (one NVLink store per peer, all in flight together) and polls its own mailbox until the
// slots of all ranks are filled — the key is its own flag, no counter, no fence between the two; the
// minimum of the slots is the round's winner on every rank.  No host, no NCCL in the loop.
constexpr int kMaxPeers = 8;
constexpr uint32_t kMailRounds = 8192;          // rounds per launch when sharded
constexpr unsigned long long kMailEmpty = ~0ull;   // no key has bit 63 set
struct Mailbox {
    unsigned long long slot[2][kMailRounds][kMaxPeers];   // [bank][round][rank]
};
struct P2P {
    int rank, world, bank;
    uint32_t idx_lo, idx_hi;                    // this rank's slice of every round
    Mailbox *const *mail;                       // [world] peer-mapped mailboxes (device array), mail[rank] is local
    unsigned long long *lkeys;                  // [rounds] this GPU's own minimum per round
    unsigned int *release;                      // CTA 0 publishes "round t is decided" here
    int *abort;                                 // set when a wait times out (a peer died): everybody leaves
    uint32_t patience;                          // > 0: stop after this many rounds without a better key
    unsigned int *rounds_run;                   // CTA 0 reports the number of rounds actually run
    // early-stop state carried from one launch of a long search to the next (the host passes the values the
    // previous launch left in `carry`): best (violation, cost) so far, rounds since it improved
    unsigned long long best_in;
    uint32_t stall_in;
    unsigned long long *carry;                  // [2] CTA 0 leaves (best, stall) here
    unsigned long long timeout_ns;              // budget of every wait (grid barrier, peers)
};

__device__ __forceinline__ unsigned long long global_ns()
{
#if defined(KAO_HOST_EMU)
    return 0;
#else
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
#endif
}
// waits in wall time (the SM clock would make the budget depend on the clock frequency)
__device__ __forceinline__ bool spin_until(const unsigned int *p, unsigned int target, int *abort_flag, unsigned long long budget_ns)
{
    const unsigned long long t0 = global_ns();
    while (*reinterpret_cast<const volatile unsigned int *>(p) < target) {
        if (*reinterpret_cast<volatile int *>(abort_flag)) return false;
        if (global_ns() - t0 > budget_ns) { atomicExch(abort_flag, 1); return false; }
    }
    return true;
}
__device__ __forceinline__ bool spin_filled(const unsigned long long *p, unsigned long long &v, int *abort_flag, unsigned long long budget_ns)
{
    const unsigned long long t0 = global_ns();
    while ((v = *reinterpret_cast<const volatile unsigned long long *>(p)) == kMailEmpty) {
        if (*reinterpret_cast<volatile int *>(abort_flag)) return false;
        if (global_ns() - t0 > budget_ns) { atomicExch(abort_flag, 1); return false; }
    }
    return true;
}

// Per-round tables of the base for the per-THREAD generator (and the delta evaluator): replica / valid-leader
// counts per slot, replicas per rack, and per-slot inverted lists (ascending partitions that hold a replica
// on / are led from the slot) so that a thread finds "the first holder of slot s from partition q on" by a
// binary search instead of a scan.  All in shared memory at plan.off_totals / plan.off_inv; rebuilt by the
// whole CTA whenever the base has changed.
struct RoundTables {
    int *cnt, *lcnt, *rc, *base, *ledn, *hoff, *loff, *inv;
    uint16_t *hold, *led;
};
__device__ __forceinline__ RoundTables round_tables(uint8_t *smem, const SmemPlan &plan)
{
    RoundTables r;
    r.cnt = reinterpret_cast<int *>(smem + plan.off_totals);
    r.lcnt = r.cnt + 256; r.rc = r.cnt + 512; r.base = r.cnt + 544;
    r.ledn = r.cnt + 548; r.hoff = r.cnt + 804; r.loff = r.cnt + 1062; r.inv = r.cnt + 1320;
    r.hold = reinterpret_cast<uint16_t *>(smem + plan.off_inv);
    r.led = r.hold + plan.cap_hold;
    return r;
}
template <int W, int THREADS>
__device__ __forceinline__ void build_round_tables(const RoundTables &rt, const SmemPlan &plan, const Params &d,
                                                   const uint32_t *s_bits, const uint8_t *s_leader)
{
    const int tid = threadIdx.x;
    for (int i = tid; i < 804; i += THREADS) if (i < 544 || i >= 548) rt.cnt[i] = 0;   // keep rt.base
    __syncthreads();
    for (int p = tid; p < d.P; p += THREADS) {
        const int ld = s_leader[p];
        bool ok = false;
#pragma unroll
        for (int w = 0; w < W; ++w) {
            const uint32_t xw = s_bits[(size_t)w * d.Ppad + p];
            for (uint32_t m = xw; m; m &= m - 1) {
                const int sl = w * 32 + __ffs(m) - 1;
                atomicAdd(&rt.cnt[sl], 1);
                atomicAdd(&rt.rc[sl >> d.log2S], 1);
            }
            if ((ld >> 5) == w) ok = (xw >> (ld & 31)) & 1u;
        }
        if (ok) atomicAdd(&rt.lcnt[ld], 1);
        atomicAdd(&rt.ledn[ld], 1);
    }
    __syncthreads();
    if (tid == 0) {
        int a = 0, b = 0;
        for (int sl = 0; sl < W * 32; ++sl) { rt.hoff[sl] = a; a += rt.cnt[sl]; rt.loff[sl] = b; b += rt.ledn[sl]; }
        rt.hoff[W * 32] = a; rt.loff[W * 32] = b;
        *rt.inv = (plan.cap_hold > 0 && a <= (int)plan.cap_hold && b <= (int)plan.cap_led) ? 1 : 0;
    }
    __syncthreads();
    if (*rt.inv) {
        // THREADS / slots segments of rows per slot: count, then write in place (ascending order)
        constexpr int NSL = W * 32, NSEG = THREADS / NSL;
        static_assert(THREADS % NSL == 0, "one thread per (segment, slot)");
        int *s_segc = reinterpret_cast<int *>(rt.led + plan.cap_led + 8);       // [2][NSEG][NSL]
        const int slot = tid % NSL, seg = tid / NSL;
        const int chunk = (d.P + NSEG - 1) / NSEG, p_lo = seg * chunk, p_hi = min(d.P, p_lo + chunk);
        const uint32_t *col = s_bits + (size_t)(slot >> 5) * d.Ppad;
        const uint32_t bit = 1u << (slot & 31);
        int hc = 0, lc = 0;
        for (int p = p_lo; p < p_hi; ++p) {
            hc += (col[p] & bit) ? 1 : 0;
            lc += ((int)s_leader[p] == slot) ? 1 : 0;
        }
        s_segc[seg * NSL + slot] = hc;
        s_segc[(NSEG + seg) * NSL + slot] = lc;
        __syncthreads();
        int hpos = rt.hoff[slot], lpos = rt.loff[slot];
        for (int g = 0; g < seg; ++g) { hpos += s_segc[g * NSL + slot]; lpos += s_segc[(NSEG + g) * NSL + slot]; }
        for (int p = p_lo; p < p_hi; ++p) {
            if (col[p] & bit) rt.hold[hpos++] = (uint16_t)p;
            if ((int)s_leader[p] == slot) rt.led[lpos++] = (uint16_t)p;
        }
    }
    __syncthreads();
}
template <int W, bool kSmall>
__device__ __forceinline__ void bind_tables(Gen<W, true, kSmall> &tg, const RoundTables &rt)
{
    tg.inv_ok = *rt.inv != 0; tg.hoff = rt.hoff; tg.loff = rt.loff; tg.hold = rt.hold; tg.led = rt.led;
}

// Column-major kernels: the 32 lanes of a warp generate 32 candidates at once (one each, per-thread
// generator) and park them in the warp's scratch; the warp then evaluates them one after the other.
// Scratch per candidate: 3 partitions, (leader slots | count << 24), 3 x W row words (16-byte aligned).
template <int W> __host__ __device__ constexpr int batch_stride() { return batch_stride_words(W); }

// All rounds of a search in ONE launch (cooperative: one CTA per SM, all co-resident).  The base
// and the tables stay in shared memory for the whole search; per round every CTA evaluates its
// share of the candidates, min-reduces into keys[t], meets the other CTAs at a grid barrier, then
// re-materialises the winner itself and patches its own shared-memory copy of the base (<= 3
// rows) — nothing but one 8-byte key crosses the chip per round.  CTA 0 mirrors the patches into
// the HBM base.
template <class Cfg, int THREADS, bool kDelta>
__global__ void __launch_bounds__(THREADS, 1)
search_persistent_kernel(Params d, SmemPlan plan, uint64_t seed, uint32_t first_round, uint32_t rounds,
                         uint32_t round_size, unsigned long long *keys, unsigned int *grid_bar, P2P pp,
                         unsigned long long *all_keys)
{
    extern __shared__ __align__(128) uint8_t smem[];
    uint32_t *s_bits = reinterpret_cast<uint32_t *>(smem + plan.off_bits);
    uint32_t *s_sw = reinterpret_cast<uint32_t *>(smem + plan.off_sw);
    uint8_t *s_leader = smem + plan.off_leader;
    Consts *s_cs = reinterpret_cast<Consts *>(smem + plan.off_consts);
    uint32_t *s_prow = reinterpret_cast<uint32_t *>(smem + plan.off_prow);
    unsigned long long *s_red = reinterpret_cast<unsigned long long *>(smem + plan.off_red);
    uint64_t *s_bar = reinterpret_cast<uint64_t *>(smem + plan.off_bar);
    int &s_abort = *reinterpret_cast<int *>(smem + plan.off_bar + 8);   // no static shared memory: the
                                                                        // dynamic limit is the full 227 KB
    uint16_t *s_D = reinterpret_cast<uint16_t *>(smem + plan.off_lists);
    uint16_t *s_DL = s_D + d.Ppad;
    int *s_counts = reinterpret_cast<int *>(smem + plan.off_lists + (size_t)d.Ppad * 4);
    int *s_scan = s_counts + 4;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int kWarps = THREADS / 32;
    constexpr int W = Cfg::W;
    const uint32_t *g_obj = Cfg::kObj > 0 ? d.planesT : d.swT;
    constexpr bool kObjShared = !(kDelta && W > 2);    // wide-row delta kernels read the objective table from HBM / L2
    // (the column-major evaluator stages no objective table: it keeps term planes, built below)
    const uint32_t obj_words = (!kObjShared || Cfg::kTrans) ? 0u : (Cfg::kObj > 0 ? (uint32_t)Cfg::kObj * W : (uint32_t)d.nentries);
    uint32_t *s_z = reinterpret_cast<uint32_t *>(smem + plan.off_z);

    if (tid == 0) mbar_init(s_bar, 1);
    __syncthreads();
    if (tid == 0) {
        const uint32_t nb = (uint32_t)W * d.Ppad * 4, ns = obj_words * d.Ppad * 4, nl = (uint32_t)d.Ppad;
        mbar_expect_tx(s_bar, nb + ns + nl + (uint32_t)sizeof(Consts));
        bulk_g2s(s_bits, d.bitsT, nb, s_bar);
        if (ns) bulk_g2s(s_sw, g_obj, ns, s_bar);
        bulk_g2s(s_leader, d.leader, nl, s_bar);
        bulk_g2s(s_cs, d.consts, (uint32_t)sizeof(Consts), s_bar);
    }
    mbar_wait(s_bar, 0);
    if constexpr (has_oh_plane<Cfg>()) build_oh_plane<W, THREADS>(s_bits, s_leader, d.Ppad);
    if constexpr (Cfg::kTrans) build_t_planes<W, THREADS>(d, s_sw, s_z, s_bits, s_leader);
    rebuild_lists<THREADS>(s_bits, s_leader, d.homeT, d.P, d.Ppad, s_D, s_DL, s_counts, s_scan);
    if constexpr (Cfg::kTrans) {
        // s_counts[2] = partitions whose leader slot is not one of their replicas (0 for every base the engine builds or
        // reaches itself): while it is 0 the leader plane T1 also answers the generator's "is led from slot s"
        if (tid == 0) s_counts[2] = 0;
        __syncthreads();
        int bad = 0;
        for (int p = tid; p < d.P; p += THREADS) {
            const int ld = s_leader[p];
            bad += (ld < W * 32 && ((s_bits[(size_t)(ld >> 5) * d.Ppad + p] >> (ld & 31)) & 1u)) ? 0 : 1;
        }
        if (bad) atomicAdd(&s_counts[2], bad);
        __syncthreads();
    }

    Gen<W, false, Cfg::kTrans> gen;        // column-major kernels: compact generator code (same candidates)
    uint32_t no_rows[kMaxOps][W];          // warp mode keeps patched rows in shared memory instead
    gen.bitsT = s_bits; gen.leader = s_leader; gen.cs = s_cs; gen.d = &d;
    gen.prow = s_prow + (size_t)warp * (Cfg::kTrans ? 32 * batch_stride<W>() : kMaxOps * W); gen.lane = lane;
    gen.D = s_D; gen.DL = s_DL;

    const uint32_t stride = gridDim.x * kWarps;
    const uint32_t first = pp.idx_lo + blockIdx.x * kWarps;
    const uint32_t iters = first < pp.idx_hi ? (pp.idx_hi - first + stride - 1) / stride : 0;
    if (tid == 0) s_abort = 0;
    // early-stop state lives behind the per-warp minima (s_red is live anyway; a separate pointer would
    // cost a register in the hot loop): [kWarps] stop flag, [kWarps+1] best (violation, cost), [kWarps+2] stall
    if (tid == 0) { s_red[kWarps] = 0; s_red[kWarps + 1] = pp.best_in; s_red[kWarps + 2] = pp.stall_in; }
    for (uint32_t t = 0; t < rounds; ++t) {
        const uint32_t round = first_round + t;
        gen.nD = s_counts[0]; gen.nL = s_counts[1];
        unsigned long long best = kKeyNone;
        if constexpr (kDelta) {
            // ---- delta mode: totals of the base once per round, then one THREAD per candidate
            const RoundTables rt = round_tables(smem, plan);
            int *s_cnt = rt.cnt, *s_lcnt = rt.lcnt, *s_rc = rt.rc, *s_base = rt.base;
            build_round_tables<W, THREADS>(rt, plan, d, s_bits, s_leader);
            // the base's own evaluation: a full pass in the first round, afterwards it IS the previous
            // winner's key (unless that key was saturated)
            if (warp == 0 && (t == 0 || s_base[2] == 0)) {
                PatchSet id;
                id.n = 0;
#pragma unroll
                for (int i = 0; i < kMaxOps; ++i) { id.p[i] = -1; id.ld[i] = 0xFF; }
                int bv, bo;
                eval_candidate<Cfg, true, kObjShared>(d, s_bits, s_leader, kObjShared ? s_sw : g_obj, s_cs, id, gen.prow, lane, bv, bo);
                if (lane == 0) { s_base[0] = bv; s_base[1] = bo; }
            }
            __syncthreads();
            Gen<W, true> tg;
            tg.bitsT = s_bits; tg.leader = s_leader; tg.cs = s_cs; tg.d = &d; tg.prow = nullptr; tg.lane = 0;
            tg.D = s_D; tg.DL = s_DL; tg.nD = s_counts[0]; tg.nL = s_counts[1];
            bind_tables(tg, rt);
            const MemRef<kObjShared> m_obj(kObjShared ? s_sw : g_obj);
            const int base_viol = s_base[0], base_obj = s_base[1];
            const uint32_t tstride = gridDim.x * THREADS;
            for (uint32_t idx = pp.idx_lo + blockIdx.x * THREADS + tid; idx < pp.idx_hi; idx += tstride) {
                PatchSet ps;
                uint32_t rows[kMaxOps][W];
                tg.run(seed, round, idx, round_size, ps, rows);
                int viol, obj;
                delta_eval<Cfg, kObjShared>(d, s_bits, s_leader, m_obj, s_cs, ps, rows, s_cnt, s_lcnt, s_rc, base_viol, base_obj, viol, obj);
                const unsigned long long key = pack_key(viol, obj, idx, d.key_obj_bits);
                if (all_keys) all_keys[idx - pp.idx_lo] = key;
                best = key < best ? key : best;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const unsigned long long w = __shfl_xor_sync(0xFFFFFFFFu, best, o);
                best = w < best ? w : best;
            }
            if (all_keys) return;                                   // key dump only: the base stays as it is
        } else if constexpr (Cfg::kTrans) {
            // ---- column-major evaluator: candidates are generated 32 at a time, one per LANE (per-thread
            // generator scanning the transposed planes), then evaluated in full one after the other by the warp
            Gen<W, true, true> tg;        // compact code (row_kth keeps its loop), same candidates
            tg.bitsT = s_bits; tg.leader = s_leader; tg.cs = s_cs; tg.d = &d; tg.prow = nullptr; tg.lane = 0;
            tg.D = s_D; tg.DL = s_DL; tg.nD = s_counts[0]; tg.nL = s_counts[1];
            tg.T = s_sw; tg.tnW = t_words(d.Ppad); tg.t_leaders_valid = s_counts[2] == 0;    // "first holder of slot s": plane scan
            constexpr int BS = batch_stride<W>();
            uint32_t *batch = s_prow + (size_t)warp * 32 * BS;
            LaneBounds<W> lb;
            lb.load(s_cs, lane, d.R);
            // the warp's best candidate of the round as (violation, cost, index) — the fields of the packed key, compared
            // field by field and packed once per round (indices rise within a warp: the first of equals stays)
            const uint32_t vcap32 = (uint32_t)key_viol_cap(d.key_obj_bits), omax = (1u << d.key_obj_bits) - 1u;
            uint32_t bv = 0xFFFFFFFFu, bc = 0, bi = 0;              // bv: no candidate yet (a violation field never exceeds 2^31 - 1)
            for (uint32_t it0 = 0; it0 < iters; it0 += 32) {
                {
                    const uint32_t idx = first + warp + (it0 + lane) * stride;
                    PatchSet ps;
                    uint32_t rows[kMaxOps][W];
                    ps.n = 0;
#pragma unroll
                    for (int i = 0; i < kMaxOps; ++i) {
                        ps.p[i] = -1; ps.ld[i] = 0xFF;
#pragma unroll
                        for (int w = 0; w < W; ++w) rows[i][w] = 0;
                    }
                    if (it0 + lane < iters && idx < pp.idx_hi) tg.run(seed, round, idx, round_size, ps, rows);
                    int pviol, pobj, pcount;
                    patch_terms<W>(d, ps, rows, pviol, pobj, pcount);
                    uint32_t *mine = batch + lane * BS;
                    // pviol <= 3 * 128, pcount <= 3 * 64, partitions < 8192 (0xFFFF = unused patch)
                    mine[0] = ((uint32_t)ps.p[0] & 0xFFFFu) | ((uint32_t)ps.p[1] << 16);
                    mine[1] = ((uint32_t)ps.p[2] & 0xFFFFu) | ((uint32_t)pcount << 16);
                    mine[2] = (uint32_t)pviol; mine[3] = (uint32_t)pobj;
                    patch_column_deltas<W>(d, ps, rows, s_bits, s_leader, reinterpret_cast<uint8_t *>(mine + kBatchHdr));
                }
                __syncwarp();
                const uint32_t nb = iters - it0 < 32u ? iters - it0 : 32u;
                for (uint32_t j = 0; j < nb; ++j) {
                    const uint32_t idx = first + warp + (it0 + j) * stride;
                    if constexpr (Cfg::kSync == 0) __syncthreads();          // all warps walk the evaluator together
                    if (idx < pp.idx_hi) {
                        const uint32_t *slot = batch + j * BS;
                        const uint4 hdr = *reinterpret_cast<const uint4 *>(slot);
                        PatchSet ps;
                        ps.p[0] = (int)(int16_t)(hdr.x & 0xFFFFu); ps.p[1] = (int)(int16_t)(hdr.x >> 16); ps.p[2] = (int)(int16_t)(hdr.y & 0xFFFFu);
                        ps.n = 0;                                           // the evaluator reads the partitions only
                        ps.ld[0] = ps.ld[1] = ps.ld[2] = 0xFF;
                        int viol, obj;
                        eval_candidate_t<Cfg, true>(d, s_sw, t_words(d.Ppad), s_bits, s_z, lb, ps, reinterpret_cast<const uint8_t *>(slot + kBatchHdr),
                                                    (int)hdr.z, (int)hdr.w, (int)(hdr.y >> 16), lane, viol, obj);
                        if (all_keys && lane == 0) all_keys[idx - pp.idx_lo] = pack_key(viol, obj, idx, d.key_obj_bits);
                        const uint32_t v = min((uint32_t)max(viol, 0), vcap32);
                        const uint32_t c = (uint32_t)obj > omax ? 0u : omax - (uint32_t)obj;
                        if (v < bv || (v == bv && c < bc)) { bv = v; bc = c; bi = idx; }
                    }
                }
                __syncwarp();                                               // the batch is consumed before it is refilled
            }
            if (bv != 0xFFFFFFFFu)
                best = ((unsigned long long)bv << (kIdxBits + d.key_obj_bits)) | ((unsigned long long)bc << kIdxBits) | (unsigned long long)(bi & kIdxMask);
            if (all_keys) return;                                           // key dump only: the base stays as it is
        } else {
        for (uint32_t it = 0; it < iters; ++it) {
            const uint32_t idx = first + warp + it * stride;
            const bool live = idx < pp.idx_hi;
            PatchSet ps;
            ps.n = 0;
#pragma unroll
            for (int i = 0; i < kMaxOps; ++i) { ps.p[i] = -1; ps.ld[i] = 0xFF; }
            if (live) gen.run(seed, round, idx, round_size, ps, no_rows);
            __syncthreads();
            if (live) {
                int viol, obj;
                eval_candidate<Cfg, true>(d, s_bits, s_leader, s_sw, s_cs, ps, gen.prow, lane, viol, obj);
                const unsigned long long key = pack_key(viol, obj, idx, d.key_obj_bits);
                best = key < best ? key : best;
            }
            __syncwarp();
        }
        }
        if (lane == 0) s_red[warp] = best;
        __syncthreads();
        if (warp == 0) {
            unsigned long long v = lane < kWarps ? s_red[lane] : kKeyNone;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const unsigned long long w = __shfl_xor_sync(0xFFFFFFFFu, v, o);
                v = w < v ? w : v;
            }
            if (pp.world == 1) {
                if (lane == 0) {
                    if (v != kKeyNone) atomicMin(keys + t, v);
                    // grid barrier: every CTA's contribution to keys[t] is visible before anyone reads it
                    __threadfence();
                    atomicAdd(grid_bar, 1u);
                    if (!spin_until(grid_bar, (t + 1) * gridDim.x, pp.abort, pp.timeout_ns)) s_abort = 1;
                    __threadfence();
                }
            } else {
                // 1. this GPU's minimum
                if (lane == 0) {
                    if (v != kKeyNone) atomicMin(pp.lkeys + t, v);
                    __threadfence();
                    atomicAdd(grid_bar, 1u);
                }
                if (blockIdx.x == 0) {
                    // 2. CTA 0 trades it with every peer over NVLink: lane r stores this rank's key into its slot
                    //    of rank r's mailbox (all stores in flight together), then polls slot r of the own mailbox
                    bool ok = true;
                    if (lane == 0) ok = spin_until(grid_bar, (t + 1) * gridDim.x, pp.abort, pp.timeout_ns);
                    ok = __shfl_sync(0xFFFFFFFFu, ok ? 1 : 0, 0) != 0;
                    unsigned long long got = kKeyNone;
                    if (ok) {
                        __threadfence();
                        const unsigned long long mine = __ldcg(pp.lkeys + t);
                        if (lane < pp.world) {
                            *reinterpret_cast<volatile unsigned long long *>(&pp.mail[lane]->slot[pp.bank][t][pp.rank]) = mine;
                            ok = spin_filled(&pp.mail[pp.rank]->slot[pp.bank][t][lane], got, pp.abort, pp.timeout_ns);
                        }
                        ok = __all_sync(0xFFFFFFFFu, ok);
                    }
                    if (ok) {
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) {
                            const unsigned long long w = __shfl_xor_sync(0xFFFFFFFFu, got, o);
                            got = w < got ? w : got;
                        }
                        if (lane == 0) {
                            keys[t] = got;
                            __threadfence();
                            atomicExch(pp.release, t + 1);            // 3. local CTAs may read keys[t]
                        }
                    } else if (lane == 0) s_abort = 1;
                } else if (lane == 0) {
                    if (!spin_until(pp.release, t + 1, pp.abort, pp.timeout_ns)) s_abort = 1;
                    __threadfence();
                }
            }
        }
        __syncthreads();
        if (s_abort) return;                                        // a peer vanished: leave, the host reports it
        // the winner becomes the base: every CTA patches its own shared-memory copy
        if (warp == 0) {
            const unsigned long long k = __ldcg(keys + t);
            if (lane == 0) {
                // early stop (same decision in every CTA and on every rank: it only depends on the keys)
                const unsigned long long vc = k >> kIdxBits;
                if (vc < s_red[kWarps + 1]) { s_red[kWarps + 1] = vc; s_red[kWarps + 2] = 0; } else ++s_red[kWarps + 2];
                if (pp.patience && s_red[kWarps + 2] >= pp.patience) s_red[kWarps] = 1;
                if (blockIdx.x == 0 && pp.rounds_run) *pp.rounds_run = t + 1;
                if (blockIdx.x == 0 && pp.carry) { pp.carry[0] = s_red[kWarps + 1]; pp.carry[1] = s_red[kWarps + 2]; }
            }
            if (kDelta && lane == 0) {
                int *s_base = reinterpret_cast<int *>(smem + plan.off_totals) + 544;
                const uint32_t kv = key_violation(k, d.key_obj_bits);
                s_base[2] = (k != kKeyNone && (uint64_t)kv < key_viol_cap(d.key_obj_bits)) ? 1 : 0;
                s_base[0] = (int)kv;
                s_base[1] = (int)key_objective(k, d.key_obj_bits);
            }
            if (k != kKeyNone) {
                PatchSet ps;
                if constexpr (Cfg::kTrans) {
                    // every lane re-materialises the same winner with the per-thread generator; lane 0 parks its rows
                    Gen<W, true, true> tg;        // compact code (row_kth keeps its loop), same candidates
                    tg.bitsT = s_bits; tg.leader = s_leader; tg.cs = s_cs; tg.d = &d; tg.prow = nullptr; tg.lane = 0;
                    tg.D = s_D; tg.DL = s_DL; tg.nD = s_counts[0]; tg.nL = s_counts[1];
                    tg.T = s_sw; tg.tnW = t_words(d.Ppad); tg.t_leaders_valid = s_counts[2] == 0;
                    uint32_t rows[kMaxOps][W];
#pragma unroll
                    for (int i = 0; i < kMaxOps; ++i)
#pragma unroll
                        for (int w = 0; w < W; ++w) rows[i][w] = 0;
                    tg.run(seed, round, (uint32_t)(k & kIdxMask), round_size, ps, rows);
                    if (lane == 0) {
#pragma unroll
                        for (int i = 0; i < kMaxOps; ++i)
#pragma unroll
                            for (int w = 0; w < W; ++w) gen.prow[i * W + w] = rows[i][w];
                    }
                } else {
                    gen.run(seed, round, (uint32_t)(k & kIdxMask), round_size, ps, no_rows);
                }
                __syncwarp();
                if constexpr (Cfg::kTrans) {                        // every lane rewrites its own slots' words
#pragma unroll
                    for (int i = 0; i < kMaxOps; ++i) {
                        if (i < ps.n) {
                            uint32_t newrow[W];
#pragma unroll
                            for (int w = 0; w < W; ++w) newrow[w] = gen.prow[i * W + w];
                            t_patch_row<W>(d, s_sw, s_z, t_words(d.Ppad), ps.p[i], newrow, ps.ld[i], lane);
                        }
                    }
                }
                if (lane == 0) {
#pragma unroll
                    for (int i = 0; i < kMaxOps; ++i) {
                        if (i < ps.n) {
                            if constexpr (Cfg::kTrans) {            // leader validity of the partition, before and after
                                const int lo = s_leader[ps.p[i]], ln = (int)ps.ld[i];
                                const bool was = lo < W * 32 && ((s_bits[(size_t)(lo >> 5) * d.Ppad + ps.p[i]] >> (lo & 31)) & 1u);
                                const bool is = ln < W * 32 && ((gen.prow[i * W + (ln >> 5)] >> (ln & 31)) & 1u);
                                s_counts[2] += (was ? 0 : -1) + (is ? 0 : 1);
                            }
                            for (int w = 0; w < W; ++w) {
                                const uint32_t v = gen.prow[i * W + w];
                                s_bits[(size_t)w * d.Ppad + ps.p[i]] = v;
                                if constexpr (has_oh_plane<Cfg>())
                                    s_bits[(size_t)(W + w) * d.Ppad + ps.p[i]] = oh_word<W>(v, ps.ld[i], w);
                                if (blockIdx.x == 0) d.bitsT[(size_t)w * d.Ppad + ps.p[i]] = v;
                            }
                            s_leader[ps.p[i]] = (uint8_t)ps.ld[i];
                            if (blockIdx.x == 0) d.leader[ps.p[i]] = (uint8_t)ps.ld[i];
                        }
                    }
                }
            }
        }
        __syncthreads();
        rebuild_lists<THREADS>(s_bits, s_leader, d.homeT, d.P, d.Ppad, s_D, s_DL, s_counts, s_scan);
        if (s_red[kWarps]) break;
    }
}

// ------------------------------------------------------------------------------------------
// instantiation lists.  X(W, NPH, kRack, kObj) for every evaluator configuration of a row width:
// rack forms {general, 8-slot, 16-slot, whole-word} x objective encodings {packed entries / dense,
// 3 mask planes} (mask planes: rows of up to 64 slots only).  One counter depth (NPH = 5: per-lane
// column counts up to 255, i.e. every P the engine accepts).
// ------------------------------------------------------------------------------------------
#define KAO_FOR_RACKS(X, W, NPH, O) X(W, NPH, 0, O) X(W, NPH, 3, O) X(W, NPH, 4, O) X(W, NPH, 5, O)
#define KAO_FOR_CFGS_NARROW(X, W, NPH) KAO_FOR_RACKS(X, W, NPH, 0) KAO_FOR_RACKS(X, W, NPH, 3)
#define KAO_FOR_CFGS_WIDE(X, W, NPH) KAO_FOR_RACKS(X, W, NPH, 0)

#define KAO_ROUND_KERNEL(W, NPH, R, O)                                                                      \
    search_round_kernel<EvalCfg<W, NPH, R, O>, threads_for<W>()>(Params, SmemPlan, uint64_t, uint32_t, uint32_t, \
                                                                   uint32_t, uint32_t, unsigned long long *,      \
                                                                   unsigned long long *)
// Column-major kernels: X(sync, pop, threads) for every built schedule (kao_set_schedule); each is
// instantiated for W = 1, 2 and for 32 partition words (compile-time offsets) / any word count.
#define KAO_FOR_SCHEDULES(X) \
    X(4, 0x22, 896) X(1, 0x22, 896) X(4, 0x22, 1024) X(4, 0x22, 768) X(4, 0x12, 896) X(2, 0x22, 896)
#define KAO_SCHEDULE_DEFAULT_SYNC 4
#define KAO_SCHEDULE_DEFAULT_POP 0x22
#define KAO_SCHEDULE_DEFAULT_THREADS 896
#define KAO_PERSISTENT_KERNEL_T(W, NW, S, POP, T)                                                            \
    search_persistent_kernel<EvalCfgT<W, NW, S, POP, T>, T, false>(Params, SmemPlan, uint64_t, uint32_t, uint32_t, \
                                                                    uint32_t, unsigned long long *, unsigned int *, P2P, \
                                                                    unsigned long long *)
#define KAO_PERSISTENT_KERNEL(W, NPH, R, O, T, DELTA)                                                       \
    search_persistent_kernel<EvalCfg<W, NPH, R, O>, T, DELTA>(Params, SmemPlan, uint64_t, uint32_t, uint32_t,      \
                                                             uint32_t, unsigned long long *, unsigned int *, P2P, \
                                                             unsigned long long *)
