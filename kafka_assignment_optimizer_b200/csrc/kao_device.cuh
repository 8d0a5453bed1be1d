// kao_device.cuh — device side of the assignment-search engine (sm_100a).
//
// One warp owns one candidate at a time.  The base assignment (replica bit-plane over rack-aligned
// broker slots, leader slot per partition) and the per-partition weight entries live in shared
// memory for the whole kernel, staged once with TMA bulk copies; a candidate is the base plus up
// to three row patches derived from (seed, round, index) by Philox4x32-10, and is evaluated IN
// FULL: every row's C1/C2/C5/C7 terms and weight, every broker column's replica and leader counts
// (C3/C4, carry-save bit-sliced counters + a cross-lane reduce-scatter), every rack total (C6).
// Model: /root/reference/README.md:139-185; search/generator spec: docs/MODEL.md.
#pragma once
#include <cuda_runtime.h>
#include <type_traits>

#include <stdint.h>

namespace kao {

constexpr int kMaxOps = 3;
// control word of a candidate in a cycle round (docs/MODEL.md 5): three ops (bits 0-1), REPLACE first (bit 2 clear),
// guided (bit 3), op 2 = R-pull (bits 4-5 = 1), op 3 = R-push (bits 7-8 = 0) with close (bit 9)
constexpr uint32_t kCycleSet = 0x21Bu, kCycleClear = 0x4u | 0x20u | 0x80u | 0x100u;
constexpr uint32_t kIdxBits = 24;
constexpr uint32_t kIdxMask = (1u << kIdxBits) - 1;
constexpr int kKeyBits = 63;                // keys < 2^63: same order as signed int64 (NCCL min)
constexpr unsigned long long kKeyNone = 0x7FFFFFFFFFFFFFFFull;
constexpr uint32_t kTag = 0x4B414F21u;
constexpr int kRowsPerLane = 4;            // rows handled per lane per 128-row tile
constexpr int kTileRows = 32 * kRowsPerLane;

// Small read-only tables, one 16-byte-aligned blob (one bulk copy into shared memory).
struct Consts {
    uint32_t bnd_rep[256];       // C3  lo | hi << 16 per slot (padding slots 0|0)
    uint32_t bnd_ldr[256];       // C4
    int32_t rack_lo[32];         // C6
    int32_t rack_hi[32];
    uint8_t slot_of_order[256];  // rack-major order index -> slot
    uint8_t order_of_slot[256];  // slot -> order index, 0xFF for padding slots
};
static_assert(sizeof(Consts) % 16 == 0, "bulk copy size");

struct Params {
    int P, Ppad, B, R, RF, NS, log2S;
    int ppr_lo, ppr_hi;
    int dense;                   // 1: weights come from dense_w (general tables in HBM)
    int nentries;                // packed weight entries per partition in use (0..4)
    int key_obj_bits;            // width of the cost field of a packed key (docs/MODEL.md 3: per problem)
    int nplanes;                 // weighted mask planes in use (0 = objective uses entries / dense)
    int plane_on_leader;         // bit c set: plane c applies to the leader one-hot, else to the row
    int plane_value[6];          // weight of each plane
    uint32_t *bitsT;             // base replica bit-plane, word-major [W][Ppad]
    uint8_t *leader;             // base leader slot [Ppad] (0xFF = none)
    const uint32_t *swT;         // packed weight entries [4][Ppad]: slot | wF << 8 | wL << 20
    const uint32_t *planesT;     // weighted mask planes [nplanes][W][Ppad], or nullptr
    const uint32_t *dense_w;     // [P][NS] wF | wL << 16, or nullptr
    const uint32_t *homeT;       // [Ppad] 4 x u8 home slots (0xFF = none)
    // term planes of the sparse objective (column-major evaluator, kao_device_t.cuh; host: kao_host.hpp)
    int nz;                      // planes in use (0..8)
    int z_on_leader;             // bit j set: plane j counts leaderships (bonus wL - wF), else replicas (wF)
    int z_value[8];              // value of a term of plane j
    uint32_t rf_mask[4];         // bit k of RF spread over a word (all ones / zero): the row pass compares bit-sliced counts with RF
    const uint8_t *zslot;        // [Ppad][8] slot of partition p's term in plane j, 0xFF = none
    uint16_t *D;                 // displaced partitions of the base, ascending
    uint16_t *DL;                // leader-displaced partitions of the base, ascending
    int *nD;                     // [0] = |D|, [1] = |DL|
    const Consts *consts;
};

inline void set_rf_masks(Params &p)
{
    for (int k = 0; k < 4; ++k) p.rf_mask[k] = ((p.RF >> k) & 1) ? 0xFFFFFFFFu : 0u;
}

// ------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------
// Packed key, smaller is better: violation | (objmax - objective) | index.  The cost field is as wide as
// the problem's largest possible objective needs (obj_bits = bit length of P * RF * max weight, fixed
// per problem by the host); the violation field takes what is left of 63 bits (15..38) and saturates.
__host__ __device__ __forceinline__ uint64_t key_viol_cap(int obj_bits)
{
    const int vbits = kKeyBits - (int)kIdxBits - obj_bits;
    return vbits >= 31 ? 0x7FFFFFFFull : ((1ull << vbits) - 1ull);
}
__host__ __device__ __forceinline__ uint64_t pack_key(int viol, int obj, uint32_t idx, int obj_bits)
{
    const uint64_t vcap = key_viol_cap(obj_bits);
    const uint32_t omax = (1u << obj_bits) - 1u;
    const uint64_t v = (uint64_t)(uint32_t)(viol < 0 ? 0 : viol) > vcap ? vcap : (uint64_t)(uint32_t)(viol < 0 ? 0 : viol);
    const uint32_t c = (uint32_t)obj > omax ? 0u : omax - (uint32_t)obj;
    return (v << (kIdxBits + obj_bits)) | ((uint64_t)c << kIdxBits) | (uint64_t)(idx & kIdxMask);
}
__host__ __device__ __forceinline__ uint32_t key_violation(uint64_t k, int obj_bits) { return (uint32_t)(k >> (kIdxBits + obj_bits)); }
__host__ __device__ __forceinline__ uint32_t key_objective(uint64_t k, int obj_bits)
{
    const uint32_t omax = (1u << obj_bits) - 1u;
    return omax - ((uint32_t)(k >> kIdxBits) & omax);
}

__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                              uint32_t k0, uint32_t k1, uint32_t (&o)[4])
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t h0 = __umulhi(0xD2511F53u, c0), l0 = 0xD2511F53u * c0;
        const uint32_t h1 = __umulhi(0xCD9E8D57u, c2), l1 = 0xCD9E8D57u * c2;
        c0 = h1 ^ c1 ^ k0; c1 = l1; c2 = h0 ^ c3 ^ k1; c3 = l0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    o[0] = c0; o[1] = c1; o[2] = c2; o[3] = c3;
}

template <int W> __device__ __forceinline__ uint32_t row_word(const uint32_t (&w)[W], int j)
{
    uint32_t x = w[0];
#pragma unroll
    for (int t = 1; t < W; ++t) x = (j == t) ? w[t] : x;
    return x;
}
template <int W> __device__ __forceinline__ bool row_has(const uint32_t (&w)[W], int s)
{
    return ((s >> 5) < W) && ((row_word<W>(w, s >> 5) >> (s & 31)) & 1u);
}
template <int W> __device__ __forceinline__ void row_flip(uint32_t (&w)[W], int s)
{
    const uint32_t m = 1u << (s & 31);
#pragma unroll
    for (int t = 0; t < W; ++t) w[t] ^= ((s >> 5) == t) ? m : 0u;
}
template <int W> __device__ __forceinline__ int row_count(const uint32_t (&w)[W])
{
    int n = 0;
#pragma unroll
    for (int t = 0; t < W; ++t) n += __popc(w[t]);
    return n;
}
// k-th (0-based) set bit in ascending slot order, -1 if fewer.  kSmall: the bit-clearing loop stays a
// loop.  (Left alone the compiler unrolls it sixteen-fold at every call site: 2,900 of the 8,500
// instructions of a search kernel for a loop that runs 0..7 times.  The column-major kernels use the
// small form; the row-major kernels keep the code that was measured.)
template <int W, bool kSmall = false> __device__ __forceinline__ int row_kth(const uint32_t (&w)[W], int k)
{
    int res = -1;
#pragma unroll
    for (int t = 0; t < W; ++t) {
        const int c = __popc(w[t]);
        if (res < 0 && k < c) {
            uint32_t m = w[t];
            if constexpr (kSmall) {
#pragma unroll 1
                for (int i = 0; i < k; ++i) m &= m - 1;
            } else {
                for (int i = 0; i < k; ++i) m &= m - 1;
            }
            res = t * 32 + __ffs(m) - 1;
        }
        k -= c;
    }
    return res;
}
__device__ __forceinline__ uint32_t mulhi32(uint32_t a, uint32_t n) { return __umulhi(a, n); }

// ------------------------------------------------------------------------------------------
// layout of the transposed planes of the column-major evaluator (kao_device_t.cuh); the per-thread
// generator below scans them too
// ------------------------------------------------------------------------------------------
// physical word of (plane q, slot s, partition word w).  The words of slot s are permuted inside every
// aligned group of 32 by XOR with 4 * (s & 7), so that the 128-bit column loads of a quarter warp (8 consecutive
// slots, same logical chunk) hit 8 different bank groups while the 32-bit row loads of a warp (32 consecutive
// words of one slot) stay conflict-free; a lane finds logical chunk j of its slot at physical chunk j ^ (s & 7)
// with one XOR.  (Fewer than 32 words per slot: not permuted.)
__host__ __device__ __forceinline__ bool t_swizzled(int nW) { return nW >= 32 && (nW & 31) == 0; }
// partition words per slot of the transposed planes and per term plane: Ppad / 32, rounded up to whole groups of
// 32 words once there are more than 32 (the padding words stay empty)
__host__ __device__ __forceinline__ int t_words(int Ppad) { const int n = Ppad >> 5; return n > 32 ? (n + 31) & ~31 : n; }
__host__ __device__ __forceinline__ int t_word(int q, int s, int w, int nW, int NSL)
{
    return (q * NSL + s) * nW + (t_swizzled(nW) ? (w ^ (4 * (s & 7))) : w);
}

// ------------------------------------------------------------------------------------------
// candidate generator (docs/MODEL.md §5): warp-uniform, every lane computes the same patches
// ------------------------------------------------------------------------------------------
struct PatchSet {
    int n;
    int p[kMaxOps];          // patched partition, -1 = unused
    uint32_t ld[kMaxOps];    // its leader slot in the candidate
};

// kThread = false: one warp generates one candidate cooperatively (patched rows go to `prow`);
// kThread = true : every thread generates its own candidate (patched rows go to the caller's registers).
// kSmall: compact code (row_kth), same candidates.
template <int W, bool kThread = false, bool kSmall = false> struct Gen {
    const uint32_t *bitsT;   // base (shared or global)
    const uint8_t *leader;
    const Consts *cs;
    const Params *d;
    uint32_t *prow;          // [kMaxOps * W] warp scratch for patched rows
    int lane;
    const uint16_t *D, *DL;  // displaced / leader-displaced partitions of the base (global or shared)
    int nD, nL;
    // thread mode only, column-major kernels: the transposed planes of the base (kao_device_t.cuh: T0 replicas, T1 leader
    // one-hot, tnW words per slot) — "the first partition from p0 on that holds / is led from / follows on slot s" is a
    // scan for the next set bit of one plane row.  t_leaders_valid: every partition is led from one of its replicas, so
    // that T1 (replica AND leader) also answers "is led from s"; else that question falls back to the scan of the leader bytes
    const uint32_t *T = nullptr;
    int tnW = 0;
    bool t_leaders_valid = false;
    // thread mode only: per-slot inverted lists of the base (ascending partitions), or inv_ok = false
    bool inv_ok = false;
    const int *hoff = nullptr, *loff = nullptr;     // [slots + 1] offsets into hold / led
    const uint16_t *hold = nullptr, *led = nullptr; // partitions holding a replica on / led from the slot

    __device__ __forceinline__ void read_row(int p, uint32_t (&row)[W], uint32_t &ld) const
    {
#pragma unroll
        for (int t = 0; t < W; ++t) row[t] = bitsT[(size_t)t * d->Ppad + p];
        ld = leader[p];
    }
    __device__ __forceinline__ void push(PatchSet &ps, int p, const uint32_t (&row)[W], uint32_t ld,
                                         uint32_t (&rows)[kMaxOps][W]) const
    {
        int slot = ps.n;
#pragma unroll
        for (int i = 0; i < kMaxOps; ++i) if (ps.p[i] == p) slot = i;   // unused entries hold -1
        if (slot == ps.n) ++ps.n;
        // static stores keep ps in registers
#pragma unroll
        for (int i = 0; i < kMaxOps; ++i) if (i == slot) { ps.p[i] = p; ps.ld[i] = ld; }
        if constexpr (kThread) {
#pragma unroll
            for (int i = 0; i < kMaxOps; ++i)
                if (i == slot) {
#pragma unroll
                    for (int t = 0; t < W; ++t) rows[i][t] = row[t];
                }
        } else if (lane == 0) {
#pragma unroll
            for (int t = 0; t < W; ++t) prow[slot * W + t] = row[t];
        }
    }
    // REPLACE on a row held in registers: replica on slot a moves to the first free broker in
    // rack-major order starting at order index o (cyclic); leadership follows the replica.
    __device__ __forceinline__ int replace(uint32_t (&row)[W], uint32_t &ld, int a, int o) const
    {
        const int B = d->B;
        int s = cs->slot_of_order[o];
        for (int tries = 0; tries < B && row_has<W>(row, s); ++tries) {
            o = (o + 1 == B) ? 0 : o + 1;
            s = cs->slot_of_order[o];
        }
        row_flip<W>(row, a);
        row_flip<W>(row, s);
        if ((int)ld == a) ld = (uint32_t)s;
        return s;
    }
    // LEADER: the partition is led from `want` if that is one of its non-leader replicas, else
    // from its k-th (ascending slot) non-leader replica.  Returns the new leader slot or -1.
    __device__ __forceinline__ int pick_leader(const uint32_t (&row)[W], uint32_t &ld, int want, uint32_t rnd) const
    {
        uint32_t m[W];
        const bool has = ((int)ld < W * 32) && row_has<W>(row, (int)ld);
#pragma unroll
        for (int t = 0; t < W; ++t) m[t] = row[t];
        if (has) row_flip<W>(m, (int)ld);
        const int cnt = row_count<W>(m);
        if (cnt < 1) return -1;
        if (want >= 0 && want < W * 32 && want != (int)ld && row_has<W>(row, want)) { ld = (uint32_t)want; return want; }
        ld = (uint32_t)row_kth<W, kSmall>(m, (int)mulhi32(rnd, (uint32_t)cnt));
        return (int)ld;
    }
    // first partition q >= p0 (cyclic), not yet patched, for which pred(q) holds; kind 0: holds a
    // replica on slot src; 1: is led from src; 2: follows (holds, not led) on src
    template <int KIND>
    __device__ __forceinline__ int find_from(const PatchSet &ps, int p0, int src) const
    {
        const int P = d->P;
        if (src < 0 || src >= W * 32) return -1;
        const uint32_t *col = bitsT + (size_t)(src >> 5) * d->Ppad;
        const uint32_t bit = 1u << (src & 31);
        if constexpr (kThread) {
            if (T != nullptr && (KIND != 1 || t_leaders_valid)) {
                // cyclic scan of one row of the transposed planes for the next set bit from p0 on, patched partitions
                // masked out: word (p0 >> 5) from bit (p0 & 31), the following words, and the first word again below p0
                constexpr int NSL = 32 * W;
                const int nWq = (P + 31) >> 5;
                const uint32_t *r0 = T + (size_t)src * tnW, *r1 = T + (size_t)(NSL + src) * tnW;
                const int sw = t_swizzled(tnW) ? 4 * (src & 7) : 0;
                int w = p0 >> 5;
                uint32_t keep = ~0u << (p0 & 31);
                for (int i = 0; i <= nWq; ++i) {
                    const int pw = w ^ sw;
                    uint32_t m = KIND == 1 ? r1[pw] : (KIND == 2 ? (r0[pw] & ~r1[pw]) : r0[pw]);
                    m &= keep;
                    if (i == nWq) m &= ~(~0u << (p0 & 31));
#pragma unroll
                    for (int j = 0; j < kMaxOps; ++j)       // unused patches hold -1: (-1 >> 5) never equals w
                        if ((ps.p[j] >> 5) == w) m &= ~(1u << (ps.p[j] & 31));
                    if (m) return 32 * w + __ffs(m) - 1;
                    keep = ~0u;
                    w = (w + 1 == nWq) ? 0 : w + 1;
                }
                return -1;
            }
            if (inv_ok) {
                // sorted list of the partitions that can match: lower_bound(p0), then walk cyclically
                const uint16_t *L = (KIND == 1) ? led + loff[src] : hold + hoff[src];
                const int n = (KIND == 1) ? loff[src + 1] - loff[src] : hoff[src + 1] - hoff[src];
                int lo = 0, hi = n;
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if ((int)L[mid] < p0) lo = mid + 1; else hi = mid;
                }
                for (int k = 0; k < n; ++k) {
                    int j = lo + k;
                    if (j >= n) j -= n;
                    const int q = L[j];
                    bool t = false;
#pragma unroll
                    for (int i = 0; i < kMaxOps; ++i) t |= (ps.p[i] == q);
                    if (t) continue;
                    if (KIND == 2 && (int)leader[q] == src) continue;
                    return q;
                }
                return -1;
            }
            int q = p0;
            for (int k = 0; k < P; ++k) {
                bool t = false;
#pragma unroll
                for (int i = 0; i < kMaxOps; ++i) t |= (ps.p[i] == q);
                bool hit = false;
                if (KIND == 0) hit = !t && (col[q] & bit);
                if (KIND == 1) hit = !t && ((int)leader[q] == src);
                if (KIND == 2) hit = !t && ((int)leader[q] != src) && (col[q] & bit);
                if (hit) return q;
                q = (q + 1 == P) ? 0 : q + 1;
            }
            return -1;
        }
        for (int k = 0; k < P; k += 32) {
            const int off = k + lane;
            int q = p0 + off;
            if (q >= P) q -= P;
            bool hit = false;
            if (off < P) {
                bool t = false;
#pragma unroll
                for (int i = 0; i < kMaxOps; ++i) t |= (ps.p[i] == q);
                if (KIND == 0) hit = !t && (col[q] & bit);
                if (KIND == 1) hit = !t && ((int)leader[q] == src);
                if (KIND == 2) hit = !t && ((int)leader[q] != src) && (col[q] & bit);
            }
            const uint32_t m = __ballot_sync(0xFFFFFFFFu, hit);
            if (m) {
                int r = p0 + k + (__ffs(m) - 1);
                if (r >= P) r -= P;
                return r;
            }
        }
        return -1;
    }

    // docs/MODEL.md §5 — must stay bit-identical to the restated generator the tests check against
    __device__ void run(uint64_t seed, uint32_t round, uint32_t idx, uint32_t round_size, PatchSet &ps,
                        uint32_t (&rows)[kMaxOps][W]) const
    {
        ps.n = 0;
#pragma unroll
        for (int i = 0; i < kMaxOps; ++i) { ps.p[i] = -1; ps.ld[i] = 0xFF; }
        if (idx + 1 == round_size) return;                       // identity candidate
        const int P = d->P, B = d->B;
        uint32_t r[4], s[4];
        philox4x32_10(idx, round, 0u, kTag, (uint32_t)seed, (uint32_t)(seed >> 32), r);
        // every fourth round (round mod 4 = 3) is a CYCLE round: every candidate is a closed three-step replica cycle — a displaced partition
        // returns to a missing home broker (guided REPLACE), a random partition moves a replica onto the broker that
        // one left (R-pull), and a holder of the now over-full home broker moves to the broker the second one left
        // (R-push, close); bits 11 / 13 ask the later steps to move a replica of the same ROLE (leader / follower) as
        // the step before, which keeps the leader totals of the three brokers as they are
        const bool cycle = (round & 3u) == 3u;
        const uint32_t ctl = cycle ? ((r[0] & ~kCycleClear) | kCycleSet) : r[0];
        const int nops = (ctl & 3u) == 0 ? 1 : ((ctl & 3u) == 3 ? 3 : 2);
        bool moved_leader = false;                               // the last REPLACE moved a leader replica
        const bool first_leader = (ctl >> 2) & 1u, gbit = (ctl >> 3) & 1u;
        uint32_t row[W], ld;
        int lo, hi;
        if (first_leader) {
            const bool guided = gbit && nL > 0;
            const int p = guided ? (int)DL[mulhi32(r[1], (uint32_t)nL)] : (int)mulhi32(r[1], (uint32_t)P);
            read_row(p, row, ld);
            lo = (int)ld;
            int want = -1;
            if (guided) { const int h0 = d->homeT[p] & 0xFF; want = (h0 == 0xFF) ? -1 : h0; }
            hi = pick_leader(row, ld, want, r[2]);
            if (hi < 0) return;
            push(ps, p, row, ld, rows);
        } else {
            const bool guided = gbit && nD > 0;
            const int p = guided ? (int)D[mulhi32(r[1], (uint32_t)nD)] : (int)mulhi32(r[1], (uint32_t)P);
            read_row(p, row, ld);
            const int n = row_count<W>(row);
            if (n == 0) return;
            int a = row_kth<W, kSmall>(row, (int)mulhi32(r[2], (uint32_t)n));
            int o = (int)mulhi32(r[3], (uint32_t)B);
            if (guided) {
                const uint32_t h4 = d->homeT[p];
                uint32_t home[W], miss[W], nonhome[W];
#pragma unroll
                for (int t = 0; t < W; ++t) home[t] = 0;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int hs = (h4 >> (8 * i)) & 0xFF;
                    if (hs != 0xFF && !row_has<W>(home, hs)) row_flip<W>(home, hs);
                }
#pragma unroll
                for (int t = 0; t < W; ++t) { miss[t] = home[t] & ~row[t]; nonhome[t] = row[t] & ~home[t]; }
                const int nm = row_count<W>(miss), nn = row_count<W>(nonhome);
                if (nm > 0) {
                    o = cs->order_of_slot[row_kth<W, kSmall>(miss, (int)mulhi32(r[3], (uint32_t)nm))];
                    if (nn > 0) a = row_kth<W, kSmall>(nonhome, (int)mulhi32(r[2], (uint32_t)nn));
                }
            }
            moved_leader = (int)ld == a;
            hi = replace(row, ld, a, o);
            lo = a;
            push(ps, p, row, ld, rows);
        }
        if (nops == 1) return;
        philox4x32_10(idx, round, 1u, kTag, (uint32_t)seed, (uint32_t)(seed >> 32), s);
        for (int k = 1; k < nops; ++k) {
            const uint32_t link = (ctl >> (4 + 3 * (k - 1))) & 3u;
            const bool close = (ctl >> (6 + 3 * (k - 1))) & 1u;
            const uint32_t ra = (k == 1) ? s[0] : s[2], rb = (k == 1) ? s[1] : s[3];
            const int start = (int)mulhi32(ra, (uint32_t)P);
            int olo = (lo >= 0 && lo < 256) ? (int)cs->order_of_slot[lo] : 0xFF;
            if (olo >= B) olo = 0;
            uint32_t rq[W], lq;
            const bool match = cycle && ((ctl >> (11 + 2 * (k - 1))) & 1u);
            if (link == 0) {                                   // R-push
                const int q = !match ? find_from<0>(ps, start, hi) : (moved_leader ? find_from<1>(ps, start, hi) : find_from<2>(ps, start, hi));
                if (q < 0) return;
                read_row(q, rq, lq);
                if (!row_has<W>(rq, hi)) return;               // led from hi without a replica there (malformed base)
                moved_leader = (int)lq == hi;
                hi = replace(rq, lq, hi, close ? olo : (int)mulhi32(rb, (uint32_t)B));
                push(ps, q, rq, lq, rows);
            } else if (link == 1) {                            // R-pull
                const int q = start;
                bool t = false;
#pragma unroll
                for (int i = 0; i < kMaxOps; ++i) t |= (ps.p[i] == q);
                if (t) return;
                read_row(q, rq, lq);
                const int nq = row_count<W>(rq);
                if (nq == 0) return;
                int src = row_kth<W, kSmall>(rq, (int)mulhi32(rb, (uint32_t)nq));
                const bool led = (int)lq < W * 32 && row_has<W>(rq, (int)lq);
                if (close && led) src = (int)lq;
                if (match && led) {                            // same role as the replica that left `lo`
                    if (moved_leader) src = (int)lq;
                    else if (nq > 1) {
                        uint32_t fol[W];
#pragma unroll
                        for (int t = 0; t < W; ++t) fol[t] = rq[t];
                        row_flip<W>(fol, (int)lq);
                        src = row_kth<W, kSmall>(fol, (int)mulhi32(rb, (uint32_t)(nq - 1)));
                    }
                }
                moved_leader = (int)lq == src;
                replace(rq, lq, src, olo);
                lo = src;
                push(ps, q, rq, lq, rows);
            } else if (link == 2) {                            // L-push
                const int q = find_from<1>(ps, start, hi);
                if (q < 0) return;
                read_row(q, rq, lq);
                int want = lo;
                if (!close) { const int h0 = d->homeT[q] & 0xFF; want = (h0 == 0xFF) ? -1 : h0; }
                const int t = pick_leader(rq, lq, want, rb);
                if (t < 0) return;
                hi = t;
                push(ps, q, rq, lq, rows);
            } else {                                           // L-pull
                const int q = find_from<2>(ps, start, lo);
                if (q < 0) return;
                read_row(q, rq, lq);
                const int old = (int)lq;
                if (pick_leader(rq, lq, lo, rb) < 0) return;
                lo = old;
                push(ps, q, rq, lq, rows);
            }
        }
    }
};

// ------------------------------------------------------------------------------------------
// full evaluation of one candidate by one warp (docs/MODEL.md §3)
// ------------------------------------------------------------------------------------------
// One three-input logic instruction (LOP3.LUT): the truth table is the byte kLut with a = 0xF0, b = 0xCC,
// c = 0xAA (e.g. majority 0xE8, a ^ b ^ c 0x96, a | b | c 0xFE, (a & b) | c 0xEA).  Spelled out because the
// compiler does not always fuse a three-input expression into one instruction.
template <int kLut> __device__ __forceinline__ uint32_t lop3(uint32_t a, uint32_t b, uint32_t c)
{
#if defined(KAO_HOST_EMU)
    uint32_t r = 0;
    if (kLut & 0x80) r |= a & b & c;
    if (kLut & 0x40) r |= a & b & ~c;
    if (kLut & 0x20) r |= a & ~b & c;
    if (kLut & 0x10) r |= a & ~b & ~c;
    if (kLut & 0x08) r |= ~a & b & c;
    if (kLut & 0x04) r |= ~a & b & ~c;
    if (kLut & 0x02) r |= ~a & ~b & c;
    if (kLut & 0x01) r |= ~a & ~b & ~c;
    return r;
#else
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, %4;" : "=r"(r) : "r"(a), "r"(b), "r"(c), "n"(kLut));
    return r;
#endif
}

// Carry-save adder: (h, l) = a + b + c  bitwise; two LOP3.
__device__ __forceinline__ void csa(uint32_t &h, uint32_t &l, uint32_t a, uint32_t b, uint32_t c)
{
    const uint32_t u = a ^ b;
    h = (a & b) | (u & c);
    l = u ^ c;
}

// Bit-sliced per-lane column counter: planes 1,2,4 + NPH high planes (8,16,...).  Rows are pushed
// four at a time (one 128-row tile): three carry-save adders fold them with the ones/twos planes
// into one weight-4 word that ripples up the higher planes (~3.5 LOP3 per pushed word).
template <int W, int NPH> struct ColCounter {
    uint32_t ones[W], twos[W], fours[W], hi[NPH][W];
    __device__ __forceinline__ void clear()
    {
#pragma unroll
        for (int t = 0; t < W; ++t) {
            ones[t] = twos[t] = fours[t] = 0;
#pragma unroll
            for (int k = 0; k < NPH; ++k) hi[k][t] = 0;
        }
    }
    // Eight rows (two tiles) form one block of seven carry-save adders with a single ripple from
    // the eights plane; the first tile parks its weight-4 word in `fa` (no row has to stay live).
    uint32_t fa[W];
    template <bool kSecond>
    __device__ __forceinline__ void push_half(const uint32_t (&x)[kRowsPerLane][W])
    {
#pragma unroll
        for (int t = 0; t < W; ++t) {
            uint32_t a2, b2, q4;
            csa(a2, ones[t], ones[t], x[0][t], x[1][t]);
            csa(b2, ones[t], ones[t], x[2][t], x[3][t]);
            csa(q4, twos[t], twos[t], a2, b2);
            if constexpr (!kSecond) {
                fa[t] = q4;
            } else {
                uint32_t cy;
                csa(cy, fours[t], fours[t], fa[t], q4);
#pragma unroll
                for (int k = 0; k < NPH; ++k) {
                    const uint32_t n = hi[k][t] & cy;
                    hi[k][t] ^= cy;
                    cy = n;
                }
            }
        }
    }
    __device__ __forceinline__ void push4(const uint32_t (&x0)[W], const uint32_t (&x1)[W],
                                          const uint32_t (&x2)[W], const uint32_t (&x3)[W])
    {
#pragma unroll
        for (int t = 0; t < W; ++t) {
            uint32_t a2, b2, c4;
            csa(a2, ones[t], ones[t], x0[t], x1[t]);
            csa(b2, ones[t], ones[t], x2[t], x3[t]);
            csa(c4, twos[t], twos[t], a2, b2);
            uint32_t cy = fours[t] & c4;
            fours[t] ^= c4;
#pragma unroll
            for (int k = 0; k < NPH; ++k) {
                const uint32_t n = hi[k][t] & cy;
                hi[k][t] ^= cy;
                cy = n;
            }
        }
    }
};

__device__ __forceinline__ uint32_t bytecounts(uint32_t x)
{
    uint32_t c = x - ((x >> 1) & 0x55555555u);
    c = (c & 0x33333333u) + ((c >> 2) & 0x33333333u);
    return (c + (c >> 4)) & 0x0F0F0F0Fu;
}

// Base address of a table, resolved once per candidate: a 32-bit shared-memory address for the
// search kernel (no generic->shared conversion per load), a global pointer for explicit populations.
#if defined(KAO_HOST_EMU)
// tests/emu compiles these device functions for the host (a warp = 32 lock-stepped fibers): there
// "shared memory" is plain memory and the PTX loads below become ordinary loads.
template <bool kShared> struct MemRef {
    const char *ga;
    explicit MemRef(const void *p) : ga(static_cast<const char *>(p)) {}
    uint4 ld128(uint32_t byte_off) const { return *reinterpret_cast<const uint4 *>(ga + byte_off); }
    uint32_t ld32(uint32_t byte_off) const { return *reinterpret_cast<const uint32_t *>(ga + byte_off); }
};
#else
template <bool kShared> struct MemRef {
    uint32_t sa;
    const char *ga;
    __device__ __forceinline__ explicit MemRef(const void *p)
    {
        if constexpr (kShared) { sa = (uint32_t)__cvta_generic_to_shared(p); ga = nullptr; }
        else { sa = 0; ga = static_cast<const char *>(p); }
    }
    __device__ __forceinline__ uint4 ld128(uint32_t byte_off) const
    {
        if constexpr (kShared) {
            uint4 v;
            asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(sa + byte_off));
            return v;
        } else {
            return __ldg(reinterpret_cast<const uint4 *>(ga + byte_off));
        }
    }
    __device__ __forceinline__ uint32_t ld32(uint32_t byte_off) const
    {
        if constexpr (kShared) {
            uint32_t v;
            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(sa + byte_off));
            return v;
        } else {
            return __ldg(reinterpret_cast<const uint32_t *>(ga + byte_off));
        }
    }
};
#endif

__device__ __forceinline__ uint32_t comp(const uint4 &v, int i)
{
    return i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w;
}

// ------------------------------------------------------------------------------------------
// per-row terms.  Two compile-time variants of the rack part:
//   kHi1 (ppr_lo == 0, ppr_hi == 1, the common "replicas of a partition sit in distinct racks"):
//        excess = popc(row) - #non-empty rack fields, with the classic non-zero-field mask;
//   general bounds: SWAR field counts and saturating field-wise subtraction.
// The slot layout makes a rack an aligned field of S = 8 / 16 slots or 1..8 whole words.
// ------------------------------------------------------------------------------------------
// kRack: 0 = general bounds, field width read at run time; 3 / 4 / 5 = the kHi1 form with 8-slot,
// 16-slot or whole-word rack fields fixed at compile time (no per-row dispatch on the layout).
template <int W, int kRack>
__device__ __forceinline__ int row_rack_terms(const uint32_t (&x)[W], int log2S_rt, int R, int lo, int hi, int RF)
{
    constexpr bool kHi1 = kRack != 0;
    const int log2S = (kRack == 3 || kRack == 4) ? kRack : log2S_rt;
    int n = 0, pen = 0;
    if (kRack != 5 && log2S == 3) {
#pragma unroll
        for (int t = 0; t < W; ++t) {
            const int pc = __popc(x[t]);
            n += pc;
            if constexpr (kHi1) {
                const uint32_t nz = (((x[t] & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x[t]) & 0x80808080u;
                pen += pc - __popc(nz);
            } else {
                const uint32_t c = bytecounts(x[t]);
                const uint32_t dd = (c | 0x80808080u) - (uint32_t)hi * 0x01010101u;
                const uint32_t m = ((dd >> 7) & 0x01010101u) * 0xFFu;
                pen += (int)(((dd & m & 0x7F7F7F7Fu) * 0x01010101u) >> 24);
                if (lo > 0) {
                    const int nv = min(max(R - 4 * t, 0), 4);
                    const uint32_t vm = nv >= 4 ? 0xFFFFFFFFu : ((1u << (8 * nv)) - 1u);
                    const uint32_t d2 = (((uint32_t)lo * 0x01010101u) | 0x80808080u) - c;
                    const uint32_t m2 = ((d2 >> 7) & 0x01010101u) * 0xFFu;
                    pen += (int)(((d2 & m2 & 0x7F7F7F7Fu & vm) * 0x01010101u) >> 24);
                }
            }
        }
    } else if (kRack != 5 && log2S == 4) {
#pragma unroll
        for (int t = 0; t < W; ++t) {
            const int pc = __popc(x[t]);
            n += pc;
            if constexpr (kHi1) {
                const uint32_t nz = (((x[t] & 0x7FFF7FFFu) + 0x7FFF7FFFu) | x[t]) & 0x80008000u;
                pen += pc - __popc(nz);
            } else {
                uint32_t c = bytecounts(x[t]);
                c = (c + (c >> 8)) & 0x00FF00FFu;
                const uint32_t dd = (c | 0x80008000u) - (uint32_t)hi * 0x00010001u;
                const uint32_t m = ((dd >> 15) & 0x00010001u) * 0xFFFFu;
                pen += (int)(((dd & m & 0x7FFF7FFFu) * 0x00010001u) >> 16);
                if (lo > 0) {
                    const int nv = min(max(R - 2 * t, 0), 2);
                    const uint32_t vm = nv >= 2 ? 0xFFFFFFFFu : (nv == 1 ? 0xFFFFu : 0u);
                    const uint32_t d2 = (((uint32_t)lo * 0x00010001u) | 0x80008000u) - c;
                    const uint32_t m2 = ((d2 >> 15) & 0x00010001u) * 0xFFFFu;
                    pen += (int)(((d2 & m2 & 0x7FFF7FFFu & vm) * 0x00010001u) >> 16);
                }
            }
        }
    } else {
        const int lw = (log2S_rt > 5 ? log2S_rt : 5) - 5;     // log2(words per rack); this branch is dead for kRack 3 / 4
        const int wpr = 1 << lw;
        int c = 0;
#pragma unroll
        for (int t = 0; t < W; ++t) {
            const int pc = __popc(x[t]);
            n += pc;
            c += pc;
            if (((t + 1) & (wpr - 1)) == 0) {
                if ((t >> lw) < R) pen += max(c - hi, 0) + max(lo - c, 0);
                c = 0;
            }
        }
    }
    return abs(n - RF) + pen;
}

constexpr int kPlanes = 13;                 // 8 per-lane planes + 5 butterfly steps: counts < 8192

template <int W, int NPH>
__device__ __forceinline__ void load_planes(uint32_t (&pl)[kPlanes], const ColCounter<W, NPH> &c, int t)
{
    pl[0] = c.ones[t]; pl[1] = c.twos[t]; pl[2] = c.fours[t];
#pragma unroll
    for (int k = 0; k < NPH; ++k) pl[3 + k] = c.hi[k][t];
#pragma unroll
    for (int k = 3 + NPH; k < kPlanes; ++k) pl[k] = 0;
}

// C3 / C4 / C6: broker columns.  pl[i] = bit-sliced per-lane counts of NI 32-column items (items
// < nA are replica words checked against bndA, the others leader words checked against bndB).
// Reduce-scatter over lanes: log2(NI) halving steps (a lane keeps half of its items and adds the
// partner's copy of them), then plain butterfly steps; every lane ends with ONE item summed over
// all 32 lanes and checks NI of its 32 columns against the bounds.  A lane's NI columns lie in
// one rack (NI <= S), so the rack totals of C6 are a segmented warp sum of the replica columns.
// Returns this lane's share of the violation.
template <int NI, int NP0>
__device__ __forceinline__ int column_violation(uint32_t (&pl)[NI][kPlanes], int lane, int nA,
                                                const uint32_t *bndA, const uint32_t *bndB,
                                                bool racks, int lead_mode, int log2S, int R, const Consts *cs)
{
    static_assert(NP0 + 5 <= kPlanes, "plane budget");
    int item = 0;
#pragma unroll
    for (int step = 0; step < 5; ++step) {
        const int mask = 1 << step;
        const bool up = (lane >> step) & 1;
        const int np = NP0 + step;                        // planes held before this step
        if ((NI >> step) >= 2) {
            const int half = NI >> (step + 1);
            item += up ? half : 0;
#pragma unroll
            for (int i = 0; i < half; ++i) {
                uint32_t carry = 0;
#pragma unroll
                for (int k = 0; k < np; ++k) {
                    const uint32_t a = pl[i][k], b = pl[i + half][k];
                    const uint32_t keep = up ? b : a, send = up ? a : b;
                    const uint32_t rcv = __shfl_xor_sync(0xFFFFFFFFu, send, mask);
                    uint32_t h, l;
                    csa(h, l, keep, rcv, carry);
                    pl[i][k] = l;
                    carry = h;
                }
                pl[i][np] = carry;
            }
        } else {
            uint32_t carry = 0;
#pragma unroll
            for (int k = 0; k < np; ++k) {
                const uint32_t rcv = __shfl_xor_sync(0xFFFFFFFFu, pl[0][k], mask);
                uint32_t h, l;
                csa(h, l, pl[0][k], rcv, carry);
                pl[0][k] = l;
                carry = h;
            }
            pl[0][np] = carry;
        }
    }
    constexpr int nsplit = (NI == 1) ? 0 : (NI == 2) ? 1 : (NI == 4) ? 2 : (NI == 8) ? 3 : 4;
    constexpr int NPF = NP0 + 5;
    const int t0 = (lane >> nsplit) * NI;                 // first of this lane's NI columns
    const bool second = item >= nA;
    const int word = second ? item - nA : item;
    const uint32_t *bnd = second ? bndB : bndA;
    uint32_t sh[NPF];
#pragma unroll
    for (int k = 0; k < NPF; ++k) sh[k] = pl[0][k] >> t0;
    int viol = 0, csum = 0;
#pragma unroll
    for (int i = 0; i < NI; ++i) {
        uint32_t c = 0;
#pragma unroll
        for (int k = 0; k < NPF; ++k) c |= ((sh[k] >> i) & 1u) << k;
        const uint32_t b = bnd[word * 32 + t0 + i];
        const int lo = (int)(b & 0xFFFFu), hi = (int)(b >> 16);
        viol += max((int)c - hi, 0) + max(lo - (int)c, 0);
        csum += (int)c;
    }
    // C2/C5: a partition whose leader slot is one of its replicas shows up exactly once in the
    // leader columns, so (#partitions - sum of leader counts) is the number of invalid leaders; the
    // caller adds P once.  lead_mode 1: items >= nA are leader words, 2: all items are.
    if (lead_mode == 2 || (lead_mode == 1 && second)) viol -= csum;
    if (racks) {
        // C6: replica columns summed per rack; leader items and padding racks form ignored groups
        const int rk = (word * 32 + t0) >> log2S;
        const int grp = (second || rk >= R) ? 0x7FFF : rk;
        const uint32_t peers = __match_any_sync(0xFFFFFFFFu, grp);
        const int tot = __reduce_add_sync(peers, csum);
        if (grp != 0x7FFF && (__ffs(peers) - 1) == lane)
            viol += max(tot - cs->rack_hi[rk], 0) + max(cs->rack_lo[rk] - tot, 0);
    }
    return viol;
}

// Objective, three encodings of the weight tables (host picks, docs/MODEL.md §3.2):
//   kObjPlanes  up to kMaxWPlanes "weighted mask planes": objective = sum_c v_c * popc(part_c & M_c[p]),
//               part = the row (follower-weight classes) or the leader one-hot (leader bonus classes)
//   kObjEntries up to 4 packed (slot, wF, wL) entries per partition
//   dense       (inside kObjEntries, runtime flag) general [P][slots] table in HBM
constexpr int kObjEntries = 0;   // kObj > 0: that many weighted mask planes (3 or 6, zero-padded):
                                 // the first 2*kObj/3 apply to the row, the last kObj/3 to the leader one-hot
constexpr int kMaxWPlanes = 6;

template <int W_, int NPH_, int kRack_, int kObj_> struct EvalCfg {
    static constexpr int W = W_, NPH = NPH_, kObj = kObj_, kRack = kRack_;
    static constexpr bool kTrans = false;      // true: column-major evaluator, kao_device_t.cuh
};
// The search kernels keep a leader one-hot plane [W][Ppad] right behind the shared-memory bit-plane
// for narrow rows scored with mask planes (the leader bytes are then not read by the evaluator).
template <class Cfg> __host__ __device__ constexpr bool has_oh_plane() { return Cfg::W <= 2 && Cfg::kObj > 0 && !Cfg::kTrans; }


// Loads one 128-row tile of the candidate: 4 consecutive rows per lane (128-bit shared-memory
// loads, conflict-free), with the candidate's row patches substituted (rare, warp-uniform test).
// kOh: the base's leader one-hot plane (row & 1 << leader, kept next to the bit-plane by the search
// kernels) is loaded instead of the leader bytes; a patched row's one-hot is rebuilt here.
template <int W, bool kShared, bool kOh>
__device__ __forceinline__ void load_tile(const MemRef<kShared> &bitsT, const MemRef<kShared> &leader, int Ppad,
                                          const PatchSet &ps, const uint32_t *prow, int lane, int u,
                                          uint4 (&xv)[W], uint4 (&ohv)[W], uint32_t &ld4)
{
    const int r0 = u * kTileRows + lane * kRowsPerLane;
#pragma unroll
    for (int t = 0; t < W; ++t) xv[t] = bitsT.ld128((uint32_t)(t * Ppad + r0) * 4u);
    if constexpr (kOh) {
#pragma unroll
        for (int t = 0; t < W; ++t) ohv[t] = bitsT.ld128((uint32_t)((W + t) * Ppad + r0) * 4u);
        ld4 = 0;
    } else {
        ld4 = leader.ld32((uint32_t)r0);
    }
    if (((ps.p[0] >> 7) == u) | ((ps.p[1] >> 7) == u) | ((ps.p[2] >> 7) == u)) {
#pragma unroll
        for (int i = 0; i < kMaxOps; ++i) {
            const int pp = ps.p[i];                       // -1 when unused: never matches a tile
            if ((pp >> 7) == u && ((pp & 127) >> 2) == lane) {
                const int rr = pp & 3;
#pragma unroll
                for (int t = 0; t < W; ++t) {
                    const uint32_t v = prow[i * W + t];
                    if (rr == 0) xv[t].x = v; else if (rr == 1) xv[t].y = v;
                    else if (rr == 2) xv[t].z = v; else xv[t].w = v;
                    if constexpr (kOh) {
                        const uint32_t o = ((int)(ps.ld[i] >> 5) == t) ? (v & (1u << (ps.ld[i] & 31u))) : 0u;
                        if (rr == 0) ohv[t].x = o; else if (rr == 1) ohv[t].y = o;
                        else if (rr == 2) ohv[t].z = o; else ohv[t].w = o;
                    }
                }
                if constexpr (!kOh) ld4 = (ld4 & ~(0xFFu << (8 * rr))) | (ps.ld[i] << (8 * rr));
            }
        }
    }
}

// Per tile, two parts over the same loaded rows:
//   part A  per row: C1 / C7 terms, leader validity (C2/C5), leader-bonus planes; per tile: the
//           carry-save column counters of replicas (C3, C6) and leaders (C4)
//   part B  per row: the follower-weight part of the objective
template <class Cfg, bool kShared, bool kCheckValid, bool kOh, bool kObjShared = kShared>
__device__ __forceinline__ void tile_pass_a(const Params &d, const MemRef<kObjShared> &objT,
                                            int lane, int u, int &viol, int &obj,
                                            const uint4 (&xv)[Cfg::W], const uint4 (&ohv)[Cfg::W], uint32_t ld4,
                                            uint32_t (&x)[kRowsPerLane][Cfg::W], uint32_t (&oh)[kRowsPerLane][Cfg::W])
{
    constexpr int W = Cfg::W;
    const int r0 = u * kTileRows + lane * kRowsPerLane;
#pragma unroll
    for (int i = 0; i < kRowsPerLane; ++i) {
#pragma unroll
        for (int t = 0; t < W; ++t) x[i][t] = comp(xv[t], i);
        const uint32_t ld = __byte_perm(ld4, 0u, 0x4440u + i);   // byte i of the four leader slots
        // leader one-hot restricted to the row (empty when the leader slot is not a replica: that
        // partition is then missing from the leader columns, which is how C2/C5 are charged)
        if constexpr (kOh) {
#pragma unroll
            for (int t = 0; t < W; ++t) oh[i][t] = comp(ohv[t], i);
        } else if constexpr (W == 2) {
            unsigned long long ob;                               // 1 << ld; PTX shl clamps: ld >= 64 gives 0
#if defined(KAO_HOST_EMU)
            ob = ld >= 64u ? 0ull : 1ull << ld;
#else
            asm("shl.b64 %0, %1, %2;" : "=l"(ob) : "l"(1ull), "r"(ld));
#endif
            oh[i][0] = x[i][0] & (uint32_t)ob;
            oh[i][1] = x[i][1] & (uint32_t)(ob >> 32);
        } else {
            const uint32_t ldbit = __funnelshift_l(0u, 1u, ld);  // 1 << (ld & 31)
#pragma unroll
            for (int t = 0; t < W; ++t) {
                const uint32_t lm = ((int)(ld >> 5) == t) ? ldbit : 0u;  // mask first: no indexed row access
                oh[i][t] = x[i][t] & lm;
            }
        }
        int rv = row_rack_terms<W, Cfg::kRack>(x[i], d.log2S, d.R, d.ppr_lo, d.ppr_hi, d.RF);
        if constexpr (kCheckValid) rv = ((r0 + i) < d.P) ? rv : 0;
        viol += rv;
    }
    if constexpr (Cfg::kObj > 0) {
        // leader-bonus planes: the one-hot has at most one bit, so "any overlap" replaces a popcount
#pragma unroll
        for (int c = 2 * Cfg::kObj / 3; c < Cfg::kObj; ++c) {
            uint4 m[W];
#pragma unroll
            for (int t = 0; t < W; ++t) m[t] = objT.ld128((uint32_t)((c * W + t) * d.Ppad + r0) * 4u);
            int cnt = 0;
#pragma unroll
            for (int i = 0; i < kRowsPerLane; ++i) {
                uint32_t hit = 0;
#pragma unroll
                for (int t = 0; t < W; ++t) hit |= oh[i][t] & comp(m[t], i);
                cnt += hit ? 1 : 0;
            }
            obj += cnt * d.plane_value[c];
        }
    }
}
template <class Cfg, bool kShared, bool kCheckValid, bool kObjShared = kShared>
__device__ __forceinline__ void tile_pass_b(const Params &d, const MemRef<kObjShared> &objT,
                                            int lane, int u, int &obj,
                                            const uint4 (&xv)[Cfg::W], uint32_t ld4)
{
    constexpr int W = Cfg::W;
    const int r0 = u * kTileRows + lane * kRowsPerLane;
    if constexpr (Cfg::kObj > 0) {
#pragma unroll
        for (int c = 0; c < 2 * Cfg::kObj / 3; ++c) {
            {
                int cnt = 0;
#pragma unroll
                for (int t = 0; t < W; ++t) {
                    const uint4 m = objT.ld128((uint32_t)((c * W + t) * d.Ppad + r0) * 4u);
#pragma unroll
                    for (int i = 0; i < kRowsPerLane; ++i) cnt += __popc(comp(xv[t], i) & comp(m, i));
                }
                obj += cnt * d.plane_value[c];
            }
        }
    } else {
        uint4 ov[4];
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (k < d.nentries) ov[k] = objT.ld128((uint32_t)(k * d.Ppad + r0) * 4u);
#pragma unroll
        for (int i = 0; i < kRowsPerLane; ++i) {
            uint32_t x[W];
#pragma unroll
            for (int t = 0; t < W; ++t) x[t] = comp(xv[t], i);
            const uint32_t ld = (ld4 >> (8 * i)) & 0xFFu;
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (k < d.nentries) {
                    const uint32_t e = comp(ov[k], i);
                    const uint32_t slot = e & 0xFFu;
                    const uint32_t xw = row_word<W>(x, (int)(slot >> 5));
                    const bool bit = __funnelshift_r(xw, 0u, slot) & 1u;
                    const uint32_t w = (slot == ld) ? (e >> 20) : ((e >> 8) & 0xFFFu);
                    obj += bit ? (int)w : 0;
                }
            if (d.dense && (!kCheckValid || (r0 + i) < d.P)) {
                const uint32_t *wrow = d.dense_w + (size_t)(r0 + i) * d.NS;
#pragma unroll
                for (int t = 0; t < W; ++t) {
                    for (uint32_t m = x[t]; m; m &= m - 1) {
                        const int s = t * 32 + __ffs(m) - 1;
                        if (s < d.NS) {
                            const uint32_t w = __ldg(wrow + s);
                            obj += (s == (int)ld) ? (int)(w >> 16) : (int)(w & 0xFFFFu);
                        }
                    }
                }
            }
        }
    }
}

// Two tiles (8 rows per lane) = one carry-save block.  Ppad is a multiple of 256, so the second
// tile of the last pair exists in memory even when it holds no real row.
template <class Cfg, bool kShared, bool kChk, bool kOh, bool kObjShared = kShared>
__device__ __forceinline__ void eval_pair(const Params &d, const MemRef<kShared> &m_bits,
                                          const MemRef<kShared> &m_leader, const MemRef<kObjShared> &m_obj,
                                          const PatchSet &ps, const uint32_t *prow, int lane, int u,
                                          ColCounter<Cfg::W, Cfg::NPH> &rc, ColCounter<Cfg::W, Cfg::NPH> &lc,
                                          int &viol, int &obj)
{
    constexpr int W = Cfg::W;
    {
        uint4 xv[W], ohv[W];
        uint32_t ld4, x[kRowsPerLane][W], oh[kRowsPerLane][W];
        load_tile<W, kShared, kOh>(m_bits, m_leader, d.Ppad, ps, prow, lane, u, xv, ohv, ld4);
        tile_pass_a<Cfg, kShared, kChk, kOh, kObjShared>(d, m_obj, lane, u, viol, obj, xv, ohv, ld4, x, oh);
        tile_pass_b<Cfg, kShared, kChk, kObjShared>(d, m_obj, lane, u, obj, xv, ld4);
        rc.template push_half<false>(x);
        lc.template push_half<false>(oh);
    }
    {
        uint4 xv[W], ohv[W];
        uint32_t ld4, x[kRowsPerLane][W], oh[kRowsPerLane][W];
        load_tile<W, kShared, kOh>(m_bits, m_leader, d.Ppad, ps, prow, lane, u + 1, xv, ohv, ld4);
        tile_pass_a<Cfg, kShared, kChk, kOh, kObjShared>(d, m_obj, lane, u + 1, viol, obj, xv, ohv, ld4, x, oh);
        tile_pass_b<Cfg, kShared, kChk, kObjShared>(d, m_obj, lane, u + 1, obj, xv, ld4);
        rc.template push_half<true>(x);
        lc.template push_half<true>(oh);
    }
}

template <class Cfg, bool kShared, bool kChk, bool kObjShared = kShared>
__device__ __forceinline__ void eval_single(const Params &d, const MemRef<kShared> &m_bits,
                                            const MemRef<kShared> &m_leader, const MemRef<kObjShared> &m_obj,
                                            const PatchSet &ps, const uint32_t *prow, int lane, int u,
                                            ColCounter<Cfg::W, Cfg::NPH> &rc, ColCounter<Cfg::W, Cfg::NPH> &lc,
                                            int &viol, int &obj)
{
    constexpr int W = Cfg::W;
    uint4 xv[W], ohv[W];
    uint32_t ld4, x[kRowsPerLane][W], oh[kRowsPerLane][W];
    load_tile<W, kShared, false>(m_bits, m_leader, d.Ppad, ps, prow, lane, u, xv, ohv, ld4);
    tile_pass_a<Cfg, kShared, kChk, false, kObjShared>(d, m_obj, lane, u, viol, obj, xv, ohv, ld4, x, oh);
    tile_pass_b<Cfg, kShared, kChk, kObjShared>(d, m_obj, lane, u, obj, xv, ld4);
    rc.push4(x[0], x[1], x[2], x[3]);
    lc.push4(oh[0], oh[1], oh[2], oh[3]);
}

// Evaluates candidate = base + patches.  kShared: the base is in shared memory; kObjShared: the objective
// table is (wide-row delta kernels keep it in HBM / L2: it is only read for the base's own evaluation).
// Outputs (same value in every lane): total violation amount and objective.
template <class Cfg, bool kShared, bool kObjShared = kShared>
__device__ void eval_candidate(const Params &d, const uint32_t *bitsT, const uint8_t *leader,
                               const uint32_t *objT, const Consts *cs, const PatchSet &ps,
                               const uint32_t *prow, int lane, int &viol_out, int &obj_out)
{
    constexpr int W = Cfg::W, NPH = Cfg::NPH;
    constexpr bool kOh = kShared && has_oh_plane<Cfg>();
    const MemRef<kShared> m_bits(bitsT), m_leader(leader);
    const MemRef<kObjShared> m_obj(objT);
    int viol = 0, obj = 0;
    const int ntiles = (d.P + kTileRows - 1) / kTileRows;
    const int nfull = d.P / kTileRows;                   // tiles made of real rows only
    ColCounter<W, NPH> rc, lc;
    rc.clear();
    lc.clear();
    if constexpr (W <= 2) {
        int u = 0;
#pragma unroll 1
        for (; u + 2 <= nfull; u += 2)
            eval_pair<Cfg, kShared, false, kOh, kObjShared>(d, m_bits, m_leader, m_obj, ps, prow, lane, u, rc, lc, viol, obj);
#pragma unroll 1
        for (; u < ntiles; u += 2)
            eval_pair<Cfg, kShared, true, kOh, kObjShared>(d, m_bits, m_leader, m_obj, ps, prow, lane, u, rc, lc, viol, obj);
    } else {
        // wide rows: one tile per iteration (the two-tile block would not fit the register file)
        int u = 0;
#pragma unroll 1
        for (; u < nfull; ++u)
            eval_single<Cfg, kShared, false, kObjShared>(d, m_bits, m_leader, m_obj, ps, prow, lane, u, rc, lc, viol, obj);
        if (u < ntiles)
            eval_single<Cfg, kShared, true, kObjShared>(d, m_bits, m_leader, m_obj, ps, prow, lane, u, rc, lc, viol, obj);
    }

    constexpr int NP0 = 3 + NPH;
    if constexpr (W <= 2) {
        // both counter sets in one pass: items 0..W-1 replica words, W..2W-1 leader words
        uint32_t pl[2 * W][kPlanes];
#pragma unroll
        for (int t = 0; t < W; ++t) {
            load_planes<W, NPH>(pl[t], rc, t);
            load_planes<W, NPH>(pl[W + t], lc, t);
        }
        viol += column_violation<2 * W, NP0>(pl, lane, W, cs->bnd_rep, cs->bnd_ldr, true, 1, d.log2S, d.R, cs);
    } else {
        uint32_t pl[W][kPlanes];
#pragma unroll
        for (int t = 0; t < W; ++t) load_planes<W, NPH>(pl[t], rc, t);
        viol += column_violation<W, NP0>(pl, lane, W, cs->bnd_rep, cs->bnd_rep, true, 0, d.log2S, d.R, cs);
#pragma unroll
        for (int t = 0; t < W; ++t) load_planes<W, NPH>(pl[t], lc, t);
        viol += column_violation<W, NP0>(pl, lane, W, cs->bnd_ldr, cs->bnd_ldr, false, 2, d.log2S, d.R, cs);
    }
    viol_out = __reduce_add_sync(0xFFFFFFFFu, viol) + d.P;          // + P: see column_violation (C2/C5)
    obj_out = __reduce_add_sync(0xFFFFFFFFu, obj);
}

// ------------------------------------------------------------------------------------------
// Delta evaluation (SURVEY.md §8(f)3, docs/MODEL.md §8): the SAME key as the full evaluator,
// computed from the base's totals and the candidate's <= 3 patched rows.  One THREAD per candidate.
// Reported separately from the full-evaluation throughput.
// ------------------------------------------------------------------------------------------
// C1 + C7 + leader validity and the objective of ONE row
template <class Cfg, bool kShared>
__device__ __forceinline__ void row_eval(const Params &d, const MemRef<kShared> &objT, int p,
                                         const uint32_t (&x)[Cfg::W], uint32_t ld, int &rv, int &ro)
{
    constexpr int W = Cfg::W;
    uint32_t oh[W], any = 0;
    const uint32_t ldbit = __funnelshift_l(0u, 1u, ld);
#pragma unroll
    for (int t = 0; t < W; ++t) {
        const uint32_t lm = ((int)(ld >> 5) == t) ? ldbit : 0u;
        oh[t] = x[t] & lm;
        any |= oh[t];
    }
    rv = row_rack_terms<W, Cfg::kRack>(x, d.log2S, d.R, d.ppr_lo, d.ppr_hi, d.RF) + (any ? 0 : 1);
    ro = 0;
    if constexpr (Cfg::kObj > 0) {
#pragma unroll
        for (int c = 0; c < Cfg::kObj; ++c) {
            int cnt = 0;
#pragma unroll
            for (int t = 0; t < W; ++t) {
                const uint32_t m = objT.ld32((uint32_t)((c * W + t) * d.Ppad + p) * 4u);
                cnt += __popc((c < 2 * Cfg::kObj / 3 ? x[t] : oh[t]) & m);
            }
            ro += cnt * d.plane_value[c];
        }
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (k < d.nentries) {
                const uint32_t e = objT.ld32((uint32_t)(k * d.Ppad + p) * 4u);
                const uint32_t slot = e & 0xFFu;
                const uint32_t xw = row_word<W>(x, (int)(slot >> 5));
                const bool bit = __funnelshift_r(xw, 0u, slot) & 1u;
                const uint32_t w = (slot == ld) ? (e >> 20) : ((e >> 8) & 0xFFFu);
                ro += bit ? (int)w : 0;
            }
        if (d.dense) {
            const uint32_t *wrow = d.dense_w + (size_t)p * d.NS;
#pragma unroll
            for (int t = 0; t < W; ++t) {
                for (uint32_t m = x[t]; m; m &= m - 1) {
                    const int s = t * 32 + __ffs(m) - 1;
                    if (s < d.NS) {
                        const uint32_t w = __ldg(wrow + s);
                        ro += (s == (int)ld) ? (int)(w >> 16) : (int)(w & 0xFFFFu);
                    }
                }
            }
        }
    }
}

__device__ __forceinline__ int band_violation(int c, uint32_t lohi)
{
    const int lo = (int)(lohi & 0xFFFFu), hi = (int)(lohi >> 16);
    return max(c - hi, 0) + max(lo - c, 0);
}

// events: (slot, +-1) pairs; applies the NET change of every distinct slot once
template <int N, class F> __device__ __forceinline__ int apply_events(const int (&slot)[N], const int (&val)[N], F cost)
{
    int dv = 0;
#pragma unroll
    for (int j = 0; j < N; ++j) {
        bool first = slot[j] >= 0;
        int net = 0;
#pragma unroll
        for (int k = 0; k < N; ++k) {
            if (k < j && slot[k] == slot[j]) first = false;
            net += (slot[k] == slot[j]) ? val[k] : 0;
        }
        if (first && net != 0) dv += cost(slot[j], net);
    }
    return dv;
}

template <int W> __device__ __forceinline__ int lone_slot(const uint32_t (&m)[W])
{
    int s = -1;
#pragma unroll
    for (int t = 0; t < W; ++t) if (m[t]) s = t * 32 + __ffs(m[t]) - 1;
    return s;
}

// cnt / lcnt: replica and (valid) leader count per slot of the BASE, rc: replica count per rack,
// base_viol / base_obj: the base's own evaluation.  Every patched partition differs from the base
// by at most one replica move and/or a leader change (MODEL 5: an op never revisits a partition).
template <class Cfg, bool kObjShared = true>
__device__ __forceinline__ void delta_eval(const Params &d, const uint32_t *s_bits, const uint8_t *s_leader,
                                           const MemRef<kObjShared> &objT, const Consts *cs, const PatchSet &ps,
                                           const uint32_t (&rows)[kMaxOps][Cfg::W], const int *cnt, const int *lcnt,
                                           const int *rc, int base_viol, int base_obj, int &viol, int &obj)
{
    constexpr int W = Cfg::W;
    viol = base_viol;
    obj = base_obj;
    int es[2 * kMaxOps], ev[2 * kMaxOps], ls[2 * kMaxOps], lv[2 * kMaxOps];
#pragma unroll
    for (int j = 0; j < 2 * kMaxOps; ++j) { es[j] = -1; ev[j] = 0; ls[j] = -1; lv[j] = 0; }
#pragma unroll
    for (int i = 0; i < kMaxOps; ++i) {
        if (i < ps.n) {
            const int p = ps.p[i];
            uint32_t xo[W], xn[W], rem[W], add[W];
#pragma unroll
            for (int t = 0; t < W; ++t) {
                xo[t] = s_bits[(size_t)t * d.Ppad + p];
                xn[t] = rows[i][t];
                rem[t] = xo[t] & ~xn[t];
                add[t] = xn[t] & ~xo[t];
            }
            const uint32_t ldo = s_leader[p], ldn = ps.ld[i];
            int rvo, roo, rvn, ron;
            row_eval<Cfg, kObjShared>(d, objT, p, xo, ldo, rvo, roo);
            row_eval<Cfg, kObjShared>(d, objT, p, xn, ldn, rvn, ron);
            viol += rvn - rvo;
            obj += ron - roo;
            es[2 * i] = lone_slot<W>(rem); ev[2 * i] = -1;
            es[2 * i + 1] = lone_slot<W>(add); ev[2 * i + 1] = 1;
            const bool oko = ((int)ldo < W * 32) && row_has<W>(xo, (int)ldo);
            const bool okn = ((int)ldn < W * 32) && row_has<W>(xn, (int)ldn);
            ls[2 * i] = oko ? (int)ldo : -1; lv[2 * i] = -1;
            ls[2 * i + 1] = okn ? (int)ldn : -1; lv[2 * i + 1] = 1;
        }
    }
    viol += apply_events<2 * kMaxOps>(es, ev, [&](int s, int net) {
        const uint32_t b = cs->bnd_rep[s];
        return band_violation(cnt[s] + net, b) - band_violation(cnt[s], b);
    });
    viol += apply_events<2 * kMaxOps>(ls, lv, [&](int s, int net) {
        const uint32_t b = cs->bnd_ldr[s];
        return band_violation(lcnt[s] + net, b) - band_violation(lcnt[s], b);
    });
    int rs[2 * kMaxOps];
#pragma unroll
    for (int j = 0; j < 2 * kMaxOps; ++j) rs[j] = es[j] < 0 ? -1 : ((es[j] >> d.log2S) < d.R ? (es[j] >> d.log2S) : -1);
    viol += apply_events<2 * kMaxOps>(rs, ev, [&](int r, int net) {
        const int lo = cs->rack_lo[r], hi = cs->rack_hi[r], c0 = rc[r], c1 = rc[r] + net;
        return (max(c1 - hi, 0) + max(lo - c1, 0)) - (max(c0 - hi, 0) + max(lo - c0, 0));
    });
}

}  // namespace kao
