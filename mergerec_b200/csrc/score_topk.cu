// score_topk.cu -- evaluator hot path B1+B2 fused (SURVEY.md section 8(a)): full-catalog scoring
//     scores[q, n] = sum_e U[q, e] * I[n, e]                (ref: module/recommender/module.py:137)
// followed by the per-row top-K                              (ref: evaluator/evaluator.py:43)
// without ever materialising the (Q, N) score matrix.
//
// Tensor-core contraction on sm_100a: tcgen05.mma kind::tf32, operands staged in shared memory by TMA
// (128-byte swizzle, K-major), fp32 accumulators in TMEM, read back with tcgen05.ld by the epilogue warps.
// fp32-faithful mode (default) is 3xTF32 on pre-split operands (hi = rna_tf32(x), lo = rna_tf32(x - hi)):
//     U.I ~= Uhi.Ilo + Ulo.Ihi + Uhi.Ihi      (error ~2^-22 per product, like an fp32 product's own rounding)
//
// Work decomposition.  A "unit" is (query block, item split): BLOCK_M * CG query rows against a contiguous
// range of 256-item tiles.  A persistent grid of CTAs (CG = 1) or CTA pairs (CG = 2, cta_group::2: 256-row
// tiles, each CTA stages its own 128 query rows and half of the item tile) walks a static unit list ordered so
// that concurrently running units share item tiles through L2 while their query blocks stay L2-resident.
// Warp roles per CTA: 0 = TMA producer, 1 = MMA issuer (leader CTA of a pair only), 2 = TMEM allocator,
// 4..7 = epilogue: thread t owns accumulator lane (= query row) t, tests the 256 scores of a tile branch-free against
// the row's running threshold (score of its K-th best so far) and appends survivors to a per-row candidate buffer
// in global memory (L2-resident); when a buffer fills, the warp finds the row's K-th largest score with a register
// bitonic network (8 keys per lane, shuffles across lanes, two rows interleaved) and keeps what is at or above it.
// After its last tile a unit sorts each row by the 64-bit key (score desc, id asc) and writes one list per row;
// lists of different splits are merged by mr_topk_merge.
//
// Two accumulator stages (2 x 256 TMEM columns) let the epilogue of tile i overlap the MMAs of tile i + 1.
#include <cuda.h>

#include <type_traits>

#include "common.cuh"
#include "topk_common.cuh"

namespace mr {
namespace st {

constexpr int kBlockM = 128;   // query rows per CTA (TMEM lanes)
constexpr int kBlockN = 256;   // items per tile (TMEM columns per accumulator stage)
// k-block = fp32 elements per pipeline stage and row: BK = 32 -> 128-byte rows (SWIZZLE_128B), BK = 16 -> 64-byte rows
// (SWIZZLE_64B): half-size stages, more of them in flight (template parameter BK of the kernel)
constexpr int kUmmaK = 8;      // tf32: 32 bytes of K per tcgen05.mma
// Epilogue warp groups (4 warps each; template parameter EG of the kernel): with EG = 2, group g drains accumulator
// stage g, i.e. every second tile, with its own per-row candidate buffers and lists.  Every mode runs ONE group by
// default.  Two groups were measured for the epilogue-bound bf16-compat mode at BASELINE config 5
// (MR_SCORE_BF16_EPI_GROUPS=2): 140.4 ms against 121.7 ms with one group, identical lists -- each group sees only every
// second tile, so its per-row threshold rises half as fast, twice as many candidates pass the filter and twice as many
// lists are sorted and merged; the filter, not the number of warps draining TMEM, is what has to get cheaper.
constexpr int kMaxEpiGroups = 2;
constexpr int kCap = 256;      // per-row candidate buffer (keys); power of two, >= 2 * MR_MAX_FUSED_TOPK
constexpr int kChunk = 16;     // accumulator columns per tcgen05.ld
constexpr int kAccStages = 2;
// BF16 (bf16-compat mode): one bf16 operand pair per stage, rows of 64 bf16 = 128 bytes (same geometry as BK = 32).
template <int CG, int BK, bool BF16> struct Cfg {
    static constexpr int kABytes = kBlockM * BK * 4;         // one of (hi, lo) of the query tile: 16 KB at BK = 32
    static constexpr int kBRows = kBlockN / CG;              // item rows staged by one CTA
    static constexpr int kBBytes = kBRows * BK * 4;          // 32 KB (CG 1) / 16 KB (CG 2) at BK = 32
    static constexpr int kStageBytes = (BF16 ? 1 : 2) * (kABytes + kBBytes);
    static constexpr int kStages = BF16 ? (CG == 1 ? 4 : 6) : BK == 32 ? (CG == 1 ? 2 : 3) : (CG == 1 ? 4 : 7);
    static constexpr int kElemsPerBlock = BF16 ? 2 * BK : BK;   // K elements per k-block
    static constexpr int kBarBytes = 256;
    static constexpr int kSmemBytes = kStages * kStageBytes + kBarBytes + 1024 /* alignment slack */;
};

struct Params {
    int64_t Q, N;
    int E, K, mode;
    int32_t id_base;
    int KB;       // k-blocks per tile = ceil(E / 32)
    int T;        // item tiles = ceil(N / 256)
    int QB;       // query blocks = ceil(Q / (128 * CG))
    int S;        // item splits
    int QG;       // query blocks per L2 group
    u64* cand;    // grid * EG * 128 * kCap keys
    float* out_val;     // (S * EG, Q, K)
    int32_t* out_id;    // (S * EG, Q, K)
    long long* dbg;     // optional timestamps of block 0 (mr_score_topk_debug_buffer), else NULL
    int l2_hint;        // 1: query loads evict_last, item loads evict_first (MR_SCORE_L2HINT, default on)
    // Pacing of the units that share an item stream (NULL = off): sync[stream * sync_windows + j] counts the units whose
    // producer has issued the loads of tile window j (sync_w tiles); a producer does not start window j + sync_lead
    // before every unit of its stream has issued window j -- or a short timeout has passed: the pacing is a performance hint
    // (it keeps the units within sync_lead windows of each other, so an item tile fetched by the first is still in L2 for the last), never
    // a correctness condition, and can therefore not deadlock.
    int32_t* sync;
    int sync_w, sync_windows, sync_lead;
    int wave;           // CTA pairs (clusters) in the grid = units that run at the same time
    int sync_giveup;    // windows after which a unit stops waiting if a member of its stream has not even started (0 = never)
};
// Parameters of the EXCL instantiations (mr_score_topk_exclude).  A type of their own: adding the fields to Params changes
// the code ptxas emits for the other instantiations.
struct ExclParams : Params {
    // items to leave out of each row's list, CSR by global query row: row q's global item ids are
    // excl_ids[excl_off[q] .. excl_off[q + 1]), ascending, duplicates allowed
    const int64_t* excl_off;
    const int32_t* excl_ids;
};
// Epilogue of an instantiation (template parameter EPI): the top-K lists, or one of the two label-rank passes --
// kEpiDiag (mr_label_score): the score key of each query's label; kEpiCount (mr_score_rank): per (split, row), the
// items of the unit that sort before the row's label.
constexpr int kEpiTopK = 0, kEpiCount = 1, kEpiDiag = 2;
// Parameters of the label-rank instantiations, a type of their own for the same reason as ExclParams.
struct RankParams : ExclParams {
    const int64_t* labels;       // (Q) global item id of each query's label
    const uint32_t* label_key;   // kEpiCount: (Q) score key of the label's score (0: no label, the row is not counted)
    uint32_t* out_key;           // kEpiDiag: (Q) score key of the label's score, 0 when the label is not in this table
    int32_t* part;               // kEpiCount: (S, Q) counts per item split
};
// kEpiLse (mr_score_lse): per (split, row), the exponential sum of the unit's eligible scores as a pair (shift k,
// sum s) with value s * 2^k in log2 units.  A type of its own, for the same reason again; labels are not read.
constexpr int kEpiLse = 3;
struct LseParams : RankParams {
    float lse_c;                 // log2(e) / temperature: the logit of score f is f * lse_c in log2 units
    int32_t* lse_shift;          // (S, Q)
    double* lse_sum;             // (S, Q)
};
// Shift range of a (shift, sum) pair: an empty sum is (kLseMinShift, 0).  Logits stay exact in the fp32 fma of the
// epilogue while |shift| <= 2^24, which bounds the supported |score / temperature| to about 1.1e7.
constexpr int kLseMinShift = -(1 << 24), kLseMaxShift = 1 << 24;
template <bool EXCL, int EPI = kEpiTopK>
using KernelParams = typename std::conditional<
    EPI == kEpiLse, LseParams,
    typename std::conditional<EPI != kEpiTopK, RankParams,
                              typename std::conditional<EXCL, ExclParams, Params>::type>::type>::type;

// ---- PTX helpers ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive_local(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint32_t bar, uint32_t cta) {
    asm volatile(
        "{\n\t.reg .b32 ra;\n\tmapa.shared::cluster.u32 ra, %0, %1;\n\tmbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}"
        ::"r"(bar), "r"(cta) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug must end in a trap (launch failure), never in a hung GPU.
__device__ __noinline__ void mbar_wait_slow(uint32_t bar, uint32_t parity, int what) {
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 4000000000LL) {
            printf("mr_score_topk: barrier wait timed out (what=%d block=%d thread=%d parity=%u)\n", what, blockIdx.x,
                   threadIdx.x, parity);
            __trap();
        }
    }
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int what) {
    if (!mbar_try_wait(bar, parity)) mbar_wait_slow(bar, parity, what);
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// L2 eviction policies for the two operand streams: the query block of a unit is re-read for every item tile and must
// stay in L2 (evict_last); item tiles are read by the handful of pairs that walk the same split and then never again
// (evict_first), so that streaming the 6 GB item table does not push the query blocks out.
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
template <int CG>
__device__ __forceinline__ void tma_load_2d_hint(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, uint64_t pol) {
    if (CG == 1) {
        asm volatile(
            "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
            ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "l"(pol) : "memory");
    } else {
        asm volatile(
            "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4}], [%2], %5;"
            ::"r"(dst), "l"(map), "r"(bar & 0xFEFFFFFFu), "r"(c0), "r"(c1), "l"(pol) : "memory");
    }
}
template <int CG>
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
    if (CG == 1) {
        asm volatile(
            "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
            ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
    } else {
        // both CTAs of the pair issue their own loads; the transaction bytes land on the leader's barrier
        asm volatile(
            "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
            ::"r"(dst), "l"(map), "r"(bar & 0xFEFFFFFFu), "r"(c0), "r"(c1) : "memory");
    }
}
template <int CG>
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    if (CG == 1) {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
    } else {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
    }
}
template <int CG>
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    if (CG == 1) {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
    } else {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc) : "memory");
    }
}
// tcgen05.commit: the barrier is arrived on when every previously issued MMA of this thread has completed
template <int CG>
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    if (CG == 1) {
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
    } else {
        asm volatile(
            "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
            ::"r"(bar), "h"((uint16_t)3) : "memory");
    }
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major shared-memory matrix descriptor: rows of BK * 4 bytes (= the swizzle span), 8-row groups 8 rows apart.
template <int BK>
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4)            // start address, 16-byte units
           | ((uint64_t)((8 * BK * 4) >> 4) << 32)        // stride byte offset between 8-row groups
           | (1ull << 46)                                 // descriptor version (sm_100)
           | ((BK == 32 ? 2ull : 4ull) << 61);            // SWIZZLE_128B / SWIZZLE_64B
}
// kind::tf32 instruction descriptor: fp32 accumulate, tf32 x tf32, both operands K-major, N = 256, M = 128 * CG
template <int CG, bool BF16>
__device__ __forceinline__ constexpr uint32_t make_idesc() {
    return (1u << 4) | ((BF16 ? 1u : 2u) << 7) | ((BF16 ? 1u : 2u) << 10) | ((uint32_t)(kBlockN >> 3) << 17) |
           ((uint32_t)((kBlockM * CG) >> 4) << 24);
}

// diagnostics: block 0 stamps clock64() per tile into dbg[role][tile][slot] (role 0 producer, 1 mma, 2 epilogue)
constexpr int kDbgTiles = 64, kDbgSlots = 4;
__device__ __forceinline__ void dbg_stamp(const Params& p, int role, uint32_t tile, int slot) {
    if (p.dbg && blockIdx.x == 0 && tile < (uint32_t)kDbgTiles) p.dbg[(role * kDbgTiles + tile) * kDbgSlots + slot] = clock64();
}

// ---- static unit schedule (identical in every role) ---------------------------------------------------------------
struct Unit {
    int qb, split, t0, t1;
    int stream;    // index of the item stream this unit walks = (query group, split): its units share every item tile
    int members;   // units on that stream (query blocks of the group)
};
__host__ __device__ __forceinline__ bool get_unit(const Params& p, int u, Unit& out) {
    const int U = p.QB * p.S;
    if (u >= U) return false;
    if (p.QG == 0) {
        // wave-aligned order (default): units are numbered query-block-major, u = qb * S + split, and wave w of the
        // grid's CTA pairs runs units [w * wave, (w + 1) * wave) -- so the pairs running at the same time walk exactly S
        // item streams, each shared by the units of that wave with the same split (wave / S of them, +- 1 when S does not
        // divide the wave), whatever S is.
        // Inside a wave the pairs are handed out split-major (pairs 0 .. m_0 - 1 walk stream 0, the next m_1 stream 1,
        // ...), so neighbouring SMs share a stream -- with S = 2 this is the 37 + 37 arrangement the numbers above were
        // measured with.
        const int w = u / p.wave;
        const int lo = w * p.wave, hi = (lo + p.wave) < U ? (lo + p.wave) : U;
        int r = u - lo, sp = 0, m = 0;
        for (; sp < p.S; ++sp) {
            m = (hi + p.S - 1 - sp) / p.S - (lo + p.S - 1 - sp) / p.S;   // number of v in [lo, hi) with v % S == sp
            if (r < m) break;
            r -= m;
        }
        const int first = lo + (sp - lo % p.S + p.S) % p.S;               // first v >= lo with v % S == sp
        const int v = first + r * p.S;
        out.split = sp;
        out.qb = v / p.S;
        out.stream = w * p.S + sp;
        out.members = m;
    } else {
        // explicit query groups (MR_SCORE_QGROUP): group g = QG query blocks x S splits, split-major inside the group
        const int per_group = p.QG * p.S;
        const int g = u / per_group, r = u - g * per_group;
        const int qg0 = g * p.QG;
        const int qgn = (p.QB - qg0) < p.QG ? (p.QB - qg0) : p.QG;
        out.split = r / qgn;
        out.qb = qg0 + (r - out.split * qgn);
        out.stream = g * p.S + out.split;
        out.members = qgn;
    }
    out.t0 = (int)(((int64_t)out.split * p.T) / p.S);
    out.t1 = (int)(((int64_t)(out.split + 1) * p.T) / p.S);
    return true;
}

// ---- warp-cooperative compaction of one row's candidate buffer ----------------------------------------------------
// Bitonic sort (descending) of kCap = 256 keys held in registers, 8 per lane: element e = lane * 8 + r.
// Strides 1, 2, 4 are register-to-register; strides >= 8 exchange with lane ^ (stride / 8) through shuffles.
// Register indices are compile-time constants, but the stage loops are NOT unrolled: `size` and the lane stride
// are run-time values, which keeps the routine at ~250 instructions instead of ~1500 (the epilogue has to stay
// inside the instruction cache; a fully unrolled network plus an unrolled filter made every tile fetch its code
// from L2 again and ran 3x slower).
__device__ __forceinline__ void cmpx(u64& a, u64& b, bool desc) {
    const bool gt = a > b;
    const u64 hi = gt ? a : b, lo = gt ? b : a;
    a = desc ? hi : lo;
    b = desc ? lo : hi;
}
// Two rows per call: the two networks are independent, which doubles the instruction-level parallelism of what is
// otherwise a chain of dependent compare-exchanges run by one warp alone on its scheduler.
__device__ __forceinline__ void warp_sort256x2(u64 (&a)[8], u64 (&b)[8], int lane) {
#pragma unroll 1
    for (int size = 2; size <= kCap; size <<= 1) {
        const bool desc_lane = ((lane * 8) & size) == 0;     // valid for size >= 8 (direction depends on the lane only)
#pragma unroll 1
        for (int lstride = size >> 4; lstride > 0; lstride >>= 1) {   // strides size/2 .. 8, in lanes
            const bool take_max = ((lane & lstride) == 0) == desc_lane;
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                const u64 oa = __shfl_xor_sync(0xffffffffu, a[r], lstride);
                const u64 ob = __shfl_xor_sync(0xffffffffu, b[r], lstride);
                a[r] = ((a[r] > oa) == take_max) ? a[r] : oa;
                b[r] = ((b[r] > ob) == take_max) ? b[r] : ob;
            }
        }
#pragma unroll
        for (int stride = 4; stride >= 1; stride >>= 1) {
            if (stride < size) {
#pragma unroll
                for (int r = 0; r < 8; ++r)
                    if ((r & stride) == 0) {
                        const bool desc = (((lane * 8) + r) & size) == 0;
                        cmpx(a[r], a[r | stride], desc);
                        cmpx(b[r], b[r | stride], desc);
                    }
            }
        }
    }
}
// Same network on 32-bit score keys (half the shuffles, min/max instead of 64-bit compare + selects): used by the
// in-loop compaction, which only needs the K-th largest SCORE to decide what survives; the order inside the buffer
// is irrelevant until the unit's final sort.
__device__ __forceinline__ void cmpx32(uint32_t& a, uint32_t& b, bool desc) {
    const uint32_t hi = a > b ? a : b, lo = a > b ? b : a;
    a = desc ? hi : lo;
    b = desc ? lo : hi;
}
__device__ __forceinline__ void warp_sort256x2_u32(uint32_t (&a)[8], uint32_t (&b)[8], int lane) {
#pragma unroll 1
    for (int size = 2; size <= kCap; size <<= 1) {
        const bool desc_lane = ((lane * 8) & size) == 0;
#pragma unroll 1
        for (int lstride = size >> 4; lstride > 0; lstride >>= 1) {
            const bool take_max = ((lane & lstride) == 0) == desc_lane;
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                const uint32_t oa = __shfl_xor_sync(0xffffffffu, a[r], lstride);
                const uint32_t ob = __shfl_xor_sync(0xffffffffu, b[r], lstride);
                a[r] = take_max ? (a[r] > oa ? a[r] : oa) : (a[r] > oa ? oa : a[r]);
                b[r] = take_max ? (b[r] > ob ? b[r] : ob) : (b[r] > ob ? ob : b[r]);
            }
        }
#pragma unroll
        for (int stride = 4; stride >= 1; stride >>= 1) {
            if (stride < size) {
#pragma unroll
                for (int r = 0; r < 8; ++r)
                    if ((r & stride) == 0) {
                        const bool desc = (((lane * 8) + r) & size) == 0;
                        cmpx32(a[r], a[r | stride], desc);
                        cmpx32(b[r], b[r | stride], desc);
                    }
            }
        }
    }
}
__device__ __forceinline__ uint32_t warp_pick32(const uint32_t (&v)[8], int e) {
    uint32_t x = 0;
#pragma unroll
    for (int r = 0; r < 8; ++r)
        if (r == (e & 7)) x = v[r];
    return __shfl_sync(0xffffffffu, x, e >> 3);
}
// Keep the keys whose score key is >= t, packed to the front of the row buffer (any order).  Returns their number.
__device__ __forceinline__ int warp_keep_ge(u64* gbuf, const u64 (&k)[8], uint32_t t, int lane) {
    int c = 0;
#pragma unroll
    for (int r = 0; r < 8; ++r) c += ((uint32_t)(k[r] >> 32) >= t) ? 1 : 0;
    int incl = c;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int n = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= off) incl += n;
    }
    int pos = incl - c;
#pragma unroll
    for (int r = 0; r < 8; ++r)
        if ((uint32_t)(k[r] >> 32) >= t) gbuf[pos++] = k[r];
    return __shfl_sync(0xffffffffu, incl, 31);
}
// Row buffer (n <= kCap keys in global memory) -> registers (zero padded), element e = lane * 8 + r.
__device__ __forceinline__ void warp_load_keys(u64 (&v)[8], const u64* gbuf, int n, int lane) {
    const uint4* g4 = reinterpret_cast<const uint4*>(gbuf + lane * 8);
#pragma unroll
    for (int h = 0; h < 4; ++h) {
        uint4 t = make_uint4(0, 0, 0, 0);
        if (lane * 8 + 2 * h < n) t = g4[h];
        v[2 * h] = ((u64)t.y << 32) | t.x;
        v[2 * h + 1] = (lane * 8 + 2 * h + 1 < n) ? (((u64)t.w << 32) | t.z) : 0ull;
    }
}
// the first `keep` sorted keys back to the row buffer
__device__ __forceinline__ void warp_store_keys(u64* gbuf, const u64 (&v)[8], int keep, int lane) {
    uint4* o4 = reinterpret_cast<uint4*>(gbuf + lane * 8);
#pragma unroll
    for (int h = 0; h < 4; ++h)
        if (lane * 8 + 2 * h < keep)
            o4[h] = make_uint4((uint32_t)v[2 * h], (uint32_t)(v[2 * h] >> 32), (uint32_t)v[2 * h + 1],
                               (uint32_t)(v[2 * h + 1] >> 32));
}
// sorted registers -> one (val, id) list of K entries; keys are zero beyond the row's candidates
__device__ __forceinline__ void warp_write_list(const Params& p, size_t o, const u64 (&v)[8], int K, int lane) {
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const int i = lane * 8 + r;
        if (i < K) {
            const u64 key = v[r];
            p.out_id[o + i] = key ? (int32_t)key_id(key) : -1;
            p.out_val[o + i] = key ? key_score(key) : -INFINITY;
        }
    }
}

// The score the top-K epilogue ranks: the fp32 accumulator, or in bf16-compat mode that accumulator rounded to bf16
// (RN-even) with the same bit operations.
template <bool BF16>
__device__ __forceinline__ float ranked_score(uint32_t bits) {
    if (BF16) {
        if ((bits & 0x7F800000u) != 0x7F800000u) bits += 0x7FFFu + ((bits >> 16) & 1u);
        bits &= 0xFFFF0000u;
    }
    return __uint_as_float(bits);
}

// ---- label-rank epilogues (RankParams) ----------------------------------------------------------------------------
// kEpiDiag: every unit walks one tile, the gathered label rows of its own query rows (host side: label_score), so query
// row `row` of CTA `rank` meets its label in accumulator column rank * 128 + row.  Two 16-column loads cover a warp's 32
// columns; each lane selects its own.
// kEpiCount: per 16-column chunk, bit j = "column j sorts before the row's label" under (score key desc, id asc):
// greater score, or equal score and smaller id (an arithmetic mask of the ids below the label), minus padding and
// excluded ids (the forward-only cursor of the EXCL top-K epilogue); the row's count grows by the popc.  No candidate
// buffer, no sort.  The float tests are the key tests: -0 == +0, and a NaN score is above every other (gt = !(f <= L));
// for a NaN label only the NaN columns with smaller ids count (Lg = +inf: gt = NaN, eq = never).
template <int CG, bool BF16, bool EXCL, int EPI>
__device__ __forceinline__ void rank_epilogue(const RankParams& p, uint32_t tmem_base, uint32_t bar_tfull,
                                              uint32_t bar_tempty, uint32_t rank, bool leader, int cluster_id,
                                              int num_clusters, int warp, int lane) {
    const int ew = (warp - 4) & 3;
    const int row = ew * 32 + lane;
    uint32_t it = 0;
    Unit u;
    for (int ui = cluster_id; get_unit(p, ui, u); ui += num_clusters) {
        const int64_t q = ((int64_t)u.qb * CG + rank) * kBlockM + row;
        const bool active = q < p.Q;
        uint32_t L = 0;
        float Lf = 0.0f, Lg = 0.0f;
        int64_t lab = 0;
        // ex_next: the id under the exclusion cursor, INT64_MAX past the end of the row.  (An int32 sentinel could be
        // reached: the last chunk of a table ending at 2^31 - 1 spans ids up to id0 + 15 > INT32_MAX.)
        int64_t ex_cur = 0, ex_end = 0;
        int64_t ex_next = INT64_MAX;
        if (EPI == kEpiCount && active) {
            L = p.label_key[q];
            lab = p.labels[q];
            Lf = key_score((u64)L << 32);
            Lg = L == 0xFFFFFFFFu ? INFINITY : Lf;
            if constexpr (EXCL) {
                ex_cur = p.excl_off[q];
                ex_end = p.excl_off[q + 1];
                const int64_t first = (int64_t)p.id_base + (int64_t)u.t0 * kBlockN;
                for (int64_t hi = ex_end; ex_cur < hi;) {
                    const int64_t mid = (ex_cur + hi) >> 1;
                    if ((int64_t)p.excl_ids[mid] < first) ex_cur = mid + 1; else hi = mid;
                }
                if (ex_cur < ex_end) ex_next = p.excl_ids[ex_cur];
            }
        }
        const uint32_t gt_keep = L == 0xFFFFFFFFu ? 0u : 0xFFFFu;   // NaN label: the NaN columns count only below its id
        int cnt = 0;
        for (int t = u.t0; t < u.t1; ++t, ++it) {
            const uint32_t acc = it & 1;
            mbar_wait(bar_tfull + 8 * acc, (it >> 1) & 1, 4);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + acc * kBlockN;
            if constexpr (EPI == kEpiDiag) {
                uint32_t a[kChunk], b[kChunk];
                tmem_ld16(taddr + rank * kBlockM + ew * 32, a);
                tmem_ld16(taddr + rank * kBlockM + ew * 32 + kChunk, b);
                tmem_ld_wait();
                // column `lane` of the warp's 32: a select tree on the bits of the lane, constant register indices only
#pragma unroll
                for (int j = 0; j < kChunk; ++j) a[j] = lane < kChunk ? a[j] : b[j];
#pragma unroll
                for (int h = kChunk / 2; h >= 1; h >>= 1)
#pragma unroll
                    for (int j = 0; j < h; ++j) a[j] = (lane & h) ? a[j + h] : a[j];
                const uint32_t bits = a[0];
                if (active) {
                    const int64_t l = p.labels[q];
                    const bool mine = l >= (int64_t)p.id_base && l < (int64_t)p.id_base + p.N;
                    p.out_key[q] = mine ? score_key(ranked_score<BF16>(bits)) : 0u;
                }
            } else {
                const int64_t n0 = (int64_t)t * kBlockN;
                const int nvalid = (int)((p.N - n0) < kBlockN ? (p.N - n0) : kBlockN);
#pragma unroll 1
                for (int c = 0; c < nvalid; c += kChunk) {
                    uint32_t v[kChunk];
                    tmem_ld16(taddr + c, v);
                    tmem_ld_wait();
                    uint32_t gt = 0, eq = 0;
#pragma unroll
                    for (int j = 0; j < kChunk; ++j) {
                        const float f = ranked_score<BF16>(v[j]);
                        gt |= !(f <= Lg) ? (1u << j) : 0u;
                        eq |= (f == Lf) ? (1u << j) : 0u;
                    }
                    const int64_t id0 = (int64_t)p.id_base + n0 + c;
                    const int64_t d = lab - id0;                          // columns of the chunk with ids below the label
                    const uint32_t below = d <= 0 ? 0u : d >= kChunk ? 0xFFFFu : (1u << d) - 1u;
                    uint32_t m = (gt & (gt_keep | below)) | (eq & below);
                    if (nvalid - c < kChunk) m &= (1u << (nvalid - c)) - 1u;
                    if constexpr (EXCL) {
                        while (ex_next < id0 + kChunk) {
                            if (ex_next >= id0) m &= ~(1u << (int)(ex_next - id0));
                            ex_next = ++ex_cur < ex_end ? (int64_t)p.excl_ids[ex_cur] : INT64_MAX;
                        }
                    }
                    cnt += __popc(m);
                }
            }
            // accumulator stage drained: hand it back to the MMA issuer
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if (CG == 1 || leader) mbar_arrive_local(bar_tempty + 8 * acc);
                else mbar_arrive_remote(bar_tempty + 8 * acc, 0);
            }
        }
        if (EPI == kEpiCount && active) p.part[(size_t)u.split * p.Q + q] = cnt;
    }
}

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// ---- log-sum-exp epilogue (LseParams) -----------------------------------------------------------------------------
// kEpiLse: the counting pass's schedule and exclusion cursor; per row, the sum of 2^(f c) over the eligible columns
// (not padding, not in the row's exclusion list) of the unit, f = the score top-K ranks, as acc * 2^k.  Each chunk adds
// its 16 terms 2^(f c - k), summed in fp32, to the fp64 accumulator.  The integer shift k only rises, and only when a
// chunk's max(f) c exceeds k + 64, to ceil(max(f) c): the terms stay below 2^64, the first term that set the shift is
// in (1/2, 1], and the rescale of acc by ldexp is exact, however many chunks raise the shift.  Special values as
// torch.logsumexp: an eligible NaN gives NaN (its term is NaN; fmaxf, which drops it, only places the shift), an
// eligible +inf gives +inf (its term is +inf; the shift stays), and a row of -inf or of no eligible item gives the
// empty pair (kLseMinShift, 0).
template <int CG, bool BF16, bool EXCL>
__device__ __forceinline__ void lse_epilogue(const LseParams& p, uint32_t tmem_base, uint32_t bar_tfull,
                                             uint32_t bar_tempty, uint32_t rank, bool leader, int cluster_id,
                                             int num_clusters, int warp, int lane) {
    const int ew = (warp - 4) & 3;
    const int row = ew * 32 + lane;
    const float lc = p.lse_c;
    uint32_t it = 0;
    Unit u;
    for (int ui = cluster_id; get_unit(p, ui, u); ui += num_clusters) {
        const int64_t q = ((int64_t)u.qb * CG + rank) * kBlockM + row;
        const bool active = q < p.Q;
        int64_t ex_cur = 0, ex_end = 0;
        int64_t ex_next = INT64_MAX;   // as in rank_epilogue
        if constexpr (EXCL) {
            if (active) {
                ex_cur = p.excl_off[q];
                ex_end = p.excl_off[q + 1];
                const int64_t first = (int64_t)p.id_base + (int64_t)u.t0 * kBlockN;
                for (int64_t hi = ex_end; ex_cur < hi;) {
                    const int64_t mid = (ex_cur + hi) >> 1;
                    if ((int64_t)p.excl_ids[mid] < first) ex_cur = mid + 1; else hi = mid;
                }
                if (ex_cur < ex_end) ex_next = p.excl_ids[ex_cur];
            }
        }
        int k = kLseMinShift;
        double acc = 0.0;
        for (int t = u.t0; t < u.t1; ++t, ++it) {
            const uint32_t stage = it & 1;
            mbar_wait(bar_tfull + 8 * stage, (it >> 1) & 1, 4);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + stage * kBlockN;
            const int64_t n0 = (int64_t)t * kBlockN;
            const int nvalid = (int)((p.N - n0) < kBlockN ? (p.N - n0) : kBlockN);
#pragma unroll 1
            for (int c = 0; c < nvalid; c += kChunk) {
                uint32_t v[kChunk];
                tmem_ld16(taddr + c, v);
                tmem_ld_wait();
                uint32_t m = nvalid - c < kChunk ? (1u << (nvalid - c)) - 1u : 0xFFFFu;
                if constexpr (EXCL) {
                    const int64_t id0 = (int64_t)p.id_base + n0 + c;
                    while (ex_next < id0 + kChunk) {
                        if (ex_next >= id0) m &= ~(1u << (int)(ex_next - id0));
                        ex_next = ++ex_cur < ex_end ? (int64_t)p.excl_ids[ex_cur] : INT64_MAX;
                    }
                }
                float f[kChunk];
                float mx = -INFINITY;
#pragma unroll
                for (int j = 0; j < kChunk; ++j) {
                    f[j] = (m >> j) & 1u ? ranked_score<BF16>(v[j]) : -INFINITY;
                    mx = fmaxf(mx, f[j]);
                }
                const float top = mx * lc;
                if (top > (float)(k + 64) && top < INFINITY) {
                    const int nk = top < (float)kLseMaxShift ? (int)ceilf(top) : kLseMaxShift;
                    acc = ldexp(acc, k - nk);
                    k = nk;
                }
                const float nkf = -(float)k;
                float s = 0.0f;
#pragma unroll
                for (int j = 0; j < kChunk; ++j) s += ex2_approx(fmaf(f[j], lc, nkf));
                acc += (double)s;
            }
            // accumulator stage drained: hand it back to the MMA issuer
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if (CG == 1 || leader) mbar_arrive_local(bar_tempty + 8 * stage);
                else mbar_arrive_remote(bar_tempty + 8 * stage, 0);
            }
        }
        if (active) {
            p.lse_shift[(size_t)u.split * p.Q + q] = k;
            p.lse_sum[(size_t)u.split * p.Q + q] = acc;
        }
    }
}

// EXCL: leave the items of the row's exclusion list (ExclParams) out of its list.  Phase 2 of the
// epilogue skips an excluded id before it enters the candidate buffer, so the running threshold stays the exact K-th
// best of the eligible items.  Inside a unit a row meets its item ids in ascending order (tiles, chunks and bits within
// a chunk ascend), so a lane-private cursor into the row's sorted list only moves forward: one register compare per
// survivor of the threshold filter, at most one load per list entry and unit.  A separate instantiation, not a run-time
// test, because the epilogue's speed depends on its code staying inside the instruction cache (DESIGN.md section 3.4).
template <int CG, int BK, bool BF16, int EG, bool EXCL, int EPI = kEpiTopK>
__global__ void __launch_bounds__(128 + 128 * EG, 1)
score_topk_kernel(const __grid_constant__ CUtensorMap map_uhi, const __grid_constant__ CUtensorMap map_ulo,
                  const __grid_constant__ CUtensorMap map_ihi, const __grid_constant__ CUtensorMap map_ilo,
                  const KernelParams<EXCL, EPI> p) {
    using C = Cfg<CG, BK, BF16>;
    constexpr int kABytes = C::kABytes;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    unsigned char* stages = smem;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::kStages * C::kStageBytes);
    // barriers: full[kStages], empty[kStages], tmem_full[2], tmem_empty[2]
    const uint32_t bar_full = smem_u32(bars);
    const uint32_t bar_empty = bar_full + 8 * C::kStages;
    const uint32_t bar_tfull = bar_empty + 8 * C::kStages;
    const uint32_t bar_tempty = bar_tfull + 8 * kAccStages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * C::kStages + 2 * kAccStages);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = CG == 1 ? 0u : cluster_ctarank();
    const bool leader = rank == 0;
    const int cluster_id = blockIdx.x / CG;
    const int num_clusters = gridDim.x / CG;
    const bool x3 = !BF16 && p.mode == 0;

    if (CG > 1) cluster_sync_all();  // both CTAs resident before the paired TMEM allocation
    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_uhi) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_ihi) : "memory");
        if (x3) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_ulo) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&map_ilo) : "memory");
        }
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < C::kStages; ++i) {
            mbar_init(bar_full + 8 * i, CG);   // producer arrivals (leader's barrier collects both CTAs)
            mbar_init(bar_empty + 8 * i, 1);   // one tcgen05.commit
        }
        for (int i = 0; i < kAccStages; ++i) {
            mbar_init(bar_tfull + 8 * i, 1);        // one tcgen05.commit
            mbar_init(bar_tempty + 8 * i, 4 * CG);  // one arrival per epilogue warp of every CTA in the pair
        }
        fence_barrier_init();
    }
    if (warp == 2) {
        if (CG == 1) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        }
    }
    tc_fence_before();
    if (CG > 1) cluster_sync_all(); else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===== TMA producer (one lane) =====
        if (lane == 0) {
            uint32_t kiter = 0;
            Unit u;
            // l2_hint: 1 = queries evict_last / items evict_first (default); 2..4 = experiment modes (MR_SCORE_L2HINT)
            const uint64_t pol_last = l2_policy_evict_last(), pol_first = l2_policy_evict_first();
            uint64_t pol_q = pol_last, pol_i = pol_first;
            if (p.l2_hint == 3) { pol_q = pol_first; pol_i = pol_last; }
            if (p.l2_hint == 4) { pol_q = pol_last; pol_i = pol_last; }
            const bool hint = p.l2_hint != 0;
            const bool hint_items = p.l2_hint != 2;          // 2: queries evict_last, items default policy
            for (int ui = cluster_id; get_unit(p, ui, u); ui += num_clusters) {
                const int qrow = (u.qb * CG + (int)rank) * kBlockM;
                int32_t* pace = p.sync ? p.sync + (size_t)u.stream * p.sync_windows : nullptr;
                // A stream whose units are spread over two waves of CTA pairs (QG * S does not fill a wave exactly, e.g.
                // 18 x 4 of 74 at BASELINE config 4) has members that start a whole unit later: a unit that still finds a
                // member absent `sync_giveup` windows into its own walk stops waiting for good instead of paying the
                // timeout at every window.
                bool peers = true;
                for (int t = u.t0; t < u.t1; ++t) {
                    // kEpiDiag: the unit's one tile is the gathered label rows of its own query rows
                    const int nrow = (EPI == kEpiDiag ? u.qb * CG * kBlockM : t * kBlockN) + (int)rank * C::kBRows;
                    if (pace && u.members > 1) {
                        const int r = t - u.t0;
                        if (r > 0 && r % p.sync_w == 0) {
                            const int j = r / p.sync_w;                     // window j starts; window j - 1 is issued
                            if (leader) atomicAdd(&pace[j - 1], 1);
                            if (peers && p.sync_giveup > 0 && j == p.sync_lead + p.sync_giveup &&
                                *reinterpret_cast<volatile int32_t*>(&pace[0]) < u.members)
                                peers = false;
                            if (j >= p.sync_lead && peers) {
                                const long long t_start = clock64();
                                while (*reinterpret_cast<volatile int32_t*>(&pace[j - p.sync_lead]) < u.members) {
                                    if (clock64() - t_start > 60000) break;    // ~40 us: give up, never block
                                    __nanosleep(200);
                                }
                            }
                        }
                    }
                    dbg_stamp(p, 0, (uint32_t)(t - u.t0), 0);
#pragma unroll 1
                    for (int kb = 0; kb < p.KB; ++kb, ++kiter) {
                        const int s = kiter % C::kStages;
                        mbar_wait(bar_empty + 8 * s, ((kiter / C::kStages) & 1) ^ 1, 1);
                        if (kb == 0) dbg_stamp(p, 0, (uint32_t)(t - u.t0), 1);
                        if (kb == p.KB - 1) dbg_stamp(p, 0, (uint32_t)(t - u.t0), 2);
                        const uint32_t full = bar_full + 8 * s;
                        const uint32_t sbase = smem_u32(stages + (size_t)s * C::kStageBytes);
                        const uint32_t bytes = (x3 ? 2u : 1u) * (uint32_t)(kABytes + C::kBBytes);
                        if (leader) mbar_arrive_expect_tx(full, bytes * CG);
                        const int kc = kb * C::kElemsPerBlock;
                        if (hint) {
                            tma_load_2d_hint<CG>(sbase, &map_uhi, full, kc, qrow, pol_q);
                            if (hint_items) tma_load_2d_hint<CG>(sbase + (BF16 ? 1 : 2) * kABytes, &map_ihi, full, kc, nrow, pol_i);
                            else tma_load_2d<CG>(sbase + (BF16 ? 1 : 2) * kABytes, &map_ihi, full, kc, nrow);
                            if (x3) {
                                tma_load_2d_hint<CG>(sbase + kABytes, &map_ulo, full, kc, qrow, pol_q);
                                if (hint_items) tma_load_2d_hint<CG>(sbase + 2 * kABytes + C::kBBytes, &map_ilo, full, kc, nrow, pol_i);
                                else tma_load_2d<CG>(sbase + 2 * kABytes + C::kBBytes, &map_ilo, full, kc, nrow);
                            }
                        } else {
                            tma_load_2d<CG>(sbase, &map_uhi, full, kc, qrow);
                            tma_load_2d<CG>(sbase + (BF16 ? 1 : 2) * kABytes, &map_ihi, full, kc, nrow);
                            if (x3) {
                                tma_load_2d<CG>(sbase + kABytes, &map_ulo, full, kc, qrow);
                                tma_load_2d<CG>(sbase + 2 * kABytes + C::kBBytes, &map_ilo, full, kc, nrow);
                            }
                        }
                        if (!leader) mbar_arrive_remote(full, 0);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (leader CTA; one lane issues) =====
        if (leader) {
            constexpr uint32_t idesc = make_idesc<CG, BF16>();
            uint32_t kiter = 0, it = 0;
            Unit u;
            for (int ui = cluster_id; get_unit(p, ui, u); ui += num_clusters) {
                for (int t = u.t0; t < u.t1; ++t, ++it) {
                    const uint32_t acc = it & 1;
                    if (lane == 0) dbg_stamp(p, 1, it, 0);
                    mbar_wait(bar_tempty + 8 * acc, ((it >> 1) & 1) ^ 1, 2);
                    tc_fence_after();
                    if (lane == 0) dbg_stamp(p, 1, it, 1);
                    const uint32_t d_tmem = tmem_base + acc * kBlockN;
#pragma unroll 1
                    for (int kb = 0; kb < p.KB; ++kb, ++kiter) {
                        const int s = kiter % C::kStages;
                        mbar_wait(bar_full + 8 * s, (kiter / C::kStages) & 1, 3);
                        tc_fence_after();
                        if (lane == 0) {
                            const uint32_t sbase = smem_u32(stages + (size_t)s * C::kStageBytes);
                            const uint64_t a_hi = make_smem_desc<BK>(sbase);
                            const uint64_t a_lo = make_smem_desc<BK>(sbase + kABytes);
                            const uint64_t b_hi = make_smem_desc<BK>(sbase + (BF16 ? 1 : 2) * kABytes);
                            const uint64_t b_lo = make_smem_desc<BK>(sbase + 2 * kABytes + C::kBBytes);
#pragma unroll
                            for (int k = 0; k < BK / kUmmaK; ++k) {
                                const uint64_t off = (uint64_t)((k * kUmmaK * 4) >> 4);  // 32 bytes of K per step
                                if (BF16) {
                                    umma_bf16<CG>(d_tmem, a_hi + off, b_hi + off, idesc, (kb | k) != 0);
                                } else if (x3) {
                                    umma_tf32<CG>(d_tmem, a_hi + off, b_lo + off, idesc, (kb | k) != 0);
                                    umma_tf32<CG>(d_tmem, a_lo + off, b_hi + off, idesc, 1u);
                                    umma_tf32<CG>(d_tmem, a_hi + off, b_hi + off, idesc, 1u);
                                } else {
                                    umma_tf32<CG>(d_tmem, a_hi + off, b_hi + off, idesc, (kb | k) != 0);
                                }
                            }
                            umma_commit<CG>(bar_empty + 8 * s);                      // stage consumed
                            if (kb == p.KB - 1) umma_commit<CG>(bar_tfull + 8 * acc);  // accumulator complete
                            if (kb == 0) dbg_stamp(p, 1, it, 2);
                            if (kb == p.KB - 1) dbg_stamp(p, 1, it, 3);
                        }
                        __syncwarp();
                    }
                }
            }
        }
    } else if (EPI != kEpiTopK && warp >= 4) {
        // ===== label-rank epilogue (a discarded branch in the top-K instantiations, whose Params have no label fields)
        if constexpr (EPI == kEpiLse)
            lse_epilogue<CG, BF16, EXCL>(p, tmem_base, bar_tfull, bar_tempty, rank, leader, cluster_id, num_clusters,
                                         warp, lane);
        else if constexpr (EPI != kEpiTopK)
            rank_epilogue<CG, BF16, EXCL, EPI>(p, tmem_base, bar_tfull, bar_tempty, rank, leader, cluster_id, num_clusters,
                                               warp, lane);
    } else if (warp >= 4) {
        // ===== epilogue: TMEM -> threshold filter -> per-row candidate buffers -> sorted top-K =====
        // Group g = (warp - 4) / 4 owns accumulator stage g, i.e. every second tile; warp ew of a group reads TMEM
        // lanes [32 ew, 32 ew + 32).  Each (group, row) keeps its own candidate buffer and threshold; the lists of
        // the two groups are merged with those of the other splits by mr_topk_merge.
        const int grp = (warp - 4) >> 2;
        const int ew = (warp - 4) & 3;
        const int row = ew * 32 + lane;
        u64* warp_buf = p.cand + (((size_t)blockIdx.x * EG + grp) * kBlockM + ew * 32) * kCap;
        u64* my_buf = warp_buf + (size_t)lane * kCap;
        const int K = p.K;
        uint32_t it = 0;
        Unit u;
        for (int ui = cluster_id; get_unit(p, ui, u); ui += num_clusters) {
            const int64_t q = ((int64_t)u.qb * CG + rank) * kBlockM + row;
            const bool active = q < p.Q;
            int cnt = 0;
            uint32_t thr = 0;                        // score key of the row's K-th best so far (0: list not full)
            float thr_f = __int_as_float(0x7FC00000);  // same threshold as a float; NaN = "everything passes"
            // EXCL: cursor into the row's exclusion list, placed on the first id >= the unit's first item; ex_next is
            // the id under the cursor (INT32_MAX past the end: no item id reaches it, since id_base + N < 2^31)
            int64_t ex_cur = 0, ex_end = 0;
            int32_t ex_next = INT32_MAX;
            if constexpr (EXCL) {
                if (active) {
                    ex_cur = p.excl_off[q];
                    ex_end = p.excl_off[q + 1];
                    const int64_t first = (int64_t)p.id_base + (int64_t)u.t0 * kBlockN;
                    for (int64_t hi = ex_end; ex_cur < hi;) {
                        const int64_t mid = (ex_cur + hi) >> 1;
                        if ((int64_t)p.excl_ids[mid] < first) ex_cur = mid + 1; else hi = mid;
                    }
                    if (ex_cur < ex_end) ex_next = p.excl_ids[ex_cur];
                }
            }
            for (int t = u.t0; t < u.t1; ++t, ++it) {
                if (EG > 1 && (int)(it & 1) != grp) continue;   // two groups: group g drains stage g
                const uint32_t acc = it & 1;
                if (threadIdx.x == 128) dbg_stamp(p, 2, it, 0);
                mbar_wait(bar_tfull + 8 * acc, (it >> 1) & 1, 4);
                tc_fence_after();
                if (threadIdx.x == 128) dbg_stamp(p, 2, it, 1);
                const int64_t n0 = (int64_t)t * kBlockN;
                const int nvalid = (int)((p.N - n0) < kBlockN ? (p.N - n0) : kBlockN);
                const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + acc * kBlockN;
                long long t_ld = 0, t_flt = 0, t_cmp = 0;
                int n_cmp = 0;
#pragma unroll 1
                for (int c = 0; c < nvalid; c += kChunk) {
                    uint32_t v[kChunk];
                    const long long c0 = p.dbg ? clock64() : 0;
                    tmem_ld16(taddr + c, v);
                    tmem_ld_wait();
                    const long long c1 = p.dbg ? clock64() : 0;
                    // Phase 1, branch-free: bit j of m = "column c + j may enter the row's list" (cheap superset test:
                    // key(f) > thr implies f > thr_f or f is NaN).  No per-element branches, so the 16 tests overlap.
                    uint32_t m = 0;
#pragma unroll
                    for (int j = 0; j < kChunk; ++j) m |= (!(__uint_as_float(v[j]) <= thr_f)) ? (1u << j) : 0u;
                    if (nvalid - c < kChunk) m &= (1u << (nvalid - c)) - 1u;
                    if (!active) m = 0;
                    // Phase 2: each lane walks its own set bits (usually none), exact key test, append.
                    const uint32_t id0 = (uint32_t)(p.id_base + (int32_t)(n0 + c));
                    while (m) {
                        const int j = __ffs(m) - 1;
                        m &= m - 1;
                        uint32_t bits = v[0];
#pragma unroll
                        for (int jj = 1; jj < kChunk; ++jj) bits = (j == jj) ? v[jj] : bits;
                        if (BF16) {
                            // the reference's bf16 autocast matmul returns bf16 scores: round the fp32 accumulator
                            // (RN-even).  Only survivors of the superset test get here -- rounding is monotone and
                            // thr_f is a bf16 value, so bf16(acc) > thr_f implies acc > thr_f.
                            if ((bits & 0x7F800000u) != 0x7F800000u) bits += 0x7FFFu + ((bits >> 16) & 1u);
                            bits &= 0xFFFF0000u;
                        }
                        const uint32_t key = score_key(__uint_as_float(bits));
                        if constexpr (EXCL) {
                            if (key > thr) {
                                const int32_t id = (int32_t)(id0 + (uint32_t)j);
                                while (ex_next < id) ex_next = ++ex_cur < ex_end ? p.excl_ids[ex_cur] : INT32_MAX;
                                if (ex_next == id) continue;
                            }
                        }
                        if (key > thr) my_buf[cnt++] = ((u64)key << 32) | (u64)(0xFFFFFFFFu - (id0 + (uint32_t)j));
                    }
                    // rows that could overflow on the next chunk are cut back to their best K, two rows per sort
                    unsigned need = __ballot_sync(0xffffffffu, cnt > kCap - kChunk);
                    const long long c2 = p.dbg ? clock64() : 0;
                    n_cmp += __popc(need);
#pragma unroll 1
                    while (need) {
                        const int L0 = __ffs(need) - 1;
                        need &= need - 1;
                        const int L1 = need ? __ffs(need) - 1 : L0;
                        if (need) need &= need - 1;
                        const int na = __shfl_sync(0xffffffffu, cnt, L0), nb = __shfl_sync(0xffffffffu, cnt, L1);
                        u64* ga = warp_buf + (size_t)L0 * kCap;
                        u64* gb = warp_buf + (size_t)L1 * kCap;
                        __syncwarp();   // the appends of lanes L0 / L1 are visible to the whole warp
                        u64 ka[8], kb[8];
                        warp_load_keys(ka, ga, na, lane);
                        warp_load_keys(kb, gb, nb, lane);
                        // K-th largest score key of each row from a 32-bit sort (na, nb > kCap - kChunk >= K here)
                        uint32_t sa[8], sb[8];
#pragma unroll
                        for (int r = 0; r < 8; ++r) { sa[r] = (uint32_t)(ka[r] >> 32); sb[r] = (uint32_t)(kb[r] >> 32); }
                        warp_sort256x2_u32(sa, sb, lane);
                        uint32_t ta = warp_pick32(sa, K - 1), tb = warp_pick32(sb, K - 1);
                        int keepa = warp_keep_ge(ga, ka, ta, lane);
                        int keepb = L1 != L0 ? warp_keep_ge(gb, kb, tb, lane) : keepa;
                        if (keepa != K || keepb != K) {
                            // more than K keys at or above the K-th score (equal scores straddle the cut): the exact
                            // (score, id) order decides -- rare, full 64-bit sort
                            warp_sort256x2(ka, kb, lane);
                            warp_store_keys(ga, ka, K, lane);
                            if (L1 != L0) warp_store_keys(gb, kb, K, lane);
                            keepa = keepb = K;
                        }
                        __syncwarp();
                        if (lane == L0 || lane == L1) {
                            const bool first = lane == L0;
                            cnt = first ? keepa : keepb;
                            thr = first ? ta : tb;
                            thr_f = thr ? key_score((u64)thr << 32) : __int_as_float(0x7FC00000);
                        }
                    }
                    if (p.dbg) {
                        const long long c3 = clock64();
                        t_ld += c1 - c0; t_flt += c2 - c1; t_cmp += c3 - c2;
                    }
                }
                if (p.dbg && blockIdx.x == 0 && threadIdx.x == 128 && it < (uint32_t)kDbgTiles) {
                    p.dbg[(3 * kDbgTiles + it) * kDbgSlots + 0] = t_ld;
                    p.dbg[(3 * kDbgTiles + it) * kDbgSlots + 1] = t_flt;
                    p.dbg[(3 * kDbgTiles + it) * kDbgSlots + 2] = t_cmp;
                    p.dbg[(3 * kDbgTiles + it) * kDbgSlots + 3] = n_cmp;
                }
                // accumulator stage drained: hand it back to the MMA issuer
                if (threadIdx.x == 128) dbg_stamp(p, 2, it, 2);
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if (CG == 1 || leader) mbar_arrive_local(bar_tempty + 8 * acc);
                    else mbar_arrive_remote(bar_tempty + 8 * acc, 0);
                }
            }
            // unit done: final sort of every row (two per call), one (val, id) list per (split, group, q)
#pragma unroll 1
            for (int L = 0; L < 32; L += 2) {
                const int64_t qL = ((int64_t)u.qb * CG + rank) * kBlockM + ew * 32 + L;
                if (qL >= p.Q) break;  // warp-uniform: rows are ascending
                const int na = __shfl_sync(0xffffffffu, cnt, L), nb = __shfl_sync(0xffffffffu, cnt, L + 1);
                __syncwarp();
                u64 ka[8], kb[8];
                warp_load_keys(ka, warp_buf + (size_t)L * kCap, na, lane);
                warp_load_keys(kb, warp_buf + (size_t)(L + 1) * kCap, nb, lane);
                warp_sort256x2(ka, kb, lane);
                const size_t list = (size_t)u.split * EG + grp;
                warp_write_list(p, (list * p.Q + qL) * K, ka, K, lane);
                if (qL + 1 < p.Q) warp_write_list(p, (list * p.Q + qL + 1) * K, kb, K, lane);
                __syncwarp();
            }
        }
    }

    // teardown: everyone (both CTAs of a pair) is done with TMEM and the barriers before they go away
    tc_fence_before();
    if (CG > 1) cluster_sync_all(); else __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        if (CG == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
        else asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    }
}

// ---- host side --------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* sym = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(sym);
    }
    return fn;
}
// (rows, E) fp32 row-major -> boxes of (32 floats, box_rows rows), 128-byte swizzle, zero fill out of bounds
static bool make_map(CUtensorMap* map, const void* ptr, int64_t rows, int E, int box_rows, int bk, bool bf16) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return false;
    cuuint64_t dims[2] = {(cuuint64_t)E, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)E * (bf16 ? 2 : 4)};
    cuuint32_t box[2] = {(cuuint32_t)(bf16 ? 2 * bk : bk), (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    return fn(map, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(ptr), dims, strides,
              box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, bk == 32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
              CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

struct Plan {
    int cg, bk, eg, QB, T, S, QG, grid;
    int64_t cand_bytes, part_bytes, sync_bytes;
    int sync_w, sync_windows;
};
static int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}
// excl: the plan of mr_score_topk_exclude, whose kernels exist only in the default geometry (BK = 32, one epilogue
// group): it ignores the experiment knobs MR_SCORE_BK and MR_SCORE_BF16_EPI_GROUPS.
// rank: the plan of the counting pass (mr_score_rank; K is ignored), same geometry: no top-K warm-up, no merge to
// bound S, and one int32 per (split, row) instead of the lists and candidate buffers.
static Plan make_plan(int64_t Q, int64_t N, int K, bool bf16, bool excl = false, bool rank = false) {
    Plan pl;
    if (rank) { excl = true; K = 1; }
    pl.eg = (!excl && bf16 && env_int("MR_SCORE_BF16_EPI_GROUPS", 1) == 2) ? 2 : 1;
    pl.cg = env_int("MR_SCORE_CTA_GROUP", 2) == 1 ? 1 : 2;
    pl.bk = (!excl && env_int("MR_SCORE_BK", 32) == 16) ? 16 : 32;
    const int sms = sm_count();
    const int clusters = sms / pl.cg;
    pl.QB = (int)((Q + (int64_t)kBlockM * pl.cg - 1) / ((int64_t)kBlockM * pl.cg));
    pl.T = (int)((N + kBlockN - 1) / kBlockN);
    pl.QG = 0;   // set below, once the number of splits is known
    // item splits: each unit pays a top-K warm-up (its first tiles pass everything and trigger bursts of row sorts),
    // measured at roughly (8 + K / 5) tile-times; units are executed in waves of `clusters`.  Pick the S that
    // minimises waves * (tiles per unit + warm-up).
    int smax = rank ? pl.T : 8192 / (pl.eg * (K > 0 ? K : 1));  // mr_topk_merge takes at most 8192 candidates per row
    if (smax > pl.T) smax = pl.T;
    if (smax < 1) smax = 1;
    int s = env_int("MR_SCORE_SPLITS", 0);
    if (s <= 0) {
        // the counting pass keeps the K-independent part: it also stands for the L2 sharing that many small units
        // lose (a wave walks S item streams, each shared by wave / S query blocks)
        const double warm = rank ? 8.0 : 8.0 + K / 5.0;
        double best = 1e300;
        s = 1;
        for (int c = 1; c <= smax; ++c) {
            const int64_t units = (int64_t)pl.QB * c;
            const int64_t waves = (units + clusters - 1) / clusters;
            const double cost = (double)waves * ((double)((pl.T + c - 1) / c) + warm);
            if (cost < best * (1.0 - 1e-9)) { best = cost; s = c; }
        }
    }
    if (s > smax) s = smax;
    pl.S = s;
    // One wave of CTA pairs walks only S item streams (get_unit's wave-aligned order), so an item tile is shared by
    // wave / S query blocks and the query operands of a wave fit L2 next to the item streams (measured at BASELINE
    // config 5 with the L2 eviction hints, as explicit groups QG x S: 37 x 2 -> 443 ms; 16 x 2 -> 447; 18 x 4 -> 466;
    // 8 x 9 -> 481; 74 x 2 -> 548).  MR_SCORE_QGROUP = explicit query groups of that many blocks (experiments).
    pl.QG = env_int("MR_SCORE_QGROUP", 0);
    if (pl.QG < 0) pl.QG = 0;
    const int64_t units = (int64_t)pl.QB * pl.S;
    pl.grid = (int)((units < clusters ? units : clusters) * pl.cg);
    if (pl.grid < pl.cg) pl.grid = pl.cg;
    pl.cand_bytes = rank ? 0 : (int64_t)sms * pl.eg * kBlockM * kCap * 8;
    pl.part_bytes = rank ? (((int64_t)pl.S * Q * 4 + 255) & ~(int64_t)255) : (int64_t)pl.S * pl.eg * Q * K * 8;
    // pacing counters: (query groups x splits) streams x windows of sync_w tiles
    pl.sync_w = env_int("MR_SCORE_PACE_TILES", 1);
    if (pl.sync_w < 1) pl.sync_w = 0;
    const int wave = pl.grid / pl.cg;
    const int groups = pl.QG ? (pl.QB + pl.QG - 1) / pl.QG : (int)((units + wave - 1) / wave);   // streams = groups x S
    pl.sync_windows = pl.sync_w ? ((pl.T + pl.S - 1) / pl.S + pl.sync_w - 1) / pl.sync_w + 2 : 0;
    pl.sync_bytes = pl.sync_w ? (((int64_t)groups * pl.S * pl.sync_windows * 4 + 255) & ~(int64_t)255) : 0;
    return pl;
}

template <int CG, int BK, bool BF16, int EG, bool EXCL = false, int EPI = kEpiTopK, class P = ExclParams>
static int launch(const Plan& pl, const CUtensorMap& muh, const CUtensorMap& mul, const CUtensorMap& mih, const CUtensorMap& mil,
                  const P& p, cudaStream_t stream) {
    using C = Cfg<CG, BK, BF16>;
    cudaError_t e = cudaFuncSetAttribute(score_topk_kernel<CG, BK, BF16, EG, EXCL, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::kSmemBytes);
    if (e != cudaSuccess) { set_error("mr_score_topk: shared memory attribute: %s", cudaGetErrorString(e)); return (int)e; }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)pl.grid);
    cfg.blockDim = dim3(128 + 128 * EG);
    cfg.dynamicSmemBytes = C::kSmemBytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    e = cudaLaunchKernelEx(&cfg, score_topk_kernel<CG, BK, BF16, EG, EXCL, EPI>, muh, mul, mih, mil,
                           static_cast<const KernelParams<EXCL, EPI>&>(p));
    if (e != cudaSuccess) { set_error("mr_score_topk: launch: %s", cudaGetErrorString(e)); return (int)e; }
    return MR_OK;
}

// kEpiDiag operand: dst row q = the item row of labels[q] (src row labels[q] - id_base), zeros when the label is not in
// [id_base, id_base + N); rows of `row_words` 16-byte words.
__global__ void gather_label_rows_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, int64_t Q, int64_t N,
                                         int row_words, int32_t id_base, const int64_t* __restrict__ labels) {
    const int64_t total = Q * row_words, gsz = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gsz) {
        const int64_t q = i / row_words, w = i - q * row_words;
        const int64_t l = labels[q] - id_base;
        dst[i] = (l >= 0 && l < N) ? src[l * row_words + w] : make_uint4(0, 0, 0, 0);
    }
}
// count[q] = the (split, q) counts of kEpiCount summed in split order, -1 for a row without a label key
__global__ void rank_finish_kernel(const int32_t* __restrict__ part, int S, int64_t Q, const uint32_t* __restrict__ label_key,
                                   int32_t* __restrict__ count) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= Q) return;
    int32_t c = 0;
    for (int s = 0; s < S; ++s) c += part[(int64_t)s * Q + q];
    count[q] = label_key[q] ? c : -1;
}
// Merges P (shift, sum) partials of kEpiLse per row, in index order: K = the largest shift, total = the sums aligned to
// it by ldexp (exact) and added in order.  label_key == NULL: writes the merged pair (out_shift, out_sum).  Otherwise
// writes logp[q] = min(0, (L c - K - log2(total)) ln 2) in fp64, stored as fp32, with L the score of the label's key:
// the label's log-probability under the softmax of the merged scores, NaN where the key is 0 (no label).  The min only
// removes the rounding above 0 (the label's own term is inside total) and keeps NaN.
__global__ void lse_finish_kernel(const int32_t* __restrict__ shift, const double* __restrict__ sum, int P, int64_t Q,
                                  const uint32_t* __restrict__ label_key, float lc, int32_t* __restrict__ out_shift,
                                  double* __restrict__ out_sum, float* __restrict__ logp) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= Q) return;
    int K = kLseMinShift;
    for (int i = 0; i < P; ++i) K = max(K, shift[(int64_t)i * Q + q]);
    double total = 0.0;
    for (int i = 0; i < P; ++i) total += ldexp(sum[(int64_t)i * Q + q], shift[(int64_t)i * Q + q] - K);
    if (!label_key) {
        out_shift[q] = K;
        out_sum[q] = total;
        return;
    }
    const uint32_t L = label_key[q];
    if (L == 0) {
        logp[q] = __int_as_float(0x7FC00000);
        return;
    }
    const double x = ((double)key_score((u64)L << 32) * (double)lc - (double)K - log2(total)) * 0.6931471805599453;
    logp[q] = (float)(x > 0.0 ? 0.0 : x);
}
// log2(e) / temperature, rounded once to fp32: the same scale in the epilogue and in the finish
static float lse_scale(float temperature) { return (float)(1.4426950408889634 / (double)temperature); }

// Fields and tensor maps shared by the two label-rank passes.  `items` / `items_lo` are the item operand of the pass
// (the table, or the gathered label rows) with `item_rows` rows.
static int rank_params(RankParams& p, CUtensorMap (&maps)[4], const Plan& pl, const float* Uhi, const float* Ulo, int64_t Q,
                       const void* items, const void* items_lo, int64_t item_rows, int64_t N, int E, int32_t id_base,
                       int mode, const int64_t* labels) {
    const bool bf16 = mode == MR_SCORE_BF16;
    p = RankParams{};
    p.Q = Q; p.N = N; p.E = E; p.K = 1; p.mode = mode; p.id_base = id_base;
    p.KB = (E + (bf16 ? 63 : 31)) / (bf16 ? 64 : 32);
    p.T = pl.T; p.QB = pl.QB; p.S = pl.S; p.QG = pl.QG; p.wave = pl.grid / pl.cg;
    p.l2_hint = env_int("MR_SCORE_L2HINT", 1);
    p.sync_w = pl.sync_w; p.sync_windows = pl.sync_windows;
    p.sync_lead = env_int("MR_SCORE_PACE_LEAD", 1);
    if (p.sync_lead < 1) p.sync_lead = 1;
    p.sync_giveup = env_int("MR_SCORE_PACE_GIVEUP", 8);
    p.labels = labels;
    const int brows = kBlockN / pl.cg;
    bool ok = make_map(&maps[0], Uhi, Q, E, kBlockM, 32, bf16) && make_map(&maps[2], items, item_rows, E, brows, 32, bf16);
    if (ok && mode == MR_SCORE_TF32X3)
        ok = make_map(&maps[1], Ulo, Q, E, kBlockM, 32, false) && make_map(&maps[3], items_lo, item_rows, E, brows, 32, false);
    else if (ok) { maps[1] = maps[0]; maps[3] = maps[2]; }
    if (!ok) { set_error("mr_score_rank: cuTensorMapEncodeTiled failed (driver without TMA support?)"); return MR_ERR_UNSUPPORTED; }
    return MR_OK;
}
template <int EPI, bool EXCL, class P>
static int launch_rank(const Plan& pl, const CUtensorMap (&m)[4], const P& p, bool bf16, cudaStream_t s) {
    if (bf16) return pl.cg == 1 ? launch<1, 32, true, 1, EXCL, EPI>(pl, m[0], m[1], m[2], m[3], p, s)
                                : launch<2, 32, true, 1, EXCL, EPI>(pl, m[0], m[1], m[2], m[3], p, s);
    return pl.cg == 1 ? launch<1, 32, false, 1, EXCL, EPI>(pl, m[0], m[1], m[2], m[3], p, s)
                      : launch<2, 32, false, 1, EXCL, EPI>(pl, m[0], m[1], m[2], m[3], p, s);
}
static int64_t align256(int64_t n) { return (n + 255) & ~(int64_t)255; }
// workspace of the label-score pass: the gathered (hi, lo) label rows
static int64_t diag_bytes(int64_t Q, int E, bool bf16) { return (bf16 ? 1 : 2) * align256(Q * E * (bf16 ? 2 : 4)); }
// partials of the log-sum-exp pass on the counting pass's plan: (S, Q) fp64 sums, then (S, Q) int32 shifts
static int64_t lse_part_bytes(const Plan& pl, int64_t Q) { return align256(pl.S * Q * 8) + align256(pl.S * Q * 4); }

}  // namespace st
}  // namespace mr

static thread_local long long* g_score_dbg = nullptr;
extern "C" int mr_score_topk_debug_buffer(void* dev_buf, int64_t bytes) {
    using namespace mr;
    MR_REQUIRE(dev_buf == nullptr || bytes >= (int64_t)(4 * st::kDbgTiles * st::kDbgSlots * 8),
               "mr_score_topk_debug_buffer: need %d bytes", 4 * st::kDbgTiles * st::kDbgSlots * 8);
    g_score_dbg = reinterpret_cast<long long*>(dev_buf);
    return MR_OK;
}

// Host-only view of the static schedule (no CUDA call: the plan and get_unit are plain arithmetic).
extern "C" int64_t mr_score_topk_schedule(int64_t Q, int64_t N, int K, int mode, int32_t* plan_out, int32_t* units_out,
                                          int64_t max_units) {
    using namespace mr;
    if (Q < 1 || N < 1 || K < 1 || K > MR_MAX_FUSED_TOPK || !plan_out) {
        set_error("mr_score_topk_schedule: need Q, N >= 1, 1 <= K <= %d and plan_out", MR_MAX_FUSED_TOPK);
        return MR_ERR_INVALID_ARG;
    }
    const st::Plan pl = st::make_plan(Q, N, K, mode == MR_SCORE_BF16);
    st::Params p{};
    p.T = pl.T; p.QB = pl.QB; p.S = pl.S; p.QG = pl.QG; p.wave = pl.grid / pl.cg;
    const int64_t U = (int64_t)pl.QB * pl.S;
    const int groups = pl.QG ? (pl.QB + pl.QG - 1) / pl.QG : (int)((U + p.wave - 1) / p.wave);
    const int32_t plan[8] = {pl.QB, pl.T, pl.S, p.wave, pl.cg, groups * pl.S, pl.sync_windows, pl.sync_w};
    for (int i = 0; i < 8; ++i) plan_out[i] = plan[i];
    if (units_out) {
        for (int64_t u = 0; u < U && u < max_units; ++u) {
            st::Unit un;
            st::get_unit(p, (int)u, un);
            int32_t* o = units_out + u * 6;
            o[0] = un.qb; o[1] = un.split; o[2] = un.t0; o[3] = un.t1; o[4] = un.stream; o[5] = un.members;
        }
    }
    return U;
}

extern "C" int64_t mr_score_topk_workspace_bytes(int64_t Q, int64_t N, int E, int K) {
    using namespace mr;
    if (Q < 0 || N < 0 || E < 1 || K < 1 || K > MR_MAX_FUSED_TOPK) {
        set_error("mr_score_topk_workspace_bytes: need Q, N >= 0, E >= 1, 1 <= K <= %d", MR_MAX_FUSED_TOPK);
        return MR_ERR_INVALID_ARG;
    }
    if (Q == 0) return 0;
    // sized for the mode that needs the most scratch (bf16-compat: two epilogue groups), so one query serves every mode
    const st::Plan pa = st::make_plan(Q, N, K, false), pb = st::make_plan(Q, N, K, true);
    const int64_t a = pa.cand_bytes + pa.part_bytes + pa.sync_bytes, b = pb.cand_bytes + pb.part_bytes + pb.sync_bytes;
    return (a > b ? a : b) + 256;
}

// mr_score_topk (excl_off == NULL) and mr_score_topk_exclude
static int score_topk_impl(const float* Uhi, const float* Ulo, int64_t Q, const float* Ihi, const float* Ilo, int64_t N,
                           int E, int K, int32_t id_base, int mode, float* out_val, int32_t* out_id, void* ws,
                           int64_t ws_bytes, mr_stream_t stream, const int64_t* excl_off, const int32_t* excl_ids) {
    using namespace mr;
    const bool excl = excl_off != nullptr;
    MR_REQUIRE(Q >= 0 && N >= 0 && E >= 1, "mr_score_topk: need Q, N >= 0 and E >= 1");
    MR_REQUIRE(K >= 1 && K <= MR_MAX_FUSED_TOPK, "mr_score_topk: K=%d outside [1,%d]", K, MR_MAX_FUSED_TOPK);
    MR_REQUIRE(mode == MR_SCORE_TF32X3 || mode == MR_SCORE_TF32X1 || mode == MR_SCORE_BF16, "mr_score_topk: unknown mode %d", mode);
    const bool bf16 = mode == MR_SCORE_BF16;
    MR_REQUIRE(E % (bf16 ? 8 : 4) == 0, "mr_score_topk: E=%d must be a multiple of %d (16-byte rows for TMA)", E, bf16 ? 8 : 4);
    MR_REQUIRE(Q < (1ll << 31) - 512 && N < (1ll << 31) - 512 && (int64_t)id_base + N < (1ll << 31),
               "mr_score_topk: Q, N and id_base + N must fit 31 bits");
    if (Q == 0) return MR_OK;
    MR_REQUIRE(Uhi && Ihi && out_val && out_id, "mr_score_topk: null pointer");
    MR_REQUIRE(mode != MR_SCORE_TF32X3 || (Ulo && Ilo), "mr_score_topk: the 3xTF32 mode needs the lo operands");
    MR_REQUIRE(host_aligned16(Uhi) && host_aligned16(Ihi) && host_aligned16(Ulo) && host_aligned16(Ilo),
               "mr_score_topk: operands must be 16-byte aligned");
    cudaStream_t s = (cudaStream_t)stream;
    if (N == 0) {  // nothing to score: every list is empty
        cudaError_t e = cudaMemsetAsync(out_id, 0xFF, (size_t)Q * K * 4, s);
        if (e == cudaSuccess) e = cudaMemsetAsync(out_val, 0xFF, (size_t)Q * K * 4, s);  // NaN payload; ids say "empty"
        if (e != cudaSuccess) { set_error("mr_score_topk: memset: %s", cudaGetErrorString(e)); return (int)e; }
        return MR_OK;
    }
    const st::Plan pl = st::make_plan(Q, N, K, bf16, excl);
    const int64_t need = pl.cand_bytes + pl.part_bytes + pl.sync_bytes + 256;
    if (!ws || ws_bytes < need) {
        set_error("mr_score_topk: workspace of %lld bytes needed, %lld given", (long long)need, (long long)ws_bytes);
        return MR_ERR_WORKSPACE;
    }
    unsigned char* w = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
    st::ExclParams p;
    p.Q = Q; p.N = N; p.E = E; p.K = K; p.mode = mode; p.id_base = id_base;
    const int bk = bf16 ? 32 : pl.bk;                 // bf16 rows are 64 elements = 128 bytes: the BK = 32 geometry
    const int kelems = bf16 ? 64 : bk;
    p.KB = (E + kelems - 1) / kelems;
    p.T = pl.T; p.QB = pl.QB; p.S = pl.S; p.QG = pl.QG; p.wave = pl.grid / pl.cg;
    p.cand = reinterpret_cast<mr::u64*>(w);
    p.dbg = g_score_dbg;
    p.l2_hint = st::env_int("MR_SCORE_L2HINT", 1);
    p.sync = nullptr; p.sync_w = pl.sync_w; p.sync_windows = pl.sync_windows;
    p.sync_lead = st::env_int("MR_SCORE_PACE_LEAD", 1);   // lead 1 / 2 / 3 at config 5: 376.5 / 379.6 / 381.2 ms
    if (p.sync_lead < 1) p.sync_lead = 1;
    p.sync_giveup = st::env_int("MR_SCORE_PACE_GIVEUP", 8);
    if (pl.sync_bytes) {
        p.sync = reinterpret_cast<int32_t*>(w + pl.cand_bytes + pl.part_bytes);
        cudaError_t e = cudaMemsetAsync(p.sync, 0, (size_t)pl.sync_bytes, s);
        if (e != cudaSuccess) { set_error("mr_score_topk: memset: %s", cudaGetErrorString(e)); return (int)e; }
    }
    float* part_val = reinterpret_cast<float*>(w + pl.cand_bytes);
    int32_t* part_id = reinterpret_cast<int32_t*>(w + pl.cand_bytes + pl.part_bytes / 2);
    p.out_val = part_val;
    p.out_id = part_id;
    p.excl_off = excl_off;
    p.excl_ids = excl_ids;

    CUtensorMap muh, mul, mih, mil;
    const int brows = st::kBlockN / pl.cg;
    bool ok = st::make_map(&muh, Uhi, Q, E, st::kBlockM, bk, bf16) && st::make_map(&mih, Ihi, N, E, brows, bk, bf16);
    if (ok && mode == MR_SCORE_TF32X3)
        ok = st::make_map(&mul, Ulo, Q, E, st::kBlockM, bk, false) && st::make_map(&mil, Ilo, N, E, brows, bk, false);
    else if (ok) { mul = muh; mil = mih; }
    if (!ok) { set_error("mr_score_topk: cuTensorMapEncodeTiled failed (driver without TMA support?)"); return MR_ERR_UNSUPPORTED; }

    int rc;
    if (excl && bf16) rc = pl.cg == 1 ? st::launch<1, 32, true, 1, true>(pl, muh, mul, mih, mil, p, s) : st::launch<2, 32, true, 1, true>(pl, muh, mul, mih, mil, p, s);
    else if (excl) rc = pl.cg == 1 ? st::launch<1, 32, false, 1, true>(pl, muh, mul, mih, mil, p, s) : st::launch<2, 32, false, 1, true>(pl, muh, mul, mih, mil, p, s);
    else if (bf16 && pl.eg == 2) rc = pl.cg == 1 ? st::launch<1, 32, true, 2>(pl, muh, mul, mih, mil, p, s) : st::launch<2, 32, true, 2>(pl, muh, mul, mih, mil, p, s);
    else if (bf16) rc = pl.cg == 1 ? st::launch<1, 32, true, 1>(pl, muh, mul, mih, mil, p, s) : st::launch<2, 32, true, 1>(pl, muh, mul, mih, mil, p, s);
    else if (bk == 32) rc = pl.cg == 1 ? st::launch<1, 32, false, 1>(pl, muh, mul, mih, mil, p, s) : st::launch<2, 32, false, 1>(pl, muh, mul, mih, mil, p, s);
    else rc = pl.cg == 1 ? st::launch<1, 16, false, 1>(pl, muh, mul, mih, mil, p, s) : st::launch<2, 16, false, 1>(pl, muh, mul, mih, mil, p, s);
    if (rc != MR_OK) return rc;
    return mr_topk_merge(part_val, part_id, pl.S * pl.eg, Q, K, K, out_val, out_id, stream);
}

extern "C" int mr_score_topk(const float* Uhi, const float* Ulo, int64_t Q, const float* Ihi, const float* Ilo, int64_t N,
                             int E, int K, int32_t id_base, int mode, float* out_val, int32_t* out_id, void* ws,
                             int64_t ws_bytes, mr_stream_t stream) {
    return score_topk_impl(Uhi, Ulo, Q, Ihi, Ilo, N, E, K, id_base, mode, out_val, out_id, ws, ws_bytes, stream, nullptr,
                           nullptr);
}

extern "C" int mr_score_topk_exclude(const float* Uhi, const float* Ulo, int64_t Q, const float* Ihi, const float* Ilo,
                                     int64_t N, int E, int K, int32_t id_base, int mode, float* out_val, int32_t* out_id,
                                     void* ws, int64_t ws_bytes, const int64_t* excl_off, const int32_t* excl_ids,
                                     mr_stream_t stream) {
    MR_REQUIRE(excl_off && excl_ids, "mr_score_topk_exclude: null pointer (excl_off / excl_ids)");
    return score_topk_impl(Uhi, Ulo, Q, Ihi, Ilo, N, E, K, id_base, mode, out_val, out_id, ws, ws_bytes, stream, excl_off,
                           excl_ids);
}

// ---- label rank against the whole catalog ------------------------------------------------------------------------
static int rank_check(const char* who, const float* Uhi, const float* Ulo, int64_t Q, const float* Ihi, const float* Ilo,
                      int64_t N, int E, int32_t id_base, int mode) {
    using namespace mr;
    MR_REQUIRE(Q >= 0 && N >= 0 && E >= 1, "%s: need Q, N >= 0 and E >= 1", who);
    MR_REQUIRE(mode == MR_SCORE_TF32X3 || mode == MR_SCORE_TF32X1 || mode == MR_SCORE_BF16, "%s: unknown mode %d", who, mode);
    const bool bf16 = mode == MR_SCORE_BF16;
    MR_REQUIRE(E % (bf16 ? 8 : 4) == 0, "%s: E=%d must be a multiple of %d (16-byte rows for TMA)", who, E, bf16 ? 8 : 4);
    MR_REQUIRE(Q < (1ll << 31) - 512 && N < (1ll << 31) - 512 && (int64_t)id_base + N < (1ll << 31),
               "%s: Q, N and id_base + N must fit 31 bits", who);
    if (Q == 0) return MR_OK;
    MR_REQUIRE(Uhi && Ihi, "%s: null pointer", who);
    MR_REQUIRE(mode != MR_SCORE_TF32X3 || (Ulo && Ilo), "%s: the 3xTF32 mode needs the lo operands", who);
    MR_REQUIRE(host_aligned16(Uhi) && host_aligned16(Ihi) && host_aligned16(Ulo) && host_aligned16(Ilo),
               "%s: operands must be 16-byte aligned", who);
    return MR_OK;
}

extern "C" int64_t mr_score_rank_workspace_bytes(int64_t Q, int64_t N, int E) {
    using namespace mr;
    if (Q < 0 || N < 0 || E < 1) {
        set_error("mr_score_rank_workspace_bytes: need Q, N >= 0 and E >= 1");
        return MR_ERR_INVALID_ARG;
    }
    if (Q == 0) return 0;
    // one scratch for both passes and every mode: the gathered fp32 (hi, lo) label rows, or the counting pass's counts
    // (the plan mr_score_rank builds: N = 0 plans as N = 1)
    const st::Plan pl = st::make_plan(Q, N > 0 ? N : 1, 1, false, true, true);
    const int64_t a = st::diag_bytes(Q, E, false), b = pl.part_bytes + pl.sync_bytes;
    return (a > b ? a : b) + 256;
}

extern "C" int mr_label_score(const float* Uhi, const float* Ulo, int64_t Q, const float* Ihi, const float* Ilo, int64_t N,
                              int E, int32_t id_base, int mode, const int64_t* labels, uint32_t* label_key, void* ws,
                              int64_t ws_bytes, mr_stream_t stream) {
    using namespace mr;
    int rc = rank_check("mr_label_score", Uhi, Ulo, Q, Ihi, Ilo, N, E, id_base, mode);
    if (rc != MR_OK || Q == 0) return rc;
    MR_REQUIRE(labels && label_key, "mr_label_score: null pointer");
    cudaStream_t s = (cudaStream_t)stream;
    if (N == 0) {
        cudaError_t e = cudaMemsetAsync(label_key, 0, (size_t)Q * 4, s);
        if (e != cudaSuccess) { set_error("mr_label_score: memset: %s", cudaGetErrorString(e)); return (int)e; }
        return MR_OK;
    }
    const bool bf16 = mode == MR_SCORE_BF16;
    const int64_t need = st::diag_bytes(Q, E, bf16) + 256;
    if (!ws || ws_bytes < need) {
        set_error("mr_label_score: workspace of %lld bytes needed, %lld given", (long long)need, (long long)ws_bytes);
        return MR_ERR_WORKSPACE;
    }
    unsigned char* w = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
    const int row_bytes = E * (bf16 ? 2 : 4);
    void* ghi = w;
    void* glo = w + st::align256(Q * row_bytes);
    int64_t blocks = (Q * (row_bytes / 16) + 255) / 256;
    const int64_t cap = (int64_t)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    st::gather_label_rows_kernel<<<(unsigned)blocks, 256, 0, s>>>(reinterpret_cast<const uint4*>(Ihi), reinterpret_cast<uint4*>(ghi),
                                                                  Q, N, row_bytes / 16, id_base, labels);
    if (mode == MR_SCORE_TF32X3)
        st::gather_label_rows_kernel<<<(unsigned)blocks, 256, 0, s>>>(reinterpret_cast<const uint4*>(Ilo),
                                                                      reinterpret_cast<uint4*>(glo), Q, N, row_bytes / 16,
                                                                      id_base, labels);
    MR_CUDA_LAUNCH_CHECK("mr_label_score");
    // one unit per query block, one tile each: the block's own gathered label rows
    st::Plan pl{};
    pl.cg = st::env_int("MR_SCORE_CTA_GROUP", 2) == 1 ? 1 : 2;
    pl.bk = 32; pl.eg = 1;
    pl.QB = (int)((Q + (int64_t)st::kBlockM * pl.cg - 1) / ((int64_t)st::kBlockM * pl.cg));
    pl.T = 1; pl.S = 1; pl.QG = 0;
    const int clusters = sm_count() / pl.cg;
    pl.grid = (pl.QB < clusters ? pl.QB : clusters) * pl.cg;
    st::RankParams p;
    CUtensorMap maps[4];
    rc = st::rank_params(p, maps, pl, Uhi, Ulo, Q, ghi, glo, Q, N, E, id_base, mode, labels);
    if (rc != MR_OK) return rc;
    p.out_key = label_key;
    return st::launch_rank<st::kEpiDiag, false>(pl, maps, p, bf16, s);
}

extern "C" int mr_score_rank(const float* Uhi, const float* Ulo, int64_t Q, const float* Ihi, const float* Ilo, int64_t N,
                             int E, int32_t id_base, int mode, const int64_t* labels, const uint32_t* label_key,
                             const int64_t* excl_off, const int32_t* excl_ids, int32_t* count, void* ws, int64_t ws_bytes,
                             mr_stream_t stream) {
    using namespace mr;
    MR_REQUIRE((excl_off == nullptr) == (excl_ids == nullptr),
               "mr_score_rank: excl_off and excl_ids must both be NULL or both be set");
    int rc = rank_check("mr_score_rank", Uhi, Ulo, Q, Ihi, Ilo, N, E, id_base, mode);
    if (rc != MR_OK || Q == 0) return rc;
    MR_REQUIRE(labels && label_key && count, "mr_score_rank: null pointer");
    cudaStream_t s = (cudaStream_t)stream;
    const st::Plan pl = st::make_plan(Q, N > 0 ? N : 1, 1, mode == MR_SCORE_BF16, true, true);
    const int64_t need = pl.part_bytes + pl.sync_bytes + 256;
    if (!ws || ws_bytes < need) {
        set_error("mr_score_rank: workspace of %lld bytes needed, %lld given", (long long)need, (long long)ws_bytes);
        return MR_ERR_WORKSPACE;
    }
    unsigned char* w = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
    int32_t* part = reinterpret_cast<int32_t*>(w);
    if (N > 0) {
        st::RankParams p;
        CUtensorMap maps[4];
        rc = st::rank_params(p, maps, pl, Uhi, Ulo, Q, Ihi, Ilo, N, N, E, id_base, mode, labels);
        if (rc != MR_OK) return rc;
        p.label_key = label_key;
        p.part = part;
        p.excl_off = excl_off;
        p.excl_ids = excl_ids;
        if (pl.sync_bytes) {
            p.sync = reinterpret_cast<int32_t*>(w + pl.part_bytes);
            cudaError_t e = cudaMemsetAsync(p.sync, 0, (size_t)pl.sync_bytes, s);
            if (e != cudaSuccess) { set_error("mr_score_rank: memset: %s", cudaGetErrorString(e)); return (int)e; }
        }
        rc = excl_off ? st::launch_rank<st::kEpiCount, true>(pl, maps, p, mode == MR_SCORE_BF16, s)
                      : st::launch_rank<st::kEpiCount, false>(pl, maps, p, mode == MR_SCORE_BF16, s);
        if (rc != MR_OK) return rc;
    }
    st::rank_finish_kernel<<<(unsigned)((Q + 255) / 256), 256, 0, s>>>(part, N > 0 ? pl.S : 0, Q, label_key, count);
    MR_CUDA_LAUNCH_CHECK("mr_score_rank");
    return MR_OK;
}

// ---- log-sum-exp of each query's scores over the whole catalog ----------------------------------------------------
extern "C" int64_t mr_score_lse_workspace_bytes(int64_t Q, int64_t N, int E) {
    using namespace mr;
    if (Q < 0 || N < 0 || E < 1) {
        set_error("mr_score_lse_workspace_bytes: need Q, N >= 0 and E >= 1");
        return MR_ERR_INVALID_ARG;
    }
    if (Q == 0) return 0;
    // the plan mr_score_lse builds (N = 0 plans as N = 1); the sync counters do not depend on the mode
    const st::Plan pl = st::make_plan(Q, N > 0 ? N : 1, 1, false, true, true);
    return st::lse_part_bytes(pl, Q) + pl.sync_bytes + 256;
}

extern "C" int mr_score_lse(const float* Uhi, const float* Ulo, int64_t Q, const float* Ihi, const float* Ilo, int64_t N,
                            int E, int32_t id_base, int mode, float temperature, const int64_t* excl_off,
                            const int32_t* excl_ids, int32_t* shift, double* sum, void* ws, int64_t ws_bytes,
                            mr_stream_t stream) {
    using namespace mr;
    MR_REQUIRE((excl_off == nullptr) == (excl_ids == nullptr),
               "mr_score_lse: excl_off and excl_ids must both be NULL or both be set");
    MR_REQUIRE(temperature > 0.0f && temperature < INFINITY, "mr_score_lse: temperature must be finite and > 0");
    // N = 0: no item operand is read (an empty table may hand in NULL), only the empty partials are written
    int rc = rank_check("mr_score_lse", Uhi, Ulo, Q, N > 0 ? Ihi : Uhi, N > 0 ? Ilo : Ulo, N, E, id_base, mode);
    if (rc != MR_OK || Q == 0) return rc;
    MR_REQUIRE(shift && sum, "mr_score_lse: null pointer");
    cudaStream_t s = (cudaStream_t)stream;
    const st::Plan pl = st::make_plan(Q, N > 0 ? N : 1, 1, mode == MR_SCORE_BF16, true, true);
    const int64_t part_bytes = st::lse_part_bytes(pl, Q);
    const int64_t need = part_bytes + pl.sync_bytes + 256;
    if (!ws || ws_bytes < need) {
        set_error("mr_score_lse: workspace of %lld bytes needed, %lld given", (long long)need, (long long)ws_bytes);
        return MR_ERR_WORKSPACE;
    }
    unsigned char* w = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
    double* psum = reinterpret_cast<double*>(w);
    int32_t* pshift = reinterpret_cast<int32_t*>(w + st::align256(pl.S * Q * 8));
    const float lc = st::lse_scale(temperature);
    if (N > 0) {
        st::LseParams p;
        CUtensorMap maps[4];
        rc = st::rank_params(p, maps, pl, Uhi, Ulo, Q, Ihi, Ilo, N, N, E, id_base, mode, nullptr);
        if (rc != MR_OK) return rc;
        p.lse_c = lc;
        p.lse_shift = pshift;
        p.lse_sum = psum;
        p.excl_off = excl_off;
        p.excl_ids = excl_ids;
        if (pl.sync_bytes) {
            p.sync = reinterpret_cast<int32_t*>(w + part_bytes);
            cudaError_t e = cudaMemsetAsync(p.sync, 0, (size_t)pl.sync_bytes, s);
            if (e != cudaSuccess) { set_error("mr_score_lse: memset: %s", cudaGetErrorString(e)); return (int)e; }
        }
        rc = excl_off ? st::launch_rank<st::kEpiLse, true>(pl, maps, p, mode == MR_SCORE_BF16, s)
                      : st::launch_rank<st::kEpiLse, false>(pl, maps, p, mode == MR_SCORE_BF16, s);
        if (rc != MR_OK) return rc;
    }
    // the S splits merged in split order (none for N = 0: the empty pair)
    st::lse_finish_kernel<<<(unsigned)((Q + 255) / 256), 256, 0, s>>>(pshift, psum, N > 0 ? pl.S : 0, Q, nullptr, lc,
                                                                       shift, sum, nullptr);
    MR_CUDA_LAUNCH_CHECK("mr_score_lse");
    return MR_OK;
}

extern "C" int mr_lse_finish(const int32_t* shift, const double* sum, int64_t P, int64_t Q, const uint32_t* label_key,
                             float temperature, float* logp, mr_stream_t stream) {
    using namespace mr;
    MR_REQUIRE(P >= 0 && P < (1 << 20) && Q >= 0 && Q < (1ll << 40), "mr_lse_finish: need 0 <= P < 2^20 and Q >= 0");
    MR_REQUIRE(temperature > 0.0f && temperature < INFINITY, "mr_lse_finish: temperature must be finite and > 0");
    if (Q == 0) return MR_OK;
    MR_REQUIRE(label_key && logp && (P == 0 || (shift && sum)), "mr_lse_finish: null pointer");
    st::lse_finish_kernel<<<(unsigned)((Q + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        shift, sum, (int)P, Q, label_key, st::lse_scale(temperature), nullptr, nullptr, logp);
    MR_CUDA_LAUNCH_CHECK("mr_lse_finish");
    return MR_OK;
}
