// ties.cu -- TIES magnitude trim, sign election and disjoint mean (SURVEY.md section 8(a): A6-A9).
//
// reference: rec_retrieval/merger/algorithms/ties.py
//   _compute_sparse_updates :8-28   keep the int(density*d) largest |m_k - base| over the WHOLE flat vector
//   _compute_final_sign     :31-52  sign vote from the fp32 sums of positive / negative survivors
//   get_ties_vectors        :55-72  survivors that agree with the elected sign, divided by their count
//   merge_ties              :75-83  base + sum_k trim_k(w_k * (m_k - base))   (no election, no mean)
//
// The trim is an exact order statistic.  Elements are ordered by the composite 64-bit key
//     key(u, j) = (bits(|u|) << 32) | (0xFFFFFFFF - j)            (larger |u| first, then LOWER index first)
// and model k keeps element j iff key >= cut[k], where cut[k] is the k_cnt-th largest key: the canonical
// tie rule of SURVEY.md section 0.1-D3 (torch.topk's own order among equal magnitudes is unspecified).
//
// Selection = "bracket and refine" on the key space, all with one streaming pass kernel:
//   fast path (stream-ordered, no host sync):
//     1. two passes over a strided sample (~0.5 M elements per model) narrow [0, 2^63) to a bracket that
//        holds the target with overwhelming probability (+-6 sigma of the sample quantile);
//     2. ONE pass over the full data counts the keys above the bracket exactly, histograms the keys inside
//        it (1024 linear bins) and stores them (~0.75 % of d) in per-CTA candidate lists;
//     3. pick the bin holding rank k_cnt, compact its candidates (<= 4096) and sort them in shared memory.
//   exact path (any input, e.g. millions of equal magnitudes; synchronous): full passes that narrow the
//     bracket 1024x each (at most 7) until the survivors fit, then steps 2-3.
// The full pass reads base + K models once ((K+1)*d*4 bytes, HBM-bound: a subtract, an AND and two compares
// per element; no atomics outside the bracket).  The build kernels read them once more and write the result.
#include <math.h>
#include <stdlib.h>

#include "common.cuh"

namespace mr {

typedef unsigned long long u64;

constexpr int kTiesBins = 1024;
constexpr int kTiesThreads = 256;
constexpr int kTiesFinalCap = 4096;
constexpr int64_t kTiesSampleQuads = 131072;  // ~0.5 M sampled elements per model (2 M narrows the bracket 2x but its two
                                              // sample passes cost more than the full pass gains: 1.44 vs 1.23 ms measured)

struct TiesState {  // one per model
    u64 lo, hi;      // inclusive bracket on composite keys
    u64 above;       // keys > hi seen by the last pass (written by pick from the pass counters)
    u64 in_bracket;  // keys inside the refined bracket
    int shift;       // bin = (key - lo) >> shift  (< kTiesBins)
    int status;      // 0 searching, 1 done, < 0 failed
};

enum {
    TIES_ST_SEARCH = 0,
    TIES_ST_DONE = 1,
    TIES_ERR_BRACKET_LOW = -1,   // more than k_cnt - 1 keys above the bracket
    TIES_ERR_BRACKET_HIGH = -2,  // target below the bracket
    TIES_ERR_TOO_MANY = -3,      // refined bracket does not fit the final sort
    TIES_ERR_CAND_OVERFLOW = -4, // a per-CTA candidate list overflowed
    TIES_ERR_INCONSISTENT = -5,
};

__device__ __forceinline__ u64 ties_key(uint32_t mag, int64_t j) {
    return ((u64)mag << 32) | (u64)(0xFFFFFFFFu - (uint32_t)j);
}
__device__ __forceinline__ int shift_for(u64 width /* hi - lo */) {
    int s = 0;
    while ((width >> s) >= (u64)kTiesBins) ++s;
    return s;
}

// ---- state init -----------------------------------------------------------------------------------
static __global__ void ties_init_kernel(TiesState* st, int K, u64* cut, int32_t* status, int64_t k_cnt, int64_t d) {
    const int k = threadIdx.x;
    if (k >= K) return;
    TiesState s;
    s.lo = 0;
    s.hi = ((u64)0x7FFFFFFFu << 32) | 0xFFFFFFFFull;
    s.above = 0;
    s.in_bracket = (u64)d;
    s.shift = shift_for(s.hi - s.lo);
    s.status = TIES_ST_SEARCH;
    if (k_cnt <= 0) { cut[k] = ~(u64)0; s.status = TIES_ST_DONE; }       // keep nothing
    else if (k_cnt >= d) { cut[k] = 0; s.status = TIES_ST_DONE; }        // keep everything
    if (st) st[k] = s;
    status[k] = s.status;
}

// ---- the pass kernel ------------------------------------------------------------------------------
struct PassCounters {
    uint32_t* hist;      // K * kTiesBins
    u64* above;          // K
    uint32_t* cand_cnt;  // K * n_threads (COLLECT): one private candidate list per thread and model
    u64* cand_keys;      // K * n_threads * cand_cap
    int cand_cap;
    int64_t j_off;       // global index of local element 0 (sharded select: keys carry GLOBAL indices); 0 otherwise
    u64* sample_keys;    // optional, sample passes only: the composite key of every sampled element, (K, sample_ld); the
    int64_t sample_ld;   // second look at the same sample then reads this contiguous cache instead of striding again
};

// Shared-memory layout of the pass kernel (dynamic): hist[K][bins] u32 | lo[K] hi[K] u64 | shift[K] i32 |
// lom[K] span[K] i32 | cn[K] notabove[K] ge[K] u32
template <int K>
struct PassSmem {
    uint32_t* hist; u64* lo; u64* hi; int* shift; int* lom; int* span; uint32_t* cn; uint32_t* notabove; uint32_t* ge;
    __device__ __forceinline__ explicit PassSmem(unsigned char* raw) {
        hist = reinterpret_cast<uint32_t*>(raw);
        lo = reinterpret_cast<u64*>(hist + K * kTiesBins);
        hi = lo + K;
        shift = reinterpret_cast<int*>(hi + K);
        lom = shift + K;
        span = lom + K;
        cn = reinterpret_cast<uint32_t*>(span + K);
        notabove = cn + K;
        ge = notabove + K;
    }
    static constexpr size_t bytes() { return (size_t)K * kTiesBins * 4 + (size_t)K * (8 + 8 + 4 * 6) + 16; }
};

// Rare path (the magnitude lies inside [lo_mag, hi_mag]): exact 64-bit classification against the bracket.
template <int K, bool COLLECT>
__device__ __noinline__ void ties_pass_edge(unsigned char* raw, uint32_t mag, int64_t j, int k, u64* cand_keys,
                                            int cand_cap) {
    PassSmem<K> sm(raw);
    const u64 key = ties_key(mag, j);
    if (key > sm.hi[k]) return;                 // above the bracket after all (already counted by the caller)
    atomicAdd(&sm.notabove[k], 1u);
    if (key < sm.lo[k]) return;                 // below it
    const uint32_t bin = (uint32_t)((key - sm.lo[k]) >> sm.shift[k]);
    atomicAdd(&sm.hist[k * kTiesBins + bin], 1u);
    (void)cand_keys; (void)cand_cap;   // keys are only stored by the inline COLLECT path of the pass kernel
}

// One streaming pass: per model, count the keys above the bracket, histogram (and optionally store) the keys inside.
// Per element and model the common path is FSUB, AND, ISUB, compare+count, compare+branch; everything 64-bit lives
// in ties_pass_edge.  VEC: all pointers 16-byte aligned (128-bit loads); otherwise scalar loads.
template <int K, bool VEC, bool W, int COLLECT>
__global__ void __launch_bounds__(kTiesThreads, K <= 8 ? 3 : 2)
ties_pass_kernel(const float* __restrict__ base, PtrPack<K> models, int64_t d, const float* __restrict__ w,
                 int64_t stride, const TiesState* __restrict__ st, PassCounters pc) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    PassSmem<K> sm(smem_raw);
    for (int i = threadIdx.x; i < K * kTiesBins; i += blockDim.x) sm.hist[i] = 0;
    if (threadIdx.x < K) {
        const TiesState s = st[threadIdx.x];
        sm.lo[threadIdx.x] = s.lo;
        sm.hi[threadIdx.x] = s.hi;
        sm.shift[threadIdx.x] = s.shift;
        sm.lom[threadIdx.x] = (int)(uint32_t)(s.lo >> 32);
        sm.span[threadIdx.x] = (int)((uint32_t)(s.hi >> 32) - (uint32_t)(s.lo >> 32));
        sm.cn[threadIdx.x] = 0;
        sm.notabove[threadIdx.x] = 0;
        sm.ge[threadIdx.x] = 0;
    }
    __syncthreads();

    uint32_t below[K];  // per-thread count of magnitudes < lo_mag (fits 32 bits: d < 2^32)
    uint32_t visited = 0;  // elements this thread looked at
    uint32_t mycnt[K];     // COLLECT: keys appended to this thread's private candidate lists
    uint32_t nab[K];       // COLLECT == 2: keys with a window magnitude that lie below the bracket
    float wreg[K];
    int lom[K];      // bracket bounds in registers: the edge call may touch shared memory, so values read through
    uint32_t span[K];  // `sm` would be reloaded from shared memory for every element
#pragma unroll
    for (int k = 0; k < K; ++k) {
        below[k] = 0;
        mycnt[k] = 0;
        nab[k] = 0;
        wreg[k] = W ? w[k] : 1.0f;
        lom[k] = sm.lom[k];
        span[k] = (uint32_t)sm.span[k];
    }

    const int64_t nq_full = d >> 2;                        // quads of 4 consecutive elements
    const int64_t nq = (d + 3) >> 2;                       // ... including a partial last one
    // sample passes (stride > 1, always even): one jittered pick per stride window, and a pick is a PAIR of quads -- the
    // 32-byte DRAM sector a 16-byte quad costs anyway -- taken by two adjacent threads
    const int64_t nsq = stride > 1 ? 2 * ((nq + stride - 1) / stride) : nq;   // sampled quads
    const int64_t gtid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t gsz = (int64_t)gridDim.x * blockDim.x;

// Common path per element and model: FSUB, AND, ISUB, one add of the sign bit, one compare OR-ed into a predicate.
// `below[k]` counts magnitudes < lo_mag; `hit` collects "some element of this quad lies inside [lo_mag, hi_mag]".
#define MR_TIES_MAG(K_, X_, B_, MAG_)                                           \
    do {                                                                        \
        float u_ = __fsub_rn((X_), (B_));                                       \
        if (W) u_ = __fmul_rn(u_, wreg[K_]);                                    \
        (MAG_) = __float_as_uint(u_) & 0x7FFFFFFFu;                             \
        const uint32_t t_ = (MAG_) - (uint32_t)lom[K_];                         \
        below[K_] += t_ >> 31; /* lo_mag, mag < 2^31: the sign bit is mag < lo_mag */ \
        hit |= t_ <= span[K_];                                                  \
    } while (0)
// Rare path.  COLLECT (the one full pass of the fast path): classify against the 64-bit bracket inline, count
// "not above" in a register and append the key to this thread's private list -- no atomics and no histogram, so
// the warp never waits on a shared-memory round trip; the histogram of the ~0.7 % collected keys is built
// afterwards by ties_cand_hist_kernel (which also corrects the "above" counter).  Otherwise (sample / exact passes, which
// need the histogram and store nothing): the out-of-line ties_pass_edge.
#define MR_TIES_EDGE(K_, MAG_, J_)                                              \
    do {                                                                        \
        if ((MAG_) - (uint32_t)lom[K_] <= span[K_]) {                           \
            if (COLLECT == 1) {                                                 \
                /* fast path: every key whose MAGNITUDE lies in [lo_mag, hi_mag] goes to the thread-private list: */ \
                /* no atomic, no shared-memory read, no 64-bit classification here -- ties_cand_hist_kernel sorts */ \
                /* the few keys outside [lo, hi] (an end magnitude, index on the wrong side) into above / ignore. */ \
                /* Millions of equal magnitudes overflow the lists: reported, and the exact path takes over.       */ \
                if (mycnt[K_] < (uint32_t)pc.cand_cap)                          \
                    pc.cand_keys[((size_t)(K_) * gsz + gtid) * pc.cand_cap + mycnt[K_]] = ties_key((MAG_), (J_) + pc.j_off); \
                ++mycnt[K_];                                                    \
            } else if (COLLECT == 2) {                                          \
                /* exact path (bracket already narrowed to <= cand_cap keys): classify against the 64-bit ends */ \
                const u64 key_ = ties_key((MAG_), (J_) + pc.j_off);             \
                if (key_ < sm.lo[K_]) {                                         \
                    ++nab[K_]; /* below the bracket: not "above", and not collected (the hist kernel cannot see it) */ \
                } else if (key_ <= sm.hi[K_]) {                                 \
                    if (mycnt[K_] < (uint32_t)pc.cand_cap)                      \
                        pc.cand_keys[((size_t)(K_) * gsz + gtid) * pc.cand_cap + mycnt[K_]] = key_; \
                    ++mycnt[K_];                                                \
                }                                                               \
            } else {                                                            \
                ties_pass_edge<K, false>(smem_raw, (MAG_), (J_) + pc.j_off, (K_), pc.cand_keys, pc.cand_cap); \
            }                                                                   \
        }                                                                       \
    } while (0)

    for (int64_t i = gtid; i < nsq; i += gsz) {
        int64_t q = i;
        if (stride > 1) {  // jitter inside the stride window so the sample does not alias with row pitches
            const int64_t pos = i >> 1;
            q = pos * stride + (int64_t)((((uint32_t)pos * 2654435761u) >> 8) % (uint32_t)stride);
            q = (q & ~(int64_t)1) + (i & 1);
            if (q >= nq) {           // the last window may be cut short
                if (pc.sample_keys)
#pragma unroll
                    for (int k = 0; k < K; ++k)
#pragma unroll
                        for (int c = 0; c < 4; ++c) pc.sample_keys[(size_t)k * pc.sample_ld + i * 4 + c] = 0;   // 0 = no element
                continue;
            }
        }
        const int64_t j0 = q << 2;
        if (VEC && q < nq_full) {
            const float4 b4 = ldg_stream4(base + j0);
            float4 xs[K];
#pragma unroll
            for (int k = 0; k < K; ++k) xs[k] = ldg_stream4(models.p[k] + j0);
#pragma unroll
            for (int k = 0; k < K; ++k) {
                uint32_t m0, m1, m2, m3;
                bool hit = false;
                MR_TIES_MAG(k, xs[k].x, b4.x, m0);
                MR_TIES_MAG(k, xs[k].y, b4.y, m1);
                MR_TIES_MAG(k, xs[k].z, b4.z, m2);
                MR_TIES_MAG(k, xs[k].w, b4.w, m3);
                if (hit) {  // rare: one branch per model and quad instead of one per element
                    MR_TIES_EDGE(k, m0, j0);
                    MR_TIES_EDGE(k, m1, j0 + 1);
                    MR_TIES_EDGE(k, m2, j0 + 2);
                    MR_TIES_EDGE(k, m3, j0 + 3);
                }
                if (stride > 1 && pc.sample_keys) {
                    u64* sk = pc.sample_keys + (size_t)k * pc.sample_ld + i * 4;
                    sk[0] = ties_key(m0, j0 + pc.j_off);
                    sk[1] = ties_key(m1, j0 + 1 + pc.j_off);
                    sk[2] = ties_key(m2, j0 + 2 + pc.j_off);
                    sk[3] = ties_key(m3, j0 + 3 + pc.j_off);
                }
            }
            visited += 4;
        } else {
            const int nvalid = (int)((d - j0) < 4 ? (d - j0) : 4);
            for (int c = 0; c < nvalid; ++c) {
                const float b = base[j0 + c];
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    uint32_t m0;
                    bool hit = false;
                    MR_TIES_MAG(k, models.p[k][j0 + c], b, m0);
                    if (hit) MR_TIES_EDGE(k, m0, j0 + c);
                    if (stride > 1 && pc.sample_keys) pc.sample_keys[(size_t)k * pc.sample_ld + i * 4 + c] = ties_key(m0, j0 + c + pc.j_off);
                }
            }
            if (stride > 1 && pc.sample_keys)
                for (int c = nvalid; c < 4; ++c)
#pragma unroll
                    for (int k = 0; k < K; ++k) pc.sample_keys[(size_t)k * pc.sample_ld + i * 4 + c] = 0;
            visited += (uint32_t)nvalid;
        }
    }
#undef MR_TIES_MAG
#undef MR_TIES_EDGE

    // above = (#magnitudes >= lo_mag) - (#of those that turned out not to be above the bracket); in a COLLECT pass the
    // second term is subtracted later by ties_cand_hist_kernel, which sees every collected key
#pragma unroll
    for (int k = 0; k < K; ++k) {
        uint32_t v = visited - below[k] - nab[k];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
        if ((threadIdx.x & 31) == 0 && v) atomicAdd(&sm.ge[k], v);
    }
    __syncthreads();
    if (threadIdx.x < K) {
        const uint32_t v = sm.ge[threadIdx.x] - sm.notabove[threadIdx.x];
        if (v) atomicAdd(&pc.above[threadIdx.x], (u64)v);
    }
    if (COLLECT) {
#pragma unroll
        for (int k = 0; k < K; ++k) pc.cand_cnt[(size_t)k * gsz + gtid] = mycnt[k];
    }
    for (int i = threadIdx.x; i < K * kTiesBins; i += blockDim.x) {
        const uint32_t v = sm.hist[i];
        if (v) atomicAdd(&pc.hist[i], v);
    }
}

// ---- histogram of the keys collected by the full pass (replaces per-element histogram atomics in that pass) ----------
static __global__ void __launch_bounds__(256)
ties_cand_hist_kernel(const TiesState* __restrict__ st, const uint32_t* __restrict__ cand_cnt,
                      const u64* __restrict__ cand_keys, int cand_cap, int n_lists, uint32_t* __restrict__ hist,
                      u64* __restrict__ above /* NULL: refinement level, histogram only */) {
    __shared__ uint32_t s_hist[kTiesBins];
    __shared__ uint32_t s_not_above;
    const int k = blockIdx.y;
    const TiesState s = st[k];
    if (s.status != TIES_ST_SEARCH) return;
    for (int i = threadIdx.x; i < kTiesBins; i += blockDim.x) s_hist[i] = 0;
    if (threadIdx.x == 0) s_not_above = 0;
    __syncthreads();
    uint32_t not_above = 0;   // collected keys <= hi: the pass counted every collected key as "above"
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < n_lists; c += gridDim.x * blockDim.x) {   // one list per thread
        uint32_t n = cand_cnt[(size_t)k * n_lists + c];
        if (n > (uint32_t)cand_cap) n = (uint32_t)cand_cap;   // overflow is reported by ties_compact_kernel
        const u64* keys = cand_keys + ((size_t)k * n_lists + c) * cand_cap;
        for (uint32_t e = 0; e < n; ++e) {
            const u64 key = keys[e];     // magnitude inside [lo_mag, hi_mag]; the key itself may fall just outside [lo, hi]
            if (key > s.hi) continue;
            ++not_above;
            if (key >= s.lo) atomicAdd(&s_hist[(uint32_t)((key - s.lo) >> s.shift)], 1u);
        }
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) not_above += __shfl_xor_sync(0xffffffffu, not_above, off);
    if ((threadIdx.x & 31) == 0 && not_above) atomicAdd(&s_not_above, not_above);
    __syncthreads();
    for (int i = threadIdx.x; i < kTiesBins; i += blockDim.x) {
        const uint32_t v = s_hist[i];
        if (v) atomicAdd(&hist[k * kTiesBins + i], v);
    }
    if (above && threadIdx.x == 0 && s_not_above) atomicAdd(&above[k], (u64)0 - (u64)s_not_above);   // two's-complement subtract
}

// ---- second look at the sparse sample: histogram of the cached keys inside the current bracket ------------------------------
// Same counters as a sample pass over the data would produce (hist of the keys in [lo, hi], `above` = keys > hi), read
// from the contiguous key cache the first pass wrote (34 MB at K = 8) instead of striding over the K + 1 vectors again.
static __global__ void __launch_bounds__(256)
ties_keys_hist_kernel(const TiesState* __restrict__ st, const u64* __restrict__ keys, int64_t ld, int64_t n,
                      uint32_t* __restrict__ hist, u64* __restrict__ above) {
    __shared__ uint32_t s_hist[kTiesBins];
    __shared__ uint32_t s_above;
    const int k = blockIdx.y;
    const TiesState s = st[k];
    if (s.status != TIES_ST_SEARCH) return;
    for (int i = threadIdx.x; i < kTiesBins; i += blockDim.x) s_hist[i] = 0;
    if (threadIdx.x == 0) s_above = 0;
    __syncthreads();
    uint32_t ab = 0;
    const u64* row = keys + (size_t)k * ld;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const u64 key = row[i];
        if (key == 0) continue;                    // slot without an element (cut-short last window)
        if (key > s.hi) ++ab;
        else if (key >= s.lo) atomicAdd(&s_hist[(uint32_t)((key - s.lo) >> s.shift)], 1u);
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) ab += __shfl_xor_sync(0xffffffffu, ab, off);
    if ((threadIdx.x & 31) == 0 && ab) atomicAdd(&s_above, ab);
    __syncthreads();
    for (int i = threadIdx.x; i < kTiesBins; i += blockDim.x) {
        const uint32_t v = s_hist[i];
        if (v) atomicAdd(&hist[k * kTiesBins + i], v);
    }
    if (threadIdx.x == 0 && s_above) atomicAdd(&above[k], (u64)s_above);
}

// ---- pick: turn a histogram into a narrower bracket ---------------------------------------------------
// rank_hi <= rank_lo are 1-based ranks (largest key = rank 1) in the population the pass visited.  The new
// bracket spans the bins holding rank_hi .. rank_lo.  strict: both ranks must fall inside the old bracket
// (exact passes, rank_hi == rank_lo == k_cnt); otherwise they are clamped to it (sample passes).
static __global__ void __launch_bounds__(kTiesBins)
ties_pick_kernel(TiesState* st, const uint32_t* __restrict__ hist, const u64* __restrict__ above_ctr, int64_t rank_hi,
                 int64_t rank_lo, int strict, int32_t* status) {
    __shared__ u64 s_suffix[kTiesBins + 1];
    __shared__ u64 s_warp[kTiesBins / 32];
    __shared__ int s_bhi, s_blo;
    const int k = blockIdx.x;
    TiesState s = st[k];
    if (s.status != TIES_ST_SEARCH) return;
    const int t = threadIdx.x;           // thread t owns bin (bins - 1 - t): an inclusive prefix scan over t
    const int bin = kTiesBins - 1 - t;   // is an inclusive suffix sum over bins
    u64 v = hist[k * kTiesBins + bin];
    // warp inclusive scan
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const u64 n = __shfl_up_sync(0xffffffffu, v, off);
        if ((t & 31) >= off) v += n;
    }
    if ((t & 31) == 31) s_warp[t >> 5] = v;
    if (t == 0) { s_bhi = -1; s_blo = -1; }
    __syncthreads();
    if (t < 32) {
        u64 x = s_warp[t];
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const u64 n = __shfl_up_sync(0xffffffffu, x, off);
            if (t >= off) x += n;
        }
        s_warp[t] = x;
    }
    __syncthreads();
    if (t >= 32) v += s_warp[(t >> 5) - 1];
    s_suffix[bin] = v;  // keys in bins >= bin
    if (t == 0) s_suffix[kTiesBins] = 0;
    __syncthreads();
    const u64 above = above_ctr ? above_ctr[k] : s.above;   // refinement level: keys above the bracket are known
    const u64 total_in = s_suffix[0];
    // bin holding rank r: the largest b with above + suffix[b] >= r
    const u64 ge = above + s_suffix[bin], gt = above + s_suffix[bin + 1];
    if (ge >= (u64)rank_hi && gt < (u64)rank_hi) s_bhi = bin;
    if (ge >= (u64)rank_lo && gt < (u64)rank_lo) s_blo = bin;
    __syncthreads();
    if (t == 0) {
        int bhi = s_bhi, blo = s_blo;
        int err = 0;
        // a rank outside the bracket is clamped to its end bins (sample passes).  The top end is the bin holding hi, not
        // bin kTiesBins - 1: a bracket narrower than 1024 << shift leaves the upper bins empty, and a bracket made of one
        // of them would start above hi -- an inverted bracket whose magnitude window wraps and takes in almost every key
        // of the vector in the full pass
        const int top = (int)((s.hi - s.lo) >> s.shift);
        if (bhi < 0) {  // rank_hi above the bracket (<= above) or below it
            if ((u64)rank_hi <= above) { if (strict) err = TIES_ERR_BRACKET_LOW; bhi = top; }
            else { if (strict) err = TIES_ERR_BRACKET_HIGH; bhi = 0; }
        }
        if (blo < 0) {
            if ((u64)rank_lo <= above) { if (strict) err = TIES_ERR_BRACKET_LOW; blo = top; }
            else { if (strict) err = TIES_ERR_BRACKET_HIGH; blo = 0; }
        }
        if (rank_hi < 1) bhi = top;
        if (err) {
            s.status = err;
        } else {
            const u64 new_lo = s.lo + ((u64)blo << s.shift);
            u64 new_hi = s.lo + (((u64)bhi + 1) << s.shift) - 1;
            if (new_hi > s.hi || bhi == top) new_hi = s.hi;
            s.above = above + s_suffix[bhi + 1];
            s.in_bracket = s_suffix[blo] - s_suffix[bhi + 1];
            s.lo = new_lo;
            s.hi = new_hi;
            s.shift = shift_for(new_hi - new_lo);
        }
        (void)total_in;
        st[k] = s;
        status[k] = s.status;
    }
}

// ---- compact the candidates of the refined bracket ------------------------------------------------------
static __global__ void __launch_bounds__(256)
ties_compact_kernel(TiesState* st, const uint32_t* __restrict__ cand_cnt, const u64* __restrict__ cand_keys,
                    int cand_cap, int n_lists, uint32_t* fin_cnt, u64* fin_keys, int32_t* status) {
    const int k = blockIdx.y;
    if (st[k].status != TIES_ST_SEARCH) return;
    const u64 lo = st[k].lo, hi = st[k].hi;
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < n_lists; c += gridDim.x * blockDim.x) {   // one list per thread
        const uint32_t n = cand_cnt[(size_t)k * n_lists + c];
        if (n > (uint32_t)cand_cap) {
            st[k].status = TIES_ERR_CAND_OVERFLOW;
            status[k] = TIES_ERR_CAND_OVERFLOW;
            continue;
        }
        const u64* keys = cand_keys + ((size_t)k * n_lists + c) * cand_cap;
        for (uint32_t e = 0; e < n; ++e) {
            const u64 key = keys[e];
            if (key >= lo && key <= hi) {
                const uint32_t pos = atomicAdd(&fin_cnt[k], 1u);
                if (pos < (uint32_t)kTiesFinalCap) fin_keys[(size_t)k * kTiesFinalCap + pos] = key;
            }
        }
    }
}

// ---- final: sort the <= 4096 survivors in shared memory and read off the cut -------------------------------
static __global__ void __launch_bounds__(1024)
ties_final_kernel(TiesState* st, const uint32_t* __restrict__ fin_cnt, const u64* __restrict__ fin_keys, int64_t k_cnt,
                  u64* cut, int32_t* status) {
    __shared__ u64 s_keys[kTiesFinalCap];
    const int k = blockIdx.x;
    TiesState s = st[k];
    if (s.status != TIES_ST_SEARCH) return;
    const uint32_t n = fin_cnt[k];
    const long long r = (long long)k_cnt - (long long)s.above;  // 1-based rank inside the bracket
    int err = 0;
    if (n > (uint32_t)kTiesFinalCap) err = TIES_ERR_TOO_MANY;
    else if ((u64)n != s.in_bracket || r < 1 || r > (long long)n) err = TIES_ERR_INCONSISTENT;
    if (err) {
        if (threadIdx.x == 0) { st[k].status = err; status[k] = err; }
        return;
    }
    int cap2 = 2;                                  // sort only as many slots as the survivors need (block-uniform)
    while (cap2 < (int)n) cap2 <<= 1;
    for (int i = threadIdx.x; i < cap2; i += blockDim.x)
        s_keys[i] = (i < (int)n) ? fin_keys[(size_t)k * kTiesFinalCap + i] : 0;  // real keys are > 0 ... or equal 0 only
    __syncthreads();                                                              // for (mag 0, j = 2^32-1): harmless
    for (int size = 2; size <= cap2; size <<= 1) {               // bitonic sort, descending
        for (int strd = size >> 1; strd > 0; strd >>= 1) {
            for (int i = threadIdx.x; i < cap2 / 2; i += blockDim.x) {
                const int a = 2 * i - (i & (strd - 1));
                const int b = a + strd;
                const bool desc = ((a & size) == 0);
                const u64 x = s_keys[a], y = s_keys[b];
                if ((x < y) == desc) { s_keys[a] = y; s_keys[b] = x; }
            }
            __syncthreads();
        }
    }
    if (threadIdx.x == 0) {
        cut[k] = s_keys[r - 1];
        st[k].status = TIES_ST_DONE;
        status[k] = TIES_ST_DONE;
    }
}

// ---- sharded select (flat vector split over ranks): final sort over the survivors of ALL ranks ---------------------------
// gathered: `world` copies of the [fin_keys (K x cap) | fin_cnt (K, padded)] region, rank-major (what one all-gather of
// every rank's region leaves).  Keys carry global indices, so the r-th largest of the union is the global cut; each rank
// then rewrites it for its own slice: an element at the cut magnitude survives iff its GLOBAL index <= the cut's.
static __global__ void __launch_bounds__(1024)
ties_final_dist_kernel(TiesState* st, const unsigned char* __restrict__ gathered, int world, size_t region_bytes,
                       size_t cnt_off, int64_t k_cnt, int64_t j_off, u64* cut_local, u64* cut_global, int32_t* status) {
    __shared__ u64 s_keys[kTiesFinalCap];
    __shared__ uint32_t s_base[65];
    const int k = blockIdx.x;
    TiesState s = st[k];
    if (s.status != TIES_ST_SEARCH) {
        if (threadIdx.x == 0 && s.status == TIES_ST_DONE && cut_global) cut_global[k] = cut_local[k];   // trivial cuts
        return;
    }
    if (threadIdx.x == 0) {
        uint32_t tot = 0;
        for (int r = 0; r < world && r < 64; ++r) {
            s_base[r] = tot;
            tot += reinterpret_cast<const uint32_t*>(gathered + (size_t)r * region_bytes + cnt_off)[k];
        }
        s_base[world < 64 ? world : 64] = tot;
    }
    __syncthreads();
    const uint32_t n = s_base[world < 64 ? world : 64];
    const long long r = (long long)k_cnt - (long long)s.above;
    int err = 0;
    if (n > (uint32_t)kTiesFinalCap) err = TIES_ERR_TOO_MANY;
    else if ((u64)n != s.in_bracket || r < 1 || r > (long long)n) err = TIES_ERR_INCONSISTENT;
    if (err) {
        if (threadIdx.x == 0) { st[k].status = err; status[k] = err; }
        return;
    }
    int cap2 = 2;
    while (cap2 < (int)n) cap2 <<= 1;
    for (int i = threadIdx.x; i < cap2; i += blockDim.x) s_keys[i] = 0;
    __syncthreads();
    for (int rk = 0; rk < world && rk < 64; ++rk) {
        const u64* keys = reinterpret_cast<const u64*>(gathered + (size_t)rk * region_bytes) + (size_t)k * kTiesFinalCap;
        const uint32_t c = s_base[rk + 1] - s_base[rk];
        for (uint32_t i = threadIdx.x; i < c; i += blockDim.x) s_keys[s_base[rk] + i] = keys[i];
    }
    __syncthreads();
    for (int size = 2; size <= cap2; size <<= 1) {
        for (int strd = size >> 1; strd > 0; strd >>= 1) {
            for (int i = threadIdx.x; i < cap2 / 2; i += blockDim.x) {
                const int a = 2 * i - (i & (strd - 1));
                const int b = a + strd;
                const bool desc = ((a & size) == 0);
                const u64 x = s_keys[a], y = s_keys[b];
                if ((x < y) == desc) { s_keys[a] = y; s_keys[b] = x; }
            }
            __syncthreads();
        }
    }
    if (threadIdx.x == 0) {
        const u64 g = s_keys[r - 1];
        if (cut_global) cut_global[k] = g;
        // local form: same magnitude, index limit shifted into this rank's coordinates
        const u64 mag = g >> 32;
        const long long jg = (long long)(0xFFFFFFFFu - (uint32_t)g);      // global index of the last survivor at `mag`
        const long long jl = jg - (long long)j_off;
        u64 c;
        if (jl < 0) c = (mag + 1) << 32;                                   // none of my elements at `mag` survives
        else c = (mag << 32) | (u64)(0xFFFFFFFFu - (uint32_t)(jl > 0xFFFFFFFFll ? 0xFFFFFFFFll : jl));
        cut_local[k] = c;
        st[k].status = TIES_ST_DONE;
        status[k] = TIES_ST_DONE;
    }
}

// ---- build kernels (A6-A9) ----------------------------------------------------------------------------------
enum { TIES_MODE_VECTORS = 0, TIES_MODE_TRIMSUM = 1, TIES_MODE_FUSED_MERGE = 2, TIES_MODE_LNS = 3 };

struct BuildArgs {
    float* out;           // VECTORS: That (K rows, ldo).  TRIMSUM / FUSED_MERGE: merged (d)
    int64_t ldo;
    uint8_t* trim_mask;   // optional (K, d) bytes
    uint8_t* elect_mask;  // optional (K, d) bytes
    const float* w;       // TRIMSUM: (K) weights applied before the trim.  FUSED_MERGE: (G, K) lambdas
    const int64_t* seg_end;   // FUSED_MERGE with P > 1
    const int32_t* seg_group;
    int P;
};

// x / c for an integer count c in [1, 16], bit-identical to IEEE division (ties.py:68, `div_`): one reciprocal
// multiply plus a Markstein FMA correction.  Exhaustively checked against x / c for every fp32 mantissa and
// c = 2..16 (DESIGN.md "TIES build"; c = 1 is exact by construction: q0 = x, r = 0).  The correction needs the
// quotient and the residual to stay normal, so a column whose survivors could leave [2^-100, 2^100] takes the IEEE
// divide instead: survivors are bounded below by their model's cut magnitude (a kernel-wide flag) and above by
// the elected same-sign sum (one compare per column; inf / NaN fail it too).
__constant__ float c_inv_count[MR_MAX_K + 1] = {1.0f,        1.0f,        1.0f / 2,  1.0f / 3,  1.0f / 4,  1.0f / 5,
                                                1.0f / 6,    1.0f / 7,    1.0f / 8,  1.0f / 9,  1.0f / 10, 1.0f / 11,
                                                1.0f / 12,   1.0f / 13,   1.0f / 14, 1.0f / 15, 1.0f / 16};
__device__ __forceinline__ float div_by_count_fast(float x, float fc, float inv) {
    const float q0 = __fmul_rn(x, inv);
    const float r = __fmaf_rn(-q0, fc, x);
    return __fmaf_rn(r, inv, q0);
}

// Sign election and disjoint mean of one column from its TRIMMED updates s[k] (0 where model k was trimmed): ties.py:31-72.
template <int K, bool TAIL>
__device__ __forceinline__ void ties_elect(const float (&s)[K], bool lo_ok, float (&res)[K], uint32_t& elect_bits) {
    float pp[K], nn[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
        pp[k] = fmaxf(s[k], 0.0f);           // ties.py:35 torch.where(s > 0, s, 0): -0.0 and NaN become +0.0 either way
        nn[k] = s[k] < 0.0f ? s[k] : 0.0f;   // ties.py:36 (fminf would keep a -0.0)
    }
    const float pos = torch_sum_dim0<K>(pp, TAIL);
    const float neg = torch_sum_dim0<K>(nn, TAIL);
    const float t = __fadd_rn(pos, neg);
    // both sums non-zero: the larger magnitude wins, ties go to + (ties.py:41-45); otherwise sign(pos + neg) with
    // 0 -> +1 (ties.py:47-50).  A NaN sum compares false and elects minus, as in the previous formulation.
    const bool both = (pos != 0.0f) && (neg != 0.0f);
    const bool plus = both ? (fabsf(pos) >= fabsf(neg)) : (t >= 0.0f);
    int cnt = 0;
    elect_bits = 0;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        res[k] = plus ? pp[k] : nn[k];        // ties.py:61-65
        const bool nz = res[k] != 0.0f;
        cnt += nz ? 1 : 0;
        elect_bits |= (nz ? 1u : 0u) << k;
    }
    // ties.py:68-70: x / cnt (cnt == 0: all zeros stay zero; cnt == 1: exact)
    const float fc = (float)(cnt > 1 ? cnt : 1);
    const float bound = fabsf(plus ? pos : neg);
    if (lo_ok && bound < 0x1p100f) {
        const float inv = c_inv_count[cnt];
#pragma unroll
        for (int k = 0; k < K; ++k) res[k] = div_by_count_fast(res[k], fc, inv);
    } else {
#pragma unroll
        // (+ 0.0f: the compiler may turn the `s < 0 ? s : 0` select above into a min, which keeps the sign of a
        //  -0.0 update; the reference's torch.where yields +0.0 there.  The fast path maps -0.0 to +0.0 by itself.)
        for (int k = 0; k < K; ++k) res[k] = __fadd_rn(__fdiv_rn(res[k], fc), 0.0f);
    }
}

// One flat column: trim, sign election, disjoint mean (or the trimmed sum for merge_ties).
// TAIL = false: the column lies in the sequential part of torch.sum(dim=0) (every column when K <= 4).
// The hot path is branch-free apart from the (never taken in practice) IEEE-divide escape.
template <int K, int MODE, bool TAIL>
__device__ __forceinline__ void ties_column(const float (&x)[K], float b, int64_t j, const u64 (&cut)[K], bool lo_ok,
                                            const float* __restrict__ wk, float (&res)[K], uint32_t& trim_bits,
                                            uint32_t& elect_bits) {
    float s[K];
    float uu[K];
    trim_bits = 0;
    elect_bits = 0;
    const uint32_t jl = 0xFFFFFFFFu - (uint32_t)j;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        float u = __fsub_rn(x[k], b);
        if (MODE == TIES_MODE_TRIMSUM) u = __fmul_rn(u, wk[k]);
        const u64 key = ((u64)(__float_as_uint(u) & 0x7FFFFFFFu) << 32) | (u64)jl;
        const bool keep = key >= cut[k];
        s[k] = keep ? u : 0.0f;
        uu[k] = u;
        trim_bits |= (keep ? 1u : 0u) << k;
    }
    if constexpr (MODE == TIES_MODE_LNS) {
        // Localize-and-Stitch (localize_and_stitch.py:33-46): mask_k = 1 on the top-k% of |tau_k|; processed mask =
        // mask / max(#active masks, 1) (an fp32 division of 1.0 or 0.0), result = processed mask * tau (a product, so
        // an unselected entry keeps tau's sign on its zero).
        const float inv = c_inv_count[__popc(trim_bits)];
        elect_bits = trim_bits;
#pragma unroll
        for (int k = 0; k < K; ++k) res[k] = __fmul_rn(((trim_bits >> k) & 1u) ? inv : 0.0f, uu[k]);
    } else if constexpr (MODE == TIES_MODE_TRIMSUM) {
        res[0] = __fadd_rn(b, torch_sum_dim0<K>(s, TAIL));   // ties.py:81-83
    } else {
        ties_elect<K, TAIL>(s, lo_ok, res, elect_bits);
    }
}

// Block table of the FUSED_MERGE mode, staged in shared memory.
struct FusedSegs {
    const float* w;        // (G, K) lambdas
    const int64_t* end;    // P ascending exclusive block ends (P > 1)
    const int32_t* grp;    // P group ids
    int P;
};

// One quad (4 consecutive flat columns) of the build pass.
// COLD = false: hot path -- all four columns exist and lie in the sequential part of torch.sum(dim=0).
// COLD = true : the few remaining quads (a partial last quad, the <= 31 trailing columns that use the interleaved
//               summation order when K >= 5); same arithmetic with per-column validity / tail decisions.
template <int K, int MODE, bool VEC, bool MASKS, bool COLD>
__device__ __forceinline__ void ties_quad(const float* __restrict__ base, const PtrPack<K>& models, int64_t d, int64_t q,
                                          const u64 (&cut)[K], bool lo_ok, const float (&wk)[K], const BuildArgs& a,
                                          const FusedSegs& fs, int& hint) {
    const int64_t j0 = q << 2;
    const int64_t tail0 = d & ~(int64_t)31;
    const int nvalid = COLD ? (int)((d - j0) < 4 ? (d - j0) : 4) : 4;
    const bool full = VEC && nvalid == 4;
    float bx[4];
    float xs[K][4];
    if (full) {
        const float4 b4 = ldg_stream4(base + j0);
        bx[0] = b4.x; bx[1] = b4.y; bx[2] = b4.z; bx[3] = b4.w;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const float4 v = ldg_stream4(models.p[k] + j0);
            xs[k][0] = v.x; xs[k][1] = v.y; xs[k][2] = v.z; xs[k][3] = v.w;
        }
    } else {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const bool ok = c < nvalid;
            bx[c] = ok ? base[j0 + c] : 0.0f;
#pragma unroll
            for (int k = 0; k < K; ++k) xs[k][c] = ok ? models.p[k][j0 + c] : 0.0f;
        }
    }
    float res[4][K];
    uint32_t tb[4], eb[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        float x[K];
#pragma unroll
        for (int k = 0; k < K; ++k) x[k] = xs[k][c];
        // the interleaved torch.sum order only exists for K >= 5 and only on the last d mod 32 columns
        if (COLD && K >= 5 && j0 + c >= tail0)
            ties_column<K, MODE, true>(x, bx[c], j0 + c, cut, lo_ok, wk, res[c], tb[c], eb[c]);
        else
            ties_column<K, MODE, false>(x, bx[c], j0 + c, cut, lo_ok, wk, res[c], tb[c], eb[c]);
    }
    if (MODE == TIES_MODE_VECTORS || MODE == TIES_MODE_LNS) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            float* o = a.out + (int64_t)k * a.ldo + j0;
            if (full) stg_stream4(o, make_float4(res[0][k], res[1][k], res[2][k], res[3][k]));
            else
#pragma unroll
                for (int c = 0; c < 4; ++c) if (c < nvalid) o[c] = res[c][k];
        }
    } else if (MODE == TIES_MODE_TRIMSUM) {
        float* o = a.out + j0;
        if (full) stg_stream4(o, make_float4(res[0][0], res[1][0], res[2][0], res[3][0]));
        else
#pragma unroll
            for (int c = 0; c < 4; ++c) if (c < nvalid) o[c] = res[c][0];
    } else {  // FUSED_MERGE: base + sum_dim0_k(w[g,k] * That[k])  (layer_wise.py:76-82 order, blocks = tensors)
        float r[4];
        int p = 0;
        if (fs.end) {
            // first block with end > j0
            if (!(j0 < fs.end[hint] && (hint == 0 || j0 >= fs.end[hint - 1]))) {
                int lo = 0, hi = fs.P - 1;
                while (lo < hi) { const int mid = (lo + hi) >> 1; if (fs.end[mid] > j0) hi = mid; else lo = mid + 1; }
                hint = lo;
            }
            p = hint;
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            bool tail;
            const float* wrow = fs.w;
            if (fs.end) {
                while (c < nvalid && j0 + c >= fs.end[p]) ++p;
                const int64_t beg = p ? fs.end[p - 1] : 0;
                const int64_t n = fs.end[p] - beg;
                tail = (K >= 5) && ((j0 + c - beg) >= (n & ~(int64_t)31));
                wrow = fs.w + fs.grp[p] * K;
            } else {
                tail = (K >= 5) && (j0 + c >= tail0);
            }
            float prod[K];
#pragma unroll
            for (int k = 0; k < K; ++k) prod[k] = __fmul_rn(wrow[k], res[c][k]);
            r[c] = __fadd_rn(bx[c], torch_sum_dim0<K>(prod, tail));
        }
        float* o = a.out + j0;
        if (full) stg_stream4(o, make_float4(r[0], r[1], r[2], r[3]));
        else
#pragma unroll
            for (int c = 0; c < 4; ++c) if (c < nvalid) o[c] = r[c];
    }
    if (MASKS) {
#pragma unroll
        for (int k = 0; k < K; ++k)
#pragma unroll
            for (int c = 0; c < 4; ++c)
                if (c < nvalid) {
                    if (a.trim_mask) a.trim_mask[(int64_t)k * d + j0 + c] = (tb[c] >> k) & 1u;
                    if (a.elect_mask) a.elect_mask[(int64_t)k * d + j0 + c] = (eb[c] >> k) & 1u;
                }
    }
}

template <int K, int MODE, bool VEC, bool MASKS>
__global__ void __launch_bounds__(kTiesThreads, K <= 8 ? 4 : 2)
ties_build_kernel(const float* __restrict__ base, PtrPack<K> models, int64_t d, const u64* __restrict__ cut_dev,
                  BuildArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    u64 cut[K];
    float wk[K];
    bool lo_ok = true;   // every survivor is at least its model's cut magnitude: >= 2^-100 keeps the fast divide exact
#pragma unroll
    for (int k = 0; k < K; ++k) {
        cut[k] = cut_dev[k];
        wk[k] = (MODE == TIES_MODE_TRIMSUM) ? a.w[k] : 0.0f;
        lo_ok = lo_ok && ((uint32_t)(cut[k] >> 32) >= (27u << 23));
    }
    // FUSED_MERGE: lambda rows and the block table in shared memory
    FusedSegs fs{nullptr, nullptr, nullptr, 1};
    if (MODE == TIES_MODE_FUSED_MERGE) {
        const int G = (int)a.ldo;  // number of lambda groups travels in ldo for this mode
        float* s_w = reinterpret_cast<float*>(smem_raw);
        int64_t* s_end = reinterpret_cast<int64_t*>(smem_raw + ((G * K * 4 + 15) & ~15));
        const bool table = a.seg_end && a.seg_group;   // a one-block table may still name a group other than 0
        int32_t* s_grp = reinterpret_cast<int32_t*>(s_end + (table ? a.P : 0));
        for (int i = threadIdx.x; i < G * K; i += blockDim.x) s_w[i] = a.w[i];
        if (table)
            for (int i = threadIdx.x; i < a.P; i += blockDim.x) { s_end[i] = a.seg_end[i]; s_grp[i] = a.seg_group[i]; }
        __syncthreads();
        fs = FusedSegs{s_w, table ? s_end : nullptr, table ? s_grp : nullptr, a.P};
    }
    const int64_t nq = (d + 3) >> 2;
    // hot quads: complete and (for K >= 5) before the interleaved-order tail of the flat vector
    const int64_t nq_hot = (K >= 5 ? (d & ~(int64_t)31) : (d & ~(int64_t)3)) >> 2;
    const int64_t gtid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t gsz = (int64_t)gridDim.x * blockDim.x;
    int hint = 0;
    for (int64_t q = gtid; q < nq_hot; q += gsz) ties_quad<K, MODE, VEC, MASKS, false>(base, models, d, q, cut, lo_ok, wk, a, fs, hint);
    for (int64_t q = nq_hot + gtid; q < nq; q += gsz) ties_quad<K, MODE, VEC, MASKS, true>(base, models, d, q, cut, lo_ok, wk, a, fs, hint);
}

// ---- speculative select + build in ONE pass over the data (VECTORS and FUSED_MERGE) --------------------------------------
// After the two sample passes the cut of every model is known to lie in a narrow bracket [lo, hi] (about 0.75 % of the
// keys).  Instead of one full pass that only counts / collects (the select) followed by a second full pass that
// builds, this kernel does both at once: it builds the output with a PROVISIONAL cut (the middle of the bracket) while
// counting the keys above the bracket and collecting the keys inside it exactly as the select's full pass does.  The
// exact cut then comes from the collected keys (cand_hist -> pick -> pick -> compact -> final, a few microseconds), and
// ties_patch_kernel recomputes only the columns whose provisional decision was wrong: the collected keys between the
// provisional and the exact cut, typically 0.05 % of the columns.  The result is bit-identical to select + build.
//
// FUSED_MERGE keeps the lambda row and the bounds of the block a thread last met in registers: a quad that lies wholly
// inside the sequential part of that block takes the hot path, any other quad looks its blocks up column by column.
constexpr int kSpecStages = 2;
__device__ __forceinline__ uint32_t spec_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void spec_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void spec_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void spec_mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok = 0;
    while (!ok)
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void spec_bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

struct SpecState {     // per model, staged in shared memory
    u64 lo, hi, mid;
};

// Rare path of the speculative pass, out of line: the key of an in-window element is appended to the thread's private
// candidate list of model k and the provisional cut decides whether the element survives for now.
static __device__ __noinline__ float spec_collect(int k, float u, int64_t j, const SpecState* s_st, uint32_t* s_cnt,
                                           const PassCounters& pc, int64_t gsz, int64_t gtid) {
    const u64 key = ties_key(__float_as_uint(u) & 0x7FFFFFFFu, j);
    const uint32_t n = s_cnt[k * kTiesThreads + threadIdx.x];
    if (n < (uint32_t)pc.cand_cap) pc.cand_keys[((size_t)k * gsz + gtid) * pc.cand_cap + n] = key;
    s_cnt[k * kTiesThreads + threadIdx.x] = n + 1;
    return (key >= s_st[k].mid) ? u : 0.0f;
}

template <int K, int MODE, bool VEC>
__global__ void __launch_bounds__(kTiesThreads, K <= 8 ? 2 : 1)
ties_spec_kernel(const float* __restrict__ base, PtrPack<K> models, int64_t d, const TiesState* __restrict__ st,
                 const u64* __restrict__ mid_dev, PassCounters pc, BuildArgs a, int blocked_tiles) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // layout: [FUSED_MERGE tables] | SpecState[K] | ge[K] u32 | lom[K] i32 | span[K] u32 | cnt[K][blockDim] u32
    // (the bracket words and the per-thread candidate counters live in shared memory, not in registers: the hot loop
    //  needs them once per model and quad, and 64 registers per thread keep four CTAs resident per SM)
    size_t off = 0;
    FusedSegs fs{nullptr, nullptr, nullptr, 1};
    if (MODE == TIES_MODE_FUSED_MERGE) {
        const int G = (int)a.ldo;   // number of lambda groups travels in ldo for this mode
        float* s_w = reinterpret_cast<float*>(smem_raw);
        off = ((size_t)G * K * 4 + 15) & ~(size_t)15;
        const bool table = a.seg_end && a.seg_group;
        int64_t* s_end = reinterpret_cast<int64_t*>(smem_raw + off);
        int32_t* s_grp = reinterpret_cast<int32_t*>(s_end + (table ? a.P : 0));
        if (table) off += (((size_t)a.P * 12) + 15) & ~(size_t)15;
        for (int i = threadIdx.x; i < G * K; i += blockDim.x) s_w[i] = a.w[i];
        if (table)
            for (int i = threadIdx.x; i < a.P; i += blockDim.x) { s_end[i] = a.seg_end[i]; s_grp[i] = a.seg_group[i]; }
        fs = FusedSegs{s_w, table ? s_end : nullptr, table ? s_grp : nullptr, a.P};
    }
    SpecState* s_st = reinterpret_cast<SpecState*>(smem_raw + off);
    uint32_t* s_ge = reinterpret_cast<uint32_t*>(s_st + K);
    uint32_t* s_lom = s_ge + K;
    uint32_t* s_span = s_lom + K;
    uint32_t* s_cnt = s_span + K;       // [K][blockDim.x]
    // VEC: the TMA ring (kSpecStages x (K + 1) x 4 KB, 128-byte aligned) and its mbarriers follow the counters
    const size_t ring_off = (off + (size_t)K * (sizeof(SpecState) + 12 + (size_t)kTiesThreads * 4) + 127) & ~(size_t)127;
    if (threadIdx.x < K) {
        const TiesState t = st[threadIdx.x];
        s_st[threadIdx.x].lo = t.lo;
        s_st[threadIdx.x].hi = t.hi;
        s_st[threadIdx.x].mid = mid_dev[threadIdx.x];
        s_ge[threadIdx.x] = 0;
        s_lom[threadIdx.x] = (uint32_t)(t.lo >> 32);
        s_span[threadIdx.x] = (uint32_t)(t.hi >> 32) - (uint32_t)(t.lo >> 32);
    }
#pragma unroll
    for (int k = 0; k < K; ++k) s_cnt[k * kTiesThreads + threadIdx.x] = 0;
    __syncthreads();

    // magnitudes below the bracket, two 16-bit counters per register (a thread sees fewer than 2^16 elements per model:
    // the grid is one resident wave and the host falls back to the two-pass path otherwise)
    constexpr int KP = (K + 1) / 2;
    uint32_t below2[KP];
#pragma unroll
    for (int i = 0; i < KP; ++i) below2[i] = 0;
    bool lo_ok = true;   // every survivor is at least the bracket's lower magnitude: >= 2^-100 keeps the fast divide exact
#pragma unroll
    for (int k = 0; k < K; ++k) lo_ok = lo_ok && (s_lom[k] >= (27u << 23));
    uint32_t visited = 0;
    const int64_t gtid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t gsz = (int64_t)gridDim.x * blockDim.x;
    const int64_t nq = (d + 3) >> 2;
    const int64_t nq_hot = (K >= 5 ? (d & ~(int64_t)31) : (d & ~(int64_t)3)) >> 2;

    // FUSED_MERGE: the block the thread is in -- [cur_lo, cur_hi) is its part where all four columns of a quad share
    // one lambda row and the sequential summation order
    int64_t cur_lo = 0, cur_hi = -1;
    int hint = 0;
    float wrow[K];
#pragma unroll
    for (int k = 0; k < K; ++k) wrow[k] = 0.0f;

    // bracket magnitudes in registers (like the build kernel keeps its cut keys)
    uint32_t lom[K], span[K];
#pragma unroll
    for (int k = 0; k < K; ++k) { lom[k] = s_lom[k]; span[k] = s_span[k]; }

    // Grid-stride over tiles of 256 quads (one quad per thread and tile).  With 16-byte aligned inputs (VEC) the tile's
    // 2K + 1... K + 1 input slices (4 KB each) are brought in by 1-D TMA bulk copies into a ring of kSpecStages shared-
    // memory stages: thread 0 keeps the next tile(s) in flight while the CTA computes, so the bytes in flight per SM
    // (2 CTAs x 2 stages x (K + 1) x 4 KB = 147 KB at K = 8) do not depend on how many registers the column logic
    // needs.  (Direct 128-bit loads left the kernel latency-bound: 52 % of the warp samples sat on the first use of
    // the loaded values at 16 warps per SM.)
    float* ring = reinterpret_cast<float*>(smem_raw + ring_off);
    const uint32_t bar0 = spec_smem_u32(smem_raw + ring_off + (size_t)kSpecStages * (K + 1) * 4096);
    const int64_t n_tiles = (nq_hot + kTiesThreads - 1) / kTiesThreads;
    auto issue_tile = [&](int64_t tile, int stage) {   // thread 0 only
        const int64_t q0 = tile * kTiesThreads;
        const uint32_t nqt = (uint32_t)((nq_hot - q0) < kTiesThreads ? (nq_hot - q0) : kTiesThreads);
        const uint32_t bytes = nqt * 16u;
        const uint32_t bar = bar0 + 8u * stage;
        spec_mbar_expect_tx(bar, bytes * (K + 1));
        float* dst = ring + (size_t)stage * (K + 1) * 1024;
        spec_bulk_load(spec_smem_u32(dst), base + (q0 << 2), bytes, bar);
#pragma unroll
        for (int k = 0; k < K; ++k) spec_bulk_load(spec_smem_u32(dst + (size_t)(k + 1) * 1024), models.p[k] + (q0 << 2), bytes, bar);
    };
    if (VEC) {
        if (threadIdx.x == 0) {
            for (int st_ = 0; st_ < kSpecStages; ++st_) spec_mbar_init(bar0 + 8u * st_, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
    }
    // VECTORS: tile `it` of CTA c is it * grid + c (grid-stride).  FUSED_MERGE: CTA c owns the contiguous tiles
    // [c * per, (c + 1) * per), so a thread's successive quads are 1024 columns apart and mostly stay inside one
    // tensor -- the cached lambda row / block bounds keep hitting (with a grid stride every quad lands in another
    // tensor and pays the block lookup: measured 1.9 vs 1.5 ms)
    const int64_t tiles_per_cta = (n_tiles + gridDim.x - 1) / gridDim.x;
    auto tile_of = [&](int64_t it) -> int64_t {
        if (blocked_tiles) return it < tiles_per_cta ? (int64_t)blockIdx.x * tiles_per_cta + it : n_tiles;
        return it * gridDim.x + blockIdx.x;
    };
    if (VEC && threadIdx.x == 0)
        for (int st_ = 0; st_ < kSpecStages; ++st_) {
            const int64_t tile = tile_of(st_);
            if (tile < n_tiles) issue_tile(tile, st_);
        }
    // (A barrier-free variant -- warps arrive on a per-stage "empty" mbarrier and thread 0 re-arms the stage one iteration
    // later -- was measured slower, 1.64 vs 1.49-1.59 ms: the CTA barrier below holds 21 % of the warp samples, but
    // re-arming right after it keeps two tile-times of prefetch distance instead of one.)
    for (int64_t it = 0;; ++it) {
        const int64_t tile = tile_of(it);
        if (tile >= n_tiles) break;
        const int64_t q = tile * kTiesThreads + threadIdx.x;
        const int64_t j0 = q << 2;
        float bx[4];
        float xs[K][4];
        if (VEC) {
            const int stage = (int)(it % kSpecStages);
            spec_mbar_wait(bar0 + 8u * stage, (uint32_t)((it / kSpecStages) & 1));
            const float4* sm4 = reinterpret_cast<const float4*>(ring + (size_t)stage * (K + 1) * 1024) + threadIdx.x;
            if (q < nq_hot) {
                const float4 b4 = sm4[0];
                bx[0] = b4.x; bx[1] = b4.y; bx[2] = b4.z; bx[3] = b4.w;
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    const float4 v = sm4[(k + 1) * 256];
                    xs[k][0] = v.x; xs[k][1] = v.y; xs[k][2] = v.z; xs[k][3] = v.w;
                }
            }
            // every thread holds its quad in registers: the stage can be refilled.  The refill is a write of the async
            // proxy, the reads above were generic ones: each thread orders its reads before it, then the CTA barrier
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncthreads();
            if (threadIdx.x == 0) {
                const int64_t next = tile_of(it + kSpecStages);
                if (next < n_tiles) issue_tile(next, stage);
            }
            if (q >= nq_hot) continue;
        } else {
            if (q >= nq_hot) continue;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                bx[c] = base[j0 + c];
#pragma unroll
                for (int k = 0; k < K; ++k) xs[k][c] = models.p[k][j0 + c];
            }
        }
        // per column: provisional trim by the magnitude window (rare: exact key test against the provisional cut and
        // collection of the key), then election + disjoint mean; xs[k][c] dies as res[c][k] is born
        float res[4][K];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            float sc[K];
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const float u = __fsub_rn(xs[k][c], bx[c]);
                const uint32_t t = (__float_as_uint(u) & 0x7FFFFFFFu) - lom[k];
                below2[k >> 1] += (t >> 31) << (16 * (k & 1));      // magnitude below the bracket: trimmed
                sc[k] = ((int)t >= 0) ? u : 0.0f;
                // inside the bracket's magnitude window (0.4 % of the elements, but some lane of a warp hits in one of
                // nine (model, column) pairs): ONE out-of-line copy of the collection path instead of 32 inlined ones
                if (t <= span[k]) sc[k] = spec_collect(k, u, j0 + c, s_st, s_cnt, pc, gsz, gtid);
            }
            uint32_t eb;
            ties_elect<K, false>(sc, lo_ok, res[c], eb);
        }
        visited += 4;

        if (MODE == TIES_MODE_VECTORS) {
#pragma unroll
            for (int k = 0; k < K; ++k) {
                float* o = a.out + (int64_t)k * a.ldo + j0;
                if (VEC) stg_stream4(o, make_float4(res[0][k], res[1][k], res[2][k], res[3][k]));
                else
#pragma unroll
                    for (int c = 0; c < 4; ++c) o[c] = res[c][k];
            }
        } else {   // FUSED_MERGE
            float r[4];
            if (!fs.end) {   // task-wise: one block, one lambda row (the tail columns are not in the hot range)
                if (cur_hi < 0) {
#pragma unroll
                    for (int k = 0; k < K; ++k) wrow[k] = fs.w[k];
                    cur_hi = 0;
                }
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    float prod[K];
#pragma unroll
                    for (int k = 0; k < K; ++k) prod[k] = __fmul_rn(wrow[k], res[c][k]);
                    r[c] = __fadd_rn(bx[c], sum_seq<K>(prod));
                }
            } else {
                if (!(j0 >= cur_lo && j0 + 4 <= cur_hi)) {
                    // left the cached block: find the block of j0 (binary search in shared memory, last hit first) and
                    // cache its sequential range and lambda row
                    if (!(j0 < fs.end[hint] && (hint == 0 || j0 >= fs.end[hint - 1]))) {
                        int lo_ = 0, hi_ = fs.P - 1;
                        while (lo_ < hi_) { const int mid_ = (lo_ + hi_) >> 1; if (fs.end[mid_] > j0) hi_ = mid_; else lo_ = mid_ + 1; }
                        hint = lo_;
                    }
                    const int64_t beg = hint ? fs.end[hint - 1] : 0;
                    const int64_t n = fs.end[hint] - beg;
                    cur_lo = beg;
                    cur_hi = (K >= 5) ? beg + (n & ~(int64_t)31) : fs.end[hint];
#pragma unroll
                    for (int k = 0; k < K; ++k) wrow[k] = fs.w[fs.grp[hint] * K + k];
                }
                if (j0 >= cur_lo && j0 + 4 <= cur_hi) {   // hot: the whole quad in the sequential part of one block
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        float prod[K];
#pragma unroll
                        for (int k = 0; k < K; ++k) prod[k] = __fmul_rn(wrow[k], res[c][k]);
                        r[c] = __fadd_rn(bx[c], sum_seq<K>(prod));
                    }
                } else {
                    // a block boundary or a block's interleaved tail inside this quad: per-column lookup
                    int pseg = hint;
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        while (j0 + c >= fs.end[pseg]) ++pseg;
                        const int64_t beg = pseg ? fs.end[pseg - 1] : 0;
                        const int64_t n = fs.end[pseg] - beg;
                        const bool tail = (K >= 5) && ((j0 + c - beg) >= (n & ~(int64_t)31));
                        const float* wr = fs.w + fs.grp[pseg] * K;
                        float prod[K];
#pragma unroll
                        for (int k = 0; k < K; ++k) prod[k] = __fmul_rn(wr[k], res[c][k]);
                        r[c] = __fadd_rn(bx[c], torch_sum_dim0<K>(prod, tail));
                    }
                }
            }
            float* o = a.out + j0;
            if (VEC) stg_stream4(o, make_float4(r[0], r[1], r[2], r[3]));
            else
#pragma unroll
                for (int c = 0; c < 4; ++c) o[c] = r[c];
        }
    }
    // the few cold columns (partial last quad; the <= 31 trailing columns that use the interleaved order when K >= 5):
    // counted and collected here, built by ties_patch_kernel with the exact cut
    for (int64_t q = nq_hot + gtid; q < nq; q += gsz) {
        const int64_t j0 = q << 2;
        const int nvalid = (int)((d - j0) < 4 ? (d - j0) : 4);
        for (int c = 0; c < nvalid; ++c) {
            const float b = base[j0 + c];
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const float u = __fsub_rn(models.p[k][j0 + c], b);
                const uint32_t mag = __float_as_uint(u) & 0x7FFFFFFFu;
                const uint32_t t = mag - lom[k];
                below2[k >> 1] += (t >> 31) << (16 * (k & 1));
                if (t <= span[k]) {
                    const uint32_t n = s_cnt[k * kTiesThreads + threadIdx.x];
                    if (n < (uint32_t)pc.cand_cap)
                        pc.cand_keys[((size_t)k * gsz + gtid) * pc.cand_cap + n] = ties_key(mag, j0 + c);
                    s_cnt[k * kTiesThreads + threadIdx.x] = n + 1;
                }
            }
        }
        visited += (uint32_t)nvalid;
    }

    // above = #magnitudes >= lo_mag; ties_cand_hist_kernel subtracts the collected keys that are not above the bracket
#pragma unroll
    for (int k = 0; k < K; ++k) {
        uint32_t v = visited - ((below2[k >> 1] >> (16 * (k & 1))) & 0xFFFFu);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0 && v) atomicAdd(&s_ge[k], v);
        pc.cand_cnt[(size_t)k * gsz + gtid] = s_cnt[k * kTiesThreads + threadIdx.x];
    }
    __syncthreads();
    if (threadIdx.x < K && s_ge[threadIdx.x]) atomicAdd(&pc.above[threadIdx.x], (u64)s_ge[threadIdx.x]);
}

// provisional cut = middle of the sample bracket (only read when the model is still searching)
static __global__ void ties_mid_kernel(const TiesState* __restrict__ st, int K, u64* __restrict__ mid) {
    const int k = threadIdx.x;
    if (k < K) mid[k] = st[k].lo + ((st[k].hi - st[k].lo) >> 1);
}

// One column rebuilt with the exact cuts (scalar accesses).
// VECTORS: a model that is trimmed under the provisional AND under the exact cut holds 0 in this column before and after
// the fix-up, so only the rows with key >= either[k] = min(provisional, exact cut) are written (about K/5 + 1 of K).
template <int K, int MODE>
__device__ __forceinline__ void ties_patch_column(const float* __restrict__ base, const PtrPack<K>& models, int64_t d, int64_t j,
                                                  const u64 (&cut)[K], const u64 (&either)[K], bool lo_ok, const BuildArgs& a) {
    float x[K], res[K];
    uint32_t tb, eb;
    const float b = base[j];
#pragma unroll
    for (int k = 0; k < K; ++k) x[k] = models.p[k][j];
    const bool flat_tail = (K >= 5) && (j >= (d & ~(int64_t)31));
    if (MODE == TIES_MODE_VECTORS) {
        if (flat_tail) ties_column<K, TIES_MODE_VECTORS, true>(x, b, j, cut, lo_ok, nullptr, res, tb, eb);
        else ties_column<K, TIES_MODE_VECTORS, false>(x, b, j, cut, lo_ok, nullptr, res, tb, eb);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const uint32_t mag = __float_as_uint(__fsub_rn(x[k], b)) & 0x7FFFFFFFu;
            if (ties_key(mag, j) >= either[k]) a.out[(int64_t)k * a.ldo + j] = res[k];
        }
    } else {
        // the election's sums run over the K models of ONE column: their order depends on the position in the flat
        // vector (VECTORS semantics of get_ties_vectors: tail = last d mod 32 columns of the whole vector)
        if (flat_tail) ties_column<K, TIES_MODE_VECTORS, true>(x, b, j, cut, lo_ok, nullptr, res, tb, eb);
        else ties_column<K, TIES_MODE_VECTORS, false>(x, b, j, cut, lo_ok, nullptr, res, tb, eb);
        const float* wr = a.w;
        bool tail = flat_tail;
        if (a.seg_end && a.seg_group) {
            int lo_ = 0, hi_ = a.P - 1;
            while (lo_ < hi_) { const int mid_ = (lo_ + hi_) >> 1; if (a.seg_end[mid_] > j) hi_ = mid_; else lo_ = mid_ + 1; }
            const int64_t beg = lo_ ? a.seg_end[lo_ - 1] : 0;
            const int64_t n = a.seg_end[lo_] - beg;
            tail = (K >= 5) && ((j - beg) >= (n & ~(int64_t)31));
            wr = a.w + a.seg_group[lo_] * K;
        }
        float prod[K];
#pragma unroll
        for (int k = 0; k < K; ++k) prod[k] = __fmul_rn(wr[k], res[k]);
        a.out[j] = __fadd_rn(b, torch_sum_dim0<K>(prod, tail));
    }
}

// Fix-up after the exact cut is known: every collected key between the provisional and the exact cut names a column
// whose provisional decision was wrong; block (0, 0) also builds the cold columns.  One candidate list per thread.
template <int K, int MODE>
__global__ void __launch_bounds__(256)
ties_patch_kernel(const float* __restrict__ base, PtrPack<K> models, int64_t d, const u64* __restrict__ cut_dev,
                  const u64* __restrict__ mid_dev, const int32_t* __restrict__ status, const uint32_t* __restrict__ cand_cnt,
                  const u64* __restrict__ cand_keys, int cand_cap, int n_lists, BuildArgs a) {
    u64 cut[K], either[K], zero[K];
    bool lo_ok = true, ok = true;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        cut[k] = cut_dev[k];
        const u64 m = mid_dev[k];
        either[k] = cut[k] < m ? cut[k] : m;
        zero[k] = 0;
        lo_ok = lo_ok && ((uint32_t)(cut[k] >> 32) >= (27u << 23));
        ok = ok && status[k] == TIES_ST_DONE;
    }
    if (!ok) return;   // a failed select: the caller sees the status and takes the exact path
    const int k = blockIdx.y;
    const u64 a_ = cut_dev[k], b_ = mid_dev[k];
    const u64 lo = a_ < b_ ? a_ : b_, hi = a_ < b_ ? b_ : a_;   // mis-decided keys: lo <= key < hi
    const int64_t hot_end = (K >= 5 ? (d & ~(int64_t)31) : (d & ~(int64_t)3));
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < n_lists; c += gridDim.x * blockDim.x) {
        uint32_t n = cand_cnt[(size_t)k * n_lists + c];
        if (n > (uint32_t)cand_cap) n = (uint32_t)cand_cap;
        const u64* keys = cand_keys + ((size_t)k * n_lists + c) * cand_cap;
        for (uint32_t e = 0; e < n; ++e) {
            const u64 key = keys[e];
            if (key >= lo && key < hi) {
                const int64_t j = (int64_t)(0xFFFFFFFFu - (uint32_t)key);
                if (j < hot_end) ties_patch_column<K, MODE>(base, models, d, j, cut, either, lo_ok, a);
            }
        }
    }
    if (blockIdx.x == 0 && blockIdx.y == 0)
        for (int64_t j = hot_end + threadIdx.x; j < d; j += blockDim.x) ties_patch_column<K, MODE>(base, models, d, j, cut, zero, lo_ok, a);   // cold columns: never built before, write every row
}

// ---- per-mode launchers of the build kernel ---------------------------------------------------------------------------
// This file is compiled five times (Makefile): MR_TIES_PART = 0 holds the selection kernels and every C entry point,
// MR_TIES_PART = 1..4 hold the 64 instantiations (K x alignment x masks) of the build kernel for ONE mode each, so that
// `make -j` compiles them side by side instead of 256 kernels in one translation unit.
#ifndef MR_TIES_PART
#define MR_TIES_PART 0
#endif
struct BuildLaunch {
    const float* base;
    const float* const* models;
    int K;
    int64_t d;
    const u64* cut;
    BuildArgs a;
    size_t smem;
    int64_t blocks;
    bool vec, masks;
    cudaStream_t st;
};
int ties_build_launch_vectors(const BuildLaunch& L);
int ties_build_launch_trimsum(const BuildLaunch& L);
int ties_build_launch_fused(const BuildLaunch& L);
int ties_build_launch_lns(const BuildLaunch& L);

struct SpecLaunch {
    const float* base;
    const float* const* models;
    int K;
    int64_t d;
    const TiesState* st;
    const u64* mid;
    const u64* cut;
    const int32_t* status;
    PassCounters pc;
    BuildArgs a;
    size_t smem;
    int n_lists;     // candidate lists available in the workspace (>= threads of the spec grid)
    bool vec;
    cudaStream_t stream;
};
// phase 0: query the grid (one resident wave) -> *blocks; phase 1: launch the speculative pass with `blocks` CTAs;
// phase 2: launch the patch kernel
int ties_spec_launch_vectors(const SpecLaunch& L, int phase, int* blocks);
int ties_spec_launch_fused(const SpecLaunch& L, int phase, int* blocks);

#if MR_TIES_PART >= 1
#if MR_TIES_PART <= 4
template <int MODE>
static int ties_build_launch_mode(const BuildLaunch& L) {
#define MR_BUILD(VEC, MASKS)                                                                                       \
    do {                                                                                                           \
        auto kern = ties_build_kernel<KK, MODE, VEC, MASKS>;                                                       \
        if (L.smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.smem); \
        kern<<<(unsigned)L.blocks, kTiesThreads, L.smem, L.st>>>(L.base, pack, L.d, L.cut, L.a);                   \
    } while (0)
    MR_DISPATCH_K(L.K, {
        PtrPack<KK> pack;
        for (int k = 0; k < KK; ++k) pack.p[k] = L.models[k];
        if (L.vec) { if (L.masks) MR_BUILD(true, true); else MR_BUILD(true, false); }
        else       { if (L.masks) MR_BUILD(false, true); else MR_BUILD(false, false); }
    });
#undef MR_BUILD
    return MR_OK;
}
#if MR_TIES_PART == 1
int ties_build_launch_vectors(const BuildLaunch& L) { return ties_build_launch_mode<TIES_MODE_VECTORS>(L); }
#elif MR_TIES_PART == 2
int ties_build_launch_trimsum(const BuildLaunch& L) { return ties_build_launch_mode<TIES_MODE_TRIMSUM>(L); }
#elif MR_TIES_PART == 3
int ties_build_launch_fused(const BuildLaunch& L) { return ties_build_launch_mode<TIES_MODE_FUSED_MERGE>(L); }
#elif MR_TIES_PART == 4
int ties_build_launch_lns(const BuildLaunch& L) { return ties_build_launch_mode<TIES_MODE_LNS>(L); }
#endif
#endif  // MR_TIES_PART <= 4
#if MR_TIES_PART >= 5
template <int MODE>
static int ties_spec_launch_mode(const SpecLaunch& L, int phase, int* blocks) {
    MR_DISPATCH_K(L.K, {
        PtrPack<KK> pack;
        for (int k = 0; k < KK; ++k) pack.p[k] = L.models[k];
        if (phase == 0 || phase == 1) {
            auto kern = L.vec ? ties_spec_kernel<KK, MODE, true> : ties_spec_kernel<KK, MODE, false>;
            if (L.smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.smem);
            if (phase == 0) {
                int per_sm = 0;
                cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kTiesThreads, L.smem);
                if (e != cudaSuccess || per_sm < 1) { set_error("mr_ties_select_build: occupancy query failed"); return e != cudaSuccess ? (int)e : MR_ERR_UNSUPPORTED; }
                int b = per_sm * sm_count();
                if (b * kTiesThreads > L.n_lists) b = L.n_lists / kTiesThreads;
                *blocks = b;
                return MR_OK;
            }
            static const int blocked_env = []() { const char* e = getenv("MR_TIES_FUSED_BLOCKED"); return e ? atoi(e) : -1; }();
            const int blocked = blocked_env >= 0 ? blocked_env : (MODE == TIES_MODE_FUSED_MERGE ? 1 : 0);
            kern<<<*blocks, kTiesThreads, L.smem, L.stream>>>(L.base, pack, L.d, L.st, L.mid, L.pc, L.a, blocked);
        } else {
            dim3 grid(64, (unsigned)KK);
            ties_patch_kernel<KK, MODE><<<grid, 256, 0, L.stream>>>(L.base, pack, L.d, L.cut, L.mid, L.status, L.pc.cand_cnt,
                                                                    L.pc.cand_keys, L.pc.cand_cap, *blocks * kTiesThreads, L.a);
        }
    });
    return MR_OK;
}
#if MR_TIES_PART == 5
int ties_spec_launch_vectors(const SpecLaunch& L, int phase, int* blocks) { return ties_spec_launch_mode<TIES_MODE_VECTORS>(L, phase, blocks); }
#elif MR_TIES_PART == 6
int ties_spec_launch_fused(const SpecLaunch& L, int phase, int* blocks) { return ties_spec_launch_mode<TIES_MODE_FUSED_MERGE>(L, phase, blocks); }
#endif
#endif  // MR_TIES_PART >= 5
#endif  // MR_TIES_PART >= 1

#if MR_TIES_PART == 0
// ---- host-side plumbing ---------------------------------------------------------------------------------------
struct TiesWs {
    TiesState* st;
    uint32_t* hist;      // K * bins       } zeroed together before every pass
    u64* above;          // K              }
    uint32_t* fin_cnt;   // K              }
    u64* mid;            // K: provisional cuts of the speculative select + build
    uint32_t* cand_cnt;  // K * n_lists
    u64* fin_keys;       // K * final cap
    u64* cand_keys;      // K * n_lists * cand_cap
    u64* sample_keys;    // K * sample_ld: key cache of the sparse sample (NULL when the "sample" is the whole vector)
    int64_t sample_ld;
    size_t zero_bytes;   // bytes from hist to the end of fin_cnt
    int n_lists, cand_cap;
    size_t total;
};

static inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// one resident wave: the pass kernel is built for 3 CTAs per SM when K <= 8 (2 above), and a 4th CTA per SM would run
// alone at a third of the occupancy after the others have finished
static int ties_pass_blocks(int K) { return sm_count() * (K <= 8 ? 3 : 2); }

// quads between two sample picks; a pick is a pair of adjacent quads (one 32-byte sector), so the stride is even and
// twice nq / sample_quads.  1 = no sampling (every quad once).
static int64_t ties_sample_stride(int64_t d, int64_t sample_quads = kTiesSampleQuads) {
    const int64_t nq = (d + 3) >> 2;
    const int64_t s = (2 * nq / sample_quads) & ~(int64_t)1;
    return s < 2 ? 1 : s;
}

// sampled element count for a given stride (must mirror the kernel's iteration domain; the jittered last quad may
// be the partial one -- the error of at most 3 elements is absorbed by the margin)
static int64_t ties_sample_count(int64_t d, int64_t stride) {
    const int64_t nq = (d + 3) >> 2;
    const int64_t npos = (nq + stride - 1) / stride;
    return stride == 1 ? d : npos * 8;
}

static void ties_sample_ranks(int64_t d, int64_t k_cnt, int64_t n_s, int64_t* r_hi, int64_t* r_lo) {
    const double rs = (double)k_cnt * (double)n_s / (double)d;
    double var = rs * (1.0 - rs / (double)n_s);
    if (var < 0) var = 0;
    const double m = 6.0 * sqrt(var) + 8.0;
    *r_hi = (int64_t)floor(rs - m);
    *r_lo = (int64_t)ceil(rs + m);
}

static TiesWs ties_layout(void* ws, int64_t d, int K) {
    TiesWs L;
    // one private candidate list per thread of the collecting grid: the select's pass kernel runs 3 (K <= 8) or 2 CTAs per
    // SM, the speculative select + build kernel up to 4
    const int n_lists = sm_count() * (K <= 8 ? 4 : 2) * kTiesThreads;
    // expected fraction of keys inside the sample bracket: the +-6 sigma rank window plus bin slack
    const int64_t stride = ties_sample_stride(d);
    const int64_t n_s = ties_sample_count(d, stride);
    int64_t r_hi, r_lo;
    ties_sample_ranks(d, d / 5, n_s, &r_hi, &r_lo);
    double frac = (double)(r_lo - r_hi + 2) / (double)n_s + 6.0 / kTiesBins * 0.25;
    if (frac > 1.0) frac = 1.0;
    const double expect = (double)d * frac / n_lists;
    int64_t cap = ((int64_t)(4.0 * expect) + 24 + 7) & ~(int64_t)7;   // Poisson tail of a mean-`expect` list: < 1e-12
    if (cap > d + 4) cap = d + 4;
    L.n_lists = n_lists;
    L.cand_cap = (int)cap;
    char* p = reinterpret_cast<char*>(ws);
    size_t off = 0;
    L.st = reinterpret_cast<TiesState*>(p + off); off += align256((size_t)K * sizeof(TiesState));
    const size_t z0 = off;
    L.hist = reinterpret_cast<uint32_t*>(p + off); off += align256((size_t)K * kTiesBins * 4);
    L.above = reinterpret_cast<u64*>(p + off); off += align256((size_t)K * 8);
    L.fin_cnt = reinterpret_cast<uint32_t*>(p + off); off += align256((size_t)K * 4);
    L.zero_bytes = off - z0;
    L.mid = reinterpret_cast<u64*>(p + off); off += align256((size_t)K * 8);
    L.cand_cnt = reinterpret_cast<uint32_t*>(p + off); off += align256((size_t)K * n_lists * 4);
    L.fin_keys = reinterpret_cast<u64*>(p + off); off += align256((size_t)K * kTiesFinalCap * 8);
    L.cand_keys = reinterpret_cast<u64*>(p + off); off += align256((size_t)K * n_lists * (size_t)cap * 8);
    L.sample_ld = stride > 1 ? (((n_s + 63) / 64) * 64) : 0;      // n_s = sampled elements = slots the sample pass writes
    L.sample_keys = stride > 1 ? reinterpret_cast<u64*>(p + off) : nullptr;
    off += align256((size_t)K * (size_t)L.sample_ld * 8);
    L.total = off;
    return L;
}

template <int K>
static int ties_launch_pass(const float* base, const float* const* models, int64_t d, const float* w, int64_t stride,
                            int collect /* 0 none, 1 magnitude window (fast path), 2 exact */, const TiesWs& L, cudaStream_t st,
                            int64_t j_off = 0, bool zero_counters = true, bool save_sample_keys = false) {
    PtrPack<K> pack;
    bool vec = host_aligned16(base);
    for (int k = 0; k < K; ++k) { pack.p[k] = models[k]; vec = vec && host_aligned16(models[k]); }
    PassCounters pc{L.hist, L.above, L.cand_cnt, L.cand_keys, L.cand_cap, j_off,
                    (save_sample_keys && stride > 1) ? L.sample_keys : nullptr, L.sample_ld};
    const size_t smem = PassSmem<K>::bytes();
    const int blocks = ties_pass_blocks(K);   // (sample passes too: a smaller grid makes them latency-bound, 70 -> 236 us)
    if (zero_counters) {
        cudaError_t e = cudaMemsetAsync(L.hist, 0, L.zero_bytes, st);
        if (e != cudaSuccess) { set_error("mr_ties_select: memset: %s", cudaGetErrorString(e)); return (int)e; }
    }
#define MR_PASS(VEC, W, COLLECT)                                                                               \
    do {                                                                                                       \
        auto kern = ties_pass_kernel<K, VEC, W, COLLECT>;                                                      \
        if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        kern<<<blocks, kTiesThreads, smem, st>>>(base, pack, d, w, stride, L.st, pc);                          \
    } while (0)
    if (vec) {
        if (w) { if (collect == 1) MR_PASS(true, true, 1); else if (collect == 2) MR_PASS(true, true, 2); else MR_PASS(true, true, 0); }
        else   { if (collect == 1) MR_PASS(true, false, 1); else if (collect == 2) MR_PASS(true, false, 2); else MR_PASS(true, false, 0); }
    } else {
        if (w) { if (collect == 1) MR_PASS(false, true, 1); else if (collect == 2) MR_PASS(false, true, 2); else MR_PASS(false, true, 0); }
        else   { if (collect == 1) MR_PASS(false, false, 1); else if (collect == 2) MR_PASS(false, false, 2); else MR_PASS(false, false, 0); }
    }
#undef MR_PASS
    MR_CUDA_LAUNCH_CHECK("mr_ties_select(pass)");
    return MR_OK;
}

// The two looks at the sparse sample that bracket the cut: the first strides over the vectors (and caches every sampled
// key), the second histograms the cached keys inside the first bracket.  With stride 1 (small vectors) both are passes
// over the data.
template <int K>
static int ties_sparse_brackets(const float* base, const float* const* models, int64_t d, const float* w, int64_t k_cnt,
                                const TiesWs& L, int32_t* status, cudaStream_t st) {
    const int64_t stride = ties_sample_stride(d);
    const int64_t n_s = ties_sample_count(d, stride);
    int64_t r_hi, r_lo;
    ties_sample_ranks(d, k_cnt, n_s, &r_hi, &r_lo);
    int rc = ties_launch_pass<K>(base, models, d, w, stride, 0, L, st, 0, true, true);
    if (rc != MR_OK) return rc;
    ties_pick_kernel<<<K, kTiesBins, 0, st>>>(L.st, L.hist, L.above, r_hi, r_lo, 0, status);
    if (stride > 1 && L.sample_keys) {
        cudaError_t e = cudaMemsetAsync(L.hist, 0, L.zero_bytes, st);
        if (e != cudaSuccess) { set_error("mr_ties_select: memset: %s", cudaGetErrorString(e)); return (int)e; }
        dim3 grid(64, (unsigned)K);
        ties_keys_hist_kernel<<<grid, 256, 0, st>>>(L.st, L.sample_keys, L.sample_ld, n_s, L.hist, L.above);
    } else {
        rc = ties_launch_pass<K>(base, models, d, w, stride, 0, L, st);
        if (rc != MR_OK) return rc;
    }
    ties_pick_kernel<<<K, kTiesBins, 0, st>>>(L.st, L.hist, L.above, r_hi, r_lo, 0, status);
    return MR_OK;
}

// n_lists: the candidate lists the collecting pass wrote = its thread count (the workspace may hold more)
static int ties_finish(const TiesWs& L, int K, int64_t k_cnt, u64* cut, int32_t* status, cudaStream_t st, int n_lists) {
    dim3 hgrid(128, (unsigned)K);
    ties_cand_hist_kernel<<<hgrid, 256, 0, st>>>(L.st, L.cand_cnt, L.cand_keys, L.cand_cap, n_lists, L.hist, L.above);
    ties_pick_kernel<<<K, kTiesBins, 0, st>>>(L.st, L.hist, L.above, k_cnt, k_cnt, 1, status);
    // second refinement level over the collected keys only (a few MB): the bin picked above holds in_bracket / 1024 keys
    // on average -- more than the final sort takes once d exceeds ~3e8 (Recformer-large: 3.2 M keys in the bracket) --
    // and composite keys are distinct, so another 1024-way split always brings it down to a handful
    cudaError_t e = cudaMemsetAsync(L.hist, 0, (size_t)K * kTiesBins * 4, st);
    if (e != cudaSuccess) { set_error("mr_ties_select: memset: %s", cudaGetErrorString(e)); return (int)e; }
    ties_cand_hist_kernel<<<hgrid, 256, 0, st>>>(L.st, L.cand_cnt, L.cand_keys, L.cand_cap, n_lists, L.hist, nullptr);
    ties_pick_kernel<<<K, kTiesBins, 0, st>>>(L.st, L.hist, nullptr, k_cnt, k_cnt, 1, status);
    dim3 grid(256, (unsigned)K);
    ties_compact_kernel<<<grid, 256, 0, st>>>(L.st, L.cand_cnt, L.cand_keys, L.cand_cap, n_lists, L.fin_cnt,
                                              L.fin_keys, status);
    ties_final_kernel<<<K, 1024, 0, st>>>(L.st, L.fin_cnt, L.fin_keys, k_cnt, cut, status);
    MR_CUDA_LAUNCH_CHECK("mr_ties_select(finish)");
    return MR_OK;
}

static int ties_check_args(const float* base, const float* const* models, int K, int64_t d, const void* cut,
                           const void* status, const void* ws, int64_t ws_bytes, const char* who) {
    MR_REQUIRE(K >= 1 && K <= MR_MAX_K, "%s: K=%d outside [1,%d]", who, K, MR_MAX_K);
    MR_REQUIRE(d >= 0 && d < ((int64_t)1 << 32), "%s: need 0 <= d < 2^32", who);
    MR_REQUIRE(cut && status, "%s: null output", who);
    if (d == 0) return MR_OK;
    MR_REQUIRE(base && models && ws, "%s: null pointer", who);
    if (ws_bytes < mr_ties_workspace_bytes(d, K)) {
        set_error("%s: workspace too small (%lld < %lld bytes)", who, (long long)ws_bytes,
                  (long long)mr_ties_workspace_bytes(d, K));
        return MR_ERR_WORKSPACE;
    }
    return MR_OK;
}
#endif  // MR_TIES_PART == 0

}  // namespace mr

#if MR_TIES_PART == 0
extern "C" int64_t mr_ties_workspace_bytes(int64_t d, int K) {
    if (d <= 0 || K < 1 || K > MR_MAX_K) return 256;
    return (int64_t)mr::ties_layout(nullptr, d, K).total;
}

extern "C" int mr_ties_select(const float* base, const float* const* models, int K, int64_t d, const float* w,
                              int64_t k_cnt, uint64_t* cut, int32_t* status, void* ws, int64_t ws_bytes,
                              mr_stream_t stream) {
    using namespace mr;
    int rc = ties_check_args(base, models, K, d, cut, status, ws, ws_bytes, "mr_ties_select");
    if (rc != MR_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (d == 0) {  // nothing to keep: cut = ~0
        ties_init_kernel<<<1, 32, 0, st>>>(nullptr, K, reinterpret_cast<u64*>(cut), status, 0, 0);
        MR_CUDA_LAUNCH_CHECK("mr_ties_select(init)");
        return MR_OK;
    }
    const TiesWs L = ties_layout(ws, d, K);
    ties_init_kernel<<<1, 32, 0, st>>>(L.st, K, reinterpret_cast<u64*>(cut), status, k_cnt, d);
    MR_CUDA_LAUNCH_CHECK("mr_ties_select(init)");
    if (k_cnt <= 0 || k_cnt >= d) return MR_OK;
    MR_DISPATCH_K(K, {
        rc = ties_sparse_brackets<KK>(base, models, d, w, k_cnt, L, status, st);   // 2^63 -> quarter-octave bins -> ~1 % bracket
        if (rc != MR_OK) return rc;
        rc = ties_launch_pass<KK>(base, models, d, w, 1, 1, L, st);
        if (rc != MR_OK) return rc;
    });
    return ties_finish(L, K, k_cnt, reinterpret_cast<u64*>(cut), status, st, ties_pass_blocks(K) * kTiesThreads);
}

// Exact path for any input (e.g. millions of equal magnitudes).  SYNCHRONOUS: reads the bracket state back after
// every pass.  At most 7 narrowing passes + 1 collecting pass over the data.
extern "C" int mr_ties_select_exact(const float* base, const float* const* models, int K, int64_t d, const float* w,
                                    int64_t k_cnt, uint64_t* cut, int32_t* status, void* ws, int64_t ws_bytes,
                                    mr_stream_t stream) {
    using namespace mr;
    int rc = ties_check_args(base, models, K, d, cut, status, ws, ws_bytes, "mr_ties_select_exact");
    if (rc != MR_OK) return rc;
    if (d == 0) return mr_ties_select(base, models, K, d, w, k_cnt, cut, status, ws, ws_bytes, stream);
    cudaStream_t st = (cudaStream_t)stream;
    const TiesWs L = ties_layout(ws, d, K);
    ties_init_kernel<<<1, 32, 0, st>>>(L.st, K, reinterpret_cast<u64*>(cut), status, k_cnt, d);
    MR_CUDA_LAUNCH_CHECK("mr_ties_select_exact(init)");
    if (k_cnt <= 0 || k_cnt >= d) return MR_OK;
    TiesState host[MR_MAX_K];
    for (int it = 0; it < 8; ++it) {
        MR_DISPATCH_K(K, {
            rc = ties_launch_pass<KK>(base, models, d, w, 1, 0, L, st);
            if (rc != MR_OK) return rc;
            ties_pick_kernel<<<KK, kTiesBins, 0, st>>>(L.st, L.hist, L.above, k_cnt, k_cnt, 1, status);
        });
        cudaError_t e = cudaMemcpyAsync(host, L.st, (size_t)K * sizeof(TiesState), cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) { set_error("mr_ties_select_exact: %s", cudaGetErrorString(e)); return (int)e; }
        bool fits = true;
        for (int k = 0; k < K; ++k) {
            if (host[k].status < 0) { set_error("mr_ties_select_exact: model %d failed with status %d", k, host[k].status); return MR_ERR_UNSUPPORTED; }
            if (host[k].status == TIES_ST_SEARCH && host[k].in_bracket > (u64)(L.cand_cap < kTiesFinalCap ? L.cand_cap : kTiesFinalCap)) fits = false;
        }
        if (fits) break;
    }
    MR_DISPATCH_K(K, {
        rc = ties_launch_pass<KK>(base, models, d, w, 1, 2, L, st);
        if (rc != MR_OK) return rc;
    });
    rc = ties_finish(L, K, k_cnt, reinterpret_cast<u64*>(cut), status, st, ties_pass_blocks(K) * kTiesThreads);
    if (rc != MR_OK) return rc;
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { set_error("mr_ties_select_exact: %s", cudaGetErrorString(e)); return (int)e; }
    return MR_OK;
}

// ---- sharded select: the single-GPU sampled-bracket algorithm with the counters summed over the ranks ------------------------
// The caller (one process per GPU) runs phases 0..5 in order on every rank and, after each phase, applies the collective
// named below to the workspace regions reported by mr_ties_dist_layout (NCCL through torch.distributed; the library
// itself never communicates):
//   phase 0  init, sparse sample pass                      -> all-reduce(sum) of the counters region
//   phase 1  pick the bracket, second sparse sample pass   -> all-reduce(sum) of the counters region
//   phase 2  pick, full pass (count + collect), histogram  -> all-reduce(sum) of the counters region
//   phase 3  pick, second-level histogram of the collected -> all-reduce(sum) of the counters region
//   phase 4  pick, compact the survivors                   -> all-gather of the survivors region
//   phase 5  (gathered given) final sort, global and local cut
// Every decision is taken from all-reduced integers, so all ranks walk the same brackets; keys carry GLOBAL indices
// (j_off + local index), which makes the result the single-GPU cut bit for bit.
extern "C" int mr_ties_dist_layout(int64_t d_local, int K, int64_t* counters_off, int64_t* counters_bytes,
                                   int64_t* survivors_off, int64_t* survivors_bytes) {
    using namespace mr;
    MR_REQUIRE(K >= 1 && K <= MR_MAX_K, "mr_ties_dist_layout: K=%d outside [1,%d]", K, MR_MAX_K);
    MR_REQUIRE(d_local >= 0 && counters_off && counters_bytes && survivors_off && survivors_bytes, "mr_ties_dist_layout: bad argument");
    char* const fake = reinterpret_cast<char*>((uintptr_t)1 << 20);     // offsets only: nothing is dereferenced
    const TiesWs L = ties_layout(fake, d_local > 0 ? d_local : 1, K);
    *counters_off = (int64_t)(reinterpret_cast<char*>(L.hist) - fake);
    *counters_bytes = (int64_t)L.zero_bytes;
    *survivors_off = (int64_t)(reinterpret_cast<char*>(L.fin_keys) - fake);
    *survivors_bytes = (int64_t)(align256((size_t)K * kTiesFinalCap * 8) + align256((size_t)K * 4));
    return MR_OK;
}

extern "C" int mr_ties_select_dist(const float* base, const float* const* models, int K, int64_t d_local, int64_t j_off,
                                   int64_t d_global, const float* w, int64_t k_cnt, int phase, const void* gathered,
                                   int world, uint64_t* cut_local, uint64_t* cut_global, int32_t* status, void* ws,
                                   int64_t ws_bytes, mr_stream_t stream) {
    using namespace mr;
    MR_REQUIRE(K >= 1 && K <= MR_MAX_K, "mr_ties_select_dist: K=%d outside [1,%d]", K, MR_MAX_K);
    MR_REQUIRE(d_local >= 0 && j_off >= 0 && d_global >= d_local + j_off && d_global < ((int64_t)1 << 32),
               "mr_ties_select_dist: need 0 <= j_off, j_off + d_local <= d_global < 2^32");
    MR_REQUIRE(k_cnt > 0 && k_cnt < d_global, "mr_ties_select_dist: trivial k_cnt is the caller's business");
    MR_REQUIRE(phase >= 0 && phase <= 5, "mr_ties_select_dist: phase %d outside [0,5]", phase);
    MR_REQUIRE(cut_local && status && ws, "mr_ties_select_dist: null pointer");
    MR_REQUIRE(d_local == 0 || (base && models), "mr_ties_select_dist: null input");
    MR_REQUIRE(world >= 1 && world <= 64, "mr_ties_select_dist: world=%d outside [1,64]", world);
    const int64_t d_ws = d_local > 0 ? d_local : 1;
    if (ws_bytes < mr_ties_workspace_bytes(d_ws, K) + (int64_t)align256((size_t)K * 4)) {
        set_error("mr_ties_select_dist: workspace too small");
        return MR_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const TiesWs L = ties_layout(ws, d_ws, K);
    // the survivors region is [fin_keys | fin_cnt copy]: fin_cnt lives among the counters (zeroed with them), so phase 4
    // copies it behind fin_keys where the all-gather picks both up
    uint32_t* fin_cnt_out = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(L.fin_keys) + align256((size_t)K * kTiesFinalCap * 8));
    // every rank samples with the SAME stride (derived from the global length) so that the global sample size is the sum
    const int64_t stride = ties_sample_stride(d_global);
    const int64_t n_s = ties_sample_count(d_global, stride);
    int64_t r_hi, r_lo;
    ties_sample_ranks(d_global, k_cnt, n_s, &r_hi, &r_lo);
    r_hi -= 8 * world;    // per-rank rounding of the sample size (partial strides at the slice ends)
    r_lo += 8 * world;
    const int n_lists = ties_pass_blocks(K) * kTiesThreads;
    int rc = MR_OK;
    cudaError_t e;
    switch (phase) {
        case 0:
            ties_init_kernel<<<1, 32, 0, st>>>(L.st, K, reinterpret_cast<u64*>(cut_local), status, k_cnt, d_global);
            MR_CUDA_LAUNCH_CHECK("mr_ties_select_dist(init)");
            [[fallthrough]];
        case 1:
            if (phase == 1) ties_pick_kernel<<<K, kTiesBins, 0, st>>>(L.st, L.hist, L.above, r_hi, r_lo, 0, status);
            e = cudaMemsetAsync(L.hist, 0, L.zero_bytes, st);
            if (e != cudaSuccess) { set_error("mr_ties_select_dist: memset: %s", cudaGetErrorString(e)); return (int)e; }
            if (d_local > 0) MR_DISPATCH_K(K, { rc = ties_launch_pass<KK>(base, models, d_local, w, stride, 0, L, st, j_off, false); });
            return rc;
        case 2:
            ties_pick_kernel<<<K, kTiesBins, 0, st>>>(L.st, L.hist, L.above, r_hi, r_lo, 0, status);
            e = cudaMemsetAsync(L.hist, 0, L.zero_bytes, st);
            if (e == cudaSuccess) e = cudaMemsetAsync(L.cand_cnt, 0, (size_t)K * n_lists * 4, st);
            if (e != cudaSuccess) { set_error("mr_ties_select_dist: memset: %s", cudaGetErrorString(e)); return (int)e; }
            if (d_local > 0) MR_DISPATCH_K(K, { rc = ties_launch_pass<KK>(base, models, d_local, w, 1, 1, L, st, j_off, false); });
            if (rc != MR_OK) return rc;
            {
                dim3 hgrid(128, (unsigned)K);
                ties_cand_hist_kernel<<<hgrid, 256, 0, st>>>(L.st, L.cand_cnt, L.cand_keys, L.cand_cap, n_lists, L.hist, L.above);
            }
            MR_CUDA_LAUNCH_CHECK("mr_ties_select_dist(collect)");
            return MR_OK;
        case 3:
            ties_pick_kernel<<<K, kTiesBins, 0, st>>>(L.st, L.hist, L.above, k_cnt, k_cnt, 1, status);
            e = cudaMemsetAsync(L.hist, 0, L.zero_bytes, st);
            if (e != cudaSuccess) { set_error("mr_ties_select_dist: memset: %s", cudaGetErrorString(e)); return (int)e; }
            {
                dim3 hgrid(128, (unsigned)K);
                ties_cand_hist_kernel<<<hgrid, 256, 0, st>>>(L.st, L.cand_cnt, L.cand_keys, L.cand_cap, n_lists, L.hist, nullptr);
            }
            MR_CUDA_LAUNCH_CHECK("mr_ties_select_dist(refine)");
            return MR_OK;
        case 4: {
            ties_pick_kernel<<<K, kTiesBins, 0, st>>>(L.st, L.hist, nullptr, k_cnt, k_cnt, 1, status);
            e = cudaMemsetAsync(L.fin_cnt, 0, (size_t)K * 4, st);
            if (e != cudaSuccess) { set_error("mr_ties_select_dist: memset: %s", cudaGetErrorString(e)); return (int)e; }
            dim3 grid(256, (unsigned)K);
            ties_compact_kernel<<<grid, 256, 0, st>>>(L.st, L.cand_cnt, L.cand_keys, L.cand_cap, n_lists, L.fin_cnt, L.fin_keys, status);
            e = cudaMemcpyAsync(fin_cnt_out, L.fin_cnt, (size_t)K * 4, cudaMemcpyDeviceToDevice, st);
            if (e != cudaSuccess) { set_error("mr_ties_select_dist: copy: %s", cudaGetErrorString(e)); return (int)e; }
            MR_CUDA_LAUNCH_CHECK("mr_ties_select_dist(compact)");
            return MR_OK;
        }
        default: {
            MR_REQUIRE(gathered, "mr_ties_select_dist: phase 5 needs the gathered survivors");
            const size_t region = align256((size_t)K * kTiesFinalCap * 8) + align256((size_t)K * 4);
            ties_final_dist_kernel<<<K, 1024, 0, st>>>(L.st, reinterpret_cast<const unsigned char*>(gathered), world, region,
                                                       align256((size_t)K * kTiesFinalCap * 8), k_cnt, j_off,
                                                       reinterpret_cast<u64*>(cut_local), reinterpret_cast<u64*>(cut_global), status);
            MR_CUDA_LAUNCH_CHECK("mr_ties_select_dist(final)");
            return MR_OK;
        }
    }
}

// get_ties_vectors / the fused TIES + lambda merge in ONE pass over the data: sample passes, then the speculative
// select + build pass, the exact cut from the collected keys, and the fix-up of the mis-decided columns.
extern "C" int mr_ties_select_build(const float* base, const float* const* models, int K, int64_t d, int64_t k_cnt, int mode,
                                    const float* w, int G, const int64_t* seg_end, const int32_t* seg_group, int P,
                                    float* out, int64_t ldo, uint64_t* cut, int32_t* status, void* ws, int64_t ws_bytes,
                                    mr_stream_t stream) {
    using namespace mr;
    int rc = ties_check_args(base, models, K, d, cut, status, ws, ws_bytes, "mr_ties_select_build");
    if (rc != MR_OK) return rc;
    MR_REQUIRE(mode == TIES_MODE_VECTORS || mode == TIES_MODE_FUSED_MERGE, "mr_ties_select_build: mode must be VECTORS or FUSED_MERGE");
    if (d == 0 || k_cnt <= 0 || k_cnt >= d) {
        // trivial cuts (keep nothing / everything): nothing to speculate about
        rc = mr_ties_select(base, models, K, d, nullptr, k_cnt, cut, status, ws, ws_bytes, stream);
        if (rc != MR_OK || d == 0) return rc;
        return mr_ties_build(base, models, K, d, cut, mode, w, G, seg_end, seg_group, P, out, ldo, nullptr, nullptr, stream);
    }
    MR_REQUIRE(out, "mr_ties_select_build: null output");
    const bool rows_out = mode == TIES_MODE_VECTORS;
    MR_REQUIRE(rows_out || w, "mr_ties_select_build: FUSED_MERGE needs the lambdas");
    MR_REQUIRE(!rows_out || ldo >= d, "mr_ties_select_build: need ldo >= d");
    MR_REQUIRE(rows_out || (G >= 1 && P >= 1 && (P == 1 || (seg_end && seg_group))),
               "mr_ties_select_build: FUSED_MERGE needs G >= 1 and a block table when P > 1");
    MR_REQUIRE(rows_out || (size_t)G * K * 4 + (size_t)P * 12 + 1024 <= (size_t)200 * 1024,
               "mr_ties_select_build: the block table (P=%d blocks, G=%d groups) does not fit shared memory", P, G);
    cudaStream_t st = (cudaStream_t)stream;
    const TiesWs L = ties_layout(ws, d, K);
    ties_init_kernel<<<1, 32, 0, st>>>(L.st, K, reinterpret_cast<u64*>(cut), status, k_cnt, d);
    MR_CUDA_LAUNCH_CHECK("mr_ties_select_build(init)");
    // Three sample passes.  The first two walk the select's sparse sample (~131 K quads) and bracket the cut to about
    // 0.75 % of the keys; the third walks a 4x denser sample but only histograms the keys inside that bracket (a rare
    // path, sparse per-CTA histograms) and halves it.  (Strided 16-byte picks cost a 32-byte DRAM sector each and run at
    // ~20 G sectors/s: 8x / 16x / 32x samples were measured slower overall, 3.02 / 3.14 / 3.67 / 4.59 ms per cfg-2 step.)  The number of columns the fix-up has to rebuild (scattered
    // 32-byte accesses, 17 per column) and the number of keys the full pass collects are both proportional to the
    // error of the sample quantile, i.e. to 1 / sqrt(sample size).
    static const int64_t dense_quads = []() { const char* e = getenv("MR_TIES_SPEC_SAMPLE_QUADS"); return e ? atoll(e) : 4 * kTiesSampleQuads; }();
    MR_DISPATCH_K(K, {
        rc = ties_sparse_brackets<KK>(base, models, d, nullptr, k_cnt, L, status, st);
        if (rc != MR_OK) return rc;
        const int64_t stride = ties_sample_stride(d, dense_quads);
        if (stride < ties_sample_stride(d)) {      // (small vectors: the sparse sample is already everything)
            const int64_t n_s = ties_sample_count(d, stride);
            int64_t r_hi, r_lo;
            ties_sample_ranks(d, k_cnt, n_s, &r_hi, &r_lo);
            rc = ties_launch_pass<KK>(base, models, d, nullptr, stride, 0, L, st);
            if (rc != MR_OK) return rc;
            ties_pick_kernel<<<KK, kTiesBins, 0, st>>>(L.st, L.hist, L.above, r_hi, r_lo, 0, status);
        }
    });
    ties_mid_kernel<<<1, 32, 0, st>>>(L.st, K, L.mid);
    cudaError_t e = cudaMemsetAsync(L.hist, 0, L.zero_bytes, st);
    if (e != cudaSuccess) { set_error("mr_ties_select_build: memset: %s", cudaGetErrorString(e)); return (int)e; }
    bool vec = host_aligned16(base) && host_aligned16(out) && (!rows_out || (ldo % 4 == 0));
    for (int k = 0; k < K; ++k) vec = vec && host_aligned16(models[k]);
    BuildArgs a{out, rows_out ? ldo : (int64_t)G, nullptr, nullptr, w, seg_end, seg_group, rows_out ? 1 : P};
    size_t smem = (size_t)K * (sizeof(SpecState) + 12 + (size_t)kTiesThreads * 4) + 32;
    if (!rows_out) smem += (((size_t)G * K * 4 + 15) & ~(size_t)15) + ((seg_end && seg_group) ? ((((size_t)P * 12) + 15) & ~(size_t)15) : 0);
    if (vec) smem = ((smem + 127) & ~(size_t)127) + (size_t)kSpecStages * (K + 1) * 4096 + 64;   // TMA ring + mbarriers
    PassCounters pc{L.hist, L.above, L.cand_cnt, L.cand_keys, L.cand_cap, 0, nullptr, 0};
    SpecLaunch S{base, models, K, d, L.st, L.mid, reinterpret_cast<const u64*>(cut), status, pc, a, smem, L.n_lists, vec, st};
    int blocks = 0;
    auto launch = rows_out ? ties_spec_launch_vectors : ties_spec_launch_fused;
    rc = launch(S, 0, &blocks);
    if (rc != MR_OK) return rc;
    {   // the kernel counts per thread in 16 bits: a grid too small for that (a tiny GPU, a huge vector) takes two passes
        const int64_t nq_hot = (K >= 5 ? (d & ~(int64_t)31) : (d & ~(int64_t)3)) >> 2;
        const int64_t per_thread = blocks > 0 ? (nq_hot + (int64_t)blocks * kTiesThreads - 1) / ((int64_t)blocks * kTiesThreads) : nq_hot;
        if (blocks < 1 || (per_thread + 2) * 4 >= 65535) {
            rc = mr_ties_select(base, models, K, d, nullptr, k_cnt, cut, status, ws, ws_bytes, stream);
            if (rc != MR_OK) return rc;
            return mr_ties_build(base, models, K, d, cut, mode, w, G, seg_end, seg_group, P, out, ldo, nullptr, nullptr, stream);
        }
    }
    rc = launch(S, 1, &blocks);
    if (rc != MR_OK) return rc;
    MR_CUDA_LAUNCH_CHECK("mr_ties_select_build(pass)");
    rc = ties_finish(L, K, k_cnt, reinterpret_cast<u64*>(cut), status, st, blocks * kTiesThreads);
    if (rc != MR_OK) return rc;
    rc = launch(S, 2, &blocks);
    if (rc != MR_OK) return rc;
    MR_CUDA_LAUNCH_CHECK("mr_ties_select_build(patch)");
    return MR_OK;
}

extern "C" int mr_ties_build(const float* base, const float* const* models, int K, int64_t d, const uint64_t* cut,
                             int mode, const float* w, int G, const int64_t* seg_end, const int32_t* seg_group, int P,
                             float* out, int64_t ldo, uint8_t* trim_mask, uint8_t* elect_mask, mr_stream_t stream) {
    using namespace mr;
    MR_REQUIRE(K >= 1 && K <= MR_MAX_K, "mr_ties_build: K=%d outside [1,%d]", K, MR_MAX_K);
    MR_REQUIRE(d >= 0 && d < ((int64_t)1 << 32), "mr_ties_build: need 0 <= d < 2^32");
    MR_REQUIRE(mode >= 0 && mode <= 3, "mr_ties_build: bad mode %d", mode);
    if (d == 0) return MR_OK;
    MR_REQUIRE(base && models && cut && out, "mr_ties_build: null pointer");
    const bool rows_out = mode == TIES_MODE_VECTORS || mode == TIES_MODE_LNS;
    MR_REQUIRE(rows_out || w, "mr_ties_build: this mode needs weights");
    MR_REQUIRE(!rows_out || ldo >= d, "mr_ties_build: need ldo >= d");
    MR_REQUIRE(mode != TIES_MODE_FUSED_MERGE || (G >= 1 && P >= 1 && (P == 1 || (seg_end && seg_group))),
               "mr_ties_build: FUSED_MERGE needs G >= 1 and a block table when P > 1");
    MR_REQUIRE(mode != TIES_MODE_FUSED_MERGE || (size_t)G * K * 4 + (size_t)P * 12 + 64 <= (size_t)224 * 1024,
               "mr_ties_build: the block table (P=%d blocks, G=%d groups) does not fit shared memory", P, G);
    cudaStream_t st = (cudaStream_t)stream;
    bool vec = host_aligned16(base) && host_aligned16(out) && (!rows_out || (ldo % 4 == 0));
    for (int k = 0; k < K; ++k) vec = vec && host_aligned16(models[k]);
    const bool masks = trim_mask || elect_mask;
    const int64_t nq = (d + 3) >> 2;
    int64_t blocks = (nq + kTiesThreads - 1) / kTiesThreads;
    const int64_t cap = (int64_t)sm_count() * 8;
    if (blocks > cap) blocks = cap;
    BuildArgs a{out, mode == TIES_MODE_FUSED_MERGE ? (int64_t)G : ldo, trim_mask, elect_mask, w, seg_end, seg_group,
                mode == TIES_MODE_FUSED_MERGE ? P : 1};
    size_t smem = 16;
    if (mode == TIES_MODE_FUSED_MERGE) smem = (((size_t)G * K * 4 + 15) & ~(size_t)15) + ((seg_end && seg_group) ? (size_t)P * 12 : 0) + 16;
    BuildLaunch L{base, models, K, d, reinterpret_cast<const u64*>(cut), a, smem, blocks, vec, masks, st};
    int rc = MR_OK;
    if (mode == TIES_MODE_VECTORS) rc = ties_build_launch_vectors(L);
    else if (mode == TIES_MODE_LNS) rc = ties_build_launch_lns(L);
    else if (mode == TIES_MODE_TRIMSUM) rc = ties_build_launch_trimsum(L);
    else rc = ties_build_launch_fused(L);
    if (rc != MR_OK) return rc;
    MR_CUDA_LAUNCH_CHECK("mr_ties_build");
    return MR_OK;
}
#endif  // MR_TIES_PART == 0
