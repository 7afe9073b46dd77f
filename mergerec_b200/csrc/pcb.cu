// pcb.cu -- PCB-merging vectors (SURVEY.md section 8(f) rank 2; reference: rec_retrieval/merger/algorithms/pcb.py:9-58).
//
//   tau_k  = m_k - base                                 A_k = clamp(|tau_k|, lo_k, hi_k)   (1% / 99% order statistics of
//   self_k = ((A_k - lo_k) / (hi_k - lo_k))^2                                                |tau_k|, found by the TIES select)
//   task_k = exp(n * self_k) * tanh(tau_k * sum_k tau_k)
//   scale_k = (clamp(task_k, q_k, max_k) - q_k) / (max_k - q_k)     q_k = the int(d (1 - density))-th smallest task_k
//   out_k  = sign(tau_k) A_k scale_k / max(sum_k scale_k, 1e-12) / n
//
// The quantile q_k of the COMPUTED values is an exact order statistic; nothing of size (K, d) is materialised besides
// the output.  Dense search: three histogram passes (11 + 11 + 10 bits of the order-preserving integer image of the
// float) that recompute task_k from base + models each time.  Fast search (round 2 rework): ONE pass over a 1/32 sample
// caches the sample's keys; two radix selects over the cached keys give the sample's order statistics R ranks below and
// above the wanted quantile (R = 6 sigma of the sampling error), i.e. a key window that holds ~2R * 32 elements of the
// full vector; ONE pass over everything counts what lies below the window and appends the keys inside it to per-warp
// lists (ballot + prefix count, no atomics); the refinement levels (2048-bin histograms, at most three) read the lists.
// Every column sum uses torch.sum(dim=0)'s order (common.cuh).  exp / tanh are CUDA's expf / tanhf; torch's CPU kernels
// use a different libm, so values agree to ~1 ulp, not bit for bit, and an element whose task value lies within that
// distance of q_k may fall on the other side of the clamp (the tests confine every difference from the reference to
// such columns).
#include <math.h>

#include <type_traits>

#include "common.cuh"

namespace mr {

constexpr int kPcbThreads = 256;
constexpr int kPcbWarps = kPcbThreads / 32;
constexpr int kPcbBins = 2048;
constexpr int kPcbSlots = 2;        // sample order statistics searched at once: window start, window end
constexpr int64_t kPcbStride = 32;  // sample of the fast path: 1 / 32 of the columns (pcb_sample_column)

struct PcbState {     // one per (slot, model); the window search uses the slot-0 entries
    uint32_t prefix;  // key bits decided so far
    uint32_t maxkey;  // order-preserving key of the row maximum
    int64_t rank;     // remaining ascending rank inside the chosen bucket
    uint32_t qkey;    // final key of the order statistic
    uint32_t wlo;     // windowed search: first key of the window
    int32_t wshift;   //                  log2(keys per bin)
    int32_t wwidth;   //                  bins of the window that belong to the search
    int32_t miss;     //                  the window did not contain the wanted rank / a list overflowed (caller falls
                      //                  back to the dense passes)
    int32_t done;     //                  qkey is final
    uint32_t wspan;   //                  last key of the window - wlo (the full pass collects wlo <= key <= wlo + wspan)
    int32_t pad;
};

// Order-preserving key: ~u for a set sign bit, u with the sign bit set otherwise.  Written as one xor with a mask built
// from the sign: the select form `(u & sign) ? ~u : (u | sign)` let nvcc compute `u | sign` as the float -|x| (an FADD),
// which turns a NaN into the canonical NaN 0x7fffffff, so +NaN weights were keyed as -0.
__device__ __forceinline__ uint32_t pcb_key(float x) {
    const uint32_t u = __float_as_uint(x);
    return u ^ ((uint32_t)((int32_t)u >> 31) | 0x80000000u);
}
__device__ __forceinline__ float pcb_unkey(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// IEEE x / y for a divisor that is used many times (a per-model range, a per-column sum) and 0 <= x.  __fdiv_rn costs
// about a dozen instructions and leaves its inline sequence for an out-of-line routine whenever ANY lane of the warp
// holds a zero / denormal / huge operand -- and here most numerators are exact zeros (80 % of the clamped balancing
// weights).  With r = RN(1 / y) prepared once: q0 = RN(x r) is within 1.5 ulp of x / y; q1 = RN(q0 + (x - q0 y) r) (the
// residual is exact in an FMA) is faithful; a second correction of a faithful quotient with a correctly rounded
// reciprocal is the correctly rounded quotient (Markstein's division theorem) -- five FMA-pipe instructions, no MUFU, no
// branch, and x = +0 gives +0.  The kernels are compiled twice: SAFE = true uses these sequences and is valid while every
// divisor and every upper clamp lies in [2^-60, 2^60] (numerators never exceed their divisors by more than that, and a
// residual can only underflow for a numerator below ~2^-100, where a last-bit difference from IEEE is 20 orders of
// magnitude under every tolerance of this floating-point path); pcb_status_kernel checks exactly this on the device and
// reports status 2 otherwise, upon which the caller reruns with MR_PCB_IEEE (SAFE = false: __fdiv_rn everywhere).
// tests/test_division_sequences.py checks the sequence exhaustively over the mantissas of x on the CPU.
template <bool SAFE>
__device__ __forceinline__ float pcb_div_by(float x, float y, float r) {
    if (!SAFE) return __fdiv_rn(x, y);
    float q = __fmul_rn(x, r);
    q = __fmaf_rn(__fmaf_rn(-q, y, x), r, q);
    q = __fmaf_rn(__fmaf_rn(-q, y, x), r, q);
    return q;
}
__device__ __forceinline__ bool pcb_safe_range(float y) { return (y >= 0x1p-60f) && (y <= 0x1p60f); }

// x / n for the integer model count n in [1, 16] and 0 <= x: reciprocal multiply + one FMA correction, bit-identical to
// the IEEE quotient inside [2^-100, 2^100] (checked exhaustively for the TIES disjoint mean, ties.cu); +0 gives +0.
template <bool SAFE>
__device__ __forceinline__ float pcb_div_count(float x, float fn, float inv) {
    if (!SAFE) return __fdiv_rn(x, fn);
    const float q0 = __fmul_rn(x, inv);
    return __fmaf_rn(__fmaf_rn(-q0, fn, x), inv, q0);
}

// Per-model clamp table in shared memory: lo, hi, the range hi - lo and its reciprocal.
template <int K>
struct PcbClamp {
    float lo[K], hi[K], rng[K], rr[K];
    __device__ __forceinline__ void load(const float* __restrict__ glo, const float* __restrict__ ghi) {   // before a barrier
        if (threadIdx.x < K) {
            const float l = glo[threadIdx.x], h = ghi[threadIdx.x];
            const float y = __fsub_rn(h, l);
            lo[threadIdx.x] = l; hi[threadIdx.x] = h; rng[threadIdx.x] = y;
            rr[threadIdx.x] = pcb_safe_range(y) ? __frcp_rn(y) : 0.0f;
        }
    }
};

// task_k of one column (pcb.py:44-53); also returns tau and A for the build kernel.
template <int K, bool SAFE>
__device__ __forceinline__ void pcb_task(float b, const float (&x)[K], const PcbClamp<K>& C, bool tail, float (&tau)[K],
                                         float (&A)[K], float (&task)[K]) {
#pragma unroll
    for (int k = 0; k < K; ++k) tau[k] = __fsub_rn(x[k], b);
    const float total = torch_sum_dim0<K>(tau, tail);
#pragma unroll
    for (int k = 0; k < K; ++k) {
        A[k] = fminf(fmaxf(fabsf(tau[k]), C.lo[k]), C.hi[k]);
        const float nrm = pcb_div_by<SAFE>(__fsub_rn(A[k], C.lo[k]), C.rng[k], C.rr[k]);
        const float self_act = expf(__fmul_rn((float)K, __fmul_rn(nrm, nrm)));
        task[k] = __fmul_rn(self_act, tanhf(__fmul_rn(tau[k], total)));
    }
}

// One quad (columns 4q .. 4q+3) of base and the K models; VEC = every pointer 16-byte aligned.  Columns past d read 0.
template <int K, bool VEC>
__device__ __forceinline__ int pcb_load_quad(const float* __restrict__ base, const PtrPack<K>& m, int64_t d, int64_t q,
                                             bool live, float (&bx)[4], float (&xs)[K][4]) {
    const int64_t j0 = q << 2;
    const int nvalid = live ? (int)((d - j0) < 4 ? (d - j0) : 4) : 0;
    if (VEC && nvalid == 4) {
        const float4 b4 = ldg_stream4(base + j0);
        bx[0] = b4.x; bx[1] = b4.y; bx[2] = b4.z; bx[3] = b4.w;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const float4 v = ldg_stream4(m.p[k] + j0);
            xs[k][0] = v.x; xs[k][1] = v.y; xs[k][2] = v.z; xs[k][3] = v.w;
        }
    } else {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const bool ok = c < nvalid;
            bx[c] = ok ? ldg_stream1(base + j0 + c) : 0.f;
#pragma unroll
            for (int k = 0; k < K; ++k) xs[k][c] = ok ? ldg_stream1(m.p[k] + j0 + c) : 0.f;
        }
    }
    return nvalid;
}

// The 1 / stride sample of the fast path: one quad of 4 adjacent columns out of every block of 4 * stride columns, at a
// hashed position inside its block.  Adjacent columns share a 32-byte DRAM sector (a pick of 4 costs what a pick of 1
// costs), and the hashed position keeps the sample from locking onto a fixed column residue of the weight matrices (a
// plain stride of 32 would only ever see columns = 0 mod 32 of a 768- or 1024-wide row -- e.g. never, or always, an outlier
// dimension of a transformer -- and a biased sample costs the fallback to the dense search).  Only whole blocks are sampled.
__host__ __device__ __forceinline__ int64_t pcb_sample_count(int64_t d, int64_t stride) { return 4 * (d / (4 * stride)); }
__host__ __device__ __forceinline__ int64_t pcb_sample_column(int64_t i, int64_t stride) {
    const int64_t c = i >> 2;
    const uint32_t h = ((uint32_t)c * 2654435761u) >> 16;
    return c * (4 * stride) + 4 * (int64_t)(h % (uint32_t)stride) + (i & 3);
}

// Radix pass over the columns (stride = 1) or over the sample (stride > 1) -- pass 0: bins = key >> 21 (+ row maxima); pass 1:
// (key >> 10) & 2047 inside prefix; pass 2: key & 1023 inside prefix.  stride = 1: the dense search (all three passes);
// stride > 1: the fast path's only pass over the sample (pass 0), which also caches the keys in skeys (K, n_vis).
// SLICE (the sharded search's sample pass): the vector is columns j_off .. j_off + d - 1 of a longer one, and the pass
// visits the elements s0 .. s0 + n_s - 1 of that vector's sample (pcb_slice_sample); otherwise s0 / j_off / n_s are
// unused and the sweep is the whole-vector one, kept apart because the slice arithmetic costs the gather-bound sample
// pass ~8 % (20 us at K = 8 BLaIR-base).
template <int K, bool SLICE>
__global__ void __launch_bounds__(kPcbThreads)
pcb_hist_kernel(const float* __restrict__ base, PtrPack<K> m, int64_t d, int64_t stride, const float* __restrict__ lo,
                const float* __restrict__ hi, int pass, PcbState* __restrict__ st, uint32_t* __restrict__ hist,
                uint32_t* __restrict__ skeys, int ieee, int64_t s0, int64_t j_off, int64_t n_s) {
    extern __shared__ uint32_t s_hist[];  // K * kPcbBins
    __shared__ PcbClamp<K> s_c;
    __shared__ uint32_t s_prefix[K];
    for (int i = threadIdx.x; i < K * kPcbBins; i += blockDim.x) s_hist[i] = 0;
    s_c.load(lo, hi);
    if (threadIdx.x < K) s_prefix[threadIdx.x] = pass ? st[threadIdx.x].prefix : 0;
    __syncthreads();
    uint32_t mx[K];
#pragma unroll
    for (int k = 0; k < K; ++k) mx[k] = 0;
    const int64_t tail0 = d & ~(int64_t)31;
    const int64_t span = (int64_t)gridDim.x * blockDim.x;
    const int64_t n_vis = SLICE ? n_s : (stride == 1 ? d : pcb_sample_count(d, stride));
    const int64_t rounds = (n_vis + span - 1) / span;  // every lane runs every round (the match below is warp-wide)
    auto sweep = [&](auto safe_tag) {
    constexpr bool SAFE = decltype(safe_tag)::value;
    for (int64_t it = 0; it < rounds; ++it) {
        const int64_t i = it * span + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        const bool live = i < n_vis;
        const int64_t j = !live ? 0 : (SLICE ? pcb_sample_column(s0 + i, stride) - j_off
                                             : (stride == 1 ? i : pcb_sample_column(i, stride)));
        float x[K], tau[K], A[K], task[K];
        const float b = live ? ldg_stream1(base + j) : 0.f;
#pragma unroll
        for (int k = 0; k < K; ++k) x[k] = live ? ldg_stream1(m.p[k] + j) : 0.f;
        pcb_task<K, SAFE>(b, x, s_c, j >= tail0, tau, A, task);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const uint32_t key = pcb_key(task[k]);
            int bin = -1;
            if (live) {
                if (pass == 0) { bin = (int)(key >> 21); mx[k] = key > mx[k] ? key : mx[k]; }
                else if (pass == 1) { if ((key >> 21) == s_prefix[k]) bin = (int)((key >> 10) & 2047u); }
                else { if ((key >> 10) == s_prefix[k]) bin = (int)(key & 1023u); }
                if (skeys) skeys[(int64_t)k * n_vis + i] = key;
            }
            const uint32_t peers = __match_any_sync(0xffffffffu, bin);  // one shared-memory atomic per distinct bin
            if (bin >= 0 && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&s_hist[k * kPcbBins + bin], __popc(peers));
        }
    }
    };
    if (ieee) sweep(std::false_type{}); else sweep(std::true_type{});   // kernel-uniform
    if (pass == 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            uint32_t v = mx[k];
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) {
                const uint32_t o = __shfl_xor_sync(0xffffffffu, v, off);
                v = o > v ? o : v;
            }
            if ((threadIdx.x & 31) == 0 && v) atomicMax(&st[k].maxkey, v);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < K * kPcbBins; i += blockDim.x)
        if (s_hist[i]) atomicAdd(&hist[i], s_hist[i]);
}

// Radix passes 1 and 2 of the sample select, over the cached keys: grid (blocks, K), both slots in one sweep.
// hist layout: (slot, model, bin).
__global__ void __launch_bounds__(kPcbThreads)
pcb_keys_hist_kernel(const uint32_t* __restrict__ skeys, int64_t n_s, int K, int pass, const PcbState* __restrict__ st,
                     uint32_t* __restrict__ hist) {
    __shared__ uint32_t s_hist[kPcbSlots * kPcbBins];
    const int k = blockIdx.y;
    for (int i = threadIdx.x; i < kPcbSlots * kPcbBins; i += blockDim.x) s_hist[i] = 0;
    uint32_t prefix[kPcbSlots];
#pragma unroll
    for (int s = 0; s < kPcbSlots; ++s) prefix[s] = st[s * K + k].prefix;
    __syncthreads();
    const uint32_t* keys = skeys + (int64_t)k * n_s;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_s; i += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t key = keys[i];
#pragma unroll
        for (int s = 0; s < kPcbSlots; ++s) {
            if (pass == 1) { if ((key >> 21) == prefix[s]) atomicAdd(&s_hist[s * kPcbBins + ((key >> 10) & 2047u)], 1u); }
            else { if ((key >> 10) == prefix[s]) atomicAdd(&s_hist[s * kPcbBins + (key & 1023u)], 1u); }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kPcbSlots * kPcbBins; i += blockDim.x)
        if (s_hist[i]) atomicAdd(&hist[((size_t)(i / kPcbBins) * K + k) * kPcbBins + (i % kPcbBins)], s_hist[i]);
}

// Block-wide (256 threads, 8 bins each) search of the first bin whose cumulative count exceeds `rank`: returns the bin
// and the count below it; a rank beyond the total returns the last bin and the total (the callers treat that as a miss).
__device__ __forceinline__ void pcb_find_bin(const uint32_t* __restrict__ h, int width, int64_t rank, int& chosen, int64_t& cum,
                                             int64_t& total) {
    __shared__ int64_t s_warp[8];
    __shared__ int64_t s_cum;
    __shared__ int s_chosen;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    uint32_t c[8];
    int64_t loc = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int b = t * 8 + i;
        c[i] = b < width ? h[b] : 0u;
        loc += c[i];
    }
    int64_t inc = loc;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int64_t v = __shfl_up_sync(0xffffffffu, inc, off);
        if (lane >= off) inc += v;
    }
    if (lane == 31) s_warp[warp] = inc;
    if (t == 0) s_chosen = -1;
    __syncthreads();
    int64_t before = 0;
    total = 0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
        if (w < warp) before += s_warp[w];
        total += s_warp[w];
    }
    int64_t run = before + inc - loc;
    if (rank >= run && rank < run + loc) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            if (rank < run + c[i]) { s_chosen = t * 8 + i; s_cum = run; break; }
            run += c[i];
        }
    }
    __syncthreads();
    if (s_chosen < 0) { chosen = width - 1; cum = total; }
    else { chosen = s_chosen; cum = s_cum; }
}

// grid (K, slots), 256 threads: find the bucket holding the slot's rank.  shared_hist = 1: every slot reads the
// histogram of slot 0 (pass 0 of the sample select).  The caller clears the histograms afterwards.
__global__ void __launch_bounds__(256)
pcb_pick_kernel(int pass, int K, int shared_hist, PcbState* __restrict__ st, const uint32_t* __restrict__ hist) {
    const int k = blockIdx.x, s = blockIdx.y;
    const uint32_t* h = hist + ((size_t)(shared_hist ? 0 : s) * K + k) * kPcbBins;
    PcbState& S = st[s * K + k];
    const int64_t rank = S.rank;
    int chosen;
    int64_t cum, total;
    pcb_find_bin(h, kPcbBins, rank, chosen, cum, total);
    if (threadIdx.x == 0) {
        S.rank = rank - cum;
        const uint32_t p = (pass == 0) ? (uint32_t)chosen : ((S.prefix << (pass == 1 ? 11 : 10)) | (uint32_t)chosen);
        S.prefix = p;
        if (pass == 2) S.qkey = p;
    }
}

// ---- windowed search (fast path) -----------------------------------------------------------------------------------
// One pass over the whole vector: elements BELOW the window are counted in registers, the keys of the elements inside
// it are appended to the warp's private list of the model (the warp-wide ballot gives every lane its slot; the running
// count is a warp-uniform register: no atomics, no shared memory).  An overflowing list sets `miss`.
template <int K, bool VEC>
__global__ void __launch_bounds__(kPcbThreads, K <= 8 ? 2 : 1)
pcb_window_kernel(const float* __restrict__ base, PtrPack<K> m, int64_t d, const float* __restrict__ lo,
                  const float* __restrict__ hi, PcbState* __restrict__ st, unsigned long long* __restrict__ below_out,
                  uint32_t* __restrict__ list_keys, uint32_t* __restrict__ list_cnt, int list_cap, int ieee) {
    __shared__ PcbClamp<K> s_c;
    __shared__ uint32_t s_wlo[K], s_wspan[K];
    s_c.load(lo, hi);
    if (threadIdx.x < K) {
        s_wlo[threadIdx.x] = st[threadIdx.x].wlo;
        s_wspan[threadIdx.x] = st[threadIdx.x].wspan;
    }
    __syncthreads();
    uint32_t mx[K], below[K], cnt[K];
#pragma unroll
    for (int k = 0; k < K; ++k) { mx[k] = 0; below[k] = 0; cnt[k] = 0; }
    const int lane = threadIdx.x & 31;
    const uint32_t lt_mask = (1u << lane) - 1u;
    const int64_t n_lists = (int64_t)gridDim.x * kPcbWarps;
    const int64_t wlist = (int64_t)blockIdx.x * kPcbWarps + (threadIdx.x >> 5);
    const int64_t tail0 = d & ~(int64_t)31;
    const int64_t nq = (d + 3) >> 2;
    const int64_t span = (int64_t)gridDim.x * blockDim.x;
    const int64_t rounds = (nq + span - 1) / span;   // every lane runs every round (the ballots are warp-wide)
    auto sweep = [&](auto safe_tag) {
    constexpr bool SAFE = decltype(safe_tag)::value;
    for (int64_t it = 0; it < rounds; ++it) {
        const int64_t q = it * span + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        float bx[4], xs[K][4];
        const int nvalid = pcb_load_quad<K, VEC>(base, m, d, q, q < nq, bx, xs);
        const bool tail = (q << 2) >= tail0;          // tail0 is a multiple of 32: a quad never straddles it
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            float x[K], tau[K], A[K], task[K];
#pragma unroll
            for (int k = 0; k < K; ++k) x[k] = xs[k][c];
            pcb_task<K, SAFE>(bx[c], x, s_c, tail, tau, A, task);
            const bool ok = c < nvalid;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const uint32_t key = pcb_key(task[k]);
                const uint32_t wl = s_wlo[k];
                const bool in = ok && (key - wl) <= s_wspan[k];   // key < wl wraps to more than any span
                below[k] += (ok && key < wl) ? 1u : 0u;
                mx[k] = (ok && key > mx[k]) ? key : mx[k];
                const uint32_t hits = __ballot_sync(0xffffffffu, in);
                if (hits) {
                    const uint32_t pos = cnt[k] + __popc(hits & lt_mask);
                    if (in && pos < (uint32_t)list_cap) list_keys[((int64_t)k * n_lists + wlist) * list_cap + pos] = key;
                    cnt[k] += __popc(hits);
                }
            }
        }
    }
    };
    if (ieee) sweep(std::false_type{}); else sweep(std::true_type{});   // kernel-uniform
#pragma unroll
    for (int k = 0; k < K; ++k) {
        uint32_t v = below[k], mv = mx[k];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            v += __shfl_xor_sync(0xffffffffu, v, off);
            const uint32_t o = __shfl_xor_sync(0xffffffffu, mv, off);
            mv = o > mv ? o : mv;
        }
        if (lane == 0) {
            if (v) atomicAdd(&below_out[k], (unsigned long long)v);
            if (mv) atomicMax(&st[k].maxkey, mv);
            list_cnt[(int64_t)k * n_lists + wlist] = cnt[k];
            if (cnt[k] > (uint32_t)list_cap) atomicExch(&st[k].miss, 1);
        }
    }
}

// One refinement level over the collected keys: one warp per list, grid (blocks, K), a shared-memory histogram of the
// current window (wwidth bins of 2^wshift keys) per CTA.
__global__ void __launch_bounds__(kPcbThreads)
pcb_list_hist_kernel(const uint32_t* __restrict__ list_keys, const uint32_t* __restrict__ list_cnt, int64_t n_lists,
                     int list_cap, const PcbState* __restrict__ st, uint32_t* __restrict__ hist) {
    __shared__ uint32_t s_hist[kPcbBins];
    const int k = blockIdx.y;
    const PcbState S = st[k];
    if (S.miss || S.done) return;
    for (int i = threadIdx.x; i < kPcbBins; i += blockDim.x) s_hist[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    for (int64_t w = (int64_t)blockIdx.x * kPcbWarps + (threadIdx.x >> 5); w < n_lists; w += (int64_t)gridDim.x * kPcbWarps) {
        uint32_t n = list_cnt[(int64_t)k * n_lists + w];
        if (n > (uint32_t)list_cap) n = (uint32_t)list_cap;
        const uint32_t* keys = list_keys + ((int64_t)k * n_lists + w) * list_cap;
        for (uint32_t e = lane; e < n; e += 32) {
            const uint32_t key = keys[e];
            if (key >= S.wlo) {
                const uint32_t bin = (key - S.wlo) >> S.wshift;
                if (bin < (uint32_t)S.wwidth) atomicAdd(&s_hist[bin], 1u);
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kPcbBins; i += blockDim.x)
        if (s_hist[i]) atomicAdd(&hist[(size_t)k * kPcbBins + i], s_hist[i]);
}

// after the sample select: the window spans the two sample order statistics (slot 0 = start, slot 1 = end; an open end
// is the smallest / largest key)
__global__ void pcb_window_init_kernel(PcbState* st, int K, int64_t q_index, int lo_open, int hi_open) {
    const int k = threadIdx.x;
    if (k < K) {
        const uint32_t a = lo_open ? 0u : st[k].qkey;
        const uint32_t b = hi_open ? 0xFFFFFFFFu : st[K + k].qkey;
        const uint64_t width = (uint64_t)(b >= a ? b - a : 0u) + 1u;    // keys in [a, b]
        int sh = 0;
        while (((uint64_t)kPcbBins << sh) < width) ++sh;
        st[k].wlo = a;
        st[k].wspan = (uint32_t)(width - 1);
        st[k].wshift = sh;
        st[k].wwidth = (int32_t)((width + ((uint64_t)1 << sh) - 1) >> sh);
        st[k].rank = q_index;      // ascending rank wanted in the FULL vector
        st[k].maxkey = 0;          // the sample's maximum is not the row maximum
        st[k].miss = 0;
        st[k].done = 0;
    }
}

// one block of 256 threads per model: find the window bin that holds the wanted rank; the first level subtracts what lies
// below the window
__global__ void __launch_bounds__(256)
pcb_window_pick_kernel(int first, PcbState* __restrict__ st, uint32_t* __restrict__ hist, unsigned long long* __restrict__ below) {
    const int k = blockIdx.x;
    uint32_t* h = hist + (size_t)k * kPcbBins;
    const bool active = !st[k].miss && !st[k].done;   // block-uniform
    if (active) {
        int64_t rank = st[k].rank;
        const int width = st[k].wwidth;
        const int64_t bl = first ? (int64_t)below[k] : 0;
        rank -= bl;
        int chosen;
        int64_t cum, total;
        pcb_find_bin(h, width, rank, chosen, cum, total);
        if (threadIdx.x == 0) {
            if (first && (rank < 0 || rank >= total)) {
                st[k].miss = 1;
            } else {
                const int sh = st[k].wshift;
                const uint32_t nlo = st[k].wlo + ((uint32_t)chosen << sh);
                st[k].rank = rank - cum;
                st[k].wlo = nlo;
                if (sh == 0) {
                    st[k].qkey = nlo;
                    st[k].done = 1;
                } else {
                    const int nsh = sh > 11 ? sh - 11 : 0;
                    st[k].wwidth = (1 << sh) >> nsh;
                    st[k].wshift = nsh;
                }
            }
        }
    }
    __syncthreads();
    for (int b = threadIdx.x; b < kPcbBins; b += blockDim.x) h[b] = 0;
    if (threadIdx.x == 0) below[k] = 0;
}

// status per model: 1 = exact result; 0 = the fast search missed (rerun with MR_PCB_DENSE); 2 = a clamp or a divisor
// of the fast division sequences lies outside [2^-60, 2^60] (rerun with MR_PCB_IEEE).  With ieee set the range is moot.
__global__ void pcb_status_kernel(const PcbState* st, int K, int fast, int ieee, const float* __restrict__ lo,
                                  const float* __restrict__ hi, int32_t* status) {
    const int k = threadIdx.x;
    if (k < K) {
        const float span = __fsub_rn(pcb_unkey(st[k].maxkey), pcb_unkey(st[k].qkey));
        const bool safe = ieee || (pcb_safe_range(hi[k]) && pcb_safe_range(__fsub_rn(hi[k], lo[k])) && pcb_safe_range(span));
        const bool found = !(st[k].miss || (fast && !st[k].done));
        status[k] = !found ? 0 : (safe ? 1 : 2);
    }
}

// rank0 / rank1: the ascending ranks the two slots search (the dense search uses slot 0 only)
__global__ void pcb_init_kernel(PcbState* st, int K, int64_t rank0, int64_t rank1) {
    const int i = threadIdx.x;
    if (i < kPcbSlots * K) {
        PcbState s;
        s.prefix = 0; s.maxkey = 0; s.rank = i < K ? rank0 : rank1; s.qkey = 0;
        s.wlo = 0; s.wshift = 0; s.wwidth = 0; s.miss = 0; s.done = 0; s.wspan = 0; s.pad = 0;
        st[i] = s;
    }
}

// Sharded search: the row maxima and the window-overflow flags of every rank meet in a region that is all-reduced with MAX
// as int32 words -- [maxkey ^ 0x80000000 (K) | miss (K)]: the xor maps the unsigned key order onto the signed order.
__global__ void pcb_export_kernel(const PcbState* st, int K, int32_t* maxreg) {
    const int k = threadIdx.x;
    if (k < K) {
        maxreg[k] = (int32_t)(st[k].maxkey ^ 0x80000000u);
        maxreg[K + k] = st[k].miss;
    }
}
__global__ void pcb_import_kernel(PcbState* st, int K, const int32_t* maxreg) {
    const int k = threadIdx.x;
    if (k < K) {
        st[k].maxkey = (uint32_t)maxreg[k] ^ 0x80000000u;
        st[k].miss = maxreg[K + k] != 0;
    }
}

template <int K, bool VEC>
__global__ void __launch_bounds__(kPcbThreads, K <= 8 ? 2 : 1)
pcb_build_kernel(const float* __restrict__ base, PtrPack<K> m, int64_t d, const float* __restrict__ lo,
                 const float* __restrict__ hi, const PcbState* __restrict__ st, float* __restrict__ out, int64_t ldo,
                 float* __restrict__ task_out, float* __restrict__ thr_out, int ieee) {
    __shared__ PcbClamp<K> s_c;
    __shared__ float s_q[K], s_max[K], s_span[K], s_rspan[K];
    s_c.load(lo, hi);
    if (threadIdx.x < K) {
        const float qv = pcb_unkey(st[threadIdx.x].qkey), mv = pcb_unkey(st[threadIdx.x].maxkey);
        const float y = __fsub_rn(mv, qv);
        s_q[threadIdx.x] = qv; s_max[threadIdx.x] = mv;
        s_span[threadIdx.x] = y; s_rspan[threadIdx.x] = pcb_safe_range(y) ? __frcp_rn(y) : 0.0f;
        if (thr_out && blockIdx.x == 0) {
            thr_out[2 * threadIdx.x] = qv;
            thr_out[2 * threadIdx.x + 1] = mv;
        }
    }
    __syncthreads();
    const float inv_n = __fdiv_rn(1.0f, (float)K);
    const int64_t tail0 = d & ~(int64_t)31;
    const int64_t nq = (d + 3) >> 2;
    const int64_t span = (int64_t)gridDim.x * blockDim.x;
    auto sweep = [&](auto safe_tag) {
    constexpr bool SAFE = decltype(safe_tag)::value;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += span) {
        float bx[4], xs[K][4];
        const int nvalid = pcb_load_quad<K, VEC>(base, m, d, q, true, bx, xs);
        const int64_t j0 = q << 2;
        const bool tail = j0 >= tail0;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            float x[K], tau[K], A[K], task[K], scale[K];
#pragma unroll
            for (int k = 0; k < K; ++k) x[k] = xs[k][c];
            pcb_task<K, SAFE>(bx[c], x, s_c, tail, tau, A, task);
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const float cl = fminf(fmaxf(task[k], s_q[k]), s_max[k]);
                scale[k] = pcb_div_by<SAFE>(__fsub_rn(cl, s_q[k]), s_span[k], s_rspan[k]);
            }
            // in [1e-12, K], or NaN: under IEEE divides (the rerun of status 2) a model whose range is 0 -- it equals
            // the base -- has NaN scales, and pcb.py's clamp(sum, min=1e-12) keeps the NaN where fmaxf alone returns
            // 1e-12.  The fast divisions only run with every divisor in range: their scales are never NaN.
            const float ssum = torch_sum_dim0<K>(scale, tail);
            const float denom = (!SAFE && ssum != ssum) ? ssum : fmaxf(ssum, (float)1e-12);
            const float rden = SAFE ? __frcp_rn(denom) : 0.0f;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                // pcb.py:54-56: sign(tau) A scale / denom / n.  Round-to-nearest commutes with the sign, so the
                // quotients are taken of the magnitude (A scale >= +0: a zero needs no special case) and the sign goes
                // on last; sign(0) = 0 makes the whole product +0, unless scale / denom is NaN (0 * NaN; IEEE divides only).
                const float w = pcb_div_count<SAFE>(pcb_div_by<SAFE>(__fmul_rn(A[k], scale[k]), denom, rden), (float)K, inv_n);
                xs[k][c] = (tau[k] != 0.0f) ? copysignf(w, tau[k]) : ((!SAFE && w != w) ? w : 0.0f);   // the input is dead: reuse its register
                if (task_out && c < nvalid) task_out[(int64_t)k * ldo + j0 + c] = task[k];
            }
        }
#pragma unroll
        for (int k = 0; k < K; ++k) {
            float* o = out + (int64_t)k * ldo + j0;
            if (VEC && nvalid == 4) stg_stream4(o, make_float4(xs[k][0], xs[k][1], xs[k][2], xs[k][3]));
            else
#pragma unroll
                for (int c = 0; c < 4; ++c) if (c < nvalid) o[c] = xs[k][c];
        }
    }
    };
    if (ieee) sweep(std::false_type{}); else sweep(std::true_type{});   // kernel-uniform
}

static inline size_t pcb_align256(size_t x) { return (x + 255) & ~(size_t)255; }

// Workspace layout.  n_s: the sample keys cached here; n_s_win: the sample the window is derived from (the whole vector's,
// which the per-warp lists are sized for).  Sizes depend on those, K and the SM count only, so query and launch agree.
struct PcbWs {
    size_t state_off, hist_off, below_off, cnt_off, keys_off, skeys_off, total;
    int64_t n_s;          // sample size
    int64_t list_total;   // list capacity per model over all warps (in keys)
    int64_t max_lists;    // upper bound on the number of warp lists
};
static PcbWs pcb_layout_n(int64_t n_s, int64_t n_s_win, int K) {
    PcbWs L;
    L.n_s = n_s;
    // sampling error of an order statistic of the sample: sigma <= sqrt(n_s) / 2 ranks; the window spans +-R = 6 sigma
    // + 16 sample ranks, i.e. about 2 R * stride elements of the full vector -- provisioned four times over
    const int64_t r_max = (int64_t)(3.0 * sqrt((double)n_s_win)) + 16;
    L.max_lists = (int64_t)sm_count() * 8 * kPcbWarps;
    L.list_total = 4 * 2 * r_max * kPcbStride + 64 * L.max_lists;
    size_t off = 0;
    L.state_off = off; off += pcb_align256((size_t)kPcbSlots * MR_MAX_K * sizeof(PcbState));
    L.hist_off = off;  off += pcb_align256((size_t)kPcbSlots * K * kPcbBins * sizeof(uint32_t));
    L.below_off = off; off += pcb_align256((size_t)MR_MAX_K * sizeof(unsigned long long));
    L.cnt_off = off;   off += pcb_align256((size_t)K * L.max_lists * sizeof(uint32_t));
    L.keys_off = off;  off += pcb_align256((size_t)K * L.list_total * sizeof(uint32_t));
    L.skeys_off = off; off += pcb_align256((size_t)K * L.n_s * sizeof(uint32_t));
    L.total = off;
    return L;
}
static PcbWs pcb_layout(int64_t d, int K) {
    const int64_t n_s = pcb_sample_count(d, kPcbStride);
    return pcb_layout_n(n_s, n_s, K);
}
// bytes of the histograms (both slots) and the below-window counters, which sit back to back
static size_t pcb_counter_bytes(const PcbWs& L) { return L.below_off + (size_t)MR_MAX_K * sizeof(unsigned long long) - L.hist_off; }

// The fast search runs where the sample is large enough to be worth it (small vectors: the dense passes are cheap and
// exact anyway).  Sharded: decided from the WHOLE vector, so that every rank takes the same path.
static bool pcb_fast(int64_t d, int flags) { return !(flags & MR_PCB_DENSE) && pcb_sample_count(d, kPcbStride) >= 4096; }

// ranks of the window's ends inside the sample (the sample's quantile +- R, R = 6 sigma of the sampling error); an end
// clipped to the sample is open
static void pcb_window_ranks(int64_t q_index, int64_t d, int64_t n_s, int64_t* r_lo, int64_t* r_hi, int* lo_open, int* hi_open) {
    const long double p = (long double)q_index / (long double)d;
    const int64_t q_s = (int64_t)(p * (long double)n_s);
    const int64_t R = (int64_t)(6.0 * sqrt((double)n_s * (double)(p * (1.0L - p)))) + 16;
    *r_lo = q_s - R; *r_hi = q_s + R;
    *lo_open = *hi_open = 0;
    if (*r_lo < 0) { *r_lo = 0; *lo_open = 1; }
    if (*r_hi > n_s - 1) { *r_hi = n_s - 1; *hi_open = 1; }
}

// The elements [s0, s0 + n) of the whole vector's sample that lie in the slice [j_off, j_off + d_local): every whole
// block of 4 * stride columns inside the slice, plus a block straddling a slice boundary when its sampled quad falls
// inside (quads are 4-aligned, slice boundaries 32-aligned or the vector's end: a quad never straddles one).  Over the
// ranks of a sharded vector the ranges partition the sample.
static void pcb_slice_sample(int64_t d_local, int64_t j_off, int64_t d_global, int64_t* s0, int64_t* n) {
    const int64_t blk = 4 * kPcbStride;
    int64_t c0 = j_off / blk, c1 = (j_off + d_local + blk - 1) / blk;
    if (c1 > d_global / blk) c1 = d_global / blk;                  // only whole blocks are sampled
    auto inside = [&](int64_t c) {
        const int64_t j = pcb_sample_column(4 * c, kPcbStride);
        return j >= j_off && j < j_off + d_local;
    };
    if (c0 < c1 && !inside(c0)) ++c0;
    if (c0 < c1 && !inside(c1 - 1)) --c1;
    if (c1 < c0) c1 = c0;
    *s0 = 4 * c0;
    *n = 4 * (c1 - c0);
}

// ---- launchers shared by the single-GPU and the sharded entry points ------------------------------------------------
// n_vis: the elements the pass visits (d, or the sample size); slice != 0: the sharded sample pass (pcb_hist_kernel SLICE)
template <int K>
static void pcb_launch_hist(const float* base, const PtrPack<K>& pk, int64_t d, int64_t stride, int64_t n_vis, bool slice,
                            int64_t s0, int64_t j_off, const float* lo, const float* hi, int pass, PcbState* state,
                            uint32_t* hist, uint32_t* skeys, int ieee, cudaStream_t st) {
    if (n_vis <= 0) return;
    const size_t hist_bytes = (size_t)K * kPcbBins * sizeof(uint32_t);
    int64_t hblocks = (n_vis + kPcbThreads - 1) / kPcbThreads;
    const int64_t hcap = (int64_t)sm_count() * 3;         // one resident wave at K = 8 (64 KB of histograms per CTA)
    if (hblocks > hcap) hblocks = hcap;
    if (slice) {
        cudaFuncSetAttribute(pcb_hist_kernel<K, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hist_bytes);
        pcb_hist_kernel<K, true><<<(unsigned)hblocks, kPcbThreads, hist_bytes, st>>>(base, pk, d, stride, lo, hi, pass, state,
                                                                                    hist, skeys, ieee, s0, j_off, n_vis);
    } else {
        cudaFuncSetAttribute(pcb_hist_kernel<K, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hist_bytes);
        pcb_hist_kernel<K, false><<<(unsigned)hblocks, kPcbThreads, hist_bytes, st>>>(base, pk, d, stride, lo, hi, pass, state,
                                                                                     hist, skeys, ieee, 0, 0, 0);
    }
}

static void pcb_launch_keys_hist(const uint32_t* skeys, int64_t n_s, int K, int pass, const PcbState* state, uint32_t* hist,
                                 cudaStream_t st) {
    if (n_s <= 0) return;
    int64_t kblocks = (n_s + kPcbThreads * 8 - 1) / (kPcbThreads * 8);
    if (kblocks > sm_count()) kblocks = sm_count();
    pcb_keys_hist_kernel<<<dim3((unsigned)kblocks, K), kPcbThreads, 0, st>>>(skeys, n_s, K, pass, state, hist);
}

// the pass over everything: one resident wave, one list per warp; the number of lists (0: nothing to do) -- the list
// kernels of a search must use the count its window pass used
template <int K>
static int64_t pcb_window_lists(int64_t d, bool vec) {
    if (d <= 0) return 0;
    int occ = 1;
    if (vec) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pcb_window_kernel<K, true>, kPcbThreads, 0);
    else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pcb_window_kernel<K, false>, kPcbThreads, 0);
    if (occ < 1) occ = 1;
    if (occ > 8) occ = 8;
    int64_t wblocks = (int64_t)sm_count() * occ;
    const int64_t nq = (d + 3) >> 2;
    if (wblocks > (nq + kPcbThreads - 1) / kPcbThreads) wblocks = (nq + kPcbThreads - 1) / kPcbThreads;
    return wblocks * kPcbWarps;
}
static int pcb_list_cap(const PcbWs& L, int64_t n_lists) { return (int)((L.list_total / n_lists) & ~(int64_t)31); }

template <int K>
static void pcb_launch_window(const float* base, const PtrPack<K>& pk, int64_t d, bool vec, const float* lo, const float* hi,
                              PcbState* state, unsigned long long* below, uint32_t* list_keys, uint32_t* list_cnt,
                              int64_t n_lists, const PcbWs& L, int ieee, cudaStream_t st) {
    if (!n_lists) return;
    const unsigned wblocks = (unsigned)(n_lists / kPcbWarps);
    const int list_cap = pcb_list_cap(L, n_lists);
    if (vec)
        pcb_window_kernel<K, true><<<wblocks, kPcbThreads, 0, st>>>(base, pk, d, lo, hi, state, below, list_keys, list_cnt,
                                                                    list_cap, ieee);
    else
        pcb_window_kernel<K, false><<<wblocks, kPcbThreads, 0, st>>>(base, pk, d, lo, hi, state, below, list_keys, list_cnt,
                                                                     list_cap, ieee);
}

static void pcb_launch_list_hist(int K, const uint32_t* list_keys, const uint32_t* list_cnt, int64_t n_lists, const PcbWs& L,
                                 const PcbState* state, uint32_t* hist, cudaStream_t st) {
    if (!n_lists) return;
    int64_t lblocks = (n_lists + kPcbWarps - 1) / kPcbWarps;
    if (lblocks > sm_count()) lblocks = sm_count();
    pcb_list_hist_kernel<<<dim3((unsigned)lblocks, K), kPcbThreads, 0, st>>>(list_keys, list_cnt, n_lists, pcb_list_cap(L, n_lists),
                                                                            state, hist);
}

template <int K>
static void pcb_launch_build(const float* base, const PtrPack<K>& pk, int64_t d, bool vec, const float* lo, const float* hi,
                             const PcbState* state, float* out, int64_t ldo, float* task_out, float* thr_out, int ieee,
                             cudaStream_t st) {
    if (d <= 0) return;
    int64_t bblocks = (((d + 3) >> 2) + kPcbThreads - 1) / kPcbThreads;
    if (bblocks > (int64_t)sm_count() * 8) bblocks = (int64_t)sm_count() * 8;
    if (vec)
        pcb_build_kernel<K, true><<<(unsigned)bblocks, kPcbThreads, 0, st>>>(base, pk, d, lo, hi, state, out, ldo, task_out,
                                                                             thr_out, ieee);
    else
        pcb_build_kernel<K, false><<<(unsigned)bblocks, kPcbThreads, 0, st>>>(base, pk, d, lo, hi, state, out, ldo, task_out,
                                                                              thr_out, ieee);
}

static bool pcb_vec(const float* base, const float* const* models, int K, const float* out, int64_t ldo, const float* task_out) {
    bool vec = host_aligned16(base) && host_aligned16(out) && (ldo % 4 == 0) && (!task_out || host_aligned16(task_out));
    for (int k = 0; k < K; ++k) vec = vec && host_aligned16(models[k]);
    return vec;
}

// Sharded search: the workspace is the single-GPU one with the sample cache sized for the slice, the lists sized for
// the whole vector's window, and the MAX region behind it.
struct PcbDistWs {
    PcbWs L;
    size_t max_off, max_bytes, total;
};
static PcbDistWs pcb_dist_layout(int64_t d_local, int64_t d_global, int K) {
    PcbDistWs D;
    // a slice of d_local columns meets at most d_local / 128 + 2 sampled blocks
    D.L = pcb_layout_n(4 * (d_local / (4 * kPcbStride) + 2), pcb_sample_count(d_global, kPcbStride), K);
    D.max_off = D.L.total;
    D.max_bytes = (size_t)2 * K * sizeof(int32_t);
    D.total = D.max_off + pcb_align256(D.max_bytes);
    return D;
}

}  // namespace mr

extern "C" int64_t mr_pcb_workspace_bytes(int64_t d, int K) {
    if (K < 1 || K > MR_MAX_K || d < 1) return 0;
    return (int64_t)mr::pcb_layout(d, K).total;
}

extern "C" int mr_pcb_vectors(const float* base, const float* const* models, int K, int64_t d, const float* clamp_lo,
                              const float* clamp_hi, int64_t q_index, int flags, int32_t* status, float* out, int64_t ldo,
                              float* task_out, float* thr_out, void* ws, int64_t ws_bytes, mr_stream_t stream) {
    using namespace mr;
    MR_REQUIRE(K >= 1 && K <= MR_MAX_K, "mr_pcb_vectors: K=%d outside [1,%d]", K, MR_MAX_K);
    MR_REQUIRE(base && models && clamp_lo && clamp_hi && out && ws && status, "mr_pcb_vectors: null pointer");
    MR_REQUIRE(d >= 1 && d < ((int64_t)1 << 32), "mr_pcb_vectors: d=%lld outside [1, 2^32)", (long long)d);
    MR_REQUIRE(q_index >= 0 && q_index < d, "mr_pcb_vectors: quantile index %lld outside [0,d)", (long long)q_index);
    MR_REQUIRE(ldo >= d, "mr_pcb_vectors: need ldo >= d");
    for (int k = 0; k < K; ++k) MR_REQUIRE(models[k] != nullptr, "mr_pcb_vectors: models[%d] is NULL", k);
    const PcbWs L = pcb_layout(d, K);
    if (ws_bytes < (int64_t)L.total) {
        set_error("mr_pcb_vectors: workspace too small (%lld < %lld bytes)", (long long)ws_bytes, (long long)L.total);
        return MR_ERR_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    char* w = reinterpret_cast<char*>(ws);
    PcbState* state = reinterpret_cast<PcbState*>(w + L.state_off);
    uint32_t* hist = reinterpret_cast<uint32_t*>(w + L.hist_off);
    unsigned long long* below = reinterpret_cast<unsigned long long*>(w + L.below_off);
    uint32_t* list_cnt = reinterpret_cast<uint32_t*>(w + L.cnt_off);
    uint32_t* list_keys = reinterpret_cast<uint32_t*>(w + L.keys_off);
    uint32_t* skeys = reinterpret_cast<uint32_t*>(w + L.skeys_off);
    const size_t hist_bytes = (size_t)K * kPcbBins * sizeof(uint32_t);           // one histogram per model
    cudaMemsetAsync(hist, 0, pcb_counter_bytes(L), st);                           // both slots + below
    const int64_t n_s = L.n_s;
    const int ieee = (flags & MR_PCB_IEEE) ? 1 : 0;
    const bool fast = pcb_fast(d, flags);
    int64_t r_lo = q_index, r_hi = q_index;
    int lo_open = 0, hi_open = 0;
    if (fast) pcb_window_ranks(q_index, d, n_s, &r_lo, &r_hi, &lo_open, &hi_open);
    pcb_init_kernel<<<1, 64, 0, st>>>(state, K, r_lo, r_hi);
    const bool vec = pcb_vec(base, models, K, out, ldo, task_out);
    MR_DISPATCH_K(K, {
        PtrPack<KK> pk;
        for (int k = 0; k < KK; ++k) pk.p[k] = models[k];
        if (!fast) {
            for (int pass = 0; pass < 3; ++pass) {      // dense radix passes over everything
                pcb_launch_hist<KK>(base, pk, d, 1, d, false, 0, 0, clamp_lo, clamp_hi, pass, state, hist, nullptr, ieee, st);
                pcb_pick_kernel<<<dim3(KK, 1), 256, 0, st>>>(pass, KK, 0, state, hist);
                cudaMemsetAsync(hist, 0, hist_bytes, st);
            }
        } else {
            // the sample: one pass computes and caches its keys, passes 1 and 2 of both order statistics read the cache
            pcb_launch_hist<KK>(base, pk, d, kPcbStride, n_s, false, 0, 0, clamp_lo, clamp_hi, 0, state, hist, skeys, ieee, st);
            pcb_pick_kernel<<<dim3(KK, kPcbSlots), 256, 0, st>>>(0, KK, 1, state, hist);
            cudaMemsetAsync(hist, 0, kPcbSlots * hist_bytes, st);
            for (int pass = 1; pass < 3; ++pass) {
                pcb_launch_keys_hist(skeys, n_s, KK, pass, state, hist, st);
                pcb_pick_kernel<<<dim3(KK, kPcbSlots), 256, 0, st>>>(pass, KK, 0, state, hist);
                cudaMemsetAsync(hist, 0, kPcbSlots * hist_bytes, st);
            }
            pcb_window_init_kernel<<<1, 32, 0, st>>>(state, KK, q_index, lo_open, hi_open);
            const int64_t n_lists = pcb_window_lists<KK>(d, vec);
            pcb_launch_window<KK>(base, pk, d, vec, clamp_lo, clamp_hi, state, below, list_keys, list_cnt, n_lists, L, ieee, st);
            for (int level = 0; level < 3; ++level) {   // 2048 bins x 2^21 keys cover the key space: three levels at most
                pcb_launch_list_hist(KK, list_keys, list_cnt, n_lists, L, state, hist, st);
                pcb_window_pick_kernel<<<KK, 256, 0, st>>>(level == 0, state, hist, below);
            }
        }
        pcb_status_kernel<<<1, 32, 0, st>>>(state, KK, fast ? 1 : 0, ieee, clamp_lo, clamp_hi, status);
        pcb_launch_build<KK>(base, pk, d, vec, clamp_lo, clamp_hi, state, out, ldo, task_out, thr_out, ieee, st);
    });
    MR_CUDA_LAUNCH_CHECK("mr_pcb_vectors");
    return MR_OK;
}

// ---- sharded search ----------------------------------------------------------------------------------------------------
// The same kernels over one rank's slice, split into phases at the points where the single-GPU search reads a count of
// the whole vector.  After each phase but the last the caller all-reduces, over the ranks, the regions that
// mr_pcb_dist_plan names (the library itself never communicates):
//   fast search (7 phases)                                                     dense search (4 phases)
//   0  init, sample pass (pass 0 over this slice's share of the sample)  SUM    0  init, dense pass 0, row maxima  SUM+MAX
//   1  pick, pass 1 over the cached sample keys                          SUM    1  pick, dense pass 1              SUM
//   2  pick, pass 2 over the cached sample keys                          SUM    2  pick, dense pass 2              SUM
//   3  pick, window, full pass (below / lists / row maxima), level 0     SUM+MAX  3  pick, status, build
//   4  pick (subtracts the global count below), list level 1             SUM
//   5  pick, list level 2                                                SUM
//   6  pick, status, build of this slice
// SUM: the histograms and below-window counters (uint32 / uint64 counts of at most d_global < 2^32, summed as int32 words:
// exact, the high words are zero); MAX: the row maxima and the list-overflow flags.  Every pick then reads the counts of
// the whole vector, so every rank takes the same decisions and reports the same status; the sample is the whole vector's
// sample (each rank visits its share, pcb_slice_sample), so the windows are the single-GPU windows.
extern "C" int mr_pcb_dist_layout(int64_t d_local, int64_t d_global, int K, int64_t* ws_bytes, int64_t* sum_off,
                                  int64_t* sum_bytes, int64_t* max_off, int64_t* max_bytes) {
    using namespace mr;
    MR_REQUIRE(K >= 1 && K <= MR_MAX_K, "mr_pcb_dist_layout: K=%d outside [1,%d]", K, MR_MAX_K);
    MR_REQUIRE(ws_bytes && sum_off && sum_bytes && max_off && max_bytes, "mr_pcb_dist_layout: null pointer");
    MR_REQUIRE(d_local >= 0 && d_local <= d_global && d_global < ((int64_t)1 << 32),
               "mr_pcb_dist_layout: need 0 <= d_local <= d_global < 2^32");
    const PcbDistWs D = pcb_dist_layout(d_local, d_global, K);
    *ws_bytes = (int64_t)D.total;
    *sum_off = (int64_t)D.L.hist_off;
    *sum_bytes = (int64_t)pcb_counter_bytes(D.L);
    *max_off = (int64_t)D.max_off;
    *max_bytes = (int64_t)D.max_bytes;
    return MR_OK;
}

extern "C" int mr_pcb_dist_plan(int64_t d_global, int flags, int32_t* collectives, int cap) {
    using namespace mr;
    MR_REQUIRE(d_global >= 1 && d_global < ((int64_t)1 << 32), "mr_pcb_dist_plan: d_global=%lld outside [1, 2^32)",
               (long long)d_global);
    MR_REQUIRE(cap >= 0 && (collectives || cap == 0), "mr_pcb_dist_plan: null pointer");
    static const int32_t kFast[7] = {MR_PCB_SUM, MR_PCB_SUM, MR_PCB_SUM, MR_PCB_SUM | MR_PCB_MAX, MR_PCB_SUM, MR_PCB_SUM, 0};
    static const int32_t kDense[4] = {MR_PCB_SUM | MR_PCB_MAX, MR_PCB_SUM, MR_PCB_SUM, 0};
    const bool fast = pcb_fast(d_global, flags);
    const int n = fast ? 7 : 4;
    for (int p = 0; p < n && p < cap; ++p) collectives[p] = fast ? kFast[p] : kDense[p];
    return n;
}

extern "C" int mr_pcb_vectors_dist(const float* base, const float* const* models, int K, int64_t d_local, int64_t j_off,
                                   int64_t d_global, const float* clamp_lo, const float* clamp_hi, int64_t q_index, int flags,
                                   int phase, int32_t* status, float* out, int64_t ldo, void* ws, int64_t ws_bytes,
                                   mr_stream_t stream) {
    using namespace mr;
    MR_REQUIRE(K >= 1 && K <= MR_MAX_K, "mr_pcb_vectors_dist: K=%d outside [1,%d]", K, MR_MAX_K);
    MR_REQUIRE(d_global >= 1 && d_global < ((int64_t)1 << 32), "mr_pcb_vectors_dist: d_global=%lld outside [1, 2^32)",
               (long long)d_global);
    MR_REQUIRE(d_local >= 0 && j_off >= 0 && j_off + d_local <= d_global,
               "mr_pcb_vectors_dist: need 0 <= j_off, 0 <= d_local, j_off + d_local <= d_global");
    MR_REQUIRE(j_off % 32 == 0 || d_local == 0, "mr_pcb_vectors_dist: j_off=%lld is not a multiple of 32", (long long)j_off);
    MR_REQUIRE(d_local % 32 == 0 || j_off + d_local == d_global,
               "mr_pcb_vectors_dist: a slice must end on a multiple of 32 columns or at d_global");
    MR_REQUIRE(q_index >= 0 && q_index < d_global, "mr_pcb_vectors_dist: quantile index %lld outside [0,d_global)",
               (long long)q_index);
    const bool fast = pcb_fast(d_global, flags);
    const int n_phases = fast ? 7 : 4;
    MR_REQUIRE(phase >= 0 && phase < n_phases, "mr_pcb_vectors_dist: phase %d outside [0,%d)", phase, n_phases);
    MR_REQUIRE(clamp_lo && clamp_hi && status && ws, "mr_pcb_vectors_dist: null pointer");
    MR_REQUIRE(d_local == 0 || (base && models && out), "mr_pcb_vectors_dist: null pointer");
    MR_REQUIRE(d_local == 0 || ldo >= d_local, "mr_pcb_vectors_dist: need ldo >= d_local");
    for (int k = 0; d_local > 0 && k < K; ++k) MR_REQUIRE(models[k] != nullptr, "mr_pcb_vectors_dist: models[%d] is NULL", k);
    const PcbDistWs D = pcb_dist_layout(d_local, d_global, K);
    if (ws_bytes < (int64_t)D.total) {
        set_error("mr_pcb_vectors_dist: workspace too small (%lld < %lld bytes)", (long long)ws_bytes, (long long)D.total);
        return MR_ERR_WORKSPACE;
    }
    const PcbWs& L = D.L;
    cudaStream_t st = (cudaStream_t)stream;
    char* w = reinterpret_cast<char*>(ws);
    PcbState* state = reinterpret_cast<PcbState*>(w + L.state_off);
    uint32_t* hist = reinterpret_cast<uint32_t*>(w + L.hist_off);
    unsigned long long* below = reinterpret_cast<unsigned long long*>(w + L.below_off);
    uint32_t* list_cnt = reinterpret_cast<uint32_t*>(w + L.cnt_off);
    uint32_t* list_keys = reinterpret_cast<uint32_t*>(w + L.keys_off);
    uint32_t* skeys = reinterpret_cast<uint32_t*>(w + L.skeys_off);
    int32_t* maxreg = reinterpret_cast<int32_t*>(w + D.max_off);
    const size_t hist_bytes = (size_t)K * kPcbBins * sizeof(uint32_t);
    const int ieee = (flags & MR_PCB_IEEE) ? 1 : 0;
    int64_t s0 = 0, n_s = 0;                                 // this slice's share of the whole vector's sample
    pcb_slice_sample(d_local, j_off, d_global, &s0, &n_s);
    int64_t r_lo = q_index, r_hi = q_index;
    int lo_open = 0, hi_open = 0;
    if (fast) pcb_window_ranks(q_index, d_global, pcb_sample_count(d_global, kPcbStride), &r_lo, &r_hi, &lo_open, &hi_open);
    const bool vec = d_local > 0 && pcb_vec(base, models, K, out, ldo, nullptr);
    MR_DISPATCH_K(K, {
        PtrPack<KK> pk;
        for (int k = 0; k < KK; ++k) pk.p[k] = d_local > 0 ? models[k] : nullptr;
        if (!fast) {
            switch (phase) {
                case 0:
                    cudaMemsetAsync(hist, 0, pcb_counter_bytes(L), st);
                    pcb_init_kernel<<<1, 64, 0, st>>>(state, KK, r_lo, r_hi);
                    pcb_launch_hist<KK>(base, pk, d_local, 1, d_local, false, 0, 0, clamp_lo, clamp_hi, 0, state, hist, nullptr, ieee, st);
                    pcb_export_kernel<<<1, 32, 0, st>>>(state, KK, maxreg);
                    break;
                case 1:
                case 2:
                    if (phase == 1) pcb_import_kernel<<<1, 32, 0, st>>>(state, KK, maxreg);
                    pcb_pick_kernel<<<dim3(KK, 1), 256, 0, st>>>(phase - 1, KK, 0, state, hist);
                    cudaMemsetAsync(hist, 0, hist_bytes, st);
                    pcb_launch_hist<KK>(base, pk, d_local, 1, d_local, false, 0, 0, clamp_lo, clamp_hi, phase, state, hist, nullptr, ieee, st);
                    break;
                default:
                    pcb_pick_kernel<<<dim3(KK, 1), 256, 0, st>>>(2, KK, 0, state, hist);
                    pcb_status_kernel<<<1, 32, 0, st>>>(state, KK, 0, ieee, clamp_lo, clamp_hi, status);
                    pcb_launch_build<KK>(base, pk, d_local, vec, clamp_lo, clamp_hi, state, out, ldo, nullptr, nullptr, ieee, st);
                    break;
            }
        } else {
            switch (phase) {
                case 0:
                    cudaMemsetAsync(hist, 0, pcb_counter_bytes(L), st);
                    pcb_init_kernel<<<1, 64, 0, st>>>(state, KK, r_lo, r_hi);
                    pcb_launch_hist<KK>(base, pk, d_local, kPcbStride, n_s, true, s0, j_off, clamp_lo, clamp_hi, 0, state, hist, skeys,
                                        ieee, st);
                    break;
                case 1:
                case 2:
                    pcb_pick_kernel<<<dim3(KK, kPcbSlots), 256, 0, st>>>(phase - 1, KK, phase == 1 ? 1 : 0, state, hist);
                    cudaMemsetAsync(hist, 0, kPcbSlots * hist_bytes, st);
                    pcb_launch_keys_hist(skeys, n_s, KK, phase, state, hist, st);
                    break;
                case 3:
                    pcb_pick_kernel<<<dim3(KK, kPcbSlots), 256, 0, st>>>(2, KK, 0, state, hist);
                    cudaMemsetAsync(hist, 0, kPcbSlots * hist_bytes, st);
                    pcb_window_init_kernel<<<1, 32, 0, st>>>(state, KK, q_index, lo_open, hi_open);
                    pcb_launch_window<KK>(base, pk, d_local, vec, clamp_lo, clamp_hi, state, below, list_keys, list_cnt,
                                          pcb_window_lists<KK>(d_local, vec), L, ieee, st);
                    pcb_export_kernel<<<1, 32, 0, st>>>(state, KK, maxreg);
                    pcb_launch_list_hist(KK, list_keys, list_cnt, pcb_window_lists<KK>(d_local, vec), L, state, hist, st);
                    break;
                case 4:
                case 5:
                    if (phase == 4) pcb_import_kernel<<<1, 32, 0, st>>>(state, KK, maxreg);
                    pcb_window_pick_kernel<<<KK, 256, 0, st>>>(phase == 4, state, hist, below);
                    pcb_launch_list_hist(KK, list_keys, list_cnt, pcb_window_lists<KK>(d_local, vec), L, state, hist, st);
                    break;
                default:
                    pcb_window_pick_kernel<<<KK, 256, 0, st>>>(0, state, hist, below);
                    pcb_status_kernel<<<1, 32, 0, st>>>(state, KK, 1, ieee, clamp_lo, clamp_hi, status);
                    pcb_launch_build<KK>(base, pk, d_local, vec, clamp_lo, clamp_hi, state, out, ldo, nullptr, nullptr, ieee, st);
                    break;
            }
        }
    });
    MR_CUDA_LAUNCH_CHECK("mr_pcb_vectors_dist");
    return MR_OK;
}
