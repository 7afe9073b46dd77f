// eval.cu -- evaluator kernels outside the tensor-core contraction (SURVEY.md section 8(a): B2-B4):
// per-row top-K of a materialised score matrix, merge of per-shard top-K lists, rank of the label,
// the hi/lo TF32 operand split, and a plain fp32 scoring kernel (CUDA cores; the "fp32 mode").
//
// reference: rec_retrieval/evaluator/evaluator.py:31-49 (torch.topk(scores, max_k, dim=1).indices),
//            rec_retrieval/evaluator/metrics.py:35-88 (`true in pred`, `pred.index(true)`),
//            rec_retrieval/module/recommender/module.py:137 (scores = user @ item.T)
//
// Order of a top-K list: score descending, then item id ascending (canonical rule, SURVEY.md 0.1-D3);
// -0.0 == +0.0 and NaN sorts first, like torch.topk.  Everything is compare-only: results are bit-exact.
#include "common.cuh"
#include "topk_common.cuh"

namespace mr {

// ---- B2: per-row top-K of a (Q, N) score matrix -------------------------------------------------------------
// One CTA per row.  Scores stream through a threshold filter into a shared-memory candidate buffer; when the
// buffer cannot take another chunk it is sorted (bitonic, descending) and cut back to K, which also raises the
// threshold.  After the first cut only ~K*ln(N/K) elements ever pass.
constexpr int kTopkThreads = 256;
constexpr int kTopkCap = 2048;               // candidate buffer (keys), power of two
constexpr int kTopkChunk = kTopkThreads * 4; // elements examined between two buffer checks

// EXCL: items of row q's exclusion list (CSR: excl_ids[excl_off[q] .. excl_off[q + 1]), ascending global ids) never
// enter the buffer.  A thread's columns are strided, so each key that passes the threshold is looked up in the row's
// list by binary search.
template <bool EXCL>
__global__ void __launch_bounds__(kTopkThreads)
topk_rows_kernel(const float* __restrict__ scores, int64_t Q, int64_t N, int64_t ld, int K, int32_t id_base,
                 float* __restrict__ out_val, int32_t* __restrict__ out_id, const int64_t* __restrict__ excl_off,
                 const int32_t* __restrict__ excl_ids) {
    __shared__ u64 s_keys[kTopkCap];
    __shared__ int s_cnt;
    __shared__ u64 s_thr;
    for (int64_t q = blockIdx.x; q < Q; q += gridDim.x) {
        const float* row = scores + q * ld;
        const bool vec = ((reinterpret_cast<uintptr_t>(row) & 15) == 0);
        const int64_t ex_beg = EXCL ? excl_off[q] : 0, ex_end = EXCL ? excl_off[q + 1] : 0;
        if (threadIdx.x == 0) { s_cnt = 0; s_thr = 0; }
        __syncthreads();
        for (int64_t c0 = 0; c0 < N; c0 += kTopkChunk) {
            const u64 thr = s_thr;
            int over = 0;  // did one of my appends land beyond the refill limit?
            const int64_t c = c0 + (int64_t)threadIdx.x * 4;
            float v[4];
            int nv = 0;
            if (c + 3 < N && vec) {
                const float4 f = ldg_stream4(row + c);
                v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
                nv = 4;
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (c + i < N) { v[i] = row[c + i]; nv = i + 1; }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if (i < nv) {
                    const u64 key = topk_key(v[i], (uint32_t)(id_base + (int32_t)(c + i)));
                    if (EXCL && key > thr) {
                        const int32_t id = id_base + (int32_t)(c + i);
                        int64_t a = ex_beg, b = ex_end;
                        while (a < b) {
                            const int64_t m = (a + b) >> 1;
                            if (excl_ids[m] < id) a = m + 1; else b = m;
                        }
                        if (a < ex_end && excl_ids[a] == id) continue;
                    }
                    if (key > thr) {
                        const int pos = atomicAdd(&s_cnt, 1);
                        s_keys[pos] = key;
                        over |= (pos >= kTopkCap - kTopkChunk);
                    }
                }
            }
            // barrier + uniform decision (s_cnt itself may already be moving again when a slow thread looks at it)
            if (__syncthreads_or(over)) {
                const int n = s_cnt;
                for (int i = n + threadIdx.x; i < kTopkCap; i += blockDim.x) s_keys[i] = 0;
                __syncthreads();
                block_bitonic_sort_desc(s_keys, kTopkCap);
                if (threadIdx.x == 0) {
                    s_cnt = n < K ? n : K;
                    if (n >= K) s_thr = s_keys[K - 1];
                }
                __syncthreads();
            }
        }
        const int n = s_cnt;
        for (int i = n + threadIdx.x; i < kTopkCap; i += blockDim.x) s_keys[i] = 0;
        __syncthreads();
        block_bitonic_sort_desc(s_keys, kTopkCap);
        for (int i = threadIdx.x; i < K; i += blockDim.x) {
            const u64 key = s_keys[i];
            if (i < n && key != 0) {
                const int32_t id = (int32_t)key_id(key);
                out_id[q * K + i] = id;
                out_val[q * K + i] = row[id - id_base];  // the original bits (keeps -0.0 / NaN payloads)
            } else {
                out_id[q * K + i] = -1;
                out_val[q * K + i] = -INFINITY;
            }
        }
        __syncthreads();
    }
}

// ---- merge L top-K lists per row (the multi-GPU / multi-split exchange step) -----------------------------------
// vals / ids: L lists of (Q, K_in), list l starting `list_stride` elements after list l - 1; entries with id < 0 are
// empty.  Output (Q, K_out) sorted by (score desc, id asc).
// Generic form (any L * K_in <= 8192, lists sorted or not): one CTA per row, bitonic sort of all candidates.
__global__ void __launch_bounds__(256)
topk_merge_kernel(const float* __restrict__ vals, const int32_t* __restrict__ ids, int64_t list_stride, int L, int64_t Q,
                  int K_in, int K_out, int NP, float* __restrict__ out_val, int32_t* __restrict__ out_id) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    u64* s_keys = reinterpret_cast<u64*>(smem_raw);
    const int total = L * K_in;
    for (int64_t q = blockIdx.x; q < Q; q += gridDim.x) {
        for (int i = threadIdx.x; i < NP; i += blockDim.x) {
            u64 key = 0;
            if (i < total) {
                const int l = i / K_in, e = i - l * K_in;
                const int64_t src = (int64_t)l * list_stride + q * K_in + e;
                const int32_t id = ids[src];
                if (id >= 0) key = topk_key(vals[src], (uint32_t)id);
            }
            s_keys[i] = key;
        }
        __syncthreads();
        block_bitonic_sort_desc(s_keys, NP);
        for (int i = threadIdx.x; i < K_out; i += blockDim.x) {
            const u64 key = (i < NP) ? s_keys[i] : 0;
            out_id[q * K_out + i] = key ? (int32_t)key_id(key) : -1;
            out_val[q * K_out + i] = key ? key_score(key) : -INFINITY;
        }
        __syncthreads();
    }
}

// Fast form for what the scoring kernel and the exchange step produce: L <= 32 SORTED lists, L * K_in <= 1024.  One WARP
// per row: the row's lists are staged in shared memory (coalesced), lane l keeps the head of list l, and K_out times the
// warp takes the maximum head (five 64-bit shuffles) and the winning lane advances -- a plain L-way merge, ~12
// instructions per output, no barriers across warps.  (A rank-counting merge -- one binary search per key and list -- was
// measured no faster than the sort: 2.85 ms for 8 lists of 100 over 65,536 rows; this form takes a fraction of that.)
// A row whose lists are not sorted (the C ABI allows it) is sorted by its warp in shared memory instead.
constexpr int kMergeWarpKeys = 1024;   // keys per row in the warp form (8 KB of shared memory per warp)
__global__ void __launch_bounds__(256)
topk_merge_warp_kernel(const float* __restrict__ vals, const int32_t* __restrict__ ids, int64_t list_stride, int L, int64_t Q,
                       int K_in, int K_out, int NP, float* __restrict__ out_val, int32_t* __restrict__ out_id) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    u64* s = reinterpret_cast<u64*>(smem_raw) + (size_t)warp * NP;
    const int total = L * K_in;
    for (int64_t q = (int64_t)blockIdx.x * wpb + warp; q < Q; q += (int64_t)gridDim.x * wpb) {
        for (int i = lane; i < NP; i += 32) {
            u64 key = 0;
            if (i < total) {
                const int l = i / K_in, e = i - l * K_in;
                const int64_t src = (int64_t)l * list_stride + q * K_in + e;
                const int32_t id = ids[src];
                if (id >= 0) key = topk_key(vals[src], (uint32_t)id);
            }
            s[i] = key;
        }
        __syncwarp();
        int unsorted = 0;
        for (int i = lane; i < total; i += 32) {
            const int e = i % K_in;
            if (e + 1 < K_in && s[i] < s[i + 1]) unsorted = 1;     // (empty slots are 0 and sit at the end of a sorted list)
        }
        if (__any_sync(0xffffffffu, unsorted)) {
            // rare: sort the row's NP keys with this warp (bitonic, descending), then read the first K_out
            for (int size = 2; size <= NP; size <<= 1) {
                for (int stride = size >> 1; stride > 0; stride >>= 1) {
                    for (int i = lane; i < (NP >> 1); i += 32) {
                        const int a = 2 * i - (i & (stride - 1));
                        const int b = a + stride;
                        const bool desc = ((a & size) == 0);
                        const u64 x = s[a], y = s[b];
                        if ((x < y) == desc) { s[a] = y; s[b] = x; }
                    }
                    __syncwarp();
                }
            }
            for (int i = lane; i < K_out; i += 32) {
                const u64 key = (i < NP) ? s[i] : 0;
                out_id[q * K_out + i] = key ? (int32_t)key_id(key) : -1;
                out_val[q * K_out + i] = key ? key_score(key) : -INFINITY;
            }
        } else {
            int pos = 0;                                              // lane l < L walks list l
            u64 cur = (lane < L) ? s[lane * K_in] : 0;
            for (int r0 = 0; r0 < K_out; r0 += 32) {
                u64 mine = 0;                                         // output r0 + lane, written coalesced after 32 steps
                const int nr = (K_out - r0) < 32 ? (K_out - r0) : 32;
                for (int r = 0; r < nr; ++r) {
                    u64 best = cur;
#pragma unroll
                    for (int off = 16; off > 0; off >>= 1) {
                        const u64 o = __shfl_xor_sync(0xffffffffu, best, off);
                        best = o > best ? o : best;
                    }
                    if (lane == r) mine = best;
                    // the winner advances; equal keys in two lists (the same id twice: legal input) -> the lowest lane
                    const unsigned win = __ballot_sync(0xffffffffu, best != 0 && cur == best);
                    if (win && lane == __ffs(win) - 1) {
                        ++pos;
                        cur = (pos < K_in) ? s[lane * K_in + pos] : 0;
                    }
                }
                if (lane < nr) {
                    out_id[q * K_out + r0 + lane] = mine ? (int32_t)key_id(mine) : -1;
                    out_val[q * K_out + r0 + lane] = mine ? key_score(mine) : -INFINITY;
                }
            }
        }
        __syncwarp();
    }
}

// ---- B3/B4 helper: position of the label inside each row's list, -1 when absent -----------------------------
__global__ void label_rank_kernel(const int32_t* __restrict__ ids, int64_t Q, int K, const int64_t* __restrict__ labels,
                                  int32_t* __restrict__ rank) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= Q) return;
    const int64_t lab = labels[q];
    int32_t r = -1;
    for (int i = 0; i < K; ++i) {
        if ((int64_t)ids[q * K + i] == lab) { r = i; break; }
    }
    rank[q] = r;
}

// ---- rank of the label against the whole row (no list, no K) ----------------------------------------------------
// count[q] = number of columns whose (score, id) key sorts before the label's, minus the row's excluded ids that do:
// the exclusion list is walked once, after the count, skipping repeated ids.  -1 when the label is not a column.
constexpr int kRankThreads = 256;
__global__ void __launch_bounds__(kRankThreads)
rank_rows_kernel(const float* __restrict__ scores, int64_t Q, int64_t N, int64_t ld, int32_t id_base,
                 const int64_t* __restrict__ labels, const int64_t* __restrict__ excl_off,
                 const int32_t* __restrict__ excl_ids, int32_t* __restrict__ count) {
    __shared__ int s_warp[kRankThreads / 32];
    for (int64_t q = blockIdx.x; q < Q; q += gridDim.x) {
        const float* row = scores + q * ld;
        const int64_t col = labels[q] - id_base;
        if (col < 0 || col >= N) {          // block-uniform
            if (threadIdx.x == 0) count[q] = -1;
            continue;
        }
        const u64 L = topk_key(row[col], (uint32_t)(id_base + (int32_t)col));
        const bool vec = ((reinterpret_cast<uintptr_t>(row) & 15) == 0);
        int c = 0;
        for (int64_t c0 = (int64_t)threadIdx.x * 4; c0 < N; c0 += kRankThreads * 4) {
            if (c0 + 3 < N && vec) {
                const float4 f = ldg_stream4(row + c0);
                const uint32_t id = (uint32_t)(id_base + (int32_t)c0);
                c += (topk_key(f.x, id) > L) + (topk_key(f.y, id + 1) > L) + (topk_key(f.z, id + 2) > L) +
                     (topk_key(f.w, id + 3) > L);
            } else {
                for (int64_t i = c0; i < c0 + 4 && i < N; ++i) c += topk_key(row[i], (uint32_t)(id_base + (int32_t)i)) > L;
            }
        }
        if (excl_off) {
            const int64_t beg = excl_off[q], end = excl_off[q + 1];
            for (int64_t i = beg + threadIdx.x; i < end; i += kRankThreads) {
                const int64_t x = (int64_t)excl_ids[i] - id_base;
                if (x >= 0 && x < N && (i == beg || excl_ids[i - 1] != excl_ids[i]))
                    c -= topk_key(row[x], (uint32_t)excl_ids[i]) > L;
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) c += __shfl_xor_sync(0xffffffffu, c, off);
        if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = c;
        __syncthreads();
        if (threadIdx.x == 0) {
            int t = 0;
            for (int w = 0; w < kRankThreads / 32; ++w) t += s_warp[w];
            count[q] = t;
        }
        __syncthreads();
    }
}

// ---- hi/lo split for the 3xTF32 contraction -----------------------------------------------------------------------
// hi = rna_tf32(x), lo = rna_tf32(x - hi) (common.cuh): x = hi + lo up to 2^-22 |x|, both exactly representable in TF32.
__global__ void split_tf32_kernel(const float* __restrict__ x, int64_t n, float* __restrict__ hi, float* __restrict__ lo) {
    const int64_t gsz = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gsz) {
        const float v = x[i];
        const float h = rna_tf32(v);
        hi[i] = h;
        lo[i] = rna_tf32(__fsub_rn(v, h));
    }
}

// fp32 -> bf16, round to nearest even (what `tensor.to(torch.bfloat16)` / autocast do); NaN stays NaN
__global__ void to_bf16_kernel(const float* __restrict__ x, int64_t n, uint16_t* __restrict__ out) {
    const int64_t gsz = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gsz) {
        const uint32_t u = __float_as_uint(x[i]);
        uint32_t r;
        if ((u & 0x7F800000u) == 0x7F800000u) r = (u & 0x007FFFFFu) ? (u | 0x00400000u) : u;   // NaN (quieted) / inf
        else r = u + 0x7FFFu + ((u >> 16) & 1u);
        out[i] = (uint16_t)(r >> 16);
    }
}

// ---- B1 in plain fp32 on CUDA cores ("fp32 mode"; also the on-device cross-check of the tensor-core path) ------------
// out[q, n] = sum_e U[q,e] * I[n,e], one fp32 FMA chain per score, sequential in e.
constexpr int kSfTile = 64, kSfBk = 16;
__global__ void __launch_bounds__(256)
scores_fp32_kernel(const float* __restrict__ U, int64_t Q, const float* __restrict__ I, int64_t N, int E,
                   float* __restrict__ out, int64_t ldo) {
    __shared__ float s_u[kSfBk][kSfTile + 1];
    __shared__ float s_i[kSfBk][kSfTile + 1];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int64_t q0 = (int64_t)blockIdx.y * kSfTile, n0 = (int64_t)blockIdx.x * kSfTile;
    float acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = 0.0f;
    for (int e0 = 0; e0 < E; e0 += kSfBk) {
        for (int i = threadIdx.x; i < kSfTile * kSfBk; i += 256) {
            const int r = i / kSfBk, e = i % kSfBk;
            const bool eok = e0 + e < E;
            s_u[e][r] = (eok && q0 + r < Q) ? U[(q0 + r) * E + e0 + e] : 0.0f;
            s_i[e][r] = (eok && n0 + r < N) ? I[(n0 + r) * E + e0 + e] : 0.0f;
        }
        __syncthreads();
#pragma unroll
        for (int e = 0; e < kSfBk; ++e) {
            float a[4], b[4];
#pragma unroll
            for (int x = 0; x < 4; ++x) { a[x] = s_u[e][ty * 4 + x]; b[x] = s_i[e][tx * 4 + x]; }
#pragma unroll
            for (int x = 0; x < 4; ++x)
#pragma unroll
                for (int y = 0; y < 4; ++y) acc[x][y] = fmaf(a[x], b[y], acc[x][y]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) {
            const int64_t q = q0 + ty * 4 + x, n = n0 + tx * 4 + y;
            if (q < Q && n < N) out[q * ldo + n] = acc[x][y];
        }
}

}  // namespace mr

// mr_topk_rows (excl_off == NULL) and mr_topk_rows_exclude
static int topk_rows_launch(const float* scores, int64_t Q, int64_t N, int64_t ld, int K, int32_t id_base, float* out_val,
                            int32_t* out_id, const int64_t* excl_off, const int32_t* excl_ids, mr_stream_t stream) {
    using namespace mr;
    MR_REQUIRE(Q >= 0 && N >= 0 && ld >= N, "mr_topk_rows: need Q >= 0 and ld >= N >= 0");
    MR_REQUIRE(K >= 1 && K <= MR_MAX_TOPK, "mr_topk_rows: K=%d outside [1,%d]", K, MR_MAX_TOPK);
    MR_REQUIRE((int64_t)K <= N || Q == 0, "mr_topk_rows: K=%d exceeds the number of items %lld", K, (long long)N);
    if (Q == 0) return MR_OK;
    MR_REQUIRE(scores && out_val && out_id, "mr_topk_rows: null pointer");
    const int64_t cap = (int64_t)sm_count() * 8;
    const unsigned blocks = (unsigned)(Q < cap ? Q : cap);
    // rows whose start is not 16-byte aligned (ld % 4 != 0) simply take the scalar loads
    if (excl_off)
        topk_rows_kernel<true><<<blocks, kTopkThreads, 0, (cudaStream_t)stream>>>(scores, Q, N, ld, K, id_base, out_val,
                                                                                  out_id, excl_off, excl_ids);
    else
        topk_rows_kernel<false><<<blocks, kTopkThreads, 0, (cudaStream_t)stream>>>(scores, Q, N, ld, K, id_base, out_val,
                                                                                   out_id, nullptr, nullptr);
    MR_CUDA_LAUNCH_CHECK("mr_topk_rows");
    return MR_OK;
}

extern "C" int mr_topk_rows(const float* scores, int64_t Q, int64_t N, int64_t ld, int K, int32_t id_base,
                            float* out_val, int32_t* out_id, mr_stream_t stream) {
    return topk_rows_launch(scores, Q, N, ld, K, id_base, out_val, out_id, nullptr, nullptr, stream);
}

extern "C" int mr_topk_rows_exclude(const float* scores, int64_t Q, int64_t N, int64_t ld, int K, int32_t id_base,
                                    float* out_val, int32_t* out_id, const int64_t* excl_off, const int32_t* excl_ids,
                                    mr_stream_t stream) {
    MR_REQUIRE(excl_off && excl_ids, "mr_topk_rows_exclude: null pointer (excl_off / excl_ids)");
    return topk_rows_launch(scores, Q, N, ld, K, id_base, out_val, out_id, excl_off, excl_ids, stream);
}

static int topk_merge_launch(const float* vals, const int32_t* ids, int64_t list_stride, int L, int64_t Q, int K_in,
                             int K_out, float* out_val, int32_t* out_id, mr_stream_t stream, const char* who) {
    using namespace mr;
    MR_REQUIRE(L >= 1 && Q >= 0 && K_in >= 1 && K_out >= 1, "%s: need L, K_in, K_out >= 1 and Q >= 0", who);
    MR_REQUIRE(K_out <= MR_MAX_TOPK, "%s: K_out=%d exceeds %d", who, K_out, MR_MAX_TOPK);
    int NP = 1;
    while (NP < L * K_in) NP <<= 1;
    MR_REQUIRE(NP <= 8192, "%s: L*K_in=%d candidates per row exceed 8192", who, L * K_in);
    if (Q == 0) return MR_OK;
    MR_REQUIRE(vals && ids && out_val && out_id, "%s: null pointer", who);
    if (L <= 32 && NP <= kMergeWarpKeys) {
        // one warp per row (sorted lists: L-way merge; otherwise the warp sorts): 8 rows per CTA
        const size_t smem = (size_t)NP * 8 * 8;
        if (smem > 48 * 1024) cudaFuncSetAttribute(topk_merge_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        const int64_t rows_blocks = (Q + 7) / 8;
        const int64_t cap = (int64_t)sm_count() * (smem > 32 * 1024 ? 3 : 8);
        const unsigned blocks = (unsigned)(rows_blocks < cap ? rows_blocks : cap);
        topk_merge_warp_kernel<<<blocks, 256, smem, (cudaStream_t)stream>>>(vals, ids, list_stride, L, Q, K_in, K_out, NP, out_val, out_id);
        MR_CUDA_LAUNCH_CHECK(who);
        return MR_OK;
    }
    const size_t smem = (size_t)NP * 8;
    if (smem > 48 * 1024) cudaFuncSetAttribute(topk_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const int64_t cap = (int64_t)sm_count() * 8;
    const unsigned blocks = (unsigned)(Q < cap ? Q : cap);
    topk_merge_kernel<<<blocks, 256, smem, (cudaStream_t)stream>>>(vals, ids, list_stride, L, Q, K_in, K_out, NP, out_val, out_id);
    MR_CUDA_LAUNCH_CHECK(who);
    return MR_OK;
}

extern "C" int mr_topk_merge(const float* vals, const int32_t* ids, int L, int64_t Q, int K_in, int K_out,
                             float* out_val, int32_t* out_id, mr_stream_t stream) {
    return topk_merge_launch(vals, ids, Q * (int64_t)K_in, L, Q, K_in, K_out, out_val, out_id, stream, "mr_topk_merge");
}

// Same merge over the exchange buffer of the sharded evaluator: L blocks of (2, Q, K_in) 32-bit words, block l = one
// rank's list -- plane 0 the fp32 scores, plane 1 the int32 global ids -- exactly what ONE all-gather of every rank's
// (2, Q, K_in) buffer produces.
extern "C" int mr_topk_merge_packed(const void* packed, int L, int64_t Q, int K_in, int K_out, float* out_val,
                                    int32_t* out_id, mr_stream_t stream) {
    const float* vals = reinterpret_cast<const float*>(packed);
    const int32_t* ids = packed ? reinterpret_cast<const int32_t*>(packed) + Q * (int64_t)K_in : nullptr;
    return topk_merge_launch(vals, ids, 2 * Q * (int64_t)K_in, L, Q, K_in, K_out, out_val, out_id, stream,
                             "mr_topk_merge_packed");
}

extern "C" int mr_label_rank(const int32_t* ids, int64_t Q, int K, const int64_t* labels, int32_t* rank,
                             mr_stream_t stream) {
    using namespace mr;
    MR_REQUIRE(Q >= 0 && K >= 1, "mr_label_rank: need Q >= 0, K >= 1");
    if (Q == 0) return MR_OK;
    MR_REQUIRE(ids && labels && rank, "mr_label_rank: null pointer");
    label_rank_kernel<<<(unsigned)((Q + 255) / 256), 256, 0, (cudaStream_t)stream>>>(ids, Q, K, labels, rank);
    MR_CUDA_LAUNCH_CHECK("mr_label_rank");
    return MR_OK;
}

extern "C" int mr_rank_rows(const float* scores, int64_t Q, int64_t N, int64_t ld, int32_t id_base, const int64_t* labels,
                            const int64_t* excl_off, const int32_t* excl_ids, int32_t* count, mr_stream_t stream) {
    using namespace mr;
    MR_REQUIRE((excl_off == nullptr) == (excl_ids == nullptr),
               "mr_rank_rows: excl_off and excl_ids must both be NULL or both be set");
    MR_REQUIRE(Q >= 0 && N >= 0 && ld >= N, "mr_rank_rows: need Q >= 0 and ld >= N >= 0");
    MR_REQUIRE((int64_t)id_base + N < (1ll << 31), "mr_rank_rows: id_base + N must fit 31 bits");
    if (Q == 0) return MR_OK;
    MR_REQUIRE(scores && labels && count, "mr_rank_rows: null pointer");
    const int64_t cap = (int64_t)sm_count() * 8;
    const unsigned blocks = (unsigned)(Q < cap ? Q : cap);
    rank_rows_kernel<<<blocks, kRankThreads, 0, (cudaStream_t)stream>>>(scores, Q, N, ld, id_base, labels, excl_off,
                                                                        excl_ids, count);
    MR_CUDA_LAUNCH_CHECK("mr_rank_rows");
    return MR_OK;
}

extern "C" int mr_split_tf32(const float* x, int64_t n, float* hi, float* lo, mr_stream_t stream) {
    using namespace mr;
    MR_REQUIRE(n >= 0, "mr_split_tf32: n < 0");
    if (n == 0) return MR_OK;
    MR_REQUIRE(x && hi && lo, "mr_split_tf32: null pointer");
    int64_t blocks = (n + 255) / 256;
    const int64_t cap = (int64_t)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    split_tf32_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, n, hi, lo);
    MR_CUDA_LAUNCH_CHECK("mr_split_tf32");
    return MR_OK;
}

extern "C" int mr_to_bf16(const float* x, int64_t n, uint16_t* out, mr_stream_t stream) {
    using namespace mr;
    MR_REQUIRE(n >= 0, "mr_to_bf16: n < 0");
    if (n == 0) return MR_OK;
    MR_REQUIRE(x && out, "mr_to_bf16: null pointer");
    int64_t blocks = (n + 255) / 256;
    const int64_t cap = (int64_t)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    to_bf16_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, n, out);
    MR_CUDA_LAUNCH_CHECK("mr_to_bf16");
    return MR_OK;
}

extern "C" int mr_scores_fp32(const float* U, int64_t Q, const float* I, int64_t N, int E, float* out, int64_t ldo,
                              mr_stream_t stream) {
    using namespace mr;
    MR_REQUIRE(Q >= 0 && N >= 0 && E >= 1 && ldo >= N, "mr_scores_fp32: need Q, N >= 0, E >= 1, ldo >= N");
    if (Q == 0 || N == 0) return MR_OK;
    MR_REQUIRE(U && I && out, "mr_scores_fp32: null pointer");
    MR_REQUIRE((Q + kSfTile - 1) / kSfTile <= 65535, "mr_scores_fp32: Q too large for this kernel (use mr_score_topk)");
    dim3 grid((unsigned)((N + kSfTile - 1) / kSfTile), (unsigned)((Q + kSfTile - 1) / kSfTile));
    scores_fp32_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(U, Q, I, N, E, out, ldo);
    MR_CUDA_LAUNCH_CHECK("mr_scores_fp32");
    return MR_OK;
}
