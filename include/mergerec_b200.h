/*
 * mergerec_b200.h -- C ABI of libmergerec_b200.so: the B200 (sm_100a) replacement for MergeRec's
 * two data-parallel hot paths (merger, evaluator).  Plain pointers and sizes only; no torch types.
 *
 * Conventions (SURVEY.md section 8(b)):
 *   - every pointer marked "dev" is a CUDA device pointer owned by the caller (PyTorch allocates all
 *     inputs, outputs and workspaces; the library owns no device memory);
 *   - every pointer marked "host" is ordinary host memory read during the call;
 *   - all entry points are stream-ordered and asynchronous: they enqueue work on `stream` and return;
 *     nothing synchronises the host;
 *   - functions never throw: the return value is 0 on success, <0 for an argument error
 *     (mr_status), >0 for a cudaError_t.  mr_last_error() gives a thread-local message.
 *   - "flat" vectors are the reference's flattened state_dicts: fp32, length d, tensors concatenated
 *     in dict order (reference: rec_retrieval/merger/utils/model_operations.py:47-63).
 *
 * Citations "ref:" are file:line under the reference checkout (DIALLab-SKKU/MergeRec).
 */
#ifndef MERGEREC_B200_H_
#define MERGEREC_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* mr_stream_t; /* == cudaStream_t */

enum mr_status {
    MR_OK = 0,
    MR_ERR_INVALID_ARG = -1,
    MR_ERR_UNSUPPORTED = -2,
    MR_ERR_WORKSPACE = -3,
};

#define MR_MAX_K 16 /* bit-exact torch.sum(dim=0) order is only defined for K <= 16 (SURVEY.md 7.3-1) */

int mr_version(void);
const char* mr_last_error(void);

/* ------------------------------------------------------------------------------------------------
 * Merger: elementwise merges over flat vectors (HBM-bound streaming kernels).
 * ---------------------------------------------------------------------------------------------- */

/* T[k, j] = models[k][j] - base[j]                       ref: merger/algorithms/task_vector.py:8-10
 * models: host array of K dev pointers (d floats each). T: dev, K rows with leading dimension ldT. */
int mr_task_vectors(const float* base, const float* const* models, int K, int64_t d, float* T,
                    int64_t ldT, mr_stream_t stream);

enum mr_merge_order {
    /* acc = base; acc = acc + fl(w_k * u_k)  k = 0..K-1    ref: merger/algorithms/task_vector.py:30-32 */
    MR_ORDER_BASE_FIRST = 0,
    /* out = base + sum_dim0_k fl(w_k * u_k) in torch.sum(dim=0) order (sequential in k; 4-way
     * interleaved on the trailing n mod 32 columns of each block when K >= 5)
     *                                                       ref: weight_learning/module/task_wise.py:43-47,
     *                                                            weight_learning/module/layer_wise.py:76-82 */
    MR_ORDER_SUM_FIRST = 1,
    /* acc = 0; acc = acc + fl(w_k * src_k); base unused      ref: merger/algorithms/linear.py:23-25 */
    MR_ORDER_LINEAR = 2,
};

/* The lambda-weighted merge (A1, A3, A4, A10 of SURVEY.md section 8(a)).
 *   src           host array of K dev pointers: fine-tuned flat models (src_is_model = 1, u_k = src_k - base
 *                 computed on the fly) or task-vector rows (src_is_model = 0, u_k = src_k).
 *   w             dev, (G, K) row-major fp32 lambdas; row g applies to blocks with seg_group == g.
 *   seg_end       dev, P ascending exclusive block ends (seg_end[P-1] == d), or NULL when P == 1
 *                 (one block [0, d), group 0; a one-entry table with a seg_group is honoured too).  Blocks are the
 *                 reference's sum(dim=0) operands: the whole vector for task-wise, one state_dict tensor each for
 *                 layer-wise.
 *   seg_group     dev, P group ids in [0, G), or NULL when P == 1.
 *   out           dev, d floats.  May alias base. */
int mr_merge_axpy(const float* base, const float* const* src, int K, int64_t d, const float* w, int G,
                  const int64_t* seg_end, const int32_t* seg_group, int P, int order, int src_is_model,
                  float* out, mr_stream_t stream);

/* The lambda-gradient reduction of collaborative merging (A5):
 *     out[g, k] = sum_{p : seg_group[p] == g} sum_{j < seg_len[p]} grad_p[j] * T[k, seg_off[p] + j]
 * Replaces the autograd backward of the reference's merge + P parameter views
 *                        ref: weight_learning/module/task_wise.py:43-47, layer_wise.py:76-82,
 *                             weight_learning/utils.py:11-15,43-51
 *   grad_ptrs   dev array of P dev pointers: the gradient of each state_dict tensor, read in place
 *               (NULL = no gradient = zeros).  Pointing all of them into one flat (d) gradient is fine.
 *   seg_off     dev, P flat offsets of the tensors;  seg_len: dev, P element counts;
 *   seg_group   dev, P group ids in [0, G) or NULL when G == 1.
 *   T           dev, K rows of d floats with leading dimension ldT (task vectors / TIES vectors).
 *   out         dev, (G, K) fp32.  Deterministic (fixed two-stage fp64 reduction tree, no atomics).
 *   ws          dev scratch of at least mr_lambda_grad_workspace_bytes(d, P, K) bytes. */
int64_t mr_lambda_grad_workspace_bytes(int64_t d, int P, int K);
int mr_lambda_grad(const float* const* grad_ptrs, const int64_t* seg_off, const int64_t* seg_len,
                   const int32_t* seg_group, int P, int64_t d, const float* T, int64_t ldT, int K, int G, float* out,
                   void* ws, int64_t ws_bytes, mr_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Merger: TIES (A6-A9).                                          ref: merger/algorithms/ties.py
 * Elements of model k are ordered by the 64-bit key (bits(|u_kj|) << 32) | (0xFFFFFFFF - j), with
 * u_kj = models[k][j] - base[j] (times w[k] when w != NULL, ties.py:20-21): larger magnitude first, lower
 * flat index first among equal magnitudes.  Model k keeps element j iff key >= cut[k], where cut[k] is the
 * k_cnt-th largest key, k_cnt = int(density * d) computed by the caller in double arithmetic (ties.py:14-15).
 * The trim is global over the flat vector like the reference.  d must be < 2^32.
 * ---------------------------------------------------------------------------------------------- */
int64_t mr_ties_workspace_bytes(int64_t d, int K);

enum mr_ties_status {
    MR_TIES_SEARCHING = 0, /* kernels still queued (never observed after a stream sync) */
    MR_TIES_DONE = 1,
    /* < 0: the sampled bracket missed or overflowed (possible on adversarial inputs, e.g. millions of equal
     * magnitudes); call mr_ties_select_exact */
};

/* Fast path, stream-ordered: cut (dev, K x uint64) and status (dev, K x int32) are written by the queued
 * kernels.  One pass over base + K models ((K+1)*d*4 bytes) plus a ~0.5 M-element sample per model. */
int mr_ties_select(const float* base, const float* const* models, int K, int64_t d, const float* w, int64_t k_cnt,
                   uint64_t* cut, int32_t* status, void* ws, int64_t ws_bytes, mr_stream_t stream);
/* Exact path for any input; SYNCHRONOUS (reads bracket state back between passes; <= 8 passes). */
int mr_ties_select_exact(const float* base, const float* const* models, int K, int64_t d, const float* w,
                         int64_t k_cnt, uint64_t* cut, int32_t* status, void* ws, int64_t ws_bytes,
                         mr_stream_t stream);

enum mr_ties_mode {
    /* out = That (K rows, leading dimension ldo): trimmed updates that agree with the elected sign, divided by
     * their per-column count (get_ties_vectors, ties.py:55-72).  w unused. */
    MR_TIES_VECTORS = 0,
    /* out = base + sum_dim0_k trim_k(w[k] * (m_k - base))   (merge_ties, ties.py:75-83).  w: dev (K); cut must
     * come from a select run with the same w. */
    MR_TIES_TRIMSUM = 1,
    /* out = base + sum_dim0_k w[g,k] * That[k] without materialising That: get_ties_vectors followed by the
     * lambda merge (A3/A4) in one pass.  w: dev (G, K); seg_end / seg_group / P as in mr_merge_axpy. */
    MR_TIES_FUSED_MERGE = 2,
    /* out = Localize-and-Stitch vectors (K rows, leading dimension ldo): tau_k * (mask_k / max(sum_j mask_j, 1)) with
     * mask_k = the top int(density * d) of |tau_k| (same select as TIES)
     *                                   ref: merger/algorithms/localize_and_stitch.py:8-49.  w unused. */
    MR_TIES_LNS = 3,
};

/* Selection and build in ONE pass over the data (mode MR_TIES_VECTORS or MR_TIES_FUSED_MERGE, unweighted trim): the
 * result of mr_ties_select(k_cnt) followed by mr_ties_build(mode), bit for bit, for (2K+1)*d*4 resp. (K+2)*d*4 bytes of
 * traffic instead of (3K+2)*d*4 / (2K+3)*d*4.  Two passes over a strided sample bracket each model's cut; ONE full pass
 * then builds `out` with a provisional cut (the middle of the bracket) while it counts the keys above the bracket and
 * collects the ~0.75 % of keys inside it; the exact cut is finished from the collected keys and only the columns whose
 * provisional decision was wrong (keys between the two cuts, ~0.05 %) are rebuilt.  Stream-ordered, no host sync.
 * cut / status / ws as for mr_ties_select: when status[k] != MR_TIES_DONE for some k the contents of `out` are
 * undefined and the caller must run mr_ties_select_exact + mr_ties_build instead.
 * ref: merger/algorithms/ties.py:8-72 (+ weight_learning/module/layer_wise.py:76-82 for FUSED_MERGE). */
int mr_ties_select_build(const float* base, const float* const* models, int K, int64_t d, int64_t k_cnt, int mode,
                         const float* w, int G, const int64_t* seg_end, const int32_t* seg_group, int P, float* out,
                         int64_t ldo, uint64_t* cut, int32_t* status, void* ws, int64_t ws_bytes, mr_stream_t stream);

/* trim_mask / elect_mask: optional dev (K, d) bytes: survived the magnitude trim / survived trim and sign
 * election (That != 0).  NULL to skip. */
int mr_ties_build(const float* base, const float* const* models, int K, int64_t d, const uint64_t* cut, int mode,
                  const float* w, int G, const int64_t* seg_end, const int32_t* seg_group, int P, float* out,
                  int64_t ldo, uint8_t* trim_mask, uint8_t* elect_mask, mr_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Evaluator (B1-B4): full-catalog scoring, per-row top-K, rank of the label.
 * Top-K lists are ordered by score descending, then item id ascending (canonical tie rule; torch.topk's own
 * order among equal scores is unspecified); -0.0 == +0.0 and NaN sorts first like torch.topk.
 * ---------------------------------------------------------------------------------------------- */
#define MR_MAX_TOPK 1024      /* mr_topk_rows / mr_topk_merge */
#define MR_MAX_FUSED_TOPK 128 /* mr_score_topk */

/* Top-K of every row of a materialised (Q, N) score matrix with row stride ld (drop-in for
 * torch.topk(scores, K, dim=1))                                   ref: evaluator/evaluator.py:43
 * out_val / out_id: dev (Q, K); ids are id_base + column.  Requires K <= N. */
int mr_topk_rows(const float* scores, int64_t Q, int64_t N, int64_t ld, int K, int32_t id_base, float* out_val,
                 int32_t* out_id, mr_stream_t stream);

/* mr_topk_rows with items left out of each row: the full-ranking protocol that removes a user's history before
 * Recall@K / NDCG@K are taken (RecBole's full-sort evaluation sets those scores to -inf).
 *   excl_off   dev int64 (Q + 1): CSR offsets by row; row q's list is excl_ids[excl_off[q] .. excl_off[q + 1])
 *   excl_ids   dev int32: global item ids, ascending within a row, duplicates allowed; a row may be empty
 * Row q never lists an item of its list; a row with fewer than K other items ends in slots of id -1, score -inf.  Ids
 * outside [id_base, id_base + N) have no effect, so every shard of a catalog takes the same lists.  Both pointers must
 * be non-NULL (even when every row is empty). */
int mr_topk_rows_exclude(const float* scores, int64_t Q, int64_t N, int64_t ld, int K, int32_t id_base, float* out_val,
                         int32_t* out_id, const int64_t* excl_off, const int32_t* excl_ids, mr_stream_t stream);

/* Merge L per-shard lists (vals / ids: dev (L, Q, K_in), sorted or not, id < 0 = empty slot) into one sorted
 * (Q, K_out) list: the exchange step after the NCCL allgather of per-GPU top-K lists (no reference
 * counterpart; the reference is single-GPU, README.md:51-53).  L * K_in <= 8192. */
int mr_topk_merge(const float* vals, const int32_t* ids, int L, int64_t Q, int K_in, int K_out, float* out_val,
                  int32_t* out_id, mr_stream_t stream);

/* The same merge over the sharded evaluator's exchange buffer: packed = dev L blocks of (2, Q, K_in) 32-bit words,
 * block l = rank l's list with plane 0 the fp32 scores and plane 1 the int32 global ids -- what ONE
 * ncclAllGather of every rank's (2, Q, K_in) buffer leaves behind (SURVEY.md section 8(e) row 1; no reference
 * counterpart, the reference is single-GPU).  L * K_in <= 8192. */
int mr_topk_merge_packed(const void* packed, int L, int64_t Q, int K_in, int K_out, float* out_val, int32_t* out_id,
                         mr_stream_t stream);

/* HOST helper (no device work): the value CPython's builtin sum() gives for the n doubles of x -- the reference's
 * `sum(ndcgs) / len(ndcgs)`, evaluator/metrics.py:61, 88.  compensated != 0: Neumaier summation as in CPython >= 3.12
 * (Python/bltinmodule.c); 0: plain left-to-right addition (older interpreters).  x: host pointer. */
double mr_float_sum(const double* x, int64_t n, int compensated);

/* rank[q] = position of labels[q] in ids[q, :K], or -1          ref: evaluator/metrics.py:51-59, 79-84 */
int mr_label_rank(const int32_t* ids, int64_t Q, int K, const int64_t* labels, int32_t* rank, mr_stream_t stream);

/* Rank of each row's label against the whole row of a materialised (Q, N) score matrix (row stride ld), with no list
 * and no K: count[q] = the number of columns that sort before column labels[q] - id_base under the top-K order
 * (score desc, id asc; -0.0 == +0.0, NaN first), leaving out the ids of row q's exclusion list, if given.  -1 when the
 * label is not in [id_base, id_base + N).  The label's own exclusion is not applied: its count is still the number of
 * eligible items ahead of it.
 *   labels     dev int64 (Q): global item ids
 *   excl_off / excl_ids   as for mr_topk_rows_exclude, both NULL (no exclusion) or both set
 *   count      dev int32 (Q) */
int mr_rank_rows(const float* scores, int64_t Q, int64_t N, int64_t ld, int32_t id_base, const int64_t* labels,
                 const int64_t* excl_off, const int32_t* excl_ids, int32_t* count, mr_stream_t stream);

/* Fused full-catalog scoring + per-row top-K: the tensor-core path (tcgen05.mma kind::tf32 fed by TMA, fp32
 * accumulators in TMEM) that never materialises the (Q, N) score matrix
 *                              ref: module/recommender/module.py:137 followed by evaluator/evaluator.py:43
 *   Uhi, Ulo   dev (Q, E) row-major: the mr_split_tf32 halves of the query embeddings
 *   Ihi, Ilo   dev (N, E) row-major: the halves of this GPU's rows of the item table (split once, reused)
 *   id_base    global id of item row 0 (shard offset); returned ids are id_base + row
 *   mode       MR_SCORE_TF32X3: Uhi.Ilo + Ulo.Ihi + Uhi.Ihi, fp32-faithful (default);
 *              MR_SCORE_TF32X1: Uhi.Ihi only (Ulo / Ilo may be NULL);
 *              MR_SCORE_BF16:   bf16-compat -- Uhi / Ihi point to BF16 arrays (mr_to_bf16; Ulo / Ilo unused), fp32
 *                               accumulation, scores rounded to bf16 before ranking: what the reference's default
 *                               `precision="bf16-mixed"` runs compute (ref: configs/base.py:41, utils.py:84), with the
 *                               canonical tie rule on the many equal bf16 scores.  Needs E % 8 == 0.
 *   out_val / out_id   dev (Q, K), sorted by (score desc, id asc); slots beyond N hold id -1, score -inf
 *   ws         dev scratch of at least mr_score_topk_workspace_bytes(Q, N, E, K) bytes
 * Requires E % 4 == 0, 16-byte aligned operands, 1 <= K <= MR_MAX_FUSED_TOPK.  Scores are exact (hence identical
 * to any fp32 summation order) whenever all products and partial sums are representable, e.g. grid embeddings. */
enum mr_score_mode { MR_SCORE_TF32X3 = 0, MR_SCORE_TF32X1 = 1, MR_SCORE_BF16 = 2 };
int64_t mr_score_topk_workspace_bytes(int64_t Q, int64_t N, int E, int K);
int mr_score_topk(const float* Uhi, const float* Ulo, int64_t Q, const float* Ihi, const float* Ilo, int64_t N, int E,
                  int K, int32_t id_base, int mode, float* out_val, int32_t* out_id, void* ws, int64_t ws_bytes,
                  mr_stream_t stream);

/* mr_score_topk with items left out of each row's list (a user's history), inside the fused kernel: an excluded item
 * never enters the row's candidates, so the list is the exact top-K of the remaining items.
 *   excl_off   dev int64 (Q + 1): CSR offsets by query row; row q's list is excl_ids[excl_off[q] .. excl_off[q + 1])
 *   excl_ids   dev int32: global item ids, ascending within a row, duplicates allowed; a row may be empty
 * Row q never lists an item of its list; a row with fewer than K other items ends in slots of id -1, score -inf.  Ids
 * outside [id_base, id_base + N) have no effect, so every shard (and every streamed chunk) of a catalog takes the same
 * lists.  Same arguments, workspace (mr_score_topk_workspace_bytes) and requirements as mr_score_topk otherwise, plus
 * non-NULL excl_off / excl_ids (even when every row is empty).  Runs in the default kernel geometry whatever the
 * MR_SCORE_BK / MR_SCORE_BF16_EPI_GROUPS experiment settings say. */
int mr_score_topk_exclude(const float* Uhi, const float* Ulo, int64_t Q, const float* Ihi, const float* Ilo, int64_t N,
                          int E, int K, int32_t id_base, int mode, float* out_val, int32_t* out_id, void* ws,
                          int64_t ws_bytes, const int64_t* excl_off, const int32_t* excl_ids, mr_stream_t stream);

/* Rank of each query's label against this GPU's rows of the item table, inside the fused scoring kernel: two
 * passes with the operands and modes of mr_score_topk, and no list.
 * mr_label_score: label_key[q] (dev uint32, Q) = the score key of (query q, item labels[q]) -- the order-preserving
 *   32-bit key of the score the top-K kernel ranks, bit for bit, computed by the same kernel on the gathered label rows
 *   -- or 0 when labels[q] is not in [id_base, id_base + N).  0 is never the key of a score.  On a sharded table,
 *   the maximum over the ranks is the label's key.
 * mr_score_rank: count[q] (dev int32, Q) = the number of this table's items that sort before the label under (score
 *   key desc, id asc), leaving out the ids of row q's exclusion list (excl_off / excl_ids as for mr_score_topk_exclude,
 *   both NULL or both set); -1 when label_key[q] == 0.  The label's own exclusion is not applied.  On a sharded table
 *   the sum of the ranks' counts is the label's 0-based rank in the whole catalog.
 *   labels     dev int64 (Q): global item ids
 *   ws         dev scratch of at least mr_score_rank_workspace_bytes(Q, N, E) bytes (both passes, every mode)
 * Requirements as for mr_score_topk (K aside).  Both run in the default kernel geometry (MR_SCORE_BK and
 * MR_SCORE_BF16_EPI_GROUPS are ignored) and need the same MR_SCORE_CTA_GROUP. */
int64_t mr_score_rank_workspace_bytes(int64_t Q, int64_t N, int E);
int mr_label_score(const float* Uhi, const float* Ulo, int64_t Q, const float* Ihi, const float* Ilo, int64_t N, int E,
                   int32_t id_base, int mode, const int64_t* labels, uint32_t* label_key, void* ws, int64_t ws_bytes,
                   mr_stream_t stream);
int mr_score_rank(const float* Uhi, const float* Ulo, int64_t Q, const float* Ihi, const float* Ilo, int64_t N, int E,
                  int32_t id_base, int mode, const int64_t* labels, const uint32_t* label_key, const int64_t* excl_off,
                  const int32_t* excl_ids, int32_t* count, void* ws, int64_t ws_bytes, mr_stream_t stream);

/* Label ranks bounded by a cap (exact below it, some value >= cap above it): mr_score_rank on a first slice of the
 * table (the probe) already finishes every row whose count reached the cap, so the rest of the table is counted only
 * for the rows still below it, gathered into a compact query set.
 * mr_rank_compact: one launch; selects the rows q with label_key[q] != 0 && probe[q] < cap in ascending q and writes
 *   *live (dev int32) = their number n, idx[i] (dev int32, Q) = their rows, out_labels / out_key (Q) = their labels and
 *   keys, and, when excl_off is set, out_excl_off (dev int64, Q + 1) = the offsets of their exclusion lists packed in
 *   the same order (out_excl_off[0] = 0; the ids follow with mr_rank_gather).
 * mr_rank_gather: compacted row i < n = row idx[i] of the query operands hi (and lo, or NULL in the bf16-compat mode),
 *   rows of row_bytes (a multiple of 16) into out_hi / out_lo, and its exclusion ids into out_excl_ids at
 *   out_excl_off[i] (the four exclusion pointers all NULL or all set).  n is the host's copy of *live.
 * mr_rank_add: count[idx[i]] += part[i] for i < n where part[i] >= 0 (count[i] without idx): the rest's counts onto the
 *   probe's. */
int mr_rank_compact(int64_t Q, const int32_t* probe, int32_t cap, const uint32_t* label_key, const int64_t* labels,
                    const int64_t* excl_off, int32_t* live, int32_t* idx, int64_t* out_labels, uint32_t* out_key,
                    int64_t* out_excl_off, mr_stream_t stream);
int mr_rank_gather(int64_t n, const int32_t* idx, int64_t row_bytes, const void* hi, const void* lo, void* out_hi,
                   void* out_lo, const int64_t* excl_off, const int32_t* excl_ids, const int64_t* out_excl_off,
                   int32_t* out_excl_ids, mr_stream_t stream);
int mr_rank_add(int64_t n, const int32_t* idx, const int32_t* part, int32_t* count, mr_stream_t stream);

/* Log-softmax of each query's label over the whole catalog, inside the fused scoring kernel: a pass of its own with
 * the operands, modes and schedule of mr_score_rank, and no list.  The logit of score f is f / temperature; f is the
 * score the top-K kernel ranks (bf16-rounded in MR_SCORE_BF16).  Supported while |f / temperature| < 1.1e7.
 * mr_score_lse: this table's partial (shift[q] dev int32, sum[q] dev fp64, Q each) = the sum over row q's eligible
 *   items (not in its exclusion list; excl_off / excl_ids as for mr_score_rank, both NULL or both set) of
 *   exp(f / temperature), as sum * 2^shift.  As torch.logsumexp: an eligible NaN gives sum = NaN, an eligible +inf
 *   gives +inf; no eligible item, or only -inf, gives the empty partial (shift = -2^24, sum = 0), also written for N = 0.
 *   temperature must be finite and > 0.  ws: dev scratch of at least mr_score_lse_workspace_bytes(Q, N, E) bytes.
 * mr_lse_finish: merges the (P, Q) partials (shift, sum: row-major, partial p of row q at p * Q + q) of the P shards of
 *   a catalog in index order, then logp[q] (dev fp32, Q) = min(0, log p) with log p = L / temperature - log(total), L
 *   the score of label_key[q] (mr_label_score, maximised over the shards), computed in fp64; NaN when label_key[q] is
 *   0.  The same temperature as mr_score_lse.  Every GPU that merges the same partials gets the same bits. */
int64_t mr_score_lse_workspace_bytes(int64_t Q, int64_t N, int E);
int mr_score_lse(const float* Uhi, const float* Ulo, int64_t Q, const float* Ihi, const float* Ilo, int64_t N, int E,
                 int32_t id_base, int mode, float temperature, const int64_t* excl_off, const int32_t* excl_ids,
                 int32_t* shift, double* sum, void* ws, int64_t ws_bytes, mr_stream_t stream);
int mr_lse_finish(const int32_t* shift, const double* sum, int64_t P, int64_t Q, const uint32_t* label_key,
                  float temperature, float* logp, mr_stream_t stream);

/* Gradient of the label log-softmax with respect to the queries, 3xTF32 only: with logp_q = f_{q,l} / T - lse_q over
 * row q's eligible items and upstream gradient g_q = gscale[q] (dev fp32, Q),
 *     dU[q] += -(g_q / T) * sum_n (p_qn - [n == labels[q]]) * I_n,    p_qn = exp(f_qn / T - lse_q),
 * summed over this table's eligible items (not in the row's exclusion list; excl_off / excl_ids as for mr_score_lse).
 * dU: dev fp32 (Q, E), 16-byte aligned; this table's contribution is added to what it holds.  The scores are recomputed
 * by the instruction sequence of mr_score_lse, and lse_q comes from the (P, Q) partials (shift, sum) of the catalog's
 * shards merged in index order, as mr_lse_finish merges them (P >= 1).  The table is walked in chunks of a fixed
 * number of items, in ascending order: the same inputs give the same bits.  A row with gscale[q] = 0 adds exactly 0;
 * rows whose label is not in the catalog or is excluded want a zero gscale (their log-softmax is NaN / -inf).
 * ws: dev scratch of at least mr_score_lse_grad_workspace_bytes(Q, N, E) bytes (0 for Q = 0 or N = 0). */
int64_t mr_score_lse_grad_workspace_bytes(int64_t Q, int64_t N, int E);
int mr_score_lse_grad(const float* Uhi, const float* Ulo, int64_t Q, const float* Ihi, const float* Ilo, int64_t N, int E,
                      int32_t id_base, float temperature, const int64_t* excl_off, const int32_t* excl_ids,
                      const int64_t* labels, const int32_t* shift, const double* sum, int64_t P, const float* gscale,
                      float* dU, void* ws, int64_t ws_bytes, mr_stream_t stream);

/* Host-only view of the kernel's static schedule for a problem shape (no CUDA call; tests/test_schedule.py).  A unit =
 * (block of 256 queries, contiguous range of 256-item tiles); the grid's CTA pairs run the units in waves of `wave`,
 * unit u on pair u % wave.  plan_out (8 int32): query blocks, item tiles, item splits S, wave, CTAs per pair, item
 * streams (each with its pacing counters), pacing windows per stream, tiles per window.  units_out (optional, 6 int32
 * per unit, at most max_units of them): query block, split, first tile, end tile, stream, units sharing that stream.
 * Returns the number of units (or an argument error < 0). */
int64_t mr_score_topk_schedule(int64_t Q, int64_t N, int K, int mode, int32_t* plan_out, int32_t* units_out,
                               int64_t max_units);

/* Diagnostics: when dev_buf != NULL, later mr_score_topk launches of this thread make block 0 record clock64()
 * stamps per tile (3 roles x 64 tiles x 4 slots of int64: tools/score_sweep.py prints them).  NULL switches it off. */
int mr_score_topk_debug_buffer(void* dev_buf, int64_t bytes);

/* out[i] = bf16(x[i]), round to nearest even (the operand conversion of MR_SCORE_BF16). */
int mr_to_bf16(const float* x, int64_t n, uint16_t* out, mr_stream_t stream);

/* hi = rna_tf32(x), lo = rna_tf32(x - hi): the operand split of the fp32-faithful 3xTF32 contraction. */
int mr_split_tf32(const float* x, int64_t n, float* hi, float* lo, mr_stream_t stream);

/* out[q, n] = sum_e U[q, e] * I[n, e] in plain fp32 on CUDA cores (row-major U (Q, E), I (N, E); out row stride
 * ldo)                                                          ref: module/recommender/module.py:137 */
int mr_scores_fp32(const float* U, int64_t Q, const float* I, int64_t N, int E, float* out, int64_t ldo,
                   mr_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Distillation step between merger and evaluator (SURVEY.md section 8(f) rank 1): per-sample catalogue
 * logits of the merged model, loss against the single-domain ("teacher") logits, gradient w.r.t. the
 * merged model's representations.   ref: module/distiller/sequence/module.py:59-76 (_forward_distill),
 * module/recommender/loss_fn.py:36-231, merge_train.py:116-126 (teacher logits from normalised embeddings).
 * Floating-point contract: fp32 arithmetic, fp64 block sums; compared at 2e-5 relative, not bit-exact.
 * ---------------------------------------------------------------------------------------------- */
#define MR_DISTILL_MAX_B 128     /* samples per call */
#define MR_DISTILL_MAX_GROUPS 64 /* (domain, up to 4 samples) groups per call */
#define MR_DISTILL_MAX_E 1024

enum mr_distill_loss_type { /* ref: merger/enums.py LossType + the two extra classes of loss_fn.py */
    MR_LOSS_CE = 0,
    MR_LOSS_KD = 1,
    MR_LOSS_MSE = 2,
    MR_LOSS_ADAMERGING = 3,
    MR_LOSS_ADAMERGING_KD = 4,
    MR_LOSS_MERGED_PSEUDO_LABEL = 5,
    MR_LOSS_MERGED_PSEUDO_LABEL_KD = 6,
    MR_LOSS_SINGLE_PSEUDO_LABEL = 7,
    MR_LOSS_SINGLE_PSEUDO_LABEL_KD = 8,
    MR_LOSS_PAIRWISE = 9,
    MR_LOSS_LISTNET = 10,
};

/* logits[b, n] = <rep[b, :], item_ptrs[sample_domain[b]][n, :]>  for n < item_rows[sample_domain[b]].
 *   rep            dev (B, E) fp32, 16-byte aligned; E a multiple of 4, <= MR_DISTILL_MAX_E
 *   item_ptrs      host array of nD dev pointers, table d is (item_rows[d], E) row-major, 16-byte aligned
 *   item_rows      host int64[nD];  sample_domain  host int32[B] (the batch's dataset_indexes)
 *   logits         dev (B, ld), ld >= the largest table used.  Every used table is read once for all of its samples.
 *                                                        ref: sequence/module.py:64-66 */
int mr_distill_logits(const float* rep, int B, int E, const float* const* item_ptrs, const int64_t* item_rows, int nD,
                      const int32_t* sample_domain, float* logits, int64_t ld, mr_stream_t stream);

/* loss[b] = loss_type(logits[b, :n_b], teacher_rows[b][:n_b]) exactly as loss_fn(merged.unsqueeze(0), single.unsqueeze(0))
 * (the caller takes the mean over b, sequence/module.py:73); grad_logits[b, :n_b] = d loss[b] / d logits (NULL: skip).
 *   teacher_rows   host array of B dev pointers (NULL entries / NULL array only for the losses that ignore the teacher)
 *   n_per_sample   host int64[B];  temperature for KD / ListNet, coefficient for the *_KD mixes, margin for PAIRWISE.
 * argmax ties take the lowest index (torch.argmax).      ref: loss_fn.py:36-231 */
int mr_distill_loss(const float* logits, int64_t ld, const float* const* teacher_rows, const int64_t* n_per_sample, int B,
                    int loss_type, float temperature, float coefficient, float margin, float* loss, float* grad_logits,
                    int64_t ldg, mr_stream_t stream);

/* grad_rep[b, :] = grad_out[b] * sum_n grad_logits[b, n] * item_ptrs[sample_domain[b]][n, :]  (grad_out NULL: 1).
 * Same host tables as mr_distill_logits; ws: dev scratch of mr_distill_grad_workspace_bytes(E) bytes. Deterministic. */
int64_t mr_distill_grad_workspace_bytes(int E);
int mr_distill_grad(const float* grad_logits, int64_t ldg, const float* grad_out, int B, int E,
                    const float* const* item_ptrs, const int64_t* item_rows, int nD, const int32_t* sample_domain,
                    float* grad_rep, void* ws, int64_t ws_bytes, mr_stream_t stream);

/* out[r, :] = x[r, :] / ||x[r, :]||_2  (may run in place)           ref: merge_train.py:122-123 */
int mr_normalize_rows(const float* x, int64_t rows, int E, float* out, mr_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * PCB-merging vectors (SURVEY.md section 8(f) rank 2).        ref: merger/algorithms/pcb.py:37-58
 * out[k, j] = sign(tau) * clamp(|tau|, lo_k, hi_k) * scale / max(sum_k scale, 1e-12) / K  with the intra- /
 * inter-balancing weights of pcb.py:44-53.  clamp_lo / clamp_hi (dev, K floats) are the int(d*0.01)-th and
 * int(d*0.99 - 1)-th smallest |tau_k| (pcb.py:17-27; obtained with mr_ties_select on the magnitudes);
 * q_index = int(d * (1 - density)) is the ascending rank of the lower clamp of the balancing weights, found here
 * exactly.  flags = 0: fast search -- a 1/32 sample (one pass, keys cached) brackets the quantile between two order
 * statistics of the sample, then ONE pass over everything counts what lies below that window and collects the keys
 * inside it; MR_PCB_DENSE: three full histogram passes instead.  The divisions by per-model ranges and per-column sums
 * use a prepared reciprocal with two FMA corrections (correctly rounded while clamps and divisors lie in
 * [2^-60, 2^60]); MR_PCB_IEEE compiles every division as an IEEE divide instead.  status (dev int32 K) per model:
 * 1 = exact result, 0 = the fast search's window missed (call again with MR_PCB_DENSE), 2 = operands outside the fast
 * divisions' range (call again with MR_PCB_IEEE).  task_out (K rows, ldo) / thr_out (K x {q, max}) are optional
 * diagnostics.  exp / tanh are CUDA's: values agree with torch's CPU kernels to ~1 ulp (floating-point contract).
 * ws: dev scratch of mr_pcb_workspace_bytes(d, K) bytes (sample keys, per-warp candidate lists, histograms). */
enum { MR_PCB_DENSE = 1, MR_PCB_IEEE = 2 };
int64_t mr_pcb_workspace_bytes(int64_t d, int K);
int mr_pcb_vectors(const float* base, const float* const* models, int K, int64_t d, const float* clamp_lo,
                   const float* clamp_hi, int64_t q_index, int flags, int32_t* status, float* out, int64_t ldo,
                   float* task_out, float* thr_out, void* ws, int64_t ws_bytes, mr_stream_t stream);

/* Sharded PCB vectors, stream-ordered (no host synchronisation): mr_pcb_vectors over a flat vector whose columns are split
 * over ranks, bit for bit the single-GPU result on this rank's columns.  Every quantity that spans columns is an order
 * statistic of a model row (clamps, quantile, row maximum) and every float sum stays inside a column, so the search is
 * the single-GPU one with its counters summed over the ranks: the sample is the whole vector's sample (each rank visits
 * the share in its slice), and the fast / dense choice is taken from d_global.  The caller runs phases
 * 0 .. n-1 in order on every rank (n and the collectives from mr_pcb_dist_plan) and, after phase p, applies to the
 * workspace regions that mr_pcb_dist_layout reports (the library never communicates itself):
 *   collectives[p] & MR_PCB_SUM: all-reduce(sum, as int32 words) of the sum region (histograms + below-window counts);
 *   collectives[p] & MR_PCB_MAX: all-reduce(max, as int32 words) of the max region (row maxima + list-overflow flags).
 * The last phase writes status (as mr_pcb_vectors; identical on every rank, since every decision is taken from reduced
 * counts) and builds this slice's vectors into out (K rows, leading dimension ldo).  Slice [j_off, j_off + d_local):
 * j_off a multiple of 32 (unless d_local == 0), the slice ends on a multiple of 32 or at d_global (then ATen's interleaved torch.sum(dim=0)
 * order on the trailing d_global mod 32 columns falls on the last rank exactly as in the single-GPU kernel), d_global <
 * 2^32; d_local == 0 is allowed (base / models / out may then be NULL: the rank contributes zero counts).  clamp_lo /
 * clamp_hi / q_index / flags: the values of the WHOLE vector, the same on every rank.  ws: dev scratch of the size
 * mr_pcb_dist_layout reports.  ref: merger/algorithms/pcb.py:37-58; SURVEY.md section 8(e) merger row. */
enum { MR_PCB_SUM = 1, MR_PCB_MAX = 2 };
int mr_pcb_dist_layout(int64_t d_local, int64_t d_global, int K, int64_t* ws_bytes, int64_t* sum_off, int64_t* sum_bytes,
                       int64_t* max_off, int64_t* max_bytes);
/* HOST helper (no device work): the number of phases (> 0) for d_global / flags; collectives[p] (p < cap) = the
 * MR_PCB_SUM / MR_PCB_MAX bits of the all-reduces after phase p (0 after the last). */
int mr_pcb_dist_plan(int64_t d_global, int flags, int32_t* collectives, int cap);
int mr_pcb_vectors_dist(const float* base, const float* const* models, int K, int64_t d_local, int64_t j_off,
                        int64_t d_global, const float* clamp_lo, const float* clamp_hi, int64_t q_index, int flags,
                        int phase, int32_t* status, float* out, int64_t ldo, void* ws, int64_t ws_bytes,
                        mr_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Sharded merger (SURVEY.md section 8(e)): the flat vector is split over ranks; the global TIES trim
 * (ref: merger/algorithms/ties.py:14-23, top-k over the WHOLE vector) is found by radix refinement of a window of
 * magnitude bit patterns.  For model k and every j < d with bits = bits(|w_k (m_k[j] - base[j])|):
 *   lo[k] <= bits < lo[k] + (2048 << shift[k])  ->  hist[k, (bits - lo[k]) >> shift[k]] += 1
 *   bits >= lo[k] + (2048 << shift[k])          ->  above[k] += 1
 * hist: dev int64 (K, 2048), above: dev int64 (K), both accumulated; the caller zeroes them, all-reduces them over the
 * ranks and picks the bin (mergerec_b200/merger/sharded.py).  lo: dev uint32 (K), shift: dev int32 (K); lo = 0,
 * shift = 20 covers every magnitude.  w: dev K floats or NULL.
 * cand (optional, dev uint32 (K, cand_cap, 2)) / cand_count (dev uint32 (K), zeroed by the caller): for the models with
 * shift[k] == 0, every in-window element also appends (bin, j); cand_count[k] may end above cand_cap (list truncated).
 * The lists resolve equal magnitudes that straddle the cut (lowest index first) without another pass. */
int mr_ties_mag_hist(const float* base, const float* const* models, int K, int64_t d, const float* w, const uint32_t* lo,
                     const int32_t* shift, int64_t* hist, int64_t* above, uint32_t* cand, uint32_t* cand_count,
                     int cand_cap, mr_stream_t stream);

/* Sharded select, stream-ordered (no host synchronisation): the sampled-bracket algorithm of mr_ties_select with every
 * counter summed over the ranks.  Keys carry GLOBAL indices (j_off + local index), so the cut is the single-GPU cut bit
 * for bit.  The caller runs phases 0..5 in order on every rank and applies, after each phase, the collective named
 * here to the workspace regions mr_ties_dist_layout reports (the library never communicates itself):
 *   phases 0-3: all-reduce(sum, as int32 words) of the counters region;  phase 4: all-gather of the survivors region;
 *   phase 5 takes the gathered survivors (`world` regions, rank-major; world == 1: the rank's own region) and writes
 *   cut_local (for mr_ties_build on this rank's slice), optionally cut_global, and status (mr_ties_status).
 * Requires 0 < k_cnt < d_global < 2^32; ws: mr_ties_workspace_bytes(max(d_local, 1), K) + 256 bytes.
 * ref: merger/algorithms/ties.py:14-23 (top-k over the WHOLE vector); SURVEY.md section 8(e) merger row. */
int mr_ties_dist_layout(int64_t d_local, int K, int64_t* counters_off, int64_t* counters_bytes, int64_t* survivors_off,
                        int64_t* survivors_bytes);
int mr_ties_select_dist(const float* base, const float* const* models, int K, int64_t d_local, int64_t j_off,
                        int64_t d_global, const float* w, int64_t k_cnt, int phase, const void* gathered, int world,
                        uint64_t* cut_local, uint64_t* cut_global, int32_t* status, void* ws, int64_t ws_bytes,
                        mr_stream_t stream);

/* DARE merge with explicit keep masks.                       ref: merger/algorithms/dare.py:9-31 (+ torch dropout)
 * out[j] = base[j] (+) sum in order k of fl( fl(w[k] * (models[k][j] - base[j])) * (keep[k, j] ? scale : 0) ),
 * scale = 1 / (1 - p) in fp32.  keep: dev uint8, K rows of leading dimension ld_keep (1 = kept).  w: dev K floats. */
int mr_merge_dare(const float* base, const float* const* models, int K, int64_t d, const float* w, const uint8_t* keep,
                  int64_t ld_keep, float scale, float* out, mr_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* MERGEREC_B200_H_ */
