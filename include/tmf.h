/*
 * tmf.h -- C ABI of libtmf.so, the sm_100a (B200) matrix-factorization hot path
 * that replaces the TensorFlow ops TeAMOFlow's `teamoflow.mf` calls.
 *
 * The reference has NO FFI/operator registry (it is pure Python over TensorFlow), so
 * there is no existing native interface to mirror; every entry point below replaces
 * the TensorFlow call sites cited beside it (paths relative to the reference repo,
 * src/teamoflow/mf/...).  INTEGRATION.md shows the ctypes binding a maintainer adds.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`;
 *   - the caller owns all buffers, including workspaces; the library allocates nothing
 *     persistent (tmf_peer_alloc is an explicit allocation the caller frees) and holds no
 *     global state (except a per-thread error string);
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*); no call
 *     synchronises the device unless its comment says so;
 *   - return value: 0 = ok, negative = TMF_E_* (message via tmf_last_error());
 *   - embedding matrices are row-major fp32 with a leading dimension `ld` (in floats),
 *     `ld % 4 == 0` and 16-byte aligned base (rows are read with 128-bit loads);
 *     columns [r, ld) must be zero;
 *   - index arrays are int32 (nnz and n_users*n_samples must be < 2^31).
 */
#ifndef TMF_H_
#define TMF_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TMF_ABI_VERSION 1

enum {
  TMF_OK = 0,
  TMF_E_INVALID = -1,  /* bad argument (shape / alignment / range) */
  TMF_E_CUDA = -2,     /* CUDA runtime error, see tmf_last_error() */
  TMF_E_WORKSPACE = -3 /* workspace too small */
};

enum { TMF_LOSS_MSE = 0, TMF_LOSS_WMRB = 1 };

typedef void* tmf_stream_t;

#if defined(__GNUC__)
#define TMF_API __attribute__((visibility("default")))
#else
#define TMF_API
#endif

TMF_API int tmf_abi_version(void);
TMF_API const char* tmf_last_error(void); /* thread-local, valid until the next failing call on this thread */

/* ------------------------------------------------------------------ setup (once per fit) */

/* row_ptr[n_rows+1] from row-major-sorted COO row ids (tf_interactions.indices[:,0],
 * loss_graphs.py:47 / utils.py:53-57). */
TMF_API int tmf_rowptr_from_sorted(const int32_t* rows, int64_t nnz, int32_t n_rows, int32_t* row_ptr, tmf_stream_t stream);

/* tf_interactions.indices ([nnz, 2], int64 like tf.sparse.SparseTensor or int32; index_bytes = 8 / 4) -> int32 row and
 * column ids in one pass.  flags[0] (device int32, zeroed by the call): bit 0 = an id outside [0, n_rows) x [0, n_cols)
 * (the reference's gather_nd raises there, matrix_factorization.py:154), bit 1 = not in row-major order. */
TMF_API int tmf_coo_split(const void* indices, int32_t index_bytes, int64_t nnz, int64_t n_rows, int64_t n_cols, int32_t* rows,
                  int32_t* cols, int32_t* flags, tmf_stream_t stream);

/* Stable counting transpose: perm = stable argsort(keys) (keys in [0, n_keys)), ptr[n_keys+1] =
 * segment starts.  Builds the item-major (CSC) view of the interactions and of the sampled
 * negatives (random_ind, matrix_factorization.py:72-73) and X^T for the embedding backward.
 * Workspace size from tmf_transpose_ws_bytes(n). */
TMF_API size_t tmf_transpose_ws_bytes(int64_t n);
TMF_API int tmf_transpose_build(const int32_t* keys, int64_t n, int32_t n_keys, int32_t* ptr, int32_t* perm,
                        void* ws, size_t ws_bytes, tmf_stream_t stream);

/* item-major list of (user, coefficient slot): for e < nnz the user is coo_rows[perm[e]], otherwise
 * (perm[e]-nnz)/n_samples (the flattened [n_users, n_samples] sample table follows the interactions). */
TMF_API int tmf_tlist_users(const int32_t* perm, int64_t n, int64_t nnz, const int32_t* coo_rows, int32_t n_samples,
                    int32_t* users_out, tmf_stream_t stream);

/* Negatives without replacement: S distinct items per user (utils.py:20-22, np.random.choice
 * replace=False) via a keyed bijection of [0, n_items); out is [n_users, S] int64 like random_ind. */
TMF_API int tmf_sample_items(int32_t n_users, int32_t n_items, int32_t n_samples, uint64_t seed, int64_t* out,
                     tmf_stream_t stream);

/* Initializers (initializer_graphs.py:34,51): iid N(0,1) / U[0,1) then a GLOBAL l2 normalise
 * x * rsqrt(max(sum x^2, 1e-12)).  w is [n_rows, ld], only columns < n_cols are filled.
 * ws: >= tmf_reduce_ws_bytes() bytes. */
TMF_API size_t tmf_reduce_ws_bytes(void);
TMF_API int tmf_fill_normal(float* w, int64_t n_rows, int32_t n_cols, int32_t ld, uint64_t seed, tmf_stream_t stream);
TMF_API int tmf_fill_uniform(float* w, int64_t n_rows, int32_t n_cols, int32_t ld, uint64_t seed, tmf_stream_t stream);
TMF_API int tmf_l2_normalize_global(float* w, int64_t n, void* ws, tmf_stream_t stream);

/* ------------------------------------------------------------------ training step */

/* Generic deterministic segment-sum of scaled rows:
 *     out[s, :] = sum_{e in [seg_ptr[s], seg_ptr[s+1])} c(e) * src[idx[e], :]
 *     c(e) = coef[cpos ? cpos[e] : e]   (coef == NULL means c(e) = 1)
 * Covers X.W (embedding_graphs.py:38,58,85), X^T.dE (its backward) and the item-major gradient
 * dE_i = dP^T E_u (backward of matrix_factorization.py:149) without ever forming dP.
 * Fixed chunking => bitwise reproducible.  ws: tmf_spmm_ws_bytes(n_entries, ld_out). */
TMF_API size_t tmf_spmm_ws_bytes(int64_t n_entries, int32_t ld_out);
TMF_API int tmf_spmm_seg(int32_t n_seg, const int32_t* seg_ptr, int64_t n_entries, const int32_t* idx,
                 const int32_t* cpos, const float* coef, const float* src, int32_t ld_src, float* out,
                 int32_t ld_out, int32_t n_cols, void* ws, size_t ws_bytes, tmf_stream_t stream);

/* Fused user-major pass of one training step (replaces matrix_factorization.py:149-167 forward and
 * the user half of :170): per user, sample scores <E_u, E_i[J_u]>, per-interaction scores, the loss
 * (MSE loss_graphs.py:47-52 / WMRB :74-88), d(sum loss)/d(score) coefficients and dE_u.
 *   loss_out[nnz]        per-interaction loss (0 where WMRB ignores a non-positive value)
 *   coef_out[nnz + n_users*n_samples]   c_k, then G[u, j] (WMRB only)
 *   coef_pos (optional, NULL = that natural order): coefficient slot e is stored at coef_out[coef_pos[e]] instead -- pass the
 *   inverse of tmf_transpose_build's permutation and the item-major pass reads its coefficients in list order (tmf_spmm_seg
 *   with cpos = NULL: coalesced) instead of gathering 4-byte values one 32-byte sector each
 *   dEu[n_users, ld]
 *   work list (optional, NULL = one item per user in natural order): n_work items (user, [a, b) slice of the
 *   user's interactions, slot); slot = -1 for whole users, otherwise the row of part_G [n_slots, ceil4(S)] /
 *   part_E [n_slots, ld] that receives the slice's partial sums (very heavy users are split for load balance and
 *   finished by tmf_user_pass_fixup).  Items should be listed heaviest first.  counter: one int32 work counter.
 *   A work item is processed by ONE warp (up to 32 resident per SM), so slices should be short enough that the whole
 *   list fills ~9.5k warp slots (InteractionPlan.slice_len: 32 ... 1024 interactions).
 */
TMF_API int tmf_user_pass(int32_t loss, int32_t n_users, int32_t n_items, int64_t nnz, const int32_t* row_ptr, const int32_t* col_idx,
                  const float* val, const float* Eu, const float* Ei, int32_t ld, int32_t n_comp,
                  const int32_t* samp, int32_t n_samples, int32_t n_work, const int32_t* work_user, const int32_t* work_a,
                  const int32_t* work_b, const int32_t* work_slot, float* part_G, float* part_E, int32_t* counter,
                  float* loss_out, float* coef_out, const int32_t* coef_pos, float* dEu, tmf_stream_t stream);

/* Sums the partial G / dE_u of split users in slice order and adds the sample term (deterministic). */
TMF_API int tmf_user_pass_fixup(int32_t loss, int32_t n_split, const int32_t* split_user, const int32_t* split_first,
                        const int32_t* split_nseg, const float* Ei, int32_t ld, const int32_t* samp, int32_t n_samples,
                        int64_t nnz, const float* part_G, const float* part_E, float* coef_out, const int32_t* coef_pos,
                        float* dEu, tmf_stream_t stream);

/* p[k] = <Eu[rows[k]], Ei[cols[k]]>  (tf.gather_nd(predictions, indices), matrix_factorization.py:154,160) */
TMF_API int tmf_pair_dots(int64_t nnz, const int32_t* rows, const int32_t* cols, const float* Eu, const float* Ei,
                  int32_t ld, float* p, tmf_stream_t stream);

/* KL loss (loss_graphs.py:111-122) in two steps.  tmf_kl_moments reduces the interactions to six additive fp64 sums
 *     moments_out[6] = {n+, sum p+, sum p+^2, n-, sum p-, sum p-^2}
 * and tmf_kl_coef_from_moments derives from them the two groups' means / variances (tf.nn.moments, :116,118), the scalar
 * loss_out[0] and d loss / d p[k] in coef_out[nnz].  Under user sharding (SURVEY 8e) the moments are global: the host sums
 * each rank's six sums (one 48-byte all-reduce) between the two calls.  ws >= tmf_reduce_ws_bytes() for both. */
TMF_API int tmf_kl_moments(int64_t nnz, const float* p, const float* val, double* moments_out, void* ws, tmf_stream_t stream);
TMF_API int tmf_kl_coef_from_moments(int64_t nnz, const float* p, const float* val, const double* moments, float* loss_out,
                             float* coef_out, void* ws, tmf_stream_t stream);

/* Adam step t=1 from zero moments (a new tf.keras.optimizers.Adam each epoch, matrix_factorization.py:176).
 * 128-bit accesses when w and g are 16-byte aligned, scalar otherwise; same bits either way. */
TMF_API int tmf_adam1(float* w, const float* g, int64_t n, float lr, tmf_stream_t stream);

/* Extension (not reference behaviour): Adam with persistent moments m, v (zero-initialised by the caller) and step count
 * `step` >= 1 -- what a single long-lived tf.keras.optimizers.Adam would do; behind fit(optimizer="adam"). */
TMF_API int tmf_adam(float* w, const float* g, float* m, float* v, int64_t n, float lr, int32_t step, tmf_stream_t stream);

/* out[0] = sum(x[0..n)) accumulated in fp64, fixed order (reduce_mean numerator, :179). ws >= tmf_reduce_ws_bytes(). */
TMF_API int tmf_reduce_sum(const float* x, int64_t n, float* out, void* ws, tmf_stream_t stream);

/* ---- BiasedLinear / ReLU embedding pieces (embedding_graphs.py:52-58, :73-87) */
TMF_API int tmf_bias_add(float* E, int64_t n_rows, int32_t n_cols, int32_t ld, const float* bias, int32_t relu, tmf_stream_t stream);
TMF_API int tmf_col_sum(const float* dE, int64_t n_rows, int32_t n_cols, int32_t ld, float* out, void* ws, size_t ws_bytes,
                tmf_stream_t stream); /* ws: 1024*ld floats */
TMF_API int tmf_relu_mask(float* dH, const float* H, int64_t n, tmf_stream_t stream); /* dH *= (H > 0) */
/* C[m,n] (ldc) = op(A) op(B), fp32 FMA chain; ta/tb: 0 = as stored, 1 = transposed. */
TMF_API int tmf_gemm_f32(int32_t ta, int32_t tb, int32_t m, int32_t n, int32_t k, const float* A, int32_t lda,
                 const float* B, int32_t ldb, float* C, int32_t ldc, tmf_stream_t stream);

/* ---- unfused forward-only loss entry points behind LossGraph.get_loss (loss_graphs.py) */
TMF_API int tmf_gather_rows2d(const float* in, int32_t n_rows, int64_t n_cols, const int64_t* index, int32_t k,
                      float* out, tmf_stream_t stream); /* gather_matrix_indices, utils.py:94-105 */
TMF_API int tmf_gather_nd2(const float* in, int64_t n_cols, const int64_t* indices2, int64_t n, float* out,
                   tmf_stream_t stream); /* tf.gather_nd(params, indices[n,2]) */
TMF_API int tmf_wmrb_forward(int64_t n_pos, const int32_t* pos_rows, const float* pos_pred, const float* sample_pred,
                     int32_t n_samples, float scale, float* loss_out, tmf_stream_t stream);

/* ------------------------------------------------------------------ scoring / top-k / metrics */

/* U.V^T (matrix_factorization.py:195) + per-row top-k (tf.math.top_k, :245,:429) as ONE kernel:
 * tcgen05 GEMM on 16-bit operands (fp16 or bf16, whichever rounds the given embeddings more accurately),
 * accumulators in TMEM, fused threshold/candidate epilogue; then an fp32/fp64 canonical rerank so indices
 * are exact.  Scores are never written to HBM.
 *   clamp != 0: scores <= 0 are +0.0 before ranking (recall_at_k path, :237).
 *   item_offset: global index of this GPU's first item (item-sharded scoring).
 *   1 <= k <= min(1024, n_items); k > 128 runs a configuration with longer candidate lists (more workspace).
 *   out_idx[n_users, k] int32 (global ids), out_score[n_users, k] fp32 canonical scores.
 * Workspace from tmf_score_topk_ws_bytes (same n_users, n_items, n_comp and k as the call). */
TMF_API size_t tmf_score_topk_ws_bytes(int64_t n_users, int64_t n_items, int32_t n_comp, int32_t k);
TMF_API int tmf_score_topk(const float* U, int64_t n_users, const float* V, int64_t n_items, int32_t n_comp, int32_t ld,
                   int32_t k, int32_t clamp, int32_t item_offset, int32_t* out_idx, float* out_score, void* ws,
                   size_t ws_bytes, tmf_stream_t stream);

/* Item-sharded scoring with an externally supplied per-row bound: row_bound[n_users] (may be NULL) holds, per
 * user, a LOWER bound of the k-th best canonical score over ALL item slabs (e.g. the k-th best score of the user
 * against any subset of the items, exchanged between GPUs).  A slab then only lists candidates that can still be in
 * the global top-k, skips the per-row warm-up, and rows with fewer than k such candidates are padded with
 * (score -inf, id INT32_MAX) entries, which lose every comparison in tmf_topk_merge*.  The merged result is
 * identical to tmf_score_topk over the concatenated slabs.  k and the workspace as for tmf_score_topk. */
TMF_API int tmf_score_topk_bounded(const float* U, int64_t n_users, const float* V, int64_t n_items, int32_t n_comp, int32_t ld,
                           int32_t k, int32_t clamp, int32_t item_offset, const float* row_bound, int32_t* out_idx,
                           float* out_score, void* ws, size_t ws_bytes, tmf_stream_t stream);

/* Top-k over each row's UNSEEN items (SURVEY 8f-3: "the best k items this user has not interacted with"; the reference
 * ranks seen items too).  ex_ptr[n_users + 1] / ex_idx form a CSR of GLOBAL item ids to exclude, each row sorted ascending
 * with distinct ids; ids outside [item_offset, item_offset + n_items) are ignored.  The result is the top-k of the unseen
 * items by (canonical score desc, id asc), bit-exact like tmf_score_topk: excluded ids are dropped inside the fused kernel
 * before they reach a row's candidate list or its threshold histogram, so the exactness argument holds with "items" read
 * as "unseen items".  clamp != 0 ranks by max(s, 0) like tmf_score_topk (zero-score ties are the lowest unseen ids).
 * Rows with fewer than k unseen items end in (score -inf, id INT32_MAX) padding, as tmf_score_topk_bounded writes it, so
 * item slabs merge with tmf_topk_merge.  k and the workspace as for tmf_score_topk. */
TMF_API int tmf_score_topk_masked(const float* U, int64_t n_users, const float* V, int64_t n_items, int32_t n_comp, int32_t ld,
                          int32_t k, int32_t clamp, int32_t item_offset, const int32_t* ex_ptr, const int32_t* ex_idx,
                          int32_t* out_idx, float* out_score, void* ws, size_t ws_bytes, tmf_stream_t stream);

/* The raw tensor-core scores s~ of tmf_score_topk's GEMM, written densely (P[n_users, n_items], small shapes only), to
 * test the error bound the exact top-k rests on.  With u~ = u rounded to the operand format and du = u - u~ (likewise v~, dv):
 *   |s~ - s| <= |du| |v| + |u~| |dv| + 2.4e-7 * k_pad * |u~| |v|,   k_pad = n_comp rounded up to a multiple of 64.
 * operand_format: -1 = chosen from the data like tmf_score_topk does (fp16 where the embeddings fit its range and it
 * rounds them more accurately than bf16), 0 = bf16, 1 = fp16.  Workspace as for tmf_score_topk with k = 1. */
TMF_API int tmf_score_dense_tc(const float* U, int64_t n_users, const float* V, int64_t n_items, int32_t n_comp, int32_t ld,
                       int32_t operand_format, float* P, void* ws, size_t ws_bytes, tmf_stream_t stream);

/* merge G per-shard top-k lists ([G, n_users, k], each row sorted as tmf_score_topk writes it) -> [n_users, k],
 * comparator (score desc, idx asc); G <= 16. */
TMF_API int tmf_topk_merge(const int32_t* idx_in, const float* score_in, int32_t n_lists, int64_t n_users, int32_t k,
                   int32_t* out_idx, float* out_score, tmf_stream_t stream);

/* dense canonical scores P[n_users, n_items] (predict(), :195) -- small shapes only. */
TMF_API int tmf_predict_dense(const float* U, int64_t n_users, const float* V, int64_t n_items, int32_t n_comp, int32_t ld,
                      float* P, tmf_stream_t stream);

/* full descending ranking of every row of P (top_k(k = n_items), :336,:367,:432,:438), ties -> lower index. */
TMF_API size_t tmf_rank_rows_ws_bytes(int64_t n_rows, int64_t n_cols);
TMF_API int tmf_rank_rows(const float* P, int64_t n_rows, int64_t n_cols, int32_t clamp, int32_t* out_idx, void* ws,
                  size_t ws_bytes, tmf_stream_t stream);

/* predict(A)'s second output (matrix_factorization.py:197-198: gather_nd(P, where(A == 0)) flattened row-major) from the
 * CSR (a_ptr, a_idx: sorted columns) of the NON-ZERO cells of A -- no dense A.  out has n_users*n_items - nnz entries. */
TMF_API int tmf_gather_unobserved(const float* P, int64_t n_users, int64_t n_items, const int32_t* a_ptr, const int32_t* a_idx,
                          float* out, tmf_stream_t stream);

/* Measurement aid (no reference counterpart): reads the rows table[idx[e]] (ld = 64 or 128 floats) for e < n the way
 * tmf_user_pass gathers embedding rows, folds them into per-thread sums written to out[148 * 8 * 256].  bench.py times it on
 * the workload's own index stream: the achievable gather rate is tmf_user_pass's roofline denominator when the table fits
 * the L2.  Indices must lie in [0, n_rows). */
TMF_API int tmf_gather_rate(const float* table, int64_t n_rows, int32_t ld, const int32_t* idx, int64_t n, float* out,
                    int64_t out_len, tmf_stream_t stream);

/* hits[u] = #{i in topk[u] : A[u,i] != 0}, relevant[u] = #{i : A[u,i] > 0} for CSR A (:248-254). */
TMF_API int tmf_metrics_hits(const int32_t* topk, int64_t n_users, int32_t k, const int32_t* a_ptr, const int32_t* a_idx,
                     const float* a_val, float* hits, float* relevant, tmf_stream_t stream);

/* dcg[u] = sum_{q<k} (2^A[u,topk[u,q]] - 1) / log2(q+2)   (:339-351) */
TMF_API int tmf_dcg(const int32_t* topk, int64_t n_users, int32_t k, const int32_t* a_ptr, const int32_t* a_idx,
            const float* a_val, float* dcg, tmf_stream_t stream);
/* idcg[u]: gains of row u sorted descending (zeros between positives and negatives), first k (:370-384) */
TMF_API int tmf_idcg(int64_t n_users, int64_t n_items, int32_t k, const int32_t* a_ptr, const float* a_val, float* idcg,
             float* row_nnz, tmf_stream_t stream);

/* fp32-accurate GEMM on the tensor cores (tcgen05 + TMEM + TMA): C[m, n] = op(A) op(B) with the same operand conventions as
 * tmf_gemm_f32 (ta: A is stored [k, m]; tb: B is stored [n, k]; row-major, leading dimensions in floats).  Every operand is split
 * exactly into three bf16 planes and the six significant plane products are accumulated in fp32 (error ~ 3 * 2^-24 |a||b| per
 * product: the 1e-5 tolerance of north_star holds).  Used for the dense contractions of the towers -- the ReLU embedding's second
 * stage and its backward (embedding_graphs.py:85-87) and X.W / X^T.dE for genuinely dense features (embedding_graphs.py:38) --
 * above a size threshold; deterministic (fixed K-split order).  ws: tmf_gemm_tc_ws_bytes(m, n, k). */
TMF_API size_t tmf_gemm_tc_ws_bytes(int64_t m, int64_t n, int64_t k);
TMF_API int tmf_gemm_tc(int32_t ta, int32_t tb, int64_t m, int64_t n, int64_t k, const float* A, int64_t lda, const float* B,
                int64_t ldb, float* C, int64_t ldc, void* ws, size_t ws_bytes, tmf_stream_t stream);

/* ------------------------------------------------------------------ multi-GPU exchange over NVLink peer memory
 * (new-build, SURVEY 8e: the reference has no distribution).  One process per GPU; a rank allocates its exchange
 * buffers with tmf_peer_alloc (plain cudaMalloc, zero-filled, SYNCHRONOUS), exports them with tmf_ipc_export (64-byte
 * handle, exchanged by the host, e.g. torch.distributed.all_gather_object) and maps the peers' buffers with
 * tmf_ipc_open.  Arrays named *_host below are HOST arrays of `world` device pointers, index = rank (the own
 * entry is the local pointer).  These three calls and tmf_peer_free/tmf_ipc_close take no stream. */
#define TMF_IPC_HANDLE_BYTES 64
#define TMF_MAX_PEERS 16
TMF_API int tmf_peer_alloc(size_t bytes, void** out);
TMF_API int tmf_peer_free(void* p);
TMF_API int tmf_ipc_export(const void* dev_ptr, void* handle_host);
TMF_API int tmf_ipc_open(const void* handle_host, void** out);
TMF_API int tmf_ipc_close(void* p);

/* Stream-ordered barrier between the ranks: pads_host[g] = rank g's pad (256 bytes, zero-initialised, in peer
 * memory: uint32 arrival slots [0, TMF_MAX_PEERS) + a private epoch counter at byte 128); every rank calls it with the
 * same, strictly increasing `epoch` (>= 1), or with epoch = 0 = "the next value of the device-side counter" (no
 * per-call argument: replayable from a CUDA graph; do not mix the two forms on one pad).  Work enqueued before the
 * barrier on any rank is visible to work enqueued after it on every rank.  A peer missing for `timeout_ms`
 * (0 = the default, 120 s) does NOT trap: the waiting rank stores 1 + (the missing rank) into the uint32 at byte 132 of
 * its own pad (sticky) and leaves the barrier; the host reads that word at its next synchronisation point and raises. */
TMF_API int tmf_peer_barrier(const void* const* pads_host, int32_t world, int32_t rank, uint32_t epoch, uint32_t timeout_ms,
                     tmf_stream_t stream);

/* all-to-all + merge + all-gather of item-sharded top-k lists in one kernel: for rows [row_lo, row_lo + n_rows) read
 * the `world` per-slab lists idx_host[g] / score_host[g] ([n_users, k] each, in rank g's memory), merge them like
 * tmf_topk_merge and store the merged rows into out_idx_host[d] / out_score_host[d] for d < n_out. */
TMF_API int tmf_topk_merge_peer(const void* const* idx_host, const void* const* score_host, int32_t world, int64_t row_lo,
                        int64_t n_rows, int32_t k, const void* const* out_idx_host, const void* const* out_score_host,
                        int32_t n_out, tmf_stream_t stream);

/* reduce-scatter + (optional Adam step 1) + all-gather of an fp32 buffer in one kernel: for elements
 * [elem_off, elem_off + n_elems) (multiples of 4) s = sum_g part_host[g][e] in rank order (deterministic; every rank
 * receives the same bits); lr < 0: dst_host[g][e] = s for every g (all-reduce of the item-side gradient dE_i between
 * the item-major pass and the update, matrix_factorization.py:171 under user sharding; dst may alias part);
 * lr >= 0: dst_host[g][e] = adam1(dst_host[rank][e], s) (the update of :176 fused in, dst = the replicated weights). */
TMF_API int tmf_peer_reduce_push(const void* const* part_host, const void* const* dst_host, int32_t world, int32_t rank,
                         int64_t elem_off, int64_t n_elems, float lr, tmf_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* TMF_H_ */
