/*
 * scd_b200 - C ABI of the B200-native clustering-and-naming hot path of Visual-AI/SCD.
 *
 * The reference has no FFI: its hot path is plain PyTorch calls inside two Python classes and two
 * driver scripts.  Each entry point below therefore cites the reference *call site(s)* whose device
 * work it replaces (paths relative to the reference checkout).  The Python layer in scd_b200/
 * keeps the reference's class / function signatures and calls these through ctypes.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (torch tensors kept alive by the host
 *     layer) unless it says "host"; no function allocates; scratch comes in through (ws, ws_bytes)
 *     sized by the matching *_workspace_bytes();
 *   - `stream` is a cudaStream_t passed as void*; calls only enqueue work, they never synchronise;
 *   - return 0 on success, non-zero on error with a message in scd_last_error() (thread local);
 *   - matrices are row-major and dense unless a leading dimension is given.
 */
#ifndef SCD_B200_H_
#define SCD_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define SCD_API __attribute__((visibility("default")))
#else
#define SCD_API
#endif

typedef void* scd_stream_t;      /* cudaStream_t */
typedef uint16_t scd_bf16_t;     /* raw bfloat16 bits */

SCD_API int scd_version(void);
SCD_API const char* scd_last_error(void);
/* Debugging aid (no reference counterpart): when non-NULL, scd_name_topk fills [pairs][16] int64 cycle
 * counters (issuer / epilogue wait times) into this device buffer; NULL switches it off. */
SCD_API void scd_debug_set_name_profile(void* dev_buf_pairs_x16_i64);

/* ---------------------------------------------------------------- k-means (a1-a4) */

/* local_utils/faster_mix_k_means_pytorch.py:177-212 pairwise_distance (copies: sskm_constrained.py:189,
 * gcd/methods/clustering/faster_mix_k_means_pytorch.py:9): out[n,k] = sum_d (X[n,d]-C[k,d])^2, direct form, fp32.
 * cost_x1000 (nullable, [N,K] int32) = round(1000*sqrt(out)): local_utils/sskm_constrained.py:116 + :324. */
SCD_API int scd_pairwise_distance(const float* X, int64_t N, int D, const float* C, int K,
                          float* out /* nullable */, int32_t* cost_x1000 /* nullable */, scd_stream_t stream);

/* E-step, faster_mix_k_means_pytorch.py:58-60 / :105-107: labels = argmin_k dist (ties -> lowest k, NaN wins),
 * mindist = min_k dist, *inertia_acc += sum(mindist) (fp64 accumulator, caller zeroes it).
 * Tensor-core path (D % 8 == 0, D >= 40, K <= 1024, X 16-byte aligned): ||x||^2 - 2 x.c + ||c||^2 with the contraction
 * issued as three bf16 tcgen05 MMAs (hi/lo split of x and c, fp32 accumulate; X is read once, as fp32).
 * Other shapes: the fp32 direct-form kernel of scd_pairwise_distance with the argmin fused (SCD_ESTEP_EXACT forces it).
 * ws holds the per-iteration centroid hi/lo planes and norms; they are recomputed from C by a small kernel unless
 * SCD_ESTEP_PLANES_READY says the previous scd_finalize_centers already left them there. */
#define SCD_ESTEP_EXACT 1          /* force the fp32 direct-form kernel */
#define SCD_ESTEP_PLANES_READY 2   /* ws already holds the operands of C: scd_finalize_centers(estep_ws = ws) wrote them */
SCD_API size_t scd_estep_workspace_bytes(int K, int D);
/* 1 when (N, D, K) takes the tensor-core path (given an aligned X and a workspace) - what the host layer needs to know
 * before it asks scd_finalize_centers to prepare the next E-step's operands. */
SCD_API int scd_estep_uses_tensor_cores(int64_t N, int D, int K);
SCD_API int scd_estep(const float* X, int64_t N, int D, const float* C, int K,
              int64_t* labels, float* mindist /* nullable */, double* inertia_acc /* nullable */, int flags,
              void* ws, size_t ws_bytes, scd_stream_t stream);

/* k-means++ seeding, faster_mix_k_means_pytorch.py:20-36 (gcd copy :82-110), without the per-centre N x c distance
 * matrix and without a host round trip per centre:
 *   scd_kpp_update: d2[i] = min(d2[i], ||X_i - X[*pick]||^2) (first != 0: plain assignment), center_out[:] = X[*pick]
 *                   (nullable), per-block fp64 sums of d2 into ws; *pick < 0 leaves d2 as it is; `center` (row-sharded
 *                   seeding, SURVEY 8e: the picked row was broadcast by the rank that owns it) replaces X[*pick];
 *   scd_kpp_select: the reference's draw  prob = d2/sum(d2); ind = first i with cumsum(prob)[i] >= r  (:31-34) resolved
 *                   on the device with fp64 prefix sums; when no row qualifies *pick keeps its value and *no_hit |= 1
 *                   (|= 2 if *pick < 0, i.e. nothing to reuse; sticky, the caller zeroes it once): the gcd copy
 *                   :104-107 reuses the previous index, the local copy :34 raises IndexError.
 *                   sums_valid = 0 recomputes the block sums from d2 first (d2 produced by scd_estep's mindist). */
SCD_API size_t scd_kpp_workspace_bytes(int64_t N);
SCD_API int scd_kpp_update(const float* X, int64_t N, int D, const int64_t* pick /* nullable when center */,
                   const float* center /* nullable, [D]: measure against this vector instead of X[*pick] */, int first,
                   float* d2, float* center_out /* nullable, [D] */, void* ws, size_t ws_bytes, scd_stream_t stream);
SCD_API int scd_kpp_select(const float* d2, int64_t N, int sums_valid, double r, int64_t* pick, int32_t* no_hit,
                   void* ws, size_t ws_bytes, scd_stream_t stream);

/* Labelled-row inertia, faster_mix_k_means_pytorch.py:108-109: *acc += sum_i ||L[i]-C[labels[i]]||^2. */
SCD_API int scd_labelled_inertia(const float* L, const int64_t* labels, int64_t n, int D, const float* C, int K,
                         double* acc, scd_stream_t stream);

/* M-step sums, faster_mix_k_means_pytorch.py:61-64 / :113-116 (native analogue: k_means_constrained/
 * sklearn_import/cluster/_k_means.pyx:29-83): sums[k,:] = sum of rows with labels==k, counts[k] = #rows.
 * Labels outside [0,K) are ignored.  sums/counts are overwritten.  Also leaves the label-sorted row order
 * in the workspace (used by scd_vote).  Split from the divide so an all-reduce can sit between. */
SCD_API size_t scd_mstep_workspace_bytes(int64_t N, int K);
SCD_API int scd_mstep_sums(const float* X, const int64_t* labels, int64_t N, int D, int K,
                   float* sums /* [K,D] */, int32_t* counts /* [K] */, void* ws, size_t ws_bytes, scd_stream_t stream);

/* Row-sharded k-means (SURVEY 8e): tail of the packed fp32 all-reduce buffer [K*D sums | K counts | inertia]:
 * out[0..K) = (float)counts, out[K] = (float)*inertia (0 when NULL).  The host layer all-reduces the buffer
 * (NCCL) between scd_mstep_sums and scd_finalize_centers(counts_f = out). */
SCD_API int scd_pack_counts_inertia(const int32_t* counts, const double* inertia /* nullable */, int K, float* out,
                            scd_stream_t stream);

/* centers = sums / counts (empty cluster -> NaN row, like torch.mean over zero rows; no relocation), and
 * faster_mix_k_means_pytorch.py:71 / :123: ws[k] = ||C_new[k]-C_old[k]||_2 (K floats, when C_old and ws are given) and
 * *shift = sum_k ws[k] (nullable: the host layer reads the K norms with the inertia and adds them itself, which
 * saves a launch).  counts_f (nullable) takes float counts instead (e.g. after a packed fp32 all-reduce).
 * estep_ws (nullable, scd_estep_workspace_bytes(K, D)): also receives the next E-step's operands of C_new (bf16 hi / lo
 * planes + ||c||^2, bit-identical to what scd_estep derives from C_new), see SCD_ESTEP_PLANES_READY. */
SCD_API int scd_finalize_centers(const float* sums, const int32_t* counts, const float* counts_f, const float* C_old,
                         float* C_new, float* shift, int K, int D, void* ws, size_t ws_bytes,
                         void* estep_ws /* nullable */, size_t estep_ws_bytes, scd_stream_t stream);

/* ---------------------------------------------------------------- naming (a8, a9, a11) */

/* zeroshot_weights [D,V] (V contiguous, clip_lang_util.py:107; row stride ldw elements; fp32 or bf16)
 * -> Wt [V,D] bf16, the K-major operand layout.  One-off per vocabulary. */
SCD_API int scd_vocab_prepare(const void* W, int w_is_bf16, int D, int64_t V, int64_t ldw, scd_bf16_t* Wt, scd_stream_t stream);
SCD_API int scd_cast_bf16(const float* in, int64_t n, scd_bf16_t* out, scd_stream_t stream);
/* out[r,:] = Wt[sel[r],:] - the K voted columns, main_unsup.py:601-602 / main_ptsup.py:668-669. */
SCD_API int scd_gather_rows_bf16(const scd_bf16_t* Wt, const int64_t* sel, int n_sel, int D, int64_t V, scd_bf16_t* out,
                         scd_stream_t stream);

/* main_unsup.py:519-529, main_ptsup.py:538-543 (and :92-96, :116-120; k=1: main_unsup.py:610-614):
 *   logits = scale * X @ Wt^T ; [softmax over V] ; top-k per row, largest first, ties -> lower index.
 * X [N,D] bf16, Wt [V,D] bf16 (D <= 768, D % 8 == 0), k <= 8.  vals [N,k] fp32 (scaled logits, or softmax
 * probabilities when want_softmax), idx [N,k] int64 = column + idx_offset (vocabulary-shard offset).
 * row_max/row_sumexp (nullable, [N]): unscaled row max and sum exp(scale*(x-max)) for cross-shard softmax.
 * The N x V score matrix is never written. */
SCD_API size_t scd_name_topk_workspace_bytes(int64_t N, int64_t V, int k);
/* Introspection (no reference counterpart): the work partition scd_name_topk uses for (N, V, k) on the current device -
 * out[0] = 256-row blocks, out[1] = vocabulary tiles per sweep, out[2] = CTA pairs launched, out[3] = most pieces any
 * row block is cut into (the (row block, tile) space is cut into one contiguous range per pair), out[4] = tiles of the
 * least loaded pair (the busiest has at most one more), out[5] = work items the busiest pair starts.  Host-only. */
SCD_API int scd_name_topk_plan(int64_t N, int64_t V, int k, int32_t* out6 /* host */);
/* The work items of one CTA pair under that partition, in execution order: out[i] = {row block, first tile, tiles,
 * piece ordinal of the row block (= partial-list slot)}.  Returns the number of items (at most max_items are written),
 * or -1 on bad arguments.  Host-only. */
SCD_API int scd_name_topk_plan_pair(int64_t N, int64_t V, int k, int pair, int32_t* out_items_x4 /* host */, int max_items);
SCD_API int scd_name_topk(const scd_bf16_t* X, int64_t N, int D, const scd_bf16_t* Wt, int64_t V, float scale, int k,
                  int want_softmax, int64_t idx_offset, float* vals, int64_t* idx,
                  float* row_max, float* row_sumexp, void* ws, size_t ws_bytes, scd_stream_t stream);

/* k-way merge of `parts` per-row top-k lists (vocabulary shards after an all-gather): [parts,N,k] -> [N,k].
 * part_vals are scaled logits (as written by scd_name_topk without softmax); with want_softmax the
 * per-part (row_max, row_sumexp) finish the softmax: p = exp(v - scale*M) / sum_p s_p*exp(scale*(m_p-M)). */
SCD_API int scd_topk_merge(const float* part_vals, const int64_t* part_idx, const float* part_max, const float* part_sum,
                   int parts, int64_t N, int k, float scale, int want_softmax, float* vals, int64_t* idx,
                   scd_stream_t stream);

/* main_unsup.py:575-582 / main_ptsup.py:636-644: per cluster c, Counter over topk_idx[cluster_of_row==c, :k_used]
 * minus `excluded` names, then most_common(M) with Python's tie order (first occurrence in the row-major
 * flattening).  out_names [K,M] int64 (-1 padded), out_counts [K,M], out_distinct [K] (#distinct names),
 * out_rows [K] (#rows in cluster).
 * A cluster's name histogram lives in a 16384-slot shared-memory table while rows * k_used <= 8192; larger clusters
 * build it in `spill` (nullable; scd_vote_spill_bytes(N, k_used) bytes of device memory, 24 bytes per top-k entry).
 * Without a spill buffer such a cluster can exhaust the table: *overflow (device int) is then set to 1 and its counts
 * are incomplete - callers must check it. */
SCD_API size_t scd_vote_workspace_bytes(int64_t N, int K);
SCD_API size_t scd_vote_spill_bytes(int64_t N, int k_used);
SCD_API int scd_vote(const int64_t* topk_idx, int k_total, int k_used, const int64_t* cluster_of_row, int64_t N, int K,
             const int64_t* excluded, int n_excluded, int M, int64_t* out_names, int32_t* out_counts,
             int32_t* out_distinct, int32_t* out_rows, int32_t* overflow, void* ws, size_t ws_bytes,
             void* spill /* nullable */, size_t spill_bytes, scd_stream_t stream);

/* Same vote when the rows were already sorted by these very cluster labels: `mstep_ws` is the workspace a
 * scd_mstep_sums(X, labels, N, D, K, ...) call on the same labels has just filled (k-means labels are what
 * main_unsup.py:575 votes with) - the counting sort is not repeated.  Per-cluster row counts are the
 * M-step's `counts`. */
SCD_API int scd_vote_presorted(const int64_t* topk_idx, int k_total, int k_used, const void* mstep_ws, int64_t N, int K,
                       const int64_t* excluded /* nullable */, int n_excluded, int M,
                       int64_t* out_names, int32_t* out_counts, int32_t* out_distinct, int32_t* overflow,
                       void* spill /* nullable */, size_t spill_bytes, scd_stream_t stream);

/* Row-sharded multi-GPU vote (SURVEY 8e): rec[i] = [label_i, name_i0 .. name_i(k_used-1)] as int32 - one record per
 * image row, so ONE all-gather moves a rank's labels and top-k names (4 * (1 + k_used) bytes per row) and
 * scd_vote_records runs the vote of main_unsup.py:575-582 on the gathered records (same outputs as scd_vote). */
SCD_API int scd_pack_vote_records(const int64_t* labels, const int64_t* topk_idx, int k_total, int k_used, int64_t n,
                          int32_t* rec /* [n, 1 + k_used] */, scd_stream_t stream);
SCD_API int scd_vote_records(const int32_t* rec, int k_used, int64_t N, int K, const int64_t* excluded /* nullable */,
                     int n_excluded, int M, int64_t* out_names, int32_t* out_counts, int32_t* out_distinct,
                     int32_t* out_rows, int32_t* overflow, void* ws, size_t ws_bytes,
                     void* spill /* nullable */, size_t spill_bytes, scd_stream_t stream);

/* ---------------------------------------------------------------- size-constrained assignment (a7) */

/* counts[k] = |{i : labels[i] == k}| (int32 [K], overwritten); labels outside [0,K) are ignored.  The size check of
 * the constrained E-step (is the plain argmin already within size_min..size_max?) and a building block of the M-step. */
SCD_API int scd_label_histogram(const int64_t* labels, int64_t N, int K, int32_t* counts, scd_stream_t stream);


/* local_utils/sskm_constrained.py:226-274 _labels_constrained (graph :277-328, OR-Tools solve :331-356):
 * minimise sum_i cost[i, labels[i]] with size_min <= |cluster k| <= size_max for every k.
 * cost: HOST int32 [N,K] = round(1000*sqrt(dist)) (scd_pairwise_distance's cost_x1000, copied to the host as the
 * reference does, :116); labels: HOST int32 [N] (the reference's labels.astype(np.int32), :265).
 * Exact optimum by successive shortest augmenting paths from the row-argmin assignment; *total_cost (nullable) is
 * the optimal objective, *n_augment (nullable) the number of unit augmentations (0 = the bounds were inactive).
 * Returns 0, 1 (bad arguments) or 2 (infeasible: the reference raises 'There was an issue with the min cost flow
 * input.', :349-350).  Host-only: no stream, no device memory. */
SCD_API int scd_constrained_assign(const int32_t* cost, int64_t N, int K, int64_t size_min, int64_t size_max,
                           int32_t* labels, int64_t* total_cost /* nullable */, int64_t* n_augment /* nullable */);

/* ---------------------------------------------------------------- multi-GPU exchange over NVLink peer memory (SURVEY 8e) */

/* The reference is single-GPU (SURVEY 2: no distributed call site); these entry points exist because north_star shards
 * the path.  One process per GPU; every rank allocates an exchange buffer and a flag pad in peer-mappable memory and
 * passes HOST tables of the G mapped device pointers (index = rank; scd_b200/peer.py builds them with torch symmetric
 * memory).  `channel` (0..7) selects one of the pad's independent barrier counters; all ranks must issue the same
 * sequence of calls per channel.  Waits are bounded (4 s) and trap with a message instead of hanging. */
SCD_API size_t scd_peer_flag_bytes(void);                 /* bytes of a flag pad; the caller zeroes it once, before first use */
SCD_API size_t scd_peer_mstep_bytes(int K, int D);        /* bytes of one M-step exchange block: [K*D sums f32 | K counts i32 | pad | inertia f64] */
SCD_API int scd_peer_barrier(void* const* peer_flags, int world, int rank, int channel, scd_stream_t stream);
/* local_utils/faster_mix_k_means_pytorch.py:61-64 + :71 over row shards: the all-reduce of the per-rank
 * [sums | counts | inertia] blocks (at byte offset buf_byte_offset of every rank's exchange buffer, filled by
 * scd_mstep_sums / scd_estep writing straight into it) fused with scd_finalize_centers: flag barrier, peer loads added in
 * rank order (bitwise identical centres on every rank), divide, move norms, next E-step operands.  counts_out (nullable,
 * [K] fp32) / inertia_out (nullable, fp64 scalar): the reduced counts and inertia. */
SCD_API int scd_finalize_centers_peer(void* const* peer_bufs, void* const* peer_flags, int world, int rank, int channel,
                              size_t buf_byte_offset, const float* C_old /* nullable */, float* C_new,
                              float* move_norms /* nullable, [K] */, float* counts_out, double* inertia_out, int K, int D,
                              void* estep_ws /* nullable */, size_t estep_ws_bytes, scd_stream_t stream);
/* main_unsup.py:575-577 over row shards: scd_pack_vote_records whose stores ARE the all-gather - record i of this rank goes
 * to row (row_offset + i) of the [N_total, 1 + k_used] int32 array at buf_byte_offset of EVERY rank's exchange buffer.
 * Follow with scd_peer_barrier before scd_vote_records reads the local copy. */
SCD_API int scd_pack_vote_records_peer(void* const* peer_bufs, int world, int rank, size_t buf_byte_offset, const int64_t* labels,
                               const int64_t* topk_idx, int k_total, int k_used, int64_t n, int64_t row_offset,
                               scd_stream_t stream);

/* The same exchange without a second sort: records leave in the label-sorted order scd_mstep_sums has just produced on this
 * rank (mstep_ws), record = [global row id = row_offset + local row, name_0 .. name_(k-1)], slot row_offset + sorted
 * position; the rank's [K + 1] offsets go to row `rank` of the [world, K + 1] int32 table at off_byte_offset of every rank's
 * buffer.  scd_vote_segments (after scd_peer_barrier) votes by walking the `world` sorted runs of each cluster:
 * rec = the local gathered array [world * per, 1 + k_used], per = rows per rank block, n_total = rows of all ranks (sizes the
 * spill tables); same outputs as scd_vote_records. */
SCD_API int scd_pack_sorted_records_peer(void* const* peer_bufs, int world, int rank, size_t rec_byte_offset, size_t off_byte_offset,
                                 const int64_t* topk_idx, int k_total, int k_used, int64_t n, int64_t row_offset,
                                 const void* mstep_ws, int K, scd_stream_t stream);
SCD_API int scd_vote_segments(const int32_t* rec, int k_used, int64_t n_total, int64_t per, int world, const int32_t* seg_offsets, int K,
                      const int64_t* excluded /* nullable */, int n_excluded, int M, int64_t* out_names, int32_t* out_counts,
                      int32_t* out_distinct, int32_t* out_rows, int32_t* overflow, void* spill /* nullable */, size_t spill_bytes,
                      scd_stream_t stream);

/* ---------------------------------------------------------------- evaluation either side of the path (SURVEY 8f, rank 4) */

/* gcd/project_utils/cluster_and_log_utils.py:45-49 (split_cluster_acc_v2: `for i in range(y_pred.size):
 * w[y_pred[i], y_true[i]] += 1`) and the match counts of main_unsup.py:149-167 evaluate_semantic_acc:
 * w [D,D] int64 (overwritten), row = predicted cluster, column = true class.  Either label vector may be int64 or
 * float64 (the drivers' `targets` are float64, main_unsup.py:118,132; the reference casts with .astype(int)).
 * first_row (nullable, [D] int64): first row index whose true class is t, N if the class never occurs (the order
 * in which evaluate_semantic_acc's defaultdict meets the classes).  mask (nullable, [N] bytes, non-zero = set) with
 * col_masked ([D] int64, overwritten): rows of true class t under the mask - :43-44's old/new class sets are the
 * classes with col_masked > 0 / column sum - col_masked > 0.  *bad (device int32, caller zeroes) |= 1 when a label
 * falls outside [0, D). */
SCD_API int scd_contingency(const void* y_pred, int pred_is_f64, const void* y_true, int true_is_f64, int64_t N, int D,
                    const uint8_t* mask /* nullable */, int64_t* w, int64_t* first_row /* nullable */,
                    int64_t* col_masked /* nullable unless mask */, int32_t* bad, scd_stream_t stream);

/* ---------------------------------------------------------------- host-side combinatorial step (a10) */

/* gcd/project_utils/cluster_utils.py:234-275 linear_assignment (called from local_utils/clip_lang_util.py:178):
 * Kuhn-Munkres on a HOST int64 cost matrix [n_rows,n_cols] with that implementation's tie-breaking.
 * out_pairs: HOST buffer of 2*min(n_rows,n_cols) int64, (row,col) pairs sorted by (row,col). */
SCD_API int scd_linear_assignment(const int64_t* cost, int n_rows, int n_cols, int64_t* out_pairs, int* n_pairs);

#ifdef __cplusplus
}
#endif
#endif /* SCD_B200_H_ */
