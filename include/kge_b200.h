/*
 * kge_b200.h -- C ABI of the B200-native KGE hot path (libkge_b200.so).
 *
 * Drop-in boundary for tail-unica/hopwise's knowledge-graph-embedding recommenders
 * (TransE / DistMult / RotatE / ComplEx).  The reference has no FFI of its own (it is
 * pure Python on torch); each entry point below names the reference Python interface it
 * replaces (paths relative to /root/reference/hopwise/).  INTEGRATION.md shows the ctypes
 * binding a hopwise maintainer would add.
 *
 * Conventions
 *   - every pointer is DEVICE memory owned by the caller (torch tensors) unless a
 *     parameter is documented "host"; the library allocates nothing persistent;
 *   - all ids are int64 (torch.long), all embedding data fp32, row-major [rows, d];
 *   - every call is asynchronous on the given cudaStream_t (passed as void*);
 *   - return value: 0 = ok, >0 = cudaError_t, <0 = KGE_E_* argument error;
 *     kge_last_error() gives a thread-local message.  No exceptions cross the ABI;
 *   - re-entrant, no global state; one process per GPU.
 */
#ifndef KGE_B200_H
#define KGE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KGE_ABI_VERSION 8

typedef void* kge_stream_t; /* cudaStream_t */

/* KGE_TORUSE (toruse.py): trains exactly like TransE (TripletMarginLoss on h + r, toruse.py:81-102: the train-step
 * kernels take it as KGE_TRANSE) and scores on the torus: -4 * sum(min(x^2, 1 - x^2)), x = frac(h) + frac(r) - frac(t)
 * (toruse.py:66-76, 131-172).  Not a contraction: CUDA-core scoring paths only.
 * KGE_TRANSH (transh.py): TransE on rows projected per relation.  The relation table has two parts, the translation
 * r and the hyperplane vector w (`norm_vec`); the reference's project() is ent - (ent * sum(w)) * w (transh.py:73-74:
 * the SUM of w's components, not <ent, w>), i.e. ent * (1 - sum(w) * w) element-wise, applied to head and both tails
 * before TransE's TripletMarginLoss / norm (transh.py:53-58, 76-107).  Recommendation triples take row
 * `ui_relation` of both parts.  TRAIN STEP ONLY: scoring (predict and full-sort over items, transh.py:109-145; the
 * reference has no KG scoring entry points for this model) goes through kge_transh_project, which writes projected
 * rows, and the KGE_TRANSE scoring entry points on those.
 * KGE_TRANSD (transd.py): every table has two parts, the embedding and a transfer vector; an entity e with transfer
 * vector e_p is projected with the relation's r_p as e + r_p * <e, e_p> (transd.py:86-91) before TransE's
 * TripletMarginLoss (transd.py:93-133).  TRAIN STEP ONLY: scoring goes through kge_transd_project, which writes
 * projected rows, and the KGE_TRANSE scoring entry points on those (the projection of an item does not depend on the
 * user, so full-sort over items is TransE over a projected table).
 * The scoring entry points refuse KGE_TRANSH and KGE_TRANSD with KGE_E_UNSUPPORTED. */
enum kge_model_kind {
  KGE_TRANSE = 0, KGE_DISTMULT = 1, KGE_ROTATE = 2, KGE_COMPLEX = 3, KGE_TORUSE = 4, KGE_TRANSH = 5, KGE_TRANSD = 6
};

enum kge_error {
  KGE_E_ARG = -1,         /* null pointer / negative size */
  KGE_E_UNSUPPORTED = -2, /* embedding_size or k outside the compiled range */
  KGE_E_STATE = -3        /* optimiser state missing for a call that needs it */
};

/* One family of embedding tables (user / entity / relation): `parts` fp32 matrices
 * [rows, d] (1 = real models, 2 = re/im) plus the row-lazy Adam state that rides with it.
 * m, v, g and row_state may be NULL for an inference-only model. */
typedef struct {
  int64_t rows;
  int32_t parts;
  int32_t _pad;
  float* w[2];        /* parameters: nn.Embedding.weight.data_ptr() */
  float* m[2];        /* Adam exp_avg */
  float* v[2];        /* Adam exp_avg_sq */
  float* g[2];        /* gradient accumulators; all-zero between steps (invariant) */
  int32_t* row_state; /* [rows][2]: {last_step, touch_step}.  last_step = optimiser step the stored
                         (w, m, v) are current for (-1 = never updated); touch_step = last step whose
                         gradient touched the row (-1 = none / taken).  Initialise to -1. */
} kge_table_t;

typedef struct {
  int32_t model;                /* enum kge_model_kind */
  int32_t d;                    /* embedding_size, 1 .. 1024 on every entry point */
  float margin;                 /* TransE / DistMult / RotatE */
  int32_t ui_relation;          /* relation row for user->item triples in loss / predict
                                   (transe.py:63, distmult.py:57: weight[-1]; rotate.py:43,
                                   complex.py:38: the [UI-Relation] token id) */
  int32_t ui_relation_fullsort; /* row used by full_sort_predict (complex.py:168-169 takes weight[-1]) */
  int32_t _pad;
  int64_t n_items;              /* items are entity rows [0, n_items) (kg_dataset.py:556-588) */
  kge_table_t user, entity, relation;
  const float* adam_table;      /* [2*adam_table_len]: {lr/(1-b1^j), 1/sqrt(1-b2^j)} for j = 0..len-1 */
  int32_t adam_table_len;
  int32_t _pad2;
} kge_model_t;

/* One training batch, the fields Interaction carries into calculate_loss
 * (transe.py:75-87).  neg_* hold k negatives per positive in the reference's j-major
 * layout out[j*n + i] (sampler.py:146-153); k = 1 is what the reference's loaders produce
 * for KG triples (knowledge_dataloader.py:51). */
typedef struct {
  const int64_t* user;
  const int64_t* item;
  const int64_t* neg_item;
  int64_t n_rec;
  const int64_t* head;
  const int64_t* relation;
  const int64_t* tail;
  const int64_t* neg_tail;
  int64_t n_kg;
  int32_t k_rec;
  int32_t k_kg;
} kge_batch_t;

/* torch.optim.Adam hyper-parameters (trainer.py:189-190) + the step about to be applied. */
/* The optimiser hopwise's trainer builds (trainer/trainer.py:165-206), applied to the touched rows:
 *   KGE_OPT_ADAM     torch.optim.Adam(lr) (also AdamW with weight_decay 0): beta1, beta2, eps; rows that skipped steps
 *                    are caught up with the zero-gradient steps dense Adam gives them
 *   KGE_OPT_SGD      torch.optim.SGD(lr): p -= lr * g
 *   KGE_OPT_ADAGRAD  torch.optim.Adagrad(lr): v += g^2; p -= lr * g / (sqrt(v) + eps)          (eps 1e-10)
 *   KGE_OPT_RMSPROP  torch.optim.RMSprop(lr): v = beta2 * v + (1 - beta2) * g^2; p -= lr * g / (sqrt(v) + eps)
 *                    (beta2 = alpha 0.99, eps 1e-8; v of a row that skipped n steps decays by alpha^n)
 * Under the last three a row without a gradient does not move, so nothing is replayed. */
enum kge_optimizer { KGE_OPT_ADAM = 0, KGE_OPT_SGD = 1, KGE_OPT_ADAGRAD = 2, KGE_OPT_RMSPROP = 3 };

typedef struct {
  float lr, beta1, beta2, eps;
  int32_t step;       /* 1-based index of the update this batch produces */
  int32_t replay_cap; /* zero-gradient steps replayed exactly per row before the closed-form tail */
  int32_t optimizer;  /* enum kge_optimizer */
  int32_t reserved;
} kge_adam_t;

int kge_abi_version(void);
const char* kge_last_error(void);

/* host: fill `out[2*len]` with the Adam bias-correction table; returns the length needed
 * for (beta1, beta2) when out == NULL. */
int kge_adam_table_fill(float lr, float beta1, float beta2, float* out_host, int32_t len);

/* ---- training ------------------------------------------------------------------------
 * kge_train_forward: replaces <Model>.calculate_loss (transe.py:75-98, distmult.py:68-95,
 * rotate.py:98-131, complex.py:95-128) AND the autograd backward of it
 * (trainer.py:261): gathers rows (catching lazily-updated rows up to step-1 on the fly),
 * scores, adds the scalar loss into *loss_out (caller zeroes it), and when with_grad != 0
 * accumulates analytic gradients into table.g and marks the touched rows in row_state. */
int kge_train_forward(const kge_model_t* model, const kge_batch_t* batch, const kge_adam_t* adam,
                      int with_grad, float* loss_out, kge_stream_t stream);

/* kge_adam_apply: replaces optimizer.step() (trainer.py:264, torch.optim.Adam) for the rows
 * touched by the accumulated gradient: replays the skipped zero-gradient steps of each row,
 * applies step `adam->step` with gradient g * grad_scale * (*grad_scale_dev), zeroes g.
 * grad_scale_dev (device, may be NULL) is the incoming gradient of the scalar loss, so that
 * loss.backward() needs no host synchronisation.  Untouched rows are caught up later (next
 * touch or kge_adam_flush), which is exactly dense Adam's trajectory. */
int kge_adam_apply(const kge_model_t* model, const kge_adam_t* adam, float grad_scale, const float* grad_scale_dev,
                   kge_stream_t stream);

/* Bring every row of every table to step `adam->step` (dense pass).  Must run before
 * weights are read by anything but this library (state_dict, predict, checkpoints). */
int kge_adam_flush(const kge_model_t* model, const kge_adam_t* adam, kge_stream_t stream);

/* kge_train_step: one whole optimisation step in one call -- kge_train_forward (with_grad) followed by
 * kge_adam_apply on the same stream: what optimizer.zero_grad(); loss = model.calculate_loss(batch);
 * loss.backward(); optimizer.step() amount to (trainer/trainer.py:247-266) on one GPU.  *loss_out must be
 * zero on entry. */
int kge_train_step(const kge_model_t* model, const kge_batch_t* batch, const kge_adam_t* adam, float grad_scale,
                   float* loss_out, kge_stream_t stream);

/* Drop a gradient that was accumulated but will not be applied. */
int kge_grad_discard(const kge_model_t* model, int32_t step, kge_stream_t stream);

/* Row-sparse gradient exchange (replaces DDP's dense all-reduce, trainer.py:82-112).
 * pack: compact this rank's touched rows of table `which` (0 user, 1 entity, 2 relation) into
 *       ids_out[count] / rows_out[count, parts*d] (order unspecified), zero them in g and clear
 *       their touch marks; *count_out (device) receives the count.  The outputs must hold
 *       min(rows, rows the batch can touch) entries.
 * add:  add a (possibly remote) packed list (unique ids) into g and mark the rows touched. */
int kge_grad_pack(const kge_model_t* model, int32_t which, int32_t step, int64_t* ids_out, float* rows_out,
                  int32_t* count_out, kge_stream_t stream);
int kge_grad_add(const kge_model_t* model, int32_t which, int32_t step, const int64_t* ids, const float* rows,
                 const int32_t* count_dev, int64_t max_count, kge_stream_t stream);

/* Host -> device staging of a batch's id vectors (replaces the blocking interaction.to(device) of
 * trainer/trainer.py:250-256): cudaMemcpyAsync from (pinned) host memory on the given copy stream. */
int kge_copy_h2d_async(void* dst_device, const void* src_host, int64_t nbytes, kge_stream_t stream);

/* Dense route of the same exchange, in the NVSwitch: sum the N ranks' copies of a symmetric buffer in place.
 * multicast_ptr = the NVLS multicast address of the buffer (16-byte aligned; n_floats % 4 == 0), i.e. one
 * address that names every rank's copy.  Rank `rank` reduces the rank-th slice with multimem.ld_reduce and
 * broadcasts the sums with multimem.st, so every copy ends up holding identical sums.  The caller puts a
 * cross-rank barrier before (all copies written) and after (all slices reduced) the call. */
int kge_multimem_all_reduce_f32(void* multicast_ptr, int64_t n_floats, int32_t rank, int32_t world,
                                kge_stream_t stream);
/* The same reduction with both cross-rank barriers and the touch marks inside one kernel (no host-launched barrier
 * rounds): signal_pads_dev = device array of `world` pointers to the ranks' symmetric signal pads (uint32 slots,
 * zero between calls; slots [slot_base, slot_base + 2*world) are used), local_flags = two zeroed uint32 in local
 * device memory, epoch = a non-zero value that differs from the previous call's.  row_state / n_mark_rows / step:
 * rows [0, n_mark_rows) of the {last_step, touch_step} array get touch_step = step (0 rows: nothing).  On return of
 * the kernel on `stream` every copy of the buffer holds the sums. */
int kge_multimem_all_reduce_fused_f32(void* multicast_ptr, int64_t n_floats, int32_t rank, int32_t world,
                                      void* const* signal_pads_dev, int32_t slot_base, uint32_t* local_flags,
                                      uint32_t epoch, int32_t* row_state, int64_t n_mark_rows, int32_t step,
                                      kge_stream_t stream);

/* kge_owner_adam_step: the optimiser step of a data-parallel job in ONE kernel, owner-sharded over the switch
 * (replaces DDP's gradient all-reduce + optimizer.step(), trainer/trainer.py:82-112, 264-266, for replicas whose
 * flat gradient and weight buffers are symmetric allocations with NVLS multicast mappings).  Rank `rank` reads the
 * sum of the `world` gradient copies of its 1/world slice through multimem.ld_reduce, applies torch.optim.Adam's
 * dense update (gradient scaled by grad_scale, bias corrections of adam->step) with its slice of the moments m / v
 * (local buffers in the same flat layout), and multicasts the new weights to every replica; this rank's gradient
 * copy (grad_local) is zeroed behind the kernel, whose closing barrier means every rank is done reading it.  Barriers before (all gradients written) and after (all slices final) run inside the kernel: see
 * kge_multimem_all_reduce_fused_f32 for signal_pads_dev / slot_base / local_flags / epoch. */
int kge_owner_adam_step(void* grad_multicast, float* grad_local, void* weight_multicast, const float* weight_local,
                        float* m, float* v, int64_t n_floats, int32_t rank, int32_t world, const kge_adam_t* adam,
                        float grad_scale,
                        void* const* signal_pads_dev, int32_t slot_base, uint32_t* local_flags, uint32_t epoch,
                        kge_stream_t stream);

/* kge_transd_project: out[i, :] = E[id_i] + RP[rel_i] * <E[id_i], EP[id_i]>  (TransD.forward, transd.py:86-91).
 * ids == NULL: rows 0..n-1 in order; rel_ids == NULL: relation row `rel_row` for every i.  emb / vec: [rows, d]
 * tables of the projected family (user or entity), rel_vec: the relation transfer-vector table. */
int kge_transd_project(const float* emb, const float* vec, const int64_t* ids, int64_t n, int32_t d,
                       const float* rel_vec, const int64_t* rel_ids, int64_t rel_row, float* out,
                       kge_stream_t stream);

/* kge_transh_project: out[i, :] = E[id_i] * (1 - sum(w) * w), w = W[rel_i]  (TransH.project, transh.py:73-74).
 * ids == NULL: rows 0..n-1 in order; rel_ids == NULL: relation row `rel_row` for every i.  TransH scores as
 * KGE_TRANSE over these projected rows (tensor-core path included). */
int kge_transh_project(const float* emb, const int64_t* ids, int64_t n, int32_t d, const float* norm_vec,
                       const int64_t* rel_ids, int64_t rel_row, float* out, kge_stream_t stream);

/* ---- scoring --------------------------------------------------------------------------
 * kge_predict: <Model>.predict / predict_kg (transe.py:100-110,128-137 and twins).
 * heads index the user tables when head_is_user != 0, else the entity tables; rels == NULL
 * means the user->item relation row. */
int kge_predict(const kge_model_t* model, const int64_t* heads, const int64_t* rels, const int64_t* tails,
                int64_t n, int head_is_user, float* out, kge_stream_t stream);

/* kge_full_sort_scores: <Model>.full_sort_predict / full_sort_predict_kg
 * (transe.py:112-126,139-154 and twins): out[n, n_targets] over entity rows [0, n_targets). */
int kge_full_sort_scores(const kge_model_t* model, const int64_t* heads, const int64_t* rels, int64_t n,
                         int head_is_user, int64_t n_targets, float* out, kge_stream_t stream);

/* kge_full_sort_topk: fuses full_sort_predict + the trainer's masking
 * (trainer.py:731-734: column 0 and history -> -inf) + torch.topk (collector.py:177) without
 * materialising [n, n_targets].  History is CSR over the n query rows (hist_off[n+1],
 * hist_items sorted ascending per row; both NULL = no history).  mask_first != 0 masks target 0
 * (the [PAD] item).  Order: score descending, id ascending (masked targets, score -inf, rank
 * last and enter only when a row has fewer than k unmasked targets).
 * Any 1 <= k <= n_targets (k > n_targets: KGE_E_ARG).  Up to k = 128 each row keeps a sorted
 * list in shared memory; above, a buffer of about 2k keys per row and target split in the
 * workspace, so the workspace grows with n * k.
 * Outputs ids_out[n,k] (int64), scores_out[n,k] (fp32, may be NULL).  workspace: device
 * scratch of kge_full_sort_topk_workspace_bytes(model, n, n_targets, k) bytes (-1: unsupported). */
int64_t kge_full_sort_topk_workspace_bytes(const kge_model_t* model, int64_t n, int64_t n_targets, int32_t k);
int kge_full_sort_topk(const kge_model_t* model, const int64_t* heads, const int64_t* rels, int64_t n,
                       int head_is_user, int64_t n_targets, const int64_t* hist_off, const int64_t* hist_items,
                       int mask_first, int32_t k, int64_t* ids_out, float* scores_out, void* workspace,
                       int64_t workspace_bytes, kge_stream_t stream);

/* kge_full_sort_rank_counts: the exact rank of listed targets over the whole masked row, without
 * materialising [n, n_targets] -- what the collector's rec.meanrank branch (collector.py, the sort
 * of every score row and _average_rank) and metrics.py's GAUC read.  Same query and masking
 * arguments as kge_full_sort_topk (rels == NULL: the user->item relation; masked targets score
 * -inf).  The listed targets are CSR over the rows: pos_off[n+1], pos_items sorted ascending per
 * row (duplicates allowed: each copy gets the same counts).  For every entry i of pos_items, over
 * the row's masked scores s and the entry's own masked score s_i:
 *   greater_out[i] = #{targets with s > s_i},  equal_out[i] = #{targets with s == s_i}
 * (the target itself included), so its average rank is greater + (equal + 1) / 2;
 * n_unmasked_out[n] = the row's unmasked targets.  Ids outside [0, n_targets) are counted as
 * masked.  Scores are bit-identical to kge_full_sort_scores / kge_full_sort_topk, counts are exact
 * integers.  workspace: device scratch of kge_full_sort_rank_workspace_bytes(model, n, n_targets,
 * n_pos) bytes with n_pos = pos_off[n]; a smaller one sets every n_unmasked_out to -1. */
int64_t kge_full_sort_rank_workspace_bytes(const kge_model_t* model, int64_t n, int64_t n_targets, int64_t n_pos);
int kge_full_sort_rank_counts(const kge_model_t* model, const int64_t* heads, const int64_t* rels, int64_t n,
                              int head_is_user, int64_t n_targets, const int64_t* hist_off, const int64_t* hist_items,
                              int mask_first, const int64_t* pos_off, const int64_t* pos_items,
                              int64_t* greater_out, int64_t* equal_out, int64_t* n_unmasked_out,
                              void* workspace, int64_t workspace_bytes, kge_stream_t stream);

/* ---- tensor-core full-sort top-k (tcgen05) -------------------------------------------------------
 * Same contract and same results as kge_full_sort_topk (ids and scores are bit-identical: the
 * fp16 tensor-core pass only filters, under a proven error bound; every reported score comes from
 * the fp32 chain), for k <= 32 and parts*d (+3 for the L2 models) <= 256.
 * kge_mma_prepare_targets converts entity rows [0, n_targets) into the tiled, power-of-two-scaled
 * fp16 operand image (128-byte aligned buffer of kge_mma_image_bytes bytes); rebuild it whenever
 * the entity table changes.
 * Rows the filter cannot bound (a candidate list that does not compact, fewer than k unmasked
 * targets, a query the fp16 scaling cannot hold) are recomputed INSIDE the call by the exact
 * kernel of kge_full_sort_topk, gated and sized on the device (no host synchronisation):
 * row_flags[n] (int32, device) = 1 for those rows, *exact_rows (int32, device) = how many.
 * debug_scores: NULL, or [n, ceil(n_targets/128)*128] fp32 receiving the raw tensor-core scores
 * (tests only).  shape: 0 = let the library pick the sweep shape, or 'a' / 'f' / 'c' (tests and
 * experiments; the image depends on it, so pass the same value to all four calls).
 * workspace: 16-byte aligned, kge_full_sort_topk_mma_workspace_bytes bytes. */
int64_t kge_mma_image_bytes(const kge_model_t* model, int64_t n_targets, int32_t shape);
int kge_mma_prepare_targets(const kge_model_t* model, int64_t n_targets, void* image, int64_t image_bytes,
                            int32_t shape, kge_stream_t stream);
int64_t kge_full_sort_topk_mma_workspace_bytes(const kge_model_t* model, int64_t n, int64_t n_targets, int32_t k,
                                               int32_t shape);
int kge_full_sort_topk_mma(const kge_model_t* model, const int64_t* heads, const int64_t* rels, int64_t n,
                           int head_is_user, int64_t n_targets, const void* image, const int64_t* hist_off,
                           const int64_t* hist_items, int mask_first, int32_t k, int64_t* ids_out, float* scores_out,
                           int32_t* row_flags, int32_t* exact_rows, void* workspace, int64_t workspace_bytes,
                           float* debug_scores, int32_t shape, kge_stream_t stream);

/* kge_topk_hits: collector.py:178-183 without the [n, I] pos_matrix: out[n, k+1] int32 =
 * hit flags of ids[n,k] against the positives CSR (pos_off[n+1], pos_items sorted) then pos_len.
 * Any k >= 1. */
int kge_topk_hits(const int64_t* ids, int64_t n, int32_t k, const int64_t* pos_off, const int64_t* pos_items,
                  int32_t* out, kge_stream_t stream);

/* ---- sampled evaluation (uni-N / pop-N) ---------------------------------------------------------------
 * kge_candidate_select: what trainer.py's _neg_sample_batch_eval (torch.full(-inf) + the scatter of the candidate
 * scores) and the collector's rec.topk / rec.meanrank branches read, from the candidate lists alone.  Row r's
 * candidates are entries [cand_off[r], cand_off[r+1]) of scores / cand_items (cand_off[0] = 0, non-decreasing, ending
 * at n_cand; offsets are clamped to [0, n_cand]); ids lie in [0, n_targets) and may repeat (a repeated id carries the
 * same score and counts once); every other target of the row scores -inf.  Every output may be NULL:
 *   ids_out[n,k] (int64) / scores_out[n,k]: the row's distinct candidates by (score desc, id asc); a row with fewer
 *     than k of them is padded with the smallest non-candidate ids, ascending, score -inf (full-sort's order for
 *     masked targets);
 *   greater_out / equal_out (both or neither): for every entry of the positives CSR (pos_off[n+1], pos_items), the
 *     counts of kge_full_sort_rank_counts over the row: a positive that is not a candidate scores -inf, so
 *     greater = the distinct candidates and equal = n_targets - the distinct candidates;
 *   n_unmasked_out[n]: the row's distinct candidates.
 * Rows pick a warp, a CTA or the workspace to sort in on the device, by length.  1 <= k <= n_targets < 2^32 - 1.
 * workspace: kge_candidate_select_workspace_bytes(n, n_cand) bytes. */
int64_t kge_candidate_select_workspace_bytes(int64_t n, int64_t n_cand);
int kge_candidate_select(const float* scores, const int64_t* cand_items, int64_t n_cand, const int64_t* cand_off,
                         int64_t n, int64_t n_targets, const int64_t* pos_off, const int64_t* pos_items, int32_t k,
                         int64_t* ids_out, float* scores_out, int64_t* greater_out, int64_t* equal_out,
                         int64_t* n_unmasked_out, void* workspace, int64_t workspace_bytes, kge_stream_t stream);

/* kge_topk_metric_sums: metrics.py:67-69,93-101,164-165,191-207,231-232 summed over users:
 * sums[5*k] float64 = per-cutoff sums of recall, mrr, ndcg, hit, precision (caller zeroes).
 * Any k >= 1. */
int kge_topk_metric_sums(const int32_t* rec_topk, int64_t n, int32_t k, double* sums, kge_stream_t stream);

/* ---- batch assembly ------------------------------------------------------------------------
 * kge_gather_columns: Interaction.__getitem__ on the id columns of a batch (interaction.py:130-139 as called
 * from general_dataloader.py:66-70 and knowledge_dataloader.py:69-75): outs[c][i] = columns[c][index[i]] for
 * n_columns <= 8 int64 columns of `rows` entries in one launch.  columns / outs are HOST arrays of device
 * pointers.  *status (device, may be NULL) becomes 1 when an index lies outside [0, rows). */
int kge_gather_columns(const int64_t* const* columns, int32_t n_columns, int64_t rows, const int64_t* index,
                       int64_t n, int64_t* const* outs, int32_t* status, kge_stream_t stream);

/* kge_assemble_batch: one RSKG training batch in one call (knowledge_dataloader.py:131-145: the KG half first --
 * kg_feat[index] then sample_by_entity_ids --, then general_dataloader.py:66-70 + abstract_dataloader.py:185-198:
 * inter_feat[index] then sample_by_user_ids), both samplers on the one MT19937 stream, uniform candidates.
 * out (device, 4*n_kg + (2 + neg_num)*n_rec int64): head | relation | tail | neg_tail | user | item | neg_item
 * (neg_item j-major).  workspace: kge_assemble_batch_workspace_bytes(...) bytes. */
int64_t kge_assemble_batch_workspace_bytes(int64_t n_kg, int64_t n_rec, int32_t neg_num);
int kge_assemble_batch(uint32_t* mt_state, const int64_t* kg_head, const int64_t* kg_rel, const int64_t* kg_tail,
                       int64_t kg_rows, const int64_t* kg_index, int64_t n_kg, const int64_t* kg_used_off,
                       const int64_t* kg_used_vals, int64_t entity_num, const int64_t* inter_user,
                       const int64_t* inter_item, int64_t inter_rows, const int64_t* rec_index, int64_t n_rec,
                       int32_t neg_num, const int64_t* rec_used_off, const int64_t* rec_used_vals, int64_t item_num,
                       int64_t* out, void* workspace, kge_stream_t stream);

/* kge_widen_ids_i32: dst[i] = src[i] for ids a loader staged as int32 (half the host->device bytes of the int64 id
 * vectors hopwise's Interaction holds, trainer.py:250-256; every id is a row index below 2^31).  16-byte aligned. */
int kge_widen_ids_i32(const int32_t* src, int64_t* dst, int64_t n, kge_stream_t stream);

/* ---- negative sampling -------------------------------------------------------------------
 * kge_sample_negatives: AbstractSampler.sample_by_key_ids with uniform sampling
 * (sampler.py:140-183, 226-227, 315-316) on numpy's MT19937 stream, bit for bit.
 * mt_state[626] (device): 624 key words, pos, status; read and advanced.  status becomes 1
 * (sticky) when some key's forbidden list covers the whole range (the reference raises for
 * that up front, sampler.py:318-336).  used_off[n_keys+1] / used_vals: CSR of sorted forbidden
 * values per key.  out[n*num] int64, j-major.
 * workspace: int32 scratch of kge_sample_workspace_bytes(n*num) bytes. */
int64_t kge_sample_workspace_bytes(int64_t total);
int kge_sample_negatives(uint32_t* mt_state, const int64_t* keys, int64_t n, int32_t num, const int64_t* used_off,
                         const int64_t* used_vals, int64_t low, int64_t high, int64_t* out, void* workspace,
                         kge_stream_t stream);
/* kge_sample_negatives_alias: the same rejection rounds with popularity-biased candidates
 * (sampler.py:68-116: AbstractSampler._build_alias_table / _pop_sampling).  Each round of L open slots
 * consumes np.random.randint(0, pop_n, L) and then np.random.random(L) from the stream; slot j takes
 * pop_keys[idx_j] when pop_prob[idx_j] > p_j, else pop_alias[idx_j].  pop_keys / pop_prob / pop_alias
 * [pop_n] (device): the alias table in the reference's key order (first occurrence in the candidates
 * list), alias stored as the aliased key id (-1 where the reference leaves -1).
 * workspace: kge_sample_alias_workspace_bytes(n*num) bytes. */
int64_t kge_sample_alias_workspace_bytes(int64_t total);
int kge_sample_negatives_alias(uint32_t* mt_state, const int64_t* keys, int64_t n, int32_t num,
                               const int64_t* used_off, const int64_t* used_vals, int64_t pop_n,
                               const int64_t* pop_keys, const double* pop_prob, const int64_t* pop_alias,
                               int64_t* out, void* workspace, kge_stream_t stream);
/* np.random.seed(seed) (legacy init_genrand) into a device state. */
int kge_mt19937_seed(uint32_t* mt_state, uint32_t seed, kge_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* KGE_B200_H */
