/*
 * kge_b200.h -- C ABI of libkge_b200.so: the B200 (sm_100a) implementation of the RotatE toolkit's
 * scoring / loss / backward / Adam / filtered-ranking hot path.
 *
 * The reference (kahrabian/KnowledgeGraphEmbedding) is pure Python and has no FFI of its own; the
 * boundary it exposes is the Python class codes/model.py:22 `KGEModel`.  Each entry point below is
 * what a ctypes binding inside that class would call; the comment on each names the reference lines
 * it replaces.  knowledgegraphembedding_b200/model.py is that binding (see INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name starts with `host_`; the caller owns all memory;
 *   - all tables are row-major fp32, indices are int64 exactly as the reference's LongTensors;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*); nothing is allocated;
 *   - return value 0 = success, negative = error; kge_last_error() gives the message (thread-local);
 *   - no C++ exceptions cross the boundary, no torch types appear in any signature.
 */
#ifndef KGE_B200_H_
#define KGE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KGE_ABI_VERSION 2

/* model.py:151-157 `model_func` keys */
enum { KGE_TRANSE = 0, KGE_DISTMULT = 1, KGE_COMPLEX = 2, KGE_ROTATE = 3, KGE_PROTATE = 4 };
/* model.py:83,104,126 `mode` strings */
enum { KGE_SINGLE = 0, KGE_HEAD_BATCH = 1, KGE_TAIL_BATCH = 2 };
/* model.py:270-279 loss kinds evaluated per positive row */
enum { KGE_LOSS_NEG_ADVERSARIAL = 0, KGE_LOSS_NEG_UNIFORM = 1, KGE_LOSS_POSITIVE = 2 };

enum {
  KGE_OK = 0,
  KGE_ERR_INVALID = -1,      /* bad argument / unsupported shape (maps to ValueError)            */
  KGE_ERR_CUDA = -2,         /* CUDA runtime error                                               */
  KGE_ERR_DEVICE = -3        /* not an sm_100 device                                             */
};

/* State of a KGEModel (model.py:23-70).  Plain struct, lives in host memory. */
typedef struct kge_model {
  int32_t model;             /* KGE_TRANSE ...                                                   */
  int32_t device;            /* CUDA ordinal the pointers live on                                */
  int64_t nentity;           /* model.py:27                                                      */
  int64_t nrelation;         /* model.py:28                                                      */
  int64_t hidden_dim;        /* model.py:29                                                      */
  int64_t entity_dim;        /* model.py:42                                                      */
  int64_t relation_dim;      /* model.py:43                                                      */
  float gamma;               /* model.py:32  gamma.item()                                        */
  float embedding_range;     /* model.py:37  embedding_range.item()                              */
  const float *entity;       /* [nentity, entity_dim]     model.py:45                            */
  const float *relation;     /* [nrelation, relation_dim] model.py:52                            */
  const float *modulus;      /* [1,1] pRotatE only, else NULL (model.py:60)                      */
} kge_model_t;

int kge_abi_version(void);
const char *kge_last_error(void);
/* Refuses anything that is not compute capability 10.x; reports SM count and L2 size. */
int kge_device_check(int device, int *sm_count, int64_t *l2_bytes);

/* ---- scoring: KGEModel.forward (model.py:72-164) + the five score functions (model.py:166-249) ----
 * mode SINGLE:      positive [B,3]; negative ignored; N must be 1; score [B,1]
 * mode HEAD_BATCH:  negative [B,N] are candidate heads; mode TAIL_BATCH: candidate tails.
 * err_flag (device int32, may be NULL) is set to 1 if an index is out of range (the row is then
 * read as id 0 instead of faulting; torch raises an index error at the same place).             */
int kge_score_forward(const kge_model_t *m, int mode, const int64_t *positive, const int64_t *negative,
                      int64_t B, int64_t N, float *score, int32_t *err_flag, void *stream);

/* autograd of the above (what loss.backward() at model.py:301 does through index_select):
 * accumulates d(sum dscore*score)/dE etc. into dense fp32 tables with vector atomics.          */
int kge_score_backward(const kge_model_t *m, int mode, const int64_t *positive, const int64_t *negative,
                       int64_t B, int64_t N, const float *dscore,
                       float *grad_entity, float *grad_relation, float *grad_modulus,
                       void *workspace, int64_t workspace_bytes, int32_t *err_flag, void *stream);

/* ---- fused train pass: model.py:268-288 (scores, self-adversarial / uniform loss) + model.py:301 ----
 * One launch per call: gather+score the N candidates of each positive row, softmax-weighted
 * logsigmoid loss in the same CTA, closed-form backward with vector atomic scatter.
 *   loss_kind NEG_*: candidates = negative[B,N] in `mode`;  POSITIVE: the positive triple itself
 *   weight: subsampling_weight [B_total] or NULL (= --uni_weight);  weight_sum: device scalar sum(weight)
 *   row_begin/row_count: this rank's slice of the batch (row_count == B_total on one GPU)
 *   row_loss [B_total]: per-row  sum_j w_ij logsig(-s_ij)  (NEG) or logsig(s_i) (POSITIVE)
 *   pos_row_loss [B_total] or NULL: with a NEG loss_kind, also run the positive triple of every row (model.py:277-279)
 *                and write logsig(s_i+) here -- fused into the same launch when the single-read path is taken
 *   score_out: optional [row_count, N] copy of the scores (tests), may be NULL
 *   workspace: kge_train_workspace_bytes(m, row_count, N) bytes of device scratch, or NULL        */
int kge_train_rows(const kge_model_t *m, int mode, int loss_kind, float adversarial_temperature,
                   const int64_t *positive, const int64_t *negative, const float *weight,
                   const float *weight_sum, int64_t B_total, int64_t row_begin, int64_t row_count,
                   int64_t N, float *row_loss, float *pos_row_loss, float *grad_entity, float *grad_relation,
                   float *grad_modulus, float *score_out, void *workspace, int64_t workspace_bytes,
                   int32_t *err_flag, void *stream);

/* ---- fused train step for one device: the call above + the Adam update of the entity table (model.py:301-303) ----
 * When kge_train_plan(m, rows, N) reports KGE_PLAN_ENTITY_ADAM, the entity-major half of the backward keeps each
 * entity's summed gradient in registers and applies torch.optim.Adam to the row in place (entity_embedding, exp_avg,
 * exp_avg_sq are updated; *m->entity is WRITTEN despite the const in kge_model_t): the dense entity gradient is never
 * materialised, zeroed or re-read (optimizer.zero_grad() at model.py:259 has nothing to clear for it).  Every entity is
 * updated, also those without a gradient this step (dense Adam semantics).  The relation table (and pRotatE's
 * modulus) keep dense gradients in grad_relation / grad_modulus and go through kge_adam_step as before.
 * With l3_coefficient != 0 the entity share of the L3 regulariser (model.py:290-297) is folded in: 3*l3*x*|x| is added
 * to the gradient and sum|x|^3 of the pre-update values is accumulated into reg_partials (zeroed here).
 * A non-zero *err_flag (bad index in this batch) cancels the update.  The whole batch must be local (row_count == B). */
typedef struct kge_entity_adam {
  float *exp_avg;            /* optimizer.state[entity_embedding]['exp_avg']     [nentity, entity_dim]  */
  float *exp_avg_sq;         /* optimizer.state[entity_embedding]['exp_avg_sq']                         */
  int32_t step;              /* 1-based, after increment (state['step'])                                */
  int32_t reserved;
  double lr, beta1, beta2, eps;
  double l3_coefficient;     /* args.regularization or 0                                                */
  double *reg_partials;      /* device doubles (>= 148 recommended) or NULL when l3_coefficient == 0     */
  int64_t n_reg_partials;
} kge_entity_adam_t;

enum { KGE_PLAN_SINGLE_READ = 1, KGE_PLAN_ENTITY_ADAM = 2 };
/* for `rows` local positive rows x N candidates: SINGLE_READ = kge_train_rows takes the single-read path (a shape AND
 * pair-density decision), ENTITY_ADAM = kge_train_rows_adam is available (shape only; bit mask of KGE_PLAN_*)      */
int kge_train_plan(const kge_model_t *m, int64_t rows, int64_t N);

int kge_train_rows_adam(const kge_model_t *m, int mode, int loss_kind, float adversarial_temperature,
                        const int64_t *positive, const int64_t *negative, const float *weight,
                        const float *weight_sum, int64_t B_total, int64_t row_count, int64_t N, float *row_loss,
                        float *pos_row_loss, float *grad_relation, float *grad_modulus, void *workspace,
                        int64_t workspace_bytes, int32_t *err_flag, const kge_entity_adam_t *host_entity_adam,
                        void *stream);

/* debug (KGE_ROW_PHASES=1): cycles per phase of the persistent row kernel, summed over CTAs, rows and launches:
 * [0] query vector, [1] candidate loop, [2] row loss, [3] fold, [4] chain rule, [5] positive triple, [6] share of [1]
 * spent waiting on the TMA mbarrier (warp 0 of each CTA).                                                          */
int kge_debug_row_phase_cycles(uint64_t *host_out8, int reset);

/* Device scratch for the single-read backward (kge_train_rows / kge_score_backward): per-pair dL/ds, the query
 * table, and the counting-sort arrays of the entity-major pass.  With workspace == NULL (or too small) the
 * two-sweep atomic kernel is used instead; results agree to rounding.                                        */
int64_t kge_train_workspace_bytes(const kge_model_t *m, int64_t rows, int64_t N);

/* Multi-GPU variant of kge_train_rows (negative loss kinds): identical work, but when the single-read path is taken
 * the entity-major pass is left to the caller (*host_entity_pass_pending = 1), who launches it per entity range with
 * kge_train_entity_pass and all-reduces each finished slice of grad_entity while the next range is computed.         */
int kge_train_rows_begin(const kge_model_t *m, int mode, int loss_kind, float adversarial_temperature,
                         const int64_t *positive, const int64_t *negative, const float *weight,
                         const float *weight_sum, int64_t B_total, int64_t row_begin, int64_t row_count, int64_t N,
                         float *row_loss, float *pos_row_loss, float *grad_entity, float *grad_relation,
                         float *grad_modulus, void *workspace, int64_t workspace_bytes, int32_t *err_flag,
                         int32_t *host_entity_pass_pending, void *stream);
int kge_train_entity_pass(const kge_model_t *m, int mode, void *workspace, int64_t row_count, int64_t N,
                          int64_t ent_begin, int64_t ent_end, int slice_index, float *grad_entity,
                          float *grad_modulus, void *stream);

/* cudaMemsetAsync(ptr, 0, bytes): clears the gradient workspace at the top of a train step (the
 * reference's optimizer.zero_grad() at model.py:259 drops the grads, autograd re-creates zero tables). */
int kge_zero(void *ptr, int64_t bytes, void *stream);

/* model.py:263-266 (`positive_sample.cuda()` ...) and :305-310 (`.item()`): stage a host batch on the device and read the
 * loss block back.  host_* are HOST pointers; pinned memory makes the H2D copy asynchronous on `stream`.              */
int kge_copy_h2d(void *dst_device, const void *host_src, int64_t bytes, void *stream);
int kge_copy_d2h_sync(void *host_dst, const void *src_device, int64_t bytes, void *stream);

/* deterministic sum of weight[0..B) into out[0] (model.py:285 `subsampling_weight.sum()`)         */
int kge_weight_sum(const float *weight, int64_t B, float *out, void *stream);

/* model.py:281-288 + 296: out[0]=positive_sample_loss out[1]=negative_sample_loss out[2]=loss
 * out[3]=regularization, from the per-row values; reg_partials (may be NULL) are the block sums of
 * |x|^3 written by kge_adam_step.                                                                */
int kge_loss_finalize(const float *pos_row, const float *neg_row, const float *weight,
                      const float *weight_sum, int64_t B, float regularization,
                      const double *reg_partials, int64_t n_reg_partials, float *out, void *stream);

/* ---- optimizer: torch.optim.Adam.step() as called at model.py:303 (defaults of run.py:266-269) ----
 * Dense fused update of up to 4 tensors in one launch.  l3 != 0 adds the gradient of the L3
 * regulariser (model.py:290-296), 3*l3*x*|x|, to `grad` (written back) and accumulates sum|x|^3
 * of the pre-update values into reg_partials[gridDim] (doubles).                                 */
typedef struct kge_adam_tensor {
  float *param; float *grad; float *exp_avg; float *exp_avg_sq;
  int64_t numel;
  int32_t step;              /* 1-based, after increment (state['step'])                         */
  int32_t l3;                /* 1: this tensor takes part in the L3 regulariser                  */
} kge_adam_tensor_t;

int kge_adam_step(const kge_adam_tensor_t *host_tensors, int n_tensors, double lr, double beta1,
                  double beta2, double eps, double l3_coefficient, double *reg_partials,
                  int64_t n_reg_partials, const int32_t *skip_flag, void *stream);
/* sum |x|^3 of the tensors flagged l3 into reg_partials (block sums, doubles): the VALUE of the L3 regulariser when the
 * update runs through kge_peer_reduce_adam, which applies the L3 gradient itself (only `param`, `numel`, `l3` are read) */
int kge_l3_partials(const kge_adam_tensor_t *host_tensors, int n_tensors, double *reg_partials,
                    int64_t n_reg_partials, void *stream);

/* ---- filtered ranking: KGEModel.test_step (model.py:346-427) with dataloader.py:134-154's filter ----
 * Step 1: per query the fixed side is folded into a query vector (model.py:214-223 etc.)
 *   queries [Q,3] int64 triples, mode HEAD_BATCH/TAIL_BATCH; qvec [Q, entity_dim]
 * pRotatE additionally needs the phase table  entity / (rho/pi)  [nentity, entity_dim] (model.py:236-238). */
int kge_eval_query_vectors(const kge_model_t *m, int mode, const int64_t *queries, int64_t Q,
                           float *qvec, int32_t *err_flag, void *stream);
int kge_eval_phase_table(const kge_model_t *m, float *phase_table, void *stream);

/* Step 2: score of the positive column, bit-identical to what step 3 computes for that column.   */
int kge_eval_positive_scores(const kge_model_t *m, int mode, const float *qvec, const int64_t *queries,
                             int64_t Q, const float *phase_table, float *pos_score, void *stream);

/* Step 3: fused all-entity scoring + filter + count.  For each query q and each entity j in
 * [ent_begin, ent_end):   counts[q] += !filtered(q,j) && j != pos(q) &&
 *                                       (s(q,j) > s_pos(q) || (s(q,j) == s_pos(q) && j < pos(q)))
 * so that rank = 1 + sum over entity shards of counts (model.py:396-411 with a stable descending sort).
 *   filter_bits [Q, ceil(nentity/32)] uint32 bitmap of the filtered columns (dataloader.py:138-144)
 *   scores_out: optional [Q, nentity] dump of s(q,j) + filter_bias (tests), may be NULL           */
int kge_eval_count_ranks(const kge_model_t *m, int mode, const float *qvec, const int64_t *queries,
                         int64_t Q, const float *phase_table, const float *pos_score,
                         const uint32_t *filter_bits, int64_t ent_begin, int64_t ent_end,
                         int32_t *counts, float *scores_out, void *stream);

/* Two-stage variant of step 3 (RotatE, pRotatE): a fast tile pass (RotatE: approximate sqrt, free association, packed
 * FP32; pRotatE: reduction by pi + one sin.approx instead of the reproducible polynomial sine) counts every candidate
 * whose order against the positive is certain under a proven error band; the few undecidable (q, j) pairs are
 * re-scored with the exact op sequence.  Counts are identical to kge_eval_count_ranks.  Models without a fast
 * variant run the exact kernel.  amb_count[1] = 1 reports an overflow of amb_pairs (caller re-runs exact).       */
int kge_eval_count_ranks_two_stage(const kge_model_t *m, int mode, const float *qvec, const int64_t *queries,
                                   int64_t Q, const float *phase_table, const float *pos_score,
                                   const uint32_t *filter_bits, int64_t ent_begin, int64_t ent_end,
                                   int32_t *counts, void *amb_pairs, int64_t amb_capacity, int32_t *amb_count,
                                   void *stream);
/* The same, and approx_scores_out (tests, may be NULL): [Q, nentity] dump, for the entities in [ent_begin, ent_end), of the
 * score each pair was decided on -- the fast pass's approximation (a filtered column as s_pos - 1; NaN where the pRotatE
 * pass gives up), or the exact score where the exact kernel runs instead (no fast variant, d > 2048, unaligned rows).
 * A fast pass zeroes amb_count; the exact kernel leaves it untouched.                                              */
int kge_eval_count_ranks_two_stage_approx(const kge_model_t *m, int mode, const float *qvec, const int64_t *queries,
                                          int64_t Q, const float *phase_table, const float *pos_score,
                                          const uint32_t *filter_bits, int64_t ent_begin, int64_t ent_end,
                                          int32_t *counts, void *amb_pairs, int64_t amb_capacity, int32_t *amb_count,
                                          float *approx_scores_out, void *stream);
/* The band of the fast pass (what the band test in tests/ pins): |approx - canonical| <= eps(approx) =
 * host_band[0] + host_band[1] * |gamma - approx| + host_band[2] * |approx| for `model` (KGE_ROTATE / KGE_PROTATE), its
 * entity_dim and (pRotatE) modulus.  KGE_ERR_INVALID for a model or entity_dim without a fast pass.               */
int kge_eval_two_stage_band(int model, int64_t entity_dim, float modulus, float *host_band);

/* ---- tcgen05 path for the dot-product models (DistMult model.py:175-182, ComplEx :184-199) in test_step ----
 * The all-entity scores are one [Q, D_e] x [D_e, nentity] contraction.  Operands are split into two TF32-exact
 * pieces (kge_eval_gemm_split: hi, lo and the row norms), a tcgen05.mma kind::tf32 kernel accumulates
 * hi*hi + hi*lo + lo*hi in tensor memory, and its epilogue counts only the candidates whose order against the
 * positive is certain under a rigorous error band; the ambiguous (q, j) pairs go to amb_pairs and are re-scored
 * with the exact op sequence of kge_eval_count_ranks, so counts are identical to that kernel's.
 * amb_count[0] = pairs appended, amb_count[1] = 1 if amb_capacity overflowed (caller falls back to
 * kge_eval_count_ranks for that chunk).  ent_begin must be a multiple of 32.                                 */
int kge_eval_gemm_supported(const kge_model_t *m);
int kge_eval_gemm_split(const float *x, int64_t rows, int64_t cols, float *hi, float *lo, float *norm, void *stream);
int kge_eval_gemm_count_ranks(const kge_model_t *m, int mode, const float *qvec, const float *qhi, const float *qlo,
                              const float *qnorm, const int64_t *queries, int64_t Q, const float *pos_score,
                              const uint32_t *filter_bits, const float *ehi, const float *elo, const float *enorm,
                              int64_t ent_begin, int64_t ent_end, int32_t *counts, void *amb_pairs,
                              int64_t amb_capacity, int32_t *amb_count, float *approx_scores_out, void *stream);
/* band(K): the relative half-width the kernel above uses, |approx - canonical| <= band * |q| * |E_j| (what the band
 * test in tests/ pins against measured tensor-core errors); approx_scores_out (tests, may be NULL): [Q, nentity] dump
 * of the tensor-core approximations for the entities in [ent_begin, ent_end).                                    */
float kge_eval_gemm_band(int64_t entity_dim);

/* ---- rank statistics: raw and tie-aware ranks from the same passes ----
 * The three step-3 entries above, counting KGE_RANK_STATS int32 counters per query instead of one:
 * stats [Q, KGE_RANK_STATS], zeroed by the caller; for the entities j != pos(q) in [ent_begin, ent_end), with s the
 * canonical score of kge_eval_count_ranks (a filtered column keeps its own score here) and "filtered" read from
 * filter_bits:
 *   [0] !filtered && s > s_pos            [3] s > s_pos
 *   [1] !filtered && s == s_pos && j < pos  [4] s == s_pos && j < pos
 *   [2] !filtered && s == s_pos && j > pos  [5] s == s_pos && j > pos
 * NaN is never greater or equal, -0.0 == +0.0, and the counters add up over entity slices.  1 + [0] + [1] is the rank of
 * kge_eval_count_ranks whenever fl(s_pos - 1) < s_pos (the filter bias of that rank); 1 + [3] + [4] is the raw rank.
 * The two-stage and tcgen05 variants take the argument rules of their count entries (amb_count[1] = 1: overflow, the
 * caller re-runs kge_eval_count_rank_stats for that chunk; ent_begin a multiple of 32 on tcgen05).              */
#define KGE_RANK_STATS 6
int kge_eval_count_rank_stats(const kge_model_t *m, int mode, const float *qvec, const int64_t *queries, int64_t Q,
                              const float *phase_table, const float *pos_score, const uint32_t *filter_bits,
                              int64_t ent_begin, int64_t ent_end, int32_t *stats, void *stream);
int kge_eval_count_rank_stats_two_stage(const kge_model_t *m, int mode, const float *qvec, const int64_t *queries,
                                        int64_t Q, const float *phase_table, const float *pos_score,
                                        const uint32_t *filter_bits, int64_t ent_begin, int64_t ent_end, int32_t *stats,
                                        void *amb_pairs, int64_t amb_capacity, int32_t *amb_count, void *stream);
int kge_eval_gemm_count_rank_stats(const kge_model_t *m, int mode, const float *qvec, const float *qhi,
                                   const float *qlo, const float *qnorm, const int64_t *queries, int64_t Q,
                                   const float *pos_score, const uint32_t *filter_bits, const float *ehi,
                                   const float *elo, const float *enorm, int64_t ent_begin, int64_t ent_end,
                                   int32_t *stats, void *amb_pairs, int64_t amb_capacity, int32_t *amb_count,
                                   void *stream);

/* ---- candidate-list ranking: each query against its own list of entities (sampled evaluation, OGB-style) ----
 * candidates [Q, ld] int64 entity ids of the predicted slot; -1 is padding (anywhere in a row); any other id outside
 * [0, nentity) sets *err_flag and counts nothing.  For the listed entries j in columns [col_begin, col_end) with
 * j != pos(q), counted as often as they are listed, stats [Q, KGE_RANK_STATS] (zeroed by the caller) receives the
 * counters of kge_eval_count_rank_stats, "filtered" read from filter_bits ([Q, ceil(nentity/32)], or NULL: nothing is
 * filtered).  s is the canonical score of kge_eval_count_ranks (bit-identical).  qvec and pos_score come from
 * kge_eval_query_vectors and kge_eval_positive_scores; pRotatE also needs kge_eval_phase_table.  The counters add up
 * over column slices.  scores_out [Q, ld] (may be NULL) receives the scores of the slice's columns: s for a listed
 * entity, s_pos where it names the positive, -inf at padding.  At most 65535*128 columns per slice.                 */
int kge_eval_candidate_rank_stats(const kge_model_t *m, int mode, const float *qvec, const int64_t *queries,
                                  int64_t Q, const float *phase_table, const float *pos_score,
                                  const int64_t *candidates, int64_t ld, int64_t col_begin, int64_t col_end,
                                  const uint32_t *filter_bits, int32_t *stats, float *scores_out, int32_t *err_flag,
                                  void *stream);

/* filter bitmap from a CSR of true entities per query (dataloader.py:138-144)                     */
int kge_eval_filter_bits(const int64_t *csr_offsets, const int32_t *csr_entities, int64_t Q,
                         int64_t nentity, uint32_t *filter_bits, void *stream);

/* Same bitmap without a host round trip per query chunk: the index of all true triples lives on the device as a
 * sorted-key CSR (built once per all_true_triples list: keys = r*nentity+t -> true heads for HEAD_BATCH,
 * h*nrelation+r -> true tails for TAIL_BATCH; run i is index_entities[index_offsets[i] .. index_offsets[i+1])),
 * and each query's key is looked up on the device.  Replaces TestDataset.__getitem__'s per-entity set probes
 * (dataloader.py:134-154) for a whole chunk of queries in one launch.                                          */
int kge_eval_filter_bits_lookup(const int64_t *index_keys, const int64_t *index_offsets, const int32_t *index_entities,
                                int64_t nkeys, const int64_t *queries, int64_t Q, int mode, int64_t nentity,
                                int64_t nrelation, uint32_t *filter_bits, void *stream);

/* The index itself built on the device (dataloader.py:122-162 builds the python set of all true triples; the host-side
 * FilterIndex sorts them with numpy): a direct-address CSR over the key space nentity*nrelation (< 2^31) by counting
 * sort -- histogram of the keys, tiled scan, scatter.  triples [ntriples,3] int64 on the device; offsets
 * [nentity*nrelation + 1] int32 and entities [ntriples] int32 are the result (run of key k = entities[offsets[k] ..
 * offsets[k+1]), order inside a run unspecified); scratch: kge_eval_filter_index_scratch_bytes().  A triple with an id
 * outside the tables sets *err_flag and is skipped.  kge_eval_filter_bits_lookup_dense is the lookup for this layout
 * (one load pair per query instead of a binary search).                                                        */
int64_t kge_eval_filter_index_scratch_bytes(int64_t nentity, int64_t nrelation);
int kge_eval_filter_index_build(const int64_t *triples, int64_t ntriples, int mode, int64_t nentity, int64_t nrelation,
                                int32_t *offsets, int32_t *entities, void *scratch, int64_t scratch_bytes,
                                int32_t *err_flag, void *stream);
int kge_eval_filter_bits_lookup_dense(const int32_t *index_offsets, const int32_t *index_entities,
                                      const int64_t *queries, int64_t Q, int mode, int64_t nentity, int64_t nrelation,
                                      uint32_t *filter_bits, void *stream);

/* ---- path queries (a, r1/.../rL, ?) and (?, r1/.../rL, a): multi-hop questions ranked by the one-hop kernels ----
 * anchors [Q] int64 entity ids; paths [Q, L] int64 hop ids: r in [0, nrelation) follows relation r, r + nrelation follows
 * it inverted, -1 pads a row after its last hop (every row has at least one hop).
 * kge_eval_path_query_vectors: qvec [Q, entity_dim], the path folded into one query vector with the non-contracted
 *   primitives of kge_eval_query_vectors (tail-batch: row(a) through hops 1..L; head-batch: from row(a), -row(a) for
 *   TransE and pRotatE, through hops L..1), so that a one-hop forward path gives that call's vector bit for bit.  It feeds
 *   kge_eval_positive_scores, the count / stats entries and kge_eval_topk as a query vector of `mode`.  A bad anchor, hop
 *   id or padding sets *err_flag (may be NULL) and folds a zero row.
 * kge_eval_path_bits_dense / kge_eval_path_bits: bits [Q, ceil(nentity/32)] = the entities reachable from the anchor along
 *   the path in the indexed triples (tail-batch: forward along hops 1..L; head-batch: backward from hop L), in the
 *   filter_bits layout, by one traversal launch per hop over the bitmaps bits and pong (same size, distinct).  The tail
 *   index ((h, r) -> tails, TAIL_BATCH build of kge_eval_filter_index_build or kge_eval_filter_bits_lookup's table) serves
 *   forward tail-batch hops and inverse head-batch hops, the head index ((r, t) -> heads) the other two; an index may be
 *   NULL (nkeys 0) when no hop of the call reads it.  answer_counts [Q] int32 (may be NULL): the size of each set.     */
int kge_eval_path_query_vectors(const kge_model_t *m, int mode, const int64_t *anchors, const int64_t *paths, int64_t Q,
                                int64_t L, float *qvec, int32_t *err_flag, void *stream);
int kge_eval_path_bits_dense(const int32_t *tail_offsets, const int32_t *tail_entities, const int32_t *head_offsets,
                             const int32_t *head_entities, const int64_t *anchors, const int64_t *paths, int64_t Q,
                             int64_t L, int mode, int64_t nentity, int64_t nrelation, uint32_t *bits, uint32_t *pong,
                             int32_t *answer_counts, void *stream);
int kge_eval_path_bits(const int64_t *tail_keys, const int64_t *tail_offsets, const int32_t *tail_entities,
                       int64_t tail_nkeys, const int64_t *head_keys, const int64_t *head_offsets,
                       const int32_t *head_entities, int64_t head_nkeys, const int64_t *anchors, const int64_t *paths,
                       int64_t Q, int64_t L, int mode, int64_t nentity, int64_t nrelation, uint32_t *bits, uint32_t *pong,
                       int32_t *answer_counts, void *stream);

/* ---- top-k link prediction: the k most plausible entities of every query (h, r, ?) / (?, r, t) ----
 * Scores are the canonical exact ones of kge_eval_count_ranks (bit-identical to that kernel and to the C oracle) for
 * every model; the [Q, nentity] score matrix is never formed.  Order: score descending, then entity id ascending; NaN
 * after every number; -0.0 == +0.0.  Results travel as uint64 keys (orderable(score) << 32) | (0xFFFFFFFF - id), so a
 * larger key is a better candidate; key 0 is an empty slot (id -1, score -inf when decoded).
 * kge_eval_topk: the k best entities in [ent_begin, ent_end) of each query vector (kge_eval_query_vectors; pRotatE also
 *   needs the phase table) that are not set in exclude_bits ([Q, ceil(nentity/32)] uint32, the filter_bits layout; may
 *   be NULL).  keys_out [Q, k] sorted best first.  scratch: kge_eval_topk_scratch_bytes() (0 or more; a negative value
 *   is an error code).  At most 65535*64 queries per call.
 * kge_eval_topk_merge: the k best of `lists` sorted key lists per query, keys_in [Q, lists, k] (entity shards of several
 *   devices, say), as keys_out [Q, k] and / or decoded ids_out int64 [Q, k] and scores_out float [Q, k]; each output
 *   may be NULL.  Keys of one query must be distinct (disjoint entity ranges).                                       */
#define KGE_TOPK_MAX 256
int64_t kge_eval_topk_scratch_bytes(const kge_model_t *m, int64_t Q, int64_t ent_begin, int64_t ent_end, int k);
int kge_eval_topk(const kge_model_t *m, int mode, const float *qvec, int64_t Q, const float *phase_table,
                  const uint32_t *exclude_bits, int64_t ent_begin, int64_t ent_end, int k, uint64_t *keys_out,
                  void *scratch, int64_t scratch_bytes, void *stream);
int kge_eval_topk_merge(const uint64_t *keys_in, int64_t Q, int lists, int k, uint64_t *keys_out, int64_t *ids_out,
                        float *scores_out, void *stream);

/* ---- similarity search: the k rows of the entity or relation table nearest to each query vector ----
 * A row is the stored row as one flat real vector of the table's width (entity_dim / relation_dim; [re | im] together
 * for double tables).  Scores are "larger is more similar", with acc() the canonical blocked sum of kge_eval_count_ranks
 * (blocks of 32 summed in index order from +0.0f, block sums added in index order; correctly rounded, non-contracted):
 *   KGE_SIM_DOT acc(q x)   KGE_SIM_COSINE acc(q x) / (|q| |x|)   KGE_SIM_L2 -sqrt(acc((q - x)^2))   KGE_SIM_L1 -acc(|q - x|)
 * with |v| = sqrt(acc(v v)); a zero row under cosine gives 0/0 = NaN.  Order and key encoding are kge_eval_topk's.
 * kge_similarity_rows: rows_out [Q, width] = the table rows ids [Q]; an id outside the table writes a zero row and sets
 *   *err_flag (may be NULL).
 * kge_similarity_norms: norms_out [n] = |v| of the table's rows (vectors == NULL, n must be the row count) or of n free
 *   vectors [n, width].
 * kge_similarity_topk: the k best rows in [row_begin, row_end) of each query vector qvec [Q, width], as keys_out [Q, k]
 *   best first; cosine needs qnorm [Q] and xnorm [rows] from kge_similarity_norms.  self_ids [Q] (may be NULL): the row
 *   left out of each query's list, -1 for none.  Merge the slices of several devices with kge_eval_topk_merge.  scratch:
 *   kge_similarity_topk_scratch_bytes() (0 or more; a negative value is an error code).  At most 65535*64 queries per
 *   call.                                                                                                          */
enum { KGE_SIM_DOT = 0, KGE_SIM_COSINE = 1, KGE_SIM_L2 = 2, KGE_SIM_L1 = 3 };
enum { KGE_TABLE_ENTITY = 0, KGE_TABLE_RELATION = 1 };
int kge_similarity_rows(const kge_model_t *m, int table, const int64_t *ids, int64_t Q, float *rows_out,
                        int32_t *err_flag, void *stream);
int kge_similarity_norms(const kge_model_t *m, int table, const float *vectors, int64_t n, float *norms_out,
                         void *stream);
int64_t kge_similarity_topk_scratch_bytes(const kge_model_t *m, int table, int64_t Q, int64_t row_begin, int64_t row_end,
                                          int k);
int kge_similarity_topk(const kge_model_t *m, int table, int metric, const float *qvec, const float *qnorm,
                        const float *xnorm, const int64_t *self_ids, int64_t Q, int64_t row_begin, int64_t row_end,
                        int k, uint64_t *keys_out, void *scratch, int64_t scratch_bytes, void *stream);

/* ---- relation prediction: which relation links h to t, for every query (h, ?, t) (queries [Q,3] int64, the relation
 *      slot is the positive for the ranks and is ignored by the top-k) ----
 * The score of relation r is the 'single'-mode score of (h, r, t) in the canonical order: bit-identical to column t of
 * the TAIL_BATCH entity scores of (h, r, ?) (kge_eval_count_ranks, kge_eval_topk) and to the C oracle.
 * kge_eval_relation_table: the relation operand, once per call: rel_table [nrelation, entity_dim] floats = (cos | sin)
 *   of relation / scale for RotatE, relation / scale for pRotatE; TransE, DistMult and ComplEx use the relation table
 *   as it is (nothing is written, rel_table may be NULL).  pRotatE also needs kge_eval_phase_table (entity side).
 * kge_eval_relation_count_ranks: for the relations in [rel_begin, rel_end), counts[q] += #{r != positive, not set in
 *   filter_bits [Q, ceil(nrelation/32)] : s > s_pos or (s == s_pos and r < positive)} (the tie rule of
 *   kge_eval_count_ranks).  pos_score from kge_eval_positive_scores in TAIL_BATCH mode on the same queries.
 *   scores_out [Q, nrelation] (may be NULL) receives the scores of the slice, a filtered column as s_pos - 1.
 * kge_eval_relation_topk: the k best relations in [rel_begin, rel_end) of each query that are not set in exclude_bits
 *   (may be NULL), as keys_out [Q, k] in the kge_eval_topk encoding (relation id in the low 32 bits), best first;
 *   merge the slices of several devices with kge_eval_topk_merge.  scratch: kge_eval_relation_topk_scratch_bytes()
 *   (0 or more; a negative value is an error code).  An h or t outside the entity table sets *err_flag (may be NULL).
 * kge_eval_relation_filter_bits: bits [Q, ceil(nrelation/32)] of the relations r with (h, r, t) true, from a sorted-key
 *   index (keys h*nentity+t int64 [nkeys], run offsets int64 [nkeys+1], relation ids int32).
 * At most 65535*64 queries per call.                                                                                 */
int kge_eval_relation_table(const kge_model_t *m, float *rel_table, void *stream);
int kge_eval_relation_count_ranks(const kge_model_t *m, const int64_t *queries, int64_t Q, const float *rel_table,
                                  const float *phase_table, const float *pos_score, const uint32_t *filter_bits,
                                  int64_t rel_begin, int64_t rel_end, int32_t *counts, float *scores_out, void *stream);
int64_t kge_eval_relation_topk_scratch_bytes(const kge_model_t *m, int64_t Q, int64_t rel_begin, int64_t rel_end, int k);
int kge_eval_relation_topk(const kge_model_t *m, const int64_t *queries, int64_t Q, const float *rel_table,
                           const float *phase_table, const uint32_t *exclude_bits, int64_t rel_begin, int64_t rel_end,
                           int k, uint64_t *keys_out, void *scratch, int64_t scratch_bytes, int32_t *err_flag,
                           void *stream);
int kge_eval_relation_filter_bits(const int64_t *index_keys, const int64_t *index_offsets, const int32_t *index_relations,
                                  int64_t nkeys, const int64_t *queries, int64_t Q, int64_t nentity, int64_t nrelation,
                                  uint32_t *bits, void *stream);

/* ---- negative sampling: TrainDataset.__getitem__ (dataloader.py:28-67) on the device ----
 * For row b (train triple triple_index[b]) draw N entity ids uniformly from the entities that are NOT in the
 * row's sorted true list true_entities[key_start[t] .. +key_len[t])  (the true heads of (r,t) for head-batch, the
 * true tails of (h,r) for tail-batch).  Counter-based Philox4x32-10 keyed by (seed, step): the same (seed, step)
 * gives the same negatives on any device, and oracle/kge_oracle.py restates the stream bit-for-bit.              */
int kge_sample_negatives(const int64_t *triple_index, const int32_t *key_start, const int32_t *key_len,
                         const int32_t *true_entities, int64_t B, int64_t N, int64_t nentity, uint64_t seed,
                         uint64_t step, int64_t *negative, void *stream);

/* ---- multi-GPU training exchange over NVLink peer memory (no counterpart in the single-device reference: run.py:241-242;
 *      it replaces "all-reduce the gradients, then optimizer.step() on every replica", model.py:301-303) ----
 * Each rank allocates one peer-visible block (kge_peer_alloc), exports it (kge_peer_export -> 64 opaque bytes the host
 * side exchanges by any means) and maps the other ranks' blocks (kge_peer_open) -- or obtains the mappings, and an
 * NVSwitch multicast mapping on top, from any symmetric-memory allocator.  The block holds the rank's gradient
 * workspace [dE | dR | dM | row losses] and a flag block of 2*KGE_PEER_MAX_RANKS uint32.
 * kge_peer_reduce_adam, called by every rank with the same epoch (1, 2, 3, ... per call) after its local train kernels:
 *   - waits until every rank has arrived (flags, bounded wait: err_flag := 2 after 60 s, or KGE_PEER_TIMEOUT_S),
 *   - one call exchanges the region [region_begin4, region_end4) of the parameter part of the workspace (float4 units; a
 *     step may be cut into several regions so that the exchange of a finished gradient slice overlaps the computation
 *     of the next one); for the groups [slice_begin4, slice_end4) of the region it owns the rank sums the G workspaces
 *     (in rank order, or inside the NVSwitch with multimem.ld_reduce when a multicast mapping is given), adds the L3
 *     gradient 3*l3*x*|x| for the tensors flagged l3 (l3_coefficient != 0; model.py:290-297), applies the Adam update
 *     (same arithmetic as kge_adam_step) to the local param / exp_avg / exp_avg_sq and
 *     pushes the new parameter values to every other rank,
 *   - sums the row-loss region of all ranks into rows_out (local, row_floats floats),
 *   - waits until every rank has pushed, then copies the rest of the region (received slices) into the local parameters.
 * host_tensors[i].grad must be the tensor's gradient view inside the local workspace (16-byte aligned offset).
 * After the call all ranks hold bit-identical parameters; exp_avg / exp_avg_sq are current only on the owning rank. */
#define KGE_PEER_MAX_RANKS 16
#define KGE_PEER_HANDLE_BYTES 64
typedef struct kge_peer_group {
  int32_t world, rank;
  void *grad[KGE_PEER_MAX_RANKS];      /* gradient workspace of every rank as mapped here; [rank] is the local one */
  void *flags[KGE_PEER_MAX_RANKS];     /* flag block of every rank as mapped here (zero-initialised)               */
  void *multicast;                     /* NVSwitch multicast mapping of the gradient workspaces (one address = all G
                                          replicas; multimem.ld_reduce / multimem.st), or NULL: unicast NVLink accesses */
} kge_peer_group_t;

int kge_peer_alloc(int device, int64_t bytes, void **ptr);
int kge_peer_free(void *ptr);
int kge_peer_export(void *ptr, void *host_handle);
int kge_peer_open(int device, const void *host_handle, void **peer_ptr);
int kge_peer_close(void *peer_ptr);
int kge_peer_reduce_adam(const kge_peer_group_t *host_group, uint32_t epoch, const kge_adam_tensor_t *host_tensors,
                         int n_tensors, int64_t param_floats, int64_t region_begin4, int64_t region_end4,
                         int64_t slice_begin4, int64_t slice_end4, int64_t row_offset, int64_t row_floats,
                         float *rows_out, double lr, double beta1, double beta2, double eps, double l3_coefficient,
                         int32_t *err_flag, void *stream);

/* ---- entity-sharded optimizer for batch-sharded multi-GPU training ("owner computes"; no counterpart in the single-device
 *      reference, it replaces model.py:301-303 across G replicas without ever forming or exchanging a dense gradient) ----
 * Rank g owns the entity rows [g*base + min(g, rem), +base (+1 if g < rem)), base = nentity / G, rem = nentity % G, and
 * is the only rank that keeps current Adam moments for them.  Every rank's peer block (kge_peer_alloc or a symmetric-
 * memory allocator; same layout everywhere) holds the rank's ENTITY TABLE itself and a gather area of
 * kge_train_gather_bytes() bytes.  One step:
 *   1. kge_train_rows_sharded: the single-read row kernel over this rank's positive rows.  Its outputs -- query vectors,
 *      dL/ds, candidate ids, target ids of the positives' gradient rows -- are stored into section `rank` of EVERY block
 *      with NVLink stores straight from the kernel; each gradient row of a positive triple is stored only into the block
 *      of the rank that owns its target entity, and each pair adds one count to the histogram in its owner's block.
 *      grad_relation / grad_modulus / row losses stay local (they go through kge_peer_reduce_adam as a small region).
 *      aux_stream (may be NULL): a second stream on which the id mirror runs next to the row kernel.
 *   2. kge_peer_barrier(channel 2, exchange_err = 1): every rank's rows are in; a bad index anywhere raises everywhere.
 *   3. kge_train_entity_sharded: counting sort of the gathered pairs that hit the owned range, entity-major backward with
 *      the fused Adam update of kge_train_rows_adam on the owned rows, and the updated row is stored into every rank's
 *      table (owner computes, all replicas take the same bits).
 *   4. kge_peer_barrier(channel 3): every rank's parameter stores have landed; the next step may read the table and
 *      overwrite the gather area.
 * Wire traffic per rank and step: (G-1)/G of the entity table inbound (the parameter rows) + the gathered (G-1) x
 * rows x (entity_dim + 2N) floats -- half of what a gradient reduce-scatter + parameter all-gather moves -- and it is
 * issued from inside the compute kernels, so no exchange kernel is exposed.  m->entity must point into block[rank]. */
typedef struct kge_shard {
  int32_t world, rank;
  void *block[KGE_PEER_MAX_RANKS];     /* base of every rank's peer block as mapped in this process; [rank] is local */
  void *multicast;                     /* NVSwitch multicast mapping of the blocks (address of block base; one
                                          multimem.st writes every replica), or NULL: one NVLink store per peer      */
  int64_t block_bytes;                 /* size of each block                                                         */
  int64_t gather_offset;               /* byte offset (multiple of 256) of the gather area inside each block         */
  int64_t rows_max;                    /* row capacity per rank of the gather area                                   */
  int32_t rows_of[KGE_PEER_MAX_RANKS]; /* positive rows each rank holds in this step (<= rows_max)                   */
} kge_shard_t;

int64_t kge_train_gather_bytes(const kge_model_t *m, int world, int64_t rows_max, int64_t N);
int64_t kge_train_shard_workspace_bytes(const kge_model_t *m, int world, int64_t rows_max, int64_t N);
int kge_train_rows_sharded(const kge_model_t *m, int mode, int loss_kind, float adversarial_temperature,
                           const int64_t *positive, const int64_t *negative, const float *weight,
                           const float *weight_sum, int64_t B_total, int64_t row_count, int64_t N, float *row_loss,
                           float *pos_row_loss, float *grad_relation, float *grad_modulus,
                           const kge_shard_t *host_shard, int32_t *err_flag, void *stream, void *aux_stream);
int kge_train_entity_sharded(const kge_model_t *m, int mode, int64_t N, const kge_shard_t *host_shard, void *workspace,
                             int64_t workspace_bytes, const kge_entity_adam_t *host_entity_adam, int32_t *err_flag,
                             void *stream);
/* cross-GPU barrier on `stream` over the flag blocks of the group (channels 2 and 3; epoch = 1, 2, 3, ... per channel);
 * exchange_err != 0: a non-zero *err_flag on any rank becomes non-zero on every rank.  phase 0 = arrive and wait; 1 =
 * arrive only and 2 = wait only (same epoch), so that independent kernels can run between the two.  Bounded wait like
 * kge_peer_reduce_adam (err_flag := 2).  The flag block must hold 8 * KGE_PEER_MAX_RANKS uint32.               */
int kge_peer_barrier(const kge_peer_group_t *host_group, int channel, uint32_t epoch, int exchange_err, int phase,
                     int32_t *err_flag, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* KGE_B200_H_ */
