/* cfl_b200.h -- C ABI of the B200-native CFL compatibility-scoring hot path.
 *
 * The reference (appier/compatibility-family-learning) has no FFI: the path is reached
 * through Python constructors that emit stock TensorFlow ops.  Each entry point below
 * replaces the TF op sequence of one reference call site (cited per function, paths
 * relative to the reference root); the Python mirror in
 * compatibility-family-learning_b200/cfl/ binds them with ctypes (INTEGRATION.md shows
 * the stub).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller unless the name ends in
 *     _host; fp32 row-major; `ld*` are leading dimensions in ELEMENTS;
 *   - nothing is allocated inside: cfl_*_workspace_bytes() tells the caller what to pass;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*) and
 *     re-entrant per stream; no global mutable state except a per-device immutable
 *     property cache;
 *   - return value: CFL_OK (0) or a negative cfl_status; cfl_last_error() returns a
 *     thread-local message.  There is NO CPU fallback: without an sm_100 device every
 *     compute call returns CFL_ERR_DEVICE.
 */
#ifndef CFL_B200_H_
#define CFL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  CFL_OK = 0,
  CFL_ERR_INVALID = -1,     /* bad argument (shape, NULL, alignment)          */
  CFL_ERR_CUDA = -2,        /* a CUDA runtime call / launch failed            */
  CFL_ERR_UNSUPPORTED = -3, /* shape outside the compiled range               */
  CFL_ERR_WORKSPACE = -4,   /* workspace too small                            */
  CFL_ERR_DEVICE = -5       /* no sm_100 device                               */
} cfl_status;

/* dist_type -- cfl/models/base.py:109 (monomer), :119 (siamese), :125 (pcd*).  CFL_PCD_SOURCE and CFL_MONOMER_SOURCE
 * are the same distances with the roles swapped (queries = TARGET items, catalog = SOURCE items); only the
 * rank-count and range-query entry points take them (cfl_pair_dist_rows, cfl_rank_counts, cfl_rank_counts_packed,
 * cfl_score_within).  The paired-loss and top-k entry points reject every mode above CFL_SIAMESE. */
typedef enum { CFL_PCD = 0, CFL_MONOMER = 1, CFL_SIAMESE = 2, CFL_PCD_SOURCE = 3, CFL_MONOMER_SOURCE = 4 } cfl_mode;
/* act_type -- cfl/models/cfl.py:579-586 (+ lrelu, cfl/ops.py:10, for hidden layers) */
typedef enum { CFL_ACT_LINEAR = 0, CFL_ACT_TANH = 1, CFL_ACT_SIGMOID = 2, CFL_ACT_RELU = 3,
               CFL_ACT_LRELU = 4 } cfl_act;

#define CFL_MAX_K 8        /* num_components                                   */
#define CFL_MAX_D 256      /* latent_size (paired kernels); all-pairs: <= 128  */
#define CFL_MAX_TOPK 128   /* k of the all-pairs ranking                       */
#define CFL_PAIR_STATS 8   /* doubles written by cfl_pair_loss_fwd             */

const char* cfl_last_error(void);
int cfl_version(void);
/* Fills SM count and compute capability of the current device. */
int cfl_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---------------------------------------------------------------------------------------
 * Stage 1 -- projection.  Replaces fully_connected_weight_norm (cfl/layers.py:80-94:
 * tf.matmul, g/sqrt(reduce_sum(square(V))), bias_add, activation) and, with
 * weight_norm = 0, tf.contrib.layers.fully_connected (cfl/models/dist.py:45-65).  The
 * input normaliser x/scale (cfl/ops.py:198-199; normalize_v2 with a single norm,
 * cfl/ops.py:107-110) is folded in as in_scale.
 *   y[b,j]  = act( (sum_i in_scale*x[b,i]*V[i,j]) * s_j + bias[j] ),  s_j = g_j/|V_:j| (or 1)
 *   z[b,j]  = sum_i in_scale*x[b,i]*V[i,j]          (optional, saved for the backward)
 *   pre[b,j]= value before the activation          (optional)
 * Arithmetic: 3xTF32 error-compensated tcgen05 MMA, fp32 accumulate (fp32-equivalent).
 * ------------------------------------------------------------------------------------- */
size_t cfl_project_fwd_workspace_bytes(int64_t B, int F, int N);
int cfl_project_fwd(const float* x, int64_t B, int F, int64_t ldx,
                    const float* V, int N, int64_t ldV,
                    const float* g, const float* bias, int weight_norm,
                    float in_scale, int act,
                    float* y, int64_t ldy, float* pre, float* z,
                    void* ws, size_t ws_bytes, void* stream);

/* Backward of the above w.r.t. (V, g, bias) -- the tf.gradients the reference gets
 * implicitly from AdamOptimizer.minimize (cfl/models/cfl.py:1083-1085,
 * cfl/models/dist.py:291-293).  dy is dL/dy (post-activation); y the saved output.
 *   accumulate != 0 adds into dV/dg/dbias (pos and neg batches share one encoder).
 *   reg_c adds the l2_regularizer gradient c*V and c*bias (cfl/models/cfl.py:870-874). */
size_t cfl_project_bwd_workspace_bytes(int64_t B, int F, int N);
int cfl_project_bwd(const float* x, int64_t B, int F, int64_t ldx,
                    const float* V, int N, int64_t ldV,
                    const float* g, const float* bias, int weight_norm, float in_scale, int act,
                    const float* y, int64_t ldy, const float* z, const float* dy, int64_t lddy,
                    float* dV, float* dg, float* dbias, int accumulate, float reg_c,
                    void* ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * Stage 2, paired rows -- DistBase.build_dist (cfl/models/base.py:107-146, identical copy
 * cfl/models/dist.py:70-89) + Thresholder (cfl/models/blocks.py:21-22) + the per-batch
 * reductions of _build_dist_losses (cfl/models/cfl.py:879-902,932-937).
 *   pcd:     a = v (target e0) [B,d];  P = source prototypes [B,K,d]
 *   monomer: a = source e0;  P = TARGET prototypes;  w = source gate softmax [B,K]
 *   siamese: a, P = the two e0 rows (K = 1)
 *   label: 1 positive pairs, 0 negative pairs, -1 no loss statistics
 * Outputs (each optional): dist[B], score[B] = max(theta,1e-6) - dist, s[B,K] softmax,
 * stats[8] doubles = { sum softplus(-/+score), #correct, sum dist, sum sqrt(dist+1e-7),
 *                      sum max(0,margin-dist), B, 0, 0 } reduced in a fixed order.
 * Direct-difference form, fp32.
 * ------------------------------------------------------------------------------------- */
size_t cfl_pair_workspace_bytes(int64_t B);
int cfl_pair_loss_fwd(int mode, const float* a, int64_t lda, const float* P, int64_t ldP,
                      const float* w, int64_t B, int K, int d,
                      const float* theta, int label, float margin,
                      float* dist, float* score, float* s, double* stats,
                      void* ws, size_t ws_bytes, void* stream);

/* Backward of the paired distance + loss (its own kernel; recomputes dist/softmax).
 * Upstream: ddist_in[B] if non-NULL, else the fused loss gradient
 *   label 1:  c_ce*sigmoid(dist-theta+) + c_lin        (cfl.py:879-882, 912-929)
 *   label 0: -c_ce*sigmoid(theta+-dist) - c_margin*[dist<margin]
 * dtheta_sum (double, optional) = -sum of the sigmoid-CE part (apply the theta>=1e-6
 * mask on the host, cfl/models/blocks.py:21).  Outputs da[B,d], dP[B,K,d], dw[B,K]. */
int cfl_pair_loss_bwd(int mode, const float* a, int64_t lda, const float* P, int64_t ldP,
                      const float* w, int64_t B, int K, int d,
                      const float* theta, int label, float margin,
                      float c_ce, float c_lin, float c_margin, const float* ddist_in,
                      float* da, int64_t ldda, float* dP, int64_t lddP, float* dw,
                      double* dtheta_sum, void* ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * Stage 2, all pairs (extension, SURVEY App. A.6: the pair scorer on the QxN cross
 * product; no reference call site).  pcd (K>=1) and siamese (K=1); monomer: cfl_score_topk_monomer.
 *   Pq[Q,K,d] query prototypes, E[N,d] catalog embeddings, mu[d] optional centring vector
 *   (distance is translation invariant; centring keeps the Gram form accurate).
 * Gram form d_k = |e|^2+|p_k|^2-2 p_k.e on tensor cores (3xTF32), soft-min epilogue and a
 * running per-query top-(k+slack) fused behind the MMA; the slack winners are rescored in
 * direct-difference form and the best k returned:
 *   top_val[Q,k] ascending exact distances, top_idx[Q,k] = idx_base + row (int64);
 *   ties -> lower index.  dist_out[Q,N] (optional, parity/debug) = un-rescored Gram values.
 * ------------------------------------------------------------------------------------- */
size_t cfl_score_topk_workspace_bytes(int64_t Q, int K, int d, int64_t N, int k);
int cfl_score_topk(int mode, const float* Pq, int64_t Q, int K, int d, int64_t ldq,
                   const float* E, int64_t N, int64_t lde, const float* mu,
                   int k, int64_t idx_base,
                   float* top_val, int64_t* top_idx, float* dist_out,
                   void* ws, size_t ws_bytes, void* stream);

/* Catalog image for the tensor-core kernel: the catalog is static across query batches, so its MMA
 * operand form (centred on mu, hi/lo tf32 split, canonical shared-memory layout, |e-mu|^2 per row)
 * is built once.  cfl_catalog_pack_bytes returns 0 when (K, d) has no tcgen05 tiling (use
 * cfl_score_topk then).  `image` must be 1024-byte aligned; mu must be the same vector later passed
 * to cfl_score_topk_packed, which is cfl_score_topk minus the per-call packing (E is still needed
 * for the direct-form rescoring of the winners). */
size_t cfl_catalog_pack_bytes(int64_t N, int K, int d);
int cfl_catalog_pack(const float* E, int64_t N, int K, int d, int64_t lde, const float* mu,
                     void* image, size_t image_bytes, void* stream);
size_t cfl_score_topk_packed_workspace_bytes(int64_t Q, int K, int d, int64_t N, int k);
int cfl_score_topk_packed(int mode, const float* Pq, int64_t Q, int K, int d, int64_t ldq,
                          const void* image, const float* E, int64_t N, int64_t lde, const float* mu,
                          int k, int64_t idx_base,
                          float* top_val, int64_t* top_idx, float* dist_out,
                          void* ws, size_t ws_bytes, void* stream);

/* The other direction of the pcd distance: rank the SOURCE items of a catalog for TARGET queries.  pcd is not
 * symmetric: dist = |v - sum_k s_k p_k|^2 takes v = e0 of the TARGET item and p_k = the K prototypes of the SOURCE
 * item (DistBase.build_dist, cfl/models/base.py:125-139).  cfl_score_topk answers "which targets go with this source";
 * cfl_score_topk_source answers "which sources is this target compatible with":
 *   Eq[Q,d] (leading dimension ldq) = e0 of the target (query) items,
 *   Pc[N,K,d] = the K prototypes of the source (catalog) items, prototype k of row c at columns [k*d,(k+1)*d) of a row
 *   of length ldp; mu[d] optional centring vector (e.g. the mean of all prototypes), the one the image was built with;
 *   dist(q,c) = pcd(v = Eq[q], P = Pc[c]).
 * cfl_source_catalog_pack builds the catalog's tensor-core image once (cfl_source_catalog_pack_bytes; 0 when N <= 0 or
 * K, d are out of range; `image` 1024-byte aligned): K planes of centred tf32 hi/lo blocks per 128-row tile and every
 * row's soft-min constants.  cfl_score_topk_source: 3xTF32 Gram form with the soft-min epilogue and running top-k
 * (the exact filter cascade of cfl_score_topk: sampled thresholds, filter, verification, exact redo), winners rescored in
 * direct-difference form.  Outputs and tie rule as cfl_score_topk: top_val[Q,k] ascending exact distances, top_idx[Q,k]
 * = idx_base + row, ties -> lower index, -1 / +inf when N < k; dist_out[Q,N] (optional) = un-rescored Gram values;
 * stats_out (optional, device) = CFL_SCORE_NSTATS counters of this call as cfl_score_topk_stats (slot [4], the
 * lower-bound pass, is always 0; all zero for catalogs short enough for the single adaptive pass).  K <= 8, d <= 128,
 * k <= 128.  No reference call site (SURVEY App. A.6). */
size_t cfl_source_catalog_pack_bytes(int64_t N, int K, int d);
int cfl_source_catalog_pack(const float* Pc, int64_t N, int K, int d, int64_t ldp, const float* mu,
                            void* image, size_t image_bytes, void* stream);
size_t cfl_score_topk_source_workspace_bytes(int64_t Q, int K, int d, int64_t N, int k);
int cfl_score_topk_source(const float* Eq, int64_t ldq, int64_t Q, int K, int d, const void* image,
                          const float* Pc, int64_t N, int64_t ldp, const float* mu, int k, int64_t idx_base,
                          float* top_val, int64_t* top_idx, float* dist_out, unsigned long long* stats_out,
                          void* ws, size_t ws_bytes, void* stream);

/* Statistics of the LAST cfl_score_topk / cfl_score_topk_packed call that used workspace `ws` with this shape
 * (packed = 1 for the _packed entry point): CFL_SCORE_NSTATS unsigned 64-bit counters copied to device memory
 * `stats_out` on `stream`: [0] keys that survived the full filter pass, summed over queries (each is rescored
 * exactly), [1] queries that used their spill list, [2] queries the probe took out of the lower-bound pass,
 * [3] queries that failed the first verification (second lower-bound round under the safe threshold, or the exact
 * redo), [4] 1 when the lower-bound pass ran, [5] queries redone by the exact kernel under the safe threshold.  All zero
 * for catalogs short enough for the single adaptive pass.  thr_out (optional, device, 3*Q floats): the per-query
 * thresholds of that call -- safe threshold tau, optimistic threshold tau_opt, redo threshold (-inf = not redone).
 * (bench.py prints the counters so that a regression to the slow paths is visible; no reference call site.) */
#define CFL_SCORE_NSTATS 8
int cfl_score_topk_stats(int64_t Q, int K, int d, int64_t N, int k, int packed, const void* ws, size_t ws_bytes,
                         unsigned long long* stats_out, float* thr_out, void* stream);

/* Monomer mode on the cross product (SURVEY App. A.6 applied to DistBase.build_dist, monomer branch,
 * cfl/models/base.py:109-117; gate cfl/models/base.py:94-105).  The roles follow the reference:
 *   Aq[Q,d]  = act(e0) of the SOURCE (query) items,  Wq[Q,K] = their gate softmax (dense, row-major),
 *   Pc[N,K,d] = the K prototypes of the TARGET (catalog) items (prototype k of row c at columns
 *   [k*d,(k+1)*d) of a row of length ldp), so the catalog side carries K*d floats per row;
 *   dist(q,c) = sum_k Wq[q,k] * |Aq[q] - Pc[c,k]|^2   (direct-difference form, fp32: values are final).
 * Outputs as cfl_score_topk: top_val ascending, top_idx = idx_base + row, ties -> lower index;
 * dist_out[Q,N] optional (parity/debug).  CUDA-core kernel (packed FP32x2), no tensor-core image. */
size_t cfl_score_topk_monomer_workspace_bytes(int64_t Q, int K, int d, int64_t N, int k);
int cfl_score_topk_monomer(const float* Aq, int64_t lda, const float* Wq, int64_t Q, int K, int d,
                           const float* Pc, int64_t N, int64_t ldp, int k, int64_t idx_base,
                           float* top_val, int64_t* top_idx, float* dist_out,
                           void* ws, size_t ws_bytes, void* stream);

/* Monomer mode, tensor-core path.  With the augmented vectors v_q = [2 w_qk a_q]_k || [-w_qk]_k and
 * c'_c = [P'_ck]_k || [|P'_ck|^2]_k (both sides centred on mu) the distance is (sum_k w_qk)|a_q|^2 - v_q.c'_c: ONE Gram
 * matrix of inner dimension K(d+1) <= 128.  cfl_monomer_pack builds the catalog's fp16 image once (1024-byte aligned,
 * cfl_monomer_pack_bytes; 0 = no tensor-core path for this shape: use cfl_score_topk_monomer).
 * cfl_score_topk_monomer_packed: thresholds from the exact CUDA-core kernel on a 1/32 sample of the tiles, the full
 * pass as a single-product fp16 tcgen05 Gram filter with a rigorous rounding margin, exact fp32 direct-form rescoring
 * of every survivor (the arithmetic of cfl_score_topk_monomer: identical bits), verification, exact redo of the
 * queries that fail it.  Outputs as cfl_score_topk_monomer.  stats_out: optional CFL_SCORE_NSTATS counters (device)
 * as cfl_score_topk_stats.  Pc / mu must be the arrays the image was built from. */
size_t cfl_monomer_pack_bytes(int64_t N, int K, int d);
int cfl_monomer_pack(const float* Pc, int64_t N, int K, int d, int64_t ldp, const float* mu, void* image,
                     size_t image_bytes, void* stream);
size_t cfl_score_topk_monomer_packed_workspace_bytes(int64_t Q, int K, int d, int64_t N, int k);
int cfl_score_topk_monomer_packed(const float* Aq, int64_t lda, const float* Wq, int64_t Q, int K, int d,
                                  const void* image, const float* Pc, int64_t N, int64_t ldp, const float* mu, int k,
                                  int64_t idx_base, float* top_val, int64_t* top_idx,
                                  unsigned long long* stats_out, void* ws, size_t ws_bytes, void* stream);

/* The other direction of the monomer distance: rank the SOURCE items of a catalog for TARGET queries.  The monomer
 * distance is directed: a and the gate w come from the source item, the K prototypes from the target item
 * (cfl/models/base.py:94-117).  cfl_score_topk_monomer answers "which targets go with this source";
 * cfl_score_topk_monomer_source answers "which sources is this target compatible with":
 *   Pq[Q,K*d] (leading dimension ldq) = the K prototypes of the target (query) items,
 *   Ac[N,d] (leading dimension lda) = act(e0) of the source (catalog) items, Wc[N,K] = their gate softmax (dense);
 *   dist(q,c) = sum_k Wc[c,k] * |Ac[c] - Pq[q,k]|^2.
 * cfl_monomer_source_pack builds the catalog's fp16 image once (the layout of cfl_monomer_pack with the rows'
 * v_c = [2 w_ck (a_c - mu)]_k || [-w_ck]_k; 1024-byte aligned; cfl_monomer_source_pack_bytes = 0 when K(d+1) > 128).
 * cfl_score_topk_monomer_source runs the stages of cfl_score_topk_monomer_packed with the roles swapped (sampled
 * thresholds on the CUDA cores, the transposed single-product fp16 Gram filter, exact rescoring, verification, exact
 * redo); with image == NULL (required when K(d+1) > 128) it runs the exact CUDA-core kernel over every tile.  Both
 * routes return identical bits.  Outputs as cfl_score_topk_monomer: top_val[Q,k] ascending exact distances,
 * top_idx[Q,k] = idx_base + row, ties -> lower index, -1 / +inf when N < k.  stats_out: optional CFL_SCORE_NSTATS
 * counters (device) as cfl_score_topk_stats (all zero on the CUDA-core route).  K <= 8, d <= 128, k <= 128;
 * N = 0 is allowed.  Ac / Wc / mu must be the arrays the image was built from. */
size_t cfl_monomer_source_pack_bytes(int64_t N, int K, int d);
int cfl_monomer_source_pack(const float* Ac, int64_t lda, const float* Wc, int64_t N, int K, int d, const float* mu,
                            void* image, size_t image_bytes, void* stream);
size_t cfl_score_topk_monomer_source_workspace_bytes(int64_t Q, int K, int d, int64_t N, int k);
int cfl_score_topk_monomer_source(const float* Pq, int64_t ldq, int64_t Q, int K, int d, const void* image,
                                  const float* Ac, int64_t lda, const float* Wc, int64_t N, const float* mu, int k,
                                  int64_t idx_base, float* top_val, int64_t* top_idx,
                                  unsigned long long* stats_out, void* ws, size_t ws_bytes, void* stream);

/* Merge R sorted lists per query (the per-rank results after ncclAllGather) into one:
 * vals[R,Q,k], idx[R,Q,k] -> top_val[Q,k], top_idx[Q,k]; order (value, index). */
int cfl_topk_merge(const float* vals, const int64_t* idx, int R, int64_t Q, int k,
                   float* top_val, int64_t* top_idx, void* stream);

/* The same merge straight from the exchange buffer of the sharded ranking: every rank packs its [Q,k] lists into ONE
 * record (cfl_topk_pack_records: [idx: Q*k int64][val: Q*k float], cfl_topk_record_bytes(Q,k) bytes, a multiple of 16),
 * one all-gather of the records, cfl_topk_merge_records over the R gathered records -- no repacking copies on either
 * side of the collective (the exchange is latency-bound: host time per step matters, see DESIGN section 5). */
size_t cfl_topk_record_bytes(int64_t Q, int k);
int cfl_topk_pack_records(const float* vals, const int64_t* idx, int64_t Q, int k, void* rec, void* stream);
int cfl_topk_merge_records(const void* recs, int R, int64_t Q, int k, float* top_val, int64_t* top_idx, void* stream);

/* Column mean of a catalog E[N,d] (the centring vector mu). */
int cfl_col_mean(const float* E, int64_t N, int d, int64_t lde, float* mu,
                 void* ws, size_t ws_bytes, void* stream);
size_t cfl_col_mean_workspace_bytes(int64_t N, int d);

/* ---------------------------------------------------------------------------------------
 * AUC -- replaces sklearn.metrics.roc_auc_score at cfl/utils.py:267-268 and the accuracy
 * counts at cfl/utils.py:247,264.  Exact integers: out[0] = 2*#{s+>s-} + #{s+==s-},
 * out[1] = n_pos, out[2] = n_neg, out[3] = #{s+>0} + #{s-<=0}.  AUC = out[0]/(2 n+ n-).
 * Radix sort of the negatives + rank/count of every positive.
 * ------------------------------------------------------------------------------------- */
size_t cfl_auc_workspace_bytes(int64_t n_pos, int64_t n_neg);
int cfl_auc(const float* pos_scores, int64_t n_pos, const float* neg_scores, int64_t n_neg,
            int64_t* out4, void* ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * Per-query all-candidate AUC -- the rank statistic of roc_auc_score (cfl/utils.py:267-268) for one
 * query against EVERY catalog row (SURVEY 8d C3, 8e), without materialising the Q x N scores.
 * Operands per mode (the pair scorer's roles, cfl/models/base.py:107-146):
 *   pcd / siamese: Pq[Q,K,d] query prototypes (ldq >= K*d), Wq NULL, E[N,d] candidate embeddings;
 *   monomer:       Pq[Q,d] query embeddings (ldq >= d), Wq[Q,K] gate softmax, E[N,K,d] candidate
 *                  prototypes (lde >= K*d); the 128-row tile of K*d floats per row must fit one CTA's shared
 *                  memory: K*d <= ~380, else CFL_ERR_UNSUPPORTED.
 *   pcd_source:    (CFL_PCD_SOURCE) Pq[Q,d] = the TARGET items' e0 (ldq >= d), Wq NULL, E[N,K,d] = the SOURCE items'
 *                  prototypes (lde >= K*d); dist(q,c) = the pcd direct form with e = Pq[q], p = E[c] (the values
 *                  cfl_score_topk_source reports).  Every K <= 8, d <= 128.
 *   monomer_source: (CFL_MONOMER_SOURCE) Pq[Q,K,d] = the TARGET items' prototypes (ldq >= K*d), E[N,d] = the SOURCE
 *                  items' a (lde >= d), Wq[N,K] = the SOURCE items' gate softmax: the gate argument belongs to
 *                  whichever side is the monomer source.  dist(q,c) = sum_k Wq[c,k] |E[c] - Pq[q,k]|^2 in the
 *                  operation order of cfl_score_topk_monomer_source.
 * The integers, sets, bits and tie rules are the same for every mode.
 * cfl_pair_dist_rows: pos_dist[q,j] = dist(q, row pos_idx[q,j]) for the J labelled positives of each
 *   query; pos_idx is LOCAL to this shard, entries outside [0,N) (e.g. -1: positive lives on another
 *   shard, or padding) give NaN.
 * cfl_rank_counts: counts[q,j,0] = #{c < N : dist(q,c) <  pos_dist[q,j]},
 *                  counts[q,j,1] = #{c < N : dist(q,c) == pos_dist[q,j]}   (int64; NaN counts nothing).
 * Both evaluate the distance in fp32 direct-difference form through one device function, so a positive
 * compares equal to itself and the counts are exact integers that ADD over catalog shards.  With n
 * candidates in total and the positives' own contributions removed, AUC_q = 2U_q / (2 J (n - J)).
 * ------------------------------------------------------------------------------------- */
#define CFL_MAX_RANK_J 32
int cfl_pair_dist_rows(int mode, const float* Pq, int64_t Q, int K, int d, int64_t ldq, const float* Wgate,
                       const float* E, int64_t N, int64_t lde, const int64_t* pos_idx, int J,
                       float* pos_dist, void* stream);
int cfl_rank_counts(int mode, const float* Pq, int64_t Q, int K, int d, int64_t ldq, const float* Wgate,
                    const float* E, int64_t N, int64_t lde, const float* pos_dist, int J,
                    int64_t* counts, void* stream);

/* The same counts over a DENSE distance matrix dense[Q, ldn] (first N columns), e.g. the dist_out of
 * cfl_score_topk: the tensor-core route for pcd -- the Gram-form distances of every (query, row) are written
 * once and counted at HBM speed; thresholds read from the same matrix (pos_dist[q,j] = dense[q, pos]) keep the
 * counts self-consistent (they are exact for the Gram-form fp32 values, which carry the 3xTF32 error of
 * cfl_score_topk's un-rescored distances instead of the direct form's). */
int cfl_dense_rank_counts(const float* dense, int64_t Q, int64_t N, int64_t ldn, const float* pos_dist, int J,
                          int64_t* counts, void* stream);

/* The same counts on the tensor cores, taken inside the fused scoring kernel's epilogue (no Q x N matrix anywhere):
 * image = cfl_catalog_pack of the same E / mu.  Every (row, query) Gram-form distance is classified against the
 * thresholds with a rounding band; pairs inside a band (exact ties included) are re-evaluated in the direct form of
 * cfl_pair_dist_rows, so counts == cfl_rank_counts(...) for pos_dist produced by cfl_pair_dist_rows.  pcd / siamese,
 * and CFL_PCD_SOURCE with the operands of cfl_rank_counts and image = cfl_source_catalog_pack of the same E / mu (its
 * workspace: cfl_rank_counts_packed_source_workspace_bytes; the forward layout, its query regions reused, so
 * cfl_rank_counts_packed_stats reads both with the same Q, K, d, N).
 * Replaces roc_auc_score over all candidates (cfl/utils.py:267-268); see csrc/rank_counts_tc.cu.  One call takes up
 * to 4096 scoring CTAs' worth of queries (>= 131072 queries; CFL_ERR_UNSUPPORTED beyond: split the query batch).
 * cfl_rank_counts_packed_stats (synchronises the stream): out[CFL_RANK_NSTATS] = {ambiguous records, largest
 * |Gram - direct| / band in units of 2^-20, records beyond half the band, queries recounted on the CUDA cores}. */
#define CFL_RANK_NSTATS 4
size_t cfl_rank_counts_packed_workspace_bytes(int64_t Q, int K, int d, int64_t N);
size_t cfl_rank_counts_packed_source_workspace_bytes(int64_t Q, int K, int d, int64_t N);
int cfl_rank_counts_packed(int mode, const float* Pq, int64_t Q, int K, int d, int64_t ldq, const float* E,
                           const void* image, int64_t N, int64_t lde, const float* mu, const float* pos_dist, int J,
                           int64_t* counts, void* ws, size_t ws_bytes, void* stream);
int cfl_rank_counts_packed_stats(int64_t Q, int K, int d, int64_t N, const void* ws, size_t ws_bytes, int64_t* out,
                                 void* stream);

/* ---------------------------------------------------------------------------------------
 * Catalog range queries (extension): every catalog row a query is compatible with.  The Thresholder
 * (cfl/models/blocks.py:21-22) scores a pair max(theta, 1e-6) - dist and the accuracy counts of
 * cfl/utils.py:247,264 call it compatible when that score is > 0, i.e. when dist < r with
 * r = max(theta, 1e-6).  For a radius r[q] per query (fp32) the result of q is the set
 *   { c < N : dist(q, c) < r[q] }   (strict; dist = the fp32 direct form of cfl_pair_dist_rows)
 * as CSR lists: rows offsets[q] .. offsets[q + 1] of out_idx (idx_base + row, int64) and out_dist (the
 * direct-form distance, bit-identical to cfl_pair_dist_rows), ordered by (distance, index).  NaN selects
 * nothing, +inf every row.  Operands per mode as cfl_rank_counts.
 * Two steps: the caller counts first -- counts[q] = cfl_rank_counts_packed / cfl_rank_counts with
 * pos_dist = r (J = 1), whose verdicts are the same arithmetic -- and lays out offsets[Q + 1] (device,
 * an exclusive scan of the counts; offsets[0] may be non-zero, out_idx / out_dist are indexed by them) and
 * the outputs; cfl_score_within then fills the segments.
 *   image != NULL (pcd / siamese, cfl_catalog_pack of E / mu; pcd_source, cfl_source_catalog_pack of E / mu): rows
 *   emitted from the tensor-core scoring epilogue (3xTF32 Gram form, rounding band, direct-form check of the pairs
 *   inside it); image == NULL: the CUDA-core direct form (monomer and monomer_source, where image must be NULL; pcd
 *   shapes without a tcgen05 tiling; pcd_source without an image).  Both routes return the same lists.  N < 2^32; one call takes up to
 *   4096 scoring CTAs' worth of queries (split larger batches).  Segments beyond 16384 rows are sorted in
 *   global memory by one CTA (correct, slower).
 * cfl_score_within_stats (synchronises the stream): out[CFL_WITHIN_NSTATS] of the last call on `ws` = {band
 * records, largest |Gram - direct| / band in units of 2^-20, records beyond half the band, queries re-emitted
 * on the CUDA cores (record list overflow), queries whose emitted row count differed from their count (0)}.
 * cfl_within_merge: the sharded result.  Rank r's list (global indices) of query q is rows offsets[r][q] ..
 * offsets[r][q + 1] of idx[r], dist[r] (offsets [R, Q + 1], idx / dist [R, ld]); out_offsets[Q + 1] = the
 * scan of the per-query sums.  The merged lists are ordered by (distance, index), independent of R. */
#define CFL_WITHIN_NSTATS 5
size_t cfl_score_within_workspace_bytes(int mode, int64_t Q, int K, int d, int64_t N);
int cfl_score_within(int mode, const float* Pq, int64_t Q, int K, int d, int64_t ldq, const float* Wgate, const float* E,
                     const void* image, int64_t N, int64_t lde, const float* mu, const float* radius,
                     const int64_t* offsets, int64_t idx_base, int64_t* out_idx, float* out_dist, void* ws,
                     size_t ws_bytes, void* stream);
int cfl_score_within_stats(const void* ws, size_t ws_bytes, int64_t* out, void* stream);
int cfl_within_merge(const int64_t* offsets, const int64_t* idx, const float* dist, int64_t ld, int R, int64_t Q,
                     const int64_t* out_offsets, int64_t* out_idx, float* out_dist, void* stream);

/* TF-1.x Adam (cfl/models/cfl.py:1083-1085): lr_t = lr*sqrt(1-b2^t)/(1-b1^t);
 * p -= lr_t*m/(sqrt(v)+eps).  grad_scale multiplies g first (1/world for DP averaging). */
int cfl_adam_step(float* p, const float* g, float* m, float* v, int64_t n, int step,
                  float lr, float beta1, float beta2, float eps, float grad_scale, void* stream);
/* Same update with the step count t read from DEVICE memory (*step_dev >= 1) when the kernel runs, so
 * a CUDA graph of the whole train step can be replayed while the count advances on the device. */
int cfl_adam_step_dev(float* p, const float* g, float* m, float* v, int64_t n, const int* step_dev,
                      float lr, float beta1, float beta2, float eps, float grad_scale, void* stream);

/* Measurement hook: when both events are non-NULL, cfl_score_topk records them (cudaEventRecord
 * on the call's stream) immediately before and after its dominant scoring kernel, so bench.py can
 * time that kernel alone inside the timed region.  Thread-local; pass NULLs to clear. */
int cfl_set_kernel_timer(void* start_event, void* stop_event);

/* Self-test of the tcgen05 3xTF32 GEMM core on one tile: D[128,N] = A[128,Kd] * B[N,Kd]^T.
 * Test-only; used by tests/ to validate descriptors and layouts in isolation. */
int cfl_selftest_umma(const float* A, const float* Bm, float* D, int N, int Kd, void* stream);

/* Self-test of the lower-bound pass's MMA: operands rounded to fp16, one tcgen05.mma.kind::f16 per 16 dimensions, fp32
 * accumulators; D[128,N] = A[128,Kd] * B[N,Kd]^T, Kd <= 128.  Test-only: tests/ measures the rounding the error margin
 * of the bound has to cover (operand rounding + accumulation inside the tensor core). */
int cfl_selftest_umma_f16(const float* A, const float* Bm, float* D, int N, int Kd, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CFL_B200_H_ */
