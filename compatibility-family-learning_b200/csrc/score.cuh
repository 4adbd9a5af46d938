// All-pairs scoring: shared declarations (plan, argument block, soft-min epilogue).
#pragma once
#include "common.cuh"
#include "topk.cuh"

namespace cfl {

// Work decomposition of one cfl_score_topk call.  The catalog is cut into `parts`
// contiguous ranges of 128-candidate tiles, the queries into tiles of `qt` queries; CTA
// (part, qtile) keeps its query tile resident and streams its catalog range.
struct ScorePlan {
  int impl;        // 1 = tcgen05 (score_umma.cu), 0 = CUDA-core kernel (score.cu)
  int qt;          // queries per query tile
  int nqt;         // number of query tiles
  int parts;       // catalog parts
  int64_t tiles;   // 128-candidate tiles in the catalog
  int kk;          // internal list length: k + slack (<= 128)
  int dpad;        // d rounded up to 8 (MMA K granularity for tf32)
};

// Tiling of the lower-bound pass (score_lb.cu): its own query tile, catalog parts and TMEM buffering.
struct LbPlan {
  int qt;      // queries per accumulator buffer (sub-tile): K*qt TMEM columns
  int sub;     // sub-tiles per CTA: every catalog tile in shared memory is multiplied with `sub` query images
  int nqt;     // CTAs along the query axis = ceil(Q / (qt*sub))
  int parts;   // catalog parts (CTAs along the catalog axis)
  int nbuf;    // TMEM accumulator buffers
};

struct ScoreArgs {
  int mode, K, d;
  int64_t Q, N, lde;
  const float* E;        // raw catalog [N, lde]
  const float* mu;       // centring vector or NULL
  const float* Pc;       // centred query prototypes [Q,K,d] (dense)
  const float* qpar;     // per query: p2[K] then pp[K*K]
  const float* qplane;   // per query: plane-bound block (qplane_stride floats)
  const void* qimg;      // tcgen05 B-operand image per query tile (score_umma.cu)
  const void* cimg;      // tcgen05 A-operand image of the catalog (cfl_catalog_pack)
  const float* e2;       // |e - mu|^2 per catalog row, padded to whole tiles (part of the image)
  tkey_t* keys;           // [parts, Q, TOPK_CAP]
  int* counts;           // [parts, Q]
  float* dist_out;       // optional dense [Q,N]
  // tcgen05 kernel pass control: phase 0 = single adaptive pass (running thresholds);
  // phase 1 = adaptive pass over every tile_stride-th tile (the sample that yields thr_init);
  // phase 2 = full pass filtering against the fixed per-query thresholds thr_init (dist <= thr).
  int phase, tile_stride;
  const float* thr_init; // [Q], phase 2
  tkey_t* spill;         // lower-bound pass: [Q, LB_SPILL] keys that did not fit their (part, query) buffer
  int* spill_cnt;        // [Q]
  const int* redo_tile;  // phase 2 redo launch: per query tile, 1 = some query must be redone (else the CTA exits)
  // Lower-bound pass (score_lb_kernel): fp16 operand planes (same 11-bit significand as tf32, twice the MMA rate).
  // The catalog plane lives behind |e|^2 in the catalog image, followed by a flag word that the pack kernel raises
  // when a centred value leaves the fp16 range, and by lbrow = (|e|^2, |e|) per row.  The query side is the
  // lower-bound image of prep_lb_kernel (2a and an orthonormal basis of the prototypes' affine hull per query),
  // its flag word, and lbq = (|a|^2 rounded down, |a| rounded up) per query.  A raised flag makes the kernel hand
  // its queries to the exact redo pass (counts = -1).
  const void* cimg16;
  const void* qimg16;
  const int* cflag16;
  const int* qflag16;
  const float2* lbrow;
  const float* lbq;
  int dbg_mode;          // timing experiments of the lower-bound pass (CFL_SCORE_DBG_MODE bits, score_lb_kernel built with
                         // -DCFL_LB_EXPERIMENTS): 1 = epilogue does nothing, 2 = no TMA / no full-barrier waits, 4 = epilogue
                         // only reads TMEM, 8 = TMEM reads + bound, no pushes, 16 = MMA issue does not wait for the epilogue
                         // (honoured only under CFL_EXPERIMENTS=1)
  ScorePlan plan;
  LbPlan lb;
  // Source-catalog call (cfl_score_topk_source): the catalog rows carry K prototypes (cimg = cfl_source_catalog_pack's
  // image, e2 = its per-row soft-min blocks), the queries one vector each (Pc = the centred vectors [Q,d], qpar =
  // |e_q - mu|^2 per query, qimg of QT vectors per tile); E = the raw prototypes [N, lde], Pq (merge) = the raw queries.
  bool src;
};

// Per-query parameter block (floats), padded to a multiple of 4 so it loads as float4:
//   [0,K)        log2(e) * |p_k|^2
//   [K,K+T)      upper triangle of p_k.p_l, row-major (k,l>=k), DIAGONAL PRE-HALVED; T=K(K+1)/2
//   [K+T]        cq = slack of the soft-min lower bound dist >= min_k d_k - cq,
//                cq = (1-1/K)/2 * max_kl |p_k-p_l|^2 (SURVEY App. A.3), padded for fp32 rounding
__host__ __device__ constexpr int qpar_tri(int K) { return K * (K + 1) / 2; }
__host__ __device__ constexpr int qpar_stride(int K) { return (K + qpar_tri(K) + 1 + 3) / 4 * 4; }

// Plane-bound block per query (K >= 2), used by the tensor-core kernel to skip the soft-min:
// dist = |e - sum_k s_k p_k|^2 with s on the plane sum(s) = 1, so dist >= the squared distance from
// e to the AFFINE HULL of the prototypes, which is a quadratic in the Gram values.  With
// n_k = |p_k|^2, D_kl = |p_k - p_l|^2, [A a; a^T alpha] = inverse of the KKT matrix [D 1; 1^T 0],
// w_j = (g_j - g_0) - (n_j - n_0)/2 for j = 1..K-1:
//   LB = |e|^2 - 2 g_0 + c0 + sum_i w_i (bm2_i + sum_{j>=i} M4_ij w_j)
//   [0,K-1)          dnh_j = -(n_j - n_0)/2
//   [K-1,2K-2)       bm2_j = -2 a_j
//   [2K-2,2K-2+T')   M4 upper triangle (i <= j), row-major: 2 A_ii on the diagonal, 4 A_ij off it
//   [2K-2+T']        c0 = alpha/2 + n_0 - margin   (-inf: bound unavailable, prototypes degenerate)
__host__ __device__ constexpr int qplane_tri(int K) { return (K - 1) * K / 2; }
__host__ __device__ constexpr int qplane_stride(int K) {
  return K < 2 ? 4 : (2 * (K - 1) + qplane_tri(K) + 1 + 3) / 4 * 4;
}
constexpr float CFL_PLANE_REL = 2.0e-4f;     // relative safety margin of the bound (fp32 / 3xTF32 rounding)

// Bytes of one query tile's tcgen05 B-operand image (score_umma.cu): [kstep][hl][chunk][nc = K*qt rows][16 B].
__host__ __device__ constexpr uint32_t qimg_tile_bytes(int dpad, int nc) { return (uint32_t)dpad * 8u * (uint32_t)nc; }

// Slots of the statistics counters of one cfl_score_topk call (cfl_score_topk_stats, cfl_b200.h; the order of
// SCORE_STAT_NAMES in cfl/_native.py).
enum ScoreStat {
  STAT_SURVIVORS = 0,              // keys that survived the full filter pass, summed over queries
  STAT_SPILL_QUERIES,              // queries that used their spill list
  STAT_PROBE_DROPPED_QUERIES,      // queries the probe took out of the lower-bound pass
  STAT_REDO_QUERIES,               // queries that failed the first verification
  STAT_LOWER_BOUND_PASS,           // 1 when the lower-bound pass ran
  STAT_EXACT_REDO_QUERIES,         // queries redone by the exact kernel under the safe threshold
};

ScorePlan make_score_plan(int64_t Q, int K, int d, int64_t N, int k, bool umma_ok);
ScorePlan make_score_plan_qt(int64_t Q, int qt, int d, int64_t N, int k, bool umma_ok);
bool score_umma_supported(int K, int d);
// Catalog image of cfl_catalog_pack (layout in score_umma.cu): behind the tf32 planes, |e - mu|^2 per row, the fp16
// plane of the lower-bound pass, its range flag and lbrow = (|e - mu|^2, |e - mu|) per row.
struct CatalogView { float* e2; unsigned char* f16; int* flag16; float2* lbrow; };
size_t catalog_image_bytes(int64_t N, int d);
CatalogView catalog_view(const void* image, int64_t N, int d);
LbPlan make_lb_plan(int64_t Q, int K, int d, int64_t tiles);
// Query image of the lower-bound pass (score_lb.cu): the fp16 image, its flag word, lbq[2 per query slot].
struct LbQimgView { unsigned char* img; int* flag; float* lbq; };
size_t score_lb_qimg_bytes(const LbPlan& p, int K, int d);
LbQimgView score_lb_qimg_view(void* base, const LbPlan& p, int K, int d);
int catalog_pack_launch(const float* E, int64_t N, int d, int64_t lde, const float* mu, void* image,
                        cudaStream_t st);
int score_umma_pack_queries(const ScoreArgs& a, void* qimg, cudaStream_t st);
int score_lb_prep_queries(const ScoreArgs& a, cudaStream_t st);   // lower-bound image + lbq of the query batch
int score_umma_launch(const ScoreArgs& a, cudaStream_t st);
int score_lb_launch(const ScoreArgs& a, cudaStream_t st);
int score_umma_qt(int K, int d);
// Source-catalog image of cfl_source_catalog_pack (layout in score_umma.cu): K*nks tf32 blocks per 128-row tile, then
// per tile the soft-min blocks of its rows, [tile][j][row], j < source_rowpar_len(K).
__host__ __device__ constexpr int source_rowpar_len(int K) { return K + qpar_tri(K); }
struct SourceCatalogView { unsigned char* blocks; float* rowpar; };
size_t source_catalog_image_bytes(int64_t N, int K, int d);
SourceCatalogView source_catalog_view(const void* image, int64_t N, int K, int d);
int source_catalog_pack_launch(const float* P, int64_t N, int K, int d, int64_t ldp, const float* mu, void* image,
                               cudaStream_t st);
int score_src_qt(int K, int d);
// query prep shared with the rank-count path (rank_counts_tc.cu): centred prototypes, soft-min and plane-bound blocks
int score_prep_queries_launch(const float* Pq, int64_t Q, int K, int d, int64_t ldq, const float* mu, float* Pc,
                              float* qpar, float* qplane, cudaStream_t st);
// the same for the source-catalog direction: centred query vectors Ec [Q,d] and |e_q - mu|^2
int score_prep_source_queries_launch(const float* Eq, int64_t Q, int d, int64_t ldq, const float* mu, float* Ec,
                                     float* e2q, cudaStream_t st);
// rank_counts.cu: the CUDA-core rank count restricted to the queries flagged in only[Q] (adds into counts)
int rank_counts_only_launch(int mode, const float* Pq, int64_t Q, int K, int d, int64_t ldq, const float* E, int64_t N,
                            int64_t lde, const float* pos_dist, int J, unsigned long long* counts, const int* only,
                            cudaStream_t st);
// cfl_score_within (within.cu): the CUDA-core emitting pass (rank_counts.cu; every query, or the ones flagged in only[Q])
// and the tensor-core one (rank_counts_tc.cu) append local rows dist < radius[q] to out[offsets[q], offsets[q + 1])
int within_emit_launch(int mode, const float* Pq, int64_t Q, int K, int d, int64_t ldq, const float* Wq, const float* E,
                       int64_t N, int64_t lde, const float* radius, const int64_t* offsets, unsigned int* cursor,
                       int64_t* out, const int* only, cudaStream_t st);
size_t within_tc_workspace_bytes(int64_t Q, int K, int d, int64_t N, bool src);
int within_tc_emit(int mode, const float* Pq, int64_t Q, int K, int d, int64_t ldq, const float* E, const void* image,
                   int64_t N, int64_t lde, const float* mu, const float* radius, const int64_t* offsets,
                   unsigned int* cursor, int64_t* out, void* ws, unsigned long long* stats, cudaStream_t st);

#ifdef __CUDACC__
__device__ __forceinline__ float fast_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fast_rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

constexpr float CFL_LOG2E = 1.4426950408889634f;
constexpr float CFL_LN2 = 0.6931471805599453f;

// Soft-min distance of one (candidate, query) pair from the Gram values g_k = p_k.e
// (SURVEY App. A.3):  s = softmax_k(2 g_k - |p_k|^2)   [the |e|^2 term cancels],
//   dist = |e|^2 - 2 sum_k s_k g_k + sum_kl s_k s_l (p_k.p_l).
// qp = the per-query parameter block above (registers or shared memory).
// Also returns mx2 = log2e * max_k(2 g_k - |p_k|^2), so that min_k d_k = |e|^2 - ln2 * mx2.
template <int K>
__device__ __forceinline__ float softmin_max2(const float (&g)[K], const float* __restrict__ qp) {
  float mx = fmaf(2.0f * CFL_LOG2E, g[0], -qp[0]);
#pragma unroll
  for (int k = 1; k < K; ++k) mx = fmaxf(mx, fmaf(2.0f * CFL_LOG2E, g[k], -qp[k]));
  return mx;
}

template <int K>
__device__ __forceinline__ float softmin_from_gram(const float (&g)[K], float e2,
                                                   const float* __restrict__ qp) {
  if (K == 1) return fmaf(-CFL_LN2, fmaf(2.0f * CFL_LOG2E, g[0], -qp[0]), e2);
  float a[K];
#pragma unroll
  for (int k = 0; k < K; ++k) a[k] = fmaf(2.0f * CFL_LOG2E, g[k], -qp[k]);
  float mx = a[0];
#pragma unroll
  for (int k = 1; k < K; ++k) mx = fmaxf(mx, a[k]);
  float sum = 0.0f;
#pragma unroll
  for (int k = 0; k < K; ++k) { a[k] = fast_ex2(a[k] - mx); sum += a[k]; }
  const float inv = fast_rcp(sum);
  float t1 = 0.0f, t2 = 0.0f;
  int o = K;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    t1 = fmaf(a[k], g[k], t1);
    float row = qp[o] * a[k];                  // diagonal is stored pre-halved
#pragma unroll
    for (int l = k + 1; l < K; ++l) row = fmaf(qp[o + l - k], a[l], row);
    o += K - k;
    t2 = fmaf(a[k], row, t2);                  // half of sum_kl a_k a_l pp_kl
  }
  // dist = e2 + inv * (-2 t1 + inv * 2 t2)
  return fmaf(inv + inv, fmaf(inv, t2, -t1), e2);
}

// ---- packed (two queries per instruction) variant for the tensor-core kernel's epilogue ---------
// sm_100 has FP32x2 FMA/ADD/MUL (FFMA2...): the soft-min of two queries of the same catalog row is
// evaluated with one instruction per pair wherever the math is FMA-shaped; max / ex2 / rcp stay
// scalar.  qp2[j] = (block_A[j], block_B[j]) with entries [0,K) NEGATED (-log2e*|p_k|^2).
typedef unsigned long long f2_t;
__device__ __forceinline__ f2_t pk2(float a, float b) {
  f2_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ void upk2(f2_t v, float& a, float& b) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
}
__device__ __forceinline__ f2_t fma2(f2_t a, f2_t b, f2_t c) {
  f2_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ f2_t add2(f2_t a, f2_t b) {
  f2_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ float max3(float a, float b, float c) {        // FMNMX3
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
__device__ __forceinline__ f2_t mul2(f2_t a, f2_t b) {
  f2_t r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}

// e2p = (|e|^2 of pair member A, of member B): one catalog row (both the same) for score_umma_kernel, two queries for
// score_src_umma_kernel, whose qp2 is then its row's block broadcast to both members.
template <int K>
__device__ __forceinline__ void softmin_pair2(const float (&gA)[K], const float (&gB)[K], f2_t e2p,
                                              const f2_t* __restrict__ qp2, float& dA, float& dB) {
  const f2_t C2 = pk2(2.0f * CFL_LOG2E, 2.0f * CFL_LOG2E);
  f2_t g[K], a[K];
#pragma unroll
  for (int k = 0; k < K; ++k) { g[k] = pk2(gA[k], gB[k]); a[k] = fma2(C2, g[k], qp2[k]); }
  if (K == 1) {
    upk2(fma2(pk2(-CFL_LN2, -CFL_LN2), a[0], e2p), dA, dB);
    return;
  }
  float mA, mB;
  upk2(a[0], mA, mB);
#pragma unroll
  for (int k = 1; k < K; ++k) { float x, y; upk2(a[k], x, y); mA = fmaxf(mA, x); mB = fmaxf(mB, y); }
  const f2_t nm = pk2(-mA, -mB);
  f2_t w[K];
  f2_t sum;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    float x, y;
    upk2(add2(a[k], nm), x, y);
    w[k] = pk2(fast_ex2(x), fast_ex2(y));
    sum = (k == 0) ? w[0] : add2(sum, w[k]);
  }
  float sA, sB;
  upk2(sum, sA, sB);
  const f2_t ninv = pk2(fast_rcp(-sA), fast_rcp(-sB));     // -1/sum
  f2_t t1, t2;
  int o = K;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    t1 = (k == 0) ? mul2(w[0], g[0]) : fma2(w[k], g[k], t1);
    f2_t row = mul2(qp2[o], w[k]);                          // diagonal is stored pre-halved
#pragma unroll
    for (int l = k + 1; l < K; ++l) row = fma2(qp2[o + l - k], w[l], row);
    o += K - k;
    t2 = (k == 0) ? mul2(w[0], row) : fma2(w[k], row, t2);  // half of sum_kl w_k w_l pp_kl
  }
  // dist = e2 - 2 inv (t1 - inv t2)
  const f2_t v = fma2(ninv, t2, t1);
  upk2(fma2(add2(ninv, ninv), v, e2p), dA, dB);
}
template <int K>
__device__ __forceinline__ void softmin_pair(const float (&gA)[K], const float (&gB)[K], float e2,
                                             const f2_t* __restrict__ qp2, float& dA, float& dB) {
  softmin_pair2<K>(gA, gB, pk2(e2, e2), qp2, dA, dB);
}

// softmin_pair2 that also returns V = sum_k s_k |p_k|^2 - |sum_k s_k p_k|^2, the spread of the prototypes under the
// soft-min weights: d dist / d(exponent k) = s_k * (-2 (e - m).(p_k - m)), so an error du on the exponents moves dist by
// at most 2 sqrt(dist * V) |du| -- the sensitivity term of the rank-count rounding band (rank_counts_tc.cu).  e2p as
// softmin_pair2: pk2(e2, e2) for a catalog row of embeddings, the two queries' |e|^2 for a source catalog.
template <int K>
__device__ __forceinline__ void softmin_pair_var(const float (&gA)[K], const float (&gB)[K], f2_t e2p,
                                                 const f2_t* __restrict__ qp2, float& dA, float& dB, float& vA, float& vB) {
  const f2_t C2 = pk2(2.0f * CFL_LOG2E, 2.0f * CFL_LOG2E);
  f2_t g[K], a[K];
#pragma unroll
  for (int k = 0; k < K; ++k) { g[k] = pk2(gA[k], gB[k]); a[k] = fma2(C2, g[k], qp2[k]); }
  if (K == 1) {
    upk2(fma2(pk2(-CFL_LN2, -CFL_LN2), a[0], e2p), dA, dB);
    vA = 0.0f; vB = 0.0f;
    return;
  }
  float mA, mB;
  upk2(a[0], mA, mB);
#pragma unroll
  for (int k = 1; k < K; ++k) { float x, y; upk2(a[k], x, y); mA = fmaxf(mA, x); mB = fmaxf(mB, y); }
  const f2_t nm = pk2(-mA, -mB);
  f2_t w[K];
  f2_t sum, sp2;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    float x, y;
    upk2(add2(a[k], nm), x, y);
    w[k] = pk2(fast_ex2(x), fast_ex2(y));
    sum = (k == 0) ? w[0] : add2(sum, w[k]);
    sp2 = (k == 0) ? mul2(w[0], qp2[0]) : fma2(w[k], qp2[k], sp2);      // -log2e * sum_k w_k |p_k|^2
  }
  float sA, sB;
  upk2(sum, sA, sB);
  const f2_t ninv = pk2(fast_rcp(-sA), fast_rcp(-sB));     // -1/sum
  f2_t t1, t2;
  int o = K;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    t1 = (k == 0) ? mul2(w[0], g[0]) : fma2(w[k], g[k], t1);
    f2_t row = mul2(qp2[o], w[k]);                          // diagonal is stored pre-halved
#pragma unroll
    for (int l = k + 1; l < K; ++l) row = fma2(qp2[o + l - k], w[l], row);
    o += K - k;
    t2 = (k == 0) ? mul2(w[0], row) : fma2(w[k], row, t2);  // half of sum_kl w_k w_l pp_kl
  }
  const f2_t v = fma2(ninv, t2, t1);
  upk2(fma2(add2(ninv, ninv), v, e2p), dA, dB);
  // V = inv * (ln2 * (-sp2')) ... with sp2 = -log2e * sum w p2:  sum s p2 = ninv * ln2 * sp2;  |m|^2 = 2 inv^2 t2
  const f2_t m2 = mul2(mul2(ninv, ninv), add2(t2, t2));
  upk2(fma2(mul2(ninv, pk2(CFL_LN2, CFL_LN2)), sp2, mul2(m2, pk2(-1.0f, -1.0f))), vA, vB);
}

// Same as softmin_from_gram, reading the pair-interleaved shared-memory block of the tensor-core
// kernel (element j of this query at qb[2*j], first K entries negated).
template <int K>
__device__ __forceinline__ float softmin_from_gram_il(const float (&g)[K], float e2,
                                                      const float* __restrict__ qb) {
  constexpr int NP = K + K * (K + 1) / 2;
  float qp[NP];
#pragma unroll
  for (int j = 0; j < NP; ++j) qp[j] = (j < K) ? -qb[2 * j] : qb[2 * j];
  return softmin_from_gram<K>(g, e2, qp);
}

// Affine-hull lower bound of two queries (packed), pl2 = pair-interleaved plane block.
template <int K>
__device__ __forceinline__ void plane_bound_pair(const float (&gA)[K], const float (&gB)[K], f2_t e2sp,
                                                 const f2_t* __restrict__ pl2, float& lA, float& lB) {
  const f2_t M1 = pk2(-1.0f, -1.0f), M2 = pk2(-2.0f, -2.0f);
  const f2_t g0 = pk2(gA[0], gB[0]);
  if constexpr (K == 1) {                                   // dist = |e|^2 + |p|^2 - 2 g exactly: c0 at [0]
    upk2(fma2(g0, M2, add2(pl2[0], e2sp)), lA, lB);
    return;
  }
  f2_t w[K > 1 ? K - 1 : 1];
#pragma unroll
  for (int j = 1; j < K; ++j) w[j - 1] = fma2(g0, M1, add2(pk2(gA[j], gB[j]), pl2[j - 1]));
  f2_t acc = fma2(g0, M2, add2(pl2[2 * (K - 1) + qplane_tri(K)], e2sp));
  int o = 2 * (K - 1);
#pragma unroll
  for (int i = 0; i < K - 1; ++i) {
    f2_t t = fma2(pl2[o], w[i], pl2[K - 1 + i]);
#pragma unroll
    for (int j = i + 1; j < K - 1; ++j) t = fma2(pl2[o + j - i], w[j], t);
    o += K - 1 - i;
    acc = fma2(w[i], t, acc);
  }
  upk2(acc, lA, lB);
}
#endif

}  // namespace cfl
