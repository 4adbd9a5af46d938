// The pair scorer in fp32 direct-difference form (DistBase.build_dist, cfl/models/base.py:107-146), shared by every
// kernel that must return or compare the SAME bits: the distances cfl_score_topk reports (merge_rescore_kernel and
// rescore_merge_kernel, score.cu), cfl_pair_dist_rows / cfl_rank_counts (rank_counts.cu) and the survivor counting of
// cfl_rank_counts_packed (rank_counts_tc.cu).  The monomer arithmetic is that of score_monomer_kernel.
#pragma once
#include "common.cuh"

namespace cfl {

// pcd / siamese: e = candidate embedding (target e0), p = the query's K prototypes.  UNROLL (the unroll of the loops
// over the dimensions) changes registers, not the order of the operations.
template <int K, int UNROLL = 4, class EAcc, class PAcc>
__device__ __forceinline__ float pcd_direct(EAcc e, PAcc p, int d) {
  float dk[K];
  float mn = 3.0e38f;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    float acc = 0.0f;
#pragma unroll UNROLL
    for (int j = 0; j < d; ++j) { const float df = e(j) - p(k, j); acc = fmaf(df, df, acc); }
    dk[k] = acc;
    mn = fminf(mn, acc);
  }
  if (K == 1) return dk[0];
  float sum = 0.0f;
#pragma unroll
  for (int k = 0; k < K; ++k) { dk[k] = expf(mn - dk[k]); sum += dk[k]; }
  const float inv = 1.0f / sum;
  float dist = 0.0f;
#pragma unroll UNROLL
  for (int j = 0; j < d; ++j) {
    float m = 0.0f;
#pragma unroll
    for (int k = 0; k < K; ++k) m = fmaf(dk[k] * inv, p(k, j), m);
    const float r = e(j) - m;
    dist = fmaf(r, r, dist);
  }
  return dist;
}

// monomer: a = the query's embedding, w = its gate softmax, e(k, j) = prototype k of the candidate.
template <int K, class EAcc, class AAcc, class WAcc>
__device__ __forceinline__ float monomer_direct(EAcc e, AAcc a, WAcc w, int d) {
  float acc = 0.0f;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    float dk = 0.0f;
#pragma unroll 4
    for (int j = 0; j < d; ++j) { const float df = a(j) + (-e(k, j)); dk = fmaf(df, df, dk); }
    acc = fmaf(w(k), dk, acc);
  }
  return acc;
}

}  // namespace cfl
