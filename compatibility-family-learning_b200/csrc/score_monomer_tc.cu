// Monomer mode on the cross product, tensor-core path (SURVEY App. A.6 applied to DistBase.build_dist, monomer branch,
// cfl/models/base.py:109-117; gate base.py:94-105):
//     dist(q, c) = sum_k w_qk |a_q - P'_ck|^2 = (sum_k w_qk) |a_q|^2 - g(q, c),
//     g(q, c)    = sum_k [ 2 w_qk a_q . P'_ck - w_qk |P'_ck|^2 ] = v_q . c'_c
// with the AUGMENTED vectors  v_q = [2 w_qk a_q]_k || [-w_qk]_k  and  c'_c = [P'_ck]_k || [|P'_ck|^2]_k  of K(d+1)
// components (both sides centred on the catalog mean mu first: the distance is translation invariant).  So the whole
// catalog pass is ONE Gram matrix, and "dist < threshold" is "g > a2 - threshold": exactly the K = 1 case of the
// lower-bound filter kernel (score_lb.cu) with the row constant |e|^2 := 0.  Pipeline of one call:
//   1. threshold sample: the exact CUDA-core kernel (score_monomer.cu) over every S-th tile -> per query the k-th best
//      (safe threshold tau: a subset's k-th best bounds the catalog's) and the r-th best (optimistic threshold
//      tau_opt: about 4k rows of the whole catalog are expected under it);
//   2. full pass on the tensor cores: score_lb_kernel<1> over the fp16 image of c' (fp32 accumulate), the rounding of
//      the single product bounded rigorously (margin in |v_q||c'_c|), survivors appended to per-query key buffers;
//   3. exact rescoring of every survivor in the direct-difference form of score_monomer_kernel (same operation
//      order: the values are final and bit-identical to the CUDA-core path), top-k by (value, index), and the
//      verification of the optimistic threshold (k survivors with dist <= tau_opt);
//   4. queries that fail it, or whose buffers overflowed, or when a value left the fp16 range: redone by the exact
//      CUDA-core kernel under no threshold (CTAs of query tiles without such a query exit at once).
// Work per score: 2 K (d+1) flop, one MMA per product; catalog bytes per row: 2 * pad16(K(d+1)) + 8.
//
// The other direction (cfl_score_topk_monomer_source): the catalog rows are SOURCE items (a_c, w_c), the queries TARGET
// items (prototypes P'_q), and the same Gram product is transposed:
//     dist(q, c) = (sum_k w_ck) |a_c|^2 - v_c . c'_q
// so the catalog image holds the sources' v_c (mono_src_pack_kernel, the layout of mono_image), the query image the
// targets' c'_q (mono_src_prep_lb_kernel), and the constant moves from the query slot to the row slot:
// lbrow = (W_c, |v_c|) with W_c = (sum_k w_ck)|a_c - mu|^2 rounded down with the slack of the forward a2, lbq = (0, |c'_q|).
// The filter is score_lb_kernel<1> unchanged.  Its margin, re-derived for the swapped roles (K = 1: no basis terms):
//   * the kernel passes (row, query) iff  g~ + tau' > e2s,  tau' = threshold rounded up (cq = 0 - tau, rounded down),
//     e2s = W_c c_e2 - c_sq |v_c| - c_abs with amax = max |c'_q| over the CTA's queries;
//   * fp16 operands: |g~ - v.c'| <= u |v||c'| + 2^-25 (|v|_1 + |c'|_1); c_sq |v_c| holds 2 (u + ulp) amax |v_c|, twice
//     the product term (the forward path halves its query norm; here both norms enter whole), and the subnormal terms
//     2 s16 |v_c| + 2 s16 amax exceed 2^-25 sqrt(dp) (|v| + |c'|) >= 2^-25 (|v|_1 + |c'|_1);
//   * fp32 evaluation: g~ + tau' loses at most ulp (|g~| + tau'), |g~| <= |v||c'| inside the c_sq term, tau' inside the
//     5e-7 slack of cq; W_c c_e2 lowers W_c by CFL_PLANE_REL, far more than the rounding of the fmaf chain;
//   * so a row with closed-form distance W_c - v.c' <= tau always passes; the rescoring's fp32 direct form differs from
//     the closed form by fp32 rounding of O(K d) non-negative terms: covered by W_c's (1 - 1e-5) and the threshold's
//     (1 + 2e-5) slack (mono_thresholds_kernel), exactly as in the forward direction.
// Rescoring (mono_rescore_src_kernel) and the sample / redo passes (score_monomer_src_kernel, score_monomer.cu) use the
// operation order of monomer_direct (direct.cuh), so the packed and the CUDA-core routes return identical bits.
#include <cuda_fp16.h>
#include <string.h>
#include "direct.cuh"
#include "score.cuh"

namespace cfl {

constexpr int MONO_QT = 16;              // query tile of the CUDA-core kernel (score_monomer.cu)
constexpr int MONO_KSTRIDE = TOPK_CAP;
constexpr int MONO_SAMPLE_STRIDE = 32;

int mono_exact_launch(const float* Aq, int64_t lda, const float* Wq, int64_t Q, int K, int d, const float* Pc, int64_t N,
                      int64_t ldp, int kk, int tile_stride, const int* redo_tile, tkey_t* keys, int* counts, int* parts_out,
                      cudaStream_t cs);
int mono_exact_parts(int64_t Q, int64_t N, int K, int d);
int mono_merge_launch(const tkey_t* keys, const int* counts, int parts, int64_t Q, int k, int64_t idx_base, float* top_val,
                      int64_t* top_idx, const float* only_redo, cudaStream_t cs);
int mono_src_exact_launch(const float* Pq, int64_t ldq, int64_t Q, int K, int d, const float* Ac, int64_t lda,
                          const float* Wc, int64_t N, int kk, int tile_stride, const int* redo_tile, tkey_t* keys,
                          int* counts, int* parts_out, cudaStream_t cs);
int mono_src_exact_parts(int64_t Q, int64_t N, int K, int d);

__host__ __device__ static inline int mono_dp(int K, int d) { return (K * (d + 1) + 15) / 16 * 16; }   // augmented dimension, padded to MMA K-steps

// ---- catalog image: fp16 plane [tile][kstep16][chunk][128 rows][8 halfs] of c', flag word, lbrow = (0, |c'|) ---------
// A source catalog (cfl_monomer_source_pack) has the same layout with the rows' v vectors and lbrow = (W_c, |v_c|).
size_t mono_image_bytes(int64_t N, int K, int d) {
  const int64_t tiles = (N + 127) / 128;
  return (size_t)tiles * (mono_dp(K, d) / 16) * 4096 + 16 + (size_t)tiles * 128 * sizeof(float2);
}
struct MonoImage { unsigned char* plane; int* flag; float2* lbrow; };
static MonoImage mono_image(const void* image, int64_t N, int K, int d) {
  MonoImage v;
  v.plane = (unsigned char*)const_cast<void*>(image);
  v.flag = (int*)(v.plane + (size_t)((N + 127) / 128) * (mono_dp(K, d) / 16) * 4096);
  v.lbrow = (float2*)((char*)v.flag + 16);
  return v;
}

__global__ void __launch_bounds__(128)
mono_pack_kernel(const float* __restrict__ P, int64_t N, int K, int d, int64_t ldp, const float* __restrict__ mu,
                 unsigned char* __restrict__ img16, int* __restrict__ flag16, float2* __restrict__ lbrow) {
  const int64_t tile = blockIdx.x;
  const int r = threadIdx.x;
  const int64_t row = tile * 128 + r;
  const int nks = mono_dp(K, d) / 16;
  float c2 = 0.0f, vmax = 0.0f;
  float nrm[CFL_MAX_K];
  for (int k = 0; k < K; ++k) {
    float s = 0.0f;
    if (row < N)
      for (int j = 0; j < d; ++j) { const float v = P[row * ldp + k * d + j] - (mu ? mu[j] : 0.0f); s = fmaf(v, v, s); }
    nrm[k] = s;
  }
  for (int ks = 0; ks < nks; ++ks)
    for (int c = 0; c < 2; ++c) {
      __align__(16) __half h[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int jj = ks * 16 + c * 8 + i;
        float v = 0.0f;
        if (row < N) {
          if (jj < K * d) v = P[row * ldp + jj] - (mu ? mu[jj % d] : 0.0f);
          else if (jj < K * d + K) v = nrm[jj - K * d];
        }
        c2 = fmaf(v, v, c2);
        vmax = fmaxf(vmax, fabsf(v));
        h[i] = __float2half_rn(v);
      }
      *(uint4*)(img16 + ((size_t)tile * nks + ks) * 4096 + (c * 128 + r) * 16) = *(const uint4*)h;
    }
  lbrow[row] = (row < N) ? make_float2(0.0f, sqrtf(c2) * 1.000001f) : make_float2(__int_as_float(0x7f800000), 0.0f);
  if (!(vmax < 60000.0f)) atomicOr(flag16, 1);               // also catches NaN / inf
}

// ---- query image of the K = 1 lower-bound kernel: row ql of image (slot / qt) = v_q; lbq = (a2 rounded down, |v|/2 up) ---
__global__ void __launch_bounds__(128)
mono_prep_lb_kernel(const float* __restrict__ Aq, int64_t lda, const float* __restrict__ Wq, int64_t Q, int K, int d,
                    const float* __restrict__ mu, int qt, int nimg, int dp, unsigned char* __restrict__ img16,
                    int* __restrict__ flag16, float* __restrict__ lbq) {
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t slot = (int64_t)blockIdx.x * 4 + w;
  if (slot >= (int64_t)nimg * qt) return;
  const int nks = dp / 16;
  const int img = (int)(slot / qt), ql = (int)(slot % qt);
  unsigned char* base = img16 + (size_t)img * nks * 2 * qt * 16;
  double a2 = 0.0, v2 = 0.0, wsum = 0.0, vmax = 0.0;
  for (int jj = lane; jj < dp; jj += 32) {
    double v = 0.0;
    if (slot < Q) {
      if (jj < K * d) {
        const int k = jj / d, j = jj % d;
        const double aj = (double)Aq[slot * lda + j] - (mu ? (double)mu[j] : 0.0);
        v = 2.0 * (double)Wq[slot * K + k] * aj;
        if (k == 0) a2 += aj * aj;
      } else if (jj < K * d + K) {
        v = -(double)Wq[slot * K + jj - K * d];
        wsum -= v;
      }
    }
    const float vf = (float)v;                                 // the image holds the fp16 rounding of the FLOAT value
    v2 += (double)vf * (double)vf;
    vmax = fmax(vmax, fabs(v));
    *(__half*)(base + ((size_t)((jj >> 4) * 2 + ((jj >> 3) & 1)) * qt + ql) * 16 + (jj & 7) * 2) = __float2half_rn(vf);
  }
  a2 = warp_sum(a2); v2 = warp_sum(v2); wsum = warp_sum(wsum);
  for (int o = 16; o > 0; o >>= 1) vmax = fmax(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
  if (!(vmax < 60000.0)) atomicOr(flag16, 1);
  if (lane == 0) {
    // dist = wsum * |a - mu|^2 - g; the rescoring arithmetic differs from this closed form by fp32 rounding of
    // O(K d) operations on values <= max(dist terms): covered by the relative slack below
    lbq[2 * slot] = __double2float_rd(wsum * a2 * (1.0 - 1.0e-5));
    lbq[2 * slot + 1] = __double2float_ru(0.5 * sqrt(v2) * 1.000001);
  }
}

// ---- source catalog image: row c = v_c = [2 w_ck (a_c - mu)]_k || [-w_ck]_k; lbrow = (W_c rounded down, |v_c| up) -----
__global__ void __launch_bounds__(128)
mono_src_pack_kernel(const float* __restrict__ A, int64_t lda, const float* __restrict__ W, int64_t N, int K, int d,
                     const float* __restrict__ mu, unsigned char* __restrict__ img16, int* __restrict__ flag16,
                     float2* __restrict__ lbrow) {
  const int64_t tile = blockIdx.x;
  const int r = threadIdx.x;
  const int64_t row = tile * 128 + r;
  const int nks = mono_dp(K, d) / 16;
  double a2 = 0.0, wsum = 0.0, v2 = 0.0;
  float vmax = 0.0f;
  if (row < N) {
    for (int j = 0; j < d; ++j) { const double x = (double)A[row * lda + j] - (mu ? (double)mu[j] : 0.0); a2 += x * x; }
    for (int k = 0; k < K; ++k) wsum += (double)W[row * K + k];
  }
  for (int ks = 0; ks < nks; ++ks)
    for (int c = 0; c < 2; ++c) {
      __align__(16) __half h[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int jj = ks * 16 + c * 8 + i;
        float v = 0.0f;
        if (row < N) {
          if (jj < K * d) {
            const int k = jj / d, j = jj % d;
            v = (float)(2.0 * (double)W[row * K + k] * ((double)A[row * lda + j] - (mu ? (double)mu[j] : 0.0)));
          } else if (jj < K * d + K) {
            v = -W[row * K + jj - K * d];
          }
        }
        v2 += (double)v * (double)v;                           // the image holds the fp16 rounding of the FLOAT value
        vmax = fmaxf(vmax, fabsf(v));
        h[i] = __float2half_rn(v);
      }
      *(uint4*)(img16 + ((size_t)tile * nks + ks) * 4096 + (c * 128 + r) * 16) = *(const uint4*)h;
    }
  // W_c: the slack the forward path gives its a2 (the rescoring's direct form differs from this closed form by fp32
  // rounding); padding rows: +inf, never pass
  lbrow[row] = (row < N) ? make_float2(__double2float_rd(wsum * a2 * (1.0 - 1.0e-5)), __double2float_ru(sqrt(v2) * 1.000001))
                         : make_float2(__int_as_float(0x7f800000), 0.0f);
  if (!(vmax < 60000.0f)) atomicOr(flag16, 1);               // also catches NaN / inf
}

// ---- query image of the source direction: row ql of image (slot / qt) = c'_q = [P'_qk - mu]_k || [|P'_qk - mu|^2]_k;
// lbq = (0, |c'_q| rounded up).  One warp per query slot, fp64.
__global__ void __launch_bounds__(128)
mono_src_prep_lb_kernel(const float* __restrict__ Pq, int64_t ldq, int64_t Q, int K, int d, const float* __restrict__ mu,
                        int qt, int nimg, int dp, unsigned char* __restrict__ img16, int* __restrict__ flag16,
                        float* __restrict__ lbq) {
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t slot = (int64_t)blockIdx.x * 4 + w;
  if (slot >= (int64_t)nimg * qt) return;
  const int nks = dp / 16;
  const int img = (int)(slot / qt), ql = (int)(slot % qt);
  unsigned char* base = img16 + (size_t)img * nks * 2 * qt * 16;
  double c2 = 0.0, vmax = 0.0;
  for (int jj = lane; jj < dp; jj += 32) {
    double v = 0.0;
    if (slot < Q) {
      if (jj < K * d) {
        v = (double)Pq[slot * ldq + jj] - (mu ? (double)mu[jj % d] : 0.0);
      } else if (jj < K * d + K) {
        const float* p = Pq + slot * ldq + (int64_t)(jj - K * d) * d;
        for (int j = 0; j < d; ++j) { const double x = (double)p[j] - (mu ? (double)mu[j] : 0.0); v += x * x; }
      }
    }
    const float vf = (float)v;
    c2 += (double)vf * (double)vf;
    vmax = fmax(vmax, fabs(v));
    *(__half*)(base + ((size_t)((jj >> 4) * 2 + ((jj >> 3) & 1)) * qt + ql) * 16 + (jj & 7) * 2) = __float2half_rn(vf);
  }
  c2 = warp_sum(c2);
  for (int o = 16; o > 0; o >>= 1) vmax = fmax(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
  if (!(vmax < 60000.0)) atomicOr(flag16, 1);
  if (lane == 0) {
    lbq[2 * slot] = 0.0f;
    lbq[2 * slot + 1] = __double2float_ru(sqrt(c2) * 1.000001);
  }
}

__global__ void mono_thresholds_kernel(const float* __restrict__ sval, int64_t Q, int k, int r_opt, float* __restrict__ tau,
                                       float* __restrict__ tau_opt, float* __restrict__ thr_filter,
                                       int* __restrict__ redo_tile, int nredo, int* __restrict__ spill_cnt) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q < nredo) redo_tile[q] = 0;
  if (q >= Q) return;
  spill_cnt[q] = 0;
  const float safe = sval[q * k + k - 1];                     // +inf when the sample held fewer than k rows
  const float opt = (safe < 3.0e38f) ? sval[q * k + r_opt - 1] : safe;
  tau[q] = safe;
  tau_opt[q] = opt;
  // the filter works on the closed form of the distance, the verification on the fp32 direct form (a sum of
  // K d + K non-negative terms: relative rounding <= (K d + K) 2^-24): keep the rows within that of the threshold
  thr_filter[q] = (opt < 3.0e38f) ? opt * (1.0f + 2.0e-5f) + 1.0e-30f : opt;
}

// ---- exact rescoring of the survivors + verification (one CTA per query) --------------------------------------------
template <int K>
__global__ void __launch_bounds__(MRG_THREADS)
mono_rescore_kernel(const tkey_t* __restrict__ keys, const int* __restrict__ counts, int parts, int64_t Q, int k,
                    const float* __restrict__ Aq, int64_t lda, const float* __restrict__ Wq, int d,
                    const float* __restrict__ P, int64_t ldp, int64_t idx_base, float* __restrict__ top_val,
                    int64_t* __restrict__ top_idx, const float* __restrict__ tau, const float* __restrict__ tau_opt,
                    float* __restrict__ thr_redo, int* __restrict__ redo_tile, const tkey_t* __restrict__ spill,
                    const int* __restrict__ spill_cnt, unsigned long long* __restrict__ stats) {
  extern __shared__ __align__(16) float s_dyn[];
  float* s_a = s_dyn;                                          // [d]
  float* s_w = s_a + d;                                        // [K]
  int* s_pref = (int*)(s_w + K);                               // [parts + 2]
  __shared__ tkey_t s[TOPK_CAP];
  __shared__ int s_fill, s_over;
  __shared__ tkey_t s_thr;
  const int t = threadIdx.x;
  const int64_t q = blockIdx.x;
  for (int i = t; i < d; i += MRG_THREADS) s_a[i] = Aq[q * lda + i];
  for (int i = t; i < K; i += MRG_THREADS) s_w[i] = Wq[q * K + i];
  if (t == 0) {
    s_fill = 0;
    s_thr = CFL_KEY_INF;
    int acc = 0, over = 0;
    for (int p = 0; p < parts; ++p) {
      s_pref[p] = acc;
      int c = counts[(int64_t)p * Q + q];
      if (c < 0) { over = 1; c = 0; }                          // the filter pass declined (fp16 range)
      acc += c > TOPK_STRIDE ? TOPK_STRIDE : c;
    }
    s_pref[parts] = acc;
    const int sc = spill_cnt[q];
    over |= sc > LB_SPILL;
    acc += sc > LB_SPILL ? LB_SPILL : sc;
    s_pref[parts + 1] = acc;
    s_over = over;
  }
  __syncthreads();
  const int total = s_pref[parts + 1];
  const bool vec4 = (d % 4 == 0) && (ldp % 4 == 0) && (((uintptr_t)P & 15u) == 0);
  for (int base = 0; base < total; base += MRG_THREADS) {
    const int f = base + t;
    const bool have = f < total;
    uint32_t idx = 0;
    float dist = 0.0f;
    if (have) {
      int p = 0;
      while (s_pref[p + 1] <= f) ++p;
      const tkey_t* src = (p < parts) ? keys + ((int64_t)p * Q + q) * TOPK_STRIDE : spill + q * (int64_t)LB_SPILL;
      idx = (uint32_t)(src[f - s_pref[p]] & 0xffffffffu);
      const float* e = P + (int64_t)idx * ldp;
      // the arithmetic of score_monomer_kernel, operation for operation (values are final)
      float acc = 0.0f;
#pragma unroll
      for (int kq = 0; kq < K; ++kq) {
        float dk = 0.0f;
        const float* ek = e + kq * d;
        if (vec4) {
          for (int j = 0; j < d; j += 4) {
            const float4 v = __ldg((const float4*)(ek + j));
            float df = s_a[j] + (-v.x);     dk = fmaf(df, df, dk);
            df = s_a[j + 1] + (-v.y);       dk = fmaf(df, df, dk);
            df = s_a[j + 2] + (-v.z);       dk = fmaf(df, df, dk);
            df = s_a[j + 3] + (-v.w);       dk = fmaf(df, df, dk);
          }
        } else {
          for (int j = 0; j < d; ++j) { const float df = s_a[j] + (-__ldg(ek + j)); dk = fmaf(df, df, dk); }
        }
        acc = fmaf(s_w[kq], dk, acc);
      }
      dist = acc;
    }
    const int f0 = s_fill;
    __syncthreads();
    if (f0 + MRG_THREADS > TOPK_CAP) mrg_compact(s, &s_fill, &s_thr, k, t);
    if (have) {
      const tkey_t key = pack_key(dist, idx);
      if (key < s_thr) s[atomicAdd(&s_fill, 1)] = key;
    }
    __syncthreads();
  }
  mrg_compact(s, &s_fill, &s_thr, k, t);
  const int fill = s_fill;
  __shared__ int s_redo;
  if (t == 0) {
    // every row outside the survivor set has dist > tau_opt (its bound exceeded it): with k survivors at or under
    // tau_opt the top-k is proven; under the safe threshold (tau_opt == tau) the survivor set always contains it
    const bool optimistic = tau_opt[q] < tau[q];
    const bool proven = !optimistic || (fill >= k && ord2f((uint32_t)(s[k - 1] >> 32)) <= tau_opt[q]);
    const int redo = (s_over || !proven) ? 1 : 0;                // (tau = +inf: every row passed the filter: proven)
    s_redo = redo;
    thr_redo[q] = redo ? 1.0f : __int_as_float(0xff800000);
    if (redo) redo_tile[q / MONO_QT] = 1;
    if (stats) {
      atomicAdd(&stats[STAT_SURVIVORS], (unsigned long long)total);
      if (spill_cnt[q] > 0) atomicAdd(&stats[STAT_SPILL_QUERIES], 1ull);
      if (redo) atomicAdd(&stats[STAT_REDO_QUERIES], 1ull);
      if (q == 0) stats[STAT_LOWER_BOUND_PASS] = 1ull;
    }
  }
  __syncthreads();
  if (s_redo) return;
  for (int i = t; i < k; i += MRG_THREADS) {
    if (i < fill) {
      top_val[q * k + i] = ord2f((uint32_t)(s[i] >> 32));
      top_idx[q * k + i] = idx_base + (int64_t)(uint32_t)(s[i] & 0xffffffffu);
    } else {
      top_val[q * k + i] = __int_as_float(0x7f800000);
      top_idx[q * k + i] = -1;
    }
  }
}

// The source direction: mono_rescore_kernel's body with the query's K prototypes in shared memory and each survivor's
// a and w read from its catalog row; the reported distance is monomer_direct (e = the query's prototypes, a / w = the
// candidate), the operation order of score_monomer_src_kernel.  (A copy rather than a shared inline body: sharing it
// changed the forward kernel's register allocation.)
template <int K>
__global__ void __launch_bounds__(MRG_THREADS)
mono_rescore_src_kernel(const tkey_t* __restrict__ keys, const int* __restrict__ counts, int parts, int64_t Q, int k,
                        const float* __restrict__ Pq, int64_t ldq, int d, const float* __restrict__ Ac, int64_t lda,
                        const float* __restrict__ Wc, int64_t idx_base, float* __restrict__ top_val,
                        int64_t* __restrict__ top_idx, const float* __restrict__ tau, const float* __restrict__ tau_opt,
                        float* __restrict__ thr_redo, int* __restrict__ redo_tile, const tkey_t* __restrict__ spill,
                        const int* __restrict__ spill_cnt, unsigned long long* __restrict__ stats) {
  extern __shared__ __align__(16) float s_dyn[];
  float* s_p = s_dyn;                                          // [K*d]
  int* s_pref = (int*)(s_p + K * d);                           // [parts + 2]
  __shared__ tkey_t s[TOPK_CAP];
  __shared__ int s_fill, s_over;
  __shared__ tkey_t s_thr;
  const int t = threadIdx.x;
  const int64_t q = blockIdx.x;
  for (int i = t; i < K * d; i += MRG_THREADS) s_p[i] = Pq[q * ldq + i];
  if (t == 0) {
    s_fill = 0;
    s_thr = CFL_KEY_INF;
    int acc = 0, over = 0;
    for (int p = 0; p < parts; ++p) {
      s_pref[p] = acc;
      int c = counts[(int64_t)p * Q + q];
      if (c < 0) { over = 1; c = 0; }                          // the filter pass declined (fp16 range)
      acc += c > TOPK_STRIDE ? TOPK_STRIDE : c;
    }
    s_pref[parts] = acc;
    const int sc = spill_cnt[q];
    over |= sc > LB_SPILL;
    acc += sc > LB_SPILL ? LB_SPILL : sc;
    s_pref[parts + 1] = acc;
    s_over = over;
  }
  __syncthreads();
  const int total = s_pref[parts + 1];
  for (int base = 0; base < total; base += MRG_THREADS) {
    const int f = base + t;
    const bool have = f < total;
    uint32_t idx = 0;
    float dist = 0.0f;
    if (have) {
      int p = 0;
      while (s_pref[p + 1] <= f) ++p;
      const tkey_t* src = (p < parts) ? keys + ((int64_t)p * Q + q) * TOPK_STRIDE : spill + q * (int64_t)LB_SPILL;
      idx = (uint32_t)(src[f - s_pref[p]] & 0xffffffffu);
      const float* a = Ac + (int64_t)idx * lda;
      const float* w = Wc + (int64_t)idx * K;
      dist = monomer_direct<K>([&](int kq, int j) { return s_p[kq * d + j]; }, [&](int j) { return __ldg(a + j); },
                               [&](int kq) { return __ldg(w + kq); }, d);
    }
    const int f0 = s_fill;
    __syncthreads();
    if (f0 + MRG_THREADS > TOPK_CAP) mrg_compact(s, &s_fill, &s_thr, k, t);
    if (have) {
      const tkey_t key = pack_key(dist, idx);
      if (key < s_thr) s[atomicAdd(&s_fill, 1)] = key;
    }
    __syncthreads();
  }
  mrg_compact(s, &s_fill, &s_thr, k, t);
  const int fill = s_fill;
  __shared__ int s_redo;
  if (t == 0) {
    // every row outside the survivor set has dist > tau_opt (its bound exceeded it): with k survivors at or under
    // tau_opt the top-k is proven; under the safe threshold (tau_opt == tau) the survivor set always contains it
    const bool optimistic = tau_opt[q] < tau[q];
    const bool proven = !optimistic || (fill >= k && ord2f((uint32_t)(s[k - 1] >> 32)) <= tau_opt[q]);
    const int redo = (s_over || !proven) ? 1 : 0;                // (tau = +inf: every row passed the filter: proven)
    s_redo = redo;
    thr_redo[q] = redo ? 1.0f : __int_as_float(0xff800000);
    if (redo) redo_tile[q / MONO_QT] = 1;
    if (stats) {
      atomicAdd(&stats[STAT_SURVIVORS], (unsigned long long)total);
      if (spill_cnt[q] > 0) atomicAdd(&stats[STAT_SPILL_QUERIES], 1ull);
      if (redo) atomicAdd(&stats[STAT_REDO_QUERIES], 1ull);
      if (q == 0) stats[STAT_LOWER_BOUND_PASS] = 1ull;
    }
  }
  __syncthreads();
  if (s_redo) return;
  for (int i = t; i < k; i += MRG_THREADS) {
    if (i < fill) {
      top_val[q * k + i] = ord2f((uint32_t)(s[i] >> 32));
      top_idx[q * k + i] = idx_base + (int64_t)(uint32_t)(s[i] & 0xffffffffu);
    } else {
      top_val[q * k + i] = __int_as_float(0x7f800000);
      top_idx[q * k + i] = -1;
    }
  }
}

struct MonoTcLayout {
  size_t keys_m, cnt_m, sval, sidx, tau, tau_opt, thr_redo, redo_tile, lbimg, keys_lb, cnt_lb, spill, spill_cnt, stats, total;
};
// parts_m = catalog parts of the CUDA-core kernel of the direction (sample and redo passes)
static MonoTcLayout mono_tc_layout(int64_t Q, int K, int d, int k, const LbPlan& lb, int parts_m) {
  MonoTcLayout L;
  size_t off = 0;
  L.keys_m = off;    off = align_up(off + (size_t)parts_m * Q * MONO_KSTRIDE * sizeof(tkey_t), 256);
  L.cnt_m = off;     off = align_up(off + (size_t)parts_m * Q * sizeof(int), 256);
  L.sval = off;      off = align_up(off + (size_t)Q * k * sizeof(float), 256);
  L.sidx = off;      off = align_up(off + (size_t)Q * k * sizeof(int64_t), 256);
  // tau[Q], tau_opt[Q], thr_redo[Q], then the redo flag per query tile of the CUDA-core kernel
  L.tau = off;       off += (size_t)Q * sizeof(float);
  L.tau_opt = off;   off += (size_t)Q * sizeof(float);
  L.thr_redo = off;  off += (size_t)Q * sizeof(float);
  L.redo_tile = off; off = align_up(off + (size_t)((Q + MONO_QT - 1) / MONO_QT + 4) * sizeof(int), 256);
  L.lbimg = off;     off = align_up(off + score_lb_qimg_bytes(lb, 1, mono_dp(K, d)), 1024);
  L.keys_lb = off;   off = align_up(off + (size_t)lb.parts * Q * TOPK_STRIDE * sizeof(tkey_t), 256);
  L.cnt_lb = off;    off = align_up(off + (size_t)lb.parts * Q * sizeof(int), 256);
  L.spill = off;     off = align_up(off + (size_t)Q * LB_SPILL * sizeof(tkey_t), 256);
  L.spill_cnt = off; off = align_up(off + (size_t)Q * sizeof(int), 256);
  L.stats = off;     off = align_up(off + CFL_SCORE_NSTATS * sizeof(unsigned long long), 256);
  L.total = off + 1024;
  return L;
}

// ---- driver stages shared by both directions ------------------------------------------------------------------------
// Sample stride of the threshold pass: every S-th tile, denser for short catalogs.
static int mono_sample_stride(int64_t tiles, int k) {
  int S = MONO_SAMPLE_STRIDE;
  while (S > 1 && (tiles / S) * 128 < 8 * (int64_t)k) S >>= 1;
  return S;
}

// Stage 1 after the sample pass: merge of its parts, then the safe / optimistic thresholds and the filter threshold.
static int mono_thresholds(const tkey_t* keys_m, const int* cnt_m, int parts_m, int64_t Q, int k, int S, char* base,
                           const MonoTcLayout& L, cudaStream_t cs) {
  float* sval = (float*)(base + L.sval);
  const int st = mono_merge_launch(keys_m, cnt_m, parts_m, Q, k, 0, sval, (int64_t*)(base + L.sidx), nullptr, cs);
  if (st != CFL_OK) return st;
  int r_opt = (4 * k + S - 1) / S;
  if (r_opt < 1) r_opt = 1;
  if (r_opt > k || S == 1) r_opt = k;
  const int nredo = (int)((Q + MONO_QT - 1) / MONO_QT);
  mono_thresholds_kernel<<<(unsigned)((Q + 255) / 256), 256, 0, cs>>>(
      sval, Q, k, r_opt, (float*)(base + L.tau), (float*)(base + L.tau_opt), (float*)(base + L.thr_redo),
      (int*)(base + L.redo_tile), nredo, (int*)(base + L.spill_cnt));        // (nredo <= Q)
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

// Stage 2: the arguments of the Gram pass on the tensor cores (K = 1 case of the lower-bound kernel) over the catalog
// image `mi` and the query image `qv`.
static ScoreArgs mono_filter_args(int64_t Q, int64_t N, int64_t tiles, int dp, int k, const LbPlan& lb, const MonoImage& mi,
                                  const LbQimgView& qv, char* base, const MonoTcLayout& L) {
  ScoreArgs a;
  memset(&a, 0, sizeof(a));
  a.mode = CFL_MONOMER; a.K = 1; a.d = dp; a.Q = Q; a.N = N;
  a.plan.impl = 1; a.plan.tiles = tiles; a.plan.dpad = dp; a.plan.kk = k;
  a.lb = lb;
  a.cimg16 = mi.plane; a.cflag16 = mi.flag; a.lbrow = mi.lbrow;
  a.qimg16 = qv.img; a.qflag16 = qv.flag; a.lbq = qv.lbq;
  a.keys = (tkey_t*)(base + L.keys_lb); a.counts = (int*)(base + L.cnt_lb);
  a.spill = (tkey_t*)(base + L.spill); a.spill_cnt = (int*)(base + L.spill_cnt);
  a.thr_init = (const float*)(base + L.thr_redo);              // filter thresholds (overwritten by the rescoring kernel later)
  a.phase = 3; a.tile_stride = 1;
  return a;
}

}  // namespace cfl

using namespace cfl;

extern "C" {

size_t cfl_monomer_pack_bytes(int64_t N, int K, int d) {
  if (N <= 0 || K < 1 || K > CFL_MAX_K || d < 1 || K * (d + 1) > 128) return 0;     // augmented dimension: 8 MMA K-steps at most
  return mono_image_bytes(N, K, d);
}

int cfl_monomer_pack(const float* Pc, int64_t N, int K, int d, int64_t ldp, const float* mu, void* image, size_t image_bytes,
                     void* stream) {
  int st = device_check();
  if (st != CFL_OK) return st;
  CFL_REQUIRE(Pc && image && N > 0 && ldp >= (int64_t)K * d, CFL_ERR_INVALID, "monomer_pack: bad arguments");
  CFL_REQUIRE(cfl_monomer_pack_bytes(N, K, d) > 0, CFL_ERR_UNSUPPORTED, "monomer_pack: K(d+1) = %d exceeds 128", K * (d + 1));
  CFL_REQUIRE(image_bytes >= mono_image_bytes(N, K, d), CFL_ERR_WORKSPACE, "monomer_pack: image buffer too small");
  CFL_REQUIRE(((uintptr_t)image & 1023u) == 0, CFL_ERR_INVALID, "monomer_pack: image must be 1024-byte aligned");
  const MonoImage v = mono_image(image, N, K, d);
  cudaStream_t cs = (cudaStream_t)stream;
  CFL_CUDA(cudaMemsetAsync(v.flag, 0, 16, cs));
  mono_pack_kernel<<<(unsigned)((N + 127) / 128), 128, 0, cs>>>(Pc, N, K, d, ldp, mu, v.plane, v.flag, v.lbrow);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

size_t cfl_score_topk_monomer_packed_workspace_bytes(int64_t Q, int K, int d, int64_t N, int k) {
  if (Q <= 0 || N <= 0) return 4096;
  const LbPlan lb = make_lb_plan(Q, 1, mono_dp(K, d), (N + 127) / 128);
  return mono_tc_layout(Q, K, d, k, lb, mono_exact_parts(Q, N, K, d)).total;
}

int cfl_score_topk_monomer_packed(const float* Aq, int64_t lda, const float* Wq, int64_t Q, int K, int d, const void* image,
                                  const float* Pc, int64_t N, int64_t ldp, const float* mu, int k, int64_t idx_base,
                                  float* top_val, int64_t* top_idx, unsigned long long* stats_out, void* ws,
                                  size_t ws_bytes, void* stream) {
  int st = device_check();
  if (st != CFL_OK) return st;
  cudaStream_t cs = (cudaStream_t)stream;
  CFL_REQUIRE(K >= 1 && K <= CFL_MAX_K && d >= 1 && K * (d + 1) <= 128, CFL_ERR_UNSUPPORTED,
              "score_topk_monomer_packed: K(d+1) = %d outside [1,128]", K * (d + 1));
  CFL_REQUIRE(k >= 1 && k <= CFL_MAX_TOPK, CFL_ERR_UNSUPPORTED, "score_topk_monomer_packed: k=%d outside [1,%d]", k, CFL_MAX_TOPK);
  CFL_REQUIRE(Q >= 0 && N > 0 && N < ((int64_t)1 << 32), CFL_ERR_INVALID, "score_topk_monomer_packed: bad Q/N");
  CFL_REQUIRE(lda >= d && ldp >= (int64_t)K * d, CFL_ERR_INVALID, "score_topk_monomer_packed: leading dimension too small");
  if (Q == 0) return CFL_OK;
  CFL_REQUIRE(Aq && Wq && Pc && image && top_val && top_idx, CFL_ERR_INVALID, "score_topk_monomer_packed: NULL argument");
  const int64_t tiles = (N + 127) / 128;
  const int dp = mono_dp(K, d);
  const LbPlan lb = make_lb_plan(Q, 1, dp, tiles);
  const MonoTcLayout L = mono_tc_layout(Q, K, d, k, lb, mono_exact_parts(Q, N, K, d));
  CFL_REQUIRE(ws && ws_bytes >= L.total, CFL_ERR_WORKSPACE, "score_topk_monomer_packed: workspace too small (%zu < %zu)",
              ws_bytes, L.total);
  char* base = (char*)ws;
  tkey_t* keys_m = (tkey_t*)(base + L.keys_m);
  int* cnt_m = (int*)(base + L.cnt_m);
  float* tau = (float*)(base + L.tau);
  float* tau_opt = (float*)(base + L.tau_opt);
  float* thr_redo = (float*)(base + L.thr_redo);
  int* redo_tile = (int*)(base + L.redo_tile);
  unsigned long long* stats = (unsigned long long*)(base + L.stats);
  CFL_CUDA(cudaMemsetAsync(stats, 0, CFL_SCORE_NSTATS * sizeof(unsigned long long), cs));

  // 1. thresholds from the exact kernel over every S-th tile
  int parts_m = 0;
  const int S = mono_sample_stride(tiles, k);
  st = mono_exact_launch(Aq, lda, Wq, Q, K, d, Pc, N, ldp, k, S, nullptr, keys_m, cnt_m, &parts_m, cs);
  if (st != CFL_OK) return st;
  st = mono_thresholds(keys_m, cnt_m, parts_m, Q, k, S, base, L, cs);
  if (st != CFL_OK) return st;

  // 2. the Gram pass on the tensor cores (K = 1 case of the lower-bound kernel)
  const LbQimgView qv = score_lb_qimg_view(base + L.lbimg, lb, 1, dp);
  const ScoreArgs a = mono_filter_args(Q, N, tiles, dp, k, lb, mono_image(image, N, K, d), qv, base, L);
  CFL_CUDA(cudaMemsetAsync(qv.flag, 0, 16, cs));
  const int64_t slots = (int64_t)lb.nqt * lb.sub * lb.qt;
  mono_prep_lb_kernel<<<(unsigned)((slots + 3) / 4), 128, 0, cs>>>(Aq, lda, Wq, Q, K, d, mu, lb.qt, lb.nqt * lb.sub, dp,
                                                                  qv.img, qv.flag, qv.lbq);
  CFL_LAUNCH_CHECK();
  timer_record(0, cs);
  st = score_lb_launch(a, cs);
  timer_record(1, cs);
  if (st != CFL_OK) return st;

  // 3. exact rescoring + verification
  const size_t rs_smem = ((size_t)d + K + lb.parts + 2 + 4) * sizeof(float);
  st = with_k(K, [&](auto KC) {
    mono_rescore_kernel<KC><<<(unsigned)Q, MRG_THREADS, rs_smem, cs>>>(
        a.keys, a.counts, lb.parts, Q, k, Aq, lda, Wq, d, Pc, ldp, idx_base, top_val, top_idx, tau, tau_opt, thr_redo,
        redo_tile, a.spill, a.spill_cnt, stats);
    CFL_LAUNCH_CHECK();
    return CFL_OK;
  });
  if (st != CFL_OK) return st;

  // 4. redo: exact CUDA-core pass for the query tiles that hold a flagged query, merged for the flagged queries only
  st = mono_exact_launch(Aq, lda, Wq, Q, K, d, Pc, N, ldp, k, 1, redo_tile, keys_m, cnt_m, &parts_m, cs);
  if (st != CFL_OK) return st;
  st = mono_merge_launch(keys_m, cnt_m, parts_m, Q, k, idx_base, top_val, top_idx, thr_redo, cs);
  if (st != CFL_OK) return st;
  if (stats_out) CFL_CUDA(cudaMemcpyAsync(stats_out, stats, CFL_SCORE_NSTATS * sizeof(unsigned long long), cudaMemcpyDeviceToDevice, cs));
  return CFL_OK;
}

// ---- the source direction -------------------------------------------------------------------------------------------
size_t cfl_monomer_source_pack_bytes(int64_t N, int K, int d) { return cfl_monomer_pack_bytes(N, K, d); }

int cfl_monomer_source_pack(const float* Ac, int64_t lda, const float* Wc, int64_t N, int K, int d, const float* mu,
                            void* image, size_t image_bytes, void* stream) {
  int st = device_check();
  if (st != CFL_OK) return st;
  CFL_REQUIRE(Ac && Wc && image && N > 0 && lda >= d, CFL_ERR_INVALID, "monomer_source_pack: bad arguments");
  CFL_REQUIRE(cfl_monomer_source_pack_bytes(N, K, d) > 0, CFL_ERR_UNSUPPORTED, "monomer_source_pack: K(d+1) = %d exceeds 128",
              K * (d + 1));
  CFL_REQUIRE(image_bytes >= mono_image_bytes(N, K, d), CFL_ERR_WORKSPACE, "monomer_source_pack: image buffer too small");
  CFL_REQUIRE(((uintptr_t)image & 1023u) == 0, CFL_ERR_INVALID, "monomer_source_pack: image must be 1024-byte aligned");
  const MonoImage v = mono_image(image, N, K, d);
  cudaStream_t cs = (cudaStream_t)stream;
  CFL_CUDA(cudaMemsetAsync(v.flag, 0, 16, cs));
  mono_src_pack_kernel<<<(unsigned)((N + 127) / 128), 128, 0, cs>>>(Ac, lda, Wc, N, K, d, mu, v.plane, v.flag, v.lbrow);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

size_t cfl_score_topk_monomer_source_workspace_bytes(int64_t Q, int K, int d, int64_t N, int k) {
  if (Q <= 0 || K < 1 || K > CFL_MAX_K || d < 1 || d > 128 || k < 1 || k > CFL_MAX_TOPK) return 4096;
  const int parts_m = mono_src_exact_parts(Q, N, K, d);
  if (N <= 0 || K * (d + 1) > 128)                             // CUDA-core route only: its keys and counts
    return align_up((size_t)parts_m * Q * MONO_KSTRIDE * sizeof(tkey_t), 256) +
           align_up((size_t)parts_m * Q * sizeof(int), 256) + 1024;
  const LbPlan lb = make_lb_plan(Q, 1, mono_dp(K, d), (N + 127) / 128);
  return mono_tc_layout(Q, K, d, k, lb, parts_m).total;
}

int cfl_score_topk_monomer_source(const float* Pq, int64_t ldq, int64_t Q, int K, int d, const void* image,
                                  const float* Ac, int64_t lda, const float* Wc, int64_t N, const float* mu, int k,
                                  int64_t idx_base, float* top_val, int64_t* top_idx, unsigned long long* stats_out,
                                  void* ws, size_t ws_bytes, void* stream) {
  int st = device_check();
  if (st != CFL_OK) return st;
  cudaStream_t cs = (cudaStream_t)stream;
  CFL_REQUIRE(K >= 1 && K <= CFL_MAX_K, CFL_ERR_UNSUPPORTED, "score_topk_monomer_source: K=%d outside [1,%d]", K, CFL_MAX_K);
  CFL_REQUIRE(d >= 1 && d <= 128, CFL_ERR_UNSUPPORTED, "score_topk_monomer_source: d=%d outside [1,128]", d);
  CFL_REQUIRE(k >= 1 && k <= CFL_MAX_TOPK, CFL_ERR_UNSUPPORTED, "score_topk_monomer_source: k=%d outside [1,%d]", k,
              CFL_MAX_TOPK);
  CFL_REQUIRE(image == nullptr || K * (d + 1) <= 128, CFL_ERR_UNSUPPORTED,
              "score_topk_monomer_source: K(d+1) = %d has no packed image (pass image = NULL)", K * (d + 1));
  CFL_REQUIRE(Q >= 0 && N >= 0 && N < ((int64_t)1 << 32), CFL_ERR_INVALID, "score_topk_monomer_source: bad Q/N");
  CFL_REQUIRE(ldq >= (int64_t)K * d && lda >= d, CFL_ERR_INVALID, "score_topk_monomer_source: leading dimension too small");
  if (Q == 0) return CFL_OK;
  CFL_REQUIRE(Pq && top_val && top_idx, CFL_ERR_INVALID, "score_topk_monomer_source: NULL argument");
  CFL_REQUIRE(N == 0 || (Ac && Wc), CFL_ERR_INVALID, "score_topk_monomer_source: NULL catalog");
  const size_t need = cfl_score_topk_monomer_source_workspace_bytes(Q, K, d, N, k);
  CFL_REQUIRE(ws && ws_bytes >= need, CFL_ERR_WORKSPACE, "score_topk_monomer_source: workspace too small (%zu < %zu)",
              ws_bytes, need);
  char* base = (char*)ws;
  int parts_m = 0;
  if (image == nullptr || N == 0) {
    // CUDA-core route: the exact kernel over every tile (keys and counts at the start of the workspace)
    tkey_t* keys_m = (tkey_t*)base;
    int* cnt_m = (int*)(base + align_up((size_t)mono_src_exact_parts(Q, N, K, d) * Q * MONO_KSTRIDE * sizeof(tkey_t), 256));
    if (stats_out) CFL_CUDA(cudaMemsetAsync(stats_out, 0, CFL_SCORE_NSTATS * sizeof(unsigned long long), cs));
    timer_record(0, cs);
    st = mono_src_exact_launch(Pq, ldq, Q, K, d, Ac, lda, Wc, N, k, 1, nullptr, keys_m, cnt_m, &parts_m, cs);
    timer_record(1, cs);
    if (st != CFL_OK) return st;
    return mono_merge_launch(keys_m, cnt_m, parts_m, Q, k, idx_base, top_val, top_idx, nullptr, cs);
  }
  const int64_t tiles = (N + 127) / 128;
  const int dp = mono_dp(K, d);
  const LbPlan lb = make_lb_plan(Q, 1, dp, tiles);
  const MonoTcLayout L = mono_tc_layout(Q, K, d, k, lb, mono_src_exact_parts(Q, N, K, d));
  tkey_t* keys_m = (tkey_t*)(base + L.keys_m);
  int* cnt_m = (int*)(base + L.cnt_m);
  float* thr_redo = (float*)(base + L.thr_redo);
  int* redo_tile = (int*)(base + L.redo_tile);
  unsigned long long* stats = (unsigned long long*)(base + L.stats);
  CFL_CUDA(cudaMemsetAsync(stats, 0, CFL_SCORE_NSTATS * sizeof(unsigned long long), cs));

  // 1. thresholds from the exact source kernel over every S-th tile
  const int S = mono_sample_stride(tiles, k);
  st = mono_src_exact_launch(Pq, ldq, Q, K, d, Ac, lda, Wc, N, k, S, nullptr, keys_m, cnt_m, &parts_m, cs);
  if (st != CFL_OK) return st;
  st = mono_thresholds(keys_m, cnt_m, parts_m, Q, k, S, base, L, cs);
  if (st != CFL_OK) return st;

  // 2. the transposed Gram pass: catalog image = the sources' v, query image = the targets' c'
  const LbQimgView qv = score_lb_qimg_view(base + L.lbimg, lb, 1, dp);
  const ScoreArgs a = mono_filter_args(Q, N, tiles, dp, k, lb, mono_image(image, N, K, d), qv, base, L);
  CFL_CUDA(cudaMemsetAsync(qv.flag, 0, 16, cs));
  const int64_t slots = (int64_t)lb.nqt * lb.sub * lb.qt;
  mono_src_prep_lb_kernel<<<(unsigned)((slots + 3) / 4), 128, 0, cs>>>(Pq, ldq, Q, K, d, mu, lb.qt, lb.nqt * lb.sub, dp,
                                                                      qv.img, qv.flag, qv.lbq);
  CFL_LAUNCH_CHECK();
  timer_record(0, cs);
  st = score_lb_launch(a, cs);
  timer_record(1, cs);
  if (st != CFL_OK) return st;

  // 3. exact rescoring + verification
  const size_t rs_smem = ((size_t)K * d + lb.parts + 2 + 4) * sizeof(float);
  st = with_k(K, [&](auto KC) {
    mono_rescore_src_kernel<KC><<<(unsigned)Q, MRG_THREADS, rs_smem, cs>>>(
        a.keys, a.counts, lb.parts, Q, k, Pq, ldq, d, Ac, lda, Wc, idx_base, top_val, top_idx, (const float*)(base + L.tau),
        (const float*)(base + L.tau_opt), thr_redo, redo_tile, a.spill, a.spill_cnt, stats);
    CFL_LAUNCH_CHECK();
    return CFL_OK;
  });
  if (st != CFL_OK) return st;

  // 4. redo of the flagged query tiles on the CUDA cores, merged for the flagged queries only
  st = mono_src_exact_launch(Pq, ldq, Q, K, d, Ac, lda, Wc, N, k, 1, redo_tile, keys_m, cnt_m, &parts_m, cs);
  if (st != CFL_OK) return st;
  st = mono_merge_launch(keys_m, cnt_m, parts_m, Q, k, idx_base, top_val, top_idx, thr_redo, cs);
  if (st != CFL_OK) return st;
  if (stats_out) CFL_CUDA(cudaMemcpyAsync(stats_out, stats, CFL_SCORE_NSTATS * sizeof(unsigned long long), cudaMemcpyDeviceToDevice, cs));
  return CFL_OK;
}

}  // extern "C"
