// Stage 2 on the Q x N cross product (SURVEY App. A.6): query prep, the CUDA-core scoring
// kernel, the part merge + direct-form rescoring kernel, the cross-rank merge kernel and the
// cfl_score_topk / cfl_topk_merge entry points.  The tensor-core scoring kernel lives in
// score_umma.cu and is used whenever its tiling supports the shape (see score_umma_supported);
// both kernels share the soft-min epilogue (score.cuh) and the top-k machinery (topk.cuh).
#include <stdlib.h>
#include "score.cuh"
#include "direct.cuh"
#include "umma.cuh"

namespace cfl {

// ---- plan --------------------------------------------------------------------------------
constexpr int SIMT_QT = 16;        // queries per CTA tile, CUDA-core kernel
constexpr int SIMT_THREADS = 128;  // one thread per candidate of a 128-row tile

static int choose_kk(int k) {
  int kk = k + 28;                 // slack so Gram-form near-ties cannot change the exact top-k
  if (kk > CFL_MAX_TOPK) kk = CFL_MAX_TOPK;
  if (kk < k) kk = k;
  return kk;
}

ScorePlan make_score_plan(int64_t Q, int K, int d, int64_t N, int k, bool umma_ok) {
  return make_score_plan_qt(Q, umma_ok ? score_umma_qt(K, d) : SIMT_QT, d, N, k, umma_ok);
}

ScorePlan make_score_plan_qt(int64_t Q, int qt, int d, int64_t N, int k, bool umma_ok) {
  ScorePlan p;
  p.impl = umma_ok ? 1 : 0;
  p.qt = qt;
  p.nqt = (int)((Q + p.qt - 1) / p.qt);
  p.tiles = (N + 127) / 128;
  int sms = sm_count();
  if (sms <= 0) sms = 148;
  int target = umma_ok ? sms : 2 * sms;
  int64_t parts = p.nqt > 0 ? target / p.nqt : 1;
  if (parts < 1) parts = 1;
  if (parts > p.tiles) parts = p.tiles;
  if (parts < 1) parts = 1;
  p.parts = (int)parts;
  p.kk = choose_kk(k);
  p.dpad = (d + 7) / 8 * 8;
  return p;
}

// ---- query prep: centre, |p_k|^2, p_k.p_l --------------------------------------------------
__global__ void prep_queries_kernel(const float* __restrict__ Pq, int64_t Q, int K, int d,
                                    int64_t ldq, const float* __restrict__ mu,
                                    float* __restrict__ Pc, float* __restrict__ qpar,
                                    float* __restrict__ qplane) {
  __shared__ float sD[4][8][8];
  __shared__ float sN[4][8];
  const int w = threadIdx.x / 32;
  int64_t q = (int64_t)blockIdx.x * (blockDim.x / 32) + w;
  int lane = threadIdx.x & 31;
  if (q >= Q) return;
  const float* src = Pq + q * ldq;
  float* dst = Pc + q * (int64_t)K * d;
  for (int i = lane; i < K * d; i += 32) {
    int j = i % d;
    dst[i] = src[i] - (mu ? mu[j] : 0.0f);
  }
  __syncwarp();
  float* qp = qpar + q * (int64_t)qpar_stride(K);
  float dmax = 0.0f, pmax = 0.0f;
  int o = K;
  for (int k = 0; k < K; ++k) {
    for (int l = k; l < K; ++l) {
      float acc = 0.0f, dkl = 0.0f;
      for (int j = lane; j < d; j += 32) {
        float a = dst[k * d + j], b = dst[l * d + j];
        acc = fmaf(a, b, acc);
        dkl = fmaf(a - b, a - b, dkl);
      }
      acc = warp_sum(acc);
      dkl = warp_sum(dkl);
      dmax = fmaxf(dmax, dkl);
      if (k == l) pmax = fmaxf(pmax, acc);
      if (lane == 0) {
        if (k == l) { qp[k] = CFL_LOG2E * acc; qp[o] = 0.5f * acc; sN[w][k] = acc; }
        else qp[o + l - k] = acc;
        sD[w][k][l] = dkl; sD[w][l][k] = dkl;
      }
    }
    o += K - k;
  }
  // slack of the lower bound, padded against fp32 rounding of the Gram form
  if (lane == 0) {
    qp[K + qpar_tri(K)] = 0.5f * (1.0f - 1.0f / K) * dmax * 1.0001f + 1e-5f * pmax;
    for (int i = K + qpar_tri(K) + 1; i < qpar_stride(K); ++i) qp[i] = 0.0f;
  }
  if (lane != 0 || qplane == nullptr) return;
  // ---- plane bound: invert the (scaled) KKT matrix [D/dmax 1; 1^T 0] in fp64 ----
  float* pl = qplane + q * (int64_t)qplane_stride(K);
  for (int i = 0; i < qplane_stride(K); ++i) pl[i] = 0.0f;
  if (K < 2) {                                               // K = 1: dist = |e|^2 + |p|^2 - 2 g exactly
    pl[0] = sN[w][0] * (1.0f - CFL_PLANE_REL);
    return;
  }
  const int ci = 2 * (K - 1) + qplane_tri(K);
  const float NEG_INF = __int_as_float(0xff800000);
  pl[ci] = NEG_INF;
  if (!(dmax > 0.0f)) return;
  const int n = K + 1;
  double M[9][18];
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < n; ++j) {
      double v = (i < K && j < K) ? (double)sD[w][i][j] / (double)dmax : ((i < K) != (j < K) ? 1.0 : 0.0);
      M[i][j] = v;
      M[i][n + j] = (i == j) ? 1.0 : 0.0;
    }
  for (int c = 0; c < n; ++c) {
    int piv = c;
    for (int r = c + 1; r < n; ++r) if (fabs(M[r][c]) > fabs(M[piv][c])) piv = r;
    if (fabs(M[piv][c]) < 1e-6) return;                       // prototypes affinely dependent
    if (piv != c) for (int j = 0; j < 2 * n; ++j) { double t = M[c][j]; M[c][j] = M[piv][j]; M[piv][j] = t; }
    const double inv = 1.0 / M[c][c];
    for (int j = 0; j < 2 * n; ++j) M[c][j] *= inv;
    for (int r = 0; r < n; ++r) {
      if (r == c) continue;
      const double f = M[r][c];
      if (f != 0.0) for (int j = 0; j < 2 * n; ++j) M[r][j] -= f * M[c][j];
    }
  }
  // inverse = M[:, n:]: A' (K x K), a' (last column), alpha' (corner); A = A'/dmax, alpha = alpha'*dmax
  double amax = 0.0;
  for (int i = 0; i < K; ++i) {
    for (int j = 0; j < K; ++j) amax = fmax(amax, fabs(M[i][n + j]));
    amax = fmax(amax, fabs(M[i][n + K]));
  }
  if (!(amax < 1.0e3)) return;                                // ill-conditioned: leave the bound off
  const double n0 = (double)sN[w][0];
  double nmax = 0.0;
  for (int k = 0; k < K; ++k) nmax = fmax(nmax, (double)sN[w][k]);
  for (int j = 1; j < K; ++j) {
    pl[j - 1] = (float)(-0.5 * ((double)sN[w][j] - n0));
    pl[K - 1 + j - 1] = (float)(-2.0 * M[j][n + K]);
  }
  int oo = 2 * (K - 1);
  for (int i = 1; i < K; ++i) {
    for (int j = i; j < K; ++j)
      pl[oo + j - i] = (float)((i == j ? 2.0 : 4.0) * M[i][n + j] / (double)dmax);
    oo += K - i;
  }
  const double alpha = M[K][n + K] * (double)dmax;
  const double margin = (double)CFL_PLANE_REL * (nmax + fabs(0.5 * alpha) + (double)dmax);
  pl[ci] = (float)(0.5 * alpha + n0 - margin);
}

int score_prep_queries_launch(const float* Pq, int64_t Q, int K, int d, int64_t ldq, const float* mu, float* Pc,
                              float* qpar, float* qplane, cudaStream_t st) {
  prep_queries_kernel<<<(unsigned)((Q + 3) / 4), 128, 0, st>>>(Pq, Q, K, d, ldq, mu, Pc, qpar, qplane);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

// ---- query prep of the source-catalog call: centred target embeddings [Q,d] and |e_q - mu|^2 ------------------------
__global__ void prep_source_queries_kernel(const float* __restrict__ Eq, int64_t Q, int d, int64_t ldq,
                                           const float* __restrict__ mu, float* __restrict__ Ec,
                                           float* __restrict__ e2q) {
  const int64_t q = (int64_t)blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
  const int lane = threadIdx.x & 31;
  if (q >= Q) return;
  float acc = 0.0f;
  for (int j = lane; j < d; j += 32) {
    const float v = Eq[q * ldq + j] - (mu ? mu[j] : 0.0f);
    Ec[q * d + j] = v;
    acc = fmaf(v, v, acc);
  }
  acc = warp_sum(acc);
  if (lane == 0) e2q[q] = acc;
}

int score_prep_source_queries_launch(const float* Eq, int64_t Q, int d, int64_t ldq, const float* mu, float* Ec,
                                     float* e2q, cudaStream_t st) {
  prep_source_queries_kernel<<<(unsigned)((Q + 3) / 4), 128, 0, st>>>(Eq, Q, d, ldq, mu, Ec, e2q);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

// ---- CUDA-core scoring kernel ---------------------------------------------------------------
template <int K>
__global__ void __launch_bounds__(SIMT_THREADS)
score_simt_kernel(ScoreArgs A) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int d = A.d;
  const int ldt = d + 1;
  tkey_t* scratch = (tkey_t*)smem_raw;                                  // [4][512]
  float* et = (float*)(scratch + (SIMT_THREADS / 32) * TOPK_CAP);      // [128][d+1]
  float* pc = et + 128 * ldt;                                         // [QT][K][d]
  float* qp = pc + SIMT_QT * K * d;                                   // [QT][K+K*K]
  float* thr = qp + SIMT_QT * qpar_stride(K);                          // [QT]
  int* cnt = (int*)(thr + SIMT_QT);                                   // [QT]

  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int part = blockIdx.x;
  const int64_t q0 = (int64_t)blockIdx.y * SIMT_QT;
  const int nq = (int)((A.Q - q0 < SIMT_QT) ? (A.Q - q0) : SIMT_QT);
  for (int i = tid; i < nq * K * d; i += SIMT_THREADS) pc[i] = A.Pc[q0 * K * d + i];
  for (int i = tid; i < nq * qpar_stride(K); i += SIMT_THREADS) qp[i] = A.qpar[q0 * qpar_stride(K) + i];
  if (tid < SIMT_QT) { thr[tid] = __int_as_float(0x7f800000); cnt[tid] = 0; }
  const int64_t t0 = A.plan.tiles * part / A.plan.parts;
  const int64_t t1 = A.plan.tiles * (part + 1) / A.plan.parts;
  tkey_t* kbase = A.keys + ((int64_t)part * A.Q + q0) * TOPK_STRIDE;
  __syncthreads();

  for (int64_t tile = t0; tile < t1; ++tile) {
    const int64_t r0 = tile * 128;
    for (int i = tid; i < 128 * d; i += SIMT_THREADS) {
      int r = i / d, j = i % d;
      int64_t row = r0 + r;
      float v = 0.0f;
      if (row < A.N) v = A.E[row * A.lde + j] - (A.mu ? A.mu[j] : 0.0f);
      et[r * ldt + j] = v;
    }
    __syncthreads();
    const int64_t row = r0 + tid;
    const float* er = et + tid * ldt;
    float e2 = 0.0f;
    for (int j = 0; j < d; ++j) e2 = fmaf(er[j], er[j], e2);
    for (int ql = 0; ql < nq; ++ql) {
      float g[K];
#pragma unroll
      for (int k = 0; k < K; ++k) g[k] = 0.0f;
      const float* pq = pc + ql * K * d;
      for (int j = 0; j < d; ++j) {
        float e = er[j];
#pragma unroll
        for (int k = 0; k < K; ++k) g[k] = fmaf(e, pq[k * d + j], g[k]);
      }
      float dist = softmin_from_gram<K>(g, e2, qp + ql * qpar_stride(K));
      if (row < A.N) {
        if (A.dist_out) A.dist_out[(q0 + ql) * A.N + row] = dist;
        if (dist < thr[ql]) {
          int slot = atomicAdd(&cnt[ql], 1);
          kbase[(int64_t)ql * TOPK_STRIDE + slot] = pack_key(dist, (uint32_t)row);
        }
      }
    }
    __syncthreads();
    for (int ql = wid; ql < nq; ql += SIMT_THREADS / 32) {
      int n = cnt[ql];
      if (n > TOPK_TRIGGER) {
        int nk = warp_compact(kbase + (int64_t)ql * TOPK_STRIDE, n, A.plan.kk,
                              scratch + wid * TOPK_CAP, lane, &thr[ql]);
        if (lane == 0) cnt[ql] = nk;
      }
    }
    __syncthreads();
  }
  for (int ql = wid; ql < nq; ql += SIMT_THREADS / 32) {
    int nk = warp_compact(kbase + (int64_t)ql * TOPK_STRIDE, cnt[ql], A.plan.kk,
                          scratch + wid * TOPK_CAP, lane, nullptr);
    if (lane == 0) A.counts[(int64_t)part * A.Q + q0 + ql] = nk;
  }
}

static size_t simt_smem_bytes(int K, int d) {
  return (size_t)(SIMT_THREADS / 32) * TOPK_CAP * sizeof(tkey_t) + (size_t)128 * (d + 1) * 4 +
         (size_t)SIMT_QT * K * d * 4 + (size_t)SIMT_QT * qpar_stride(K) * 4 + SIMT_QT * 8 + 64;
}

template <int K>
static int launch_simt(const ScoreArgs& a, cudaStream_t st) {
  size_t smem = simt_smem_bytes(K, a.d);
  CFL_CUDA(cudaFuncSetAttribute(score_simt_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)smem));
  dim3 grid(a.plan.parts, a.plan.nqt);
  score_simt_kernel<K><<<grid, SIMT_THREADS, smem, st>>>(a);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

// ---- merge of the catalog parts + direct-form rescoring + final sort ---------------------
// Exact distance of the kk survivors in direct-difference form (pcd_direct, direct.cuh: the arithmetic of
// cfl/models/base.py:129-138) on the raw rows, then (value, index) order, best k written out.
template <int K>
__global__ void __launch_bounds__(MRG_THREADS, 8)            // 32 registers: eight blocks per SM
merge_rescore_kernel(const tkey_t* __restrict__ keys, const int* __restrict__ counts, int parts, int64_t Q, int kk, int k,
                     const float* __restrict__ Pq, int64_t ldq, int d, const float* __restrict__ E, int64_t lde,
                     int64_t idx_base, float* __restrict__ top_val, int64_t* __restrict__ top_idx,
                     const float* __restrict__ only_redo,
                     // compact exact redo: blocks [Q, Q + cq) merge the compact tile's slots (own buffers, query map)
                     int cq, const tkey_t* __restrict__ ckeys, const int* __restrict__ ccounts, int cparts,
                     const float* __restrict__ cthr, const int* __restrict__ cmap) {
  __shared__ tkey_t s[TOPK_CAP];
  __shared__ int s_fill;
  __shared__ tkey_t s_thr;
  const int t = threadIdx.x;
  int64_t qk = blockIdx.x;                                  // position in the key buffers
  int64_t q = qk;                                           // the query it stands for
  if (qk >= Q) {
    qk -= Q;
    if (!(cthr[qk] > __int_as_float(0xff800000))) return;
    q = cmap[qk];
    keys = ckeys; counts = ccounts; parts = cparts; Q = cq;
  } else if (only_redo != nullptr && !(only_redo[qk] > __int_as_float(0xff800000))) {
    return;                                                 // second merge after a lower-bound pass: only the redone queries
  }
  const int fill = block_merge_topkk(keys, counts, parts, Q, qk, kk, s, &s_fill, &s_thr);
  const float* pq = Pq + q * ldq;
  if (t < fill) {
    const uint32_t idx = (uint32_t)(s[t] & 0xffffffffu);
    const float* e = E + (int64_t)idx * lde;
    const float dist = pcd_direct<K, 1>([&](int j) { return e[j]; }, [&](int kq, int j) { return pq[kq * d + j]; }, d);
    s[t] = pack_key(dist, idx);
  }
  __syncthreads();
  if (t == 0) s_fill = fill;
  __syncthreads();
  mrg_compact(s, &s_fill, &s_thr, kk, t);           // re-sort by the exact values
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

// The merge of cfl_score_topk_source (no lower-bound pass, no compact redo): the query row Eq[q] is the embedding e and
// catalog row Pc[idx] holds the K prototypes p of the direct form.
template <int K>
__global__ void __launch_bounds__(MRG_THREADS, 8)
merge_rescore_src_kernel(const tkey_t* __restrict__ keys, const int* __restrict__ counts, int parts, int64_t Q, int kk,
                         int k, const float* __restrict__ Eq, int64_t ldq, int d, const float* __restrict__ Pc, int64_t ldp,
                         int64_t idx_base, float* __restrict__ top_val, int64_t* __restrict__ top_idx) {
  __shared__ tkey_t s[TOPK_CAP];
  __shared__ int s_fill;
  __shared__ tkey_t s_thr;
  const int t = threadIdx.x;
  const int64_t q = blockIdx.x;
  const int fill = block_merge_topkk(keys, counts, parts, Q, q, kk, s, &s_fill, &s_thr);
  const float* e = Eq + q * ldq;
  if (t < fill) {
    const uint32_t idx = (uint32_t)(s[t] & 0xffffffffu);
    const float* p = Pc + (int64_t)idx * ldp;
    const float dist = pcd_direct<K, 1>([&](int j) { return e[j]; }, [&](int kq, int j) { return p[kq * d + j]; }, d);
    s[t] = pack_key(dist, idx);
  }
  __syncthreads();
  if (t == 0) s_fill = fill;
  __syncthreads();
  mrg_compact(s, &s_fill, &s_thr, kk, t);
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

// ---- merge after the lower-bound filter pass: EVERY surviving row is scored exactly -------------
// The keys of score_lb_kernel carry a lower bound, not the distance, so nothing may be discarded before its exact value
// is known.  Stage 1 (all survivors): each warp takes 32 survivors per round and gathers their rows RSC_CH dimensions
// at a time (16-byte loads, eight rows' segments per instruction) into its own slice of shared memory; every thread then
// owns one row and accumulates d_k = |e - p_k|^2, from which dist = sum_k s_k d_k - sum_{k<l} s_k s_l |p_k - p_l|^2 (the
// same quantity as the direct form, SURVEY App. A.3, good to a few ulp) picks the kk best.  The gather is software
// pipelined: the loads of the next chunk -- the next round's first chunk during the last one -- are issued before the
// current chunk is computed, so they stay in flight through the arithmetic, the selection and its barriers.  Stage 2
// stages the kk best rows with all threads and rescores them in the direct-difference form (pcd_direct), then sorts by
// (value, index), exactly as merge_rescore_kernel does.
constexpr int RSC_CH = 32;                 // dimensions per gathered chunk: 8 float4 per thread for the warp's 32 rows
constexpr int RSC_LD = RSC_CH + 4;         // row stride in floats: 16 B aligned, conflict-free LDS.128 / STS.128
constexpr int RSC_CAP = 2 * TOPK_CAP;      // candidate keys under the admission bound

// Row of the survivor f (0 when f >= total): the list p with s_pref[p] <= f < s_pref[p + 1], by binary search.
// Lists 0..parts-1 are the part buffers, list `parts` is the query's spill list.
__device__ __forceinline__ uint32_t rsc_row(int f, int total, const int* s_pref, int parts, const tkey_t* __restrict__ keys,
                                            const tkey_t* __restrict__ spill, int64_t Q, int64_t q) {
  if (f >= total) return 0u;
  int lo = 0, hi = parts;
  while (lo < hi) {
    const int m = (lo + hi) >> 1;
    if (s_pref[m + 1] <= f) lo = m + 1; else hi = m;
  }
  const tkey_t* src = (lo < parts) ? keys + ((int64_t)lo * Q + q) * TOPK_STRIDE : spill + q * (int64_t)LB_SPILL;
  return (uint32_t)(src[f - s_pref[lo]] & 0xffffffffu);
}

// Loads dimensions [c0, c0 + RSC_CH) of the warp's 32 rows (row r of the warp = the row of lane r): instruction i reads
// float4 (lane & 7) of row 4i + (lane >> 3).  Without 16-byte aligned rows (vec = false) the same elements come in
// 4-byte loads.  Dimensions >= d read as 0.
__device__ __forceinline__ void rsc_load(float4 (&v)[RSC_CH / 4], const float* __restrict__ E, int64_t lde, int d, bool vec,
                                         uint32_t idx, int c0, int lane) {
  const int j = c0 + 4 * (lane & 7);
#pragma unroll
  for (int i = 0; i < RSC_CH / 4; ++i) {
    const uint32_t r = __shfl_sync(0xffffffffu, idx, 4 * i + (lane >> 3));
    const float* e = E + (int64_t)r * lde + j;
    if (vec) {
      v[i] = (j < d) ? __ldg((const float4*)e) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    } else {
      v[i] = make_float4(j < d ? __ldg(e) : 0.0f, j + 1 < d ? __ldg(e + 1) : 0.0f, j + 2 < d ? __ldg(e + 2) : 0.0f,
                         j + 3 < d ? __ldg(e + 3) : 0.0f);
    }
  }
}

// The kk best of the candidate buffer, sorted ascending; the sort covers the smallest of TOPK_CAP, RSC_CAP keys that
// holds the fill.  Same result and admission bound as mrg_compact.
__device__ __forceinline__ void rsc_compact(tkey_t* s, int* s_fill, tkey_t* s_thr, int kk, int t) {
  const int fill = *s_fill;
  if (fill <= TOPK_CAP) {
    mrg_compact(s, s_fill, s_thr, kk, t);
    return;
  }
  for (int i = fill + t; i < RSC_CAP; i += MRG_THREADS) s[i] = CFL_KEY_INF;
  __syncthreads();
  coop_sort_generic<MRG_THREADS, RSC_CAP>(s, t);   // ends with a block barrier
  if (t == 0) {
    const int nf = fill < kk ? fill : kk;
    *s_fill = nf;
    if (nf >= kk) *s_thr = s[kk - 1];
  }
  __syncthreads();
}

template <int K>
__global__ void __launch_bounds__(MRG_THREADS, 2)            // <= 128 registers: two blocks per SM (at three, K >= 2 spills)
rescore_merge_kernel(const tkey_t* __restrict__ keys, const int* __restrict__ counts, int parts, int64_t Q,
                     int kk, int k, const float* __restrict__ Pq, int64_t ldq, int d,
                     const float* __restrict__ E, int64_t lde, int64_t idx_base,
                     float* __restrict__ top_val, int64_t* __restrict__ top_idx,
                     const float* __restrict__ tau, const float* __restrict__ tau_opt, int qt,
                     float* __restrict__ thr_redo, int* __restrict__ redo_tile, unsigned long long* __restrict__ stats,
                     const tkey_t* __restrict__ spill, const int* __restrict__ spill_cnt,
                     const float* __restrict__ only_redo, const float* __restrict__ prev_redo,
                     float* __restrict__ second_round) {
  extern __shared__ __align__(16) float s_dyn[];
  // Second round (only_redo != NULL): only the queries whose optimistic threshold was not confirmed, filtered again
  // under the safe threshold (the caller passes tau as tau_opt).  Every other query keeps the first round's verdict
  // (prev_redo: -inf = done, else the threshold of its exact redo).
  if (only_redo != nullptr && !(only_redo[blockIdx.x] > __int_as_float(0xff800000))) {
    if (threadIdx.x == 0) {
      const float pr = prev_redo[blockIdx.x];
      thr_redo[blockIdx.x] = pr;
      if (pr > __int_as_float(0xff800000)) {
        redo_tile[blockIdx.x / qt] = 1;
        if (stats) atomicAdd(&stats[STAT_EXACT_REDO_QUERIES], 1ull);
      }
    }
    return;
  }
  const int dp = (d + RSC_CH - 1) / RSC_CH * RSC_CH;        // d padded to whole chunks
  float* s_pq = s_dyn;                                       // [K][dp], zero padded
  float* s_rows = s_pq + K * dp;                             // stage 1: [warps][32][RSC_LD]; stage 2: [rows][dp + 1]
  int* s_pref = (int*)(s_rows + (MRG_THREADS / 32) * 32 * RSC_LD);   // [parts + 2]
  __shared__ tkey_t s[RSC_CAP];
  __shared__ int s_fill;
  __shared__ tkey_t s_thr;
  __shared__ float s_D[K * K];
  const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
  const int64_t q = blockIdx.x;
  for (int i = t; i < K * dp; i += MRG_THREADS) {
    const int kq = i / dp, j = i % dp;
    s_pq[i] = (j < d) ? Pq[q * ldq + kq * d + j] : 0.0f;
  }
  __shared__ int s_over, s_redo;
  if (t == 0) {
    // under an optimistic threshold only rows with dist <= tau_opt can be in a VERIFIED top-kk
    s_fill = 0;
    s_thr = (tau_opt[q] < tau[q]) ? pack_key(tau_opt[q] * (1.0f + 1e-5f) + 1e-30f, 0u) : CFL_KEY_INF;
    int acc = 0, over = 0;
    for (int p = 0; p < parts; ++p) {
      s_pref[p] = acc;
      int c = counts[(int64_t)p * Q + q];
      if (c < 0) { over = 1; c = 0; }                          // the filter pass declined (fp16 range): exact redo
      // (keys beyond a full part buffer went to the query's spill list; only ITS overflow loses keys)
      acc += c > TOPK_STRIDE ? TOPK_STRIDE : c;
    }
    s_pref[parts] = acc;                                     // list `parts` = this query's spill list
    int sc = spill_cnt[q];
    over |= sc > LB_SPILL;
    acc += sc > LB_SPILL ? LB_SPILL : sc;
    s_pref[parts + 1] = acc;
    s_over = over;
  }
  __syncthreads();
  for (int i = t; i < K * K; i += MRG_THREADS) {
    const int a = i / K, b = i % K;
    float acc = 0.0f;
    for (int j = 0; j < d; ++j) { const float df = s_pq[a * dp + j] - s_pq[b * dp + j]; acc = fmaf(df, df, acc); }
    s_D[i] = acc;
  }
  const int total = s_pref[parts + 1];
  const bool vec = (d % 4 == 0) && (lde % 4 == 0) && ((reinterpret_cast<uintptr_t>(E) & 15u) == 0);
  float* my_rows = s_rows + wid * 32 * RSC_LD;
  // round r: thread t scores survivor f = 256 r + t; idx / nidx are the rows of this round and the next
  int f = t;
  uint32_t idx = rsc_row(f, total, s_pref, parts, keys, spill, Q, q);
  uint32_t nidx = rsc_row(f + MRG_THREADS, total, s_pref, parts, keys, spill, Q, q);
  float4 v[RSC_CH / 4];
  if (f - lane < total) rsc_load(v, E, lde, d, vec, idx, 0, lane);
  __syncthreads();                                           // s_D
  for (int base = 0; base < total; base += MRG_THREADS, f += MRG_THREADS) {
    float dk[K];
#pragma unroll
    for (int kq = 0; kq < K; ++kq) dk[kq] = 0.0f;
    if (f - lane < total) {                                  // the warp has survivors this round (warp-uniform)
      for (int c0 = 0; c0 < dp; c0 += RSC_CH) {
        __syncwarp();
#pragma unroll
        for (int i = 0; i < RSC_CH / 4; ++i)
          *(float4*)(my_rows + (4 * i + (lane >> 3)) * RSC_LD + 4 * (lane & 7)) = v[i];
        __syncwarp();
        if (c0 + RSC_CH < dp) rsc_load(v, E, lde, d, vec, idx, c0 + RSC_CH, lane);
        else if (f - lane + MRG_THREADS < total) rsc_load(v, E, lde, d, vec, nidx, 0, lane);
        const float4* er = (const float4*)(my_rows + lane * RSC_LD);
#pragma unroll
        for (int j4 = 0; j4 < RSC_CH / 4; ++j4) {
          const float4 e4 = er[j4];
#pragma unroll
          for (int kq = 0; kq < K; ++kq) {
            const float4 p4 = *(const float4*)(s_pq + kq * dp + c0 + j4 * 4);
            const float a0 = e4.x - p4.x, a1 = e4.y - p4.y, a2 = e4.z - p4.z, a3 = e4.w - p4.w;
            dk[kq] = fmaf(a3, a3, fmaf(a2, a2, fmaf(a1, a1, fmaf(a0, a0, dk[kq]))));
          }
        }
      }
    }
    const uint32_t row = idx;
    idx = nidx;
    nidx = rsc_row(f + 2 * MRG_THREADS, total, s_pref, parts, keys, spill, Q, q);
    float dist = dk[0];
    if (K > 1) {
      float mn = dk[0];
#pragma unroll
      for (int kq = 1; kq < K; ++kq) mn = fminf(mn, dk[kq]);
      float w[K], sum = 0.0f;
#pragma unroll
      for (int kq = 0; kq < K; ++kq) { w[kq] = __expf(mn - dk[kq]); sum += w[kq]; }
      const float inv = 1.0f / sum;
      float lin = 0.0f, quad = 0.0f;
#pragma unroll
      for (int a = 0; a < K; ++a) {
        lin = fmaf(w[a], dk[a], lin);
#pragma unroll
        for (int b = a + 1; b < K; ++b) quad = fmaf(w[a] * w[b], s_D[a * K + b], quad);
      }
      dist = inv * (lin - inv * quad);
    }
    // selection protocol of block_merge_topkk: uniform branch on the fill level read between barriers
    const int f0 = s_fill;
    __syncthreads();
    if (f0 + MRG_THREADS > RSC_CAP) rsc_compact(s, &s_fill, &s_thr, kk, t);
    if (f < total) {
      const tkey_t key = pack_key(dist, row);
      if (key < s_thr) s[atomicAdd(&s_fill, 1)] = key;
    }
    __syncthreads();
  }
  rsc_compact(s, &s_fill, &s_thr, kk, t);
  const int fill = s_fill;
  // Verification.  The filter kept every row whose LOWER BOUND is under the threshold, so a key count
  // proves nothing; the exact values do: if kk survivors have dist <= tau_opt, no row outside the
  // survivor set (all of which have dist >= bound > tau_opt) can belong to the top-kk.  Under the safe
  // threshold (tau_opt == tau) the survivor set always contains the top-kk.  Otherwise -- or when a
  // key buffer overflowed -- the query is handed to the exact kernel (thr_redo / redo_tile).
  if (t == 0) {
    const bool optimistic = tau_opt[q] < tau[q];
    const bool proven = !optimistic || (fill >= kk && ord2f((uint32_t)(s[kk - 1] >> 32)) <= tau_opt[q] * (1.0f - 4e-6f));
    const int redo = (s_over || !proven) ? 1 : 0;
    s_redo = redo;
    thr_redo[q] = redo ? tau[q] : __int_as_float(0xff800000);
    if (redo) redo_tile[q / qt] = 1;
    // a second lower-bound round can help only when the optimistic threshold was the problem: not for overflowing
    // buffers, raised range flags or queries the probe took out (tau_opt = -inf)
    if (second_round)
      second_round[q] = (redo && !s_over && tau_opt[q] > __int_as_float(0xff800000)) ? tau[q] : __int_as_float(0xff800000);
    if (stats && only_redo != nullptr && redo) atomicAdd(&stats[STAT_EXACT_REDO_QUERIES], 1ull);
    if (stats && only_redo == nullptr) {                     // statistics of the call (cfl_score_topk_stats)
      atomicAdd(&stats[STAT_SURVIVORS], (unsigned long long)total);
      if (spill_cnt[q] > 0) atomicAdd(&stats[STAT_SPILL_QUERIES], 1ull);
      if (!(tau_opt[q] > __int_as_float(0xff800000))) atomicAdd(&stats[STAT_PROBE_DROPPED_QUERIES], 1ull);
      if (redo) atomicAdd(&stats[STAT_REDO_QUERIES], 1ull);
      if (q == 0) stats[STAT_LOWER_BOUND_PASS] = 1ull;
    }
  }
  __syncthreads();
  if (s_redo) return;
  {                                                          // stage 2: direct form for the kk survivors,
    const int ld2 = dp + 1;                                  // rows staged in full (stride dp+1: conflict-free)
    const int nst = ((MRG_THREADS / 32) * 32 * RSC_LD) / ld2;  // rows the staging area holds at once
    if (nst > 0) {
      for (int r0 = 0; r0 < fill; r0 += nst) {
        const int nr = (fill - r0 < nst) ? fill - r0 : nst;
        // every thread loads: element i of the nr x (dp / 4) float4 grid, eight loads in flight before the stores
        const int n4 = dp / 4, ne = nr * n4;
        for (int i0 = 0; i0 < ne; i0 += 8 * MRG_THREADS) {
          float4 w4[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int i = i0 + u * MRG_THREADS + t;
            const int rr = i / n4, j = 4 * (i - rr * n4);
            w4[u] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
            if (i < ne && j < d) {
              const float* e = E + (int64_t)(uint32_t)(s[r0 + rr] & 0xffffffffu) * lde + j;
              if (vec) w4[u] = __ldg((const float4*)e);
              else w4[u] = make_float4(__ldg(e), j + 1 < d ? __ldg(e + 1) : 0.0f, j + 2 < d ? __ldg(e + 2) : 0.0f,
                                       j + 3 < d ? __ldg(e + 3) : 0.0f);
            }
          }
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int i = i0 + u * MRG_THREADS + t;
            const int rr = i / n4, j = 4 * (i - rr * n4);
            if (i < ne) {
              float* o = s_rows + rr * ld2 + j;
              o[0] = w4[u].x; o[1] = w4[u].y; o[2] = w4[u].z; o[3] = w4[u].w;
            }
          }
        }
        __syncthreads();
        float dist = 0.0f;
        uint32_t ridx = 0u;
        if (t < nr) {
          ridx = (uint32_t)(s[r0 + t] & 0xffffffffu);
          const float* er = s_rows + t * ld2;
          dist = pcd_direct<K>([&](int j) { return er[j]; }, [&](int kq, int j) { return s_pq[kq * dp + j]; }, d);
        }
        __syncthreads();                                     // staged rows and keys read
        if (t < nr) s[r0 + t] = pack_key(dist, ridx);
      }
    } else {                                                 // very wide rows: straight from global memory
      for (int kidx = t; kidx < fill; kidx += MRG_THREADS) {
        const uint32_t ridx = (uint32_t)(s[kidx] & 0xffffffffu);
        const float* er = E + (int64_t)ridx * lde;
        const float dist = pcd_direct<K>([&](int j) { return er[j]; }, [&](int kq, int j) { return s_pq[kq * dp + j]; }, d);
        s[kidx] = pack_key(dist, ridx);
      }
    }
  }
  __syncthreads();
  if (t == 0) s_fill = fill;
  __syncthreads();
  mrg_compact(s, &s_fill, &s_thr, kk, t);
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

// ---- thresholds from the sample pass ------------------------------------------------------
// tau[q] = kk-th smallest distance among the sampled candidates of ALL parts.  Any subset's kk-th
// best is an upper bound of the catalog's kk-th best, so every member of the final top-kk
// satisfies dist <= tau[q].  The optimistic bound tau_opt[q] is the r_opt-th best of the 1/S sample: about r_opt*S
// candidates of the whole range lie under it -- several times kk, but not guaranteed (the verification checks).
// Radix selection: only the VALUES of the kk-th and r_opt-th
// smallest distances are needed, so four 8-bit passes over the 32-bit ordered distances (staged in
// shared memory when they fit) replace the ~20 cooperative sorts of block_merge_topkk.
constexpr int SEL_THREADS = 1024;              // few blocks (one per query) when Q is small: they must be wide
constexpr int SEL_SMEM_KEYS = 24576;            // 148 parts x kk keys of an adaptive sample pass fit (96 KB)

__device__ __forceinline__ uint32_t radix_select(const uint32_t* __restrict__ sv, const tkey_t* __restrict__ keys,
                                                 const int* __restrict__ s_pref, int parts, int64_t Q, int64_t q,
                                                 int total, bool in_smem, int rank, int* hist, int* s_sel) {
  // rank is 1-based; returns the ordered-uint value of the rank-th smallest
  const int t = threadIdx.x, nt = blockDim.x;
  uint32_t prefix = 0, mask = 0;
  int want = rank;
  for (int shift = 24; shift >= 0; shift -= 8) {
    for (int i = t; i < 256; i += nt) hist[i] = 0;
    __syncthreads();
    if (in_smem) {
      for (int i = t; i < total; i += nt) {
        const uint32_t v = sv[i];
        if ((v & mask) == prefix) atomicAdd(&hist[(v >> shift) & 255u], 1);
      }
    } else {
      for (int p = 0; p < parts; ++p) {
        const int c = s_pref[p + 1] - s_pref[p];
        const tkey_t* src = keys + ((int64_t)p * Q + q) * TOPK_STRIDE;
        for (int i = t; i < c; i += nt) {
          const uint32_t v = (uint32_t)(src[i] >> 32);
          if ((v & mask) == prefix) atomicAdd(&hist[(v >> shift) & 255u], 1);
        }
      }
    }
    __syncthreads();
    if (t < 32) {                                            // warp 0: find the bin holding the want-th key
      int loc[8], sum = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) { loc[j] = hist[t * 8 + j]; sum += loc[j]; }
      int incl = sum;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const int n = __shfl_up_sync(0xffffffffu, incl, o); if (t >= o) incl += n; }
      const int excl = incl - sum;
      if (want > excl && want <= incl) {
        int acc = excl;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (want > acc && want <= acc + loc[j]) { s_sel[0] = t * 8 + j; s_sel[1] = want - acc; }
          acc += loc[j];
        }
      }
    }
    __syncthreads();
    prefix |= (uint32_t)s_sel[0] << shift;
    mask |= 255u << shift;
    want = s_sel[1];
    __syncthreads();
  }
  return prefix;
}

__global__ void __launch_bounds__(SEL_THREADS)
select_threshold_kernel(const tkey_t* __restrict__ keys, const int* __restrict__ counts, int parts,
                        int64_t Q, int kk, float* __restrict__ tau, float* __restrict__ tau_opt, int r_opt, int smem_keys) {
  extern __shared__ uint32_t s_sel_dyn[];
  int* s_pref = (int*)s_sel_dyn;                             // [parts + 1]
  uint32_t* sv = s_sel_dyn + parts + 1;                      // [smem_keys]
  __shared__ int hist[256];
  __shared__ int s_sel[2];
  const int t = threadIdx.x;
  const int64_t q = blockIdx.x;
  if (t == 0) {
    int acc = 0;
    for (int p = 0; p < parts; ++p) {
      s_pref[p] = acc;
      const int c = counts[(int64_t)p * Q + q];
      acc += c > TOPK_STRIDE ? TOPK_STRIDE : (c < 0 ? 0 : c);
    }
    s_pref[parts] = acc;
  }
  __syncthreads();
  const int total = s_pref[parts];
  const float INF = __int_as_float(0x7f800000);
  if (total < kk) {
    if (t == 0) { tau[q] = INF; if (tau_opt) tau_opt[q] = INF; }
    return;
  }
  const bool in_smem = total <= smem_keys;
  if (in_smem) {
    for (int p = 0; p < parts; ++p) {
      const int c = s_pref[p + 1] - s_pref[p];
      const tkey_t* src = keys + ((int64_t)p * Q + q) * TOPK_STRIDE;
      for (int i = t; i < c; i += blockDim.x) sv[s_pref[p] + i] = (uint32_t)(src[i] >> 32);
    }
    __syncthreads();
  }
  const uint32_t vk = radix_select(sv, keys, s_pref, parts, Q, q, total, in_smem, kk, hist, s_sel);
  const float safe = ord2f(vk);
  float opt = safe;
  if (tau_opt && r_opt >= 1 && r_opt < kk)
    opt = ord2f(radix_select(sv, keys, s_pref, parts, Q, q, total, in_smem, r_opt, hist, s_sel));
  if (t == 0) { tau[q] = safe; if (tau_opt) tau_opt[q] = opt; }
}

// Probe of the lower-bound filter: score_lb_kernel over a few tiles per part under tau_opt.  A query
// whose projected number of survivors over the whole range would swamp its key buffers (prototypes
// nearly affinely dependent, or so far apart that the soft-min is one-hot: the affine-hull bound is
// off or loose) is taken out of the lower-bound pass (tau_opt = -inf: nothing is pushed, verification
// fails, the exact kernel redoes it) -- and a query tile with no live query costs nothing there.
__global__ void probe_classify_kernel(const int* __restrict__ counts, int parts, int64_t Q, float scale,
                                      float limit, float* __restrict__ tau_opt, const int* __restrict__ spill_cnt) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= Q) return;
  long long tot = spill_cnt ? spill_cnt[q] : 0;
  for (int p = 0; p < parts; ++p) tot += counts[(int64_t)p * Q + q];
  if ((float)tot * scale > limit) tau_opt[q] = __int_as_float(0xff800000);
}

// After the filter pass under the optimistic thresholds: a query whose parts hold fewer than kk keys
// in total may have lost members of its top-kk; it is redone under the safe threshold.  (A part's
// count is either the number of rows it pushed or, after a compaction, still >= kk.)
__global__ void verify_counts_kernel(const int* __restrict__ counts, int parts, int64_t Q, int kk, int qt,
                                     const float* __restrict__ tau, const float* __restrict__ tau_opt,
                                     float* __restrict__ thr_redo, int* __restrict__ redo_tile,
                                     unsigned long long* __restrict__ stats) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= Q) return;
  long long tot = 0;
  bool over = false;                                         // a lower-bound pass buffer overflowed
  for (int p = 0; p < parts; ++p) {
    const int c = counts[(int64_t)p * Q + q];
    tot += c;
    over |= c > TOPK_STRIDE;
  }
  const bool redo = over || (tot < kk && tau_opt[q] < tau[q]);
  thr_redo[q] = redo ? tau[q] : __int_as_float(0xff800000);
  if (redo) redo_tile[q / qt] = 1;
  if (stats) {
    atomicAdd(&stats[STAT_SURVIVORS], (unsigned long long)tot);
    if (redo) atomicAdd(&stats[STAT_REDO_QUERIES], 1ull);
  }
}

// ---- cross-rank merge: rank-based merge of R sorted lists --------------------------------
__device__ __forceinline__ bool lex_less(float va, int64_t ia, float vb, int64_t ib) {
  return va < vb || (va == vb && (uint64_t)ia < (uint64_t)ib);
}

// vals / idx of rank r start rs_v / rs_i BYTES after those of rank r - 1 (contiguous [R,Q,k] arrays, or the gathered
// exchange records [R][idx | val] of cfl_topk_pack_records).
// exchange record of one rank: [idx: n int64][val: n float][pad to 16 bytes], n = Q * k
__host__ __device__ inline size_t topk_record_bytes(int64_t n) { return ((size_t)n * 12 + 15) / 16 * 16; }
__global__ void topk_pack_records_kernel(const float* __restrict__ vals, const int64_t* __restrict__ idx, int64_t n,
                                         char* __restrict__ rec) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  ((int64_t*)rec)[i] = idx[i];
  ((float*)(rec + (size_t)n * 8))[i] = vals[i];
}

__global__ void __launch_bounds__(128)
topk_merge_kernel(const char* __restrict__ vals_b, const char* __restrict__ idx_b, size_t rs_v, size_t rs_i, int R,
                  int64_t Q, int k, float* __restrict__ top_val, int64_t* __restrict__ top_idx) {
  const int64_t q = blockIdx.x;
  for (int e = threadIdx.x; e < R * k; e += blockDim.x) {
    int r = e / k, j = e % k;
    float v = ((const float*)(vals_b + (size_t)r * rs_v))[q * k + j];
    int64_t id = ((const int64_t*)(idx_b + (size_t)r * rs_i))[q * k + j];
    int rank = j;
    for (int r2 = 0; r2 < R; ++r2) {
      if (r2 == r) continue;
      const float* lv = (const float*)(vals_b + (size_t)r2 * rs_v) + q * k;
      const int64_t* li = (const int64_t*)(idx_b + (size_t)r2 * rs_i) + q * k;
      // r2 < r: count elements <= e ; r2 > r: count elements < e   (stable merge rank)
      int lo = 0, hi = k;
      while (lo < hi) {
        int mid = (lo + hi) >> 1;
        bool before = (r2 < r) ? !lex_less(v, id, lv[mid], li[mid]) : lex_less(lv[mid], li[mid], v, id);
        if (before) lo = mid + 1; else hi = mid;
      }
      rank += lo;
    }
    if (rank < k) { top_val[q * k + rank] = v; top_idx[q * k + rank] = id; }
  }
}

}  // namespace cfl

using namespace cfl;

// Tuning knobs of cfl_score_topk (DESIGN.md "Experiment knobs"): read from the environment in ONE place per call.
// Results never depend on them.  The ones that switch work off for timing experiments (CFL_SCORE_DBG_MODE) or force a
// path outside its validated range (CFL_SCORE_FORCE_LB) are honoured only under CFL_EXPERIMENTS=1.
struct ScoreKnobs {
  int sample_stride = 32;     // tools/knob_sweep.py: 32 beats 16 by 7 % on the C3 step (the sample pass halves; r_opt = 16)
  int64_t min_tiles = 16;     // tiles per part below which one adaptive exact pass is used (tools/small_q_probe.py: the
                              // sampled two-pass path wins from Q = 1 on a 1 M-row catalog)
  int opt_mult = 4;           // optimistic threshold = ceil(opt_mult * kk / stride)-th best of the sample
  bool no_cascade = false, no_optimistic = false, no_lb = false, no_probe = false, force_lb = false;
  int dbg_mode = 0;
};
static ScoreKnobs read_knobs() {
  ScoreKnobs k;
  const char* e;
  if ((e = getenv("CFL_SCORE_SAMPLE_STRIDE"))) k.sample_stride = atoi(e);
  if ((e = getenv("CFL_SCORE_MIN_TILES"))) k.min_tiles = atoll(e);
  if ((e = getenv("CFL_SCORE_OPT_MULT"))) k.opt_mult = atoi(e);
  k.no_cascade = getenv("CFL_SCORE_NO_CASCADE") != nullptr;
  k.no_optimistic = getenv("CFL_SCORE_NO_OPTIMISTIC") != nullptr;
  k.no_lb = getenv("CFL_SCORE_NO_LB") != nullptr;
  k.no_probe = getenv("CFL_SCORE_NO_PROBE") != nullptr;
  if ((e = getenv("CFL_EXPERIMENTS")) && atoi(e) != 0) {
    k.force_lb = getenv("CFL_SCORE_FORCE_LB") != nullptr;
    if ((e = getenv("CFL_SCORE_DBG_MODE"))) k.dbg_mode = atoi(e);
  }
  return k;
}
static bool score_two_pass(const ScoreKnobs& kn, const ScorePlan& plan, bool dense) {
  return kn.sample_stride > 1 && !dense && plan.tiles / plan.parts >= kn.min_tiles;
}
static bool score_lb_pass(const ScoreKnobs& kn, int K) {
  // the affine hull of K prototypes has K-1 dimensions: for K > 4 it swallows so much of a low-dimensional embedding
  // that the bound stops rejecting (measured: K=8 survivors overflow at d=20..64), so those shapes keep the exact
  // filter (optimistic threshold + exact counts)
  return !kn.no_lb && (K <= 4 || kn.force_lb);
}

// Compact exact redo: the (rare) queries that still need the exact kernel after the lower-bound rounds are gathered
// into ONE query tile, so that every SM works on a slice of the catalog for them -- the in-place redo below keeps a
// query in its own tile, i.e. on a few CTAs that each walk a large part of the catalog.
struct CerLayout { size_t idx, thr, flag, pc, qpar, qplane, qimg, total; };
static CerLayout cer_layout(int K, int d, int qt, int dpad) {
  CerLayout L;
  size_t off = 0;
  L.idx = off;    off = align_up(off + (size_t)qt * sizeof(int), 256);
  L.thr = off;    off = align_up(off + (size_t)qt * sizeof(float), 256);
  L.flag = off;   off = align_up(off + 16, 256);
  L.pc = off;     off = align_up(off + (size_t)qt * K * d * sizeof(float), 256);
  L.qpar = off;   off = align_up(off + (size_t)qt * qpar_stride(K) * sizeof(float), 256);
  L.qplane = off; off = align_up(off + (size_t)qt * qplane_stride(K) * sizeof(float), 1024);
  L.qimg = off;   off = align_up(off + qimg_tile_bytes(dpad, K * qt), 1024);
  L.total = off;
  return L;
}

// One block.  Takes the first `cap` flagged queries (thr[q] > -inf) in query order: idx_c / thr_c / gathered prototype
// and parameter rows; un-flags them in thr, rebuilds the per-tile flags for what is left, flag_c = "something taken".
__global__ void __launch_bounds__(256)
redo_compact_kernel(float* __restrict__ thr, int64_t Q, int cap, int K, int d, int plan_qt, int nqt,
                    const float* __restrict__ Pc, const float* __restrict__ qpar, const float* __restrict__ qplane,
                    int* __restrict__ idx_c, float* __restrict__ thr_c, int* __restrict__ flag_c,
                    float* __restrict__ Pc_c, float* __restrict__ qpar_c, float* __restrict__ qplane_c,
                    int* __restrict__ redo_tile, int dpad, float* __restrict__ qimg_c) {
  __shared__ int s_cnt[256];
  __shared__ int s_total;
  const int t = threadIdx.x;
  const float NEG_INF = __int_as_float(0xff800000);
  const int64_t per = (Q + 255) / 256;
  const int64_t lo = (int64_t)t * per, hi = lo + per < Q ? lo + per : Q;
  int mine = 0;
  for (int64_t q = lo; q < hi; ++q) mine += thr[q] > NEG_INF ? 1 : 0;
  s_cnt[t] = mine;
  for (int i = t; i < nqt; i += 256) redo_tile[i] = 0;
  for (int i = t; i < cap; i += 256) { idx_c[i] = 0; thr_c[i] = NEG_INF; }
  __syncthreads();
  if (t == 0) {
    int run = 0;
    for (int i = 0; i < 256; ++i) { const int c = s_cnt[i]; s_cnt[i] = run; run += c; }
    s_total = run;
    *flag_c = run > 0 ? 1 : 0;
  }
  __syncthreads();
  int pos = s_cnt[t];
  for (int64_t q = lo; q < hi; ++q) {
    const float v = thr[q];
    if (!(v > NEG_INF)) continue;
    if (pos < cap) { idx_c[pos] = (int)q; thr_c[pos] = v; thr[q] = NEG_INF; }
    else redo_tile[q / plan_qt] = 1;                           // left to the in-place redo
    ++pos;
  }
  __syncthreads();
  const int R = s_total < cap ? s_total : cap;
  const int qps = qpar_stride(K), pbs = qplane_stride(K), kd = K * d;
  for (int i = t; i < R * kd; i += 256) Pc_c[i] = Pc[(int64_t)idx_c[i / kd] * kd + i % kd];
  for (int i = t; i < R * qps; i += 256) qpar_c[i] = qpar[(int64_t)idx_c[i / qps] * qps + i % qps];
  for (int i = t; i < R * pbs; i += 256) qplane_c[i] = qplane[(int64_t)idx_c[i / pbs] * pbs + i % pbs];
  for (int i = R * kd + t; i < cap * kd; i += 256) Pc_c[i] = 0.0f;
  for (int i = R * qps + t; i < cap * qps; i += 256) qpar_c[i] = 0.0f;
  for (int i = R * pbs + t; i < cap * pbs; i += 256) qplane_c[i] = 0.0f;
  if (R == 0) return;                                          // the exact kernel's CTAs leave on flag_c
  __syncthreads();
  // tcgen05 B-operand image of the compact tile (the layout of pack_queries_kernel, score_umma.cu): cap = the query tile
  const int nc = K * cap, nks = dpad / 8;
  for (int e = t; e < nks * 2 * nc; e += 256) {
    const int n = e % nc, c = (e / nc) % 2, ks = e / (2 * nc);
    const int k = n / cap, ql = n % cap;
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    float* xp = &x.x;
    if (ql < R) {
      const float* src = Pc_c + ((int64_t)ql * K + k) * d;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int j = ks * 8 + c * 4 + i;
        if (j < d) xp[i] = src[j];
      }
    }
    float4 hi4, lo4;
    umma::split_tf32x4(x, hi4, lo4);
    const size_t step = (size_t)ks * 4 * nc;
    ((float4*)qimg_c)[step + (size_t)(0 * 2 + c) * nc + n] = hi4;
    ((float4*)qimg_c)[step + (size_t)(1 * 2 + c) * nc + n] = lo4;
  }
}

// Workspace of one cfl_score_topk[_packed] call under plan p: the byte offset of every region.  Only the tensor-core
// plan has the lower-bound pass's spill lists, the statistics and the compact-redo area.
struct ScoreWs {
  size_t pc, qpar, qplane;            // centred prototypes [Q,K,d]; soft-min and plane-bound blocks per query
  size_t qimg, lbimg;                 // query images of the exact kernel and of the lower-bound pass
  size_t keys, counts;                // key buffers [parts,Q,TOPK_STRIDE] and counts [parts,Q] of the larger tiling
  size_t cimg;                        // catalog image, packed here by cfl_score_topk (empty for the _packed entry)
  size_t tau, tau_opt;                // per query: safe and optimistic thresholds
  size_t thr_redo, redo_tile;         // per query: threshold of the exact redo (-inf = none); per query tile: 1 = redo
  size_t thr_redo2, redo_tile2;       // the same after the second lower-bound round
  size_t lb2;                         // per query: threshold of the second lower-bound round, -inf = none
  size_t spill, spill_cnt;            // lower-bound pass: [Q,LB_SPILL] keys that did not fit their buffer, count [Q]
  size_t stats;                       // CFL_SCORE_NSTATS counters (ScoreStat)
  size_t cer;                         // compact exact redo: cer_layout at the next 1024-byte aligned ADDRESS from here
  CerLayout cl;
  size_t total;
};

// src (cfl_score_topk_source): one vector per query (pc = [Q,d], qpar = |e_q - mu|^2, a query image of qt vectors per
// tile), no lower-bound pass (no lbimg, spill lists or compact-redo area) and never an own catalog image.
static ScoreWs score_ws(int64_t Q, int K, int d, int64_t N, const ScorePlan& p, bool own_image, bool src = false) {
  ScoreWs w = {};
  const bool lbp = p.impl && !src;
  const LbPlan lb = lbp ? make_lb_plan(Q, K, d, p.tiles) : LbPlan{0, 0, 0, 0, 0};
  const int kparts = p.parts > lb.parts ? p.parts : lb.parts;          // key buffers serve both tilings
  const int Kq = src ? 1 : K;                                          // vectors per query
  size_t off = 0;
  w.pc = off;         off = align_up(off + (size_t)Q * Kq * d * 4, 256);
  w.qpar = off;       w.qplane = off + (size_t)Q * (src ? 1 : qpar_stride(K)) * 4;
  off = align_up(off + (size_t)Q * (src ? 1 : qpar_stride(K) + qplane_stride(K)) * 4, 256);
  w.qimg = off;       off = align_up(off + (p.impl ? (size_t)p.nqt * qimg_tile_bytes(p.dpad, Kq * p.qt) : 0), 1024);
  w.lbimg = off;      off = align_up(off + (lbp ? score_lb_qimg_bytes(lb, K, d) : 0), 1024);
  w.keys = off;       off = align_up(off + (size_t)kparts * Q * TOPK_STRIDE * sizeof(tkey_t), 256);
  w.counts = off;     off = align_up(off + (size_t)kparts * Q * sizeof(int), 1024);
  w.cimg = off;       off = align_up(off + ((p.impl && own_image) ? catalog_image_bytes(N, d) : 0), 1024);
  w.tau = off;        off += (size_t)Q * sizeof(float);
  w.tau_opt = off;    off += (size_t)Q * sizeof(float);
  w.thr_redo = off;   off += (size_t)Q * sizeof(float);
  w.redo_tile = off;  off += (size_t)(p.nqt + 4) * sizeof(int);
  w.thr_redo2 = off;  off += (size_t)Q * sizeof(float);
  w.redo_tile2 = off; off += (size_t)(p.nqt + 4) * sizeof(int);
  w.lb2 = off;        off = align_up(off + (size_t)(Q + 4) * sizeof(float), 256);
  if (p.impl) {
    if (!src) {
      w.spill = off;  w.spill_cnt = off + (size_t)Q * LB_SPILL * sizeof(tkey_t);
      off = align_up(w.spill_cnt + (size_t)Q * sizeof(int), 256);
    }
    w.stats = off;    off = align_up(off + CFL_SCORE_NSTATS * sizeof(unsigned long long), 256);
    if (!src) {
      w.cl = cer_layout(K, d, p.qt, p.dpad);
      w.cer = off;    off = align_up(off + w.cl.total, 1024);
    }
  }
  w.total = off + 1024;
  return w;
}

static size_t score_ws_bytes(int64_t Q, int K, int d, int64_t N, int k, bool own_image) {
  if (Q <= 0 || N <= 0) return 4096;
  // the plan (hence the size) differs between the two kernels: take the larger
  size_t s = score_ws(Q, K, d, N, make_score_plan(Q, K, d, N, k, false), own_image).total;
  if (score_umma_qt(K, d) > 0) {
    const size_t s1 = score_ws(Q, K, d, N, make_score_plan(Q, K, d, N, k, true), own_image).total;
    if (s1 > s) s = s1;
  }
  return s + 1024;
}

// One cfl_score_topk call as its stages see it: the caller's arguments, plan, knobs, workspace, and the argument block
// of the tensor-core kernels, which the stages update as the call proceeds.
struct ScoreCall {
  const float* Pq; int64_t ldq; int k; int64_t idx_base; float* top_val; int64_t* top_idx;
  ScorePlan plan; ScoreKnobs kn; ScoreWs ws; char* base; cudaStream_t cs;
  ScoreArgs a;
  template <class T> T* at(size_t off) const { return (T*)(base + off); }
};

// What the final merge_rescore_kernel launch reads besides the call's key buffers.
struct MergeInput {
  int parts;                          // catalog parts of the key buffers
  const float* only = nullptr;        // after a lower-bound pass: only the queries with only[q] > -inf are merged
  // compact exact redo (cparts = 0: none): key buffers, counts, parts, per-slot thresholds, slot -> query map
  const tkey_t* ckeys = nullptr; const int* ccounts = nullptr; int cparts = 0;
  const float* cthr = nullptr; const int* cmap = nullptr;
};

// Stage: centred prototypes and parameter blocks; on the tensor-core plan also the catalog image (packed into the
// workspace unless the caller packed it), its views and the query images.
static int prep_and_pack(ScoreCall& c, const void* image) {
  ScoreArgs& a = c.a;
  prep_queries_kernel<<<(unsigned)((a.Q + 3) / 4), 128, 0, c.cs>>>(c.Pq, a.Q, a.K, a.d, c.ldq, a.mu, (float*)a.Pc,
                                                                   (float*)a.qpar, (float*)a.qplane);
  CFL_LAUNCH_CHECK();
  if (c.plan.impl != 1) return CFL_OK;
  if (!image) {
    void* own = c.base + c.ws.cimg;
    const int st = catalog_pack_launch(a.E, a.N, a.d, a.lde, a.mu, own, c.cs);
    if (st != CFL_OK) return st;
    image = own;
  }
  const CatalogView cv = catalog_view(image, a.N, a.d);
  a.cimg = image; a.e2 = cv.e2; a.cimg16 = cv.f16; a.cflag16 = cv.flag16; a.lbrow = cv.lbrow;
  const LbQimgView qv = score_lb_qimg_view(c.base + c.ws.lbimg, a.lb, a.K, a.d);
  a.qimg16 = qv.img; a.qflag16 = qv.flag; a.lbq = qv.lbq;
  return score_umma_pack_queries(a, c.base + c.ws.qimg, c.cs);
}

// Stage: the thresholds.  Long catalog ranges are scored in two passes: a sparse sample pass (every S-th tile) whose
// merged kk-th best distance bounds the final threshold (tau), then the full pass that only filters against a fixed
// bound (no barriers, no compaction).
static int sample_thresholds(ScoreCall& c) {
  ScoreArgs& a = c.a;
  const ScorePlan& plan = c.plan;
  const int64_t Q = a.Q;
  const int sstride = c.kn.sample_stride;
  float* tau = c.at<float>(c.ws.tau);
  // Threshold selection: one block per query.  Many queries -> narrow blocks with 32 KB of staged keys each (a whole
  // wave of them is resident; a query with more keys selects from global memory); few queries -> wide blocks that
  // stage up to 148 parts x kk keys.
  const int sel_threads = Q >= 2 * (int64_t)sm_count() ? 256 : SEL_THREADS;
  const int sel_cap = Q >= 2 * (int64_t)sm_count() ? 8192 : SEL_SMEM_KEYS;
  auto sel_keys = [&](int64_t bound) { return (int)(bound < sel_cap ? (bound < 1024 ? 1024 : bound) : sel_cap); };
  CFL_SMEM_LIMIT(select_threshold_kernel, ((size_t)plan.parts + 1 + SEL_SMEM_KEYS) * sizeof(uint32_t));
  // Sample = every sstride-th tile of each part.  When a few collect-everything tiles per
  // part already give a bound tau_a under which the sample yields <= ~384 keys per buffer,
  // the sample itself is scored in filter mode (no barriers); otherwise it runs adaptively.
  const int64_t tpp = plan.tiles / plan.parts;
  const int64_t tiles_b = (tpp + sstride - 1) / sstride;
  int64_t tiles_a = ((int64_t)plan.kk * tiles_b + 384 * (int64_t)plan.parts - 1) / (384 * (int64_t)plan.parts);
  if (tiles_a < 1) tiles_a = 1;
  // The cascade needs a pass-B sample several times larger than pass A's: tau_a (kk-th best of pass A) leaves
  // about kk * |B| / |A| rows of pass B under it, and pass B must find at least kk of them to define the
  // thresholds (with |B| ~ |A| -- short part ranges, e.g. a few queries on 148 parts -- a seventh of the queries
  // ended up without thresholds and fell through to the exact redo pass).  Pass A visits up to tiles_a + 1 tiles.
  const bool cascade = tiles_a <= 7 && tiles_a * 128 * plan.parts >= 2 * plan.kk && tiles_b >= 4 * (tiles_a + 1) &&
                       !c.kn.no_cascade;
  int st;
  if (cascade) {
    a.phase = 2; a.thr_init = nullptr;                 // +inf thresholds: keep every sampled row
    a.tile_stride = (int)((tpp + tiles_a - 1) / tiles_a);
    if (a.tile_stride < 1) a.tile_stride = 1;
    // guard: ceil(range / stride) <= 7 tiles even for the longest part range
    while ((tpp + 1 + a.tile_stride - 1) / a.tile_stride > 7) ++a.tile_stride;
    st = score_umma_launch(a, c.cs);
    if (st != CFL_OK) return st;
    const int nk = sel_keys((int64_t)plan.parts * 7 * 128);   // pass A: at most 7 tiles of 128 rows per part
    select_threshold_kernel<<<(unsigned)Q, sel_threads, ((size_t)plan.parts + 1 + nk) * sizeof(uint32_t), c.cs>>>(
        a.keys, a.counts, plan.parts, Q, plan.kk, tau, nullptr, 0, nk);
    CFL_LAUNCH_CHECK();
    a.phase = 2; a.tile_stride = sstride; a.thr_init = tau;
    st = score_umma_launch(a, c.cs);
  } else {
    a.phase = 1; a.tile_stride = sstride; a.thr_init = nullptr;
    st = score_umma_launch(a, c.cs);
  }
  if (st != CFL_OK) return st;
  // The full pass filters under an OPTIMISTIC threshold (r_opt-th best of the sample: about 4*kk rows of the whole
  // range pass instead of sstride*kk), which lets the bounds reject almost every (row, query).  Each query is then
  // verified, and the rare query that fails is redone under the safe bound.
  CFL_CUDA(cudaMemsetAsync(c.at<unsigned long long>(c.ws.stats), 0, CFL_SCORE_NSTATS * sizeof(unsigned long long), c.cs));
  int r_opt = (int)((c.kn.opt_mult * (int64_t)plan.kk + sstride - 1) / sstride);
  if (c.kn.no_optimistic) r_opt = 0;
  const int nk = sel_keys((int64_t)plan.parts * TOPK_STRIDE);
  select_threshold_kernel<<<(unsigned)Q, sel_threads, ((size_t)plan.parts + 1 + nk) * sizeof(uint32_t), c.cs>>>(
      a.keys, a.counts, plan.parts, Q, plan.kk, tau, c.at<float>(c.ws.tau_opt), r_opt, nk);
  CFL_LAUNCH_CHECK();
  CFL_CUDA(cudaMemsetAsync(c.at<int>(c.ws.redo_tile), 0, (size_t)plan.nqt * sizeof(int), c.cs));
  return CFL_OK;
}

// One round of rescore_merge_kernel over the lower-bound pass's survivors: the threshold they were filtered under and
// where the verdicts go.
struct RescoreRound {
  const float* tau_opt;               // threshold of the filter pass (the safe tau in the second round)
  float* thr_redo;                    // per query: threshold of the exact redo, -inf = verified and written
  int* redo_tile;                     // per query tile: 1 = some query must be redone
  const float* only;                  // second round: the queries it rescores (> -inf); NULL in the first
  const float* prev;                  // second round: the first round's thr_redo, kept by every other query
  float* second;                      // first round: the thresholds of the second round (lb2)
};
static int rescore_round(const ScoreCall& c, const RescoreRound& r) {
  const ScoreArgs& a = c.a;
  const int dp = (a.d + RSC_CH - 1) / RSC_CH * RSC_CH;
  const size_t smem = ((size_t)a.K * dp + (size_t)(MRG_THREADS / 32) * 32 * RSC_LD + a.lb.parts + 2 + 4) * sizeof(float);
  return with_k(a.K, [&](auto K) {
    CFL_SMEM_LIMIT(rescore_merge_kernel<K>, smem);
    rescore_merge_kernel<K><<<(unsigned)a.Q, MRG_THREADS, smem, c.cs>>>(
        a.keys, a.counts, a.lb.parts, a.Q, c.plan.kk, c.k, c.Pq, c.ldq, a.d, a.E, a.lde, c.idx_base, c.top_val,
        c.top_idx, c.at<float>(c.ws.tau), r.tau_opt, c.plan.qt, r.thr_redo, r.redo_tile,
        c.at<unsigned long long>(c.ws.stats), a.spill, a.spill_cnt, r.only, r.prev, r.second);
    CFL_LAUNCH_CHECK();
    return CFL_OK;
  });
}

// Stage: the single-product lower-bound filter (K <= 4), its survivors rescored exactly by rescore_merge_kernel, which
// also verifies the optimistic threshold.  Verdicts in thr_redo2 / redo_tile2.
static int lower_bound_rounds(ScoreCall& c) {
  ScoreArgs& a = c.a;
  const int64_t Q = a.Q;
  float* tau_opt = c.at<float>(c.ws.tau_opt);
  float* lb2 = c.at<float>(c.ws.lb2);
  int st = score_lb_prep_queries(a, c.cs);
  if (st != CFL_OK) return st;
  if (!c.kn.no_probe) {
    const int64_t tpp_lb = c.plan.tiles / a.lb.parts;    // the lower-bound pass has its own catalog parts
    int probe_stride = (int)((tpp_lb + 3) / 4);          // about 4 tiles per part
    if (probe_stride < 1) probe_stride = 1;
    const int64_t probe_tiles = (tpp_lb + probe_stride - 1) / probe_stride;
    a.phase = 3; a.tile_stride = probe_stride;
    CFL_CUDA(cudaMemsetAsync(a.spill_cnt, 0, (size_t)Q * sizeof(int), c.cs));
    st = score_lb_launch(a, c.cs);
    if (st != CFL_OK) return st;
    // only the pathological regimes (most rows survive) are taken out: 4x the total key capacity
    const float limit = 4.0f * ((float)a.lb.parts * (float)TOPK_STRIDE + (float)LB_SPILL);
    probe_classify_kernel<<<(unsigned)((Q + 255) / 256), 256, 0, c.cs>>>(
        a.counts, a.lb.parts, Q, (float)tpp_lb / (float)probe_tiles, limit, tau_opt, a.spill_cnt);
    CFL_LAUNCH_CHECK();
    a.phase = 2; a.tile_stride = 1;
    timer_record(0, c.cs);
  }
  CFL_CUDA(cudaMemsetAsync(a.spill_cnt, 0, (size_t)Q * sizeof(int), c.cs));
  a.phase = 3; st = score_lb_launch(a, c.cs); a.phase = 2;
  timer_record(1, c.cs);
  if (st != CFL_OK) return st;
  float* thr_redo = c.at<float>(c.ws.thr_redo);
  st = rescore_round(c, {tau_opt, thr_redo, c.at<int>(c.ws.redo_tile), nullptr, nullptr, lb2});
  if (st != CFL_OK) return st;
  // Second chance for the queries whose optimistic threshold was not confirmed (fewer than kk survivors under
  // it): the lower-bound pass again, under the SAFE threshold and only for them -- query tiles without such a
  // query leave at once -- then the exact rescoring of THEIR survivors.  Bounded by one more filter pass; the
  // exact 3xTF32 redo (a few CTAs per query tile walk the whole catalog) remains for overflowing buffers,
  // raised range flags and the queries the probe took out.
  int* redo_tile2 = c.at<int>(c.ws.redo_tile2);
  CFL_CUDA(cudaMemsetAsync(redo_tile2, 0, (size_t)c.plan.nqt * sizeof(int), c.cs));
  CFL_CUDA(cudaMemsetAsync(a.spill_cnt, 0, (size_t)Q * sizeof(int), c.cs));
  a.thr_init = lb2;
  a.phase = 3; st = score_lb_launch(a, c.cs); a.phase = 2;
  if (st != CFL_OK) return st;
  return rescore_round(c, {c.at<float>(c.ws.tau), c.at<float>(c.ws.thr_redo2), redo_tile2, lb2, thr_redo, nullptr});
}

// Stage: the exact 3xTF32 filter (K > 4 or CFL_SCORE_NO_LB) under the optimistic threshold; verify_counts_kernel
// flags the queries with fewer than kk keys.  Verdicts in thr_redo / redo_tile.
static int exact_filter(ScoreCall& c) {
  const int st = score_umma_launch(c.a, c.cs);
  timer_record(1, c.cs);
  if (st != CFL_OK) return st;
  const int64_t Q = c.a.Q;
  verify_counts_kernel<<<(unsigned)((Q + 255) / 256), 256, 0, c.cs>>>(
      c.a.counts, c.plan.parts, Q, c.plan.kk, c.plan.qt, c.at<float>(c.ws.tau), c.at<float>(c.ws.tau_opt),
      c.at<float>(c.ws.thr_redo), c.at<int>(c.ws.redo_tile), c.at<unsigned long long>(c.ws.stats));
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

// Stage: the exact kernel redoes the flagged queries (thr_redo > -inf) under the safe threshold.
static int exact_redo(ScoreCall& c, bool lb_pass, float* thr_redo, int* redo_tile, MergeInput& m) {
  ScoreArgs& a = c.a;
  const ScorePlan& plan = c.plan;
  int st;
  if (lb_pass && plan.nqt > 1) {
    // compact exact redo: up to one query tile of flagged queries, every SM on a slice of the catalog.  Its key
    // buffers live in the spill lists (free once the rescoring rounds are done): [parts][qt][TOPK_STRIDE] + counts.
    int sms_c = sm_count();
    if (sms_c <= 0) sms_c = 148;
    int64_t pc_parts = ((int64_t)a.Q * LB_SPILL) / ((int64_t)plan.qt * (TOPK_STRIDE + 1));
    if (pc_parts > sms_c) pc_parts = sms_c;
    if (pc_parts > plan.tiles) pc_parts = plan.tiles;
    if (pc_parts >= 1) {
      const CerLayout& CL = c.ws.cl;
      char* cer = (char*)align_up((size_t)(uintptr_t)(c.base + c.ws.cer), 1024);
      int* cmap = (int*)(cer + CL.idx);
      float* cthr = (float*)(cer + CL.thr);
      int* flag_c = (int*)(cer + CL.flag);
      tkey_t* ckeys = a.spill;
      int* ccounts = (int*)(a.spill + (size_t)pc_parts * plan.qt * TOPK_STRIDE);
      redo_compact_kernel<<<1, 256, 0, c.cs>>>(thr_redo, a.Q, plan.qt, a.K, a.d, plan.qt, plan.nqt, a.Pc, a.qpar,
                                               a.qplane, cmap, cthr, flag_c, (float*)(cer + CL.pc),
                                               (float*)(cer + CL.qpar), (float*)(cer + CL.qplane), redo_tile, plan.dpad,
                                               (float*)(cer + CL.qimg));
      CFL_LAUNCH_CHECK();
      m.ckeys = ckeys; m.ccounts = ccounts; m.cparts = (int)pc_parts; m.cthr = cthr; m.cmap = cmap;
      ScoreArgs b = a;
      b.Q = plan.qt; b.Pc = (const float*)(cer + CL.pc); b.qpar = (const float*)(cer + CL.qpar);
      b.qplane = (const float*)(cer + CL.qplane); b.qimg = cer + CL.qimg;
      b.keys = ckeys; b.counts = ccounts;
      b.thr_init = cthr; b.redo_tile = flag_c; b.phase = 2; b.tile_stride = 1; b.dist_out = nullptr;
      b.plan.nqt = 1; b.plan.parts = m.cparts;
      st = score_umma_launch(b, c.cs);
      if (st != CFL_OK) return st;
    }
  }
  a.thr_init = thr_redo; a.redo_tile = redo_tile;
  if (lb_pass && a.lb.parts > plan.parts) {
    // After a lower-bound pass only the redone queries use the exact kernel's key buffers, and the buffers exist
    // for the lower-bound tiling's (more numerous) catalog parts: cut the catalog that finely, so that the few
    // query tiles with something to redo are spread over more SMs (the others leave at once).
    ScoreArgs r = a;
    r.plan.parts = a.lb.parts;
    st = score_umma_launch(r, c.cs);
    m.parts = a.lb.parts;
  } else {
    st = score_umma_launch(a, c.cs);
  }
  a.redo_tile = nullptr;
  m.only = lb_pass ? thr_redo : nullptr;
  return st;
}

// Shared body of cfl_score_topk (image == NULL: packed into the workspace on every call) and
// cfl_score_topk_packed (image built once by cfl_catalog_pack).
static int score_topk_impl(int mode, const float* Pq, int64_t Q, int K, int d, int64_t ldq,
                           const float* E, const void* image, int64_t N, int64_t lde, const float* mu,
                           int k, int64_t idx_base, float* top_val, int64_t* top_idx, float* dist_out,
                           void* ws, size_t ws_bytes, cudaStream_t cs) {
  int st = device_check();
  if (st != CFL_OK) return st;
  CFL_REQUIRE(mode == CFL_PCD || mode == CFL_SIAMESE, CFL_ERR_UNSUPPORTED,
              "score_topk: mode %d not supported on the cross product (pcd, siamese)", mode);
  CFL_REQUIRE(mode != CFL_SIAMESE || K == 1, CFL_ERR_INVALID, "score_topk: siamese needs K=1");
  CFL_REQUIRE(K >= 1 && K <= CFL_MAX_K, CFL_ERR_UNSUPPORTED, "score_topk: K=%d outside [1,%d]", K, CFL_MAX_K);
  CFL_REQUIRE(d >= 1 && d <= 128, CFL_ERR_UNSUPPORTED, "score_topk: d=%d outside [1,128]", d);
  CFL_REQUIRE(k >= 1 && k <= CFL_MAX_TOPK, CFL_ERR_UNSUPPORTED, "score_topk: k=%d outside [1,%d]", k, CFL_MAX_TOPK);
  CFL_REQUIRE(Q >= 0 && N >= 0 && N < ((int64_t)1 << 32), CFL_ERR_INVALID, "score_topk: bad Q/N");
  CFL_REQUIRE(ldq >= (int64_t)K * d && lde >= d, CFL_ERR_INVALID, "score_topk: leading dimension too small");
  if (Q == 0) return CFL_OK;
  CFL_REQUIRE(Pq && top_val && top_idx, CFL_ERR_INVALID, "score_topk: NULL argument");
  CFL_REQUIRE(N == 0 || E, CFL_ERR_INVALID, "score_topk: NULL catalog");
  bool umma_ok = N > 0 && score_umma_supported(K, d);
  CFL_REQUIRE(!image || umma_ok, CFL_ERR_UNSUPPORTED, "score_topk_packed: shape K=%d d=%d has no tcgen05 tiling", K, d);
  ScoreCall c;
  c.Pq = Pq; c.ldq = ldq; c.k = k; c.idx_base = idx_base; c.top_val = top_val; c.top_idx = top_idx;
  c.plan = make_score_plan(Q, K, d, N > 0 ? N : 1, k, umma_ok);
  c.kn = read_knobs();
  c.ws = score_ws(Q, K, d, N, c.plan, image == nullptr);
  c.base = (char*)ws;
  c.cs = cs;
  CFL_REQUIRE(ws && ws_bytes >= c.ws.total, CFL_ERR_WORKSPACE, "score_topk: workspace too small (%zu < %zu)",
              ws_bytes, c.ws.total);
  const ScorePlan& plan = c.plan;
  ScoreArgs& a = c.a;
  a = ScoreArgs{};
  a.mode = mode; a.K = K; a.d = d; a.Q = Q; a.N = N; a.lde = lde; a.E = E; a.mu = mu;
  a.Pc = c.at<float>(c.ws.pc); a.qpar = c.at<float>(c.ws.qpar); a.qplane = c.at<float>(c.ws.qplane);
  a.qimg = c.at<char>(c.ws.qimg);
  a.keys = c.at<tkey_t>(c.ws.keys); a.counts = c.at<int>(c.ws.counts); a.dist_out = dist_out;
  a.tile_stride = 1;
  a.dbg_mode = c.kn.dbg_mode;
  a.plan = plan;
  a.lb = plan.impl ? make_lb_plan(Q, K, d, plan.tiles) : LbPlan{0, 0, 0, 0, 0};
  MergeInput m;
  m.parts = plan.parts;
  if (N == 0) {
    CFL_CUDA(cudaMemsetAsync(a.counts, 0, (size_t)plan.parts * Q * sizeof(int), cs));
  } else {
    st = prep_and_pack(c, image);
    if (st != CFL_OK) return st;
    if (plan.impl != 1) {
      timer_record(0, cs);
      st = with_k(K, [&](auto KC) { return launch_simt<KC>(a, cs); });
      timer_record(1, cs);
    } else if (!score_two_pass(c.kn, plan, dist_out != nullptr)) {
      timer_record(0, cs);
      a.phase = 0; a.tile_stride = 1; a.thr_init = nullptr;
      st = score_umma_launch(a, cs);
      timer_record(1, cs);
    } else {
      st = sample_thresholds(c);
      if (st != CFL_OK) return st;
      a.spill = c.at<tkey_t>(c.ws.spill); a.spill_cnt = c.at<int>(c.ws.spill_cnt);
      a.phase = 2; a.tile_stride = 1; a.thr_init = c.at<float>(c.ws.tau_opt);
      timer_record(0, cs);                 // bench.py times the dominant launch: the full filter pass
      const bool lb_pass = score_lb_pass(c.kn, K);
      st = lb_pass ? lower_bound_rounds(c) : exact_filter(c);
      if (st != CFL_OK) return st;
      float* thr_redo = c.at<float>(lb_pass ? c.ws.thr_redo2 : c.ws.thr_redo);
      int* redo_tile = c.at<int>(lb_pass ? c.ws.redo_tile2 : c.ws.redo_tile);
      st = exact_redo(c, lb_pass, thr_redo, redo_tile, m);
    }
    if (st != CFL_OK) return st;
  }
  // after a lower-bound pass the verified queries are already written; only the redone ones remain
  return with_k(K, [&](auto KC) {
    merge_rescore_kernel<KC><<<(unsigned)(Q + (m.cparts ? plan.qt : 0)), MRG_THREADS, 0, cs>>>(
        a.keys, a.counts, m.parts, Q, plan.kk, k, Pq, ldq, d, E, lde, idx_base, top_val, top_idx, m.only, plan.qt,
        m.ckeys, m.ccounts, m.cparts, m.cthr, m.cmap);
    CFL_LAUNCH_CHECK();
    return CFL_OK;
  });
}

// The source-catalog call: the exact filter cascade of score_topk_impl on score_src_umma_kernel (sample thresholds,
// exact filter under the optimistic threshold, in-place exact redo, merge with direct-form rescoring).  There is no
// lower-bound pass and no CUDA-core kernel: every K <= 8, d <= 128 has a tensor-core tiling (score_src_qt).
static ScorePlan source_plan(int64_t Q, int K, int d, int64_t N, int k) {
  return make_score_plan_qt(Q, score_src_qt(K, d), d, N > 0 ? N : 1, k, true);
}

static int score_topk_source_impl(const float* Eq, int64_t ldq, int64_t Q, int K, int d, const void* image,
                                  const float* Pc, int64_t N, int64_t ldp, const float* mu, int k, int64_t idx_base,
                                  float* top_val, int64_t* top_idx, float* dist_out, unsigned long long* stats_out,
                                  void* ws, size_t ws_bytes, cudaStream_t cs) {
  int st = device_check();
  if (st != CFL_OK) return st;
  CFL_REQUIRE(K >= 1 && K <= CFL_MAX_K, CFL_ERR_UNSUPPORTED, "score_topk_source: K=%d outside [1,%d]", K, CFL_MAX_K);
  CFL_REQUIRE(d >= 1 && d <= 128, CFL_ERR_UNSUPPORTED, "score_topk_source: d=%d outside [1,128]", d);
  CFL_REQUIRE(k >= 1 && k <= CFL_MAX_TOPK, CFL_ERR_UNSUPPORTED, "score_topk_source: k=%d outside [1,%d]", k, CFL_MAX_TOPK);
  CFL_REQUIRE(Q >= 0 && N >= 0 && N < ((int64_t)1 << 32), CFL_ERR_INVALID, "score_topk_source: bad Q/N");
  CFL_REQUIRE(ldq >= d && ldp >= (int64_t)K * d, CFL_ERR_INVALID, "score_topk_source: leading dimension too small");
  if (stats_out) CFL_CUDA(cudaMemsetAsync(stats_out, 0, CFL_SCORE_NSTATS * sizeof(unsigned long long), cs));
  if (Q == 0) return CFL_OK;
  CFL_REQUIRE(Eq && top_val && top_idx, CFL_ERR_INVALID, "score_topk_source: NULL argument");
  CFL_REQUIRE(N == 0 || (Pc && image), CFL_ERR_INVALID, "score_topk_source: NULL catalog or image");
  CFL_REQUIRE(((uintptr_t)image & 1023u) == 0, CFL_ERR_INVALID, "score_topk_source: image must be 1024-byte aligned");
  ScoreCall c;
  c.Pq = Eq; c.ldq = ldq; c.k = k; c.idx_base = idx_base; c.top_val = top_val; c.top_idx = top_idx;
  c.plan = source_plan(Q, K, d, N, k);
  c.kn = read_knobs();
  c.ws = score_ws(Q, K, d, N, c.plan, false, true);
  c.base = (char*)ws;
  c.cs = cs;
  CFL_REQUIRE(ws && ws_bytes >= c.ws.total, CFL_ERR_WORKSPACE, "score_topk_source: workspace too small (%zu < %zu)",
              ws_bytes, c.ws.total);
  const ScorePlan& plan = c.plan;
  ScoreArgs& a = c.a;
  a = ScoreArgs{};
  a.src = true;
  a.mode = CFL_PCD; a.K = K; a.d = d; a.Q = Q; a.N = N; a.lde = ldp; a.E = Pc; a.mu = mu;
  a.Pc = c.at<float>(c.ws.pc); a.qpar = c.at<float>(c.ws.qpar);
  a.qimg = c.at<char>(c.ws.qimg);
  a.keys = c.at<tkey_t>(c.ws.keys); a.counts = c.at<int>(c.ws.counts); a.dist_out = dist_out;
  a.tile_stride = 1;
  a.plan = plan;
  MergeInput m;
  m.parts = plan.parts;
  bool two_pass = false;
  if (N == 0) {
    CFL_CUDA(cudaMemsetAsync(a.counts, 0, (size_t)plan.parts * Q * sizeof(int), cs));
  } else {
    st = score_prep_source_queries_launch(Eq, Q, d, ldq, mu, (float*)a.Pc, (float*)a.qpar, cs);
    if (st != CFL_OK) return st;
    const SourceCatalogView v = source_catalog_view(image, N, K, d);
    a.cimg = v.blocks; a.e2 = v.rowpar;
    st = score_umma_pack_queries(a, c.base + c.ws.qimg, cs);
    if (st != CFL_OK) return st;
    if (!score_two_pass(c.kn, plan, dist_out != nullptr)) {
      timer_record(0, cs);
      a.phase = 0; a.tile_stride = 1; a.thr_init = nullptr;
      st = score_umma_launch(a, cs);
      timer_record(1, cs);
    } else {
      two_pass = true;
      st = sample_thresholds(c);
      if (st != CFL_OK) return st;
      a.phase = 2; a.tile_stride = 1; a.thr_init = c.at<float>(c.ws.tau_opt);
      timer_record(0, cs);
      st = exact_filter(c);
      if (st != CFL_OK) return st;
      st = exact_redo(c, false, c.at<float>(c.ws.thr_redo), c.at<int>(c.ws.redo_tile), m);
    }
    if (st != CFL_OK) return st;
  }
  st = with_k(K, [&](auto KC) {
    merge_rescore_src_kernel<KC><<<(unsigned)Q, MRG_THREADS, 0, cs>>>(a.keys, a.counts, m.parts, Q, plan.kk, k, Eq, ldq, d,
                                                                       Pc, ldp, idx_base, top_val, top_idx);
    CFL_LAUNCH_CHECK();
    return CFL_OK;
  });
  if (st != CFL_OK) return st;
  if (stats_out && two_pass)
    CFL_CUDA(cudaMemcpyAsync(stats_out, c.at<unsigned long long>(c.ws.stats), CFL_SCORE_NSTATS * sizeof(unsigned long long),
                             cudaMemcpyDeviceToDevice, cs));
  return CFL_OK;
}

extern "C" {

size_t cfl_source_catalog_pack_bytes(int64_t N, int K, int d) {
  if (N <= 0 || score_src_qt(K, d) == 0) return 0;
  return source_catalog_image_bytes(N, K, d);
}

int cfl_source_catalog_pack(const float* Pc, int64_t N, int K, int d, int64_t ldp, const float* mu, void* image,
                            size_t image_bytes, void* stream) {
  int st = device_check();
  if (st != CFL_OK) return st;
  CFL_REQUIRE(score_src_qt(K, d) != 0, CFL_ERR_UNSUPPORTED, "source_catalog_pack: K=%d d=%d outside K <= %d, d <= 128", K,
              d, CFL_MAX_K);
  CFL_REQUIRE(Pc && image && N > 0 && N < ((int64_t)1 << 32) && ldp >= (int64_t)K * d, CFL_ERR_INVALID,
              "source_catalog_pack: bad arguments");
  CFL_REQUIRE(image_bytes >= source_catalog_image_bytes(N, K, d), CFL_ERR_WORKSPACE,
              "source_catalog_pack: image buffer too small");
  CFL_REQUIRE(((uintptr_t)image & 1023u) == 0, CFL_ERR_INVALID, "source_catalog_pack: image must be 1024-byte aligned");
  return source_catalog_pack_launch(Pc, N, K, d, ldp, mu, image, (cudaStream_t)stream);
}

size_t cfl_score_topk_source_workspace_bytes(int64_t Q, int K, int d, int64_t N, int k) {
  if (Q <= 0 || score_src_qt(K, d) == 0) return 4096;
  return score_ws(Q, K, d, N, source_plan(Q, K, d, N, k), false, true).total + 1024;
}

int cfl_score_topk_source(const float* Eq, int64_t ldq, int64_t Q, int K, int d, const void* image, const float* Pc,
                          int64_t N, int64_t ldp, const float* mu, int k, int64_t idx_base, float* top_val,
                          int64_t* top_idx, float* dist_out, unsigned long long* stats_out, void* ws, size_t ws_bytes,
                          void* stream) {
  return score_topk_source_impl(Eq, ldq, Q, K, d, image, Pc, N, ldp, mu, k, idx_base, top_val, top_idx, dist_out,
                                stats_out, ws, ws_bytes, (cudaStream_t)stream);
}

size_t cfl_score_topk_workspace_bytes(int64_t Q, int K, int d, int64_t N, int k) {
  return score_ws_bytes(Q, K, d, N, k, true);
}
size_t cfl_score_topk_packed_workspace_bytes(int64_t Q, int K, int d, int64_t N, int k) {
  return score_ws_bytes(Q, K, d, N, k, false);
}

size_t cfl_catalog_pack_bytes(int64_t N, int K, int d) {
  if (N <= 0 || score_umma_qt(K, d) == 0) return 0;
  return catalog_image_bytes(N, d);
}

int cfl_catalog_pack(const float* E, int64_t N, int K, int d, int64_t lde, const float* mu, void* image,
                     size_t image_bytes, void* stream) {
  int st = device_check();
  if (st != CFL_OK) return st;
  CFL_REQUIRE(E && image && N > 0 && lde >= d, CFL_ERR_INVALID, "catalog_pack: bad arguments");
  CFL_REQUIRE(score_umma_supported(K, d), CFL_ERR_UNSUPPORTED, "catalog_pack: shape K=%d d=%d has no tcgen05 tiling", K, d);
  CFL_REQUIRE(image_bytes >= catalog_image_bytes(N, d), CFL_ERR_WORKSPACE, "catalog_pack: image buffer too small");
  CFL_REQUIRE(((uintptr_t)image & 1023u) == 0, CFL_ERR_INVALID, "catalog_pack: image must be 1024-byte aligned");
  return catalog_pack_launch(E, N, d, lde, mu, image, (cudaStream_t)stream);
}

int cfl_score_topk(int mode, const float* Pq, int64_t Q, int K, int d, int64_t ldq,
                   const float* E, int64_t N, int64_t lde, const float* mu, int k,
                   int64_t idx_base, float* top_val, int64_t* top_idx, float* dist_out, void* ws,
                   size_t ws_bytes, void* stream) {
  return score_topk_impl(mode, Pq, Q, K, d, ldq, E, nullptr, N, lde, mu, k, idx_base, top_val, top_idx,
                         dist_out, ws, ws_bytes, (cudaStream_t)stream);
}

int cfl_score_topk_packed(int mode, const float* Pq, int64_t Q, int K, int d, int64_t ldq,
                          const void* image, const float* E, int64_t N, int64_t lde, const float* mu, int k,
                          int64_t idx_base, float* top_val, int64_t* top_idx, float* dist_out, void* ws,
                          size_t ws_bytes, void* stream) {
  CFL_REQUIRE(image, CFL_ERR_INVALID, "score_topk_packed: NULL image");
  return score_topk_impl(mode, Pq, Q, K, d, ldq, E, image, N, lde, mu, k, idx_base, top_val, top_idx,
                         dist_out, ws, ws_bytes, (cudaStream_t)stream);
}

int cfl_score_topk_stats(int64_t Q, int K, int d, int64_t N, int k, int packed, const void* ws, size_t ws_bytes,
                         unsigned long long* stats_out, float* thr_out, void* stream) {
  int st = device_check();
  if (st != CFL_OK) return st;
  CFL_REQUIRE(ws && stats_out && Q > 0 && N > 0, CFL_ERR_INVALID, "score_topk_stats: bad arguments");
  const bool umma_ok = score_umma_supported(K, d);
  ScorePlan plan = make_score_plan(Q, K, d, N, k, umma_ok);
  const ScoreKnobs kn = read_knobs();
  cudaStream_t cs = (cudaStream_t)stream;
  if (!umma_ok || !score_two_pass(kn, plan, false)) {         // short catalogs / CUDA-core shapes: one adaptive pass, no statistics
    CFL_CUDA(cudaMemsetAsync(stats_out, 0, CFL_SCORE_NSTATS * sizeof(unsigned long long), cs));
    if (thr_out) CFL_CUDA(cudaMemsetAsync(thr_out, 0, (size_t)3 * Q * sizeof(float), cs));
    return CFL_OK;
  }
  const ScoreWs w = score_ws(Q, K, d, N, plan, packed == 0);
  CFL_REQUIRE(ws_bytes >= w.total, CFL_ERR_WORKSPACE, "score_topk_stats: workspace too small (%zu < %zu)", ws_bytes,
              w.total);
  const char* stats = (const char*)ws + w.stats;
  const char* tau = (const char*)ws + w.tau;                  // tau, tau_opt and thr_redo are consecutive
  CFL_CUDA(cudaMemcpyAsync(stats_out, stats, CFL_SCORE_NSTATS * sizeof(unsigned long long), cudaMemcpyDeviceToDevice, cs));
  if (thr_out) CFL_CUDA(cudaMemcpyAsync(thr_out, tau, (size_t)3 * Q * sizeof(float), cudaMemcpyDeviceToDevice, cs));
  return CFL_OK;
}

int cfl_topk_merge(const float* vals, const int64_t* idx, int R, int64_t Q, int k, float* top_val,
                   int64_t* top_idx, void* stream) {
  int st = device_check();
  if (st != CFL_OK) return st;
  CFL_REQUIRE(vals && idx && top_val && top_idx && R >= 1 && Q >= 0 && k >= 1, CFL_ERR_INVALID,
              "topk_merge: bad arguments");
  if (Q == 0) return CFL_OK;
  topk_merge_kernel<<<(unsigned)Q, 128, 0, (cudaStream_t)stream>>>((const char*)vals, (const char*)idx, (size_t)Q * k * sizeof(float),
                                                                   (size_t)Q * k * sizeof(int64_t), R, Q, k, top_val, top_idx);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

size_t cfl_topk_record_bytes(int64_t Q, int k) { return topk_record_bytes(Q * (int64_t)k); }

int cfl_topk_pack_records(const float* vals, const int64_t* idx, int64_t Q, int k, void* rec, void* stream) {
  int st = device_check();
  if (st != CFL_OK) return st;
  CFL_REQUIRE(Q >= 0 && k >= 1 && (Q == 0 || (vals && idx && rec)), CFL_ERR_INVALID, "topk_pack_records: bad arguments");
  const int64_t n = Q * (int64_t)k;
  if (n == 0) return CFL_OK;
  topk_pack_records_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(vals, idx, n, (char*)rec);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

int cfl_topk_merge_records(const void* recs, int R, int64_t Q, int k, float* top_val, int64_t* top_idx, void* stream) {
  int st = device_check();
  if (st != CFL_OK) return st;
  CFL_REQUIRE(recs && top_val && top_idx && R >= 1 && Q >= 0 && k >= 1, CFL_ERR_INVALID, "topk_merge_records: bad arguments");
  if (Q == 0) return CFL_OK;
  const int64_t n = Q * (int64_t)k;
  const size_t rb = topk_record_bytes(n);
  topk_merge_kernel<<<(unsigned)Q, 128, 0, (cudaStream_t)stream>>>((const char*)recs + (size_t)n * 8, (const char*)recs, rb, rb, R, Q, k,
                                                                   top_val, top_idx);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

}  // extern "C"
