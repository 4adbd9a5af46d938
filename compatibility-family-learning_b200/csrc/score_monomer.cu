// Stage 2 on the Q x N cross product, monomer mode (SURVEY App. A.6; the pair scorer is
// DistBase.build_dist, cfl/models/base.py:109-117):
//     dist(q, c) = sum_k w_qk * | a_q - P'_ck |^2
// with the roles the reference gives them -- a_q = act(e0) and w_q = softmax(gate) of the SOURCE
// (query) item, P'_c = the K prototypes of the TARGET (catalog) item, so here the catalog carries
// K*d floats per row and the query side is small.
//
// The distance is evaluated in direct-difference form in fp32 (the arithmetic of the paired kernel),
// so the values are final: no centring, no rescoring pass.  One thread owns one catalog row of a
// 128-row tile and 16 queries; prototype k of the tile is staged through shared memory (coalesced
// row segments), the query vectors sit in shared memory as query PAIRS so the inner loop is packed
// FP32x2 (add.f32x2 + fma.f32x2: two queries per instruction), and the running per-query top-k is the
// machinery of topk.cuh (append buffers in the workspace, warp compaction, block merge).
#include <stdlib.h>
#include "score.cuh"

namespace cfl {

constexpr int MONO_QT = 16;        // queries per CTA (8 packed pairs per thread)
constexpr int MONO_THREADS = 128;  // one thread per catalog row of a tile
constexpr int MONO_KSTRIDE = TOPK_CAP;   // keys per (part, query) buffer: the adaptive mode never holds more than 512

struct MonoArgs {
  int K, d;
  int64_t Q, N, lda, ldp;
  const float* A;    // [Q, lda]  query embeddings a_q
  const float* W;    // [Q, K]    query gate weights (softmax), dense
  const float* P;    // [N, ldp]  catalog prototypes, prototype k of row c at columns [k*d, (k+1)*d)
  tkey_t* keys;      // [parts, Q, MONO_KSTRIDE]
  int* counts;       // [parts, Q]
  float* dist_out;   // optional dense [Q, N]
  int parts, kk;
  int64_t tiles;
  int tile_stride;          // visit every tile_stride-th tile of a part (the threshold sample of the tensor-core path)
  const int* redo_tile;     // optional [ceil(Q / MONO_QT)]: a CTA whose query tile has nothing to redo exits at once
};

// VW = floats per staging load: 4 / 2 when d and ldp are multiples of it and the catalog is aligned to it (128- /
// 64-bit loads: the element walk costs address arithmetic per load, so wider loads cut the overhead), else 1.
template <int VW>
__global__ void __launch_bounds__(MONO_THREADS)
score_monomer_kernel(MonoArgs A) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int K = A.K, d = A.d;
  const int ldt = d + 1;                                              // odd-ish stride: conflict-free row reads
  tkey_t* scratch = (tkey_t*)smem_raw;                                // [4][512] compaction scratch
  f2_t* aq2 = (f2_t*)(scratch + (MONO_THREADS / 32) * TOPK_CAP);      // [d][QT/2]: element j of queries (2p, 2p+1)
  float* wq = (float*)(aq2 + (size_t)d * (MONO_QT / 2));              // [K][QT]
  float* thr = wq + K * MONO_QT;                                      // [QT]
  int* cnt = (int*)(thr + MONO_QT);                                   // [QT]
  float* et = (float*)(cnt + MONO_QT);                                // [128][d+1] prototype k of the tile

  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int part = blockIdx.x;
  if (A.redo_tile != nullptr && A.redo_tile[blockIdx.y] == 0) return;
  const int64_t q0 = (int64_t)blockIdx.y * MONO_QT;
  const int nq = (int)((A.Q - q0 < MONO_QT) ? (A.Q - q0) : MONO_QT);
  for (int i = tid; i < MONO_QT * d; i += MONO_THREADS) {
    const int ql = i / d, j = i % d;
    ((float*)aq2)[j * MONO_QT + ql] = ql < nq ? A.A[(q0 + ql) * A.lda + j] : 0.0f;
  }
  for (int i = tid; i < MONO_QT * K; i += MONO_THREADS) {
    const int ql = i / K, k = i % K;
    wq[k * MONO_QT + ql] = ql < nq ? A.W[(q0 + ql) * K + k] : 0.0f;
  }
  if (tid < MONO_QT) { thr[tid] = __int_as_float(0x7f800000); cnt[tid] = 0; }
  const int64_t t0 = A.tiles * part / A.parts;
  const int64_t t1 = A.tiles * (part + 1) / A.parts;
  tkey_t* kbase = A.keys + ((int64_t)part * A.Q + q0) * MONO_KSTRIDE;
  // staging walk: element i = r*dv + j of a [128][dv] prototype tile (dv = d / VW vector loads per row), advanced
  // by 128 without divisions
  const int dv = d / VW;
  const int sr0 = tid / dv, sj0 = tid % dv, sdr = MONO_THREADS / dv, sdj = MONO_THREADS % dv;

  // tile_stride > 1: the tiles whose GLOBAL index is a multiple of it (a sample whose density does not depend on the parts)
  for (int64_t tile = (t0 + A.tile_stride - 1) / A.tile_stride * A.tile_stride; tile < t1; tile += A.tile_stride) {
    const int64_t r0 = tile * 128;
    f2_t acc[MONO_QT / 2];
#pragma unroll
    for (int p = 0; p < MONO_QT / 2; ++p) acc[p] = pk2(0.0f, 0.0f);
    for (int k = 0; k < K; ++k) {
      __syncthreads();                                   // queries loaded / previous prototype consumed
      for (int i = tid, r = sr0, j = sj0; i < 128 * dv; i += MONO_THREADS) {
        const int64_t row = r0 + r;
        const float* src = A.P + row * A.ldp + (int64_t)k * d + VW * j;
        float* dst = et + r * ldt + VW * j;
        if (VW == 4) {
          const float4 v = row < A.N ? *(const float4*)src : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
          dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
        } else if (VW == 2) {
          const float2 v = row < A.N ? *(const float2*)src : make_float2(0.0f, 0.0f);
          dst[0] = v.x; dst[1] = v.y;
        } else {
          dst[0] = row < A.N ? *src : 0.0f;
        }
        r += sdr; j += sdj;
        if (j >= dv) { j -= dv; ++r; }
      }
      __syncthreads();
      const float* er = et + tid * ldt;
      f2_t dk[MONO_QT / 2];
#pragma unroll
      for (int p = 0; p < MONO_QT / 2; ++p) dk[p] = pk2(0.0f, 0.0f);
      for (int j = 0; j < d; ++j) {
        const float ne = -er[j];
        const f2_t ne2 = pk2(ne, ne);
        const ulonglong2* aj = (const ulonglong2*)(aq2 + (size_t)j * (MONO_QT / 2));
#pragma unroll
        for (int p = 0; p < MONO_QT / 4; ++p) {
          const ulonglong2 a = aj[p];
          const f2_t d0 = add2(a.x, ne2), d1 = add2(a.y, ne2);
          dk[2 * p] = fma2(d0, d0, dk[2 * p]);
          dk[2 * p + 1] = fma2(d1, d1, dk[2 * p + 1]);
        }
      }
      const f2_t* wk = (const f2_t*)(wq + k * MONO_QT);
#pragma unroll
      for (int p = 0; p < MONO_QT / 2; ++p) acc[p] = fma2(wk[p], dk[p], acc[p]);
    }
    const int64_t row = r0 + tid;
    if (row < A.N) {
#pragma unroll
      for (int p = 0; p < MONO_QT / 2; ++p) {
        float dv[2];
        upk2(acc[p], dv[0], dv[1]);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int ql = 2 * p + h;
          if (ql < nq) {
            if (A.dist_out) A.dist_out[(q0 + ql) * A.N + row] = dv[h];
            if (dv[h] < thr[ql]) {
              const int slot = atomicAdd(&cnt[ql], 1);
              kbase[(int64_t)ql * MONO_KSTRIDE + slot] = pack_key(dv[h], (uint32_t)row);
            }
          }
        }
      }
    }
    __syncthreads();
    for (int ql = wid; ql < nq; ql += MONO_THREADS / 32) {
      const int n = cnt[ql];
      if (n > TOPK_TRIGGER) {
        const int nk = warp_compact(kbase + (int64_t)ql * MONO_KSTRIDE, n, A.kk, scratch + wid * TOPK_CAP, lane, &thr[ql]);
        if (lane == 0) cnt[ql] = nk;
      }
    }
  }
  __syncthreads();
  for (int ql = wid; ql < nq; ql += MONO_THREADS / 32) {
    const int nk = warp_compact(kbase + (int64_t)ql * MONO_KSTRIDE, cnt[ql], A.kk, scratch + wid * TOPK_CAP, lane, nullptr);
    if (lane == 0) A.counts[(int64_t)part * A.Q + q0 + ql] = nk;
  }
}

// The other direction (cfl_score_topk_monomer_source): the catalog rows are SOURCE items (a_c, w_c), the queries TARGET
// items (K prototypes each), dist(q, c) = sum_k w_ck |a_c - P'_qk|^2.  One thread owns one source row of a 128-row tile
// and 16 queries; the tile's a and w are staged once per tile, the queries' K prototypes sit in shared memory as query
// PAIRS, negated, so the inner loop is packed FP32x2 as above.  Operation order of monomer_direct (direct.cuh): over k,
// over j, a_j + (-p_kj), fmaf; then fmaf(w_k, dk, acc) -- the values are final.
struct MonoSrcArgs {
  int K, d;
  int64_t Q, N, ldq, lda;
  const float* P;    // [Q, ldq]  query prototypes, prototype k of query q at columns [k*d, (k+1)*d)
  const float* A;    // [N, lda]  catalog embeddings a_c
  const float* W;    // [N, K]    catalog gate weights (softmax), dense
  tkey_t* keys;      // [parts, Q, MONO_KSTRIDE]
  int* counts;       // [parts, Q]
  int parts, kk;
  int64_t tiles;
  int tile_stride;
  const int* redo_tile;
};

constexpr int MONO_SRC_CTAS_PER_SM = 4;   // 125 registers x 128 threads, no spills (at 8 CTAs per SM ptxas spills)

__global__ void __launch_bounds__(MONO_THREADS, MONO_SRC_CTAS_PER_SM)
score_monomer_src_kernel(MonoSrcArgs A) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int K = A.K, d = A.d, kd = K * d;
  const int ldt = d | 1;                                              // odd stride: conflict-free row reads
  tkey_t* scratch = (tkey_t*)smem_raw;                                // [4][512] compaction scratch
  f2_t* np2 = (f2_t*)(scratch + (MONO_THREADS / 32) * TOPK_CAP);      // [K*d][QT/2]: -P'_(k,j) of queries (2p, 2p+1)
  float* thr = (float*)(np2 + (size_t)kd * (MONO_QT / 2));            // [QT]
  int* cnt = (int*)(thr + MONO_QT);                                   // [QT]
  float* wt = (float*)(cnt + MONO_QT);                                // [K][128] gate weights of the tile's rows
  float* at = wt + K * MONO_THREADS;                                  // [128][ldt] embeddings of the tile's rows

  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int part = blockIdx.x;
  if (A.redo_tile != nullptr && A.redo_tile[blockIdx.y] == 0) return;
  const int64_t q0 = (int64_t)blockIdx.y * MONO_QT;
  const int nq = (int)((A.Q - q0 < MONO_QT) ? (A.Q - q0) : MONO_QT);
  for (int i = tid; i < MONO_QT * kd; i += MONO_THREADS) {
    const int ql = i / kd, kj = i % kd;
    ((float*)np2)[kj * MONO_QT + ql] = ql < nq ? -A.P[(q0 + ql) * A.ldq + kj] : 0.0f;
  }
  if (tid < MONO_QT) { thr[tid] = __int_as_float(0x7f800000); cnt[tid] = 0; }
  const int64_t t0 = A.tiles * part / A.parts;
  const int64_t t1 = A.tiles * (part + 1) / A.parts;
  tkey_t* kbase = A.keys + ((int64_t)part * A.Q + q0) * MONO_KSTRIDE;
  const int sr0 = tid / d, sj0 = tid % d, sdr = MONO_THREADS / d, sdj = MONO_THREADS % d;

  for (int64_t tile = (t0 + A.tile_stride - 1) / A.tile_stride * A.tile_stride; tile < t1; tile += A.tile_stride) {
    const int64_t r0 = tile * 128;
    __syncthreads();                                     // queries loaded / previous tile consumed
    for (int i = tid, r = sr0, j = sj0; i < 128 * d; i += MONO_THREADS) {
      const int64_t row = r0 + r;
      at[r * ldt + j] = row < A.N ? A.A[row * A.lda + j] : 0.0f;
      r += sdr; j += sdj;
      if (j >= d) { j -= d; ++r; }
    }
    for (int i = tid; i < 128 * K; i += MONO_THREADS) {
      const int r = i / K, k = i % K;
      const int64_t row = r0 + r;
      wt[k * MONO_THREADS + r] = row < A.N ? A.W[row * K + k] : 0.0f;
    }
    __syncthreads();
    const float* ar = at + tid * ldt;
    f2_t acc[MONO_QT / 2];
#pragma unroll
    for (int p = 0; p < MONO_QT / 2; ++p) acc[p] = pk2(0.0f, 0.0f);
    for (int k = 0; k < K; ++k) {
      f2_t dk[MONO_QT / 2];
#pragma unroll
      for (int p = 0; p < MONO_QT / 2; ++p) dk[p] = pk2(0.0f, 0.0f);
      const ulonglong2* pk = (const ulonglong2*)(np2 + (size_t)k * d * (MONO_QT / 2));
      for (int j = 0; j < d; ++j) {
        const float a = ar[j];
        const f2_t a2 = pk2(a, a);
        const ulonglong2* pj = pk + j * (MONO_QT / 4);
#pragma unroll
        for (int p = 0; p < MONO_QT / 4; ++p) {
          const ulonglong2 np = pj[p];
          const f2_t d0 = add2(a2, np.x), d1 = add2(a2, np.y);
          dk[2 * p] = fma2(d0, d0, dk[2 * p]);
          dk[2 * p + 1] = fma2(d1, d1, dk[2 * p + 1]);
        }
      }
      const float w = wt[k * MONO_THREADS + tid];
      const f2_t w2 = pk2(w, w);
#pragma unroll
      for (int p = 0; p < MONO_QT / 2; ++p) acc[p] = fma2(w2, dk[p], acc[p]);
    }
    const int64_t row = r0 + tid;
    if (row < A.N) {
#pragma unroll
      for (int p = 0; p < MONO_QT / 2; ++p) {
        float dv[2];
        upk2(acc[p], dv[0], dv[1]);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int ql = 2 * p + h;
          if (ql < nq && dv[h] < thr[ql]) {
            const int slot = atomicAdd(&cnt[ql], 1);
            kbase[(int64_t)ql * MONO_KSTRIDE + slot] = pack_key(dv[h], (uint32_t)row);
          }
        }
      }
    }
    __syncthreads();
    for (int ql = wid; ql < nq; ql += MONO_THREADS / 32) {
      const int n = cnt[ql];
      if (n > TOPK_TRIGGER) {
        const int nk = warp_compact(kbase + (int64_t)ql * MONO_KSTRIDE, n, A.kk, scratch + wid * TOPK_CAP, lane, &thr[ql]);
        if (lane == 0) cnt[ql] = nk;
      }
    }
  }
  __syncthreads();
  for (int ql = wid; ql < nq; ql += MONO_THREADS / 32) {
    const int nk = warp_compact(kbase + (int64_t)ql * MONO_KSTRIDE, cnt[ql], A.kk, scratch + wid * TOPK_CAP, lane, nullptr);
    if (lane == 0) A.counts[(int64_t)part * A.Q + q0 + ql] = nk;
  }
}

// Merge of the catalog parts; the keys already carry exact distances.
__global__ void __launch_bounds__(MRG_THREADS)
merge_plain_kernel(const tkey_t* __restrict__ keys, const int* __restrict__ counts, int parts, int64_t Q, int kk,
                   int k, int64_t idx_base, float* __restrict__ top_val, int64_t* __restrict__ top_idx,
                   const float* __restrict__ only_redo = nullptr) {
  __shared__ tkey_t s[TOPK_CAP];
  __shared__ int s_fill;
  __shared__ tkey_t s_thr;
  const int t = threadIdx.x;
  const int64_t q = blockIdx.x;
  // second merge of the tensor-core path: only the queries that were redone by this kernel's exact pass
  if (only_redo != nullptr && !(only_redo[q] > __int_as_float(0xff800000))) return;
  const int fill = block_merge_topkk(keys, counts, parts, Q, q, kk, s, &s_fill, &s_thr, MONO_KSTRIDE);
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

static size_t mono_smem_bytes(int K, int d) {
  return (size_t)(MONO_THREADS / 32) * TOPK_CAP * sizeof(tkey_t) + (size_t)d * MONO_QT * 4 + (size_t)K * MONO_QT * 4 +
         MONO_QT * 8 + (size_t)128 * (d + 1) * 4;
}

static size_t mono_src_smem_bytes(int K, int d) {
  return (size_t)(MONO_THREADS / 32) * TOPK_CAP * sizeof(tkey_t) + (size_t)K * d * MONO_QT * 4 + MONO_QT * 8 +
         (size_t)K * MONO_THREADS * 4 + (size_t)MONO_THREADS * (d | 1) * 4;
}

struct MonoPlan { int nqt, parts; int64_t tiles; };

// One wave: the grid is sized to the CTAs that are RESIDENT at once (64 registers x 128 threads -> 8 per SM;
// 228 KB of shared memory per SM, 1 KB reserved per CTA), because only resident warps hide the staging latency
// and a second, partial wave would idle most SMs (measured: 4 CTAs per SM left 76 % of the warp slots empty,
// 8 per SM ran 1.1 waves).  smem = dynamic shared memory of one CTA of the kernel being planned.
static MonoPlan mono_plan_smem(int64_t Q, int64_t N, size_t smem, int64_t max_resident) {
  MonoPlan p;
  p.nqt = (int)((Q + MONO_QT - 1) / MONO_QT);
  p.tiles = (N + 127) / 128;
  int sms = sm_count();
  if (sms <= 0) sms = 148;
  int64_t resident = (228 * 1024) / (int64_t)(smem + 1024);
  if (resident > max_resident) resident = max_resident;  // register-limited CTAs per SM
  if (resident < 1) resident = 1;
  const char* e = getenv("CFL_MONO_CTAS_PER_SM");
  if (e && atoi(e) > 0) resident = atoi(e);
  int64_t parts = p.nqt > 0 ? (resident * sms) / p.nqt : 1;
  if (parts > p.tiles) parts = p.tiles;
  if (parts < 1) parts = 1;
  p.parts = (int)parts;
  return p;
}
static MonoPlan mono_plan(int64_t Q, int64_t N, int K, int d) {
  return mono_plan_smem(Q, N, mono_smem_bytes(K, d), 8);                 // 64 registers x 128 threads
}
static MonoPlan mono_src_plan(int64_t Q, int64_t N, int K, int d) {
  return mono_plan_smem(Q, N, mono_src_smem_bytes(K, d), MONO_SRC_CTAS_PER_SM);
}

// Launch of the CUDA-core kernel for the tensor-core path (score_monomer_tc.cu): threshold sample (tile_stride > 1)
// and exact redo (redo_tile != NULL); keys [parts, Q, MONO_KSTRIDE], counts [parts, Q].
int mono_exact_launch(const float* Aq, int64_t lda, const float* Wq, int64_t Q, int K, int d, const float* Pc, int64_t N,
                      int64_t ldp, int kk, int tile_stride, const int* redo_tile, tkey_t* keys, int* counts, int* parts_out,
                      cudaStream_t cs) {
  MonoPlan plan = mono_plan(Q, N, K, d);
  MonoArgs a;
  a.K = K; a.d = d; a.Q = Q; a.N = N; a.lda = lda; a.ldp = ldp; a.A = Aq; a.W = Wq; a.P = Pc;
  a.keys = keys; a.counts = counts; a.dist_out = nullptr;
  a.parts = plan.parts; a.kk = kk; a.tiles = plan.tiles; a.tile_stride = tile_stride; a.redo_tile = redo_tile;
  *parts_out = plan.parts;
  const size_t smem = mono_smem_bytes(K, d);
  int vw = 1;
  if (d % 4 == 0 && ldp % 4 == 0 && ((uintptr_t)Pc & 15u) == 0) vw = 4;
  else if (d % 2 == 0 && ldp % 2 == 0 && ((uintptr_t)Pc & 7u) == 0) vw = 2;
  dim3 grid(plan.parts, plan.nqt);
  switch (vw) {
    case 4:
      CFL_CUDA(cudaFuncSetAttribute(score_monomer_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      score_monomer_kernel<4><<<grid, MONO_THREADS, smem, cs>>>(a); break;
    case 2:
      CFL_CUDA(cudaFuncSetAttribute(score_monomer_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      score_monomer_kernel<2><<<grid, MONO_THREADS, smem, cs>>>(a); break;
    default:
      CFL_CUDA(cudaFuncSetAttribute(score_monomer_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      score_monomer_kernel<1><<<grid, MONO_THREADS, smem, cs>>>(a); break;
  }
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}
int mono_exact_parts(int64_t Q, int64_t N, int K, int d) { return mono_plan(Q, N, K, d).parts; }

// The same for the source direction (score_monomer_src_kernel): every S-th tile, the flagged query tiles, or (tile_stride
// 1, redo_tile NULL) the whole catalog.
int mono_src_exact_launch(const float* Pq, int64_t ldq, int64_t Q, int K, int d, const float* Ac, int64_t lda,
                          const float* Wc, int64_t N, int kk, int tile_stride, const int* redo_tile, tkey_t* keys,
                          int* counts, int* parts_out, cudaStream_t cs) {
  MonoPlan plan = mono_src_plan(Q, N > 0 ? N : 1, K, d);
  *parts_out = plan.parts;
  if (N == 0) {
    CFL_CUDA(cudaMemsetAsync(counts, 0, (size_t)plan.parts * Q * sizeof(int), cs));
    return CFL_OK;
  }
  MonoSrcArgs a;
  a.K = K; a.d = d; a.Q = Q; a.N = N; a.ldq = ldq; a.lda = lda; a.P = Pq; a.A = Ac; a.W = Wc;
  a.keys = keys; a.counts = counts;
  a.parts = plan.parts; a.kk = kk; a.tiles = plan.tiles; a.tile_stride = tile_stride; a.redo_tile = redo_tile;
  const size_t smem = mono_src_smem_bytes(K, d);
  CFL_CUDA(cudaFuncSetAttribute(score_monomer_src_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  score_monomer_src_kernel<<<dim3(plan.parts, plan.nqt), MONO_THREADS, smem, cs>>>(a);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}
int mono_src_exact_parts(int64_t Q, int64_t N, int K, int d) { return mono_src_plan(Q, N > 0 ? N : 1, K, d).parts; }
int mono_merge_launch(const tkey_t* keys, const int* counts, int parts, int64_t Q, int k, int64_t idx_base, float* top_val,
                      int64_t* top_idx, const float* only_redo, cudaStream_t cs) {
  merge_plain_kernel<<<(unsigned)Q, MRG_THREADS, 0, cs>>>(keys, counts, parts, Q, k, k, idx_base, top_val, top_idx, only_redo);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

}  // namespace cfl

using namespace cfl;

extern "C" {

size_t cfl_score_topk_monomer_workspace_bytes(int64_t Q, int K, int d, int64_t N, int k) {
  (void)k;
  if (Q <= 0) return 4096;
  MonoPlan p = mono_plan(Q, N > 0 ? N : 1, K, d);
  return align_up((size_t)p.parts * Q * MONO_KSTRIDE * sizeof(tkey_t), 256) +
         align_up((size_t)p.parts * Q * sizeof(int), 256) + 1024;
}

int cfl_score_topk_monomer(const float* Aq, int64_t lda, const float* Wq, int64_t Q, int K, int d,
                           const float* Pc, int64_t N, int64_t ldp, int k, int64_t idx_base,
                           float* top_val, int64_t* top_idx, float* dist_out,
                           void* ws, size_t ws_bytes, void* stream) {
  int st = device_check();
  if (st != CFL_OK) return st;
  cudaStream_t cs = (cudaStream_t)stream;
  CFL_REQUIRE(K >= 1 && K <= CFL_MAX_K, CFL_ERR_UNSUPPORTED, "score_topk_monomer: K=%d outside [1,%d]", K, CFL_MAX_K);
  CFL_REQUIRE(d >= 1 && d <= 128, CFL_ERR_UNSUPPORTED, "score_topk_monomer: d=%d outside [1,128]", d);
  CFL_REQUIRE(k >= 1 && k <= CFL_MAX_TOPK, CFL_ERR_UNSUPPORTED, "score_topk_monomer: k=%d outside [1,%d]", k, CFL_MAX_TOPK);
  CFL_REQUIRE(Q >= 0 && N >= 0 && N < ((int64_t)1 << 32), CFL_ERR_INVALID, "score_topk_monomer: bad Q/N");
  CFL_REQUIRE(lda >= d && ldp >= (int64_t)K * d, CFL_ERR_INVALID, "score_topk_monomer: leading dimension too small");
  if (Q == 0) return CFL_OK;
  CFL_REQUIRE(Aq && Wq && top_val && top_idx, CFL_ERR_INVALID, "score_topk_monomer: NULL argument");
  CFL_REQUIRE(N == 0 || Pc, CFL_ERR_INVALID, "score_topk_monomer: NULL catalog");
  MonoPlan plan = mono_plan(Q, N > 0 ? N : 1, K, d);
  const size_t keys_bytes = align_up((size_t)plan.parts * Q * MONO_KSTRIDE * sizeof(tkey_t), 256);
  const size_t need = keys_bytes + align_up((size_t)plan.parts * Q * sizeof(int), 256);
  CFL_REQUIRE(ws && ws_bytes >= need, CFL_ERR_WORKSPACE, "score_topk_monomer: workspace too small (%zu < %zu)",
              ws_bytes, need);
  MonoArgs a;
  a.K = K; a.d = d; a.Q = Q; a.N = N; a.lda = lda; a.ldp = ldp; a.A = Aq; a.W = Wq; a.P = Pc;
  a.keys = (tkey_t*)ws; a.counts = (int*)((char*)ws + keys_bytes); a.dist_out = dist_out;
  a.parts = plan.parts; a.kk = k; a.tiles = plan.tiles; a.tile_stride = 1; a.redo_tile = nullptr;
  if (N == 0) {
    CFL_CUDA(cudaMemsetAsync(a.counts, 0, (size_t)plan.parts * Q * sizeof(int), cs));
  } else {
    const size_t smem = mono_smem_bytes(K, d);
    const char* ev = getenv("CFL_MONO_VW");
    const int vmax = ev ? atoi(ev) : 4;
    int vw = 1;
    if (vmax >= 4 && d % 4 == 0 && ldp % 4 == 0 && ((uintptr_t)Pc & 15u) == 0) vw = 4;
    else if (vmax >= 2 && d % 2 == 0 && ldp % 2 == 0 && ((uintptr_t)Pc & 7u) == 0) vw = 2;
    dim3 grid(plan.parts, plan.nqt);
#define CFL_MONO_CASE(VV)                                                                                          \
  case VV:                                                                                                         \
    CFL_CUDA(cudaFuncSetAttribute(score_monomer_kernel<VV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
    timer_record(0, cs);                                                                                           \
    score_monomer_kernel<VV><<<grid, MONO_THREADS, smem, cs>>>(a);                                                 \
    break;
    switch (vw) { CFL_MONO_CASE(4) CFL_MONO_CASE(2) default: CFL_MONO_CASE(1) }
#undef CFL_MONO_CASE
    timer_record(1, cs);
    CFL_LAUNCH_CHECK();
  }
  merge_plain_kernel<<<(unsigned)Q, MRG_THREADS, 0, cs>>>(a.keys, a.counts, plan.parts, Q, a.kk, k, idx_base,
                                                          top_val, top_idx);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

}  // extern "C"
