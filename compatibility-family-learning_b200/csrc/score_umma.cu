// Fused all-pairs scoring kernel for sm_100a: the Gram pipeline of gram_pipe.cuh (3xTF32 tcgen05.mma into double-
// buffered TMEM accumulators) with a soft-min epilogue and running per-query top-k behind the MMA; the Q x N score matrix
// never reaches HBM.
//
// Both operands are consumed as pre-split (hi, lo) tf32 images in the canonical K-major SWIZZLE_NONE layout (umma.cuh),
// both laid out by this file:
//   * the CATALOG image is built once per catalog by cfl_catalog_pack (centred on mu, split, one 8 KB block per (tile,
//     K-step), plus |e|^2 per row and the lower-bound pass's planes) -- the catalog is static across query batches, so
//     no per-query work is spent on it;
//   * the QUERY image of the CTA's query tile (<= 96 KB) is packed per call and stays resident in shared memory for the
//     whole kernel.
// Epilogue (16 warps): the K Gram values of a group of 4, 8 or 16 queries for the thread's catalog row, the affine-hull
// lower bound and the soft-min distance (score.cuh), threshold test, warp-aggregated push into the per-query buffers
// (topk.cuh), cooperative compaction of over-full buffers.
// Work per score: 2*K*d flops (x3 MMAs); catalog bytes per row per query tile: 8*dpad + 4.
//
// score_src_umma_kernel is the same kernel for the other direction of the asymmetric pcd distance (cfl_score_topk_source):
// the catalog rows are SOURCE items with K prototypes each (cfl_source_catalog_pack: K planes of tf32 blocks per tile and
// each row's soft-min block), the queries are TARGET embeddings (one vector each).  The Gram values land in TMEM where the
// forward kernel puts them; the soft-min constants belong to the row and |e_q|^2 to the query.  It has no plane bound: the
// affine hull is per row.  Catalog bytes per row per query tile: K*8*dpad + 4*(K + K(K+1)/2).
#include <cuda_fp16.h>
#include "gram_pipe.cuh"

namespace cfl {

using namespace umma;

constexpr size_t SU_B_BUDGET = 96 * 1024;             // query image per CTA

int score_umma_qt(int K, int d) {
  if (K < 1 || K > CFL_MAX_K || d < 1 || d > 128) return 0;
  const int dpad = (d + 7) / 8 * 8;
  const int gq = K <= 2 ? 16 : (K <= 4 ? 8 : 4);
  const int cand[] = {128, 64, 48, 32, 16, 8};
  for (int qt : cand) {
    int nc = K * qt;
    if (nc > 256 || nc % 16 != 0 || qt % gq != 0) continue;
    if (qimg_tile_bytes(dpad, nc) > SU_B_BUDGET) continue;
    return qt;
  }
  return 0;
}

bool score_umma_supported(int K, int d) {
  if (getenv("CFL_FORCE_SIMT")) return false;
  return score_umma_qt(K, d) != 0;
}

// ---- catalog image ----------------------------------------------------------------------------
// [tile][kstep][hl][chunk][row 0..127][4 floats]  (8 KB per (tile,kstep)), then e2[tiles*128].
// ... then the fp16 plane of the lower-bound pass: [tile][kstep16][chunk 0|1][row 0..127][8 halfs] (4 KB per
// (tile, 16 columns)), then one flag word (non-zero: a centred value left the fp16 range, plane unusable).
static size_t catalog_e2_offset(int64_t N, int d) {
  return (size_t)((N + 127) / 128) * ((d + 7) / 8) * GP_ASTAGE;
}
static size_t catalog_f16_offset(int64_t N, int d) {
  return catalog_e2_offset(N, d) + (size_t)((N + 127) / 128) * 128 * sizeof(float);
}
static size_t catalog_f16_bytes(int64_t N, int d) {
  const int64_t tiles = (N + 127) / 128;
  return (size_t)tiles * ((d + 15) / 16) * (GP_ASTAGE / 2);
}
// ... then lbrow[tiles*128] float2 = (|e - mu|^2, |e - mu|) per row, (+inf, 0) for the padding rows of the last tile:
// what the lower-bound pass needs per row (its margin has a term in |e|), one 8-byte load per row and tile.
static size_t catalog_lbrow_offset(int64_t N, int d) {
  return catalog_f16_offset(N, d) + catalog_f16_bytes(N, d) + 16;
}
size_t catalog_image_bytes(int64_t N, int d) {
  const int64_t tiles = (N + 127) / 128;
  return catalog_lbrow_offset(N, d) + (size_t)tiles * 128 * sizeof(float2);
}
CatalogView catalog_view(const void* image, int64_t N, int d) {
  unsigned char* img = (unsigned char*)const_cast<void*>(image);
  CatalogView v;
  v.e2 = (float*)(img + catalog_e2_offset(N, d));
  v.f16 = img + catalog_f16_offset(N, d);
  v.flag16 = (int*)(v.f16 + catalog_f16_bytes(N, d));
  v.lbrow = (float2*)(img + catalog_lbrow_offset(N, d));
  return v;
}

__global__ void __launch_bounds__(128)
pack_catalog_kernel(const float* __restrict__ E, int64_t N, int d, int64_t lde,
                    const float* __restrict__ mu, unsigned char* __restrict__ img, float* __restrict__ e2g,
                    unsigned char* __restrict__ img16, int* __restrict__ flag16, float2* __restrict__ lbrow) {
  const int64_t tile = blockIdx.x;
  const int r = threadIdx.x;
  const int64_t row = tile * 128 + r;
  const int nks = (d + 7) / 8;
  float e2 = 0.0f;
  float vmax = 0.0f;
  const int nks16 = (d + 15) / 16;
  for (int ks = 0; ks < nks; ++ks) {
    float v[8];
#pragma unroll
    for (int jj = 0; jj < 8; ++jj) {
      const int j = ks * 8 + jj;
      v[jj] = (row < N && j < d) ? E[row * lde + j] - (mu ? mu[j] : 0.0f) : 0.0f;
      e2 = fmaf(v[jj], v[jj], e2);
    }
    float4 h0, l0, h1, l1;
    split_tf32x4(make_float4(v[0], v[1], v[2], v[3]), h0, l0);
    split_tf32x4(make_float4(v[4], v[5], v[6], v[7]), h1, l1);
    unsigned char* st = img + ((size_t)tile * nks + ks) * GP_ASTAGE;
    *(float4*)(st + ((0 * 2 + 0) * 128 + r) * 16) = h0;
    *(float4*)(st + ((0 * 2 + 1) * 128 + r) * 16) = h1;
    *(float4*)(st + ((1 * 2 + 0) * 128 + r) * 16) = l0;
    *(float4*)(st + ((1 * 2 + 1) * 128 + r) * 16) = l1;
    // the same 8 centred values as halfs: chunk (ks & 1) of fp16 K-step ks >> 1
    __align__(16) __half h[8];
#pragma unroll
    for (int jj = 0; jj < 8; ++jj) { h[jj] = __float2half_rn(v[jj]); vmax = fmaxf(vmax, fabsf(v[jj])); }
    unsigned char* st16 = img16 + ((size_t)tile * nks16 + (ks >> 1)) * (GP_ASTAGE / 2);
    *(uint4*)(st16 + ((ks & 1) * 128 + r) * 16) = *(const uint4*)h;
  }
  if (nks & 1) {                                             // odd number of 8-column steps: zero the last half K-step
    unsigned char* st16 = img16 + ((size_t)tile * nks16 + (nks >> 1)) * (GP_ASTAGE / 2);
    *(uint4*)(st16 + (1 * 128 + r) * 16) = make_uint4(0u, 0u, 0u, 0u);
  }
  e2g[row] = e2;
  lbrow[row] = (row < N) ? make_float2(e2, sqrtf(e2)) : make_float2(__int_as_float(0x7f800000), 0.0f);
  if (!(vmax < 60000.0f)) atomicOr(flag16, 1);               // also catches NaN / inf
}

int catalog_pack_launch(const float* E, int64_t N, int d, int64_t lde, const float* mu, void* image,
                        cudaStream_t st) {
  const int64_t tiles = (N + 127) / 128;
  const CatalogView v = catalog_view(image, N, d);
  CFL_CUDA(cudaMemsetAsync(v.flag16, 0, 16, st));
  pack_catalog_kernel<<<(unsigned)tiles, 128, 0, st>>>(E, N, d, lde, mu, (unsigned char*)image, v.e2, v.f16, v.flag16,
                                                       v.lbrow);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

// ---- source-catalog image ----------------------------------------------------------------------
// [tile][k][kstep][hl][chunk][row 0..127][4 floats]  (8 KB per (tile, k, kstep): prototype k of the tile's rows, centred on
// mu, in the block format of the catalog image), then rowpar[tile][j][row 0..127], j < K + K(K+1)/2: log2(e)*|p_k|^2 and
// the upper triangle of p_k.p_l with the diagonal pre-halved (the first entries of the qpar format, score.cuh), zeros for
// the padding rows of the last tile.  The epilogue reads its row's block once per tile, coalesced.
static size_t source_rowpar_offset(int64_t N, int K, int d) {
  return (size_t)((N + 127) / 128) * K * ((d + 7) / 8) * GP_ASTAGE;
}
size_t source_catalog_image_bytes(int64_t N, int K, int d) {
  return source_rowpar_offset(N, K, d) + (size_t)((N + 127) / 128) * 128 * source_rowpar_len(K) * sizeof(float);
}
SourceCatalogView source_catalog_view(const void* image, int64_t N, int K, int d) {
  unsigned char* img = (unsigned char*)const_cast<void*>(image);
  return SourceCatalogView{img, (float*)(img + source_rowpar_offset(N, K, d))};
}

template <int K>
__global__ void __launch_bounds__(128)
pack_source_catalog_kernel(const float* __restrict__ P, int64_t N, int d, int64_t ldp, const float* __restrict__ mu,
                           unsigned char* __restrict__ img, float* __restrict__ rowpar) {
  const int64_t tile = blockIdx.x;
  const int r = threadIdx.x;
  const int64_t row = tile * 128 + r;
  const bool valid = row < N;
  const float* src = P + (valid ? row : 0) * ldp;
  const int nks = (d + 7) / 8;
  constexpr int T = qpar_tri(K);
  float tri[T];
#pragma unroll
  for (int o = 0; o < T; ++o) tri[o] = 0.0f;
  for (int ks = 0; ks < nks; ++ks) {
    float v[K][8];
#pragma unroll
    for (int k = 0; k < K; ++k)
#pragma unroll
      for (int jj = 0; jj < 8; ++jj) {
        const int j = ks * 8 + jj;
        v[k][jj] = (valid && j < d) ? src[k * d + j] - (mu ? mu[j] : 0.0f) : 0.0f;
      }
    int o = 0;
#pragma unroll
    for (int k = 0; k < K; ++k)
#pragma unroll
      for (int l = k; l < K; ++l, ++o)
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) tri[o] = fmaf(v[k][jj], v[l][jj], tri[o]);
#pragma unroll
    for (int k = 0; k < K; ++k) {
      float4 h0, l0, h1, l1;
      split_tf32x4(make_float4(v[k][0], v[k][1], v[k][2], v[k][3]), h0, l0);
      split_tf32x4(make_float4(v[k][4], v[k][5], v[k][6], v[k][7]), h1, l1);
      unsigned char* st = img + (((size_t)tile * K + k) * nks + ks) * GP_ASTAGE;
      *(float4*)(st + ((0 * 2 + 0) * 128 + r) * 16) = h0;
      *(float4*)(st + ((0 * 2 + 1) * 128 + r) * 16) = h1;
      *(float4*)(st + ((1 * 2 + 0) * 128 + r) * 16) = l0;
      *(float4*)(st + ((1 * 2 + 1) * 128 + r) * 16) = l1;
    }
  }
  float* rp = rowpar + (size_t)tile * 128 * source_rowpar_len(K) + r;
  int o = 0;
#pragma unroll
  for (int k = 0; k < K; ++k)
#pragma unroll
    for (int l = k; l < K; ++l, ++o) {
      if (l == k) rp[k * 128] = CFL_LOG2E * tri[o];
      rp[(K + o) * 128] = (l == k) ? 0.5f * tri[o] : tri[o];
    }
}

int source_catalog_pack_launch(const float* P, int64_t N, int K, int d, int64_t ldp, const float* mu, void* image,
                               cudaStream_t st) {
  const SourceCatalogView v = source_catalog_view(image, N, K, d);
  return with_k(K, [&](auto KC) {
    pack_source_catalog_kernel<KC><<<(unsigned)((N + 127) / 128), 128, 0, st>>>(P, N, d, ldp, mu, v.blocks, v.rowpar);
    CFL_LAUNCH_CHECK();
    return CFL_OK;
  });
}

// Query tile of the source-catalog kernel: QT vectors, a valid MMA N (a multiple of 16) with K*QT <= 256 TMEM columns
// per accumulator buffer; QT = 16 always qualifies, so every K <= 8 and d <= 128 has a tiling.
int score_src_qt(int K, int d) {
  if (K < 1 || K > CFL_MAX_K || d < 1 || d > 128) return 0;
  const int dpad = (d + 7) / 8 * 8;
  const int cand[] = {128, 64, 48, 32, 16};
  for (int qt : cand) {
    if (K * qt > 256 || qt % gram_gq(K) != 0) continue;
    if (qimg_tile_bytes(dpad, qt) > SU_B_BUDGET) continue;
    return qt;
  }
  return 0;
}

// Shared memory of the exact kernel: the Gram pipeline's regions with the compaction scratch in front of the query blocks
// and, behind them, running thresholds, key counts and compaction requests.
struct SuLayout { GramLayout g; uint32_t thr, cnt, need; };
template <bool SRC = false>
__host__ __device__ inline SuLayout su_layout(int K, int qt, int dpad) {
  SuLayout L;
  L.g = gram_layout<SRC>(K, qt, dpad, TOPK_STRIDE * 8u);
  uint32_t off = L.g.back;
  L.thr = off;     off += (uint32_t)qt * 4u;
  L.cnt = off;     off += (uint32_t)qt * 4u;
  L.need = off;    off += 16u;
  gram_layout_end(L.g, off);
  return L;
}

// ---- query (B operand) image: [qtile][kstep][hl][chunk][row n = k*QT + ql][4 floats] -----------
__global__ void pack_queries_kernel(const float* __restrict__ Pc, int64_t Q, int K, int d, int qt,
                                    int dpad, float* __restrict__ img) {
  const int nc = K * qt;
  const int nks = dpad / 8;
  const int qtile = blockIdx.x;
  float* base = (float*)((char*)img + (size_t)qtile * qimg_tile_bytes(dpad, nc));
  for (int e = threadIdx.x; e < nks * 2 * nc; e += blockDim.x) {
    int n = e % nc;
    int c = (e / nc) % 2;
    int ks = e / (2 * nc);
    int k = n / qt, ql = n % qt;
    int64_t q = (int64_t)qtile * qt + ql;
    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
    float* xp = &x.x;
    if (q < Q) {
      const float* src = Pc + (q * K + k) * (int64_t)d;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        int j = ks * 8 + c * 4 + i;
        if (j < d) xp[i] = src[j];
      }
    }
    float4 hi, lo;
    split_tf32x4(x, hi, lo);
    size_t step = (size_t)ks * 4 * nc;                       // float4 units per K-step: 4*nc
    ((float4*)base)[step + (size_t)(0 * 2 + c) * nc + n] = hi;
    ((float4*)base)[step + (size_t)(1 * 2 + c) * nc + n] = lo;
  }
}

int score_umma_pack_queries(const ScoreArgs& a, void* qimg, cudaStream_t st) {
  pack_queries_kernel<<<a.plan.nqt, 256, 0, st>>>(a.Pc, a.Q, a.src ? 1 : a.K, a.d, a.plan.qt, a.plan.dpad, (float*)qimg);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

__device__ __forceinline__ void epi_bar_sync() {
  asm volatile("bar.sync 1, %0;" ::"n"(GP_EPI_THREADS) : "memory");
}

// ---- the kernels ---------------------------------------------------------------------------
// SRC = false: score_umma_kernel (catalog of embeddings, queries of K prototypes); SRC = true: score_src_umma_kernel
// (catalog of K prototypes per row, queries of one vector).
template <int K, bool SRC>
__device__ __forceinline__ void score_umma_body(const ScoreArgs& A) {
  extern __shared__ __align__(1024) unsigned char smem[];
  constexpr int GQ = gram_gq(K);
  const int QT = A.plan.qt;
  const SuLayout L = su_layout<SRC>(K, QT, A.plan.dpad);
  const GramPipe P = gram_pipe(smem, L.g, K, QT, A.plan.dpad);
  tkey_t* scratch = (tkey_t*)(smem + L.g.front);
  float* thr = (float*)(smem + L.thr);
  int* cnt = (int*)(smem + L.cnt);
  int* need = (int*)(smem + L.need);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int part = blockIdx.x, qtile = blockIdx.y;
  const bool redo = A.redo_tile != nullptr;
  if (redo && A.redo_tile[qtile] == 0) return;               // nothing to redo for this query tile
  const int64_t q0 = (int64_t)qtile * QT;
  const int nq = (int)((A.Q - q0 < QT) ? (A.Q - q0) : QT);
  const int64_t t0 = A.plan.tiles * part / A.plan.parts;
  const int64_t t1 = A.plan.tiles * (part + 1) / A.plan.parts;
  const int ts = A.tile_stride;                              // phase 1 visits every ts-th tile
  const int ntiles = (int)((t1 - t0 + ts - 1) / ts);
  const bool filter = A.phase == 2;

  // ---- one-time setup ----
  if constexpr (SRC) {
    gram_init(P);
    for (int i = tid; i < QT; i += GP_THREADS) P.qpar[i] = (i < nq) ? A.qpar[q0 + i] : 0.0f;     // |e_q - mu|^2
  } else {
    gram_setup<K>(P, A.qpar, A.qplane, q0, nq, QT);
  }
  // padding queries of the last tile get thr = -inf: they can never be pushed
  // phase 2: fixed thresholds from the sample pass, bumped one ulp so that the strict compare
  // below implements dist <= tau (every candidate tied with the bound must be kept)
  for (int i = tid; i < QT; i += GP_THREADS) {
    float th = __int_as_float(i < nq ? 0x7f800000 : 0xff800000);
    if (filter && i < nq && A.thr_init != nullptr) {
      const float tau = A.thr_init[q0 + i];
      th = (tau < 3.0e38f) ? nextafterf(tau, 3.4e38f) : tau;
    }
    thr[i] = th;
    cnt[i] = 0;
  }
  if (tid < 4) need[tid] = 0;
  const uint32_t tmem_base = gram_start(P);

  if (warp == GP_NEPI) {
    gram_mma<SRC ? K : 1>(P, tmem_base, ntiles);
  } else if (warp == GP_NEPI + 1) {
    gram_tma<SRC ? K : 1>(P, A.qimg, qtile, A.cimg, t0, ts, ntiles);
  } else {
    // ======================================= epilogue ========================================
    constexpr int QPS = qpar_stride(K);
    const int lq = warp & 3, sub = warp >> 2;
    const int lrow = lq * 32 + lane;
    const uint32_t lane_lt = (1u << lane) - 1u;
    const bool dense = A.dist_out != nullptr;
    tkey_t* kbase = A.keys + ((int64_t)part * A.Q + q0) * TOPK_STRIDE;
    // dist >= squared distance from e to the affine hull of the query's prototypes (a quadratic in
    // the Gram values, score.cuh): in the usual regime it is within a few percent of dist, so almost
    // every (row, query) is rejected by ~11 packed FMAs per query pair and the soft-min runs only for
    // the queries of a group where some lane survives.  When the bound is loose for the data at hand
    // (prototypes far apart relative to the spread of the distances) each warp measures its hit rate
    // and switches the test off.
    constexpr int PBS = qplane_stride(K);
    bool bound_on = !SRC && (K > 1) && !dense;
    constexpr int NRP = source_rowpar_len(K);
    int grp_seen = 0, grp_skipped = 0;
    for (int t = 0; t < ntiles; ++t) {
      const int64_t tile = t0 + (int64_t)t * ts;
      const int64_t row = tile * 128 + lrow;
      const bool valid = row < A.N;
      float e2 = 0.0f;
      f2_t rq[SRC ? NRP : 1];                                // SRC: the row's soft-min block, broadcast to a query pair
      if constexpr (SRC) {
        const float* rp = A.e2 + tile * 128 * NRP + lrow;
#pragma unroll
        for (int j = 0; j < NRP; ++j) {
          const float v = __ldg(rp + j * 128);
          rq[j] = (j < K) ? pk2(-v, -v) : pk2(v, v);
        }
      } else {
        e2 = __ldg(A.e2 + row);                              // padded to whole tiles
      }
      const uint32_t taddr = gram_acquire(P, tmem_base, t, lq);
      const int nslot = filter ? 2 + ((t >> 2) & 1) : (t & 1);
      const int trig = filter ? TOPK_STRIDE / 2 : TOPK_TRIGGER;
      // push the passing lanes of query ql (warp-uniform call) into its key buffer
      auto push = [&](int ql, bool pass, float dv) {
        const uint32_t m = __ballot_sync(0xffffffffu, pass);
        if (m == 0) return;
        const int leader = __ffs(m) - 1;
        int basei = 0;
        if (lane == leader) {
          basei = atomicAdd(&cnt[ql], __popc(m));
          if (basei + __popc(m) > trig) need[nslot] = 1;
        }
        basei = __shfl_sync(0xffffffffu, basei, leader);
        if (pass) kbase[(int64_t)ql * TOPK_STRIDE + basei + __popc(m & lane_lt)] = pack_key(dv, (uint32_t)row);
      };
      for (int g = sub; g * GQ < nq; g += GP_WPQ) {
        float gk[K][GQ];
        gram_load_group<K, GQ>(taddr, QT, g, gk);
        const float* qg = P.qpar + g * GQ * QPS;               // GQ/2 pair blocks of 2*QPS floats
        float tg[GQ];
#pragma unroll
        for (int i = 0; i < GQ; i += 4) {
          const float4 t4 = *(const float4*)(thr + g * GQ + i);
          tg[i] = t4.x; tg[i + 1] = t4.y; tg[i + 2] = t4.z; tg[i + 3] = t4.w;
        }
        if constexpr (K > 1 && !SRC) {
          if (bound_on) {
            const float e2s = e2 * (1.0f - CFL_PLANE_REL);
            const f2_t e2sp = pk2(e2s, e2s);
            float lb[GQ];
            bool nd = false;
#pragma unroll
            for (int pi = 0; pi < GQ / 2; ++pi) {
              f2_t pv[PBS];
              load_pair_block<PBS>(P.qpl + (g * (GQ / 2) + pi) * PBS * 2, pv);
              float gA[K], gB[K];
#pragma unroll
              for (int k = 0; k < K; ++k) { gA[k] = gk[k][2 * pi]; gB[k] = gk[k][2 * pi + 1]; }
              plane_bound_pair<K>(gA, gB, e2sp, pv, lb[2 * pi], lb[2 * pi + 1]);
              nd |= (lb[2 * pi] < tg[2 * pi]) | (lb[2 * pi + 1] < tg[2 * pi + 1]);
            }
            ++grp_seen;
            if (!__any_sync(0xffffffffu, nd && valid)) { ++grp_skipped; continue; }
            uint32_t nb = 0;
#pragma unroll
            for (int i = 0; i < GQ; ++i) nb |= (lb[i] < tg[i]) ? (1u << i) : 0u;
            if (!valid) nb = 0;
            const uint32_t anyn = __reduce_or_sync(0xffffffffu, nb);
            if (__popc(anyn) <= GQ / 4) {                      // a few queries: soft-min only for those
#pragma unroll
              for (int i = 0; i < GQ; ++i) {
                if (anyn & (1u << i)) {                        // warp-uniform
                  float gi[K];
#pragma unroll
                  for (int k = 0; k < K; ++k) gi[k] = gk[k][i];
                  const float dv = softmin_from_gram_il<K>(gi, e2, qg + (i >> 1) * QPS * 2 + (i & 1));
                  push(g * GQ + i, valid && dv < tg[i], dv);
                }
              }
              continue;
            }
          }
        }
        float dist[GQ];
#pragma unroll
        for (int pi = 0; pi < GQ / 2; ++pi) {
          float gA[K], gB[K];
#pragma unroll
          for (int k = 0; k < K; ++k) { gA[k] = gk[k][2 * pi]; gB[k] = gk[k][2 * pi + 1]; }
          if constexpr (SRC) {
            const f2_t e2q = *(const f2_t*)(P.qpar + g * GQ + 2 * pi);
            softmin_pair2<K>(gA, gB, e2q, rq, dist[2 * pi], dist[2 * pi + 1]);
          } else {
            f2_t qv[QPS];
            load_pair_block<QPS>(qg + pi * QPS * 2, qv);
            softmin_pair<K>(gA, gB, e2, qv, dist[2 * pi], dist[2 * pi + 1]);
          }
        }
        uint32_t bits = 0;
#pragma unroll
        for (int i = 0; i < GQ; ++i) bits |= (dist[i] < tg[i]) ? (1u << i) : 0u;
        if (!valid) bits = 0;
        if (dense && valid && A.phase != 1) {
#pragma unroll
          for (int i = 0; i < GQ; ++i)
            if (g * GQ + i < nq) A.dist_out[(q0 + g * GQ + i) * A.N + row] = dist[i];
        }
        // which queries of the group have at least one passing lane (usually 0-2 of them)
        const uint32_t anyq = __reduce_or_sync(0xffffffffu, bits);
        if (anyq) {
#pragma unroll
          for (int i = 0; i < GQ; ++i)
            if (anyq & (1u << i)) push(g * GQ + i, (bits >> i) & 1u, dist[i]);     // warp-uniform
        }
      }
      // hit-rate check of the plane bound: in the filter pass over tiles [0,16); in the adaptive
      // passes over tiles [16,32), once the running thresholds have tightened
      if (bound_on) {
        if (!filter && t == 15) { grp_seen = 0; grp_skipped = 0; }
        if (t == (filter ? 15 : 31) && grp_skipped * 2 < grp_seen) bound_on = false;
      }
      gram_release(P, t);
      // ---- compaction point: all epilogue warps sort one over-full buffer together ----
      // adaptive phases: checked every tile (a tile adds <= 128 keys per query, buffers hold 512);
      // filter phase: every 4th tile (<= 512 new keys, buffers hold 1024) and it almost never fires.
      // The decision must be identical in every warp although faster warps may already be pushing
      // for the next tile: pushes raise need[slot] (slot = parity of the tile / 4-tile epoch), which
      // is stable once every warp has passed the barrier below.
      if (!filter || (t & 3) == 3) {
        epi_bar_sync();
        if (need[nslot]) {
          for (int qb = 0; qb < nq; qb += 32) {
            const int ql0 = qb + lane;
            const uint32_t over = __ballot_sync(0xffffffffu, ql0 < nq && cnt[ql0] > trig);
            for (uint32_t m = over; m; m &= m - 1) {          // identical in every warp
              const int ql = qb + __ffs(m) - 1;
              if (filter) {
                coop_compact_big<GP_EPI_THREADS>(kbase + (int64_t)ql * TOPK_STRIDE, cnt[ql], A.plan.kk, scratch, tid, &cnt[ql], &thr[ql]);
              } else {
                coop_compact<GP_EPI_THREADS>(kbase + (int64_t)ql * TOPK_STRIDE, cnt[ql], A.plan.kk, scratch, tid, &cnt[ql], &thr[ql]);
              }
            }
          }
          if (tid == 0) need[nslot] = 0;
          epi_bar_sync();
        }
      }
    }
    if (!filter) {
      for (int ql = 0; ql < nq; ++ql) {
        coop_compact<GP_EPI_THREADS>(kbase + (int64_t)ql * TOPK_STRIDE, cnt[ql], A.plan.kk, scratch, tid, &cnt[ql], nullptr);
        if (tid == 0) A.counts[(int64_t)part * A.Q + q0 + ql] = cnt[ql];
      }
    } else {
      epi_bar_sync();                                         // all pushes done; lists stay unsorted
      for (int ql = tid; ql < nq; ql += GP_EPI_THREADS) {
        // a redo launch restarts only the queries it was asked to redo (thr_init > -inf)
        if (redo && !(A.thr_init[q0 + ql] > __int_as_float(0xff800000))) continue;
        A.counts[(int64_t)part * A.Q + q0 + ql] = cnt[ql];
      }
    }
  }
  gram_finish(P, tmem_base);
}

template <int K>
__global__ void __launch_bounds__(GP_THREADS, 1)
score_umma_kernel(ScoreArgs A) {
  score_umma_body<K, false>(A);
}

template <int K>
__global__ void __launch_bounds__(GP_THREADS, 1)
score_src_umma_kernel(ScoreArgs A) {
  score_umma_body<K, true>(A);
}

template <int K, bool SRC>
static int launch_umma(const ScoreArgs& a, cudaStream_t st) {
  size_t smem = su_layout<SRC>(K, a.plan.qt, a.plan.dpad).g.total + 1024;   // slack for the alignment of the dynamic segment
  dim3 grid(a.plan.parts, a.plan.nqt);
  if constexpr (SRC) {
    CFL_SMEM_LIMIT(score_src_umma_kernel<K>, smem);
    score_src_umma_kernel<K><<<grid, GP_THREADS, smem, st>>>(a);
  } else {
    CFL_SMEM_LIMIT(score_umma_kernel<K>, smem);
    score_umma_kernel<K><<<grid, GP_THREADS, smem, st>>>(a);
  }
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

int score_umma_launch(const ScoreArgs& a, cudaStream_t st) {
  return with_k(a.K, [&](auto K) { return a.src ? launch_umma<K, true>(a, st) : launch_umma<K, false>(a, st); });
}

}  // namespace cfl
