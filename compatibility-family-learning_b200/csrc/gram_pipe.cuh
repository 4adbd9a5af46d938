// The tcgen05 Gram pipeline of the exact kernels: score_umma_kernel (score_umma.cu) and rank_count_umma_kernel /
// within_emit_umma_kernel (rank_counts_tc.cu) run it and differ only in their epilogues.
//
//   D[c, k*QT + q] = e_c . p_{q,k}        M = 128 catalog rows (TMEM lanes), N = NC = K*QT columns,
//                                         MMA-K = the embedding dimension (8 per K-step), 3xTF32 (umma.cuh)
//
// The source-catalog kernel score_src_umma_kernel (score_umma.cu) runs the same pipeline in the other direction: the
// catalog rows carry K prototype planes and the query tile one vector per query, D[c, k*QT + q] = p_{c,k} . e_q.  Its
// tiles have PLANES = K A planes, each multiplied by the same QT-column B image into its own QT columns (gram_mma /
// gram_tma template argument; 1 for the other kernels).
//
// A CTA (part, qtile) keeps its query tile's tf32 hi/lo image resident in shared memory and streams a range of 128-row
// tiles of the packed catalog image (score_umma.cu).  18 warps:
//   warp  GP_NEPI      one lane issues tcgen05.mma (3 per K-step) and tcgen05.commit       (gram_mma)
//   warp  GP_NEPI+1    one lane drives the TMA engine: cp.async.bulk of the query image, then one or two 8 KB K-steps
//                      of the catalog per ring stage (mbarrier expect_tx / complete_tx)      (gram_tma)
//   warps 0..GP_NEPI-1 the caller's epilogue: four warps per TMEM lane quarter, the thread's TMEM lane = its catalog
//                      row; gram_load_group reads the K Gram values of a group of queries.  The accumulators are
//                      double-buffered in TMEM (2*NC columns) so the epilogue of tile t overlaps the MMAs of tile t+1.
#pragma once
#include "score.cuh"
#include "umma.cuh"

namespace cfl {

constexpr int GP_NEPI = 16;                         // epilogue warps (TMEM lane quarters x 4)
constexpr int GP_WPQ = GP_NEPI / 4;                 // epilogue warps per TMEM lane quarter
constexpr int GP_EPI_THREADS = GP_NEPI * 32;
constexpr int GP_THREADS = (GP_NEPI + 2) * 32;      // + the MMA warp and the TMA warp
constexpr int GP_NSTAGE = 6;                        // ring stages of up to 2 K-steps (16 KB) each
constexpr uint32_t GP_ASTAGE = 4u * 128u * 16u;     // one K-step of the catalog image: [hl][chunk][128 rows][16 B] = 8 KB

// queries per epilogue group: K x GQ Gram values are live per thread (register budget)
__host__ __device__ constexpr int gram_gq(int K) { return K <= 2 ? 16 : (K <= 4 ? 8 : 4); }

// Shared memory of one CTA: the query image, the catalog ring, the caller's front region (front_bytes, a multiple of 16),
// the pair-interleaved soft-min (qpar) and plane-bound (qpl) blocks, the caller's back region from `back` on, then the
// mbarriers and the TMEM address slot, placed by gram_layout_end once the caller knows where its back region ends.
// The front region sits at a fixed distance from the 1024-aligned end of the query image, so the epilogue addresses a
// buffer there with an immediate offset instead of one more live register.
// SRC (the source-catalog kernel): a query image of QT vectors, and qpar holds one float per query, |e_q - mu|^2; no
// plane-bound block.
struct GramLayout { uint32_t b_img, a_ring, front, qpar, qpl, back, bars, tmem_slot, total; };
template <bool SRC = false>
__host__ __device__ inline GramLayout gram_layout(int K, int qt, int dpad, uint32_t front_bytes) {
  GramLayout L;
  uint32_t off = 0;
  L.b_img = off;   off += qimg_tile_bytes(dpad, SRC ? qt : K * qt);           off = (off + 1023u) & ~1023u;
  L.a_ring = off;  off += GP_NSTAGE * 2u * GP_ASTAGE;
  L.front = off;   off += front_bytes;
  L.qpar = off;    off += (uint32_t)qt * (uint32_t)(SRC ? 1 : qpar_stride(K)) * 4u;      off = (off + 15u) & ~15u;
  L.qpl = off;     off += (uint32_t)qt * (uint32_t)(SRC ? 0 : qplane_stride(K)) * 4u;    off = (off + 15u) & ~15u;
  L.back = off;
  return L;
}
__host__ __device__ inline void gram_layout_end(GramLayout& L, uint32_t back_end) {
  uint32_t off = (back_end + 15u) & ~15u;
  L.bars = off;    off += (2u * GP_NSTAGE + 5u) * 8u;
  L.tmem_slot = off; off += 16u;
  L.total = off;
}

struct GramPipe {
  unsigned char* b_img;
  unsigned char* a_ring;
  float* qpar;
  float* qpl;
  uint64_t* full;       // [GP_NSTAGE] ring stage loaded      (TMA -> MMA)
  uint64_t* empty;      // [GP_NSTAGE] ring stage consumed    (MMA -> TMA)
  uint64_t* tfull;      // [2] accumulator buffer complete    (MMA -> epilogue)
  uint64_t* tempty;     // [2] accumulator buffer read        (epilogue -> MMA)
  uint64_t* bfull;      // query image resident               (TMA -> MMA)
  uint32_t* tmem_slot;
  int NC;               // accumulator columns per buffer: K * QT
  int nks, kss;         // K-steps per tile, K-steps per ring stage
  uint32_t ncols;       // TMEM columns allocated: 2 * NC rounded up to a power of two
};

__device__ __forceinline__ GramPipe gram_pipe(unsigned char* smem, const GramLayout& L, int K, int QT, int dpad) {
  GramPipe P;
  P.b_img = smem + L.b_img;
  P.a_ring = smem + L.a_ring;
  P.qpar = (float*)(smem + L.qpar);
  P.qpl = (float*)(smem + L.qpl);
  P.full = (uint64_t*)(smem + L.bars);
  P.empty = P.full + GP_NSTAGE;
  P.tfull = P.empty + GP_NSTAGE;
  P.tempty = P.tfull + 2;
  P.bfull = P.tempty + 2;
  P.tmem_slot = (uint32_t*)(smem + L.tmem_slot);
  P.NC = K * QT;
  P.nks = dpad / 8;
  P.kss = (P.nks % 2 == 0) ? 2 : 1;
  P.ncols = 32;
  while ((int)P.ncols < 2 * P.NC) P.ncols <<= 1;
  return P;
}

// First half of the one-time setup: barriers and TMEM columns (MMA warp).
__device__ __forceinline__ void gram_init(const GramPipe& P) {
  const int tid = threadIdx.x, warp = tid >> 5;
  if (warp == GP_NEPI) {
    if ((tid & 31) == 0) {
      for (int s = 0; s < GP_NSTAGE; ++s) { umma::mbar_init(&P.full[s], 1); umma::mbar_init(&P.empty[s], 1); }
      umma::mbar_init(&P.tfull[0], 1); umma::mbar_init(&P.tfull[1], 1);
      umma::mbar_init(&P.tempty[0], GP_EPI_THREADS); umma::mbar_init(&P.tempty[1], GP_EPI_THREADS);
      umma::mbar_init(P.bfull, 1);
      umma::fence_barrier_init();
    }
    __syncwarp();
    umma::tmem_alloc(P.tmem_slot, P.ncols);
  }
}

// gram_init, and the per-query blocks of queries [q0, q0 + nq) stored interleaved by query PAIR,
// qpar[(pair*QPS + j)*2 + (q&1)], with the soft-min block's first K entries negated: ready for softmin_pair /
// plane_bound_pair.  The padding queries of the tile get zeros.  The caller stages its own epilogue state, then calls
// gram_start.
template <int K>
__device__ __forceinline__ void gram_setup(const GramPipe& P, const float* __restrict__ qpar,
                                           const float* __restrict__ qplane, int64_t q0, int nq, int QT) {
  const int tid = threadIdx.x;
  gram_init(P);
  constexpr int QPS = qpar_stride(K);
  for (int i = tid; i < QT * QPS; i += GP_THREADS) {
    const int ql = i / QPS, j = i % QPS;
    float v = (ql < nq) ? qpar[(q0 + ql) * QPS + j] : 0.0f;
    if (j < K) v = -v;
    P.qpar[((ql >> 1) * QPS + j) * 2 + (ql & 1)] = v;
  }
  constexpr int PBS = qplane_stride(K);
  for (int i = tid; i < QT * PBS; i += GP_THREADS) {
    const int ql = i / PBS, j = i % PBS;
    P.qpl[((ql >> 1) * PBS + j) * 2 + (ql & 1)] = (ql < nq) ? qplane[(q0 + ql) * PBS + j] : 0.0f;
  }
}

// Second half: every thread's staging is visible and the TMEM allocation is known.  Returns the TMEM base address.
__device__ __forceinline__ uint32_t gram_start(const GramPipe& P) {
  umma::tc_fence_before();
  __syncthreads();
  umma::tc_fence_after();
  return *P.tmem_slot;
}

// MMA warp: one lane issues the A-steps of ntiles catalog tiles, tile t into accumulator buffer t & 1.  A tile is
// PLANES * nks A-steps; step s multiplies A block s by B K-step s % nks into the columns [(s / nks) * N, +N) of the
// buffer, N = NC / PLANES, starting a fresh sum when s % nks == 0.
template <int PLANES = 1>
__device__ __forceinline__ void gram_mma(const GramPipe& P, uint32_t tmem_base, int ntiles) {
  using namespace umma;
  if (!elect_one()) return;
  mbar_wait(P.bfull, 0);
  const uint32_t N = (uint32_t)(P.NC / PLANES);
  const Step3Desc sd = make_step3(N, make_idesc_tf32(128, N));
  const uint32_t a_base = smem_u32(P.a_ring), b_base = smem_u32(P.b_img);
  const uint32_t b_step = 4u * N * 16u;
  int stage = 0; uint32_t phase = 0;
  for (int t = 0; t < ntiles; ++t) {
    const int buf = t & 1;
    mbar_wait(&P.tempty[buf], ((uint32_t)(t >> 1) & 1u) ^ 1u);
    tc_fence_after();
    const uint32_t d_tmem = tmem_base + (uint32_t)(buf * P.NC);
    for (int s = 0; s < PLANES * P.nks; s += P.kss) {
      mbar_wait(&P.full[stage], phase);
      tc_fence_after();
      const int ks = PLANES == 1 ? s : s % P.nks;             // kss divides nks: a stage never straddles two planes
      const uint32_t d_col = PLANES == 1 ? d_tmem : d_tmem + (uint32_t)(s / P.nks) * N;
      for (int j = 0; j < P.kss; ++j)
        mma_step3(sd, d_col, a_base + (stage * 2 + j) * GP_ASTAGE, b_base + (ks + j) * b_step, ks + j == 0);
      mma_commit(&P.empty[stage]);
      if (++stage == GP_NSTAGE) { stage = 0; phase ^= 1u; }
    }
    mma_commit(&P.tfull[buf]);
  }
}

// TMA warp: one lane loads query tile qtile's image, then streams the catalog tiles t0, t0 + ts, ... (ntiles of them,
// PLANES * nks A blocks each) through the ring.
template <int PLANES = 1>
__device__ __forceinline__ void gram_tma(const GramPipe& P, const void* qimg, int qtile, const void* cimg, int64_t t0,
                                         int ts, int ntiles) {
  using namespace umma;
  if (!elect_one()) return;
  const uint32_t bbytes = qimg_tile_bytes(8 * P.nks, P.NC / PLANES);
  const unsigned char* qsrc = (const unsigned char*)qimg + (size_t)qtile * bbytes;
  mbar_arrive_expect_tx(P.bfull, bbytes);
  for (uint32_t o = 0; o < bbytes; o += 32768u) {
    uint32_t n = bbytes - o < 32768u ? bbytes - o : 32768u;
    bulk_g2s(P.b_img + o, qsrc + o, n, P.bfull);
  }
  int stage = 0; uint32_t phase = 0;
  for (int t = 0; t < ntiles; ++t) {
    const unsigned char* src = (const unsigned char*)cimg + (size_t)(t0 + (int64_t)t * ts) * PLANES * P.nks * GP_ASTAGE;
    for (int ks = 0; ks < PLANES * P.nks; ks += P.kss) {
      mbar_wait(&P.empty[stage], phase ^ 1u);
      mbar_arrive_expect_tx(&P.full[stage], (uint32_t)P.kss * GP_ASTAGE);
      bulk_g2s(P.a_ring + stage * 2 * GP_ASTAGE, src + (size_t)ks * GP_ASTAGE, (uint32_t)P.kss * GP_ASTAGE, &P.full[stage]);
      if (++stage == GP_NSTAGE) { stage = 0; phase ^= 1u; }
    }
  }
}

// Epilogue: waits for tile t's accumulators; returns the TMEM address of lane quarter lq in its buffer.
__device__ __forceinline__ uint32_t gram_acquire(const GramPipe& P, uint32_t tmem_base, int t, int lq) {
  const int buf = t & 1;
  umma::mbar_wait(&P.tfull[buf], (uint32_t)(t >> 1) & 1u);
  umma::tc_fence_after();
  return tmem_base + ((uint32_t)(lq * 32) << 16) + (uint32_t)(buf * P.NC);
}
// Epilogue: this thread is done reading tile t's accumulators.
__device__ __forceinline__ void gram_release(const GramPipe& P, int t) {
  umma::tc_fence_before();
  umma::mbar_arrive(&P.tempty[t & 1]);
}

// gk[k][i] = e . p_{k} of query g*GQ + i, for the thread's catalog row
template <int K, int GQ>
__device__ __forceinline__ void gram_load_group(uint32_t taddr, int QT, int g, float (&gk)[K][GQ]) {
#pragma unroll
  for (int k = 0; k < K; ++k) {
    if constexpr (GQ == 16)     umma::tmem_ld16(taddr + (uint32_t)(k * QT + g * GQ), gk[k]);
    else if constexpr (GQ == 8) umma::tmem_ld8(taddr + (uint32_t)(k * QT + g * GQ), gk[k]);
    else                        umma::tmem_ld4(taddr + (uint32_t)(k * QT + g * GQ), gk[k]);
  }
  umma::tmem_ld_wait();
}

// The N-float blocks of a query pair, interleaved as gram_setup stores them: v[j] = (block_A[j], block_B[j]).
template <int N>
__device__ __forceinline__ void load_pair_block(const float* blk, f2_t (&v)[N]) {
  const ulonglong2* src = (const ulonglong2*)blk;
#pragma unroll
  for (int j = 0; j < N; j += 2) { const ulonglong2 u = src[j >> 1]; v[j] = u.x; v[j + 1] = u.y; }
}

// The MMA warp frees the TMEM columns once every role is done.
__device__ __forceinline__ void gram_finish(const GramPipe& P, uint32_t tmem_base) {
  umma::tc_fence_before();
  __syncthreads();
  if ((threadIdx.x >> 5) == GP_NEPI) umma::tmem_dealloc(tmem_base, P.ncols);
}

}  // namespace cfl
