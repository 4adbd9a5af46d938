// Lower-bound filter pass of the all-pairs scoring (phase 3 of cfl_score_topk on long catalogs): its own tiling,
// its own query image, its own kernel.  See score_umma.cu for the exact 3xTF32 kernel and score.cu for the host side.
#include <cuda_fp16.h>
#include <stdlib.h>
#include "score.cuh"
#include "umma.cuh"

namespace cfl {

using namespace umma;

// =====================================================================================================
// Lower-bound filter pass (phase 3): the dominant launch of a long-catalog call.
//
// dist(e, q) = |e - sum_k s_k p_k|^2 with s in the simplex, hence dist >= the squared distance from e to the AFFINE
// HULL of the query's prototypes.  With a = the point of that hull closest to the origin (the catalog mean: both
// sides are centred) and u_1..u_{K-1} an orthonormal basis of span{p_j - p_0}, a is orthogonal to every u_j and
//     hull distance^2 = |e|^2 - 2 e.a + |a|^2 - sum_j (e.u_j)^2 .
// The tensor cores produce, per (row, query), the K inner products e.(2a), e.u_1 .. e.u_{K-1} -- ONE fp16 MMA per
// 16 dimensions (kind::f16, fp32 accumulators in TMEM; fp16 carries tf32's 11-bit significand) -- and the epilogue
// decides "bound <= threshold" as
//     e.(2a) - cq(query) + sum_j (e.u_j)^2  >  e2s(row)
// i.e. K-1 packed FP32x2 FMAs and one packed add per query PAIR, then a 3-input max tree and ONE compare per group; nothing else is evaluated, nothing
// is voted on, and a passing (row, query) is appended by its own lane.  The soft-min never runs here: every
// survivor is rescored exactly by rescore_merge_kernel (score.cu), which also verifies the optimistic threshold.
//
// Rigour.  e2s = |e|^2 lowered by a bound on everything the single-product evaluation can lose:
//   * operands rounded to fp16: |d(e.x)| <= u |e||x| + 2^-25 (|e|_1 + |x|_1) (subnormals), u = 1.1 * 2^-10 -- the 0.1
//     covers the fp32 accumulation inside the tensor core, measured at <= 1.6 * 2^-24 |e||x| (tools/tmem_probe.cu,
//     profiles/r2_01_tmem_probe.md);
//   * sum_j C_j^2 >= sum_j c_j^2 - 2 sqrt(K-1) |e| eta,  eta = the bound above with |x| = 1, because sum c_j^2 <= |e|^2;
//   * the fp32 evaluation of both sides (CFL_PLANE_REL |e|^2 and 4K ulp terms).
// cq = |a|^2 - threshold is rounded down.  A value outside the fp16 range (flag words raised by the pack kernels)
// sends the CTA's queries to the exact redo pass (counts = -1).
//
// Pipeline.  Measured on B200 (profiles/r2_02_pass_c.md): tcgen05.mma M=128 costs 43 + N/2 clk per instruction, one
// tile of d = 64 is only ~500 clk of tensor work, and the hand-shake "MMA done -> epilogue warps wake -> tcgen05.ld ->
// arrive -> MMA warp wakes" takes about as long, so two accumulator buffers cannot keep the tensor pipe busy.  The
// query tile is therefore sized so that THREE (or four) accumulator buffers fit the 512 TMEM columns; epilogue warps
// release a buffer as soon as its accumulators are in registers, then evaluate the bound and append.
constexpr float CFL_TF32_PRODUCT_U = 1.1f / 1024.0f;
constexpr int LB_NEPI = 16;                          // epilogue warps (4 per TMEM lane quarter)
constexpr int LB_THREADS = (LB_NEPI + 2) * 32;
constexpr int LB_NSTAGE = 6;                         // ring stages of up to 4 K-steps (16 KB) each
constexpr uint32_t LB_BLK = 2u * 128u * 16u;         // one K-step of the fp16 catalog plane: [chunk][128 rows][16 B]
constexpr uint32_t LB_STAGE = 4u * LB_BLK;
constexpr int LB_MAXBUF = 4;
// CFL_SCORE_DBG_MODE experiments (tools/passc_probe.py) exist only in builds with CFL_NVCC_EXTRA=-DCFL_LB_EXPERIMENTS: a
// load of the mode word plus a branch per check sits on the critical path of every step otherwise.
#ifdef CFL_LB_EXPERIMENTS
#define LB_DBG(A, bits) (((A).dbg_mode & (bits)) != 0)
#else
#define LB_DBG(A, bits) false
#endif
#ifdef CFL_LB_TRACE
// timing trace of CTA (0,0) (tools/lb_trace.py; builds with CFL_NVCC_EXTRA=-DCFL_LB_TRACE only): per tile
// [0] MMA warp starts the tile, [2] tile issued, [3] epilogue warp 0 before the tfull wait, [4] after it,
// [5] accumulators in registers, [6] bound evaluated / appends done
__device__ unsigned long long g_lb_trace[8 * 4096];
#define LB_TRACE(slot, tile) do { if (blockIdx.x == 0 && blockIdx.y == 0 && (tile) < 4096) g_lb_trace[(tile) * 8 + (slot)] = clock64(); } while (0)
#else
#define LB_TRACE(slot, tile) do { } while (0)
#endif
// A sub-tile holds 4 query groups of GQ queries: epilogue warp `sub` of every TMEM lane quarter owns group `sub`, i.e.
// K*GQ <= 48 accumulator columns per (row, step) in registers.  K*4*GQ = 192 TMEM columns per buffer where K divides 48.
__host__ __device__ constexpr int lb_gq(int K) {
  return K == 1 ? 48 : K == 2 ? 24 : K == 3 ? 16 : K == 4 ? 12 : K == 5 ? 8 : K == 6 ? 8 : K == 7 ? 4 : 6;
}

// Tiling of the pass.  A sub-tile = 4 groups of lb_gq(K) queries = one accumulator buffer of K*qt TMEM columns.  A CTA
// keeps `sub` query images resident and multiplies every catalog tile it streams with all of them, so the catalog
// plane is fetched from L2 once per qt*sub queries: with one image per CTA the pass is bound by the L2 -> SM traffic
// of the re-read plane (measured ~20 B/clk/SM with every SM streaming), not by the tensor pipe.  parts = catalog
// ranges so that parts * nqt ~ the SM count.  Cost model (clk per CTA): tiles * max(sub * tensor, L2) from the
// measured laws tensor = nkm * (43 + N/2), L2 = tile bytes / 20.
LbPlan make_lb_plan(int64_t Q, int K, int d, int64_t tiles) {
  const int qt = 4 * lb_gq(K);
  const int nc = K * qt;
  const int nkm = (d + 15) / 16;
  const int nbuf = 512 / nc > LB_MAXBUF ? LB_MAXBUF : 512 / nc;
  int sms = sm_count(); if (sms <= 0) sms = 148;
  const double tile_clk = nkm * (43.0 + nc / 2.0);              // tensor work per (catalog tile, sub-tile)
  const double l2_clk = nkm * 4096.0 / 20.0;
  LbPlan best{qt, 1, (int)((Q + qt - 1) / qt), 1, nbuf};
  double best_cost = 1e30;
  int sub_lo = 1, sub_hi = 4;
  {                                                            // experiments: force the number of query images per CTA
    const char* e = getenv("CFL_EXPERIMENTS");
    if (e && atoi(e) != 0 && (e = getenv("CFL_LB_SUB")) && atoi(e) >= 1 && atoi(e) <= 4) sub_lo = sub_hi = atoi(e);
  }
  for (int sub = sub_lo; sub <= sub_hi; ++sub) {
    const size_t smem = (size_t)sub * nkm * 2 * nc * 16 + (size_t)LB_NSTAGE * LB_STAGE + 8192;
    if (smem > 200 * 1024) break;
    const int64_t nqt = (Q + (int64_t)qt * sub - 1) / ((int64_t)qt * sub);
    int64_t parts = sms / nqt; if (parts < 1) parts = 1; if (parts > tiles) parts = tiles;
    const double per_cta = (double)((tiles + parts - 1) / parts);
    const double rounds = (double)((nqt * parts + sms - 1) / sms);
    const double step = sub * tile_clk > l2_clk ? sub * tile_clk : l2_clk;
    const double cost = per_cta * rounds * step;
    if (cost < best_cost * 0.999) { best_cost = cost; best = LbPlan{qt, sub, (int)nqt, (int)parts, nbuf}; }
    if ((int64_t)qt * sub >= Q) break;
  }
  return best;
}

static size_t lb_qimg_image_bytes(const LbPlan& p, int K, int d) {
  return (size_t)p.nqt * p.sub * p.qt * ((d + 15) / 16) * 2 * K * 16;
}
size_t score_lb_qimg_bytes(const LbPlan& p, int K, int d) {      // images + flag word + lbq[2 per query slot]
  return lb_qimg_image_bytes(p, K, d) + 16 + (size_t)p.nqt * p.sub * p.qt * 2 * sizeof(float);
}
LbQimgView score_lb_qimg_view(void* base, const LbPlan& p, int K, int d) {
  LbQimgView v;
  v.img = (unsigned char*)base;
  v.flag = (int*)(v.img + lb_qimg_image_bytes(p, K, d));
  v.lbq = (float*)((char*)v.flag + 16);
  return v;
}

// fp16 lower-bound image: [qtile][kstep16][chunk][row n][8 halfs] with n = g*(GQ*K) + k*GQ + i for the query
// ql = g*GQ + i of the tile: the K columns of a query GROUP are contiguous in TMEM (one run of tcgen05.ld), and the
// two queries of a pair sit in adjacent columns = adjacent registers = one FP32x2 operand.  Row k = 0 holds 2a,
// rows k >= 1 the basis vectors.  One warp per query slot, fp64 (modified Gram-Schmidt, every vector
// re-orthogonalised: "twice is enough").
__global__ void __launch_bounds__(128)
prep_lb_kernel(const float* __restrict__ Pc, int64_t Q, int K, int d, int qt, int nqt, int dpad,
               unsigned char* __restrict__ img16, int* __restrict__ flag16, float* __restrict__ lbq) {
  __shared__ double su[4][CFL_MAX_K - 1][128];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t slot = (int64_t)blockIdx.x * 4 + w;
  if (slot >= (int64_t)nqt * qt) return;
  const int GQ = lb_gq(K), NC = K * qt, nks16 = (dpad + 15) / 16;
  const int qtile = (int)(slot / qt), ql = (int)(slot % qt);
  const int g = ql / GQ, gi = ql % GQ;
  unsigned char* base = img16 + (size_t)qtile * nks16 * 2 * NC * 16;
  auto store = [&](int k, int j, double x) {
    const int n = g * (GQ * K) + k * GQ + gi;
    *(__half*)(base + ((size_t)((j >> 4) * 2 + ((j >> 3) & 1)) * NC + n) * 16 + (j & 7) * 2) = __float2half_rn((float)x);
  };
  if (slot >= Q) {                                             // padding queries of the last tile: zero rows
    for (int k = 0; k < K; ++k)
      for (int j = lane; j < nks16 * 16; j += 32) store(k, j, 0.0);
    return;
  }
  const float* pq = Pc + slot * (int64_t)K * d;
  double p0[4], a[4];
#pragma unroll
  for (int m = 0; m < 4; ++m) { const int j = lane + 32 * m; p0[m] = (j < d) ? (double)pq[j] : 0.0; a[m] = p0[m]; }
  for (int k = 1; k < K; ++k) {
    double v[4];
    double n0 = 0.0;
#pragma unroll
    for (int m = 0; m < 4; ++m) { const int j = lane + 32 * m; v[m] = (j < d) ? (double)pq[k * d + j] - p0[m] : 0.0; n0 += v[m] * v[m]; }
    n0 = warp_sum(n0);
    double nrm = 0.0;
    for (int pass = 0; pass < 3; ++pass) {                     // pass 2 re-orthogonalises the NORMALISED vector
      for (int i = 1; i < k; ++i) {
        double c = 0.0;
#pragma unroll
        for (int m = 0; m < 4; ++m) c += v[m] * su[w][i - 1][lane + 32 * m];
        c = warp_sum(c);
#pragma unroll
        for (int m = 0; m < 4; ++m) v[m] -= c * su[w][i - 1][lane + 32 * m];
      }
      if (pass >= 1) {
        nrm = 0.0;
#pragma unroll
        for (int m = 0; m < 4; ++m) nrm += v[m] * v[m];
        nrm = warp_sum(nrm);
        const double inv = (nrm > 1e-280) ? rsqrt(nrm) : 0.0;  // p_k - p_0 exactly inside the previous span: no new direction
#pragma unroll
        for (int m = 0; m < 4; ++m) v[m] *= inv;
      }
    }
#pragma unroll
    for (int m = 0; m < 4; ++m) su[w][k - 1][lane + 32 * m] = v[m];
    __syncwarp();
    (void)n0;
  }
  for (int pass = 0; pass < 2; ++pass)
    for (int i = 1; i < K; ++i) {
      double c = 0.0;
#pragma unroll
      for (int m = 0; m < 4; ++m) c += a[m] * su[w][i - 1][lane + 32 * m];
      c = warp_sum(c);
#pragma unroll
      for (int m = 0; m < 4; ++m) a[m] -= c * su[w][i - 1][lane + 32 * m];
    }
  double a2 = 0.0, vmax = 0.0;
#pragma unroll
  for (int m = 0; m < 4; ++m) { a2 += a[m] * a[m]; vmax = fmax(vmax, fabs(2.0 * a[m])); }
  a2 = warp_sum(a2);
  for (int m = 0; m < 4; ++m) {
    const int j = lane + 32 * m;
    if (j >= nks16 * 16) continue;
    store(0, j, j < d ? 2.0 * a[m] : 0.0);
    for (int k = 1; k < K; ++k) store(k, j, j < d ? su[w][k - 1][j] : 0.0);
  }
  if (!(vmax < 60000.0)) atomicOr(flag16, 1);                  // also catches NaN / inf
  if (lane == 0) {
    lbq[2 * slot] = __double2float_rd(a2);
    lbq[2 * slot + 1] = __double2float_ru(sqrt(a2));
  }
}

int score_lb_prep_queries(const ScoreArgs& a, cudaStream_t st) {
  unsigned char* img16 = (unsigned char*)const_cast<void*>(a.qimg16);
  int* flag16 = const_cast<int*>(a.qflag16);
  CFL_CUDA(cudaMemsetAsync(flag16, 0, 16, st));
  const int64_t slots = (int64_t)a.lb.nqt * a.lb.sub * a.lb.qt;   // one image per sub-tile of qt queries
  prep_lb_kernel<<<(unsigned)((slots + 3) / 4), 128, 0, st>>>(a.Pc, a.Q, a.K, a.d, a.lb.qt, a.lb.nqt * a.lb.sub, a.plan.dpad,
                                                             img16, flag16, const_cast<float*>(a.lbq));
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

// NCOLS consecutive TMEM columns of this warp's 32 lanes -> registers, as a run of x16 / x8 / x4 loads
template <int NCOLS, int OFF = 0>
__device__ __forceinline__ void tmem_ld_cols(uint32_t taddr, float (&v)[NCOLS]) {
  if constexpr (NCOLS - OFF >= 16) {
    tmem_ld16(taddr + OFF, *reinterpret_cast<float(*)[16]>(&v[OFF]));
    tmem_ld_cols<NCOLS, OFF + 16>(taddr, v);
  } else if constexpr (NCOLS - OFF >= 8) {
    tmem_ld8(taddr + OFF, *reinterpret_cast<float(*)[8]>(&v[OFF]));
    tmem_ld_cols<NCOLS, OFF + 8>(taddr, v);
  } else if constexpr (NCOLS - OFF >= 4) {
    tmem_ld4(taddr + OFF, *reinterpret_cast<float(*)[4]>(&v[OFF]));
    tmem_ld_cols<NCOLS, OFF + 4>(taddr, v);
  }
}

constexpr int LB_WQ = 64;                            // entries of a warp's survivor queue (16 B each)
struct LbLayout {
  uint32_t b_img, a_ring, ncq, cnt, red, wq, bars, tmem_slot, total;
};
__host__ __device__ inline LbLayout lb_layout(int K, int qt, int sub, int nkm) {
  LbLayout L;
  uint32_t off = 0;
  L.b_img = off;   off += (uint32_t)sub * (uint32_t)nkm * 2u * (uint32_t)(K * qt) * 16u;  off = (off + 1023u) & ~1023u;
  L.a_ring = off;  off += LB_NSTAGE * LB_STAGE;
  L.ncq = off;     off += (uint32_t)(qt * sub) * 4u;                      off = (off + 15u) & ~15u;
  L.cnt = off;     off += (uint32_t)(qt * sub) * 4u;                      off = (off + 15u) & ~15u;
  L.red = off;     off += 32u * 4u;
  L.wq = off;      off += (uint32_t)LB_NEPI * LB_WQ * 16u;
  L.bars = off;    off += (2u * LB_NSTAGE + 2u * LB_MAXBUF + 1u) * 8u;
  L.tmem_slot = off; off += 16u;
  L.total = off;
  return L;
}

// Appends the entries of a warp's survivor queue to the per-(part, query) key buffers (warp-uniform call): lane e takes
// entry e, one shared-memory atomic + one 8-byte store per surviving (row, query).
__device__ __forceinline__ void lb_flush_queue(const uint4* wq, int fill, int lane, int QT, int g0, int nq, int* cnt,
                                               tkey_t* kbase, tkey_t* spill, int* spill_cnt, int64_t q0) {
  __syncwarp();
  for (int e = lane; e < fill; e += 32) {
    const uint4 en = wq[e];
    unsigned long long nb = ((unsigned long long)en.w << 32) | en.z;
    const tkey_t key = pack_key(0.0f, en.x);
    while (nb) {
      const int ql = (int)en.y * QT + g0 + __ffsll((long long)nb) - 1;
      nb &= nb - 1;
      if (ql >= nq) continue;                                  // padding queries never pass (ncq = -inf); belt and braces
      const int slot = atomicAdd(&cnt[ql], 1);
      if (slot < TOPK_STRIDE) {
        kbase[(int64_t)ql * TOPK_STRIDE + slot] = key;
      } else {                                                 // this part's buffer is full: spill list of the query
        const int sp = atomicAdd(&spill_cnt[q0 + ql], 1);
        if (sp < LB_SPILL) spill[(q0 + ql) * (int64_t)LB_SPILL + sp] = key;
      }
    }
  }
  __syncwarp();
}

// Sequence of "steps" u = (catalog tile t, sub-tile s): accumulator buffer u mod NBUF, A = the tile's ring stage(s),
// B = query image s.  A ring stage is handed back to the TMA producer after its LAST sub-tile.
template <int KSS>
__device__ __forceinline__ void lb_mma_loop(const ScoreArgs& A, uint32_t a_base, uint32_t b_base, uint32_t tmem_base, int NC,
                                            int NBUF, int SUB, int nkm, int ntiles, uint64_t* full, uint64_t* empty,
                                            uint64_t* tfull, uint64_t* tempty) {
  const uint32_t idesc = make_idesc_f16(128, (uint32_t)NC);
  const uint32_t b_step = 2u * (uint32_t)NC * 16u;            // bytes per K-step of a query image
  const uint32_t b_img = (uint32_t)nkm * b_step;               // bytes per query image
  const int nsteps = nkm / KSS;                                // ring stages per catalog tile
  const uint32_t full0 = smem_u32(full), empty0 = smem_u32(empty), tfull0 = smem_u32(tfull), tempty0 = smem_u32(tempty);
  int stage0 = 0; uint32_t phase0 = 0;                         // first ring stage of tile t
  int buf = 0; uint32_t bphase = 0;                            // accumulator buffer of the step and the parity of its use count
  if (ntiles > 0) {
    mbar_wait_addr(tempty0, 1u);
    if (!LB_DBG(A, 2)) mbar_wait_addr(full0, 0u);
    tc_fence_after();
  }
  for (int t = 0; t < ntiles; ++t) {
    LB_TRACE(0, t);
    for (int sq = 0; sq < SUB; ++sq) {
      const uint32_t d_tmem = tmem_base + (uint32_t)(buf * NC);
      int nbuf_i = buf + 1; uint32_t nbphase = bphase;
      if (nbuf_i == NBUF) { nbuf_i = 0; nbphase ^= 1u; }
      const bool last_sub = sq == SUB - 1;
      int stage = stage0; uint32_t phase = phase0;
      for (int sidx = 0; sidx < nsteps; ++sidx) {
        const uint32_t a_st = a_base + (uint32_t)stage * LB_STAGE;
        const uint32_t b_st = b_base + (uint32_t)sq * b_img + (uint32_t)(sidx * KSS) * b_step;
        int nstage = stage + 1; uint32_t nphase = phase;
        if (nstage == LB_NSTAGE) { nstage = 0; nphase ^= 1u; }
        const bool last = sidx == nsteps - 1;
#pragma unroll
        for (int j = 0; j < KSS; ++j) {
          if (j == KSS - 1) {                                  // look ahead: barriers of the next stage / step
            bool fence = false;
            if (last && (!last_sub || t + 1 < ntiles) && !LB_DBG(A, 16)) { mbar_wait_addr(tempty0 + (uint32_t)nbuf_i * 8u, nbphase ^ 1u); fence = true; }
            // the next stage holds catalog data not yet waited for: the tile's further stages during its first
            // sub-tile, the next tile's first stage after the last sub-tile
            const bool need_full = last ? (last_sub && t + 1 < ntiles) : (sq == 0);
            if (need_full && !LB_DBG(A, 2)) { mbar_wait_addr(full0 + (uint32_t)nstage * 8u, nphase); fence = true; }
            if (fence) tc_fence_after();
          }
          if (!LB_DBG(A, 64))                              // 64: no MMAs at all, only the barrier traffic (timing only)
          mma_f16(d_tmem, make_smem_desc(a_st + (uint32_t)j * LB_BLK, 128u * 16u, 128u),
                  make_smem_desc(b_st + (uint32_t)j * b_step, (uint32_t)NC * 16u, 128u), idesc, (sidx | j) ? 1u : 0u);
        }
        if (last_sub) mma_commit_addr(empty0 + (uint32_t)stage * 8u);
        stage = nstage; phase = nphase;
      }
      mma_commit_addr(tfull0 + (uint32_t)buf * 8u);
      buf = nbuf_i; bphase = nbphase;
      if (last_sub) { stage0 = stage; phase0 = phase; }
    }
    LB_TRACE(2, t);
  }
}

template <int K>
__global__ void __launch_bounds__(LB_THREADS, 1)
score_lb_kernel(ScoreArgs A) {
  extern __shared__ __align__(1024) unsigned char smem[];
  constexpr int GQ = lb_gq(K);
  constexpr int GC = GQ * K;                                   // TMEM columns of one query group
  const int QT = A.lb.qt;                                      // queries per sub-tile (one accumulator buffer)
  const int SUB = A.lb.sub;                                    // sub-tiles (query images) of this CTA
  const int QC = QT * SUB;                                     // queries per CTA
  const int NC = K * QT;
  const int NBUF = A.lb.nbuf;
  const int nkm = (A.plan.dpad + 15) / 16;                     // MMA K-steps (16 halfs) per tile
  const int kss = (nkm % 4 == 0) ? 4 : ((nkm % 2 == 0) ? 2 : 1);   // K-steps (4 KB blocks) per ring stage
  const LbLayout L = lb_layout(K, QT, SUB, nkm);
  unsigned char* b_img = smem + L.b_img;
  unsigned char* a_ring = smem + L.a_ring;
  float* ncq = (float*)(smem + L.ncq);                         // -cq per query of the tile
  int* cnt = (int*)(smem + L.cnt);
  float* red = (float*)(smem + L.red);
  uint64_t* full = (uint64_t*)(smem + L.bars);
  uint64_t* empty = full + LB_NSTAGE;
  uint64_t* tfull = empty + LB_NSTAGE;
  uint64_t* tempty = tfull + LB_MAXBUF;
  uint64_t* bfull = tempty + LB_MAXBUF;
  uint32_t* tmem_slot = (uint32_t*)(smem + L.tmem_slot);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int part = blockIdx.x, qtile = blockIdx.y;
  const int64_t q0 = (int64_t)qtile * QC;
  const int nq = (int)((A.Q - q0 < QC) ? (A.Q - q0) : QC);
  const int64_t t0 = A.plan.tiles * part / A.lb.parts;
  const int64_t t1 = A.plan.tiles * (part + 1) / A.lb.parts;
  const int ts = A.tile_stride;
  const int ntiles = (int)((t1 - t0 + ts - 1) / ts);
  if (*A.cflag16 != 0 || *A.qflag16 != 0) {                    // a value outside the fp16 range: exact redo pass
    for (int ql = tid; ql < nq; ql += LB_THREADS) A.counts[(int64_t)part * A.Q + q0 + ql] = -1;
    return;
  }
  if (A.thr_init != nullptr) {                                 // no live query in this tile: nothing to do
    bool live = false;
    for (int i = tid; i < nq; i += LB_THREADS) live |= A.thr_init[q0 + i] > __int_as_float(0xff800000);
    if (!__syncthreads_or(live)) {
      for (int ql = tid; ql < nq; ql += LB_THREADS) A.counts[(int64_t)part * A.Q + q0 + ql] = 0;
      return;
    }
  }
  if (warp == LB_NEPI) {
    if (lane == 0) {
      for (int s = 0; s < LB_NSTAGE; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
      for (int b = 0; b < LB_MAXBUF; ++b) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], LB_NEPI); }   // one arrival per epilogue WARP
      mbar_init(bfull, 1);
      fence_barrier_init();
    }
    __syncwarp();
    tmem_alloc(tmem_slot, 512);
  }
  // largest |a| of the tile: one margin factor for the whole CTA
  float am = 0.0f;
  for (int i = tid; i < nq; i += LB_THREADS) am = fmaxf(am, A.lbq[2 * (q0 + i) + 1]);
  am = warp_max(am);
  if (lane == 0) red[warp] = am;
  // cq = |a|^2 - threshold, rounded down (stored negated); padding / dead queries get +inf (never pass), no threshold
  // -inf (always pass)
  for (int i = tid; i < QC; i += LB_THREADS) {
    float c = __int_as_float(0x7f800000);
    if (i < nq) {
      const float tau = A.thr_init ? A.thr_init[q0 + i] : __int_as_float(0x7f800000);
      const float a2 = A.lbq[2 * (q0 + i)];
      if (tau > 3.0e38f) c = __int_as_float(0xff800000);
      else if (tau > -3.0e38f) c = __fsub_rd(a2, nextafterf(tau, 3.4e38f)) - 5.0e-7f * (a2 + fabsf(tau));
    }
    ncq[i] = -c;
    cnt[i] = 0;
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == LB_NEPI) {
    // ================================ MMA issuer (one elected lane) =================================
    // One thread issues; what limits it is the latency of its OWN instruction stream (a dependent SASS instruction
    // costs ~5 clk when a single thread runs): ~25 instructions of address arithmetic and R2UR moves per MMA make the
    // issue slower than the tensor pipe (tools/umma_rate.cu).  The loop is therefore written so that ptxas keeps every
    // operand in uniform registers: all values derive from kernel parameters and shared-memory addresses, the K-steps
    // of a ring stage are unrolled at compile time, and the barrier waits for the NEXT stage / accumulator buffer are
    // issued before the stage's last MMA, while the queued MMAs still execute.
    if (elect_one()) {
      mbar_wait(bfull, 0);
      switch (kss) {
        case 4: lb_mma_loop<4>(A, smem_u32(a_ring), smem_u32(b_img), tmem_base, NC, NBUF, SUB, nkm, ntiles, full, empty, tfull, tempty); break;
        case 2: lb_mma_loop<2>(A, smem_u32(a_ring), smem_u32(b_img), tmem_base, NC, NBUF, SUB, nkm, ntiles, full, empty, tfull, tempty); break;
        default: lb_mma_loop<1>(A, smem_u32(a_ring), smem_u32(b_img), tmem_base, NC, NBUF, SUB, nkm, ntiles, full, empty, tfull, tempty); break;
      }
    }
  } else if (warp == LB_NEPI + 1) {
    // ================================ TMA producer (one lane) ===============================
    if (elect_one()) {
      const uint32_t bbytes = (uint32_t)SUB * (uint32_t)nkm * 2u * (uint32_t)NC * 16u;   // SUB consecutive query images
      const unsigned char* qsrc = (const unsigned char*)A.qimg16 + (size_t)qtile * bbytes;
      mbar_arrive_expect_tx(bfull, bbytes);
      for (uint32_t o = 0; o < bbytes; o += 32768u) {
        const uint32_t n = bbytes - o < 32768u ? bbytes - o : 32768u;
        bulk_g2s(b_img + o, qsrc + o, n, bfull);
      }
      int stage = 0; uint32_t phase = 0;
      for (int t = 0; t < (LB_DBG(A, 2) ? 0 : ntiles); ++t) {
        const unsigned char* src = (const unsigned char*)A.cimg16 + (size_t)(t0 + (int64_t)t * ts) * nkm * LB_BLK;
        for (int ks = 0; ks < nkm; ks += kss) {
          mbar_wait(&empty[stage], phase ^ 1u);
          mbar_arrive_expect_tx(&full[stage], (uint32_t)kss * LB_BLK);
          bulk_g2s(a_ring + stage * LB_STAGE, src + (size_t)ks * LB_BLK, (uint32_t)kss * LB_BLK, &full[stage]);
          if (++stage == LB_NSTAGE) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else {
    // ======================================= epilogue ========================================
    // Warp (lane quarter lq, sub) owns query group `sub` of every sub-tile: per step it waits for the accumulators,
    // moves its K*GQ columns to registers (tcgen05.ld), releases the buffer at once (the MMA of step u + NBUF never
    // waits for CUDA-core work), then evaluates the bound: K-1 packed FMAs + one packed add per query pair, a 3-input
    // max tree, ONE compare; the rare survivors are appended by their own lane.
    const int lq = warp & 3, sub = warp >> 2;
    const int lrow = lq * 32 + lane;
    tkey_t* kbase = A.keys + ((int64_t)part * A.Q + q0) * TOPK_STRIDE;
    float amax = 0.0f;
    for (int i = 0; i < LB_THREADS / 32; ++i) amax = fmaxf(amax, red[i]);
    const float s16 = 5.97e-8f * sqrtf((float)(nkm * 16));    // 2^-24 sqrt(d): twice the subnormal term
    const float rk = sqrtf((float)(K - 1));
    const float ulp = (float)(4 * K) * 5.97e-8f;
    const float c_e2 = 1.0f - CFL_PLANE_REL - (2.0f * rk * (CFL_TF32_PRODUCT_U + s16) + ulp) * 1.0001f;
    const float c_sq = ((2.0f * CFL_TF32_PRODUCT_U + 2.0f * ulp) * amax + 2.0f * s16 * (1.0f + rk)) * 1.0001f;
    const float c_abs = 2.0f * s16 * amax * 1.0001f;
    float2 er_next = (ntiles > 0) ? __ldg(A.lbrow + t0 * 128 + lrow) : make_float2(0.f, 0.f);   // one tile ahead
    const uint32_t taddr0 = tmem_base + ((uint32_t)(lq * 32) << 16) + (uint32_t)(sub * GC);
    const float* ncq_w = ncq + sub * GQ;
    uint4* wq = (uint4*)(smem + L.wq) + warp * LB_WQ;
    int wq_fill = 0;
    int buf = 0; uint32_t bphase = 0;
    for (int t = 0; t < ntiles; ++t) {
      const uint32_t row = (uint32_t)((t0 + (int64_t)t * ts) * 128 + lrow);
      const float2 er = er_next;
      if (t + 1 < ntiles) er_next = __ldg(A.lbrow + (t0 + (int64_t)(t + 1) * ts) * 128 + lrow);
      // |e|^2 lowered by the error bound of the single-product evaluation; +inf for the padding rows
      const float e2s = fmaf(er.x, c_e2, fmaf(-c_sq, er.y, -c_abs));
      for (int sq = 0; sq < SUB; ++sq) {
        if (tid == 0) LB_TRACE(3, t * SUB + sq);
        mbar_wait(&tfull[buf], bphase);
        tc_fence_after();
        if (tid == 0) LB_TRACE(4, t * SUB + sq);
        float v[GC];
        if (!LB_DBG(A, 1)) {
          tmem_ld_cols<GC>(taddr0 + (uint32_t)(buf * NC), v);
          tmem_ld_wait();
        }
        if (tid == 0) LB_TRACE(5, t * SUB + sq);
        tc_fence_before();                                     // the accumulators are in registers: release the buffer
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty[buf]);
        if (++buf == NBUF) { buf = 0; bphase ^= 1u; }
        if (LB_DBG(A, 5)) continue;                          // experiments: no epilogue work / TMEM reads only
        // t_i = e.(2a) - cq_i + sum_j (e.u_j)^2 ; the (row, query) survives iff t_i > e2s(row)
        // (evaluated in place: v[i], i < GQ, becomes t_i)
        const float2* ncq2 = (const float2*)(ncq_w + sq * QT);
#pragma unroll
        for (int pi = 0; pi < GQ / 2; ++pi) {
          const float2 c2 = LB_DBG(A, 32) ? make_float2(e2s, e2s) : ncq2[pi];   // 32: no shared-memory reads (timing only)
          f2_t acc = add2(pk2(v[2 * pi], v[2 * pi + 1]), pk2(c2.x, c2.y));
#pragma unroll
          for (int k = 1; k < K; ++k) {
            const f2_t c = pk2(v[k * GQ + 2 * pi], v[k * GQ + 2 * pi + 1]);
            acc = fma2(c, c, acc);
          }
          upk2(acc, v[2 * pi], v[2 * pi + 1]);
        }
        // max over the group as a two-level tree of 3-input maxima: the triples' maxima locate the survivors cheaply
        constexpr int NT3 = (GQ + 2) / 3;
        float m3[NT3];
#pragma unroll
        for (int j = 0; j < NT3; ++j) {
          const int i0 = 3 * j, i1 = 3 * j + 1 < GQ ? 3 * j + 1 : i0, i2 = 3 * j + 2 < GQ ? 3 * j + 2 : i0;
          m3[j] = max3(v[i0], v[i1], v[i2]);
        }
        float m = m3[0];
#pragma unroll
        for (int j = 1; j < NT3; j += 2) m = (j + 1 < NT3) ? max3(m, m3[j], m3[j + 1]) : fmaxf(m, m3[j]);
        if (tid == 0) LB_TRACE(6, t * SUB + sq);
        const bool hit = m > e2s && !LB_DBG(A, 8);
        const uint32_t hb = __ballot_sync(0xffffffffu, hit);
        if (hb != 0) {
          // Rare per lane (a fraction of a percent), but about every second warp-step has one: the survivors go to
          // the warp's queue in shared memory -- (row, sub-tile, mask of the group's surviving queries), position by
          // ballot, no atomics -- and are appended to the per-query key buffers in batches of >= 32 entries, so the
          // latency of the shared-memory atomics and the dependent global stores is paid once per batch.
          const int nh = __popc(hb);
          if (wq_fill + nh > LB_WQ) { lb_flush_queue(wq, wq_fill, lane, QT, sub * GQ, nq, cnt, kbase, A.spill, A.spill_cnt, q0); wq_fill = 0; }
          if (hit) {
            unsigned long long nb = 0;
#pragma unroll
            for (int j = 0; j < NT3; ++j)
              if (m3[j] > e2s) {
#pragma unroll
                for (int i = 3 * j; i < 3 * j + 3 && i < GQ; ++i) nb |= (v[i] > e2s) ? (1ull << i) : 0ull;
              }
            wq[wq_fill + __popc(hb & ((1u << lane) - 1u))] = make_uint4(row, (uint32_t)sq, (uint32_t)nb, (uint32_t)(nb >> 32));
          }
          wq_fill += nh;
          __syncwarp();
        }
        if (tid == 0) LB_TRACE(7, t * SUB + sq);
      }
    }
    lb_flush_queue(wq, wq_fill, lane, QT, sub * GQ, nq, cnt, kbase, A.spill, A.spill_cnt, q0);
    asm volatile("bar.sync 1, %0;" ::"n"(LB_NEPI * 32) : "memory");
    // counts may exceed TOPK_STRIDE: the excess went to the query's spill list
    for (int ql = tid; ql < nq; ql += LB_NEPI * 32) A.counts[(int64_t)part * A.Q + q0 + ql] = cnt[ql];
  }
  tc_fence_before();
  __syncthreads();
  if (warp == LB_NEPI) tmem_dealloc(tmem_base, 512);
}

template <int K>
static int launch_lb(const ScoreArgs& a, cudaStream_t st) {
  const LbLayout L = lb_layout(K, a.lb.qt, a.lb.sub, (a.plan.dpad + 15) / 16);
  const size_t smem = L.total + 1024;                          // slack for the alignment of the dynamic segment
  CFL_SMEM_LIMIT(score_lb_kernel<K>, smem);
  dim3 grid(a.lb.parts, a.lb.nqt);
  score_lb_kernel<K><<<grid, LB_THREADS, smem, st>>>(a);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

#ifdef CFL_LB_TRACE
extern "C" int cfl_lb_trace_read(unsigned long long* host, int n) {
  return (int)cudaMemcpyFromSymbol(host, g_lb_trace, (size_t)n * sizeof(unsigned long long));
}
#endif

// ---- self-test of the pass's MMA: D[128, N] = A[128, Kd] B[N, Kd]^T, operands rounded to fp16 (RN), ONE kind::f16 MMA
// per 16 dimensions, fp32 accumulators: what the error margin of the lower bound (CFL_TF32_PRODUCT_U) is about.
__global__ void __launch_bounds__(160)
lb_selftest_kernel(const float* __restrict__ Af, const float* __restrict__ Bf, float* __restrict__ D, int N, int Kd) {
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ uint64_t bar;
  __shared__ uint32_t slot;
  const int tid = threadIdx.x, warp = tid >> 5;
  const int nks = (Kd + 15) / 16;
  const uint32_t a_step = 2u * 128u * 16u, b_step = 2u * (uint32_t)N * 16u;
  unsigned char* a_img = smem;
  unsigned char* b_img = smem + (size_t)nks * a_step;
  if (tid == 0) { mbar_init(&bar, 1); fence_barrier_init(); }
  if (tid < 128) {
    for (int ks = 0; ks < nks; ++ks)
      for (int c = 0; c < 2; ++c) {
        __align__(16) __half h[8];
        for (int i = 0; i < 8; ++i) { const int j = ks * 16 + c * 8 + i; h[i] = __float2half_rn(j < Kd ? Af[(size_t)tid * Kd + j] : 0.0f); }
        *(uint4*)(a_img + (size_t)ks * a_step + (c * 128 + tid) * 16) = *(const uint4*)h;
        for (int n = tid; n < N; n += 128) {
          for (int i = 0; i < 8; ++i) { const int j = ks * 16 + c * 8 + i; h[i] = __float2half_rn(j < Kd ? Bf[(size_t)n * Kd + j] : 0.0f); }
          *(uint4*)(b_img + (size_t)ks * b_step + ((size_t)c * N + n) * 16) = *(const uint4*)h;
        }
      }
    fence_proxy_async();
  }
  uint32_t ncols = 32;
  while ((int)ncols < N) ncols <<= 1;
  if (warp == 4) tmem_alloc(&slot, ncols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tb = slot;
  if (warp == 4) {
    if (elect_one()) {
      const uint32_t idesc = make_idesc_f16(128, (uint32_t)N);
      for (int ks = 0; ks < nks; ++ks)
        mma_f16(tb, make_smem_desc(smem_u32(a_img) + ks * a_step, 128u * 16u, 128u),
                make_smem_desc(smem_u32(b_img) + ks * b_step, (uint32_t)N * 16u, 128u), idesc, ks ? 1u : 0u);
      mma_commit(&bar);
    }
  } else {
    mbar_wait(&bar, 0);
    tc_fence_after();
    for (int c0 = 0; c0 < N; c0 += 8) {
      float v[8];
      tmem_ld8(tb + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, v);
      tmem_ld_wait();
      for (int j = 0; j < 8; ++j) D[(size_t)tid * N + c0 + j] = v[j];
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tb, ncols);
}

int score_lb_launch(const ScoreArgs& a, cudaStream_t st) {
  return with_k(a.K, [&](auto K) { return launch_lb<K>(a, st); });
}

}  // namespace cfl

extern "C" int cfl_selftest_umma_f16(const float* A, const float* Bm, float* D, int N, int Kd, void* stream) {
  using namespace cfl;
  int st = device_check();
  if (st != CFL_OK) return st;
  CFL_REQUIRE(A && Bm && D, CFL_ERR_INVALID, "selftest_umma_f16: NULL argument");
  CFL_REQUIRE(N >= 16 && N <= 256 && N % 16 == 0, CFL_ERR_INVALID, "selftest_umma_f16: N must be a multiple of 16 in [16,256]");
  CFL_REQUIRE(Kd >= 1 && Kd <= 128, CFL_ERR_INVALID, "selftest_umma_f16: Kd must be in [1,128]");
  const int nks = (Kd + 15) / 16;
  const size_t smem = (size_t)nks * (2 * 128 * 16 + 2 * (size_t)N * 16) + 1024;
  CFL_SMEM_LIMIT(lb_selftest_kernel, smem);
  lb_selftest_kernel<<<1, 160, smem, (cudaStream_t)stream>>>(A, Bm, D, N, Kd);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}
