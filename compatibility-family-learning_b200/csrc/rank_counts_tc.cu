// Per-query all-candidate AUC on the tensor cores (SURVEY 8d C3, 8e): the rank counts of cfl_rank_counts
//   counts[q,j] = ( #{c : dist(q,c) < t[q,j]},  #{c : dist(q,c) == t[q,j]} )
// taken INSIDE the epilogue of the fused scoring kernel -- the Q x N distances never reach HBM (the earlier
// tensor-core route wrote and re-read a dense 4 GB matrix).  roc_auc_score of cfl/utils.py:267-268 over every
// catalog row follows from these integers (cfl.ranking.auc_from_rank_counts).
//
// The kernel runs the Gram pipeline of gram_pipe.cuh (packed catalog image through a TMA ring, 3xTF32 tcgen05.mma into
// double-buffered TMEM accumulators, the same as score_umma_kernel) with the soft-min of score.cuh and a counting epilogue:
//   * every (row, query) distance D~ (Gram form, 3xTF32) gets a rounding band
//       m = S * (REL1 + REL2 * sqrt(D~ * V)),   S = |e|^2 + max_k |p_k|^2,   V = spread of the prototypes under the
//     soft-min weights (softmin_pair_var: the sensitivity of the distance to an error of the soft-min exponents, which
//     carry an absolute error proportional to S -- zero when the soft-min is saturated or K = 1);
//   * every pair is counted at once against each of the query's J thresholds by the sign of t - D~ (per-thread packed
//     4-bit counters, one predicated add per (row, query, threshold); a thread keeps its TMEM lane = catalog row
//     position for the whole pass; flushed through a warp reduction every 15 tiles);
//   * a pair with SOME threshold inside its band (min_j |t_j - D~| <= m, two thresholds per packed add + 3-input min;
//     exact ties included) -- a few 1e-4 of all pairs -- also goes to a record list: rank_fix_kernel evaluates it in
//     fp32 direct-difference form with the SAME device function as cfl_pair_dist_rows / cfl_rank_counts (direct.cuh)
//     and, for every threshold inside the band, replaces the fast verdict by the exact < / == verdicts.
// The counts therefore equal cfl_rank_counts' whenever |D~ - direct| <= m for every pair.  REL1 / REL2 are set to >= 4x
// the largest deviation measured over the bench and test shapes (tools/rank_counts_perf.py prints the observed
// maximum of |D~ - direct| / m over all ambiguous records; rank_fix_kernel reports it in the call's statistics and
// tests/test_rank_counts.py asserts the headroom).  A query whose records do not fit the list is recounted from
// scratch by the CUDA-core kernel (rank_count_kernel, restricted by `only`).
//
// SRC (pcd_source: rank_count_src_umma_kernel / within_emit_src_umma_kernel, the fix kernels rank_fix_src_kernel /
// within_fix_src_kernel): the pipeline of score_src_umma_kernel -- the catalog rows are SOURCE items with K prototype
// planes (cfl_source_catalog_pack), the queries TARGET embeddings (one vector each, a query image packed with K = 1).
// The row's soft-min block is broadcast to each query pair, |e_q - mu|^2 is per query, and the band takes
// S = |e_q - mu|^2 + max_k |p_ck - mu|^2 (the row's first K block entries).  There is no skip test: the affine hull
// belongs to the row, not to the query.  The records are checked with pcd_direct(e = query row, p = catalog row), the
// values cfl_score_topk_source reports.
#include "gram_pipe.cuh"
#include <stdlib.h>
#include "direct.cuh"

namespace cfl {

using namespace umma;

constexpr int RT_JC = 8;                            // thresholds per launch (J > 8: several launches)
constexpr int RT_QT_MAX = 64;
constexpr float RT_REL1_DEFAULT = 1.0f / 262144.0f;     // 2^-18: Gram-form (3xTF32) + direct-form rounding, relative to S
constexpr float RT_REL2_DEFAULT = 1.0f / 2097152.0f;    // 2^-21: exponent error relative to S (sensitivity term)

// query tile: <= RT_QT_MAX and, with the query groups of gram_gq(K), at most NGW groups per epilogue warp (rank_umma_body);
// the source tile also keeps K*qt <= 256 TMEM columns per accumulator buffer (score_src_qt)
int rank_tc_qt(int K, int d, bool src = false) {
  int qt = src ? score_src_qt(K, d) : score_umma_qt(K, d);
  return qt > RT_QT_MAX ? RT_QT_MAX : qt;
}

struct RtArgs {
  int K, d, J, j0;                // this launch counts thresholds [j0, j0 + min(RT_JC, J - j0))
  int64_t Q, N;
  int qt, nqt, parts, dpad;
  int64_t tiles;
  const float* qpar;              // per query: soft-min block (SRC: |e_q - mu|^2)
  const float* qplane;            // per query: affine-hull bound block (score.cuh); SRC: unused
  const void* qimg;
  const void* cimg;
  const float* e2;                // per row: |e - mu|^2; SRC: the rows' soft-min blocks (source_catalog_view().rowpar)
  const float* thr;               // [Q, J]
  unsigned long long* counts;     // [Q, J, 2]
  uint4* recs;                    // ambiguous (query, row) records
  unsigned int rec_slice;         // records per CTA slice of the list
  unsigned int* rec_n;            // [CTAs] records written per slice
  int* only;                      // [Q]: 1 = records dropped, recount this query from scratch
  float rel1, rel2;
  // emitting pass only
  const int64_t* offsets;         // [Q + 1]: segment of query q = out[offsets[q], offsets[q + 1])
  unsigned int* cursor;           // [Q]: rows appended so far
  int64_t* out;                   // local catalog rows
};

// Shared memory of the counting / emitting kernels: the Gram pipeline's regions and, behind the query blocks, the
// epilogue's thresholds, max_k |p_k|^2, skip-test constants per query, per-threshold counts and records written.
struct RtLayout { GramLayout g; uint32_t thr, qm, skp, cs, rcn; };
template <bool SRC = false>
__host__ __device__ inline RtLayout rt_layout(int K, int qt, int dpad) {
  RtLayout L;
  L.g = gram_layout<SRC>(K, qt, dpad, 0u);
  uint32_t off = L.g.back;
  L.thr = off;     off += (uint32_t)qt * RT_JC * 4u;
  L.qm = off;      off += (uint32_t)qt * 4u;                           off = (off + 15u) & ~15u;
  L.skp = off;     off += (uint32_t)qt * 16u;                          // per query: (tmax, kappa0, kappa1, -)
  L.cs = off;      off += (uint32_t)qt * RT_JC * 4u;
  L.rcn = off;     off += 16u;
  gram_layout_end(L.g, off);
  return L;
}

// cnt += inc when x > 0 (x = t - D~: the pair is closer than the threshold), without a branch.
__device__ __forceinline__ void count_pos(uint32_t& cnt, float x, uint32_t inc) {
  asm("{\n\t.reg .pred p;\n\t"
      "setp.gt.f32 p, %1, 0f00000000;\n\t"
      "@p add.u32 %0, %0, %2;\n\t}"
      : "+r"(cnt)
      : "f"(x), "r"(inc));
}
__device__ __forceinline__ float sqrt_approx(float x) {
  float y;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// The Gram pipeline and the classifying epilogue, shared by the counting kernel (EMIT = false: packed counters, J
// thresholds) and the emitting kernel of cfl_score_within (EMIT = true, J = 1: a pair with D~ < t - m is appended to its
// query's result segment at once, a pair inside the band goes to the record list exactly as for the counts).  Both
// instantiations classify with the same arithmetic, so the emitted set and the count of the same radius agree pair for pair.
template <int K, bool SRC, bool EMIT>
__device__ __forceinline__ void rank_umma_body(const RtArgs& A) {
  extern __shared__ __align__(1024) unsigned char smem[];
  // SRC at K <= 2 (qt = 64): smaller query groups where 16 needs local memory (-Xptxas -v): 4 (count) / 16 (emit) at
  // K = 1, 8 at K = 2
  constexpr int GQ = SRC && K <= 2 ? (K == 1 ? (EMIT ? 16 : 4) : 8) : gram_gq(K);
  // query groups per warp: ceil((qt / GQ) / GP_WPQ), qt <= 64 (48 at K = 5)
  constexpr int NGW = SRC && K <= 2 ? 16 / GQ : K <= 2 ? 1 : (K <= 4 ? 2 : 3);
  constexpr int QPS = qpar_stride(K);
  constexpr int NRP = source_rowpar_len(K);
  const int QT = A.qt;
  const RtLayout L = rt_layout<SRC>(K, QT, A.dpad);
  const GramPipe P = gram_pipe(smem, L.g, K, QT, A.dpad);
  float* thr = (float*)(smem + L.thr);
  float* qm = (float*)(smem + L.qm);
  float4* skp = (float4*)(smem + L.skp);
  unsigned int* cs = (unsigned int*)(smem + L.cs);
  unsigned int* rcn = (unsigned int*)(smem + L.rcn);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int part = blockIdx.x, qtile = blockIdx.y;
  const int64_t q0 = (int64_t)qtile * QT;
  const int nq = (int)((A.Q - q0 < QT) ? (A.Q - q0) : QT);
  const int64_t t0 = A.tiles * part / A.parts;
  const int64_t t1 = A.tiles * (part + 1) / A.parts;
  const int ntiles = (int)(t1 - t0);
  const int jn = (A.J - A.j0 < RT_JC) ? (A.J - A.j0) : RT_JC;

  if constexpr (SRC) {
    gram_init(P);
    for (int i = tid; i < QT; i += GP_THREADS) P.qpar[i] = (i < nq) ? A.qpar[q0 + i] : 0.0f;     // |e_q - mu|^2
  } else {
    gram_setup<K>(P, A.qpar, A.qplane, q0, nq, QT);
  }
  // thresholds: NaN (no positive in the slot), padding slots and padding queries become -inf = "count nothing"
  for (int i = tid; i < QT * RT_JC; i += GP_THREADS) {
    const int ql = i / RT_JC, j = i % RT_JC;
    float t = __int_as_float(0xff800000);
    if (ql < nq && j < jn) {
      const float v = A.thr[(q0 + ql) * A.J + A.j0 + j];
      if (v == v) t = fminf(v, 3.4028234e38f);             // +inf -> FLT_MAX: t - D~ stays -inf for padding rows
    }
    thr[i] = t;
    cs[i] = 0u;
  }
  for (int ql = tid; ql < QT && !SRC; ql += GP_THREADS) {   // SRC: the prototypes belong to the row
    float pm = 0.0f;
    if (ql < nq)
      for (int k = 0; k < K; ++k) pm = fmaxf(pm, A.qpar[(q0 + ql) * QPS + k]);      // log2(e) |p_k|^2
    qm[ql] = pm * CFL_LN2;                                    // max_k |p_k|^2
  }
  // Skip test of a whole query group (epilogue): with LB <= D~ the affine-hull lower bound and Vq >= V,
  //   D~ - m(D~) >= LB - S (rel1 + rel2 sqrt(LB Vq)) >= LB (1 - S k1) - S k0   (AM-GM with c = sqrt(Vq / tmax)),
  // k0 = rel1 + rel2 Vq / (2c), k1 = rel2 c / 2: when that exceeds the query's largest threshold the pair is farther than
  // every threshold and outside every band -- nothing to count, nothing to record.
  for (int ql = tid; ql < QT && !SRC; ql += GP_THREADS) {
    float tmax = __int_as_float(0xff800000);
    float k0 = A.rel1, k1 = 0.0f;
    if (ql < nq) {
      for (int j = 0; j < jn; ++j) {
        const float v = A.thr[(q0 + ql) * A.J + A.j0 + j];
        if (v == v) tmax = fmaxf(tmax, fminf(v, 3.4028234e38f));
      }
      if (K > 1) {
        const float cq = A.qpar[(q0 + ql) * QPS + K + qpar_tri(K)];       // >= (1 - 1/K) / 2 * max_kl |p_k - p_l|^2
        const float vq = cq / (0.5f * (1.0f - 1.0f / (float)K));          // >= the prototypes' spread under any weights
        const float c = sqrtf(vq / fmaxf(tmax, 1.0e-30f));
        k0 = A.rel1 + 0.5f * A.rel2 * vq / fmaxf(c, 1.0e-30f);
        k1 = 0.5f * A.rel2 * c;
        if (!(c == c) || !(k0 == k0) || !(k1 == k1) || k1 > 1.0e30f) { k0 = __int_as_float(0x7f800000); k1 = 0.0f; }   // never skip
      }
    }
    skp[ql] = make_float4(tmax, k0 * 1.0001f, k1 * 1.0001f, 0.0f);
  }
  if (tid == 0) *rcn = 0u;
  const unsigned int cta = blockIdx.y * gridDim.x + blockIdx.x;
  uint4* myrecs = A.recs + (size_t)cta * A.rec_slice;
  const uint32_t tmem_base = gram_start(P);

  if (warp == GP_NEPI) {
    gram_mma<SRC ? K : 1>(P, tmem_base, ntiles);
  } else if (warp == GP_NEPI + 1) {
    gram_tma<SRC ? K : 1>(P, A.qimg, qtile, A.cimg, t0, 1, ntiles);
  } else {
    // ======================================= epilogue ========================================
    const int lq = warp & 3, sub = warp >> 2;
    const int lrow = lq * 32 + lane;
    const uint32_t lane_lt = (1u << lane) - 1u;
    const float INF = __int_as_float(0x7f800000);
    // c[gi][i]: eight packed 4-bit counters (threshold j in nibble j) for query i of this warp's gi-th group
    uint32_t c[NGW][GQ];
#pragma unroll
    for (int gi = 0; gi < NGW; ++gi)
#pragma unroll
      for (int i = 0; i < GQ; ++i) c[gi][i] = 0u;

    auto flush = [&]() {
#pragma unroll
      for (int gi = 0; gi < NGW; ++gi) {
        const int g = sub + gi * GP_WPQ;
        if (g * GQ < nq) {                                    // warp-uniform
#pragma unroll
          for (int i = 0; i < GQ; ++i) {
            const uint32_t x = c[gi][i];
            c[gi][i] = 0u;
            const uint32_t ev = x & 0x0f0f0f0fu, od = (x >> 4) & 0x0f0f0f0fu;      // thresholds 0,2,4,6 | 1,3,5,7
            const uint32_t r0 = __reduce_add_sync(0xffffffffu, ev & 0x00ff00ffu);          // j = 0 | 4
            const uint32_t r1 = __reduce_add_sync(0xffffffffu, od & 0x00ff00ffu);          // j = 1 | 5
            const uint32_t r2 = __reduce_add_sync(0xffffffffu, (ev >> 8) & 0x00ff00ffu);   // j = 2 | 6
            const uint32_t r3 = __reduce_add_sync(0xffffffffu, (od >> 8) & 0x00ff00ffu);   // j = 3 | 7
            if (lane < RT_JC) {                               // lane j adds threshold j's sum
              const uint32_t lo2 = (lane & 1) ? r1 : r0, hi2 = (lane & 1) ? r3 : r2;
              const uint32_t r = (lane & 2) ? hi2 : lo2;
              const uint32_t v = (lane & 4) ? (r >> 16) : (r & 0xffffu);
              if (v) atomicAdd(cs + (g * GQ + i) * RT_JC + lane, v);
            }
          }
        }
      }
    };

    int since_flush = 0;
    // the skip test pays when most groups are far from every threshold (labelled positives near the top of the ranking:
    // the usual evaluation); each warp measures its hit rate over the first 16 tiles and switches the test off otherwise
    bool bound_on = !SRC;
    int grp_seen = 0, grp_skipped = 0;
    for (int t = 0; t < ntiles; ++t) {
      const int64_t row = (t0 + t) * 128 + lrow;
      const bool valid = row < A.N;
      float e2 = 0.0f;
      // SRC: the row's soft-min block, read where it is used, per query pair (L1 hits after the first); held in registers
      // across the TMEM loads and the group loop it pushed the counting kernel into local memory
      const float* rp = A.e2 + (t0 + t) * 128 * NRP + lrow;
      if constexpr (!SRC) e2 = __ldg(A.e2 + row);            // padded to whole tiles
      const uint32_t taddr = gram_acquire(P, tmem_base, t, lq);
#pragma unroll
      for (int gi = 0; gi < NGW; ++gi) {
        const int g = sub + gi * GP_WPQ;
        if (g * GQ >= nq) continue;                           // warp-uniform
        float gk[K][GQ];
        gram_load_group<K, GQ>(taddr, QT, g, gk);
        if (!SRC && bound_on) {
          constexpr int PBS = qplane_stride(K);
          const float e2s = e2 * (1.0f - CFL_PLANE_REL);
          const f2_t e2sp = pk2(e2s, e2s);
          bool need = false;
#pragma unroll
          for (int pi = 0; pi < GQ / 2; ++pi) {
            f2_t pv[PBS];
            load_pair_block<PBS>(P.qpl + (g * (GQ / 2) + pi) * PBS * 2, pv);
            float gA[K], gB[K], lbA, lbB;
#pragma unroll
            for (int k = 0; k < K; ++k) { gA[k] = gk[k][2 * pi]; gB[k] = gk[k][2 * pi + 1]; }
            plane_bound_pair<K>(gA, gB, e2sp, pv, lbA, lbB);
            const int ql = g * GQ + 2 * pi;
            const float4 sa = skp[ql], sb = skp[ql + 1];
            const float SA = e2 + qm[ql], SB = e2 + qm[ql + 1];
            const float fa = fmaf(-SA, sa.z, 1.0f), fb = fmaf(-SB, sb.z, 1.0f);     // 1 - S k1: must stay positive
            const float va = fmaf(lbA, fa, -SA * sa.y);
            const float vb = fmaf(lbB, fb, -SB * sb.y);
            need |= !(va > sa.x) | !(vb > sb.x) | !(fminf(fa, fb) > 0.0f);
          }
          ++grp_seen;
          if (!__any_sync(0xffffffffu, need && valid)) { ++grp_skipped; continue; }
        }
        const float* qg = P.qpar + g * GQ * QPS;
        float dist[GQ], var[GQ];
#pragma unroll
        for (int pi = 0; pi < GQ / 2; ++pi) {
          float gA[K], gB[K];
#pragma unroll
          for (int k = 0; k < K; ++k) { gA[k] = gk[k][2 * pi]; gB[k] = gk[k][2 * pi + 1]; }
          if constexpr (SRC) {
            const f2_t e2q = *(const f2_t*)(P.qpar + g * GQ + 2 * pi);
            f2_t rq[NRP];                                     // the row's block broadcast to the query pair
#pragma unroll
            for (int j = 0; j < NRP; ++j) {
              const float v = __ldg(rp + j * 128);
              rq[j] = (j < K) ? pk2(-v, -v) : pk2(v, v);
            }
            softmin_pair_var<K>(gA, gB, e2q, rq, dist[2 * pi], dist[2 * pi + 1], var[2 * pi], var[2 * pi + 1]);
          } else {
            f2_t qv[QPS];
            load_pair_block<QPS>(qg + pi * QPS * 2, qv);
            softmin_pair_var<K>(gA, gB, pk2(e2, e2), qv, dist[2 * pi], dist[2 * pi + 1], var[2 * pi], var[2 * pi + 1]);
          }
        }
        float pm = 0.0f;                                     // SRC: max_k |p_k|^2 of the row
        if constexpr (SRC) {
#pragma unroll
          for (int k = 0; k < K; ++k) pm = fmaxf(pm, __ldg(rp + k * 128));      // log2(e) |p_k|^2
          pm *= CFL_LN2;
        }
        uint32_t amb = 0u, sure = 0u;
#pragma unroll
        for (int i = 0; i < GQ; ++i) {
          const int ql = g * GQ + i;
          // band m = S * (rel1 + rel2 * sqrt(D~ * V)); var[] keeps it for the record
          const float S = SRC ? P.qpar[ql] + pm : e2 + qm[ql];
          const float sens = K == 1 ? 0.0f : sqrt_approx(fmaxf(dist[i], 0.0f) * fmaxf(var[i], 0.0f));
          const float m = S * fmaf(A.rel2, sens, A.rel1);
          var[i] = m;
          if (!valid) dist[i] = INF;                          // padding rows: t - inf = -inf, never counted, never in a band
          const f2_t nd = pk2(-dist[i], -dist[i]);
          const ulonglong2 ta = *(const ulonglong2*)(thr + ql * RT_JC);
          const ulonglong2 tb = *(const ulonglong2*)(thr + ql * RT_JC + 4);
          const f2_t tp[RT_JC / 2] = {ta.x, ta.y, tb.x, tb.y};
          float near = INF;
          if constexpr (EMIT) {                               // one radius in slot 0; slot 1 is padding (-inf)
            float x, y;
            upk2(add2(tp[0], nd), x, y);
            near = fminf(fminf(fabsf(x), fabsf(y)), near);
            if (x > m) sure |= 1u << i;                       // closer than t - m: inside whatever the direct form says
          } else {
#pragma unroll
            for (int jp = 0; jp < RT_JC / 2; ++jp) {
              float x, y;
              upk2(add2(tp[jp], nd), x, y);                   // t_j - D~ for two thresholds
              near = fminf(fminf(fabsf(x), fabsf(y)), near);
              count_pos(c[gi][i], x, 1u << (8 * jp));
              count_pos(c[gi][i], y, 1u << (8 * jp + 4));
            }
          }
          if (!(near > m)) amb |= 1u << i;                    // some threshold inside the band (or NaN)
        }
        if constexpr (EMIT) {
          // sure pairs straight to the query's segment: one ballot and one cursor atomic per (warp, query)
          if (__any_sync(0xffffffffu, sure != 0u)) {
#pragma unroll
            for (int i = 0; i < GQ; ++i) {
              const bool mine = (sure >> i) & 1u;
              const uint32_t mk = __ballot_sync(0xffffffffu, mine);
              if (mk == 0u) continue;                         // warp-uniform
              const int64_t q = q0 + g * GQ + i;
              const int leader = __ffs(mk) - 1;
              unsigned int basei = 0;
              if (lane == leader) basei = atomicAdd(A.cursor + q, (unsigned int)__popc(mk));
              basei = __shfl_sync(0xffffffffu, basei, leader);
              if (mine) {
                const int64_t at = (int64_t)basei + __popc(mk & lane_lt);
                const int64_t o = A.offsets[q];
                if (at < A.offsets[q + 1] - o) A.out[o + at] = row;     // beyond the count: reported by the finish kernel
              }
            }
          }
        }
        if (__any_sync(0xffffffffu, amb != 0u)) {
#pragma unroll
          for (int i = 0; i < GQ; ++i) {
            const bool mine = (amb >> i) & 1u;
            const uint32_t mk = __ballot_sync(0xffffffffu, mine);
            if (mk == 0u) continue;                           // warp-uniform
            const int ql = g * GQ + i;
            const int leader = __ffs(mk) - 1;
            unsigned int basei = 0;
            if (lane == leader) basei = atomicAdd(rcn, (unsigned int)__popc(mk));
            basei = __shfl_sync(0xffffffffu, basei, leader);
            if (mine) {
              const unsigned int at = basei + (unsigned int)__popc(mk & lane_lt);
              if (at < A.rec_slice) {
                myrecs[at] = make_uint4((uint32_t)(q0 + ql), (uint32_t)row, __float_as_uint(dist[i]), __float_as_uint(var[i]));
              } else {
                A.only[q0 + ql] = 1;
              }
            }
          }
        }
      }
      if (t == 15 && grp_skipped * 2 < grp_seen) bound_on = false;
      gram_release(P, t);
      if constexpr (!EMIT) {
        if (++since_flush == 15) { flush(); since_flush = 0; }
      }
    }
    if constexpr (!EMIT) flush();
    asm volatile("bar.sync 1, %0;" ::"n"(GP_EPI_THREADS) : "memory");
    if constexpr (!EMIT) {
      for (int i = tid; i < nq * RT_JC; i += GP_EPI_THREADS) {
        const int ql = i / RT_JC, j = i % RT_JC;
        if (j < jn && cs[i]) atomicAdd(&A.counts[((q0 + ql) * A.J + A.j0 + j) * 2], (unsigned long long)cs[i]);
      }
    }
    if (tid == 0) A.rec_n[cta] = *rcn < A.rec_slice ? *rcn : A.rec_slice;
  }
  gram_finish(P, tmem_base);
}

template <int K>
__global__ void __launch_bounds__(GP_THREADS, 1)     // 18 warps = 5 on one sub-partition: 5 x 32 x 96 registers is its whole file
rank_count_umma_kernel(RtArgs A) {
  rank_umma_body<K, false, false>(A);
}

// cfl_score_within's emitting pass (J = 1: A.thr = the radii)
template <int K>
__global__ void __launch_bounds__(GP_THREADS, 1)
within_emit_umma_kernel(RtArgs A) {
  rank_umma_body<K, false, true>(A);
}

// the same two passes over a source catalog (pcd_source)
template <int K>
__global__ void __launch_bounds__(GP_THREADS, 1)
rank_count_src_umma_kernel(RtArgs A) {
  rank_umma_body<K, true, false>(A);
}

template <int K>
__global__ void __launch_bounds__(GP_THREADS, 1)
within_emit_src_umma_kernel(RtArgs A) {
  rank_umma_body<K, true, true>(A);
}

// Exact verdicts of the ambiguous pairs: one thread per record, the direct-form device function of direct.cuh on the raw
// rows (bit-identical to cfl_pair_dist_rows / cfl_rank_counts; the operands are staged in shared memory -- the slice's
// query tile once per block, 32 catalog rows per warp and step with coalesced loads -- which changes no arithmetic).  stats: [0] records, [1] max |D~ - direct| / m in units
// of 2^-20, [2] records whose deviation exceeded m / 2.
constexpr int FX_THREADS = 128;
constexpr int FX_BLOCKS = 4;                        // blocks per list slice
// EMIT (cfl_score_within, J = 1): a record whose direct-form distance is below the radius is appended to its query's
// segment instead of correcting a count.  SRC: the query tile holds one vector per query and each record's K*d-float
// row is read in place (128 of them would not fit shared memory at K*d = 1024).
template <int K, bool SRC, bool EMIT>
__device__ __forceinline__ void
rank_fix_body(const uint4* __restrict__ recs_all, const unsigned int* __restrict__ rec_n, unsigned int slice,
              const float* __restrict__ Pq, int64_t ldq, const float* __restrict__ E, int64_t lde, int64_t N, int64_t Q,
              int d, int qt, int parts, const float* __restrict__ thr, int J, int j0, const int* __restrict__ only,
              unsigned long long* __restrict__ counts, unsigned long long* __restrict__ stats,
              const int64_t* __restrict__ offsets, unsigned int* __restrict__ cursor, int64_t* __restrict__ out) {
  extern __shared__ __align__(16) float fx_smem[];
  const unsigned int n = rec_n[blockIdx.y];                  // grid.y = the scoring kernel's CTAs, one list slice each
  if (n == 0 || (unsigned int)blockIdx.x * FX_THREADS >= n) return;
  const uint4* recs = recs_all + (size_t)blockIdx.y * slice;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int KD = SRC ? d : K * d, ldp = KD + 1, lder = d + 1;
  float* pq = fx_smem;                                       // [qt][K*d + 1]: the slice's query tile (SRC: [qt][d + 1])
  float* er = pq + (size_t)qt * ldp;                         // [FX_THREADS][d + 1]: one catalog row per thread (not SRC)
  const int64_t q0 = (int64_t)(blockIdx.y / parts) * qt;     // CTA (part, qtile) of the scoring kernel = qtile * parts + part
  const int nq = (int)((Q - q0 < qt) ? (Q - q0) : qt);
  for (int i = tid; i < nq * KD; i += FX_THREADS) {
    const int ql = i / KD, e = i - ql * KD;
    pq[ql * ldp + e] = Pq[(q0 + ql) * ldq + e];
  }
  __syncthreads();
  unsigned long long worst = 0, over = 0;
  for (unsigned int c0 = blockIdx.x * FX_THREADS; c0 < n; c0 += gridDim.x * FX_THREADS) {
    const unsigned int i = c0 + tid;
    const bool have = i < n;
    const uint4 r = have ? recs[i] : make_uint4(0u, 0u, 0u, 0u);
    const int64_t q = r.x, row = r.y;
    const bool live = have && !only[q] && row < N;
    // the warp gathers its 32 rows with coalesced loads; every thread then walks its own row in shared memory
    if constexpr (!SRC) {
    __syncwarp();
    for (int rr = 0; rr < 32; ++rr) {
      const int64_t rw = __shfl_sync(0xffffffffu, (unsigned int)r.y, rr);
      const bool ok = __shfl_sync(0xffffffffu, live ? 1 : 0, rr) != 0;
      if (!ok) continue;                                     // warp-uniform
      float* dst = er + (wid * 32 + rr) * lder;
      for (int j = lane; j < d; j += 32) dst[j] = E[rw * lde + j];
    }
    __syncwarp();
    }
    if (!live) continue;
    const float* qv = pq + (int)(q - q0) * ldp;
    float dist;
    if constexpr (SRC) {
      const float* pr = E + row * lde;
      dist = pcd_direct<K, 1>([&](int j) { return qv[j]; }, [&](int k, int j) { return __ldg(pr + k * d + j); }, d);
    } else {
      const float* ev = er + tid * lder;
      dist = pcd_direct<K>([&](int j) { return ev[j]; }, [&](int k, int j) { return qv[k * d + j]; }, d);
    }
    const float Dg = __uint_as_float(r.z), m = __uint_as_float(r.w);
    if constexpr (EMIT) {
      if (dist < thr[q]) {                                   // every record of a J = 1 pass lies inside its band
        const int64_t at = atomicAdd(cursor + q, 1u);
        const int64_t o = offsets[q];
        if (at < offsets[q + 1] - o) out[o + at] = row;
      }
    } else {
    for (int j = 0; j < RT_JC && j0 + j < J; ++j) {
      const float t = thr[q * J + j0 + j];
      if (!(t == t)) continue;                               // NaN: no positive in this slot
      const float x = fminf(t, 3.4028234e38f) + (-Dg);       // the scoring kernel's arithmetic, bit for bit
      if (fabsf(x) > m) continue;                            // outside the band: the fast verdict stands
      const int fast = x > 0.0f ? 1 : 0;                     // what the scoring kernel counted
      const int lt = dist < t ? 1 : 0;
      if (lt != fast) atomicAdd(&counts[((q * J) + j0 + j) * 2], (unsigned long long)(long long)(lt - fast));
      if (dist == t) atomicAdd(&counts[((q * J) + j0 + j) * 2 + 1], 1ull);
    }
    }
    const float dev = fabsf(Dg - dist);
    const float ratio = m > 0.0f ? dev / m : (dev > 0.0f ? 4096.0f : 0.0f);
    const unsigned long long u = (unsigned long long)fminf(ratio * 1048576.0f, 4.0e9f);
    if (u > worst) worst = u;
    if (ratio > 0.5f) ++over;
  }
  if (stats) {
    if (worst) atomicMax(&stats[1], worst);
    if (over) atomicAdd(&stats[2], over);
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&stats[0], (unsigned long long)n);
  }
}

template <int K>
__global__ void __launch_bounds__(FX_THREADS)
rank_fix_kernel(const uint4* __restrict__ recs_all, const unsigned int* __restrict__ rec_n, unsigned int slice,
                const float* __restrict__ Pq, int64_t ldq, const float* __restrict__ E, int64_t lde, int64_t N, int64_t Q,
                int d, int qt, int parts, const float* __restrict__ thr, int J, int j0, const int* __restrict__ only,
                unsigned long long* __restrict__ counts, unsigned long long* __restrict__ stats) {
  rank_fix_body<K, false, false>(recs_all, rec_n, slice, Pq, ldq, E, lde, N, Q, d, qt, parts, thr, J, j0, only, counts,
                                 stats, nullptr, nullptr, nullptr);
}

template <int K>
__global__ void __launch_bounds__(FX_THREADS)
rank_fix_src_kernel(const uint4* __restrict__ recs_all, const unsigned int* __restrict__ rec_n, unsigned int slice,
                    const float* __restrict__ Pq, int64_t ldq, const float* __restrict__ E, int64_t lde, int64_t N,
                    int64_t Q, int d, int qt, int parts, const float* __restrict__ thr, int J, int j0,
                    const int* __restrict__ only, unsigned long long* __restrict__ counts,
                    unsigned long long* __restrict__ stats) {
  rank_fix_body<K, true, false>(recs_all, rec_n, slice, Pq, ldq, E, lde, N, Q, d, qt, parts, thr, J, j0, only, counts,
                                stats, nullptr, nullptr, nullptr);
}

template <int K>
__global__ void __launch_bounds__(FX_THREADS)
within_fix_kernel(const uint4* __restrict__ recs_all, const unsigned int* __restrict__ rec_n, unsigned int slice,
                  const float* __restrict__ Pq, int64_t ldq, const float* __restrict__ E, int64_t lde, int64_t N,
                  int64_t Q, int d, int qt, int parts, const float* __restrict__ radius, const int* __restrict__ only,
                  unsigned long long* __restrict__ stats, const int64_t* __restrict__ offsets,
                  unsigned int* __restrict__ cursor, int64_t* __restrict__ out) {
  rank_fix_body<K, false, true>(recs_all, rec_n, slice, Pq, ldq, E, lde, N, Q, d, qt, parts, radius, 1, 0, only, nullptr,
                                stats, offsets, cursor, out);
}

template <int K>
__global__ void __launch_bounds__(FX_THREADS)
within_fix_src_kernel(const uint4* __restrict__ recs_all, const unsigned int* __restrict__ rec_n, unsigned int slice,
                      const float* __restrict__ Pq, int64_t ldq, const float* __restrict__ E, int64_t lde, int64_t N,
                      int64_t Q, int d, int qt, int parts, const float* __restrict__ radius, const int* __restrict__ only,
                      unsigned long long* __restrict__ stats, const int64_t* __restrict__ offsets,
                      unsigned int* __restrict__ cursor, int64_t* __restrict__ out) {
  rank_fix_body<K, true, true>(recs_all, rec_n, slice, Pq, ldq, E, lde, N, Q, d, qt, parts, radius, 1, 0, only, nullptr,
                               stats, offsets, cursor, out);
}

// queries whose records were dropped are recounted from scratch: clear what the fast path added
__global__ void rank_zero_flagged_kernel(const int* __restrict__ only, int64_t Q, int J, unsigned long long* counts,
                                         unsigned long long* stats) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= Q || !only[q]) return;
  for (int i = 0; i < 2 * J; ++i) counts[q * 2 * J + i] = 0ull;
  if (stats) atomicAdd(&stats[3], 1ull);
}

static void rank_tc_rel(float* rel1, float* rel2) {
  *rel1 = RT_REL1_DEFAULT; *rel2 = RT_REL2_DEFAULT;
  const char* x = getenv("CFL_EXPERIMENTS");
  if (!x || atoi(x) == 0) return;
  const char* e;
  if ((e = getenv("CFL_RANK_REL1"))) *rel1 = (float)atof(e);
  if ((e = getenv("CFL_RANK_REL2"))) *rel2 = (float)atof(e);
}

static unsigned int rank_tc_rec_cap(int64_t Q, int64_t N) {
  const char* e = getenv("CFL_EXPERIMENTS");
  if (e && atoi(e) != 0 && (e = getenv("CFL_RANK_REC_CAP")) && atoi(e) > 0) {     // tests: force the overflow path
    const unsigned int c = (unsigned int)atoi(e);
    return c < 1048576u ? c : 1048576u;
  }
  double pairs = (double)Q * (double)N;
  double cap = pairs / 256.0;
  if (cap < 1048576.0) cap = 1048576.0;
  if (cap > 268435456.0) cap = 268435456.0;
  return (unsigned int)cap;
}

// SRC: the forward layout, so that cfl_rank_counts_packed_stats finds the statistics at the same offset; the source query
// regions (centred query vectors, |e_q - mu|^2, the query image of one vector per query) reuse the forward ones.
struct RtWs { size_t pc, qpar, qimg, recs, recn, only, stats, total; };
static RtWs rank_tc_ws(int64_t Q, int K, int d, int64_t N, bool src = false) {
  RtWs w;
  const int qt = rank_tc_qt(K, d);
  const int nqt = qt > 0 ? (int)((Q + qt - 1) / qt) : 0;
  const int dpad = (d + 7) / 8 * 8;
  size_t off = 0;
  w.pc = off;    off = align_up(off + (size_t)Q * K * d * 4, 256);
  w.qpar = off;  off = align_up(off + (size_t)Q * (qpar_stride(K) + qplane_stride(K)) * 4, 256);
  w.qimg = off;  off = align_up(off + (size_t)nqt * qimg_tile_bytes(dpad, K * qt), 1024);
  w.recs = off;  off = align_up(off + (size_t)rank_tc_rec_cap(Q, N) * sizeof(uint4), 256);
  w.recn = off;  off = align_up(off + 4096 * sizeof(unsigned int), 256);
  w.only = off;  off = align_up(off + (size_t)Q * sizeof(int), 256);
  w.stats = off; off = align_up(off + CFL_RANK_NSTATS * sizeof(unsigned long long), 256);
  if (src) {     // Q*d centred vectors and Q norms always fit the forward pc / qpar regions; the query image of sqt
                 // vectors per tile fits the forward one unless Q is small against the tile (then it goes behind stats)
    const int sqt = rank_tc_qt(K, d, true);
    const int snqt = sqt > 0 ? (int)((Q + sqt - 1) / sqt) : 0;
    const size_t sbytes = (size_t)snqt * qimg_tile_bytes(dpad, sqt);
    if (sbytes > (size_t)nqt * qimg_tile_bytes(dpad, K * qt)) {
      off = align_up(off, 1024);
      w.qimg = off;  off = align_up(off + sbytes, 256);
    }
  }
  w.total = off + 1024;
  return w;
}

// The fix kernel stages the slice's query tile (K*d floats per query; SRC: d) and, forward, one d-float row per thread.
__host__ inline size_t fix_smem_bytes(bool src, int K, int d, int qt) {
  return ((size_t)qt * ((src ? 1 : K) * d + 1) + (src ? 0 : (size_t)FX_THREADS * (d + 1))) * sizeof(float);
}

template <int K, bool SRC>
static int rank_tc_launch(const RtArgs& a, const float* Pq, int64_t ldq, const float* E, int64_t lde,
                          unsigned long long* stats, cudaStream_t cs) {
  auto kern = SRC ? rank_count_src_umma_kernel<K> : rank_count_umma_kernel<K>;
  auto fix = SRC ? rank_fix_src_kernel<K> : rank_fix_kernel<K>;
  const size_t smem = rt_layout<SRC>(K, a.qt, a.dpad).g.total + 1024;
  CFL_SMEM_LIMIT(kern, smem);
  kern<<<dim3((unsigned)a.parts, (unsigned)a.nqt), GP_THREADS, smem, cs>>>(a);
  CFL_LAUNCH_CHECK();
  const size_t fx_smem = fix_smem_bytes(SRC, K, a.d, a.qt);
  CFL_SMEM_LIMIT(fix, fx_smem);
  fix<<<dim3(FX_BLOCKS, (unsigned)(a.parts * a.nqt)), FX_THREADS, fx_smem, cs>>>(
      a.recs, a.rec_n, a.rec_slice, Pq, ldq, E, lde, a.N, a.Q, a.d, a.qt, a.parts, a.thr, a.J, a.j0, a.only, a.counts, stats);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

// Query prep shared by the counting and the emitting pass: centred prototypes, soft-min and plane-bound blocks, the
// packed query image, the grid, the record list (cleared flags) and the band constants.
// src (pcd_source): the source-catalog call's prep (centred query vectors, |e_q - mu|^2, a query image with K = 1).
static int rank_tc_prepare(const char* what, bool src, const float* Pq, int64_t Q, int K, int d, int64_t ldq,
                           const void* image, int64_t N, const float* mu, void* ws, const RtWs& w, RtArgs& a,
                           cudaStream_t cs) {
  const int qt = rank_tc_qt(K, d, src);
  CFL_REQUIRE(qt > 0 && (src || score_umma_supported(K, d)), CFL_ERR_UNSUPPORTED,
              "%s: shape K=%d d=%d has no tcgen05 tiling", what, K, d);
  char* base = (char*)ws;
  float* Pc = (float*)(base + w.pc);
  float* qpar = (float*)(base + w.qpar);
  float* qplane = src ? nullptr : qpar + (size_t)Q * qpar_stride(K);
  int st = src ? score_prep_source_queries_launch(Pq, Q, d, ldq, mu, Pc, qpar, cs)
               : score_prep_queries_launch(Pq, Q, K, d, ldq, mu, Pc, qpar, qplane, cs);
  if (st != CFL_OK) return st;
  ScoreArgs sa = {};
  sa.K = K; sa.d = d; sa.Q = Q; sa.Pc = Pc; sa.src = src;
  sa.plan.qt = qt; sa.plan.nqt = (int)((Q + qt - 1) / qt); sa.plan.dpad = (d + 7) / 8 * 8;
  st = score_umma_pack_queries(sa, base + w.qimg, cs);
  if (st != CFL_OK) return st;

  a.K = K; a.d = d; a.Q = Q; a.N = N;
  a.qt = qt; a.nqt = sa.plan.nqt; a.dpad = sa.plan.dpad;
  a.tiles = (N + 127) / 128;
  int sms = sm_count();
  if (sms <= 0) sms = 148;
  int64_t parts = sms / a.nqt;
  if (parts < 1) parts = 1;
  if (parts > a.tiles) parts = a.tiles;
  a.parts = (int)parts;
  a.qpar = qpar; a.qplane = qplane; a.qimg = base + w.qimg;
  if (src) {
    const SourceCatalogView v = source_catalog_view(image, N, K, d);
    a.cimg = v.blocks; a.e2 = v.rowpar;
  } else {
    a.cimg = image; a.e2 = catalog_view(image, N, d).e2;
  }
  CFL_REQUIRE((int64_t)a.parts * a.nqt <= 4096, CFL_ERR_UNSUPPORTED, "%s: Q=%lld needs more than 4096 CTAs", what,
              (long long)Q);
  a.recs = (uint4*)(base + w.recs); a.rec_slice = rank_tc_rec_cap(Q, N) / (unsigned int)(a.parts * a.nqt);
  a.rec_n = (unsigned int*)(base + w.recn);
  a.only = (int*)(base + w.only);
  rank_tc_rel(&a.rel1, &a.rel2);
  CFL_CUDA(cudaMemsetAsync(a.only, 0, (size_t)Q * sizeof(int), cs));
  return CFL_OK;
}

__global__ void within_reset_flagged_kernel(const int* __restrict__ only, int64_t Q, unsigned int* cursor,
                                            unsigned long long* stats) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= Q || !only[q]) return;
  cursor[q] = 0u;
  atomicAdd(&stats[3], 1ull);
}

template <int K, bool SRC>
static int within_tc_launch(const RtArgs& a, const float* Pq, int64_t ldq, const float* E, int64_t lde,
                            unsigned long long* stats, cudaStream_t cs) {
  auto kern = SRC ? within_emit_src_umma_kernel<K> : within_emit_umma_kernel<K>;
  auto fix = SRC ? within_fix_src_kernel<K> : within_fix_kernel<K>;
  const size_t smem = rt_layout<SRC>(K, a.qt, a.dpad).g.total + 1024;
  CFL_SMEM_LIMIT(kern, smem);
  kern<<<dim3((unsigned)a.parts, (unsigned)a.nqt), GP_THREADS, smem, cs>>>(a);
  CFL_LAUNCH_CHECK();
  const size_t fx_smem = fix_smem_bytes(SRC, K, a.d, a.qt);
  CFL_SMEM_LIMIT(fix, fx_smem);
  fix<<<dim3(FX_BLOCKS, (unsigned)(a.parts * a.nqt)), FX_THREADS, fx_smem, cs>>>(
      a.recs, a.rec_n, a.rec_slice, Pq, ldq, E, lde, a.N, a.Q, a.d, a.qt, a.parts, a.thr, a.only, stats, a.offsets,
      a.cursor, a.out);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

size_t within_tc_workspace_bytes(int64_t Q, int K, int d, int64_t N, bool src) {
  return rank_tc_ws(Q, K, d, N, src).total;
}

// Emitting pass of cfl_score_within on the tensor cores (pcd / siamese / pcd_source): sure rows straight from the scoring epilogue,
// band rows after the direct-form check, queries whose records overflowed the list re-emitted from scratch on the
// CUDA cores.  cursor[Q] must be zero; stats as CFL_WITHIN_NSTATS.
int within_tc_emit(int mode, const float* Pq, int64_t Q, int K, int d, int64_t ldq, const float* E, const void* image,
                   int64_t N, int64_t lde, const float* mu, const float* radius, const int64_t* offsets,
                   unsigned int* cursor, int64_t* out, void* ws, unsigned long long* stats, cudaStream_t cs) {
  const bool src = mode == CFL_PCD_SOURCE;
  const RtWs w = rank_tc_ws(Q, K, d, N, src);
  RtArgs a = {};
  int st = rank_tc_prepare("score_within", src, Pq, Q, K, d, ldq, image, N, mu, ws, w, a, cs);
  if (st != CFL_OK) return st;
  a.J = 1; a.j0 = 0; a.thr = radius;
  a.offsets = offsets; a.cursor = cursor; a.out = out;
  CFL_CUDA(cudaMemsetAsync(a.rec_n, 0, 4096 * sizeof(unsigned int), cs));
  st = with_k(K, [&](auto KC) {
    return src ? within_tc_launch<KC, true>(a, Pq, ldq, E, lde, stats, cs)
               : within_tc_launch<KC, false>(a, Pq, ldq, E, lde, stats, cs);
  });
  if (st != CFL_OK) return st;
  within_reset_flagged_kernel<<<(unsigned)((Q + 255) / 256), 256, 0, cs>>>(a.only, Q, cursor, stats);
  CFL_LAUNCH_CHECK();
  return within_emit_launch(mode, Pq, Q, K, d, ldq, nullptr, E, N, lde, radius, offsets, cursor, out, a.only, cs);
}

}  // namespace cfl

using namespace cfl;

extern "C" {

size_t cfl_rank_counts_packed_workspace_bytes(int64_t Q, int K, int d, int64_t N) {
  if (Q <= 0 || N <= 0 || K < 1 || K > CFL_MAX_K || d < 1 || d > 128) return 4096;
  return rank_tc_ws(Q, K, d, N).total;
}

size_t cfl_rank_counts_packed_source_workspace_bytes(int64_t Q, int K, int d, int64_t N) {
  if (Q <= 0 || N <= 0 || K < 1 || K > CFL_MAX_K || d < 1 || d > 128) return 4096;
  return rank_tc_ws(Q, K, d, N, true).total;
}

int cfl_rank_counts_packed(int mode, const float* Pq, int64_t Q, int K, int d, int64_t ldq, const float* E,
                           const void* image, int64_t N, int64_t lde, const float* mu, const float* pos_dist, int J,
                           int64_t* counts, void* ws, size_t ws_bytes, void* stream) {
  int st = device_check();
  if (st != CFL_OK) return st;
  CFL_REQUIRE(mode == CFL_PCD || mode == CFL_SIAMESE || mode == CFL_PCD_SOURCE, CFL_ERR_UNSUPPORTED,
              "rank_counts_packed: mode %d not supported (pcd, siamese, pcd_source)", mode);
  const bool src = mode == CFL_PCD_SOURCE;
  CFL_REQUIRE(mode != CFL_SIAMESE || K == 1, CFL_ERR_INVALID, "rank_counts_packed: siamese needs K=1");
  CFL_REQUIRE(K >= 1 && K <= CFL_MAX_K, CFL_ERR_UNSUPPORTED, "rank_counts_packed: K=%d outside [1,%d]", K, CFL_MAX_K);
  CFL_REQUIRE(d >= 1 && d <= 128, CFL_ERR_UNSUPPORTED, "rank_counts_packed: d=%d outside [1,128]", d);
  CFL_REQUIRE(J >= 1 && J <= CFL_MAX_RANK_J, CFL_ERR_UNSUPPORTED, "rank_counts_packed: J=%d outside [1,%d]", J, CFL_MAX_RANK_J);
  CFL_REQUIRE(Q >= 0 && N >= 0 && N < ((int64_t)1 << 32) && Q < ((int64_t)1 << 31), CFL_ERR_INVALID, "rank_counts_packed: bad Q/N");
  CFL_REQUIRE(ldq >= (src ? d : (int64_t)K * d) && lde >= (src ? (int64_t)K * d : d), CFL_ERR_INVALID,
              "rank_counts_packed: leading dimension too small");
  if (Q == 0) return CFL_OK;
  CFL_REQUIRE(Pq && pos_dist && counts, CFL_ERR_INVALID, "rank_counts_packed: NULL argument");
  cudaStream_t cs = (cudaStream_t)stream;
  CFL_CUDA(cudaMemsetAsync(counts, 0, (size_t)Q * J * 2 * sizeof(int64_t), cs));
  if (N == 0) return CFL_OK;
  CFL_REQUIRE(E && image, CFL_ERR_INVALID, "rank_counts_packed: NULL catalog / image");
  CFL_REQUIRE(!src || ((uintptr_t)image & 1023u) == 0, CFL_ERR_INVALID, "rank_counts_packed: image must be 1024-byte aligned");
  CFL_REQUIRE(rank_tc_qt(K, d, src) > 0 && (src || score_umma_supported(K, d)), CFL_ERR_UNSUPPORTED,
              "rank_counts_packed: shape K=%d d=%d has no tcgen05 tiling", K, d);
  const RtWs w = rank_tc_ws(Q, K, d, N, src);
  CFL_REQUIRE(ws && ws_bytes >= w.total, CFL_ERR_WORKSPACE, "rank_counts_packed: workspace too small (%zu < %zu)",
              ws_bytes, w.total);
  RtArgs a = {};
  st = rank_tc_prepare("rank_counts_packed", src, Pq, Q, K, d, ldq, image, N, mu, ws, w, a, cs);
  if (st != CFL_OK) return st;
  a.J = J;
  a.thr = pos_dist; a.counts = (unsigned long long*)counts;
  unsigned long long* stats = (unsigned long long*)((char*)ws + w.stats);
  CFL_CUDA(cudaMemsetAsync(stats, 0, CFL_RANK_NSTATS * sizeof(unsigned long long), cs));
  timer_record(0, cs);
  for (int j0 = 0; j0 < J; j0 += RT_JC) {
    a.j0 = j0;
    CFL_CUDA(cudaMemsetAsync(a.rec_n, 0, 4096 * sizeof(unsigned int), cs));
    st = with_k(K, [&](auto KC) {
      return src ? rank_tc_launch<KC, true>(a, Pq, ldq, E, lde, stats, cs)
                 : rank_tc_launch<KC, false>(a, Pq, ldq, E, lde, stats, cs);
    });
    if (st != CFL_OK) return st;
  }
  timer_record(1, cs);
  // queries whose ambiguous records overflowed the list (the flags are final only now: a later threshold chunk may
  // have raised one): clear them and recount them from scratch on the CUDA cores
  rank_zero_flagged_kernel<<<(unsigned)((Q + 255) / 256), 256, 0, cs>>>(a.only, Q, J, a.counts, stats);
  CFL_LAUNCH_CHECK();
  return rank_counts_only_launch(mode, Pq, Q, K, d, ldq, E, N, lde, pos_dist, J, a.counts, a.only, cs);
}

int cfl_rank_counts_packed_stats(int64_t Q, int K, int d, int64_t N, const void* ws, size_t ws_bytes, int64_t* out,
                                 void* stream) {
  int st = device_check();
  if (st != CFL_OK) return st;
  CFL_REQUIRE(out, CFL_ERR_INVALID, "rank_counts_packed_stats: NULL argument");
  for (int i = 0; i < CFL_RANK_NSTATS; ++i) out[i] = 0;
  if (Q <= 0 || N <= 0) return CFL_OK;
  const RtWs w = rank_tc_ws(Q, K, d, N);
  CFL_REQUIRE(ws && ws_bytes >= w.total, CFL_ERR_WORKSPACE, "rank_counts_packed_stats: workspace too small");
  cudaStream_t cs = (cudaStream_t)stream;
  CFL_CUDA(cudaMemcpyAsync(out, (const char*)ws + w.stats, CFL_RANK_NSTATS * sizeof(int64_t), cudaMemcpyDeviceToHost, cs));
  CFL_CUDA(cudaStreamSynchronize(cs));
  return CFL_OK;
}

}  // extern "C"
