// Per-query all-candidate AUC (SURVEY 8d C3 "per-query all-candidate AUC with J planted positives",
// 8e "AUC across ranks"): the rank statistic of roc_auc_score (cfl/utils.py:267-268) for ONE query
// against EVERY catalog row, without materialising the Q x N scores.
//
//   cfl_pair_dist_rows : t[q,j] = dist(query q, catalog row pos_idx[q,j])        (the labelled positives)
//   cfl_rank_counts    : counts[q,j] = ( #{c : dist(q,c) < t[q,j]},  #{c : dist(q,c) == t[q,j]} )  over a shard
//
// Both evaluate the pair scorer (DistBase.build_dist, cfl/models/base.py:107-146) in fp32
// direct-difference form through the SAME device function, operation for operation, so a positive
// compares equal to itself and the integer counts are exact for the fp32 distances; they add over
// catalog shards (int64 all-reduce), which makes the AUC independent of the sharding.  The pcd
// arithmetic is that of merge_rescore_kernel (score.cu), i.e. of the values cfl_score_topk reports;
// the monomer arithmetic is that of score_monomer_kernel.
//
// The source modes swap the roles (queries = target items, catalog rows = source items): pcd_source takes e = the
// query's e0 and p = the row's K prototypes (merge_rescore_src_kernel's values), monomer_source takes the query's
// K prototypes and the row's a and gate w (mono_rescore_src_kernel's values).  The bodies below take the role as a
// template argument; the kernels of the forward modes keep their names and code, the source modes have their own.
#include "score.cuh"
#include "direct.cuh"

namespace cfl {

constexpr int RC_QT = 8;          // queries per CTA
constexpr int RC_THREADS = 128;   // one thread per catalog row of a 128-row tile
constexpr int RC_MAX_J = 32;
constexpr size_t RC_SMEM_MAX = 200 * 1024;

// Roles of the query and the catalog row.  Floats per catalog row staged in shared memory / per query:
//   RC_PCD      row e0 [d],          query K prototypes [K*d]
//   RC_MONO     row K prototypes,    query a [d] (gate Wq per query)
//   RC_PCD_SRC  row K prototypes,    query e0 [d]
//   RC_MONO_SRC row a [d] + gate [K] (Wq per row), query K prototypes
constexpr int RC_PCD = 0, RC_MONO = 1, RC_PCD_SRC = 2, RC_MONO_SRC = 3;
__host__ __device__ constexpr int rc_role(int mode) {
  return mode == CFL_MONOMER ? RC_MONO : mode == CFL_PCD_SOURCE ? RC_PCD_SRC : mode == CFL_MONOMER_SOURCE ? RC_MONO_SRC
                                                                                                          : RC_PCD;
}
__host__ __device__ constexpr int rc_row_floats(int role, int K, int d) {
  return role == RC_PCD ? d : role == RC_MONO_SRC ? d + K : K * d;
}
__host__ __device__ constexpr int rc_query_floats(int role, int K, int d) {
  return role == RC_MONO || role == RC_PCD_SRC ? d : K * d;
}

struct RcArgs {
  int mode, K, d, J;
  int64_t Q, N, ldq, lde;
  const float* Pq;         // [Q, ldq] rc_query_floats per query (roles above)
  const float* Wq;         // the monomer gate: [Q, K] (monomer), [N, K] (monomer_source)
  const float* E;          // [N, lde] catalog rows (roles above; monomer_source: a, its gate in Wq)
  const float* thr;        // [Q, J] distances of the positives (NaN = no positive)
  const int64_t* pos_idx;  // [Q, J] gather kernel
  float* pos_dist;         // [Q, J] gather kernel output
  unsigned long long* counts;   // [Q, J, 2]
  const int* only;         // optional [Q]: count only the flagged queries (fallback of cfl_rank_counts_packed)
  int parts;
  int64_t tiles;
};
// emitting variant (cfl_score_within, J = 1): rows dist < thr[q] appended to out[offsets[q], offsets[q + 1])
struct RcEmit {
  const int64_t* offsets;
  unsigned int* cursor;
  int64_t* out;
};

// Four queries per pass through a catalog row: every shared-memory load of the row serves four distance
// evaluations and the query operands arrive as one 128-bit broadcast load (the first version issued two
// 32-bit loads per FMA and sat at 66 % of the LSU pipe).  Per query the operation sequence is exactly that of
// pcd_direct / monomer_direct above, so the values -- and the counts -- are bit-identical to theirs.
template <int K>
__device__ __forceinline__ void pcd_direct4(const float* __restrict__ er, const float4* __restrict__ q4, int d,
                                            float (&dist)[4]) {
  float dk[4][K];
  float mn[4] = {3.0e38f, 3.0e38f, 3.0e38f, 3.0e38f};
#pragma unroll
  for (int k = 0; k < K; ++k) {
    float acc[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll 4
    for (int j = 0; j < d; ++j) {
      const float e = er[j];
      const float4 p = q4[(k * d + j) * 2];
      float df;
      df = e - p.x; acc[0] = fmaf(df, df, acc[0]);
      df = e - p.y; acc[1] = fmaf(df, df, acc[1]);
      df = e - p.z; acc[2] = fmaf(df, df, acc[2]);
      df = e - p.w; acc[3] = fmaf(df, df, acc[3]);
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) { dk[c][k] = acc[c]; mn[c] = fminf(mn[c], acc[c]); }
  }
  if (K == 1) {
#pragma unroll
    for (int c = 0; c < 4; ++c) dist[c] = dk[c][0];
    return;
  }
  float inv[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    float sum = 0.0f;
#pragma unroll
    for (int k = 0; k < K; ++k) { dk[c][k] = expf(mn[c] - dk[c][k]); sum += dk[c][k]; }
    inv[c] = 1.0f / sum;
    dist[c] = 0.0f;
  }
#pragma unroll 2
  for (int j = 0; j < d; ++j) {
    const float e = er[j];
    float m[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const float4 p = q4[(k * d + j) * 2];
      m[0] = fmaf(dk[0][k] * inv[0], p.x, m[0]);
      m[1] = fmaf(dk[1][k] * inv[1], p.y, m[1]);
      m[2] = fmaf(dk[2][k] * inv[2], p.z, m[2]);
      m[3] = fmaf(dk[3][k] * inv[3], p.w, m[3]);
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) { const float r = e - m[c]; dist[c] = fmaf(r, r, dist[c]); }
  }
}

// The source roles: e = the query (four of them in q4), p = the row's K prototypes (er[k * d + j]) -- pcd_direct's
// operation order with the swapped accessors.
template <int K>
__device__ __forceinline__ void pcd_src_direct4(const float* __restrict__ er, const float4* __restrict__ q4, int d,
                                                float (&dist)[4]) {
  float dk[4][K];
  float mn[4] = {3.0e38f, 3.0e38f, 3.0e38f, 3.0e38f};
#pragma unroll
  for (int k = 0; k < K; ++k) {
    float acc[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll 4
    for (int j = 0; j < d; ++j) {
      const float p = er[k * d + j];
      const float4 e = q4[j * 2];
      float df;
      df = e.x - p; acc[0] = fmaf(df, df, acc[0]);
      df = e.y - p; acc[1] = fmaf(df, df, acc[1]);
      df = e.z - p; acc[2] = fmaf(df, df, acc[2]);
      df = e.w - p; acc[3] = fmaf(df, df, acc[3]);
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) { dk[c][k] = acc[c]; mn[c] = fminf(mn[c], acc[c]); }
  }
  if (K == 1) {
#pragma unroll
    for (int c = 0; c < 4; ++c) dist[c] = dk[c][0];
    return;
  }
  float inv[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    float sum = 0.0f;
#pragma unroll
    for (int k = 0; k < K; ++k) { dk[c][k] = expf(mn[c] - dk[c][k]); sum += dk[c][k]; }
    inv[c] = 1.0f / sum;
    dist[c] = 0.0f;
  }
#pragma unroll 2
  for (int j = 0; j < d; ++j) {
    const float4 e = q4[j * 2];
    float m[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const float p = er[k * d + j];
      m[0] = fmaf(dk[0][k] * inv[0], p, m[0]);
      m[1] = fmaf(dk[1][k] * inv[1], p, m[1]);
      m[2] = fmaf(dk[2][k] * inv[2], p, m[2]);
      m[3] = fmaf(dk[3][k] * inv[3], p, m[3]);
    }
    float r;
    r = e.x - m[0]; dist[0] = fmaf(r, r, dist[0]);
    r = e.y - m[1]; dist[1] = fmaf(r, r, dist[1]);
    r = e.z - m[2]; dist[2] = fmaf(r, r, dist[2]);
    r = e.w - m[3]; dist[3] = fmaf(r, r, dist[3]);
  }
}

// monomer_source: the row is a (er[0, d)) and its gate (er[d, d + K)), the queries' K prototypes in q4 -- monomer_direct
// with e = the query's prototypes, a / w = the row's.
template <int K>
__device__ __forceinline__ void monomer_src_direct4(const float* __restrict__ er, const float4* __restrict__ p4, int d,
                                                    float (&dist)[4]) {
  float acc[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
  for (int k = 0; k < K; ++k) {
    float dk[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll 4
    for (int j = 0; j < d; ++j) {
      const float a = er[j];
      const float4 p = p4[(k * d + j) * 2];
      float df;
      df = a + (-p.x); dk[0] = fmaf(df, df, dk[0]);
      df = a + (-p.y); dk[1] = fmaf(df, df, dk[1]);
      df = a + (-p.z); dk[2] = fmaf(df, df, dk[2]);
      df = a + (-p.w); dk[3] = fmaf(df, df, dk[3]);
    }
    const float w = er[d + k];
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[c] = fmaf(w, dk[c], acc[c]);
  }
#pragma unroll
  for (int c = 0; c < 4; ++c) dist[c] = acc[c];
}

template <int K>
__device__ __forceinline__ void monomer_direct4(const float* __restrict__ er, const float4* __restrict__ a4,
                                                const float* __restrict__ w /* [4][K] */, int d, float (&dist)[4]) {
  float acc[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
  for (int k = 0; k < K; ++k) {
    float dk[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll 4
    for (int j = 0; j < d; ++j) {
      const float ne = -er[k * d + j];
      const float4 a = a4[j * 2];
      float df;
      df = a.x + ne; dk[0] = fmaf(df, df, dk[0]);
      df = a.y + ne; dk[1] = fmaf(df, df, dk[1]);
      df = a.z + ne; dk[2] = fmaf(df, df, dk[2]);
      df = a.w + ne; dk[3] = fmaf(df, df, dk[3]);
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[c] = fmaf(w[c * K + k], dk[c], acc[c]);
  }
#pragma unroll
  for (int c = 0; c < 4; ++c) dist[c] = acc[c];
}

// VW = floats per staging load (4 when the row length, the row stride and the base pointer allow 128-bit loads); VW = 0
// (pcd_source when 128 rows of K*d floats do not fit shared memory): no staging, each thread reads its row in place
// through L1, in the same order.
// EMIT: instead of counting, the rows closer than the (single) threshold are appended to their query's segment -- one
// ballot and one cursor atomic per (warp, query); with `only`, for the flagged queries alone.
template <int K, int ROLE, int VW, bool EMIT>
__device__ __forceinline__ void rank_count_body(const RcArgs& A, const RcEmit& X) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int d = A.d, J = A.J;
  const int ew = rc_row_floats(ROLE, K, d);   // floats per catalog row
  const int qw = rc_query_floats(ROLE, K, d); // floats per query
  const int ldt = ew + 1;
  float4* q4 = (float4*)smem_raw;                             // [qw][2]: element i of queries 0-3 | 4-7 (zero padded)
  float* et = (float*)(q4 + 2 * qw);                          // [128][ew+1] (none when VW = 0)
  float* ws = et + (VW == 0 ? 0 : 128 * ldt);                // [QT][K] (monomer)
  float* thr = ws + RC_QT * K;                                // [QT][J]
  int* cnt = (int*)(thr + RC_QT * J);                         // [4 warps][QT][J][2]

  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int part = blockIdx.x;
  const int64_t q0 = (int64_t)blockIdx.y * RC_QT;
  const int nq = (int)((A.Q - q0 < RC_QT) ? (A.Q - q0) : RC_QT);
  unsigned emit_mask = 0xffffffffu;
  if (A.only != nullptr) {                                   // restricted recount: leave unless a query here is flagged
    int flagged = 0;
    for (int ql = 0; ql < nq; ++ql) flagged |= A.only[q0 + ql];
    if (!flagged) return;
    if constexpr (EMIT) {
      emit_mask = 0u;
      for (int ql = 0; ql < nq; ++ql) emit_mask |= (A.only[q0 + ql] != 0 ? 1u : 0u) << ql;
    }
  }
  for (int i = tid; i < RC_QT * qw; i += RC_THREADS) {
    const int ql = i / qw, e = i % qw;
    ((float*)q4)[e * RC_QT + ql] = ql < nq ? A.Pq[(q0 + ql) * A.ldq + e] : 0.0f;
  }
  if (ROLE == RC_MONO) for (int i = tid; i < RC_QT * K; i += RC_THREADS) ws[i] = i < nq * K ? A.Wq[q0 * K + i] : 0.0f;
  for (int i = tid; i < nq * J; i += RC_THREADS) thr[i] = A.thr[q0 * J + i];
  for (int i = tid; i < (RC_THREADS / 32) * RC_QT * J * 2; i += RC_THREADS) cnt[i] = 0;
  int* mycnt = cnt + wid * RC_QT * J * 2;
  const int64_t t0 = A.tiles * part / A.parts;
  const int64_t t1 = A.tiles * (part + 1) / A.parts;
  const int dv = (ROLE == RC_MONO_SRC ? d : ew) / (VW > 0 ? VW : 1);   // staging loads per row from E
  const int sr0 = tid / dv, sj0 = tid % dv, sdr = RC_THREADS / dv, sdj = RC_THREADS % dv;

  for (int64_t tile = t0; tile < t1; ++tile) {
    const int64_t r0 = tile * 128;
    __syncthreads();
    for (int i = tid, r = sr0, j = sj0; VW > 0 && i < 128 * dv; i += RC_THREADS) {
      const int64_t row = r0 + r;
      const float* src = A.E + row * A.lde + VW * j;
      float* dst = et + r * ldt + VW * j;
      if (VW == 4) {
        const float4 v = row < A.N ? *(const float4*)src : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
        dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
      } else {
        dst[0] = row < A.N ? *src : 0.0f;
      }
      r += sdr; j += sdj;
      if (j >= dv) { j -= dv; ++r; }
    }
    if (ROLE == RC_MONO_SRC)                                   // the row's gate behind its a
      for (int i = tid; i < 128 * K; i += RC_THREADS) {
        const int64_t row = r0 + i / K;
        et[(i / K) * ldt + d + i % K] = row < A.N ? A.Wq[row * K + i % K] : 0.0f;
      }
    __syncthreads();
    const bool valid = r0 + tid < A.N;
    const float* er = VW > 0 ? et + tid * ldt : A.E + (valid ? r0 + tid : 0) * A.lde;
    for (int qh = 0; qh * 4 < nq; ++qh) {
      float dist[4];
      if (ROLE == RC_MONO)          monomer_direct4<K>(er, q4 + qh, ws + qh * 4 * K, d, dist);
      else if (ROLE == RC_PCD_SRC)  pcd_src_direct4<K>(er, q4 + qh, d, dist);
      else if (ROLE == RC_MONO_SRC) monomer_src_direct4<K>(er, q4 + qh, d, dist);
      else                          pcd_direct4<K>(er, q4 + qh, d, dist);
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int ql = qh * 4 + c;
        if (ql < nq) {                                         // warp-uniform
          if constexpr (EMIT) {
            const bool mine = valid && dist[c] < thr[ql];
            const unsigned lt = __ballot_sync(0xffffffffu, mine);
            if (lt != 0u && ((emit_mask >> ql) & 1u)) {        // warp-uniform
              const int64_t q = q0 + ql;
              unsigned int basei = 0;
              if (lane == 0) basei = atomicAdd(X.cursor + q, (unsigned int)__popc(lt));
              basei = __shfl_sync(0xffffffffu, basei, 0);
              if (mine) {
                const int64_t at = (int64_t)basei + __popc(lt & ((1u << lane) - 1u));
                const int64_t o = X.offsets[q];
                if (at < X.offsets[q + 1] - o) X.out[o + at] = r0 + tid;   // beyond the count: reported at the finish
              }
            }
          } else {
          for (int j = 0; j < J; ++j) {
            const float t = thr[ql * J + j];
            const unsigned lt = __ballot_sync(0xffffffffu, valid && dist[c] < t);
            const unsigned eq = __ballot_sync(0xffffffffu, valid && dist[c] == t);
            if (lane == 0) {
              mycnt[(ql * J + j) * 2] += __popc(lt);
              mycnt[(ql * J + j) * 2 + 1] += __popc(eq);
            }
          }
          }
        }
      }
    }
  }
  if constexpr (EMIT) return;
  __syncthreads();
  for (int i = tid; i < nq * J * 2; i += RC_THREADS) {
    unsigned long long s = 0;
    for (int w = 0; w < RC_THREADS / 32; ++w) s += (unsigned long long)cnt[w * RC_QT * J * 2 + i];
    if (A.only != nullptr && !A.only[q0 + i / (J * 2)]) continue;
    if (s) atomicAdd(&A.counts[q0 * J * 2 + i], s);
  }
}

template <int K, bool MONO, int VW>
__global__ void __launch_bounds__(RC_THREADS)
rank_count_kernel(RcArgs A) {
  rank_count_body<K, MONO ? RC_MONO : RC_PCD, VW, false>(A, RcEmit{});
}

template <int K, bool MONO, int VW>
__global__ void __launch_bounds__(RC_THREADS)
within_emit_kernel(RcArgs A, RcEmit X) {
  rank_count_body<K, MONO ? RC_MONO : RC_PCD, VW, true>(A, X);
}

// the source modes (MONO: monomer_source, else pcd_source)
template <int K, bool MONO, int VW>
__global__ void __launch_bounds__(RC_THREADS)
rank_count_src_kernel(RcArgs A) {
  rank_count_body<K, MONO ? RC_MONO_SRC : RC_PCD_SRC, VW, false>(A, RcEmit{});
}

template <int K, bool MONO, int VW>
__global__ void __launch_bounds__(RC_THREADS)
within_emit_src_kernel(RcArgs A, RcEmit X) {
  rank_count_body<K, MONO ? RC_MONO_SRC : RC_PCD_SRC, VW, true>(A, X);
}

// One thread per (query, positive): the same device functions on rows gathered from global memory.
template <int K, int ROLE>
__device__ __forceinline__ void dist_rows_body(const RcArgs& A) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= A.Q * A.J) return;
  const int64_t q = i / A.J;
  const int64_t row = A.pos_idx[i];
  float dist = __int_as_float(0x7fc00000);                   // NaN: no positive here
  if (row >= 0 && row < A.N) {
    const float* er = A.E + row * A.lde;
    const float* qv = A.Pq + q * A.ldq;
    const int d = A.d;
    if (ROLE == RC_MONO) {
      const float* wv = A.Wq + q * K;
      dist = monomer_direct<K>([&](int k, int j) { return er[k * d + j]; }, [&](int j) { return qv[j]; },
                               [&](int k) { return wv[k]; }, d);
    } else if (ROLE == RC_PCD_SRC) {
      dist = pcd_direct<K>([&](int j) { return qv[j]; }, [&](int k, int j) { return er[k * d + j]; }, d);
    } else if (ROLE == RC_MONO_SRC) {
      const float* wv = A.Wq + row * K;
      dist = monomer_direct<K>([&](int k, int j) { return qv[k * d + j]; }, [&](int j) { return er[j]; },
                               [&](int k) { return wv[k]; }, d);
    } else {
      dist = pcd_direct<K>([&](int j) { return er[j]; }, [&](int k, int j) { return qv[k * d + j]; }, d);
    }
  }
  A.pos_dist[i] = dist;
}

template <int K, bool MONO>
__global__ void pair_dist_rows_kernel(RcArgs A) {
  dist_rows_body<K, MONO ? RC_MONO : RC_PCD>(A);
}

template <int K, bool MONO>
__global__ void source_dist_rows_kernel(RcArgs A) {
  dist_rows_body<K, MONO ? RC_MONO_SRC : RC_PCD_SRC>(A);
}

// Counts over a DENSE distance matrix (the tensor-core route: cfl_score_topk's dist_out holds the Gram-form
// distance of every (query, row); thresholds taken from the same matrix make the counts self-consistent).
// grid (chunks, Q): each CTA streams a slice of one query's row with 128-bit loads.
constexpr int DRC_THREADS = 256;
template <int JM>
__global__ void __launch_bounds__(DRC_THREADS)
dense_rank_count_kernel(const float* __restrict__ dense, int64_t N, int64_t ldn, const float* __restrict__ thr, int J,
                        unsigned long long* __restrict__ counts) {
  __shared__ float st[JM];
  __shared__ unsigned int sc[JM * 2];
  const int64_t q = blockIdx.y;
  const int t = threadIdx.x;
  if (t < JM) st[t] = t < J ? thr[q * J + t] : __int_as_float(0x7fc00000);   // NaN pads: count nothing
  if (t < 2 * JM) sc[t] = 0u;
  __syncthreads();
  const float* row = dense + q * ldn;
  const int64_t per = (N + gridDim.x - 1) / gridDim.x;
  const int64_t lo = (int64_t)blockIdx.x * per;
  const int64_t hi = lo + per < N ? lo + per : N;
  unsigned int lt[JM], eq[JM];
  float tj[JM];
#pragma unroll
  for (int j = 0; j < JM; ++j) { lt[j] = 0u; eq[j] = 0u; tj[j] = st[j]; }
  for (int64_t i = lo + t; i < hi; i += DRC_THREADS) {
    const float v = row[i];
#pragma unroll
    for (int j = 0; j < JM; ++j) { lt[j] += v < tj[j]; eq[j] += v == tj[j]; }
  }
#pragma unroll
  for (int j = 0; j < JM; ++j) {
    unsigned int a = lt[j], b = eq[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
    if ((t & 31) == 0) { if (a) atomicAdd(&sc[2 * j], a); if (b) atomicAdd(&sc[2 * j + 1], b); }
  }
  __syncthreads();
  if (t < 2 * J && sc[t]) atomicAdd(&counts[q * J * 2 + t], (unsigned long long)sc[t]);
}

static size_t rc_smem_bytes(int K, int d, int J, int role, bool staged = true) {
  const int ew = rc_row_floats(role, K, d), qw = rc_query_floats(role, K, d);
  return (size_t)RC_QT * qw * 4 + (staged ? (size_t)128 * (ew + 1) * 4 : 0) + (size_t)RC_QT * K * 4 +
         (size_t)RC_QT * J * 4 + (size_t)(RC_THREADS / 32) * RC_QT * J * 2 * 4;
}

template <int K, bool MONO, bool SRC>
static int rc_launch(const RcArgs& a, bool gather, const RcEmit* emit, cudaStream_t cs) {
  constexpr int role = SRC ? (MONO ? RC_MONO_SRC : RC_PCD_SRC) : (MONO ? RC_MONO : RC_PCD);
  if (gather) {
    const int64_t n = a.Q * a.J;
    if (SRC) source_dist_rows_kernel<K, MONO><<<(unsigned)((n + 127) / 128), 128, 0, cs>>>(a);
    else pair_dist_rows_kernel<K, MONO><<<(unsigned)((n + 127) / 128), 128, 0, cs>>>(a);
  } else {
    // pcd_source rows of K*d floats: staged while 128 of them fit, read in place beyond (VW = 0)
    const bool staged = rc_smem_bytes(K, a.d, a.J, role) <= RC_SMEM_MAX;
    const size_t smem = rc_smem_bytes(K, a.d, a.J, role, staged);
    const int ea = role == RC_MONO_SRC ? a.d : rc_row_floats(role, K, a.d);
    const bool v4 = ea % 4 == 0 && a.lde % 4 == 0 && ((uintptr_t)a.E & 15u) == 0;
    void (*kern)(RcArgs);
    void (*ekern)(RcArgs, RcEmit);
    if constexpr (!SRC) {
      kern = v4 ? rank_count_kernel<K, MONO, 4> : rank_count_kernel<K, MONO, 1>;
      ekern = v4 ? within_emit_kernel<K, MONO, 4> : within_emit_kernel<K, MONO, 1>;
    } else if constexpr (MONO) {                               // d + K floats per row: always staged
      kern = v4 ? rank_count_src_kernel<K, true, 4> : rank_count_src_kernel<K, true, 1>;
      ekern = v4 ? within_emit_src_kernel<K, true, 4> : within_emit_src_kernel<K, true, 1>;
    } else {
      kern = !staged ? rank_count_src_kernel<K, false, 0>
                     : v4 ? rank_count_src_kernel<K, false, 4> : rank_count_src_kernel<K, false, 1>;
      ekern = !staged ? within_emit_src_kernel<K, false, 0>
                      : v4 ? within_emit_src_kernel<K, false, 4> : within_emit_src_kernel<K, false, 1>;
    }
    // one wave: as many catalog parts as keep every CTA resident at once (only resident warps hide the
    // shared-memory latency; a partial second wave idles most SMs)
    int resident = 0;
    if (emit) {
      CFL_CUDA(cudaFuncSetAttribute(ekern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      CFL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, ekern, RC_THREADS, smem));
    } else {
      CFL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      CFL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, kern, RC_THREADS, smem));
    }
    if (resident < 1) resident = 1;
    int sms = sm_count();
    if (sms <= 0) sms = 148;
    const int64_t nqt = (a.Q + RC_QT - 1) / RC_QT;
    int64_t parts = ((int64_t)resident * sms) / nqt;
    if (parts > a.tiles) parts = a.tiles;
    if (parts < 1) parts = 1;
    RcArgs b = a;
    b.parts = (int)parts;
    dim3 grid((unsigned)parts, (unsigned)nqt);
    if (emit) ekern<<<grid, RC_THREADS, smem, cs>>>(b, *emit);
    else kern<<<grid, RC_THREADS, smem, cs>>>(b);
  }
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

static int rc_dispatch(const RcArgs& a, bool gather, cudaStream_t cs, const RcEmit* emit = nullptr) {
  const int role = rc_role(a.mode);
#define CFL_RC_CASE(KK)                                                       \
  case KK:                                                                    \
    switch (role) {                                                           \
      case RC_MONO: return rc_launch<KK, true, false>(a, gather, emit, cs);   \
      case RC_PCD_SRC: return rc_launch<KK, false, true>(a, gather, emit, cs); \
      case RC_MONO_SRC: return rc_launch<KK, true, true>(a, gather, emit, cs); \
      default: return rc_launch<KK, false, false>(a, gather, emit, cs);       \
    }
  switch (a.K) {
    CFL_RC_CASE(1) CFL_RC_CASE(2) CFL_RC_CASE(3) CFL_RC_CASE(4)
    CFL_RC_CASE(5) CFL_RC_CASE(6) CFL_RC_CASE(7) CFL_RC_CASE(8)
  }
#undef CFL_RC_CASE
  return CFL_ERR_UNSUPPORTED;
}

static int rc_check(const char* what, int mode, const float* Pq, int64_t Q, int K, int d, int64_t ldq, const float* Wq,
                    const float* E, int64_t N, int64_t lde, int J) {
  CFL_REQUIRE(mode >= CFL_PCD && mode <= CFL_MONOMER_SOURCE, CFL_ERR_INVALID, "%s: bad mode %d", what, mode);
  CFL_REQUIRE(mode != CFL_SIAMESE || K == 1, CFL_ERR_INVALID, "%s: siamese needs K=1", what);
  CFL_REQUIRE(K >= 1 && K <= CFL_MAX_K, CFL_ERR_UNSUPPORTED, "%s: K=%d outside [1,%d]", what, K, CFL_MAX_K);
  CFL_REQUIRE(d >= 1 && d <= 128, CFL_ERR_UNSUPPORTED, "%s: d=%d outside [1,128]", what, d);
  CFL_REQUIRE(J >= 1 && J <= RC_MAX_J, CFL_ERR_UNSUPPORTED, "%s: J=%d outside [1,%d]", what, J, RC_MAX_J);
  CFL_REQUIRE(Q >= 0 && N >= 0, CFL_ERR_INVALID, "%s: bad Q/N", what);
  const int role = rc_role(mode);
  const int64_t ldq_min = rc_query_floats(role, K, d), lde_min = role == RC_MONO_SRC ? d : rc_row_floats(role, K, d);
  CFL_REQUIRE(ldq >= ldq_min && lde >= lde_min, CFL_ERR_INVALID, "%s: leading dimension too small", what);
  CFL_REQUIRE(Q == 0 || (Pq && (role != RC_MONO || Wq)), CFL_ERR_INVALID, "%s: NULL query argument", what);
  CFL_REQUIRE(Q == 0 || N == 0 || (E && (role != RC_MONO_SRC || Wq)), CFL_ERR_INVALID, "%s: NULL catalog", what);
  // the tile of a monomer catalog (K*d floats per row) must fit the shared memory of one CTA
  CFL_REQUIRE(role != RC_MONO || rc_smem_bytes(K, d, J, role) <= RC_SMEM_MAX, CFL_ERR_UNSUPPORTED,
              "%s: K*d = %d too large for the monomer rank-count tile", what, K * d);
  return CFL_OK;
}

int rank_counts_only_launch(int mode, const float* Pq, int64_t Q, int K, int d, int64_t ldq, const float* E, int64_t N,
                            int64_t lde, const float* pos_dist, int J, unsigned long long* counts, const int* only,
                            cudaStream_t st) {
  RcArgs a = {};
  a.mode = mode; a.K = K; a.d = d; a.J = J; a.Q = Q; a.N = N; a.ldq = ldq; a.lde = lde;
  a.Pq = Pq; a.E = E; a.thr = pos_dist; a.counts = counts; a.only = only;
  a.tiles = (N + 127) / 128;
  a.parts = 1;
  return rc_dispatch(a, false, st);
}

int within_emit_launch(int mode, const float* Pq, int64_t Q, int K, int d, int64_t ldq, const float* Wq, const float* E,
                       int64_t N, int64_t lde, const float* radius, const int64_t* offsets, unsigned int* cursor,
                       int64_t* out, const int* only, cudaStream_t st) {
  RcArgs a = {};
  a.mode = mode; a.K = K; a.d = d; a.J = 1; a.Q = Q; a.N = N; a.ldq = ldq; a.lde = lde;
  a.Pq = Pq; a.Wq = Wq; a.E = E; a.thr = radius; a.only = only;
  a.tiles = (N + 127) / 128;
  a.parts = 1;
  const RcEmit x = {offsets, cursor, out};
  return rc_dispatch(a, false, st, &x);
}

}  // namespace cfl

using namespace cfl;

extern "C" {

int cfl_pair_dist_rows(int mode, const float* Pq, int64_t Q, int K, int d, int64_t ldq, const float* Wq,
                       const float* E, int64_t N, int64_t lde, const int64_t* pos_idx, int J,
                       float* pos_dist, void* stream) {
  int st = device_check();
  if (st != CFL_OK) return st;
  st = rc_check("pair_dist_rows", mode, Pq, Q, K, d, ldq, Wq, E, N, lde, J);
  if (st != CFL_OK) return st;
  if (Q == 0) return CFL_OK;
  CFL_REQUIRE(pos_idx && pos_dist, CFL_ERR_INVALID, "pair_dist_rows: NULL argument");
  RcArgs a = {};
  a.mode = mode; a.K = K; a.d = d; a.J = J; a.Q = Q; a.N = N; a.ldq = ldq; a.lde = lde;
  a.Pq = Pq; a.Wq = Wq; a.E = E; a.pos_idx = pos_idx; a.pos_dist = pos_dist;
  return rc_dispatch(a, true, (cudaStream_t)stream);
}

int cfl_rank_counts(int mode, const float* Pq, int64_t Q, int K, int d, int64_t ldq, const float* Wq,
                    const float* E, int64_t N, int64_t lde, const float* pos_dist, int J,
                    int64_t* counts, void* stream) {
  int st = device_check();
  if (st != CFL_OK) return st;
  st = rc_check("rank_counts", mode, Pq, Q, K, d, ldq, Wq, E, N, lde, J);
  if (st != CFL_OK) return st;
  if (Q == 0) return CFL_OK;
  CFL_REQUIRE(pos_dist && counts, CFL_ERR_INVALID, "rank_counts: NULL argument");
  cudaStream_t cs = (cudaStream_t)stream;
  CFL_CUDA(cudaMemsetAsync(counts, 0, (size_t)Q * J * 2 * sizeof(int64_t), cs));
  if (N == 0) return CFL_OK;
  RcArgs a = {};
  a.mode = mode; a.K = K; a.d = d; a.J = J; a.Q = Q; a.N = N; a.ldq = ldq; a.lde = lde;
  a.Pq = Pq; a.Wq = Wq; a.E = E; a.thr = pos_dist; a.counts = (unsigned long long*)counts;
  a.tiles = (N + 127) / 128;
  a.parts = 1;                                   // set per kernel instance in rc_launch (one wave)
  return rc_dispatch(a, false, cs);
}

int cfl_dense_rank_counts(const float* dense, int64_t Q, int64_t N, int64_t ldn, const float* pos_dist, int J,
                          int64_t* counts, void* stream) {
  int st = device_check();
  if (st != CFL_OK) return st;
  CFL_REQUIRE(J >= 1 && J <= RC_MAX_J, CFL_ERR_UNSUPPORTED, "dense_rank_counts: J=%d outside [1,%d]", J, RC_MAX_J);
  CFL_REQUIRE(Q >= 0 && N >= 0 && ldn >= N && Q <= 65535, CFL_ERR_INVALID, "dense_rank_counts: bad Q/N/ldn");
  if (Q == 0) return CFL_OK;
  CFL_REQUIRE(pos_dist && counts && (N == 0 || dense), CFL_ERR_INVALID, "dense_rank_counts: NULL argument");
  cudaStream_t cs = (cudaStream_t)stream;
  CFL_CUDA(cudaMemsetAsync(counts, 0, (size_t)Q * J * 2 * sizeof(int64_t), cs));
  if (N == 0) return CFL_OK;
  int sms = sm_count();
  if (sms <= 0) sms = 148;
  int64_t chunks = (8 * (int64_t)sms + Q - 1) / Q;                 // ~8 CTAs per SM in flight
  const int64_t max_chunks = (N + 4 * DRC_THREADS - 1) / (4 * DRC_THREADS);
  if (chunks > max_chunks) chunks = max_chunks;
  if (chunks < 1) chunks = 1;
  dim3 grid((unsigned)chunks, (unsigned)Q);
  unsigned long long* c64 = (unsigned long long*)counts;
  if (J <= 8) dense_rank_count_kernel<8><<<grid, DRC_THREADS, 0, cs>>>(dense, N, ldn, pos_dist, J, c64);
  else if (J <= 16) dense_rank_count_kernel<16><<<grid, DRC_THREADS, 0, cs>>>(dense, N, ldn, pos_dist, J, c64);
  else dense_rank_count_kernel<32><<<grid, DRC_THREADS, 0, cs>>>(dense, N, ldn, pos_dist, J, c64);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

}  // extern "C"
