// Catalog range queries (cfl_score_within): every catalog row c with dist(q, c) < r_q, exact, as CSR lists ordered by
// (distance, index).  "Compatible" in the Thresholder's sense (cfl/models/blocks.py:21-22, the accuracy counts of
// cfl/utils.py:247,264) is r = max(theta, 1e-6): the score r - dist is > 0 exactly when dist < r.
//
// The caller has counted every query's result (cfl_rank_counts_packed / cfl_rank_counts with pos_dist = r, J = 1) and
// laid out the segments: offsets[q] .. offsets[q + 1] of out_idx / out_dist.  This file runs the rest:
//   1. emit   -- the local rows of every segment, in no particular order (rank_counts_tc.cu: the tensor-core scoring
//               epilogue, sure rows at once, band rows after the direct-form check; rank_counts.cu: the CUDA-core kernel
//               for monomer catalogs, shapes without a tcgen05 tiling and queries whose band records overflowed);
//   2. rescore -- every emitted row's distance in the fp32 direct form of direct.cuh (the bits cfl_pair_dist_rows
//               returns), written in place as the key (orderable(dist) << 32) | row;
//   3. finish  -- one CTA per query sorts its keys (bitonic; in shared memory up to WN_BIG keys, in place in global
//               memory beyond) and writes idx_base + row and the distance.
// The emitted rows and then the keys live in out_idx until the finish overwrites them: nothing is allocated.
// cfl_within_merge merges the per-rank lists of a sharded catalog (rank-based placement, as cfl_topk_merge).
#include "score.cuh"
#include "direct.cuh"

namespace cfl {

constexpr int WR_THREADS = 128;           // rescore: one element per thread, 32 rows staged per warp
constexpr int WN_SMALL = 1024, WN_SMALL_THREADS = 256;
constexpr int WN_BIG = 16384, WN_BIG_THREADS = 1024;     // 128 KB of keys in shared memory

// largest q with offsets[q] <= i (offsets non-decreasing, offsets[0] <= i < offsets[Q])
__device__ __forceinline__ int64_t seg_of(const int64_t* __restrict__ offsets, int64_t Q, int64_t i) {
  int64_t lo = 0, hi = Q;                 // invariant: offsets[lo] <= i < offsets[hi]
  while (hi - lo > 1) {
    const int64_t mid = (lo + hi) >> 1;
    if (offsets[mid] <= i) lo = mid; else hi = mid;
  }
  return lo;
}

// SRC (pcd_source / monomer_source): the direct form with the roles swapped, the accessors of merge_rescore_src_kernel
// (score.cu) and mono_rescore_src_kernel (score_monomer_tc.cu), so the bits are those cfl_score_topk_source /
// _monomer_source report.  STAGED: the warp gathers its rows into shared memory (every forward call; pcd_source while
// 128 rows of K*d floats fit); otherwise each thread reads its row in place (monomer_source: d + K floats).
template <int K, bool MONO, bool SRC, bool STAGED>
__device__ __forceinline__ void within_rescore_body(const float* __restrict__ Pq, int64_t ldq, const float* __restrict__ Wq,
                                                    const float* __restrict__ E, int64_t lde, int64_t N, int d, int64_t Q,
                                                    const int64_t* __restrict__ offsets,
                                                    const unsigned int* __restrict__ cursor, int64_t* __restrict__ out) {
  extern __shared__ __align__(16) float wr_smem[];
  const int ew = MONO || SRC ? K * d : d, lder = ew + 1;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int64_t begin = offsets[0], end = offsets[Q];
  for (int64_t c0 = begin + (int64_t)blockIdx.x * WR_THREADS; c0 < end; c0 += (int64_t)gridDim.x * WR_THREADS) {
    const int64_t i = c0 + tid;
    int64_t q = 0, row = 0;
    bool live = false;
    if (i < end) {
      q = seg_of(offsets, Q, i);
      live = i - offsets[q] < (int64_t)cursor[q];          // an unfilled slot (count mismatch) stays a dead key
      if (live) {
        row = out[i];
        live = row >= 0 && row < N;
      }
    }
    if constexpr (STAGED) {
    __syncwarp();
    for (int rr = 0; rr < 32; ++rr) {                      // the warp gathers its 32 rows with coalesced loads
      const int64_t rw = __shfl_sync(0xffffffffu, row, rr);
      if (!__shfl_sync(0xffffffffu, live ? 1 : 0, rr)) continue;      // warp-uniform
      float* dst = wr_smem + (wid * 32 + rr) * lder;
      for (int j = lane; j < ew; j += 32) dst[j] = E[rw * lde + j];
    }
    __syncwarp();
    }
    if (i >= end) continue;
    unsigned long long key = CFL_KEY_INF;
    if (live) {
      const float* ev = STAGED ? wr_smem + tid * lder : E + row * lde;
      const float* qv = Pq + q * ldq;
      float dist;
      if (SRC && MONO) {                                   // e = the query's prototypes, a / w = the row's
        const float* wv = Wq + row * K;
        dist = monomer_direct<K>([&](int k, int j) { return qv[k * d + j]; }, [&](int j) { return ev[j]; },
                                 [&](int k) { return wv[k]; }, d);
      } else if (SRC) {                                    // e = the query row, p = the row's prototypes (shared when STAGED)
        dist = pcd_direct<K, 1>([&](int j) { return qv[j]; }, [&](int k, int j) { return ev[k * d + j]; }, d);
      } else if (MONO) {
        const float* wv = Wq + q * K;
        dist = monomer_direct<K>([&](int k, int j) { return ev[k * d + j]; }, [&](int j) { return qv[j]; },
                                 [&](int k) { return wv[k]; }, d);
      } else {
        dist = pcd_direct<K>([&](int j) { return ev[j]; }, [&](int k, int j) { return qv[k * d + j]; }, d);
      }
      key = pack_key(dist, (uint32_t)row);
    }
    out[i] = (int64_t)key;
  }
}

template <int K, bool MONO>
__global__ void __launch_bounds__(WR_THREADS)
within_rescore_kernel(const float* __restrict__ Pq, int64_t ldq, const float* __restrict__ Wq,
                      const float* __restrict__ E, int64_t lde, int64_t N, int d, int64_t Q,
                      const int64_t* __restrict__ offsets, const unsigned int* __restrict__ cursor,
                      int64_t* __restrict__ out) {
  within_rescore_body<K, MONO, false, true>(Pq, ldq, Wq, E, lde, N, d, Q, offsets, cursor, out);
}

template <int K, bool MONO, bool STAGED>
__global__ void __launch_bounds__(WR_THREADS)
within_rescore_src_kernel(const float* __restrict__ Pq, int64_t ldq, const float* __restrict__ Wq,
                          const float* __restrict__ E, int64_t lde, int64_t N, int d, int64_t Q,
                          const int64_t* __restrict__ offsets, const unsigned int* __restrict__ cursor,
                          int64_t* __restrict__ out) {
  within_rescore_body<K, MONO, true, STAGED>(Pq, ldq, Wq, E, lde, N, d, Q, offsets, cursor, out);
}

// Ascending sort of s[0, n) by NT threads; positions n .. P-1 (P = next power of two) act as +inf keys that are never
// touched.  Bitonic network in the form whose every comparator puts the smaller key first (the first step of a merge
// compares mirrored positions), so a comparator with its upper end beyond n is a no-op.  s may be shared or global.
template <int NT>
__device__ __forceinline__ void sort_keys(unsigned long long* s, int64_t n, int tid) {
  int64_t P = 1;
  while (P < n) P <<= 1;
  for (int64_t size = 2; size <= P; size <<= 1) {
    const int64_t half = size >> 1;
    for (int64_t c = tid; c < P / 2; c += NT) {
      const int64_t base = (c / half) * size, off = c % half;
      const int64_t i = base + off, j = base + size - 1 - off;
      if (j < n) {
        const unsigned long long a = s[i], b = s[j];
        if (a > b) { s[i] = b; s[j] = a; }
      }
    }
    __syncthreads();
    for (int64_t stride = half >> 1; stride > 0; stride >>= 1) {
      for (int64_t c = tid; c < P / 2; c += NT) {
        const int64_t i = ((c & ~(stride - 1)) << 1) | (c & (stride - 1));
        const int64_t j = i + stride;
        if (j < n) {
          const unsigned long long a = s[i], b = s[j];
          if (a > b) { s[i] = b; s[j] = a; }
        }
      }
      __syncthreads();
    }
  }
}

// One CTA per query whose result size n lies in (n_lo, n_hi].  stats[4] counts the queries whose emitting pass did not
// append exactly n rows (must stay 0: the verdicts of the count and of the emission are the same arithmetic).
template <int CAP, int NT>
__global__ void __launch_bounds__(NT)
within_finish_kernel(const int64_t* __restrict__ offsets, const unsigned int* __restrict__ cursor, int64_t n_lo,
                     int64_t n_hi, int64_t idx_base, int64_t* __restrict__ out_idx, float* __restrict__ out_dist,
                     unsigned long long* __restrict__ stats) {
  extern __shared__ __align__(16) unsigned long long wn_keys[];
  const int64_t q = blockIdx.x;
  const int64_t b = offsets[q], n = offsets[q + 1] - b;
  if (n <= n_lo || n > n_hi) return;
  const int tid = threadIdx.x;
  if (tid == 0 && (int64_t)cursor[q] != n) atomicAdd(&stats[4], 1ull);
  unsigned long long* seg = (unsigned long long*)(out_idx + b);
  unsigned long long* s = seg;
  if (n <= CAP) {
    s = wn_keys;
    for (int64_t i = tid; i < n; i += NT) s[i] = seg[i];
    __syncthreads();
  }
  sort_keys<NT>(s, n, tid);
  for (int64_t i = tid; i < n; i += NT) {
    const unsigned long long key = s[i];
    const bool ok = key != CFL_KEY_INF;
    out_idx[b + i] = ok ? idx_base + (int64_t)(key & 0xffffffffull) : -1;
    out_dist[b + i] = ok ? ord2f((uint32_t)(key >> 32)) : __int_as_float(0x7fc00000);
  }
}

// Sharded merge: element i of rank r's list of query q lands at out_offsets[q] + (its position in its own list) + (the
// number of smaller (distance, index) entries in every other rank's list of q, by binary search).  Global indices are
// unique, so the positions form a permutation and the result does not depend on the rank count.
__device__ __forceinline__ bool key_less(float da, int64_t ia, float db, int64_t ib) {
  const uint32_t a = f2ord(da), b = f2ord(db);
  return a < b || (a == b && ia < ib);
}

__global__ void within_merge_kernel(const int64_t* __restrict__ offs, const int64_t* __restrict__ idx,
                                    const float* __restrict__ dist, int64_t ld, int R, int64_t Q,
                                    const int64_t* __restrict__ out_offsets, int64_t* __restrict__ out_idx,
                                    float* __restrict__ out_dist) {
  const int64_t total = (int64_t)R * ld;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int r = (int)(e / ld);
    const int64_t i = e - (int64_t)r * ld;
    const int64_t* o = offs + (int64_t)r * (Q + 1);
    if (i < o[0] || i >= o[Q]) continue;
    const int64_t q = seg_of(o, Q, i);
    const float dv = dist[e];
    const int64_t iv = idx[e];
    int64_t pos = out_offsets[q] + (i - o[q]);
    for (int r2 = 0; r2 < R; ++r2) {
      if (r2 == r) continue;
      const int64_t* o2 = offs + (int64_t)r2 * (Q + 1);
      const float* d2 = dist + (int64_t)r2 * ld;
      const int64_t* i2 = idx + (int64_t)r2 * ld;
      int64_t lo = o2[q], hi = o2[q + 1];               // first entry not smaller than (dv, iv)
      const int64_t start = lo;
      while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (key_less(d2[mid], i2[mid], dv, iv)) lo = mid + 1; else hi = mid;
      }
      pos += lo - start;
    }
    out_idx[pos] = iv;
    out_dist[pos] = dv;
  }
}

struct WsLayout { size_t stats, cursor, tc, total; };
static WsLayout within_ws(int mode, int64_t Q, int K, int d, int64_t N) {
  WsLayout w;
  size_t off = 0;
  w.stats = off;  off = align_up(off + CFL_WITHIN_NSTATS * sizeof(unsigned long long), 256);
  w.cursor = off; off = align_up(off + (size_t)(Q > 0 ? Q : 0) * sizeof(unsigned int), 1024);
  w.tc = off;
  if (mode == CFL_PCD_SOURCE && Q > 0 && N > 0) off += within_tc_workspace_bytes(Q, K, d, N, true);
  else if ((mode == CFL_PCD || mode == CFL_SIAMESE) && Q > 0 && N > 0 && score_umma_supported(K, d))
    off += within_tc_workspace_bytes(Q, K, d, N, false);
  w.total = off;
  return w;
}

template <int K, bool MONO, bool SRC>
static int within_rescore_launch(const float* Pq, int64_t ldq, const float* Wq, const float* E, int64_t lde, int64_t N,
                                 int d, int64_t Q, const int64_t* offsets, const unsigned int* cursor, int64_t* out,
                                 cudaStream_t cs) {
  int sms = sm_count();
  if (sms <= 0) sms = 148;
  if constexpr (SRC) {
    const size_t smem = (size_t)WR_THREADS * (K * d + 1) * sizeof(float);
    if (!MONO && smem <= 200 * 1024) {
      CFL_SMEM_LIMIT((within_rescore_src_kernel<K, false, true>), smem);
      within_rescore_src_kernel<K, false, true><<<(unsigned)(sms * 8), WR_THREADS, smem, cs>>>(Pq, ldq, Wq, E, lde, N, d,
                                                                                             Q, offsets, cursor, out);
    } else {
      within_rescore_src_kernel<K, MONO, false><<<(unsigned)(sms * 8), WR_THREADS, 0, cs>>>(Pq, ldq, Wq, E, lde, N, d, Q,
                                                                                          offsets, cursor, out);
    }
  } else {
    const size_t smem = (size_t)WR_THREADS * ((MONO ? K * d : d) + 1) * sizeof(float);
    CFL_SMEM_LIMIT((within_rescore_kernel<K, MONO>), smem);
    within_rescore_kernel<K, MONO><<<(unsigned)(sms * 8), WR_THREADS, smem, cs>>>(Pq, ldq, Wq, E, lde, N, d, Q, offsets,
                                                                               cursor, out);
  }
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

}  // namespace cfl

using namespace cfl;

extern "C" {

size_t cfl_score_within_workspace_bytes(int mode, int64_t Q, int K, int d, int64_t N) {
  if (K < 1 || K > CFL_MAX_K || d < 1 || d > 128) return 4096;
  return within_ws(mode, Q, K, d, N).total;
}

int cfl_score_within(int mode, const float* Pq, int64_t Q, int K, int d, int64_t ldq, const float* Wq, const float* E,
                     const void* image, int64_t N, int64_t lde, const float* mu, const float* radius,
                     const int64_t* offsets, int64_t idx_base, int64_t* out_idx, float* out_dist, void* ws,
                     size_t ws_bytes, void* stream) {
  int st = device_check();
  if (st != CFL_OK) return st;
  CFL_REQUIRE(mode >= CFL_PCD && mode <= CFL_MONOMER_SOURCE, CFL_ERR_INVALID, "score_within: bad mode %d", mode);
  CFL_REQUIRE(mode != CFL_SIAMESE || K == 1, CFL_ERR_INVALID, "score_within: siamese needs K=1");
  CFL_REQUIRE(K >= 1 && K <= CFL_MAX_K, CFL_ERR_UNSUPPORTED, "score_within: K=%d outside [1,%d]", K, CFL_MAX_K);
  CFL_REQUIRE(d >= 1 && d <= 128, CFL_ERR_UNSUPPORTED, "score_within: d=%d outside [1,128]", d);
  CFL_REQUIRE(Q >= 0 && N >= 0 && N < ((int64_t)1 << 32) && Q < ((int64_t)1 << 31), CFL_ERR_INVALID,
              "score_within: bad Q/N");
  const bool mono = mode == CFL_MONOMER, msrc = mode == CFL_MONOMER_SOURCE, src = mode == CFL_PCD_SOURCE || msrc;
  // per query: K*d floats (pcd, monomer_source) or d (monomer, pcd_source); per row: the other one
  const bool qd = mono || mode == CFL_PCD_SOURCE;
  CFL_REQUIRE(ldq >= (qd ? d : (int64_t)K * d) && lde >= (qd ? (int64_t)K * d : d), CFL_ERR_INVALID,
              "score_within: leading dimension too small");
  CFL_REQUIRE(!(mono || msrc) || image == nullptr, CFL_ERR_UNSUPPORTED,
              "score_within: monomer runs on the CUDA cores (image NULL)");
  CFL_REQUIRE(!mono || (size_t)(128 * (K * d + 1) + 9 * d + 8 * K + 72) * 4 <= 200 * 1024, CFL_ERR_UNSUPPORTED,
              "score_within: K*d = %d too large for the monomer tile", K * d);
  CFL_REQUIRE(mode != CFL_PCD_SOURCE || ((uintptr_t)image & 1023u) == 0, CFL_ERR_INVALID,
              "score_within: image must be 1024-byte aligned");
  if (Q == 0) return CFL_OK;
  CFL_REQUIRE(Pq && radius && offsets && (!(mono || msrc) || Wq) && (N == 0 || E), CFL_ERR_INVALID,
              "score_within: NULL argument");
  const WsLayout w = within_ws(mode, Q, K, d, N);
  CFL_REQUIRE(ws && ws_bytes >= w.total, CFL_ERR_WORKSPACE, "score_within: workspace too small (%zu < %zu)", ws_bytes,
              w.total);
  cudaStream_t cs = (cudaStream_t)stream;
  char* base = (char*)ws;
  unsigned long long* stats = (unsigned long long*)(base + w.stats);
  unsigned int* cursor = (unsigned int*)(base + w.cursor);
  CFL_CUDA(cudaMemsetAsync(stats, 0, CFL_WITHIN_NSTATS * sizeof(unsigned long long), cs));
  CFL_CUDA(cudaMemsetAsync(cursor, 0, (size_t)Q * sizeof(unsigned int), cs));
  if (N > 0) {
    CFL_REQUIRE(out_idx && out_dist, CFL_ERR_INVALID, "score_within: NULL output");
    if (image != nullptr) {
      st = within_tc_emit(mode, Pq, Q, K, d, ldq, E, image, N, lde, mu, radius, offsets, cursor, out_idx, base + w.tc,
                          stats, cs);
    } else {
      st = within_emit_launch(mode, Pq, Q, K, d, ldq, Wq, E, N, lde, radius, offsets, cursor, out_idx, nullptr, cs);
    }
    if (st != CFL_OK) return st;
#define CFL_WR_CASE(KK)                                                                                              \
  case KK:                                                                                                           \
    st = src ? (msrc ? within_rescore_launch<KK, true, true>(Pq, ldq, Wq, E, lde, N, d, Q, offsets, cursor, out_idx, cs) \
                     : within_rescore_launch<KK, false, true>(Pq, ldq, Wq, E, lde, N, d, Q, offsets, cursor, out_idx, cs)) \
             : mono ? within_rescore_launch<KK, true, false>(Pq, ldq, Wq, E, lde, N, d, Q, offsets, cursor, out_idx, cs)  \
                    : within_rescore_launch<KK, false, false>(Pq, ldq, Wq, E, lde, N, d, Q, offsets, cursor, out_idx, cs); \
    break;
    switch (K) {
      CFL_WR_CASE(1) CFL_WR_CASE(2) CFL_WR_CASE(3) CFL_WR_CASE(4)
      CFL_WR_CASE(5) CFL_WR_CASE(6) CFL_WR_CASE(7) CFL_WR_CASE(8)
    }
#undef CFL_WR_CASE
    if (st != CFL_OK) return st;
  }
  // two finish launches: small segments at high occupancy, large ones with 1024 threads (global memory beyond WN_BIG)
  CFL_SMEM_LIMIT((within_finish_kernel<WN_BIG, WN_BIG_THREADS>), WN_BIG * sizeof(unsigned long long));
  within_finish_kernel<WN_SMALL, WN_SMALL_THREADS><<<(unsigned)Q, WN_SMALL_THREADS, WN_SMALL * sizeof(unsigned long long),
                                                     cs>>>(offsets, cursor, -1, WN_SMALL, idx_base, out_idx, out_dist,
                                                           stats);
  CFL_LAUNCH_CHECK();
  within_finish_kernel<WN_BIG, WN_BIG_THREADS><<<(unsigned)Q, WN_BIG_THREADS, WN_BIG * sizeof(unsigned long long), cs>>>(
      offsets, cursor, WN_SMALL, INT64_MAX, idx_base, out_idx, out_dist, stats);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

int cfl_score_within_stats(const void* ws, size_t ws_bytes, int64_t* out, void* stream) {
  int st = device_check();
  if (st != CFL_OK) return st;
  CFL_REQUIRE(out && ws && ws_bytes >= CFL_WITHIN_NSTATS * sizeof(int64_t), CFL_ERR_INVALID,
              "score_within_stats: bad argument");
  cudaStream_t cs = (cudaStream_t)stream;
  CFL_CUDA(cudaMemcpyAsync(out, ws, CFL_WITHIN_NSTATS * sizeof(int64_t), cudaMemcpyDeviceToHost, cs));
  CFL_CUDA(cudaStreamSynchronize(cs));
  return CFL_OK;
}

int cfl_within_merge(const int64_t* offsets, const int64_t* idx, const float* dist, int64_t ld, int R, int64_t Q,
                     const int64_t* out_offsets, int64_t* out_idx, float* out_dist, void* stream) {
  int st = device_check();
  if (st != CFL_OK) return st;
  CFL_REQUIRE(R >= 1 && Q >= 0 && ld >= 0, CFL_ERR_INVALID, "within_merge: bad R/Q/ld");
  if (Q == 0 || ld == 0) return CFL_OK;
  CFL_REQUIRE(offsets && idx && dist && out_offsets && out_idx && out_dist, CFL_ERR_INVALID, "within_merge: NULL argument");
  int sms = sm_count();
  if (sms <= 0) sms = 148;
  int64_t blocks = ((int64_t)R * ld + 255) / 256;
  if (blocks > (int64_t)sms * 16) blocks = (int64_t)sms * 16;
  within_merge_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(offsets, idx, dist, ld, R, Q, out_offsets,
                                                                          out_idx, out_dist);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

}  // extern "C"
