// Stage 1: projection of item features onto the e0 / prototype heads, forward + backward.
// Replaces fully_connected_weight_norm (cfl/layers.py:80-94) and the plain FC of
// FCEncoder (cfl/models/dist.py:45-65).
//
// Forward:  the GEMM runs on tcgen05 tensor cores as error-compensated 3xTF32
//           (project_umma.cu) whenever the shape fits its tiling (F % 8 == 0, 16-byte aligned
//           rows, N <= 256); the fp32 CUDA-core tile kernel below covers the remaining shapes
//           (tiny / odd F) and is the reference point for the tensor-core kernel's parity test.
// Backward: dV = x^T dpre with the weight-norm column terms (SURVEY App. A.5).  The GEMM runs on tcgen05
//           tensor cores as 3xTF32 (project_bwd_umma.cu) for B >= 256 and N <= 256; the fp32 CUDA-core
//           kernel below covers the rest.  Both split the batch into slabs reduced in a fixed order
//           (deterministic).
#include "common.cuh"

namespace cfl {

int project_fwd_umma(const float* x, int64_t B, int F, int64_t ldx, const float* V, int N,
                     int64_t ldV, const float* scaler, const float* bias, float in_scale, int act,
                     float* y, int64_t ldy, float* pre, float* z, void* ws, size_t ws_bytes,
                     cudaStream_t st);                       // project_umma.cu
size_t project_fwd_umma_workspace(int64_t B, int F, int N);  // project_umma.cu
bool project_fwd_umma_supported(const float* x, int64_t B, int F, int64_t ldx, int N);
// project_bwd_umma.cu: dV partials on the tensor cores, Cpart[slabs][F][N]
bool project_bwd_umma_supported(int64_t B, int F, int N);
int project_bwd_umma_slabs(int64_t B, int F);
int project_bwd_umma(const float* x, int64_t B, int F, int64_t ldx, const float* dy, int64_t lddy, const float* y,
                     int64_t ldy, int act, int N, float* Cpart, cudaStream_t st);

// ---- column scaler s_j = g_j / |V_:j| ----------------------------------------------------
// one block per 32 columns, 32 row slices per block (four independent accumulators per thread keep four loads in
// flight: the 8-slice version walked F / 8 dependent loads per thread, 16 us at F = 1024 on a handful of CTAs),
// fixed-order reduction over the slices.
constexpr int CN_SLICES = 32;
__global__ void __launch_bounds__(32 * CN_SLICES)
colnorm_kernel(const float* __restrict__ V, int F, int N, int64_t ldV,
               const float* __restrict__ g, float* __restrict__ scaler,
               float* __restrict__ norm_out) {
  __shared__ float sm[CN_SLICES][33];
  int j = blockIdx.x * 32 + threadIdx.x;
  float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
  if (j < N) {
    int i = threadIdx.y;
    for (; i + 3 * CN_SLICES < F; i += 4 * CN_SLICES) {
      const float v0 = V[(int64_t)i * ldV + j], v1 = V[(int64_t)(i + CN_SLICES) * ldV + j];
      const float v2 = V[(int64_t)(i + 2 * CN_SLICES) * ldV + j], v3 = V[(int64_t)(i + 3 * CN_SLICES) * ldV + j];
      a0 = fmaf(v0, v0, a0); a1 = fmaf(v1, v1, a1); a2 = fmaf(v2, v2, a2); a3 = fmaf(v3, v3, a3);
    }
    for (; i < F; i += CN_SLICES) { const float v = V[(int64_t)i * ldV + j]; a0 = fmaf(v, v, a0); }
  }
  sm[threadIdx.y][threadIdx.x] = (a0 + a1) + (a2 + a3);
  __syncthreads();
  if (threadIdx.y == 0 && j < N) {
    float t = 0.0f;
#pragma unroll
    for (int r = 0; r < CN_SLICES; ++r) t += sm[r][threadIdx.x];
    float n = sqrtf(t);                                   // no epsilon: layers.py:81
    if (norm_out) norm_out[j] = n;
    scaler[j] = (g ? g[j] : 1.0f) / n;
  }
}

// ---- fp32 tile GEMM (64x64x16, 4x4 per thread) with the fused epilogue -------------------
constexpr int TM = 64, TN = 64, TK = 16;

template <bool TRANS_A>
__device__ __forceinline__ void tile_mainloop(const float* __restrict__ A, int64_t lda,
                                              const float* __restrict__ Bm, int64_t ldb, int64_t M,
                                              int N, int64_t k0, int64_t k1, int64_t m0, int n0,
                                              float (&acc)[4][4]) {
  // C[m,n] = sum_k A(m,k) * B(k,n);  TRANS_A: A(m,k) stored at A[k*lda + m]
  __shared__ float As[TK][TM + 4];
  __shared__ float Bs[TK][TN + 4];
  const int tid = threadIdx.x;
  const int tx = tid % 16, ty = tid / 16;
  for (int64_t kk = k0; kk < k1; kk += TK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int e = tid + i * 256;
      if (TRANS_A) {
        int k = e / TM, m = e % TM;
        int64_t gk = kk + k, gm = m0 + m;
        As[k][m] = (gk < k1 && gm < M) ? A[gk * lda + gm] : 0.0f;
      } else {
        int m = e / TK, k = e % TK;
        int64_t gk = kk + k, gm = m0 + m;
        As[k][m] = (gk < k1 && gm < M) ? A[gm * lda + gk] : 0.0f;
      }
      int k = e / TN, n = e % TN;
      int64_t gk = kk + k;
      int gn = n0 + n;
      Bs[k][n] = (gk < k1 && gn < N) ? Bm[gk * ldb + gn] : 0.0f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < TK; ++k) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = As[k][ty * 4 + i]; b[i] = Bs[k][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(256)
project_fwd_simt(const float* __restrict__ x, int64_t B, int F, int64_t ldx,
                 const float* __restrict__ V, int N, int64_t ldV,
                 const float* __restrict__ scaler, const float* __restrict__ bias, float in_scale,
                 int act, float* __restrict__ y, int64_t ldy, float* __restrict__ pre,
                 float* __restrict__ z) {
  float acc[4][4] = {};
  int64_t m0 = (int64_t)blockIdx.y * TM;
  int n0 = blockIdx.x * TN;
  tile_mainloop<false>(x, ldx, V, ldV, B, N, 0, F, m0, n0, acc);
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int64_t b = m0 + ty * 4 + i;
    if (b >= B) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int n = n0 + tx * 4 + j;
      if (n >= N) continue;
      float zz = acc[i][j] * in_scale;
      float p = zz * (scaler ? scaler[n] : 1.0f) + (bias ? bias[n] : 0.0f);
      if (z) z[b * ldy + n] = zz;
      if (pre) pre[b * ldy + n] = p;
      y[b * ldy + n] = apply_act(p, act);
    }
  }
}

// Small batches (the reference trains at B = 100): one 128-row tile cannot fill the GPU, and its
// F/8 K-steps would run serially on one SM.  Split the feature dimension over CTAs instead
// (fp32 FFMA partial sums per slice), then reduce the slices in a fixed order with the epilogue.
__global__ void __launch_bounds__(256)
project_fwd_splitk(const float* __restrict__ x, int64_t B, int F, int64_t ldx,
                   const float* __restrict__ V, int N, int64_t ldV, int fslice,
                   float* __restrict__ part) {
  float acc[4][4] = {};
  int64_t m0 = (int64_t)blockIdx.y * TM;
  int n0 = blockIdx.x * TN;
  int64_t k0 = (int64_t)blockIdx.z * fslice;
  int64_t k1 = k0 + fslice; if (k1 > F) k1 = F;
  tile_mainloop<false>(x, ldx, V, ldV, B, N, k0, k1, m0, n0, acc);
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
  float* P = part + (int64_t)blockIdx.z * B * N;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int64_t b = m0 + ty * 4 + i;
    if (b >= B) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int n = n0 + tx * 4 + j;
      if (n < N) P[b * N + n] = acc[i][j];
    }
  }
}
__global__ void project_fwd_splitk_final(const float* __restrict__ part, int slices, int64_t B, int N,
                                         const float* __restrict__ scaler, const float* __restrict__ bias,
                                         float in_scale, int act, float* __restrict__ y, int64_t ldy,
                                         float* __restrict__ pre, float* __restrict__ z) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * N) return;
  int64_t b = i / N; int n = (int)(i % N);
  float a = 0.0f;
  for (int s = 0; s < slices; ++s) a += part[(int64_t)s * B * N + i];
  float zz = a * in_scale;
  float p = zz * (scaler ? scaler[n] : 1.0f) + (bias ? bias[n] : 0.0f);
  if (z) z[b * ldy + n] = zz;
  if (pre) pre[b * ldy + n] = p;
  y[b * ldy + n] = apply_act(p, act);
}

static int splitk_slices(int64_t B, int F, int N, int* fslice) {
  int64_t tiles = ((B + TM - 1) / TM) * ((N + TN - 1) / TN);
  int sms = sm_count(); if (sms <= 0) sms = 148;
  int64_t want = (2 * (int64_t)sms + tiles - 1) / tiles;     // ~2 CTAs per SM
  int64_t maxs = (F + 63) / 64;                              // at least 64 features per slice
  if (want > maxs) want = maxs;
  if (want < 1) want = 1;
  int fs = (int)((F + want - 1) / want);
  fs = (fs + TK - 1) / TK * TK;
  *fslice = fs;
  return (int)((F + fs - 1) / fs);
}
static bool use_splitk(int64_t B) { return B <= 1024; }   // <= 8 tcgen05 tiles would leave 140 SMs idle: split F over ~2 CTAs per SM instead

// ---- backward ----------------------------------------------------------------------------
__device__ __forceinline__ float dpre_of(const float* __restrict__ dy, int64_t lddy,
                                         const float* __restrict__ y, int64_t ldy, int act,
                                         int64_t b, int n) {
  float g = dy[b * lddy + n];
  if (act != CFL_ACT_LINEAR) g *= act_grad_from_y(y[b * ldy + n], act);
  return g;
}

// column statistics per batch slab: q_j = sum_b dpre*z, db_j = sum_b dpre  (double partials)
__global__ void colstats_kernel(const float* __restrict__ dy, int64_t lddy,
                                const float* __restrict__ y, int64_t ldy,
                                const float* __restrict__ z, int act, int64_t B, int N,
                                int64_t rows_per_slab, double* __restrict__ part) {
  __shared__ double sq[8][33], sb[8][33];
  int j = blockIdx.x * 32 + threadIdx.x;
  int64_t r0 = (int64_t)blockIdx.y * rows_per_slab;
  int64_t r1 = r0 + rows_per_slab; if (r1 > B) r1 = B;
  double q = 0.0, db = 0.0;
  if (j < N)
    for (int64_t b = r0 + threadIdx.y; b < r1; b += 8) {
      float g = dpre_of(dy, lddy, y, ldy, act, b, j);
      db += (double)g;
      if (z) q += (double)g * (double)z[b * ldy + j];
    }
  sq[threadIdx.y][threadIdx.x] = q; sb[threadIdx.y][threadIdx.x] = db;
  __syncthreads();
  if (threadIdx.y == 0 && j < N) {
    double tq = 0.0, tb = 0.0;
#pragma unroll
    for (int r = 0; r < 8; ++r) { tq += sq[r][threadIdx.x]; tb += sb[r][threadIdx.x]; }
    part[((int64_t)blockIdx.y * N + j) * 2 + 0] = tq;
    part[((int64_t)blockIdx.y * N + j) * 2 + 1] = tb;
  }
}

__global__ void colstats_final(const double* __restrict__ part, int slabs, int N,
                               const float* __restrict__ norm, const float* __restrict__ bias,
                               int weight_norm, int accumulate, float reg_c,
                               float* __restrict__ qn3, float* __restrict__ dg,
                               float* __restrict__ dbias, const float* __restrict__ g) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= N) return;
  double q = 0.0, db = 0.0;
  for (int s = 0; s < slabs; ++s) { q += part[((int64_t)s * N + j) * 2]; db += part[((int64_t)s * N + j) * 2 + 1]; }
  if (weight_norm) {
    float n = norm[j];
    float gg = g ? g[j] : 1.0f;
    qn3[j] = (float)(gg * q / ((double)n * n * n));        // g q / n^3
    if (dg) dg[j] = (accumulate ? dg[j] : 0.0f) + (float)(q / n);
  }
  if (dbias) dbias[j] = (accumulate ? dbias[j] : 0.0f) + (float)db + (bias ? reg_c * bias[j] : 0.0f);
}

// partial dV over one batch slab: C[f,n] = sum_{b in slab} x[b,f] * dpre[b,n]
__global__ void __launch_bounds__(256)
project_bwd_gemm(const float* __restrict__ x, int64_t B, int F, int64_t ldx,
                 const float* __restrict__ dy, int64_t lddy, const float* __restrict__ y,
                 int64_t ldy, int act, int N, int64_t rows_per_slab, float* __restrict__ Cpart) {
  __shared__ float As[TK][TM + 4];
  __shared__ float Bs[TK][TN + 4];
  float acc[4][4] = {};
  const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
  int64_t f0 = (int64_t)blockIdx.y * TM;
  int n0 = blockIdx.x * TN;
  int64_t k0 = (int64_t)blockIdx.z * rows_per_slab;
  int64_t k1 = k0 + rows_per_slab; if (k1 > B) k1 = B;
  for (int64_t kk = k0; kk < k1; kk += TK) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int e = tid + i * 256;
      int k = e / TM, m = e % TM;
      int64_t gb = kk + k, gf = f0 + m;
      As[k][m] = (gb < k1 && gf < F) ? x[gb * ldx + gf] : 0.0f;
      int n = e % TN;
      int gn = n0 + n;
      Bs[k][n] = (gb < k1 && gn < N) ? dpre_of(dy, lddy, y, ldy, act, gb, gn) : 0.0f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < TK; ++k) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = As[k][ty * 4 + i]; b[i] = Bs[k][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
  float* C = Cpart + (int64_t)blockIdx.z * F * N;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int64_t f = f0 + ty * 4 + i;
    if (f >= F) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int n = n0 + tx * 4 + j;
      if (n < N) C[f * N + n] = acc[i][j];
    }
  }
}

// dV[f,n] (+)= in_scale*s_n*sum_slabs C - V[f,n]*qn3[n] + reg_c*V[f,n]
__global__ void project_bwd_final(const float* __restrict__ Cpart, int slabs, int F, int N,
                                  const float* __restrict__ V, int64_t ldV,
                                  const float* __restrict__ scaler, const float* __restrict__ qn3,
                                  float in_scale, float reg_c, int accumulate,
                                  float* __restrict__ dV) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t total = (int64_t)F * N;
  if (i >= total) return;
  int64_t f = i / N; int n = (int)(i % N);
  float c = 0.0f;
  for (int s = 0; s < slabs; ++s) c += Cpart[(int64_t)s * total + i];
  float v = V[f * ldV + n];
  float r = c * in_scale * (scaler ? scaler[n] : 1.0f) - (qn3 ? v * qn3[n] : 0.0f) + reg_c * v;
  dV[i] = (accumulate ? dV[i] : 0.0f) + r;
}

static int bwd_slabs(int64_t B) {
  int64_t s = (B + 2047) / 2048;
  if (s < 1) s = 1;
  if (s > 16) s = 16;
  return (int)s;
}

}  // namespace cfl

using namespace cfl;

extern "C" {

size_t cfl_project_fwd_workspace_bytes(int64_t B, int F, int N) {
  size_t sk = 0;
  if (use_splitk(B)) { int fs; sk = (size_t)splitk_slices(B, F, N, &fs) * (size_t)B * N * sizeof(float) + 256; }
  size_t um = project_fwd_umma_workspace(B, F, N);
  return align_up((size_t)N * 2 * sizeof(float), 256) + (sk > um ? sk : um) + 512;
}

int cfl_project_fwd(const float* x, int64_t B, int F, int64_t ldx, const float* V, int N,
                    int64_t ldV, const float* g, const float* bias, int weight_norm,
                    float in_scale, int act, float* y, int64_t ldy, float* pre, float* z,
                    void* ws, size_t ws_bytes, void* stream) {
  int st = device_check();
  if (st != CFL_OK) return st;
  CFL_REQUIRE(x && V && y && B >= 0 && F > 0 && N > 0, CFL_ERR_INVALID, "project_fwd: bad arguments");
  CFL_REQUIRE(ldx >= F && ldV >= N && ldy >= N, CFL_ERR_INVALID, "project_fwd: leading dimension too small");
  CFL_REQUIRE(act >= CFL_ACT_LINEAR && act <= CFL_ACT_LRELU, CFL_ERR_INVALID, "project_fwd: bad act %d", act);
  CFL_REQUIRE(ws && ws_bytes >= cfl_project_fwd_workspace_bytes(B, F, N), CFL_ERR_WORKSPACE,
              "project_fwd: workspace too small");
  if (B == 0) return CFL_OK;
  cudaStream_t cs = (cudaStream_t)stream;
  Workspace W(ws, ws_bytes);
  float* scaler = nullptr;
  if (weight_norm) {
    scaler = W.take<float>(N);
    colnorm_kernel<<<(N + 31) / 32, dim3(32, CN_SLICES), 0, cs>>>(V, F, N, ldV, g, scaler, nullptr);
    CFL_LAUNCH_CHECK();
  }
  if (use_splitk(B)) {
    int fs;
    const int slices = splitk_slices(B, F, N, &fs);
    W.off = align_up(W.off, 256);
    float* part = (float*)(W.base + W.off);
    dim3 grid((N + TN - 1) / TN, (unsigned)((B + TM - 1) / TM), slices);
    project_fwd_splitk<<<grid, 256, 0, cs>>>(x, B, F, ldx, V, N, ldV, fs, part);
    CFL_LAUNCH_CHECK();
    const int64_t total = B * N;
    project_fwd_splitk_final<<<(unsigned)((total + 255) / 256), 256, 0, cs>>>(part, slices, B, N, scaler, bias,
                                                                         in_scale, act, y, ldy, pre, z);
    CFL_LAUNCH_CHECK();
    return CFL_OK;
  }
  if (project_fwd_umma_supported(x, B, F, ldx, N)) {
    W.off = align_up(W.off, 256);
    return project_fwd_umma(x, B, F, ldx, V, N, ldV, scaler, bias, in_scale, act, y, ldy, pre, z,
                            W.base + W.off, W.size - W.off, cs);
  }
  dim3 grid((N + TN - 1) / TN, (unsigned)((B + TM - 1) / TM));
  project_fwd_simt<<<grid, 256, 0, cs>>>(x, B, F, ldx, V, N, ldV, scaler, bias, in_scale, act, y,
                                         ldy, pre, z);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

size_t cfl_project_bwd_workspace_bytes(int64_t B, int F, int N) {
  int slabs = bwd_slabs(B);
  int gslabs = slabs;                                      // the tensor-core dV GEMM cuts the batch its own way
  if (project_bwd_umma_supported(B, F, N)) gslabs = project_bwd_umma_slabs(B, F);
  return align_up((size_t)N * 3 * sizeof(float), 256) +
         align_up((size_t)slabs * N * 2 * sizeof(double), 256) +
         align_up((size_t)gslabs * F * N * sizeof(float), 256) + 1024;
}

int cfl_project_bwd(const float* x, int64_t B, int F, int64_t ldx, const float* V, int N,
                    int64_t ldV, const float* g, const float* bias, int weight_norm,
                    float in_scale, int act, const float* y, int64_t ldy, const float* z,
                    const float* dy, int64_t lddy, float* dV, float* dg, float* dbias,
                    int accumulate, float reg_c, void* ws, size_t ws_bytes, void* stream) {
  int st = device_check();
  if (st != CFL_OK) return st;
  CFL_REQUIRE(x && V && dy && dV && B >= 0 && F > 0 && N > 0, CFL_ERR_INVALID, "project_bwd: bad arguments");
  CFL_REQUIRE(act == CFL_ACT_LINEAR || y, CFL_ERR_INVALID, "project_bwd: non-linear act needs y");
  CFL_REQUIRE(!weight_norm || z, CFL_ERR_INVALID, "project_bwd: weight_norm needs the saved z");
  CFL_REQUIRE(ldx >= F && ldV >= N && lddy >= N && (!y || ldy >= N), CFL_ERR_INVALID,
              "project_bwd: leading dimension too small");
  CFL_REQUIRE(ws && ws_bytes >= cfl_project_bwd_workspace_bytes(B, F, N), CFL_ERR_WORKSPACE,
              "project_bwd: workspace too small");
  cudaStream_t cs = (cudaStream_t)stream;
  Workspace W(ws, ws_bytes);
  int slabs = bwd_slabs(B);
  float* scaler = W.take<float>(N);
  float* norm = W.take<float>(N);
  float* qn3 = W.take<float>(N);
  double* part = W.take<double>((size_t)slabs * N * 2);
  const bool tc = project_bwd_umma_supported(B, F, N);
  const int gslabs = tc ? project_bwd_umma_slabs(B, F) : slabs;
  float* Cpart = W.take<float>((size_t)gslabs * F * N);
  int64_t rps = (B + slabs - 1) / slabs;
  rps = (rps + TK - 1) / TK * TK;
  if (rps < TK) rps = TK;
  if (weight_norm) {
    colnorm_kernel<<<(N + 31) / 32, dim3(32, CN_SLICES), 0, cs>>>(V, F, N, ldV, g, scaler, norm);
    CFL_LAUNCH_CHECK();
  }
  colstats_kernel<<<dim3((N + 31) / 32, slabs), dim3(32, 8), 0, cs>>>(
      dy, lddy, y, ldy, weight_norm ? z : nullptr, act, B, N, rps, part);
  CFL_LAUNCH_CHECK();
  colstats_final<<<(N + 127) / 128, 128, 0, cs>>>(part, slabs, N, norm, bias, weight_norm,
                                                 accumulate, reg_c, qn3, dg, dbias, g);
  CFL_LAUNCH_CHECK();
  if (tc) {
    st = project_bwd_umma(x, B, F, ldx, dy, lddy, y, ldy, act, N, Cpart, cs);
    if (st != CFL_OK) return st;
  } else {
    dim3 grid((N + TN - 1) / TN, (F + TM - 1) / TM, slabs);
    project_bwd_gemm<<<grid, 256, 0, cs>>>(x, B, F, ldx, dy, lddy, y, ldy, act, N, rps, Cpart);
    CFL_LAUNCH_CHECK();
  }
  int64_t total = (int64_t)F * N;
  project_bwd_final<<<(unsigned)((total + 255) / 256), 256, 0, cs>>>(
      Cpart, gslabs, F, N, V, ldV, weight_norm ? scaler : nullptr, weight_norm ? qn3 : nullptr,
      in_scale, reg_c, accumulate, dV);
  CFL_LAUNCH_CHECK();
  return CFL_OK;
}

}  // extern "C"
