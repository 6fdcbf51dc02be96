// train.cu - training-mode building blocks of the patch embedding (SURVEY.md 8f "next" #4): batch-statistics BatchNorm
// and the backward of the mini-PointNet through both max-pools, the concat and the gather.
//
// What the reference trains (src/models/apf.py:335-346 keeps every parameter whose name contains "encoder" trainable;
// Pix4Point trains everything): the tokenizer's convolutions and BatchNorms in TRAIN mode - nn.BatchNorm1d/2d normalise
// with the statistics of the batch (biased variance, eps from the module), update the running estimates with momentum
// 0.1 and the unbiased variance (apf.py:129-143, pix4point.py:135-156) - and autograd through
//   Encoder.forward      apf.py:145-181   conv/BN/ReLU x2, conv, max over k, concat [global || local], conv/BN/ReLU, conv, max
//   P3Embed.forward      pix4point.py:171-189  gather, conv, conv/BN/ReLU, max, concat, conv/BN/ReLU x2, max
// Everything here is fp32 on CUDA cores (per-channel sums accumulate in fp64 across blocks); the host side
// (p3tok/train.py) strings the blocks together as torch.autograd.Functions.  Parity target: the float64 oracle
// oracle/train.py, itself pinned against the reference's own autograd (tests/golden/apf_train.npz, p4p_train.npz).
//
//   p3tok_linear_f32 (mlp_f32.cu)   Y = X W^T + b (+ per-group bias)       forward GEMMs and dX = dY W (W passed transposed)
//   p3tok_linear_tn_f32             dW[N,K] += dY[M,N]^T X[M,K]             weight gradients (split over M, fp32 atomics)
//   p3tok_colstats_f32              per-channel sum, sum of squares         BatchNorm batch statistics (fp64 accumulators)
//   p3tok_bn_act_f32                y = act(gamma (z - mean) rstd + beta)
//   p3tok_bn_bwd_stats_f32 / p3tok_bn_bwd_apply_f32   BatchNorm(+ReLU) backward: dgamma, dbeta and dz
//   p3tok_group_max_arg_f32 / p3tok_group_max_bwd_f32 max over k with the first arg-max (torch.max) and its scatter
//   p3tok_group_sum_f32             sum over the k rows of a group          gradient of the expanded global feature
//   p3tok_scatter_rows_add_f32      gradient of the kNN gather: every point collects the gradients of all its rows
//   p3tok_build_rows_f32            the gathered row matrix of p3tok_rows    (forward input of the training path)
//   p3tok_apf_rows_bwd_f32          adjoint of the APF rows: gradient to the input points (neighbour and centre terms)
//   p3tok_gather_points_bwd_f32     adjoint of p3tok_gather_points (index_points, fps, the centres)
#include "embed.cuh"

namespace p3tok {

static inline unsigned tr_grid(int64_t total, int threads, int64_t cap = 148 * 32) {
  int64_t b = (total + threads - 1) / threads;
  return (unsigned)(b < 1 ? 1 : (b > cap ? cap : b));
}

// ---- dW[N,K] (+)= dY[M,N]^T X[M,K]: 64 x 64 outputs per CTA, 4 x 4 per thread, the M range split over gridDim.z
constexpr int TN_T = 64, TN_MM = 16;
__global__ void __launch_bounds__(256)
sgemm_tn_kernel(const float* __restrict__ dY, const float* __restrict__ X, int64_t M, int N, int K, float* __restrict__ dW,
                int64_t rows_per_slice) {
  __shared__ float As[TN_MM][TN_T + 4];   // dY tile: [m][n]
  __shared__ float Bs[TN_MM][TN_T + 4];   // X tile:  [m][k]
  const int t = threadIdx.x, tn = t >> 4, tk = t & 15;
  const int n0 = blockIdx.x * TN_T, k0 = blockIdx.y * TN_T;
  const int64_t m_begin = (int64_t)blockIdx.z * rows_per_slice;
  const int64_t m_end = m_begin + rows_per_slice < M ? m_begin + rows_per_slice : M;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int64_t m0 = m_begin; m0 < m_end; m0 += TN_MM) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {               // 16 x 64 elements per tile, 256 threads x 4
      const int e = t + i * 256;
      const int mm = e >> 6, c = e & 63;
      const int64_t m = m0 + mm;
      As[mm][c] = (m < m_end && n0 + c < N) ? dY[m * N + n0 + c] : 0.f;
      Bs[mm][c] = (m < m_end && k0 + c < K) ? X[m * K + k0 + c] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int mm = 0; mm < TN_MM; ++mm) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = As[mm][tn * 4 + i]; b[i] = Bs[mm][tk * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int n = n0 + tn * 4 + i;
    if (n >= N) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + tk * 4 + j;
      if (k < K) atomicAdd(&dW[(size_t)n * K + k], acc[i][j]);
    }
  }
}

// ---- per-channel sums: every thread walks a strip of rows of ONE column group, fp32 inside the strip, fp64 across strips
__global__ void __launch_bounds__(256)
colstats_kernel(const float* __restrict__ X, int64_t M, int N, int64_t rows_per_block, double* __restrict__ sum,
                double* __restrict__ sumsq) {
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const int rlane = threadIdx.x >> 5;                         // 8 row lanes
  const int64_t m0 = (int64_t)blockIdx.y * rows_per_block, m1 = m0 + rows_per_block < M ? m0 + rows_per_block : M;
  double s = 0.0, q = 0.0;
  if (c < N) {
    float fs = 0.f, fq = 0.f;
    int n = 0;
    for (int64_t m = m0 + rlane; m < m1; m += 8) {
      const float v = X[m * N + c];
      fs += v;
      fq = fmaf(v, v, fq);
      if (++n == 64) { s += fs; q += fq; fs = fq = 0.f; n = 0; }
    }
    s += fs; q += fq;
  }
  __shared__ double rs[8][32], rq[8][32];
  rs[rlane][threadIdx.x & 31] = s;
  rq[rlane][threadIdx.x & 31] = q;
  __syncthreads();
  if (rlane == 0 && c < N) {
#pragma unroll
    for (int r = 1; r < 8; ++r) { s += rs[r][threadIdx.x & 31]; q += rq[r][threadIdx.x & 31]; }
    atomicAdd(&sum[c], s);
    atomicAdd(&sumsq[c], q);
  }
}

__global__ void bn_act_kernel(const float* __restrict__ Z, int64_t total, int N, const float* __restrict__ mean,
                              const float* __restrict__ rstd, const float* __restrict__ gamma, const float* __restrict__ beta,
                              int relu, float* __restrict__ Y) {
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(e % N);
    float y = fmaf((Z[e] - mean[c]) * rstd[c], gamma[c], beta[c]);
    if (relu) y = fmaxf(y, 0.f);
    Y[e] = y;
  }
}

// s1[c] = sum dy', s2[c] = sum dy' xhat with dy' = dy * [y > 0] (ReLU) and xhat = (z - mean) rstd
__global__ void __launch_bounds__(256)
bn_bwd_stats_kernel(const float* __restrict__ dY, const float* __restrict__ Z, int64_t M, int N, const float* __restrict__ mean,
                    const float* __restrict__ rstd, const float* __restrict__ gamma, const float* __restrict__ beta, int relu,
                    int64_t rows_per_block, double* __restrict__ s1, double* __restrict__ s2) {
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const int rlane = threadIdx.x >> 5;
  const int64_t m0 = (int64_t)blockIdx.y * rows_per_block, m1 = m0 + rows_per_block < M ? m0 + rows_per_block : M;
  double a = 0.0, b = 0.0;
  if (c < N) {
    const float mu = mean[c], rs = rstd[c], g = gamma[c], be = beta[c];
    float fa = 0.f, fb = 0.f;
    int n = 0;
    for (int64_t m = m0 + rlane; m < m1; m += 8) {
      const float xh = (Z[m * N + c] - mu) * rs;
      float dy = dY[m * N + c];
      if (relu && !(fmaf(xh, g, be) > 0.f)) dy = 0.f;
      fa += dy;
      fb = fmaf(dy, xh, fb);
      if (++n == 64) { a += fa; b += fb; fa = fb = 0.f; n = 0; }
    }
    a += fa; b += fb;
  }
  __shared__ double ra[8][32], rb[8][32];
  ra[rlane][threadIdx.x & 31] = a;
  rb[rlane][threadIdx.x & 31] = b;
  __syncthreads();
  if (rlane == 0 && c < N) {
#pragma unroll
    for (int r = 1; r < 8; ++r) { a += ra[r][threadIdx.x & 31]; b += rb[r][threadIdx.x & 31]; }
    atomicAdd(&s1[c], a);
    atomicAdd(&s2[c], b);
  }
}

// dz = gamma rstd (dy' - s1/M - xhat s2/M)
__global__ void bn_bwd_apply_kernel(const float* __restrict__ dY, const float* __restrict__ Z, int64_t total, int N, double invM,
                                    const float* __restrict__ mean, const float* __restrict__ rstd, const float* __restrict__ gamma,
                                    const float* __restrict__ beta, int relu, const double* __restrict__ s1,
                                    const double* __restrict__ s2, float* __restrict__ dZ) {
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(e % N);
    const float xh = (Z[e] - mean[c]) * rstd[c];
    float dy = dY[e];
    if (relu && !(fmaf(xh, gamma[c], beta[c]) > 0.f)) dy = 0.f;
    const float m1 = (float)(s1[c] * invM), m2 = (float)(s2[c] * invM);
    dZ[e] = gamma[c] * rstd[c] * (dy - m1 - xh * m2);
  }
}

__global__ void group_max_arg_kernel(const float* __restrict__ X, int64_t G, int k, int C, float* __restrict__ out,
                                     int32_t* __restrict__ arg) {
  const int64_t total = G * C;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g = e / C;
    const int c = (int)(e - g * C);
    const float* p = X + g * k * C + c;
    float m = p[0];
    int a = 0;
    for (int r = 1; r < k; ++r) {
      const float v = p[(int64_t)r * C];
      if (v > m) { m = v; a = r; }               // strict: the FIRST maximum, like torch.max(dim)
    }
    out[e] = m;
    arg[e] = a;
  }
}

// dX[(g*k + r), c] (+)= (r == arg[g,c]) ? dOut[g,c] : 0
__global__ void group_max_bwd_kernel(const float* __restrict__ dOut, const int32_t* __restrict__ arg, int64_t G, int k, int C,
                                     int accumulate, float* __restrict__ dX) {
  const int64_t total = G * k * C;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(e % C);
    const int64_t row = e / C;
    const int64_t g = row / k;
    const int r = (int)(row - g * k);
    const float v = arg[g * C + c] == r ? dOut[g * C + c] : 0.f;
    dX[e] = accumulate ? dX[e] + v : v;
  }
}

__global__ void group_sum_kernel(const float* __restrict__ X, int64_t G, int k, int C, float* __restrict__ out) {
  const int64_t total = G * C;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g = e / C;
    const int c = (int)(e - g * C);
    const float* p = X + g * k * C + c;
    float s = 0.f;
    for (int r = 0; r < k; ++r) s += p[(int64_t)r * C];
    out[e] = s;
  }
}

// gradient of the gather (pix4point.py:92-102): dRows (B,G,k,3+D) -> dP (B,N,3) += , dF (B,N,D) +=
__global__ void scatter_rows_add_kernel(const float* __restrict__ dRows, const int32_t* __restrict__ idx, int64_t B, int64_t N,
                                        int64_t Gk, int D, float* __restrict__ dP, float* __restrict__ dF) {
  const int W = 3 + D;
  const int64_t total = B * Gk * W;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(e % W);
    const int64_t row = e / W;
    const int64_t b = row / Gk;
    const int64_t p = b * N + idx[row];
    const float v = dRows[e];
    if (c < 3) { if (dP) atomicAdd(&dP[p * 3 + c], v); }
    else if (dF) atomicAdd(&dF[p * D + (c - 3)], v);
  }
}

// adjoint of the APF rows (build_rows kind 0): output group bj reads input group g = perm[bj]; its row n is
// [x[nbr] - x[ctr] || x[ctr]].  One thread per (output group, channel): d rel goes to the neighbour (one atomic per element),
// sum_n (d ctr - d rel) is reduced over the group's k rows in a register and added to the centre with one atomic.
template <typename IdxT>
__global__ void apf_rows_bwd_kernel(const float* __restrict__ dRows, const int64_t* __restrict__ ctr_idx,
                                    const IdxT* __restrict__ knn_idx, const int64_t* __restrict__ perm, int64_t N, int64_t G,
                                    int k, int C, int64_t BG, float* __restrict__ dX) {
  const int64_t total = BG * C;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(e % C);
    const int64_t bj = e / C;
    const int64_t b = bj / G;
    const int64_t g = perm ? perm[bj] : (bj - b * G);
    const IdxT* nbr = knn_idx + (b * G + g) * k;
    const float* d = dRows + bj * k * 2 * C + c;
    float acc = 0.f;
    for (int n = 0; n < k; ++n) {
      const float drel = d[(int64_t)n * 2 * C], dctr = d[(int64_t)n * 2 * C + C];
      atomicAdd(&dX[(b * N + (int64_t)nbr[n]) * C + c], drel);
      acc += dctr - drel;
    }
    atomicAdd(&dX[(b * N + ctr_idx[b * G + g]) * C + c], acc);
  }
}

// adjoint of gather_points: dX[b, idx[b,s], c] += dOut[b, s, c]
__global__ void gather_points_bwd_kernel(const float* __restrict__ dOut, int64_t N, int C, const int64_t* __restrict__ idx,
                                         int64_t S, int64_t total, float* __restrict__ dX) {
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(e % C);
    const int64_t bs = e / C;
    const int64_t b = bs / S;
    atomicAdd(&dX[(b * N + idx[bs]) * C + c], dOut[e]);
  }
}

}  // namespace p3tok

using namespace p3tok;

extern "C" int p3tok_linear_tn_f32(const float* dY, const float* X, int64_t M, int64_t N, int64_t K, float* dW, int accumulate,
                                   void* stream) {
  P3_REQUIRE(M >= 0 && N > 0 && K > 0 && N < (1 << 24) && K < (1 << 24), P3TOK_ERR_INVALID, "linear_tn_f32: bad shape");
  P3_REQUIRE(dW && (M == 0 || (dY && X)), P3TOK_ERR_INVALID, "linear_tn_f32: null pointer");
  cudaStream_t s = as_stream(stream);
  if (!accumulate) P3_CUDA(cudaMemsetAsync(dW, 0, (size_t)N * K * sizeof(float), s));
  if (M == 0) return P3TOK_OK;
  const int gn = (int)((N + TN_T - 1) / TN_T), gk = (int)((K + TN_T - 1) / TN_T);
  // enough M slices to fill the GPU (~4 CTAs per SM), each a multiple of the 16-row tile and at least 256 rows
  int64_t slices = (148 * 4 + gn * gk - 1) / (gn * gk);
  int64_t rows = (M + slices - 1) / slices;
  rows = (rows + 255) / 256 * 256;
  slices = (M + rows - 1) / rows;
  P3_REQUIRE(slices < 65536, P3TOK_ERR_UNSUPPORTED, "linear_tn_f32: too many rows");
  sgemm_tn_kernel<<<dim3((unsigned)gn, (unsigned)gk, (unsigned)slices), 256, 0, s>>>(dY, X, M, (int)N, (int)K, dW, rows);
  P3_LAUNCH_CHECK("sgemm_tn_kernel");
  return P3TOK_OK;
}

static int64_t strip_rows(int64_t M, int N) {
  const int64_t cgroups = (N + 31) / 32;
  int64_t strips = (148 * 8 + cgroups - 1) / cgroups;
  int64_t rows = (M + strips - 1) / strips;
  rows = (rows + 63) / 64 * 64;
  return rows < 64 ? 64 : rows;
}

extern "C" int p3tok_colstats_f32(const float* X, int64_t M, int64_t N, double* sum, double* sumsq, void* stream) {
  P3_REQUIRE(M >= 0 && N > 0 && N < (1 << 24), P3TOK_ERR_INVALID, "colstats_f32: bad shape");
  P3_REQUIRE(sum && sumsq && (M == 0 || X), P3TOK_ERR_INVALID, "colstats_f32: null pointer");
  cudaStream_t s = as_stream(stream);
  P3_CUDA(cudaMemsetAsync(sum, 0, (size_t)N * sizeof(double), s));
  P3_CUDA(cudaMemsetAsync(sumsq, 0, (size_t)N * sizeof(double), s));
  if (M == 0) return P3TOK_OK;
  const int64_t rows = strip_rows(M, (int)N);
  const int64_t strips = (M + rows - 1) / rows;
  P3_REQUIRE(strips < 65536, P3TOK_ERR_UNSUPPORTED, "colstats_f32: too many rows");
  colstats_kernel<<<dim3((unsigned)((N + 31) / 32), (unsigned)strips), 256, 0, s>>>(X, M, (int)N, rows, sum, sumsq);
  P3_LAUNCH_CHECK("colstats_kernel");
  return P3TOK_OK;
}

extern "C" int p3tok_bn_act_f32(const float* Z, int64_t M, int64_t N, const float* mean, const float* rstd, const float* gamma,
                                const float* beta, int relu, float* Y, void* stream) {
  P3_REQUIRE(M >= 0 && N > 0, P3TOK_ERR_INVALID, "bn_act_f32: bad shape");
  if (M == 0) return P3TOK_OK;
  P3_REQUIRE(Z && mean && rstd && gamma && beta && Y, P3TOK_ERR_INVALID, "bn_act_f32: null pointer");
  bn_act_kernel<<<tr_grid(M * N, 256), 256, 0, as_stream(stream)>>>(Z, M * N, (int)N, mean, rstd, gamma, beta, relu, Y);
  P3_LAUNCH_CHECK("bn_act_kernel");
  return P3TOK_OK;
}

extern "C" int p3tok_bn_bwd_stats_f32(const float* dY, const float* Z, int64_t M, int64_t N, const float* mean, const float* rstd,
                                      const float* gamma, const float* beta, int relu, double* s1, double* s2, void* stream) {
  P3_REQUIRE(M >= 0 && N > 0, P3TOK_ERR_INVALID, "bn_bwd_stats_f32: bad shape");
  P3_REQUIRE(s1 && s2 && (M == 0 || (dY && Z && mean && rstd && gamma && beta)), P3TOK_ERR_INVALID, "bn_bwd_stats_f32: null pointer");
  cudaStream_t s = as_stream(stream);
  P3_CUDA(cudaMemsetAsync(s1, 0, (size_t)N * sizeof(double), s));
  P3_CUDA(cudaMemsetAsync(s2, 0, (size_t)N * sizeof(double), s));
  if (M == 0) return P3TOK_OK;
  const int64_t rows = strip_rows(M, (int)N);
  const int64_t strips = (M + rows - 1) / rows;
  P3_REQUIRE(strips < 65536, P3TOK_ERR_UNSUPPORTED, "bn_bwd_stats_f32: too many rows");
  bn_bwd_stats_kernel<<<dim3((unsigned)((N + 31) / 32), (unsigned)strips), 256, 0, s>>>(dY, Z, M, (int)N, mean, rstd, gamma, beta, relu,
                                                                                        rows, s1, s2);
  P3_LAUNCH_CHECK("bn_bwd_stats_kernel");
  return P3TOK_OK;
}

extern "C" int p3tok_bn_bwd_apply_f32(const float* dY, const float* Z, int64_t M, int64_t N, int64_t count, const float* mean,
                                      const float* rstd, const float* gamma, const float* beta, int relu, const double* s1,
                                      const double* s2, float* dZ, void* stream) {
  P3_REQUIRE(M >= 0 && N > 0 && count > 0, P3TOK_ERR_INVALID, "bn_bwd_apply_f32: bad shape");
  if (M == 0) return P3TOK_OK;
  P3_REQUIRE(dY && Z && mean && rstd && gamma && beta && s1 && s2 && dZ, P3TOK_ERR_INVALID, "bn_bwd_apply_f32: null pointer");
  bn_bwd_apply_kernel<<<tr_grid(M * N, 256), 256, 0, as_stream(stream)>>>(dY, Z, M * N, (int)N, 1.0 / (double)count, mean, rstd, gamma,
                                                                          beta, relu, s1, s2, dZ);
  P3_LAUNCH_CHECK("bn_bwd_apply_kernel");
  return P3TOK_OK;
}

extern "C" int p3tok_group_max_arg_f32(const float* X, int64_t G, int64_t k, int64_t C, float* out, int32_t* arg, void* stream) {
  P3_REQUIRE(G >= 0 && k > 0 && C > 0 && k < (1 << 30), P3TOK_ERR_INVALID, "group_max_arg_f32: bad shape");
  if (G == 0) return P3TOK_OK;
  P3_REQUIRE(X && out && arg, P3TOK_ERR_INVALID, "group_max_arg_f32: null pointer");
  group_max_arg_kernel<<<tr_grid(G * C, 256), 256, 0, as_stream(stream)>>>(X, G, (int)k, (int)C, out, arg);
  P3_LAUNCH_CHECK("group_max_arg_kernel");
  return P3TOK_OK;
}

extern "C" int p3tok_group_max_bwd_f32(const float* dOut, const int32_t* arg, int64_t G, int64_t k, int64_t C, int accumulate,
                                       float* dX, void* stream) {
  P3_REQUIRE(G >= 0 && k > 0 && C > 0, P3TOK_ERR_INVALID, "group_max_bwd_f32: bad shape");
  if (G == 0) return P3TOK_OK;
  P3_REQUIRE(dOut && arg && dX, P3TOK_ERR_INVALID, "group_max_bwd_f32: null pointer");
  group_max_bwd_kernel<<<tr_grid(G * k * C, 256), 256, 0, as_stream(stream)>>>(dOut, arg, G, (int)k, (int)C, accumulate, dX);
  P3_LAUNCH_CHECK("group_max_bwd_kernel");
  return P3TOK_OK;
}

extern "C" int p3tok_group_sum_f32(const float* X, int64_t G, int64_t k, int64_t C, float* out, void* stream) {
  P3_REQUIRE(G >= 0 && k > 0 && C > 0, P3TOK_ERR_INVALID, "group_sum_f32: bad shape");
  if (G == 0) return P3TOK_OK;
  P3_REQUIRE(X && out, P3TOK_ERR_INVALID, "group_sum_f32: null pointer");
  group_sum_kernel<<<tr_grid(G * C, 256), 256, 0, as_stream(stream)>>>(X, G, (int)k, (int)C, out);
  P3_LAUNCH_CHECK("group_sum_kernel");
  return P3TOK_OK;
}

extern "C" int p3tok_scatter_rows_add_f32(const float* dRows, const int32_t* idx, int64_t B, int64_t N, int64_t G, int64_t k, int64_t D,
                                          float* dP, float* dF, void* stream) {
  P3_REQUIRE(B >= 0 && N > 0 && G >= 0 && k > 0 && D >= 0, P3TOK_ERR_INVALID, "scatter_rows_add_f32: bad shape");
  if (B * G == 0) return P3TOK_OK;
  P3_REQUIRE(dRows && idx && (dP || dF), P3TOK_ERR_INVALID, "scatter_rows_add_f32: null pointer");
  scatter_rows_add_kernel<<<tr_grid(B * G * k * (3 + D), 256), 256, 0, as_stream(stream)>>>(dRows, idx, B, N, G * k, (int)D, dP, dF);
  P3_LAUNCH_CHECK("scatter_rows_add_kernel");
  return P3TOK_OK;
}

extern "C" int p3tok_build_rows_f32(const p3tok_rows* rows, float* X, void* stream) {
  P3_REQUIRE(rows && rows->kind >= 0 && rows->kind <= 1, P3TOK_ERR_INVALID, "build_rows_f32: APF (0) or P4P (1) rows expected");
  P3_REQUIRE(rows->B >= 0 && rows->G >= 0 && rows->k > 0, P3TOK_ERR_INVALID, "build_rows_f32: bad B/G/k");
  if (rows->B * rows->G == 0) return P3TOK_OK;
  P3_REQUIRE(X && rows->x && rows->knn_idx, P3TOK_ERR_INVALID, "build_rows_f32: null pointer");
  P3_REQUIRE(rows->kind != 0 || rows->ctr_idx, P3TOK_ERR_INVALID, "build_rows_f32: APF rows need ctr_idx");
  P3_REQUIRE(rows->kind != 1 || rows->feats, P3TOK_ERR_INVALID, "build_rows_f32: P4P rows need feats");
  return build_rows_f32(rows, 0, rows->B * rows->G, X, as_stream(stream));
}

extern "C" int p3tok_apf_rows_bwd_f32(const p3tok_rows* rows, const float* dRows, float* dX, void* stream) {
  P3_REQUIRE(rows && rows->kind == 0, P3TOK_ERR_INVALID, "apf_rows_bwd_f32: APF (kind 0) rows expected");
  P3_REQUIRE(rows->B >= 0 && rows->N > 0 && rows->G >= 0 && rows->k > 0 && rows->k < (1 << 30) && rows->C > 0,
             P3TOK_ERR_INVALID, "apf_rows_bwd_f32: bad shape");
  P3_REQUIRE(rows->idx_dtype == P3TOK_I64 || rows->idx_dtype == P3TOK_I32, P3TOK_ERR_INVALID, "apf_rows_bwd_f32: bad idx_dtype");
  const int64_t BG = rows->B * rows->G;
  if (BG == 0) return P3TOK_OK;
  P3_REQUIRE(dRows && dX && rows->ctr_idx && rows->knn_idx, P3TOK_ERR_INVALID, "apf_rows_bwd_f32: null pointer");
  cudaStream_t s = as_stream(stream);
  if (rows->idx_dtype == P3TOK_I64)
    apf_rows_bwd_kernel<int64_t><<<tr_grid(BG * rows->C, 256), 256, 0, s>>>(
        dRows, rows->ctr_idx, static_cast<const int64_t*>(rows->knn_idx), rows->perm, rows->N, rows->G, (int)rows->k, rows->C, BG, dX);
  else
    apf_rows_bwd_kernel<int32_t><<<tr_grid(BG * rows->C, 256), 256, 0, s>>>(
        dRows, rows->ctr_idx, static_cast<const int32_t*>(rows->knn_idx), rows->perm, rows->N, rows->G, (int)rows->k, rows->C, BG, dX);
  P3_LAUNCH_CHECK("apf_rows_bwd_kernel");
  return P3TOK_OK;
}

extern "C" int p3tok_gather_points_bwd_f32(const float* dOut, int64_t B, int64_t N, int64_t C, const int64_t* idx, int64_t S, float* dX,
                                           void* stream) {
  P3_REQUIRE(B >= 0 && N > 0 && C > 0 && S >= 0, P3TOK_ERR_INVALID, "gather_points_bwd_f32: bad shape");
  const int64_t total = B * S * C;
  if (total == 0) return P3TOK_OK;
  P3_REQUIRE(dOut && idx && dX, P3TOK_ERR_INVALID, "gather_points_bwd_f32: null pointer");
  gather_points_bwd_kernel<<<tr_grid(total, 256), 256, 0, as_stream(stream)>>>(dOut, N, (int)C, idx, S, total, dX);
  P3_LAUNCH_CHECK("gather_points_bwd_kernel");
  return P3TOK_OK;
}
