// train_vit.cu - training-mode building blocks of the ViT block stack that consumes the tokens (SURVEY.md 8f "next" #4
// on top of "next" #3): what autograd needs to carry dL/dlogits back to the tokenizer.
//
// The reference freezes the pre-trained blocks but trains the tokenizer THROUGH them (src/models/apf.py:335-346: every
// parameter whose name contains "encoder" or "head" stays trainable - point_encoder.*, encoder_norm.*, head.*), so a training
// step differentiates   APFViTLayer x 12 (src/models/apf_utils.py:268-293: LayerNorm -> attention -> residual; adapter and
// MLP on a second pair of LayerNorms; three-way sum)  ->  encoder_norm  ->  max over tokens  ->  ClassificationHead
// (apf.py:219-252, BatchNorm1d in TRAIN mode)   with respect to its input.  The GEMMs are p3tok_linear_f32 /
// p3tok_linear_tn_f32 (forward, dX = dY W, dW = dY^T X); this file adds the pieces that are not GEMMs:
//
//   p3tok_ln_fwd_f32 / p3tok_ln_bwd_f32 / p3tok_ln_param_grad_f32   nn.LayerNorm with saved row statistics
//   p3tok_attn_fwd_f32 / p3tok_attn_bwd_f32                           softmax(q k^T scale) v per (cloud, head), probabilities kept
//   p3tok_ew_f32                                                      a x + b y, masked scaling (dropout / DropPath), GELU and ReLU
//                                                                     with their derivatives
// fp32 on CUDA cores, like train.cu: the serving path is the tensor-core one, this path exists so that the kernels can stand
// in for the reference inside its trainers.  Parity target: oracle/train.py (float64), itself pinned against the reference's
// autograd (tests/golden/vit_train.npz, vit_train_full.npz).
#include "embed.cuh"

namespace p3tok {

__device__ __forceinline__ float tv_warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float tv_warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

static inline unsigned tv_grid(int64_t total, int threads, int64_t cap = 148 * 32) {
  int64_t b = (total + threads - 1) / threads;
  return (unsigned)(b < 1 ? 1 : (b > cap ? cap : b));
}

// ---- LayerNorm: one warp per row; two-pass statistics (mean, then the centred second moment), biased variance
__global__ void __launch_bounds__(256)
ln_fwd_kernel(const float* __restrict__ X, int64_t M, int D, const float* __restrict__ gamma, const float* __restrict__ beta,
              float eps, float* __restrict__ Y, float* __restrict__ mean, float* __restrict__ rstd) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * 8;
  for (int64_t m = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); m < M; m += nw) {
    const float* x = X + m * D;
    float s = 0.f;
    for (int c = lane; c < D; c += 32) s += x[c];
    const float mu = tv_warp_sum(s) / (float)D;
    float q = 0.f;
    for (int c = lane; c < D; c += 32) {
      const float d = x[c] - mu;
      q = fmaf(d, d, q);
    }
    const float rs = 1.f / sqrtf(tv_warp_sum(q) / (float)D + eps);
    if (Y)
      for (int c = lane; c < D; c += 32) {
        const float xh = (x[c] - mu) * rs;
        Y[m * D + c] = gamma ? fmaf(xh, gamma[c], beta ? beta[c] : 0.f) : xh;
      }
    if (lane == 0) {
      if (mean) mean[m] = mu;
      if (rstd) rstd[m] = rs;
    }
  }
}

// dX (+)= rstd (g dy - mean_c(g dy) - xhat mean_c(g dy xhat))
__global__ void __launch_bounds__(256)
ln_bwd_kernel(const float* __restrict__ dY, const float* __restrict__ X, int64_t M, int D, const float* __restrict__ mean,
              const float* __restrict__ rstd, const float* __restrict__ gamma, int accumulate, float* __restrict__ dX) {
  const int lane = threadIdx.x & 31;
  const int64_t nw = (int64_t)gridDim.x * 8;
  for (int64_t m = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); m < M; m += nw) {
    const float* x = X + m * D;
    const float* dy = dY + m * D;
    const float mu = mean[m], rs = rstd[m];
    float a = 0.f, b = 0.f;
    for (int c = lane; c < D; c += 32) {
      const float g = gamma ? gamma[c] * dy[c] : dy[c];
      a += g;
      b = fmaf(g, (x[c] - mu) * rs, b);
    }
    a = tv_warp_sum(a) / (float)D;
    b = tv_warp_sum(b) / (float)D;
    for (int c = lane; c < D; c += 32) {
      const float g = gamma ? gamma[c] * dy[c] : dy[c];
      const float v = rs * (g - a - (x[c] - mu) * rs * b);
      dX[m * D + c] = accumulate ? dX[m * D + c] + v : v;
    }
  }
}

// dgamma[c] = sum_m dy xhat, dbeta[c] = sum_m dy: column strips, fp32 inside a strip of 64 rows per lane, fp64 across.
// kPartial: strip y stores its sums to dgamma[y][D] / dbeta[y][D] (a workspace; strip_sum_f64 adds the strips in order).
template <bool kPartial>
__global__ void __launch_bounds__(256)
ln_param_grad_kernel(const float* __restrict__ dY, const float* __restrict__ X, int64_t M, int D, const float* __restrict__ mean,
                     const float* __restrict__ rstd, int64_t rows_per_block, double* __restrict__ dgamma,
                     double* __restrict__ dbeta) {
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const int rlane = threadIdx.x >> 5;
  const int64_t m0 = (int64_t)blockIdx.y * rows_per_block, m1 = m0 + rows_per_block < M ? m0 + rows_per_block : M;
  double a = 0.0, b = 0.0;
  if (c < D) {
    float fa = 0.f, fb = 0.f;
    int n = 0;
    for (int64_t m = m0 + rlane; m < m1; m += 8) {
      const float dy = dY[m * D + c];
      fa = fmaf(dy, (X[m * D + c] - mean[m]) * rstd[m], fa);
      fb += dy;
      if (++n == 64) { a += fa; b += fb; fa = fb = 0.f; n = 0; }
    }
    a += fa; b += fb;
  }
  __shared__ double ra[8][32], rb[8][32];
  ra[rlane][threadIdx.x & 31] = a;
  rb[rlane][threadIdx.x & 31] = b;
  __syncthreads();
  if (rlane == 0 && c < D) {
#pragma unroll
    for (int r = 1; r < 8; ++r) { a += ra[r][threadIdx.x & 31]; b += rb[r][threadIdx.x & 31]; }
    if constexpr (kPartial) {
      dgamma[(size_t)blockIdx.y * D + c] = a;
      dbeta[(size_t)blockIdx.y * D + c] = b;
    } else {
      atomicAdd(&dgamma[c], a);
      atomicAdd(&dbeta[c], b);
    }
  }
}

// ---- attention (apf_utils.py:141-153): one CTA per (cloud, head); K and V of the head in shared memory (row pitch hd + 1:
// lanes that walk keys and lanes that walk channels are both conflict-free), a warp per query row.
// qkv (B*G, 3D): [q | k | v], head h = columns h*hd .. of each third.  P (B*heads, G, G) is kept for the backward.
constexpr int AT_WARPS = 8;

__device__ __forceinline__ void at_load_heads(const float* __restrict__ src0, const float* __restrict__ src1, int64_t pitch0,
                                              int64_t pitch1, int G, int hd, float* __restrict__ s0, float* __restrict__ s1) {
  for (int e = threadIdx.x; e < G * hd; e += AT_WARPS * 32) {
    const int j = e / hd, d = e - j * hd;
    s0[j * (hd + 1) + d] = src0[(int64_t)j * pitch0 + d];
    s1[j * (hd + 1) + d] = src1[(int64_t)j * pitch1 + d];
  }
}

__global__ void __launch_bounds__(AT_WARPS * 32)
attn_fwd_kernel(const float* __restrict__ qkv, int G, int heads, int hd, float scale, float* __restrict__ O,
                float* __restrict__ P) {
  extern __shared__ float at_sm[];
  const int D = heads * hd, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* Ks = at_sm;
  float* Vs = Ks + (size_t)G * (hd + 1);
  float* qw = Vs + (size_t)G * (hd + 1) + (size_t)warp * (hd + G);
  float* pw = qw + hd;
  const int64_t b = blockIdx.x / heads;
  const int h = (int)(blockIdx.x - b * heads);
  const float* base = qkv + b * G * 3 * D + h * hd;
  at_load_heads(base + D, base + 2 * D, 3 * D, 3 * D, G, hd, Ks, Vs);
  __syncthreads();
  float* Pb = P + (int64_t)blockIdx.x * G * G;
  for (int i = warp; i < G; i += AT_WARPS) {
    for (int d = lane; d < hd; d += 32) qw[d] = base[(int64_t)i * 3 * D + d];
    __syncwarp();
    float mx = -INFINITY;
    for (int j = lane; j < G; j += 32) {
      const float* kr = Ks + (size_t)j * (hd + 1);
      float s = 0.f;
      for (int d = 0; d < hd; ++d) s = fmaf(qw[d], kr[d], s);
      s *= scale;
      pw[j] = s;
      mx = fmaxf(mx, s);
    }
    mx = tv_warp_max(mx);
    float sum = 0.f;
    for (int j = lane; j < G; j += 32) {
      const float e = expf(pw[j] - mx);
      pw[j] = e;
      sum += e;
    }
    const float inv = 1.f / tv_warp_sum(sum);
    for (int j = lane; j < G; j += 32) {
      const float p = pw[j] * inv;
      pw[j] = p;
      Pb[(int64_t)i * G + j] = p;
    }
    __syncwarp();
    for (int d = lane; d < hd; d += 32) {
      float o = 0.f;
      for (int j = 0; j < G; ++j) o = fmaf(pw[j], Vs[(size_t)j * (hd + 1) + d], o);
      O[(b * G + i) * D + h * hd + d] = o;
    }
    __syncwarp();
  }
}

// Backward for dO: phase 1 walks query rows (K, V in shared memory): dP = dO V^T, dS = P (dP - sum_j dP P) scale, dq = dS K;
// dS and P are left TRANSPOSED in the scratch so that phase 2, which walks keys (Q, dO in the same shared memory),
// reads its columns as rows: dk = dS^T q, dv = P^T dO.  PT / dST: (B*heads, G, G) each, only ever touched by their own CTA.
__global__ void __launch_bounds__(AT_WARPS * 32)
attn_bwd_kernel(const float* __restrict__ qkv, const float* __restrict__ P, const float* __restrict__ dO, int G, int heads, int hd,
                float scale, float* __restrict__ PT, float* __restrict__ dST, float* __restrict__ dqkv) {
  extern __shared__ float at_sm[];
  const int D = heads * hd, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* S0 = at_sm;                                   // K, then Q
  float* S1 = S0 + (size_t)G * (hd + 1);               // V, then dO
  float* vw = S1 + (size_t)G * (hd + 1) + (size_t)warp * (hd + 2 * G);
  float* aw = vw + hd;
  float* bw = aw + G;
  const int64_t b = blockIdx.x / heads;
  const int h = (int)(blockIdx.x - b * heads);
  const float* base = qkv + b * G * 3 * D + h * hd;
  const float* dOb = dO + b * G * D + h * hd;
  float* dbase = dqkv + b * G * 3 * D + h * hd;
  const float* Pb = P + (int64_t)blockIdx.x * G * G;
  float* PTb = PT + (int64_t)blockIdx.x * G * G;
  float* dSTb = dST + (int64_t)blockIdx.x * G * G;
  at_load_heads(base + D, base + 2 * D, 3 * D, 3 * D, G, hd, S0, S1);
  __syncthreads();
  for (int i = warp; i < G; i += AT_WARPS) {
    for (int d = lane; d < hd; d += 32) vw[d] = dOb[(int64_t)i * D + d];
    __syncwarp();
    float delta = 0.f;
    for (int j = lane; j < G; j += 32) {
      const float* vr = S1 + (size_t)j * (hd + 1);
      float dp = 0.f;
      for (int d = 0; d < hd; ++d) dp = fmaf(vw[d], vr[d], dp);
      const float p = Pb[(int64_t)i * G + j];
      aw[j] = p;
      bw[j] = dp;
      delta = fmaf(p, dp, delta);
    }
    delta = tv_warp_sum(delta);
    for (int j = lane; j < G; j += 32) {
      const float p = aw[j];
      const float ds = p * (bw[j] - delta) * scale;
      bw[j] = ds;
      PTb[(int64_t)j * G + i] = p;
      dSTb[(int64_t)j * G + i] = ds;
    }
    __syncwarp();
    for (int d = lane; d < hd; d += 32) {
      float dq = 0.f;
      for (int j = 0; j < G; ++j) dq = fmaf(bw[j], S0[(size_t)j * (hd + 1) + d], dq);
      dbase[(int64_t)i * 3 * D + d] = dq;
    }
    __syncwarp();
  }
  __syncthreads();                                     // every row of PT / dST written; K, V no longer needed
  at_load_heads(base, dOb, 3 * D, D, G, hd, S0, S1);
  __syncthreads();
  for (int j = warp; j < G; j += AT_WARPS) {
    for (int i = lane; i < G; i += 32) {
      aw[i] = PTb[(int64_t)j * G + i];
      bw[i] = dSTb[(int64_t)j * G + i];
    }
    __syncwarp();
    for (int d = lane; d < hd; d += 32) {
      float dk = 0.f, dv = 0.f;
      for (int i = 0; i < G; ++i) {
        dk = fmaf(bw[i], S0[(size_t)i * (hd + 1) + d], dk);
        dv = fmaf(aw[i], S1[(size_t)i * (hd + 1) + d], dv);
      }
      dbase[(int64_t)j * 3 * D + D + d] = dk;
      dbase[(int64_t)j * 3 * D + 2 * D + d] = dv;
    }
    __syncwarp();
  }
}

// ---- element-wise: out = f(A, B)
enum { EW_AXPBY = 0, EW_MUL = 1, EW_GELU = 2, EW_GELU_BWD = 3, EW_RELU = 4, EW_RELU_BWD = 5 };

template <int OP>
__global__ void ew_kernel(const float* A, const float* Bv, float alpha, float beta, int64_t total, int64_t bdiv, float* out) {
  // no __restrict__: `out` may be A or B (in-place updates of the residual / gradient streams)
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const float a = A[e];
    float r;
    if (OP == EW_AXPBY) r = fmaf(alpha, a, beta * Bv[e]);
    else if (OP == EW_MUL) r = alpha * a * Bv[bdiv > 1 ? e / bdiv : e];
    else if (OP == EW_GELU) r = 0.5f * a * (1.f + erff(a * 0.70710678118654752f));
    else if (OP == EW_GELU_BWD)
      r = Bv[e] * (0.5f * (1.f + erff(a * 0.70710678118654752f)) + a * expf(-0.5f * a * a) * 0.39894228040143268f);
    else if (OP == EW_RELU) r = fmaxf(a, 0.f);
    else r = a > 0.f ? Bv[e] : 0.f;
    out[e] = r;
  }
}

static size_t attn_smem_bytes(int64_t G, int64_t hd, int row_bufs) {
  return (size_t)(2 * G * (hd + 1) + AT_WARPS * (hd + row_bufs * G)) * sizeof(float);
}

}  // namespace p3tok

using namespace p3tok;

extern "C" int p3tok_ln_fwd_f32(const float* X, int64_t M, int64_t D, const float* gamma, const float* beta, float eps, float* Y,
                                float* mean, float* rstd, void* stream) {
  P3_REQUIRE(M >= 0 && D > 0 && D < (1 << 24), P3TOK_ERR_INVALID, "ln_fwd_f32: bad shape");
  if (M == 0) return P3TOK_OK;
  P3_REQUIRE(X && (Y || mean || rstd), P3TOK_ERR_INVALID, "ln_fwd_f32: null pointer");
  ln_fwd_kernel<<<tv_grid(M, 8), 256, 0, as_stream(stream)>>>(X, M, (int)D, gamma, beta, eps, Y, mean, rstd);
  P3_LAUNCH_CHECK("ln_fwd_kernel");
  return P3TOK_OK;
}

extern "C" int p3tok_ln_bwd_f32(const float* dY, const float* X, int64_t M, int64_t D, const float* mean, const float* rstd,
                                const float* gamma, int accumulate, float* dX, void* stream) {
  P3_REQUIRE(M >= 0 && D > 0 && D < (1 << 24), P3TOK_ERR_INVALID, "ln_bwd_f32: bad shape");
  if (M == 0) return P3TOK_OK;
  P3_REQUIRE(dY && X && mean && rstd && dX, P3TOK_ERR_INVALID, "ln_bwd_f32: null pointer");
  ln_bwd_kernel<<<tv_grid(M, 8), 256, 0, as_stream(stream)>>>(dY, X, M, (int)D, mean, rstd, gamma, accumulate, dX);
  P3_LAUNCH_CHECK("ln_bwd_kernel");
  return P3TOK_OK;
}

extern "C" int p3tok_ln_param_grad_f32(const float* dY, const float* X, int64_t M, int64_t D, const float* mean, const float* rstd,
                                       double* dgamma, double* dbeta, void* stream) {
  P3_REQUIRE(M >= 0 && D > 0 && D < (1 << 24), P3TOK_ERR_INVALID, "ln_param_grad_f32: bad shape");
  P3_REQUIRE(dgamma && dbeta && (M == 0 || (dY && X && mean && rstd)), P3TOK_ERR_INVALID, "ln_param_grad_f32: null pointer");
  cudaStream_t s = as_stream(stream);
  P3_CUDA(cudaMemsetAsync(dgamma, 0, (size_t)D * sizeof(double), s));
  P3_CUDA(cudaMemsetAsync(dbeta, 0, (size_t)D * sizeof(double), s));
  if (M == 0) return P3TOK_OK;
  const int64_t cgroups = (D + 31) / 32;
  int64_t strips = (148 * 8 + cgroups - 1) / cgroups;
  int64_t rows = (M + strips - 1) / strips;
  rows = (rows + 63) / 64 * 64;
  strips = (M + rows - 1) / rows;
  P3_REQUIRE(strips < 65536, P3TOK_ERR_UNSUPPORTED, "ln_param_grad_f32: too many rows");
  ln_param_grad_kernel<false><<<dim3((unsigned)cgroups, (unsigned)strips), 256, 0, s>>>(dY, X, M, (int)D, mean, rstd, rows, dgamma, dbeta);
  P3_LAUNCH_CHECK("ln_param_grad_kernel");
  return P3TOK_OK;
}

extern "C" int p3tok_ln_param_grad_det_f32(const float* dY, const float* X, int64_t M, int64_t D, const float* mean, const float* rstd,
                                           double* dgamma, double* dbeta, void* workspace, int64_t workspace_bytes, void* stream) {
  P3_REQUIRE(M >= 0 && D > 0 && D < (1 << 24), P3TOK_ERR_INVALID, "ln_param_grad_det_f32: bad shape");
  P3_REQUIRE(dgamma && dbeta && (M == 0 || (dY && X && mean && rstd)), P3TOK_ERR_INVALID, "ln_param_grad_det_f32: null pointer");
  cudaStream_t s = as_stream(stream);
  if (M == 0) {
    P3_CUDA(cudaMemsetAsync(dgamma, 0, (size_t)D * sizeof(double), s));
    P3_CUDA(cudaMemsetAsync(dbeta, 0, (size_t)D * sizeof(double), s));
    return P3TOK_OK;
  }
  const int rc = colsum_det_begin(workspace, workspace_bytes, M, D, "ln_param_grad_det_f32");
  if (rc != P3TOK_OK) return rc;
  const int64_t rows = strip_rows(M, (int)D), strips = (M + rows - 1) / rows;   // the strips of p3tok_ln_param_grad_f32
  double* part = static_cast<double*>(workspace);
  ln_param_grad_kernel<true><<<dim3((unsigned)((D + 31) / 32), (unsigned)strips), 256, 0, s>>>(dY, X, M, (int)D, mean, rstd, rows, part,
                                                                                               part + strips * D);
  P3_LAUNCH_CHECK("ln_param_grad_kernel");
  return strip_sum_f64(part, M, (int)D, dgamma, dbeta, s);
}

static int attn_shape_ok(int64_t B, int64_t G, int64_t heads, int64_t hd, int row_bufs, const char* who) {
  P3_REQUIRE(B >= 0 && G > 0 && heads > 0 && hd > 0 && B * heads < (1ll << 31) && G < (1 << 15) && hd <= 256, P3TOK_ERR_INVALID,
             "%s: bad shape", who);
  P3_REQUIRE(attn_smem_bytes(G, hd, row_bufs) <= 227 * 1024, P3TOK_ERR_UNSUPPORTED,
             "%s: G = %lld tokens x head dim %lld does not fit one CTA's shared memory", who, (long long)G, (long long)hd);
  return P3TOK_OK;
}

extern "C" int p3tok_attn_fwd_f32(const float* qkv, int64_t B, int64_t G, int64_t heads, int64_t hd, float scale, float* O, float* P,
                                  void* stream) {
  const int rc = attn_shape_ok(B, G, heads, hd, 1, "attn_fwd_f32");
  if (rc != P3TOK_OK) return rc;
  if (B == 0) return P3TOK_OK;
  P3_REQUIRE(qkv && O && P, P3TOK_ERR_INVALID, "attn_fwd_f32: null pointer");
  const size_t smem = attn_smem_bytes(G, hd, 1);
  P3_CUDA(cudaFuncSetAttribute(attn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  attn_fwd_kernel<<<(unsigned)(B * heads), AT_WARPS * 32, smem, as_stream(stream)>>>(qkv, (int)G, (int)heads, (int)hd, scale, O, P);
  P3_LAUNCH_CHECK("attn_fwd_kernel");
  return P3TOK_OK;
}

extern "C" int p3tok_attn_bwd_f32(const float* qkv, const float* P, const float* dO, int64_t B, int64_t G, int64_t heads, int64_t hd,
                                  float scale, float* scratch, float* dqkv, void* stream) {
  const int rc = attn_shape_ok(B, G, heads, hd, 2, "attn_bwd_f32");
  if (rc != P3TOK_OK) return rc;
  if (B == 0) return P3TOK_OK;
  P3_REQUIRE(qkv && P && dO && scratch && dqkv, P3TOK_ERR_INVALID, "attn_bwd_f32: null pointer");
  const size_t smem = attn_smem_bytes(G, hd, 2);
  P3_CUDA(cudaFuncSetAttribute(attn_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  attn_bwd_kernel<<<(unsigned)(B * heads), AT_WARPS * 32, smem, as_stream(stream)>>>(
      qkv, P, dO, (int)G, (int)heads, (int)hd, scale, scratch, scratch + B * heads * G * G, dqkv);
  P3_LAUNCH_CHECK("attn_bwd_kernel");
  return P3TOK_OK;
}

extern "C" int p3tok_ew_f32(int op, const float* A, const float* Bv, float alpha, float beta, int64_t total, int64_t bdiv, float* out,
                            void* stream) {
  P3_REQUIRE(op >= EW_AXPBY && op <= EW_RELU_BWD && total >= 0 && bdiv >= 1, P3TOK_ERR_INVALID, "ew_f32: bad op / size");
  if (total == 0) return P3TOK_OK;
  const bool needs_b = op != EW_GELU && op != EW_RELU;
  P3_REQUIRE(A && out && (!needs_b || Bv), P3TOK_ERR_INVALID, "ew_f32: null pointer");
  cudaStream_t s = as_stream(stream);
  const unsigned grid = tv_grid(total, 256);
  switch (op) {
    case EW_AXPBY: ew_kernel<EW_AXPBY><<<grid, 256, 0, s>>>(A, Bv, alpha, beta, total, bdiv, out); break;
    case EW_MUL: ew_kernel<EW_MUL><<<grid, 256, 0, s>>>(A, Bv, alpha, beta, total, bdiv, out); break;
    case EW_GELU: ew_kernel<EW_GELU><<<grid, 256, 0, s>>>(A, Bv, alpha, beta, total, bdiv, out); break;
    case EW_GELU_BWD: ew_kernel<EW_GELU_BWD><<<grid, 256, 0, s>>>(A, Bv, alpha, beta, total, bdiv, out); break;
    case EW_RELU: ew_kernel<EW_RELU><<<grid, 256, 0, s>>>(A, Bv, alpha, beta, total, bdiv, out); break;
    default: ew_kernel<EW_RELU_BWD><<<grid, 256, 0, s>>>(A, Bv, alpha, beta, total, bdiv, out); break;
  }
  P3_LAUNCH_CHECK("ew_kernel");
  return P3TOK_OK;
}
