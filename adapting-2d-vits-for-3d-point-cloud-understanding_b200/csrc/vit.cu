// vit.cu - the ViT block stack that consumes the tokens (SURVEY.md 8f "next" #3).
//
// Replaces the block loop, encoder_norm and token max of AdaptPointFormer.forward (reference src/models/apf.py:361-366)
// with APFViTLayer = attention + bottleneck adapter + MLP (src/models/apf_utils.py:106-293), eval mode.
//
// At BASELINE config 2 (B = 128 clouds x G = 128 tokens = 16384 rows, D = 384) every GEMM of a layer is 7-14 us of tensor
// work, so a layer is bound by the NUMBER of kernels (each has ~10 us of launch / pipeline fill / drain) and by the GEMM
// epilogues, not by the MMAs.  The host therefore folds a layer (p3tok/apf_model.py::fold_vit_layer) into four GEMMs:
//   LayerNorm affines move into the weights that consume them (W' = W diag(gamma), b' = b + W beta), so norm2 and
//   adapter_norm (same statistics, different affine) become ONE affine-free normalisation feeding ONE GEMM
//   [fc1 ; down_proj] (N = H + R) whose epilogue applies GELU to the first H columns and ReLU to the last R, and
//   [fc2 | scale * up_proj] (K = H + R) consumes that matrix whole: x_out = 2 x + [h | dn] [Wfc2 | s Wup]^T + b.
// Data flow per layer (M = B*G rows, fp32 residual stream x updated in place, bf16 activations in the workspace):
//   ln_rows_kernel          xh = bf16((x - mean) / std)
//   tc_linear               qkv = xh Wqkv'^T + b'                     (tcgen05, bf16 out, 16 epilogue warps)   embed_tc.cu
//   attention_small_kernel  o  = softmax(q k^T / sqrt(hd)) v          (G <= 128: persistent over (cloud, head) items;
//   / attention_kernel                                                 longer sequences: one CTA per 128 query rows)
//   tc_linear               x += o Wproj^T + b                        (TMA reduce-add epilogue)          apf_utils.py:279-283
//   ln_rows_kernel          xh = bf16((x - mean) / std);  x = 2 x     (adapter's own "+ x" and the layer's, :233 and :292)
//   tc_linear               hd = [gelu | relu](xh [Wfc1' ; Wdown']^T + b')                               :217-225, :288
//   tc_linear               x += hd [Wfc2 | s Wup]^T + b
// then norm_max_kernel: pooled[b] = max over tokens of encoder_norm(x[b]).
// Both residual GEMMs add into x with TMA reduce stores (cp.reduce.async.bulk.tensor .add.f32): the first version loaded
// x in the epilogue (32 lanes x 128 B rows), and that load's latency - exposed once per 32x32 piece - was most of the
// kernel (proj: 25 us for 3.4 us of MMA work).
//
// Attention (sequence 128-196, head dim 32/64: 5 % of the FLOPs, bound by the exp / element-wise work on the scores)
// is a flash-style kernel on warp-level bf16 mma (ldmatrix fragments, fp32 online softmax in the log2 domain with the
// scale folded into one FFMA per score).  Measurements and what bounds each kernel: DESIGN.md 6c.
#include <math.h>
#include <stdlib.h>

#include "embed.cuh"

namespace p3tok {

// ------------------------------------------------------------------------------------------------ LayerNorm
// One warp per row, the row in registers (float4 index lane + 32 i, D <= 1024), two passes (mean, then centred
// variance - what torch computes up to rounding), biased variance, eps inside the square root.
constexpr int LN_MAX_V4 = 8;

// NV4 = float4 slots per lane (3 for D = 384, 6 for 768, 8 generic); every warp normalises TWO rows per pass, all loads of
// both rows issued before the first reduction (the kernel is a chain of exposed latencies: load, 2 x 5 shuffles, store).
template <int NV4, bool SPLIT>
__global__ void __launch_bounds__(256)
ln_rows_kernel(float* __restrict__ x, int64_t M, int D, float eps, const float* __restrict__ w,
               const float* __restrict__ bvec, __nv_bfloat16* __restrict__ out, float rescale, const float* __restrict__ add,
               float* __restrict__ out_f32) {
  // add != null: the rows are first replaced by x + add (Pix4Point re-adds the positional embedding in front of every block,
  // src/models/pix4point.py:254-255) - the sum is what the block normalises AND what its residual carries, so it is written back.
  // out_f32 != null: the (affine) normalised rows also leave in fp32 (the final norm of PointViT.forward, line 256).
  // SPLIT: out is [M, 2D] = [hi | lo] with hi = bf16(v), lo = bf16(v - hi): the split operand of the bf16x3 GEMMs.
  const int lane = threadIdx.x & 31;
  const int64_t row0 = ((int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 2;
  if (row0 >= M) return;
  const int nv = D >> 2;
  const bool two = row0 + 1 < M;   // warp-uniform
  float4 v[2][NV4];
  float s[2] = {0.f, 0.f};
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    float4* xr = reinterpret_cast<float4*>(x + (row0 + (two ? r : 0)) * D);
#pragma unroll
    for (int i = 0; i < NV4; ++i) {
      const int j = lane + 32 * i;
      v[r][i] = j < nv ? xr[j] : make_float4(0.f, 0.f, 0.f, 0.f);
      if (add && j < nv) {
        const float4 a4 = reinterpret_cast<const float4*>(add + (row0 + (two ? r : 0)) * D)[j];
        v[r][i].x += a4.x; v[r][i].y += a4.y; v[r][i].z += a4.z; v[r][i].w += a4.w;
      }
    }
  }
#pragma unroll
  for (int r = 0; r < 2; ++r) {
#pragma unroll
    for (int i = 0; i < NV4; ++i) s[r] += (v[r][i].x + v[r][i].y) + (v[r][i].z + v[r][i].w);
    if ((rescale != 1.f || add) && (r == 0 || two)) {   // the residual stream leaves this kernel multiplied (the layer's "2 x") / shifted
      float4* xr = reinterpret_cast<float4*>(x + (row0 + r) * D);
#pragma unroll
      for (int i = 0; i < NV4; ++i) {
        const int j = lane + 32 * i;
        if (j < nv) xr[j] = make_float4(v[r][i].x * rescale, v[r][i].y * rescale, v[r][i].z * rescale, v[r][i].w * rescale);
      }
    }
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    s[0] += __shfl_xor_sync(0xffffffffu, s[0], o);
    s[1] += __shfl_xor_sync(0xffffffffu, s[1], o);
  }
  const float mean[2] = {s[0] / (float)D, s[1] / (float)D};
  float q[2] = {0.f, 0.f};
#pragma unroll
  for (int r = 0; r < 2; ++r) {
#pragma unroll
    for (int i = 0; i < NV4; ++i) {
      const int j = lane + 32 * i;
      if (j < nv) {
        const float a = v[r][i].x - mean[r], b = v[r][i].y - mean[r], c = v[r][i].z - mean[r], d = v[r][i].w - mean[r];
        q[r] += (a * a + b * b) + (c * c + d * d);
      }
    }
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    q[0] += __shfl_xor_sync(0xffffffffu, q[0], o);
    q[1] += __shfl_xor_sync(0xffffffffu, q[1], o);
  }
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    if (r == 1 && !two) break;
    const float rstd = 1.f / sqrtf(q[r] / (float)D + eps);
    __nv_bfloat16* orow = out + (row0 + r) * (SPLIT ? 2 * D : D);
#pragma unroll
    for (int i = 0; i < NV4; ++i) {
      const int j = lane + 32 * i;
      if (j < nv) {
        float a = (v[r][i].x - mean[r]) * rstd, b = (v[r][i].y - mean[r]) * rstd, c = (v[r][i].z - mean[r]) * rstd,
              d = (v[r][i].w - mean[r]) * rstd;
        if (w) {   // warp-uniform
          const float4 ww = reinterpret_cast<const float4*>(w)[j], bb = reinterpret_cast<const float4*>(bvec)[j];
          a = fmaf(a, ww.x, bb.x); b = fmaf(b, ww.y, bb.y); c = fmaf(c, ww.z, bb.z); d = fmaf(d, ww.w, bb.w);
        }
        if (out_f32) reinterpret_cast<float4*>(out_f32 + (row0 + r) * D)[j] = make_float4(a, b, c, d);
        if constexpr (SPLIT) {
          const __nv_bfloat162 h0 = __floats2bfloat162_rn(a, b), h1 = __floats2bfloat162_rn(c, d);
          const float2 f0 = __bfloat1622float2(h0), f1 = __bfloat1622float2(h1);
          const __nv_bfloat162 l0 = __floats2bfloat162_rn(a - f0.x, b - f0.y), l1 = __floats2bfloat162_rn(c - f1.x, d - f1.y);
          reinterpret_cast<uint2*>(orow)[j] = make_uint2(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1));
          reinterpret_cast<uint2*>(orow + D)[j] = make_uint2(*reinterpret_cast<const uint32_t*>(&l0), *reinterpret_cast<const uint32_t*>(&l1));
        } else if (out) {
          __nv_bfloat162 lo = __floats2bfloat162_rn(a, b);
          __nv_bfloat162 hi = __floats2bfloat162_rn(c, d);
          reinterpret_cast<uint2*>(orow)[j] = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
        }
      }
    }
  }
}

// w == nullptr: plain normalisation (the affine lives in the consuming GEMM's weights)
// rescale != 1: x is also multiplied in place (x <- rescale * x) after it has been read
// split: out is [M, 2D] = [hi | lo] (bf16x3 stack) instead of [M, D]
static int layernorm_bf16(float* x, int64_t M, int D, float eps, const float* w, const float* b, __nv_bfloat16* out,
                          float rescale, cudaStream_t s, const float* add = nullptr, float* out_f32 = nullptr, bool split = false) {
  P3_REQUIRE(D % 4 == 0 && D > 0 && D <= 128 * LN_MAX_V4, P3TOK_ERR_UNSUPPORTED, "layernorm: D=%d must be a multiple of 4, <= %d", D,
             128 * LN_MAX_V4);
  P3_REQUIRE(x && (out || out_f32) && (!w == !b) && (!split || out), P3TOK_ERR_INVALID, "layernorm: null pointer");
  if (M == 0) return P3TOK_OK;
  const unsigned blocks = (unsigned)((M + 15) / 16);   // 8 warps x 2 rows
  if (split) {
    if (D <= 384) ln_rows_kernel<3, true><<<blocks, 256, 0, s>>>(x, M, D, eps, w, b, out, rescale, add, out_f32);
    else if (D <= 768) ln_rows_kernel<6, true><<<blocks, 256, 0, s>>>(x, M, D, eps, w, b, out, rescale, add, out_f32);
    else ln_rows_kernel<LN_MAX_V4, true><<<blocks, 256, 0, s>>>(x, M, D, eps, w, b, out, rescale, add, out_f32);
  } else {
    if (D <= 384) ln_rows_kernel<3, false><<<blocks, 256, 0, s>>>(x, M, D, eps, w, b, out, rescale, add, out_f32);
    else if (D <= 768) ln_rows_kernel<6, false><<<blocks, 256, 0, s>>>(x, M, D, eps, w, b, out, rescale, add, out_f32);
    else ln_rows_kernel<LN_MAX_V4, false><<<blocks, 256, 0, s>>>(x, M, D, eps, w, b, out, rescale, add, out_f32);
  }
  P3_LAUNCH_CHECK("ln_rows_kernel");
  return P3TOK_OK;
}

// encoder_norm + max over the tokens of a cloud (apf.py:364-366).  One CTA per cloud, warp per token row.
__global__ void __launch_bounds__(256)
norm_max_kernel(const float* __restrict__ x, int G, int D, float eps, const float* __restrict__ w, const float* __restrict__ b,
                float* __restrict__ pooled, int skip) {   // skip: leading rows of every sequence left out of the max (a cls token)
  __shared__ float4 red[8][32 * LN_MAX_V4];   // [warp][D/4], 32 KB
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nv = D >> 2;
  const float* xb = x + (size_t)blockIdx.x * G * D;
  float4 mx[LN_MAX_V4];
#pragma unroll
  for (int i = 0; i < LN_MAX_V4; ++i) mx[i] = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
  for (int r = warp + skip; r < G; r += 8) {
    const float4* xr = reinterpret_cast<const float4*>(xb + (size_t)r * D);
    float4 v[LN_MAX_V4];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < LN_MAX_V4; ++i) {
      const int j = lane + 32 * i;
      v[i] = j < nv ? xr[j] : make_float4(0.f, 0.f, 0.f, 0.f);
      s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float mean = s / (float)D;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < LN_MAX_V4; ++i) {
      const int j = lane + 32 * i;
      if (j < nv) {
        const float a = v[i].x - mean, bq = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
        q += (a * a + bq * bq) + (c * c + d * d);
      }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
    const float rstd = 1.f / sqrtf(q / (float)D + eps);
#pragma unroll
    for (int i = 0; i < LN_MAX_V4; ++i) {
      const int j = lane + 32 * i;
      if (j < nv) {
        const float4 ww = reinterpret_cast<const float4*>(w)[j], bb = reinterpret_cast<const float4*>(b)[j];
        mx[i].x = fmaxf(mx[i].x, fmaf((v[i].x - mean) * rstd, ww.x, bb.x));
        mx[i].y = fmaxf(mx[i].y, fmaf((v[i].y - mean) * rstd, ww.y, bb.y));
        mx[i].z = fmaxf(mx[i].z, fmaf((v[i].z - mean) * rstd, ww.z, bb.z));
        mx[i].w = fmaxf(mx[i].w, fmaf((v[i].w - mean) * rstd, ww.w, bb.w));
      }
    }
  }
#pragma unroll
  for (int i = 0; i < LN_MAX_V4; ++i) red[warp][lane + 32 * i] = mx[i];
  __syncthreads();
  for (int j = threadIdx.x; j < nv; j += blockDim.x) {
    float4 m = red[0][j];
#pragma unroll
    for (int wv = 1; wv < 8; ++wv) {
      const float4 o = red[wv][j];
      m.x = fmaxf(m.x, o.x); m.y = fmaxf(m.y, o.y); m.z = fmaxf(m.z, o.z); m.w = fmaxf(m.w, o.w);
    }
    reinterpret_cast<float4*>(pooled + (size_t)blockIdx.x * D)[j] = m;
  }
}

// ------------------------------------------------------------------------------------------------ attention
__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&t);
}

__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

constexpr int AT_Q = 128, AT_KV = 64, AT_THREADS = 256;   // query rows per CTA (8 warps x 16), keys per block

// 16-byte asynchronous global -> shared copy; `ok` false zero-fills (rows past the end of the cloud)
__device__ __forceinline__ void cp_async16(void* dst, const void* src, bool ok) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst);
  const int n = ok ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(src), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// bf16x3 (X3): every operand is a split pair hi = bf16(v), lo = bf16(v - hi) (hi + lo carries 16 mantissa bits) staged in a
// second tile `lo` elements behind the hi tile; a product a.b is evaluated as a_hi.b_hi + a_lo.b_hi + a_hi.b_lo (the lo.lo
// term is 2^-18 of it) on the same m16n8k16 fragments: 3x the MMAs, the fp32 online softmax unchanged.
template <int HD, bool X3>
constexpr int attention_smem_bytes() { return (AT_Q + 4 * AT_KV) * (HD + 8) * 2 * (X3 ? 2 : 1); }

// {hi, lo} bf16x2 pairs of (a, b): hi rounded as pack2 rounds, lo = the rounding error of hi, rounded
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  const float2 f = __bfloat1622float2(h);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = pack2(a - f.x, b - f.y);
}

// One 64-key block of the flash loop for a warp's 16 query rows: scores (raw), ragged-block mask, online softmax in the
// log2 domain, O += P V.  sK / sV: the block's [key][d] tiles (padded rows of RP elements).  Shared by both kernels.
// X3: qal holds the lo fragments of Q, and the lo tiles of K / V sit `lo` elements behind sK / sV.
template <int HD, bool X3>
__device__ __forceinline__ void attention_block(const uint32_t (&qa)[HD / 16][4], const uint32_t (&qal)[HD / 16][4],
                                                const __nv_bfloat16* sK, const __nv_bfloat16* sV, int lo, int kv0, int G,
                                                float scale_log2e, int lane, float (&o)[HD / 8][4], float& m0, float& m1, float& l0,
                                                float& l1) {
  constexpr int KS = HD / 16, DT = HD / 8, RP = HD + 8;
  const int t = lane & 3;
  float sc[AT_KV / 8][4];
#pragma unroll
  for (int nt = 0; nt < AT_KV / 8; ++nt) {
    sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = 0.f;
#pragma unroll
    for (int k2 = 0; k2 < KS; k2 += 2) {   // one x4: keys nt*8..+7, d chunks (k2*16, +8, +16, +24) = b0,b1 of two k steps
      uint32_t kb[4];
      const __nv_bfloat16* kp = &sK[(nt * 8 + (lane & 7)) * RP + k2 * 16 + (lane >> 3) * 8];
      ldsm_x4(kb, (uint32_t)__cvta_generic_to_shared(kp));
      if constexpr (X3) {                  // the two correction terms first: Q_hi K_lo, Q_lo K_hi
        uint32_t kl[4];
        ldsm_x4(kl, (uint32_t)__cvta_generic_to_shared(kp + lo));
        mma_bf16_16816(sc[nt], qa[k2], kl[0], kl[1]);
        mma_bf16_16816(sc[nt], qa[k2 + 1], kl[2], kl[3]);
        mma_bf16_16816(sc[nt], qal[k2], kb[0], kb[1]);
        mma_bf16_16816(sc[nt], qal[k2 + 1], kb[2], kb[3]);
      }
      mma_bf16_16816(sc[nt], qa[k2], kb[0], kb[1]);
      mma_bf16_16816(sc[nt], qa[k2 + 1], kb[2], kb[3]);
    }
  }
  if (kv0 + AT_KV > G) {   // ragged last block: keys past G never win the max and contribute 2^-inf = 0
#pragma unroll
    for (int nt = 0; nt < AT_KV / 8; ++nt) {
      const int col = kv0 + nt * 8 + 2 * t;
      if (col >= G) sc[nt][0] = sc[nt][2] = -INFINITY;
      if (col + 1 >= G) sc[nt][1] = sc[nt][3] = -INFINITY;
    }
  }
  float bm0 = -INFINITY, bm1 = -INFINITY;
#pragma unroll
  for (int nt = 0; nt < AT_KV / 8; ++nt) {
    bm0 = fmaxf(bm0, fmaxf(sc[nt][0], sc[nt][1]));
    bm1 = fmaxf(bm1, fmaxf(sc[nt][2], sc[nt][3]));
  }
  bm0 = fmaxf(bm0, __shfl_xor_sync(0xffffffffu, bm0, 1));
  bm0 = fmaxf(bm0, __shfl_xor_sync(0xffffffffu, bm0, 2));
  bm1 = fmaxf(bm1, __shfl_xor_sync(0xffffffffu, bm1, 1));
  bm1 = fmaxf(bm1, __shfl_xor_sync(0xffffffffu, bm1, 2));
  const float n0 = fmaxf(m0, bm0), n1 = fmaxf(m1, bm1);   // finite: every block holds at least one valid key
  const float c0 = ex2f((m0 - n0) * scale_log2e), c1 = ex2f((m1 - n1) * scale_log2e);   // 0 on the first block (m = -inf)
  m0 = n0; m1 = n1;
  const float ms0 = -n0 * scale_log2e, ms1 = -n1 * scale_log2e;
  l0 *= c0; l1 *= c1;
#pragma unroll
  for (int i = 0; i < DT; ++i) { o[i][0] *= c0; o[i][1] *= c0; o[i][2] *= c1; o[i][3] *= c1; }
#pragma unroll
  for (int nt = 0; nt < AT_KV / 8; ++nt) {
    sc[nt][0] = ex2f(fmaf(sc[nt][0], scale_log2e, ms0)); sc[nt][1] = ex2f(fmaf(sc[nt][1], scale_log2e, ms0));
    sc[nt][2] = ex2f(fmaf(sc[nt][2], scale_log2e, ms1)); sc[nt][3] = ex2f(fmaf(sc[nt][3], scale_log2e, ms1));
    l0 += sc[nt][0] + sc[nt][1];   // the row sums take the unrounded fp32 p
    l1 += sc[nt][2] + sc[nt][3];
  }
  // O += P V: the score accumulators of two adjacent key tiles are exactly one A fragment
#pragma unroll
  for (int kk = 0; kk < AT_KV / 16; ++kk) {
    uint32_t pa[4], pl[4];
    if constexpr (X3) {
      split2(sc[2 * kk][0], sc[2 * kk][1], pa[0], pl[0]);
      split2(sc[2 * kk][2], sc[2 * kk][3], pa[1], pl[1]);
      split2(sc[2 * kk + 1][0], sc[2 * kk + 1][1], pa[2], pl[2]);
      split2(sc[2 * kk + 1][2], sc[2 * kk + 1][3], pa[3], pl[3]);
    } else {
      pa[0] = pack2(sc[2 * kk][0], sc[2 * kk][1]);
      pa[1] = pack2(sc[2 * kk][2], sc[2 * kk][3]);
      pa[2] = pack2(sc[2 * kk + 1][0], sc[2 * kk + 1][1]);
      pa[3] = pack2(sc[2 * kk + 1][2], sc[2 * kk + 1][3]);
    }
#pragma unroll
    for (int dt = 0; dt < DT; dt += 2) {   // one x4.trans: keys kk*16 (+8), d tiles dt and dt+1 -> b0,b1 of each
      uint32_t vb[4];
      const __nv_bfloat16* vp = &sV[(kk * 16 + ((lane >> 3) & 1) * 8 + (lane & 7)) * RP + (dt + (lane >> 4)) * 8];
      ldsm_x4_t(vb, (uint32_t)__cvta_generic_to_shared(vp));
      if constexpr (X3) {                  // P_hi V_lo, P_lo V_hi
        uint32_t vl[4];
        ldsm_x4_t(vl, (uint32_t)__cvta_generic_to_shared(vp + lo));
        mma_bf16_16816(o[dt], pa, vl[0], vl[1]);
        mma_bf16_16816(o[dt + 1], pa, vl[2], vl[3]);
        mma_bf16_16816(o[dt], pl, vb[0], vb[1]);
        mma_bf16_16816(o[dt + 1], pl, vb[2], vb[3]);
      }
      mma_bf16_16816(o[dt], pa, vb[0], vb[1]);
      mma_bf16_16816(o[dt + 1], pa, vb[2], vb[3]);
    }
  }
}

// normalise by the row sums and store the warp's 16 rows (rows past G are skipped).  ob: row pitch D, or (X3) 2D with the
// lo half of the split output D columns behind the hi half.
template <int HD, bool X3>
__device__ __forceinline__ void attention_store(float (&o)[HD / 8][4], float l0, float l1, __nv_bfloat16* ob, int q0, int G, int D,
                                                int lane) {
  const int g = lane >> 2, t = lane & 3;
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
  l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float i0 = 1.f / l0, i1 = 1.f / l1;
  const int r0 = q0 + g, r1 = q0 + g + 8;
  const size_t ld = X3 ? 2 * (size_t)D : (size_t)D;
#pragma unroll
  for (int dt = 0; dt < HD / 8; ++dt) {
    if constexpr (X3) {   // __fmul_rn: lo is the rounding error of the product as stored, in every kernel (no FMA contraction)
      uint32_t h, l;
      if (r0 < G) {
        split2(__fmul_rn(o[dt][0], i0), __fmul_rn(o[dt][1], i0), h, l);
        *reinterpret_cast<uint32_t*>(ob + r0 * ld + dt * 8 + 2 * t) = h;
        *reinterpret_cast<uint32_t*>(ob + r0 * ld + D + dt * 8 + 2 * t) = l;
      }
      if (r1 < G) {
        split2(__fmul_rn(o[dt][2], i1), __fmul_rn(o[dt][3], i1), h, l);
        *reinterpret_cast<uint32_t*>(ob + r1 * ld + dt * 8 + 2 * t) = h;
        *reinterpret_cast<uint32_t*>(ob + r1 * ld + D + dt * 8 + 2 * t) = l;
      }
    } else {
      if (r0 < G) *reinterpret_cast<uint32_t*>(ob + (size_t)r0 * D + dt * 8 + 2 * t) = pack2(o[dt][0] * i0, o[dt][1] * i0);
      if (r1 < G) *reinterpret_cast<uint32_t*>(ob + (size_t)r1 * D + dt * 8 + 2 * t) = pack2(o[dt][2] * i1, o[dt][3] * i1);
    }
  }
}

// CTAs per SM the attention kernels are built for.  X3 doubles the staged tiles: the persistent form's two item buffers
// take 216 KB at head dim 64 and 120 KB at 32 - one CTA per SM either way, so both keep the double buffering (the next
// item's copy hides behind this item's 3x MMA work) rather than give it up for a second resident CTA at head dim 32.
template <int HD, bool X3, bool SMALL>
constexpr int attention_ctas_per_sm() { return X3 ? (SMALL ? 1 : (HD == 32 ? 2 : 1)) : (HD == 32 ? 3 : 2); }

// qkv (B*G, 3D) bf16: column which*D + head*HD + d (AttentionLayer's reshape(B,N,3,heads,hd), apf_utils.py:143).
// out (B*G, D) bf16: column head*HD + d ((attn @ v).transpose(1,2).reshape(B,N,C), apf_utils.py:155).
// X3: qkv (B*G, 6D) = [hi | lo] (lo of column c at 3D + c), out (B*G, 2D) = [hi | lo].
// grid (ceil(G/128), heads, B).  Q and the K / V blocks are staged row-major in padded shared memory by cp.async, two key
// blocks in flight (for G <= 128 the whole (cloud, head) is requested up front: one exposed memory latency per CTA
// instead of three - the first version, load -> barrier -> compute per block, was latency-bound at 32 us per 16 k rows);
// fragments come from ldmatrix (V through .trans: the [key][d] tile is already the k-major B operand of P V).
// Lane (g = lane/4, t = lane%4) of a warp owns query rows g and g+8 of the warp's 16 (the m16n8k16 accumulator layout),
// so row maxima / sums need only the two quad shuffles.  Scores stay raw; p = 2^(s*c - m*c) with c = log2(e)/sqrt(hd).
template <int HD, bool X3>
__global__ void __launch_bounds__(AT_THREADS, (attention_ctas_per_sm<HD, X3, false>()))
attention_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ out, int G, int D, float scale_log2e) {
  constexpr int KS = HD / 16;          // k steps of q k^T
  constexpr int DT = HD / 8;           // n tiles of the output
  constexpr int RP = HD + 8;           // padded row (16-byte aligned, conflict-free ldmatrix)
  constexpr int CPR = HD / 8;          // 16-byte chunks per row
  constexpr int NH = X3 ? 2 : 1;       // tiles per operand: hi (, lo)
  extern __shared__ __align__(16) uint8_t at_smem[];
  __nv_bfloat16* sQ = reinterpret_cast<__nv_bfloat16*>(at_smem);
  __nv_bfloat16* sKV = sQ + NH * AT_Q * RP;   // buffer j: K at sKV + j * 2 * NH * AT_KV * RP (lo tile behind), V right behind it
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int head = blockIdx.y, b = blockIdx.z;
  const int qb = blockIdx.x * AT_Q;
  const int q0 = qb + warp * 16;
  const size_t ld = (size_t)3 * NH * D;
  const __nv_bfloat16* base = qkv + (size_t)b * G * ld + (size_t)head * HD;
  const int nblk = (G + AT_KV - 1) / AT_KV;

  auto load_kv = [&](int blk) {
    __nv_bfloat16* k = sKV + (size_t)(blk & 1) * 2 * NH * AT_KV * RP;
    __nv_bfloat16* v = k + NH * AT_KV * RP;
    const int kv0 = blk * AT_KV;
    for (int c = tid; c < AT_KV * CPR; c += AT_THREADS) {
      const int r = c / CPR, ch = c % CPR;
      const bool ok = kv0 + r < G;
      const __nv_bfloat16* rowp = base + (size_t)(ok ? kv0 + r : 0) * ld + ch * 8;
#pragma unroll
      for (int h = 0; h < NH; ++h) {
        cp_async16(&k[h * AT_KV * RP + r * RP + ch * 8], rowp + h * 3 * D + D, ok);
        cp_async16(&v[h * AT_KV * RP + r * RP + ch * 8], rowp + h * 3 * D + 2 * D, ok);
      }
    }
  };
  for (int c = tid; c < AT_Q * CPR; c += AT_THREADS) {
    const int r = c / CPR, ch = c % CPR;
    const bool ok = qb + r < G;
#pragma unroll
    for (int h = 0; h < NH; ++h)
      cp_async16(&sQ[h * AT_Q * RP + r * RP + ch * 8], base + (size_t)(ok ? qb + r : 0) * ld + h * 3 * D + ch * 8, ok);
  }
  load_kv(0);
  cp_async_commit();                   // group: Q + block 0
  if (nblk > 1) load_kv(1);
  cp_async_commit();                   // group: block 1 (possibly empty)

  const bool active = q0 < G;          // warps whose 16 rows lie past G only help with the copies
  uint32_t qa[KS][4], qal[KS][4];
  float o[DT][4];
#pragma unroll
  for (int i = 0; i < DT; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;   // running maxima of the RAW scores, running sums

  for (int blk = 0; blk < nblk; ++blk) {
    cp_async_wait<1>();                // everything but the most recent group has landed: this block (and Q)
    __syncthreads();
    const int kv0 = blk * AT_KV;
    const __nv_bfloat16* sK = sKV + (size_t)(blk & 1) * 2 * NH * AT_KV * RP;
    const __nv_bfloat16* sV = sK + NH * AT_KV * RP;
    if (blk == 0) {
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {   // lanes 0-15: rows 0-15 at column ks*16; lanes 16-31: the same rows at column ks*16 + 8
        const __nv_bfloat16* qp = &sQ[(warp * 16 + (lane & 15)) * RP + ks * 16 + (lane >> 4) * 8];
        ldsm_x4(qa[ks], (uint32_t)__cvta_generic_to_shared(qp));
        if constexpr (X3) ldsm_x4(qal[ks], (uint32_t)__cvta_generic_to_shared(qp + AT_Q * RP));
      }
    }
    if (active) attention_block<HD, X3>(qa, qal, sK, sV, AT_KV * RP, kv0, G, scale_log2e, lane, o, m0, m1, l0, l1);
    __syncthreads();                   // every warp is done with buffer blk & 1
    if (blk + 2 < nblk) load_kv(blk + 2);
    cp_async_commit();                 // one group per iteration keeps the wait_group<1> accounting uniform
  }
  if (active) attention_store<HD, X3>(o, l0, l1, out + (size_t)b * G * NH * D + (size_t)head * HD, q0, G, D, lane);
}

// Persistent form for short sequences (G <= 128: one query block, at most two key blocks - BASELINE config 2): a CTA walks
// (cloud, head) items, and while it computes item i the whole of item i+1 (Q, K, V: 30 KB at head dim 32) is already in
// flight into the other half of shared memory.  The non-persistent kernel above pays one exposed L2 round trip per CTA and
// runs 3.5 rounds of CTAs per SM at config 2 (24 us per layer); here only the first item of a CTA waits.
template <int HD, bool X3>
constexpr int attention_small_smem_bytes() { return 2 * 3 * AT_Q * (HD + 8) * 2 * (X3 ? 2 : 1); }

template <int HD, bool X3>
__global__ void __launch_bounds__(AT_THREADS, (attention_ctas_per_sm<HD, X3, true>()))
attention_small_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ out, int G, int D, int heads, int items,
                       float scale_log2e) {
  constexpr int KS = HD / 16, DT = HD / 8, RP = HD + 8, CPR = HD / 8;
  constexpr int NH = X3 ? 2 : 1;
  constexpr int BUF = 3 * NH * AT_Q * RP;   // elements per item buffer: Q, K, V of 128 rows each (X3: each hi then lo)
  extern __shared__ __align__(16) uint8_t at_smem[];
  __nv_bfloat16* sm = reinterpret_cast<__nv_bfloat16*>(at_smem);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const size_t ld = (size_t)3 * NH * D;
  const int nblk = (G + AT_KV - 1) / AT_KV;   // 1 or 2
  const int kv_rows = nblk * AT_KV;
  const int q0 = warp * 16;
  const bool active = q0 < G;

  auto load_item = [&](int item, int buf) {
    const int b = item / heads, head = item - b * heads;
    const __nv_bfloat16* base = qkv + (size_t)b * G * ld + (size_t)head * HD;
    __nv_bfloat16* q = sm + (size_t)buf * BUF;
    __nv_bfloat16* k = q + NH * AT_Q * RP;
    __nv_bfloat16* v = k + NH * AT_Q * RP;
    for (int c = tid; c < AT_Q * CPR; c += AT_THREADS) {
      const int r = c / CPR, ch = c % CPR;
      const bool ok = r < G;
      const __nv_bfloat16* rowp = base + (size_t)(ok ? r : 0) * ld + ch * 8;
#pragma unroll
      for (int h = 0; h < NH; ++h) {
        cp_async16(&q[h * AT_Q * RP + r * RP + ch * 8], rowp + h * 3 * D, ok);
        if (r < kv_rows) {
          cp_async16(&k[h * AT_Q * RP + r * RP + ch * 8], rowp + h * 3 * D + D, ok);
          cp_async16(&v[h * AT_Q * RP + r * RP + ch * 8], rowp + h * 3 * D + 2 * D, ok);
        }
      }
    }
  };

  int buf = 0;
  if ((int)blockIdx.x < items) load_item(blockIdx.x, 0);
  cp_async_commit();
  for (int item = blockIdx.x; item < items; item += gridDim.x) {
    const int next = item + gridDim.x;
    if (next < items) load_item(next, buf ^ 1);   // the other buffer was released by the barrier that ended the previous item
    cp_async_commit();
    cp_async_wait<1>();                            // this item's group has landed
    __syncthreads();
    const __nv_bfloat16* sQ = sm + (size_t)buf * BUF;
    const __nv_bfloat16* sKa = sQ + NH * AT_Q * RP;
    const __nv_bfloat16* sVa = sKa + NH * AT_Q * RP;
    if (active) {
      uint32_t qa[KS][4], qal[KS][4];
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        const __nv_bfloat16* qp = &sQ[(q0 + (lane & 15)) * RP + ks * 16 + (lane >> 4) * 8];
        ldsm_x4(qa[ks], (uint32_t)__cvta_generic_to_shared(qp));
        if constexpr (X3) ldsm_x4(qal[ks], (uint32_t)__cvta_generic_to_shared(qp + AT_Q * RP));
      }
      float o[DT][4];
#pragma unroll
      for (int i = 0; i < DT; ++i) o[i][0] = o[i][1] = o[i][2] = o[i][3] = 0.f;
      float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
      for (int blk = 0; blk < nblk; ++blk)
        attention_block<HD, X3>(qa, qal, sKa + blk * AT_KV * RP, sVa + blk * AT_KV * RP, AT_Q * RP, blk * AT_KV, G, scale_log2e, lane,
                                o, m0, m1, l0, l1);
      const int b = item / heads, head = item - b * heads;
      attention_store<HD, X3>(o, l0, l1, out + (size_t)b * G * NH * D + (size_t)head * HD, q0, G, D, lane);
    }
    __syncthreads();   // every warp is done with this buffer: the next iteration prefetches into it
    buf ^= 1;
  }
}

static int num_sms_vit() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

template <int HD, bool X3>
static int attention_configure() {
  P3_CUDA(cudaFuncSetAttribute(attention_kernel<HD, X3>, cudaFuncAttributeMaxDynamicSharedMemorySize, attention_smem_bytes<HD, X3>()));
  P3_CUDA(cudaFuncSetAttribute(attention_small_kernel<HD, X3>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               attention_small_smem_bytes<HD, X3>()));
  return P3TOK_OK;
}

template <int HD, bool X3>
static void attention_launch(const __nv_bfloat16* qkv, int64_t B, int64_t G, int D, int heads, __nv_bfloat16* out, float scale_log2e,
                             bool small, cudaStream_t s) {
  if (small) {   // persistent, next item prefetched
    const int items = (int)(B * heads);
    const int slots = num_sms_vit() * attention_ctas_per_sm<HD, X3, true>();
    const unsigned nblocks = (unsigned)(items < slots ? items : slots);
    attention_small_kernel<HD, X3><<<nblocks, AT_THREADS, attention_small_smem_bytes<HD, X3>(), s>>>(qkv, out, (int)G, D, heads, items,
                                                                                                  scale_log2e);
  } else {
    dim3 grid((unsigned)((G + AT_Q - 1) / AT_Q), (unsigned)heads, (unsigned)B);
    attention_kernel<HD, X3><<<grid, AT_THREADS, attention_smem_bytes<HD, X3>(), s>>>(qkv, out, (int)G, D, scale_log2e);
  }
}

// x3 = false: qkv (B*G, 3D) -> out (B*G, D), bf16.  x3 = true: the split forms (B*G, 6D) -> (B*G, 2D).
static int attention_bf16(const __nv_bfloat16* qkv, int64_t B, int64_t G, int D, int heads, __nv_bfloat16* out, cudaStream_t s,
                          bool x3 = false) {
  P3_REQUIRE(heads > 0 && D % heads == 0, P3TOK_ERR_INVALID, "attention: D=%d not divisible by heads=%d", D, heads);
  const int hd = D / heads;
  P3_REQUIRE(hd == 32 || hd == 64, P3TOK_ERR_UNSUPPORTED, "attention: head dim %d (supported: 32, 64)", hd);
  P3_REQUIRE(B <= 65535 && heads <= 65535, P3TOK_ERR_UNSUPPORTED, "attention: B=%lld / heads=%d exceed the grid", (long long)B, heads);
  P3_REQUIRE(qkv && out, P3TOK_ERR_INVALID, "attention: null pointer");
  P3_REQUIRE((reinterpret_cast<uintptr_t>(qkv) & 15) == 0, P3TOK_ERR_UNSUPPORTED, "attention: qkv must be 16-byte aligned");
  if (B * G == 0) return P3TOK_OK;
  const float scale_log2e = (float)((1.0 / sqrt((double)hd)) * 1.4426950408889634);
  static thread_local bool configured[32] = {false};   // attention_kernel<64> needs 55 KB of dynamic shared memory
  int dev = 0;
  P3_CUDA(cudaGetDevice(&dev));
  if (dev < 32 && !configured[dev]) {
    int rc;
    if ((rc = attention_configure<32, false>()) || (rc = attention_configure<64, false>()) || (rc = attention_configure<32, true>()) ||
        (rc = attention_configure<64, true>()))
      return rc;
    configured[dev] = true;
  }
  static int small_on = -1;
  if (small_on < 0) { const char* e = getenv("P3TOK_ATTN_SMALL"); small_on = e ? atoi(e) : 1; }
  const bool small = small_on && G <= AT_Q;
  if (x3) {
    if (hd == 32) attention_launch<32, true>(qkv, B, G, D, heads, out, scale_log2e, small, s);
    else attention_launch<64, true>(qkv, B, G, D, heads, out, scale_log2e, small, s);
  } else {
    if (hd == 32) attention_launch<32, false>(qkv, B, G, D, heads, out, scale_log2e, small, s);
    else attention_launch<64, false>(qkv, B, G, D, heads, out, scale_log2e, small, s);
  }
  if (small) P3_LAUNCH_CHECK("attention_small_kernel");
  else P3_LAUNCH_CHECK("attention_kernel");
  return P3TOK_OK;
}

// ------------------------------------------------------------------------------------------------ orchestration
struct VitWs {
  int64_t a, qkv, h, total;
};
static int64_t pad64(int64_t n) { return (n + 63) / 64 * 64; }
// x3: every activation matrix is stored split, [hi | lo] at twice the width, and the [gelu | relu] matrix is padded to
// pad64(H + R) columns (the reduction length of fc2u)
static VitWs vit_layout(int64_t M, int64_t D, int64_t H, int64_t R, bool x3) {
  VitWs w;
  int64_t off = 0;
  const int64_t nh = x3 ? 2 : 1;
  auto take = [&](int64_t bytes) { int64_t o = off; off += align_up(bytes, 1024); return o; };
  w.a = take(M * D * 2 * nh);       // normalised rows / attention output
  w.qkv = take(M * 3 * D * 2 * nh);
  w.h = take(M * (x3 ? pad64(H + R) : H + R) * 2 * nh);      // [gelu(fc1) | relu(down)]
  w.total = off + 1024;
  return w;
}
int64_t apf_vit_workspace(int64_t B, int64_t G, int64_t D, int64_t H, int64_t R, bool x3) { return vit_layout(B * G, D, H, R, x3).total; }

// wide layers whose width is no multiple of 192 or 256 (fc1 + bottleneck: 1600): the least-padding rule of tc_linear would
// pick 64-column tiles; full-rate 256-column tiles with a partly empty last tile cost less
static int wide_tile(int n) { return (n > 1024 && n % 192 != 0 && n % 256 != 0) ? 256 : 0; }

// bf16-output GEMM whose N may exceed what one tc_linear launch stages (2048 columns): column slices of the weight
// matrix write column slices of the output (ViT-B: 3D = 2304, H + R = 3136).  Slices are multiples of 256 columns, so a
// GELU/ReLU boundary (gelu_cols, a multiple of 64) falls inside at most one slice and is passed relative to it.
// x3: A and out are split matrices, W the [W_hi | W_hi | W_lo] form (K = 3 x its reduction length); a slice writes hi at
// column n0 and lo at column N + n0 of out [M, 2N].  The split epilogue needs the 8-warp form.
static int linear_wide(const __nv_bfloat16* A, int64_t M, int K, const __nv_bfloat16* W, int N, const float* bias, int relu,
                       int gelu_cols, __nv_bfloat16* out, cudaStream_t s, bool x3 = false) {
  const int parts = (N + 2047) / 2048;
  const int per = parts == 1 ? N : ((N + parts - 1) / parts + 255) / 256 * 256;
  for (int n0 = 0; n0 < N; n0 += per) {
    const int n = N - n0 < per ? N - n0 : per;
    TcExtra ex;
    int do_relu = relu;
    if (gelu_cols > n0) {             // this slice starts with GELU columns
      ex.gelu = 1;
      ex.gelu_cols = gelu_cols - n0 < n ? gelu_cols - n0 : n;
      if (ex.gelu_cols == n) do_relu = 0;
    }
    ex.bn = wide_tile(n);
    if (x3) {
      ex.x3 = 1;
      ex.out_split = 1;
      ex.split_n = N;
    } else {
      ex.ldc = N;
      ex.epi16 = 1;
    }
    int rc = tc_linear_ex(A, M, K, W + (size_t)n0 * K, n, bias + n0, do_relu, ex, out + n0, nullptr, s);
    if (rc) return rc;
  }
  return P3TOK_OK;
}

}  // namespace p3tok

using namespace p3tok;

extern "C" int64_t p3tok_apf_vit_workspace_bytes(int64_t B, int64_t G, int64_t D, int64_t H, int64_t R) {
  if (B < 0 || G < 0 || D <= 0 || H <= 0 || R < 0) return -1;
  return apf_vit_workspace(B, G, D, H, R, false);
}

extern "C" int64_t p3tok_vit_x3_workspace_bytes(int64_t B, int64_t G, int64_t D, int64_t H, int64_t R) {
  if (B < 0 || G < 0 || D <= 0 || H <= 0 || R < 0) return -1;
  return apf_vit_workspace(B, G, D, H, R, true);
}

extern "C" int p3tok_layernorm_bf16(const float* x, int64_t M, int64_t D, float eps, const float* w, const float* b, void* out,
                                    void* stream) {
  P3_REQUIRE(M >= 0 && D > 0, P3TOK_ERR_INVALID, "layernorm: bad shape");
  return layernorm_bf16(const_cast<float*>(x), M, (int)D, eps, w, b, (__nv_bfloat16*)out, 1.f, as_stream(stream));
}

extern "C" int p3tok_attention_bf16(const void* qkv, int64_t B, int64_t G, int64_t D, int64_t heads, void* out, void* stream) {
  P3_REQUIRE(B >= 0 && G >= 0 && D > 0 && D % 8 == 0, P3TOK_ERR_INVALID, "attention: bad shape");
  return attention_bf16((const __nv_bfloat16*)qkv, B, G, (int)D, (int)heads, (__nv_bfloat16*)out, as_stream(stream));
}

extern "C" int p3tok_layernorm_split(const float* x, int64_t M, int64_t D, float eps, const float* w, const float* b, void* out,
                                     void* stream) {
  P3_REQUIRE(M >= 0 && D > 0, P3TOK_ERR_INVALID, "layernorm: bad shape");
  return layernorm_bf16(const_cast<float*>(x), M, (int)D, eps, w, b, (__nv_bfloat16*)out, 1.f, as_stream(stream), nullptr, nullptr, true);
}

extern "C" int p3tok_attention_x3(const void* qkv, int64_t B, int64_t G, int64_t D, int64_t heads, void* out, void* stream) {
  P3_REQUIRE(B >= 0 && G >= 0 && D > 0 && D % 8 == 0, P3TOK_ERR_INVALID, "attention: bad shape");
  return attention_bf16((const __nv_bfloat16*)qkv, B, G, (int)D, (int)heads, (__nv_bfloat16*)out, as_stream(stream), true);
}

extern "C" int p3tok_linear_bf16_ex(const void* A, int64_t M, int64_t K, const void* W, int64_t N, const float* bias, int act,
                                    int64_t gelu_cols, const float* residual, float res_mul, float out_scale, void* out_bf16,
                                    float* out_f32, void* stream) {
  P3_REQUIRE(M >= 0 && K > 0 && N > 0 && K < (1 << 24) && N < (1 << 24), P3TOK_ERR_INVALID, "linear_bf16_ex: bad shape");
  P3_REQUIRE(act >= 0 && act <= 3, P3TOK_ERR_INVALID, "linear_bf16_ex: act %d", act);
  if (M == 0) return P3TOK_OK;
  P3_REQUIRE(A && W && (out_bf16 || out_f32), P3TOK_ERR_INVALID, "linear_bf16_ex: null pointer");
  P3_REQUIRE(!residual || out_f32, P3TOK_ERR_INVALID, "linear_bf16_ex: a residual needs the f32 output");
  P3_REQUIRE(act != 3 || (gelu_cols > 0 && gelu_cols < N && gelu_cols % 64 == 0), P3TOK_ERR_INVALID,
             "linear_bf16_ex: act 3 needs 0 < gelu_cols < N, a multiple of 64");
  TcExtra ex;
  ex.gelu = act >= 2;
  ex.gelu_cols = act == 3 ? (int)gelu_cols : 0;
  ex.residual = residual;
  ex.res_mul = res_mul;
  ex.out_scale = residual ? out_scale : 1.f;
  ex.bn = wide_tile((int)N);
  return tc_linear_ex((const __nv_bfloat16*)A, M, (int)K, (const __nv_bfloat16*)W, (int)N, bias, act == 1 || act == 3, ex,
                      (__nv_bfloat16*)out_bf16, out_f32, as_stream(stream));
}

// The block stack in its two flavours:
//   APFViTLayer (apf_utils.py:236-293): R > 0 adapter columns ride in the fc1 / fc2 GEMMs, the layer output carries 2 x
//   timm Block (pix4point.py:254-255 `feats = blk(feats + pos_embed)`; timm 1.0.16 vision_transformer.Block, the dependency the
//              reference pins in requirements.txt): R = 0, plain residuals, the positional embedding re-added in front of
//              every block (fused into the block's first normalisation pass), a cls row at the head of every sequence.
// x3: the fp32-accurate form - split activations, [W_hi | W_hi | W_lo] weights, the bf16x3 attention (include/p3tok.h).
static int vit_forward(float* x, int64_t B, int64_t G, int64_t D, int64_t heads, int64_t H, int64_t R, const p3tok_vit_layer* layers,
                       int64_t n_layers, const float* pos, float res_mul, const float* final_norm_w, const float* final_norm_b,
                       float eps, float* out_norm, float* pooled_out, int pool_skip, void* workspace, int64_t workspace_bytes,
                       cudaStream_t s, bool x3) {
  P3_REQUIRE(B >= 0 && G >= 0 && D > 0 && H > 0 && R >= 0 && heads > 0 && n_layers >= 0, P3TOK_ERR_INVALID, "vit: bad shape");
  P3_REQUIRE(D % 8 == 0 && H % 64 == 0 && R % 8 == 0, P3TOK_ERR_UNSUPPORTED, "vit: D, R must be multiples of 8, H of 64");
  P3_REQUIRE(D <= 128 * LN_MAX_V4, P3TOK_ERR_UNSUPPORTED, "vit: D=%lld > %d", (long long)D, 128 * LN_MAX_V4);
  P3_REQUIRE(D % heads == 0 && (D / heads == 32 || D / heads == 64), P3TOK_ERR_UNSUPPORTED,
             "vit: head dim %lld (supported: 32, 64)", (long long)(D / heads));
  P3_REQUIRE(B * G < (1ll << 31) - 256, P3TOK_ERR_UNSUPPORTED, "vit: too many token rows");
  P3_REQUIRE(eps > 0.f && eps < 1.f, P3TOK_ERR_INVALID, "vit: ln_eps %g", (double)eps);
  P3_REQUIRE(pool_skip >= 0 && pool_skip < (G > 0 ? G : 1), P3TOK_ERR_INVALID, "vit: pool_skip %d", pool_skip);
  P3_REQUIRE(!x3 || D % 64 == 0, P3TOK_ERR_UNSUPPORTED, "vit(x3): D=%lld must be a multiple of 64", (long long)D);
  const int64_t M = B * G;
  if (M == 0) return P3TOK_OK;
  P3_REQUIRE(x && workspace && (n_layers == 0 || layers), P3TOK_ERR_INVALID, "vit: null pointer");
  P3_REQUIRE((!pooled_out && !out_norm) || (final_norm_w && final_norm_b), P3TOK_ERR_INVALID, "vit: outputs need the final norm");
  const VitWs L = vit_layout(M, D, H, R, x3);
  P3_REQUIRE(workspace_bytes >= L.total, P3TOK_ERR_WORKSPACE, "vit: workspace %lld < %lld bytes", (long long)workspace_bytes,
             (long long)L.total);
  uint8_t* ws = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 1023) & ~(uintptr_t)1023);
  __nv_bfloat16* a = reinterpret_cast<__nv_bfloat16*>(ws + L.a);
  __nv_bfloat16* qkv = reinterpret_cast<__nv_bfloat16*>(ws + L.qkv);
  __nv_bfloat16* h = reinterpret_cast<__nv_bfloat16*>(ws + L.h);
  const int HR = (int)(x3 ? pad64(H + R) : H + R);   // x3: fc1d rows / fc2u reduction padded with zeros (GELU(0) = ReLU(0) = 0)
  const int kx = x3 ? 3 : 1;                           // reduction length multiplier of the weight matrices
  int rc;
  for (int64_t li = 0; li < n_layers; ++li) {
    const p3tok_vit_layer& w = layers[li];
    P3_REQUIRE(w.qkv_w && w.qkv_b && w.proj_w && w.proj_b && w.fc1d_w && w.fc1d_b && w.fc2u_w && w.fc2u_b, P3TOK_ERR_INVALID,
               "vit: layer %lld has a null parameter", (long long)li);
    // attention branch: x (+= pos) ; x += proj(attention(norm1(x)))                       (apf_utils.py:279-283)
    if ((rc = layernorm_bf16(x, M, (int)D, eps, nullptr, nullptr, a, 1.f, s, pos, nullptr, x3))) return rc;
    if ((rc = linear_wide(a, M, kx * (int)D, (const __nv_bfloat16*)w.qkv_w, (int)(3 * D), w.qkv_b, 0, 0, qkv, s, x3))) return rc;
    if ((rc = attention_bf16(qkv, B, G, (int)D, (int)heads, a, s, x3))) return rc;
    {
      TcExtra ex;
      ex.residual = x; ex.res_mul = 1.f; ex.out_scale = 1.f; ex.epi16 = 1; ex.x3 = x3;
      if ((rc = tc_linear_ex(a, M, kx * (int)D, (const __nv_bfloat16*)w.proj_w, (int)D, w.proj_b, 0, ex, nullptr, x, s))) return rc;
    }
    // adapter + MLP on the same x: out = mlp(norm2(x)) + [scale * up(relu(down(adapter_norm(x)))) + x] + x   (:284-292)
    // the normalisation pass also leaves res_mul x behind (2 for APFViTLayer, 1 for a timm Block), so that the last GEMM,
    // like proj, only ADDS into the stream
    if ((rc = layernorm_bf16(x, M, (int)D, eps, nullptr, nullptr, a, res_mul, s, nullptr, nullptr, x3))) return rc;
    if ((rc = linear_wide(a, M, kx * (int)D, (const __nv_bfloat16*)w.fc1d_w, HR, w.fc1d_b, 1, (int)H, h, s, x3))) return rc;
    {
      TcExtra ex;
      ex.residual = x; ex.res_mul = 1.f; ex.out_scale = 1.f; ex.epi16 = 1; ex.x3 = x3;
      if ((rc = tc_linear_ex(h, M, kx * HR, (const __nv_bfloat16*)w.fc2u_w, (int)D, w.fc2u_b, 0, ex, nullptr, x, s))) return rc;
    }
  }
  if (out_norm) {
    if ((rc = layernorm_bf16(x, M, (int)D, eps, final_norm_w, final_norm_b, nullptr, 1.f, s, nullptr, out_norm))) return rc;
  }
  if (pooled_out) {
    norm_max_kernel<<<(unsigned)B, 256, 0, s>>>(x, (int)G, (int)D, eps, final_norm_w, final_norm_b, pooled_out, pool_skip);
    P3_LAUNCH_CHECK("norm_max_kernel");
  }
  return P3TOK_OK;
}

static int apf_vit_forward(float* x, int64_t B, int64_t G, int64_t D, int64_t heads, int64_t H, int64_t R, const p3tok_vit_layer* layers,
                           int64_t n_layers, const float* final_norm_w, const float* final_norm_b, float ln_eps, float* pooled_out,
                           void* workspace, int64_t workspace_bytes, void* stream, bool x3) {
  P3_REQUIRE(R > 0, P3TOK_ERR_INVALID, "apf_vit: the adapter bottleneck R must be positive (use p3tok_vit_forward for plain blocks)");
  return vit_forward(x, B, G, D, heads, H, R, layers, n_layers, nullptr, 2.f, final_norm_w, final_norm_b, ln_eps, nullptr, pooled_out, 0,
                     workspace, workspace_bytes, as_stream(stream), x3);
}

extern "C" int p3tok_apf_vit_forward(float* x, int64_t B, int64_t G, int64_t D, int64_t heads, int64_t H, int64_t R,
                                     const p3tok_vit_layer* layers, int64_t n_layers, const float* final_norm_w,
                                     const float* final_norm_b, float ln_eps, float* pooled_out, void* workspace,
                                     int64_t workspace_bytes, void* stream) {
  return apf_vit_forward(x, B, G, D, heads, H, R, layers, n_layers, final_norm_w, final_norm_b, ln_eps, pooled_out, workspace,
                         workspace_bytes, stream, false);
}

extern "C" int p3tok_apf_vit_forward_x3(float* x, int64_t B, int64_t G, int64_t D, int64_t heads, int64_t H, int64_t R,
                                        const p3tok_vit_layer* layers, int64_t n_layers, const float* final_norm_w,
                                        const float* final_norm_b, float ln_eps, float* pooled_out, void* workspace,
                                        int64_t workspace_bytes, void* stream) {
  return apf_vit_forward(x, B, G, D, heads, H, R, layers, n_layers, final_norm_w, final_norm_b, ln_eps, pooled_out, workspace,
                         workspace_bytes, stream, true);
}

extern "C" int p3tok_vit_forward(float* x, int64_t B, int64_t S, int64_t D, int64_t heads, int64_t H, const p3tok_vit_layer* layers,
                                 int64_t n_layers, const float* pos, const float* final_norm_w, const float* final_norm_b,
                                 float ln_eps, float* out_norm, float* pooled_out, int64_t pool_skip, void* workspace,
                                 int64_t workspace_bytes, void* stream) {
  return vit_forward(x, B, S, D, heads, H, 0, layers, n_layers, pos, 1.f, final_norm_w, final_norm_b, ln_eps, out_norm, pooled_out,
                     (int)pool_skip, workspace, workspace_bytes, as_stream(stream), false);
}

extern "C" int p3tok_vit_forward_x3(float* x, int64_t B, int64_t S, int64_t D, int64_t heads, int64_t H, const p3tok_vit_layer* layers,
                                    int64_t n_layers, const float* pos, const float* final_norm_w, const float* final_norm_b,
                                    float ln_eps, float* out_norm, float* pooled_out, int64_t pool_skip, void* workspace,
                                    int64_t workspace_bytes, void* stream) {
  return vit_forward(x, B, S, D, heads, H, 0, layers, n_layers, pos, 1.f, final_norm_w, final_norm_b, ln_eps, out_norm, pooled_out,
                     (int)pool_skip, workspace, workspace_bytes, as_stream(stream), true);
}
