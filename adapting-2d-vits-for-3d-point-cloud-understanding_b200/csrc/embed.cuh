// embed.cuh - internal interfaces shared by the patch-embedding paths.
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"

namespace p3tok {

// rows of the first layer's input, built from the fused-gather description (p3tok_rows).
// X: (ngroups_chunk*k, cin) f32 for groups [g_begin, g_begin+g_count) in OUTPUT (permuted) order.
int build_rows_f32(const p3tok_rows* rows, int64_t g_begin, int64_t g_count, float* X, cudaStream_t s);

int64_t patch_embed_f32_workspace(const p3tok_mlp* mlp, int64_t ngroups, int64_t k);
int patch_embed_f32(const p3tok_rows* rows, const p3tok_mlp* mlp, void* ws, int64_t ws_bytes, float* tokens,
                    cudaStream_t s);

int64_t patch_embed_bf16_workspace(const p3tok_mlp* mlp, int64_t ngroups, int64_t k);
// tokens: f32 (tokens_bf16 = 0) or bf16 (tokens_bf16 = 1), [ngroups, out_dim]
int patch_embed_bf16(const p3tok_rows* rows, const p3tok_mlp* mlp, void* ws, int64_t ws_bytes, void* tokens, int tokens_bf16,
                     cudaStream_t s);

// bf16x3 (fp32-accurate tensor-core) mode, embed_tc.cu
int64_t patch_embed_x3_workspace(const p3tok_mlp* mlp, int64_t ngroups, int64_t k);
int patch_embed_x3(const p3tok_rows* rows, const p3tok_mlp* mlp, void* ws, int64_t ws_bytes, float* tokens, cudaStream_t s);

// extra epilogue of tc_linear for the ViT blocks (vit.cu): GELU, fp32 residual stream, column-slice outputs
struct TcExtra {
  int gelu = 0;                    // exact GELU after the bias ...
  int gelu_cols = 0;               // ... on columns < gelu_cols (0 = all); `relu` then applies to the remaining columns
  int epi16 = 0;                   // 16 epilogue warps instead of 8 (bf16-only outputs; small-M GEMMs whose tiles are epilogue-bound)
  int bn = 0;                      // N-tile width override (multiple of 64, <= 256); 0 = least padding
  const float* residual = nullptr; // out_f32 = res_mul * residual + out_scale * value
  float res_mul = 1.f, out_scale = 1.f;
  int64_t ldc = 0;                 // row pitch of out_bf16 in elements (0 = N)
  int x3 = 0;                      // bf16x3 split operands: A [M, 2Kp] = [hi | lo], W [N, 3Kp] = [W_hi | W_hi | W_lo], K = 3Kp
  int out_split = 0;               // out_bf16 is [M, 2N] = [hi | lo] of the fp32 result ...
  int split_n = 0;                 // ... or a column slice of a [M, 2 split_n] split matrix: lo at column split_n + c (0 = N)
};
int tc_linear_ex(const __nv_bfloat16* A, int64_t M, int K, const __nv_bfloat16* W, int N, const float* bias, int relu,
                 const TcExtra& ex, __nv_bfloat16* out_bf16, float* out_f32, cudaStream_t s);

// vit.cu
int64_t apf_vit_workspace(int64_t B, int64_t G, int64_t D, int64_t H, int64_t R, bool x3);

// train.cu: the column-strip reductions (rows per strip from the shapes only) and their deterministic finish
bool ws_ok(const void* ws, int64_t ws_bytes, int64_t need);      // need bytes available, 16-byte aligned
int64_t strip_rows(int64_t M, int N);
int colsum_det_begin(const void* ws, int64_t ws_bytes, int64_t M, int64_t N, const char* who);
// out0[c] / out1[c] = sum in ascending strip order of part[0][strip][c] / part[1][strip][c], part = [2][strips][N] fp64
int strip_sum_f64(const double* part, int64_t M, int N, double* out0, double* out1, cudaStream_t s);

static inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

}  // namespace p3tok
