/*
 * p3tok.h - C ABI of the B200-native point-patch tokenizer (libp3tok.so).
 *
 * The reference (Irish-77/adapting-2D-ViTs-for-3D-point-cloud-understanding) has no FFI layer:
 * its boundary is plain Python callables (SURVEY.md 8b).  Every entry point below names the
 * reference callable it replaces (path:line relative to the reference tree); the Python side
 * (p3tok/ops.py) binds these with ctypes and registers them as torch custom ops.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless said otherwise;
 *   - the caller owns every buffer (inputs, outputs, workspace); the library allocates nothing
 *     persistent and keeps no state besides per-process kernel attributes;
 *   - work is enqueued on `stream` (a cudaStream_t passed as void*); the library never
 *     synchronises the device;
 *   - return value: P3TOK_OK or an error code; p3tok_last_error() (thread-local, host string)
 *     describes the last failure of the calling thread;
 *   - outputs are fully overwritten; row-major contiguous layouts as written in each comment.
 */
#ifndef P3TOK_H_
#define P3TOK_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define P3TOK_ABI_VERSION 3

#if defined(__GNUC__)
#define P3TOK_API __attribute__((visibility("default")))
#else
#define P3TOK_API
#endif

enum p3tok_status {
  P3TOK_OK = 0,
  P3TOK_ERR_INVALID = 1,     /* bad shape / null pointer / index out of contract */
  P3TOK_ERR_UNSUPPORTED = 2, /* valid request outside the implemented envelope (k, N, alignment) */
  P3TOK_ERR_CUDA = 3,        /* a CUDA call or launch failed; see p3tok_last_error() */
  P3TOK_ERR_WORKSPACE = 4    /* workspace too small; see the matching *_workspace_bytes() */
};

/* kNN distance flavour */
enum p3tok_knn_mode {
  P3TOK_KNN_APF_SQ = 0,   /* src/data/sampler.py:47-62  ((-2*dot)+|c|^2)+|p|^2, K=3 FMA chain */
  P3TOK_KNN_P4P_CDIST = 1 /* src/models/pix4point.py:87  cdist mm path: K=5 FMA chain, clamp, sqrt */
};

enum p3tok_dtype { P3TOK_F32 = 0, P3TOK_BF16 = 1, P3TOK_I32 = 2, P3TOK_I64 = 3,
                   P3TOK_BF16X3 = 4 /* precision mode / weight form of the fp32-accurate tensor-core path, see p3tok_patch_embed */ };

P3TOK_API int p3tok_abi_version(void);
P3TOK_API const char* p3tok_last_error(void);
/* number of kernels this library has launched in this process (diagnostic; bench.py reports it) */
P3TOK_API int64_t p3tok_kernel_launches(void);

/* ---- a1/a2: farthest point sampling ----------------------------------------------------------
 * Replaces furthest_point_sample (src/data/sampler.py:4-30) and farthest_point_sampling
 * (src/models/pix4point.py:8-53; its min(n_samples,N) clamp is applied by the Python wrapper).
 * x: B clouds x N points, point p of cloud b at x[(b*N+p)*pt_stride + 0..2] (pt_stride >= 3, so
 * an (B,N,4) xyz+height tensor is read in place, no .contiguous() copy).
 * start_idx: (B) int64, first pick per cloud (the reference draws torch.randint, sampler.py:20).
 * out_idx: (B,G) int64.  dist = ((dx*dx)+(dy*dy))+(dz*dz) unfused; argmax keeps the lowest index.
 * N <= 131072.  G > N repeats index 0 once the cloud is exhausted, like the reference.
 * One CTA per cloud up to 8192 points, a thread-block cluster per cloud beyond; the cluster size (<= 12288 points per
 * CTA) is chosen per launch so that all B clouds are resident at once (cudaOccupancyMaxActiveClusters). */
P3TOK_API int p3tok_fps(const float* x, int64_t B, int64_t N, int64_t pt_stride, const int64_t* start_idx,
              int64_t G, int64_t* out_idx, void* stream);

/* farthest_point_sampling (src/models/pix4point.py:8-53) on D-dimensional points, 1 <= D <= 16: the reference sums the
 * squared differences over ALL D coordinates (line 44, torch.sum(..., dim=2)).  x: point p of cloud b at
 * x[(b*N+p)*pt_stride + 0..D-1] (pt_stride >= D).  The D squares are added in the order torch's CPU sum kernel adds a
 * contiguous last dimension (four interleaved partial sums below 8 elements, 8 vector lanes from 8 on - spelled out in
 * csrc/fps_nd.cu and oracle/p3tok_oracle.c, checked bit for bit against torch.sum), so the picks equal the reference's for
 * every D; for D <= 3 they equal p3tok_fps's.  min_dist_ws: (B,N) f32 scratch owned by the caller (the running minima;
 * contents on entry are ignored).  One CTA per cloud, any N < 2^31; the xyz case belongs on p3tok_fps. */
P3TOK_API int p3tok_fps_nd(const float* x, int64_t B, int64_t N, int64_t D, int64_t pt_stride, const int64_t* start_idx,
                 int64_t G, int64_t* out_idx, float* min_dist_ws, void* stream);

/* ---- a5: index_points (src/data/sampler.py:77-94) / torch.gather of centres (pix4point.py:176)
 * x (B,N,C) f32, idx (B,S) int64 -> out (B,S,C).  S may be G or G*k. */
P3TOK_API int p3tok_gather_points(const float* x, int64_t B, int64_t N, int64_t C, const int64_t* idx,
                        int64_t S, float* out, void* stream);

/* ---- a3/a4: kNN query -----------------------------------------------------------------------
 * Replaces _square_distance + knn_point (src/data/sampler.py:47-75) and the cdist+topk inside
 * group_knn (src/models/pix4point.py:79-89).  centres: (B,G,3) contiguous query points.
 * idx_out: (B,G,k) of idx_dtype (P3TOK_I64 for the APF flavour, P3TOK_I32 for Pix4Point's
 * `.int()`), ascending by (distance, index) - the canonical instance of torch.topk's
 * implementation-defined tie order.  dist_out: optional (B,G,k) f32 distances (may be NULL).
 * 1 <= k <= 128, k <= N. */
P3TOK_API int p3tok_knn(const float* x, int64_t B, int64_t N, int64_t pt_stride, const float* centres,
              int64_t G, int64_t k, int mode, void* idx_out, int idx_dtype, float* dist_out,
              void* stream);

/* Spatially sorted variant of p3tok_knn for clouds of at most 131072 points (same contract, same results bit for bit):
 * a preparation kernel sorts every cloud along a Z-order curve into `workspace` (clouds beyond 8192 points as segments of
 * <= 8192 consecutive points, each sorted on its own), then one warp per centre evaluates only the 32-point blocks whose
 * bounding box can still contain one of the k nearest neighbours.
 * p3tok_knn_workspace_bytes returns the scratch size in bytes, or 0 when the variant does not apply (N > 131072). */
P3TOK_API int64_t p3tok_knn_workspace_bytes(int64_t B, int64_t N);
P3TOK_API int p3tok_knn_sorted(const float* x, int64_t B, int64_t N, int64_t pt_stride, const float* centres,
                     int64_t G, int64_t k, int mode, void* idx_out, int idx_dtype, float* dist_out,
                     void* workspace, int64_t workspace_bytes, void* stream);

/* The two halves of p3tok_knn_sorted as separate calls.  p3tok_knn_prepare depends only on the clouds, so a caller can
 * enqueue it on a second stream while p3tok_fps picks the centres on the first (p3tok/modules.py does; the two kernels
 * share the SMs), then p3tok_knn_query - after a stream dependency on the preparation - answers the query from the
 * workspace.  Same contract and results as p3tok_knn / p3tok_knn_sorted. */
P3TOK_API int p3tok_knn_prepare(const float* x, int64_t B, int64_t N, int64_t pt_stride, void* workspace,
                      int64_t workspace_bytes, void* stream);
P3TOK_API int p3tok_knn_query(const void* workspace, int64_t workspace_bytes, int64_t B, int64_t N, const float* centres,
                    int64_t G, int64_t k, int mode, void* idx_out, int idx_dtype, float* dist_out, void* stream);

/* _square_distance materialised (src/data/sampler.py:47-62): src (B,S,3) contiguous, dst: point n of cloud b at
 * dst[(b*N+n)*dst_stride + 0..2] -> out (B,S,N) f32 = ((-2*dot) + |src|^2) + |dst|^2 with the K=3 FMA chain of
 * P3TOK_KNN_APF_SQ (bit-exact restatement of the reference's matmul form; values may be slightly negative, no clamp).
 * The tokenizer itself never materialises this matrix (p3tok_knn*); B*S*N < 2^40. */
P3TOK_API int p3tok_square_distance(const float* src, int64_t B, int64_t S, const float* dst, int64_t N,
                          int64_t dst_stride, float* out, void* stream);

/* ---- a7: Morton order of the centres (src/models/apf_utils.py:66-104, resolution 1024) -------
 * centres (B,G,3) -> perm (B,G) int64 = stable ascending argsort of the 30-bit Z-order code;
 * codes_out optional (B,G) int64.  G <= 8192. */
P3TOK_API int p3tok_morton_order(const float* centres, int64_t B, int64_t G, int64_t* perm,
                       int64_t* codes_out, void* stream);

/* ---- a6: Group.forward materialised (src/models/apf.py:52-112) --------------------------------
 * x (B,N,C) f32 contiguous; fps_idx (B,G) i64; knn_idx (B,G,k) i64; perm (B,G) i64 or NULL.
 * neigh (B,G,k,2C) = [x[nbr]-x[centre] || x[centre]], center (B,G,3) = xyz of the centre, both
 * in the permuted group order (output group j = input group perm[b,j]). */
P3TOK_API int p3tok_apf_group(const float* x, int64_t B, int64_t N, int64_t C, const int64_t* fps_idx,
                    const int64_t* knn_idx, const int64_t* perm, int64_t G, int64_t k,
                    float* neigh, float* center, void* stream);

/* ---- a4 (gather half of group_knn, src/models/pix4point.py:92-102) ---------------------------
 * pnts (B,N,3), feats (B,N,D) channel-last, idx (B,G,k) int32 -> grouped_pnts (B,G,k,3),
 * grouped_feats (B,G,k,D).  Absolute coordinates: Pix4Point does not centre-normalise. */
P3TOK_API int p3tok_group_gather(const float* pnts, const float* feats, int64_t B, int64_t N, int64_t D,
                       const int32_t* idx, int64_t G, int64_t k, float* grouped_pnts,
                       float* grouped_feats, void* stream);

/* ---- a8/a10: mini-PointNet patch embedding ---------------------------------------------------
 * One descriptor covers both model families (eval-mode BatchNorm already folded into the
 * weights by the host, p3tok/fold.py):
 *   rows X (ngroups*k, cin)
 *   -> n_pre per-point layers  h = act(W_i h + b_i)           (APF: 3, P3Embed: 1 [conv1 folded])
 *   -> g = max over the k rows of a group                     (apf.py:160 / pix4point.py:185)
 *   -> h = relu(W_mid_g g + W_mid_f h + b_mid)                (concat layer split, apf.py:162-163)
 *   -> o = act_out(W_out h + b_out);  token = max over k      (apf.py:167 / pix4point.py:188)
 * Matrices are row-major [out, in] in `wdtype` (P3TOK_F32 for the fp32 path, P3TOK_BF16 for the
 * tcgen05 path); biases are always f32. */
typedef struct p3tok_mlp {
  int32_t cin;
  int32_t n_pre;
  int32_t pre_dim[4];
  int32_t pre_relu[4];
  int32_t mid_dim;
  int32_t out_dim;
  int32_t out_relu;
  int32_t wdtype;
  const void* w_pre[4];
  const float* b_pre[4];
  const void* w_mid_g;
  const void* w_mid_f;
  const float* b_mid;
  const void* w_out;
  const float* b_out;
} p3tok_mlp;

/* Where the rows come from (fused gather, no (B,G,k,2C) tensor in HBM):
 *   kind 0 (APF):  row = [x[b,nbr,:C]-x[b,ctr,:C] || x[b,ctr,:C]]  (cin = 2C), groups emitted in
 *                  `perm` order when perm != NULL (Morton order as the OUTPUT row, apf.py:99-110)
 *   kind 1 (P4P):  row = [pnts[b,nbr,:3] || feats[b,nbr,:D]]        (cin = 3+D)
 *   kind 2 (rows): X given directly as (ngroups*k, cin) f32 in `x` (Encoder.forward on a
 *                  materialised (B,G,k,2C) tensor, apf.py:171-181) */
typedef struct p3tok_rows {
  int32_t kind;
  int32_t C;              /* channels of x (APF: 3 or 4; P4P: 3) */
  int32_t D;              /* feature channels (P4P) */
  int32_t idx_dtype;      /* dtype of knn_idx: P3TOK_I64 or P3TOK_I32 */
  int64_t B, N, G, k;
  const float* x;         /* (B,N,C) or rows */
  const float* feats;     /* (B,N,D) channel-last, P4P only */
  const int64_t* ctr_idx; /* (B,G) APF only */
  const void* knn_idx;    /* (B,G,k) */
  const int64_t* perm;    /* (B,G) or NULL */
} p3tok_rows;

/* Workspace size in bytes for p3tok_patch_embed with these shapes (host computation only). */
P3TOK_API int64_t p3tok_patch_embed_workspace_bytes(const p3tok_mlp* mlp, int64_t ngroups, int64_t k,
                                          int precision);

/* Replaces Encoder.forward (src/models/apf.py:145-181) and the conv/pool half of one
 * P3Embed.forward iteration (src/models/pix4point.py:179-188).
 * precision: P3TOK_F32 (CUDA-core FFMA, fp32 accumulate; rtol 1e-4 contract), P3TOK_BF16 (tcgen05 tensor cores, bf16
 * operands, fp32 accumulate in TMEM; rtol 1e-2 contract) or P3TOK_BF16X3 - the rtol 1e-4 contract ON the tensor cores:
 * every operand is carried as hi + lo bf16 halves and a.w = a_hi.w_hi + a_lo.w_hi + a_hi.w_lo accumulates in fp32; the
 * descriptor then holds (wdtype P3TOK_BF16X3) a first layer with cin <= 16 as f32 [out, cin] and every other matrix as
 * bf16 [out, 3 * pad64(in)] = [W_hi | W_hi | W_lo] (p3tok/fold.py prepares them); all widths multiples of 64.
 * tokens: (B*G, out_dim) of tokens_dtype, group order as described in p3tok_rows.  tokens_dtype: P3TOK_F32 (the
 * reference's dtype) or, with precision P3TOK_BF16 only, P3TOK_BF16 - the patch max is rounded once, in the epilogue
 * that produces it, so a bf16 consumer (the ViT blocks) or a host reader moves half the bytes. */
P3TOK_API int p3tok_patch_embed(const p3tok_rows* rows, const p3tok_mlp* mlp, int precision, int tokens_dtype,
                      void* workspace, int64_t workspace_bytes, void* tokens, void* stream);

/* ---- building blocks exported for tests and for the "next" rows (pix4point.py:245 proj) -------
 * C[M,N] = act(A[M,K] W[N,K]^T + bias[N] + gbias[m / rows_per_group, N]) in fp32 on CUDA cores.
 * gbias may be NULL. */
P3TOK_API int p3tok_linear_f32(const float* A, int64_t M, int64_t K, const float* W, int64_t N,
                     const float* bias, const float* gbias, int64_t rows_per_group, int relu,
                     float* C, void* stream);

/* Tensor-core version (tcgen05, bf16 operands A[M,K], W[N,K]; K % 8 == 0, N % 8 == 0; fp32 accumulate).
 * Any subset of the outputs may be requested: out_bf16 [M,N] bf16, out_f32 [M,N] f32, out_max32
 * [ceil(M/32), N] f32 = max over each 32 consecutive rows (the fused patch max-pool for k = 32). */
P3TOK_API int p3tok_linear_bf16(const void* A, int64_t M, int64_t K, const void* W, int64_t N, const float* bias,
                      const float* gbias, int64_t rows_per_group, int relu, void* out_bf16,
                      float* out_f32, float* out_max32, void* stream);

/* fp32 in, fp32 out, on the tensor cores: C[M,N] = act(A[M,K] W[N,K]^T + bias + gbias) with both operands split on the fly
 * into hi = bf16(v), lo = bf16(v - hi) and a w = a_hi w_hi + a_lo w_hi + a_hi w_lo evaluated as ONE tcgen05 GEMM over the
 * three-fold reduction length (fp32 accumulate; ~1e-5 of max against float64).  N % 8 == 0, N <= 2048; relu 0 / 1.
 * workspace >= p3tok_linear_x3_workspace_bytes(M, K, N).  Used by the training path when P3TOK_TRAIN_TC=1. */
P3TOK_API int64_t p3tok_linear_x3_workspace_bytes(int64_t M, int64_t K, int64_t N);
P3TOK_API int p3tok_linear_x3_f32(const float* A, int64_t M, int64_t K, const float* W, int64_t N, const float* bias,
                        const float* gbias, int64_t rows_per_group, int relu, float* C, void* workspace,
                        int64_t workspace_bytes, void* stream);

/* ---- "next" row 1 (SURVEY 8f): Pix4Point token head, src/models/pix4point.py:213-218 and 245-252 -----------
 * feats_out (B,1+G,E): row 0 = cls_token, rows 1.. = proj(tokens) with proj = Linear(W->E);
 * pos_out   (B,1+G,E): row 0 = cls_pos,   rows 1.. = Linear(H->E)(GELU(Linear(3->H)(centres))) (exact erf GELU).
 * tokens (B,G,W) channel-last, centres (B,G,3); weights row-major [out,in] f32; hidden_ws: caller scratch of
 * B*G*H floats.  fp32 on CUDA cores. */
P3TOK_API int p3tok_token_head_f32(const float* tokens, const float* centres, int64_t B, int64_t G, int64_t W, int64_t E,
                         int64_t H, const float* proj_w, const float* proj_b, const float* pos_w1,
                         const float* pos_b1, const float* pos_w2, const float* pos_b2,
                         const float* cls_token, const float* cls_pos, float* hidden_ws, float* feats_out,
                         float* pos_out, void* stream);

/* ---- "next" row 3 (SURVEY 8f): the ViT block stack consuming the tokens ------------------------------------
 * One APFViTLayer (src/models/apf_utils.py:236-293): x += proj(attention(norm1(x)));  out = mlp(norm2(x)) +
 * adapter(x) + x with adapter(x) = scale * up(relu(down(adapter_norm(x)))) + x (apf_utils.py:197-233) - so the
 * layer output carries 2*x, as the reference computes it.  Attention is the explicit softmax(q k^T / sqrt(hd)) v of
 * AttentionLayer (apf_utils.py:133-160); mlp = fc1 -> exact (erf) GELU -> fc2 (timm Mlp).  Eval mode: DropPath and
 * dropout are the identity.  ln_eps: the eps of norm1 / norm2 / adapter_norm / encoder_norm (nn.LayerNorm default 1e-5).
 * The descriptor holds the layer FOLDED by the host (p3tok/apf_model.py::fold_vit_layer, like the BatchNorm folding of
 * p3tok_mlp), matrices row-major [out,in] bf16, biases f32; g1/b1, g2/b2, ga/ba = affine of norm1, norm2, adapter_norm:
 *   qkv_w  [3D, D]   = qkv.weight * diag(g1)                       qkv_b  = qkv.bias + qkv.weight b1
 *   proj_w [D, D]    = proj.weight                                 proj_b = proj.bias
 *   fc1d_w [H+R, D]  = [fc1.weight diag(g2) ; down_proj.weight diag(ga)]
 *   fc1d_b [H+R]     = [fc1.bias + fc1.weight b2 ; down_proj.bias + down_proj.weight ba]
 *   fc2u_w [D, H+R]  = [fc2.weight | scale * up_proj.weight]       fc2u_b = fc2.bias + scale * up_proj.bias */
typedef struct p3tok_vit_layer {
  const void* qkv_w; const float* qkv_b;
  const void* proj_w; const float* proj_b;
  const void* fc1d_w; const float* fc1d_b;
  const void* fc2u_w; const float* fc2u_b;
} p3tok_vit_layer;

/* Workspace bytes for p3tok_apf_vit_forward (host computation only). */
P3TOK_API int64_t p3tok_apf_vit_workspace_bytes(int64_t B, int64_t G, int64_t D, int64_t H, int64_t R);

/* Replaces the block loop + encoder_norm + token max of AdaptPointFormer.forward (src/models/apf.py:361-366).
 * x (B,G,D) f32: the tokens; overwritten IN PLACE by the output of the last block (the fp32 residual stream).
 * layers: HOST array of n_layers descriptors (device pointers inside).  heads: D/heads must be 32 or 64.
 * H = mlp hidden width (multiple of 64), R = adapter bottleneck (multiple of 8).
 * final_norm_w/b [D] + pooled_out (B,D) f32: pooled = max over the G tokens of LayerNorm(x) (apf.py:364-366);
 * pass pooled_out = NULL to skip.  GEMMs on tcgen05 (bf16 operands, fp32 accumulate), attention on bf16 mma with
 * fp32 softmax; the bf16 contract of the tokenizer (rtol 1e-2) holds after 12 layers, see tests/test_gpu_vit.py. */
P3TOK_API int p3tok_apf_vit_forward(float* x, int64_t B, int64_t G, int64_t D, int64_t heads, int64_t H, int64_t R,
                          const p3tok_vit_layer* layers, int64_t n_layers, const float* final_norm_w,
                          const float* final_norm_b, float ln_eps, float* pooled_out, void* workspace,
                          int64_t workspace_bytes, void* stream);

/* The same stack for plain pre-norm ViT blocks - the timm `Block`s Pix4Point runs (src/models/pix4point.py:248-256; timm
 * 1.0.16 is the reference's pinned dependency, requirements.txt): x = x + proj(attn(norm1(x))); x = x + fc2(gelu(fc1(norm2(x)))).
 * x (B,S,D) f32 = [cls ; tokens], updated in place.  pos (B,S,D) f32 or NULL: added to x in front of EVERY block (line 255
 * `feats = blk(feats + pos_embed)`; fused into the block's first normalisation pass).  Layers use the same folded descriptor
 * with no adapter columns: fc1d_w [H, D] = fc1.weight diag(g2), fc2u_w [D, H] = fc2.weight.
 * out_norm (B,S,D) f32 or NULL: LayerNorm(x; final_norm) - what PointViT.forward returns (line 256);
 * pooled_out (B,D) f32 or NULL: max over the rows s >= pool_skip of LayerNorm(x) (forward_cls_feat's 'max' feature over the
 * tokens without the cls row: pool_skip = 1).  Workspace: p3tok_apf_vit_workspace_bytes(B, S, D, H, 0). */
P3TOK_API int p3tok_vit_forward(float* x, int64_t B, int64_t S, int64_t D, int64_t heads, int64_t H,
                      const p3tok_vit_layer* layers, int64_t n_layers, const float* pos, const float* final_norm_w,
                      const float* final_norm_b, float ln_eps, float* out_norm, float* pooled_out, int64_t pool_skip,
                      void* workspace, int64_t workspace_bytes, void* stream);

/* The fp32-accurate forms of the two stacks above (bf16x3 on the tensor cores, the rtol 1e-4 contract of the fp32 tokenizer):
 * every GEMM operand is a split pair v = hi + lo with hi = bf16(v), lo = bf16(v - hi), and a product is evaluated as
 * a_hi.b_hi + a_lo.b_hi + a_hi.b_lo on tcgen05 (GEMMs) or mma.sync (attention: scores and P V; softmax in fp32).  Same
 * arguments and the same p3tok_vit_layer descriptor, whose matrices then hold the x3 form, with Dp = D (D must be a multiple
 * of 64) and HRp = pad64(H + R) (p3tok_vit_forward_x3: R = 0):
 *   qkv_w  [3D, 3D]     proj_w [D, 3D]     fc1d_w [HRp, 3D]     fc2u_w [D, 3 HRp]       (bf16)
 *   each W [out, in] of the bf16 layout above stored as [W_hi | W_hi | W_lo], in padded to a multiple of 64 with zeros
 *   (p3tok/fold.py split_x3, from the float64 folded matrix); fc1d_w's rows H + R .. HRp - 1 are zero and fc1d_b has HRp
 *   entries (zero past H + R): GELU(0) = ReLU(0) = 0, so the padding adds nothing.  Biases f32.
 * Workspace: p3tok_vit_x3_workspace_bytes(B, G, D, H, R) (p3tok_vit_forward_x3: R = 0). */
P3TOK_API int64_t p3tok_vit_x3_workspace_bytes(int64_t B, int64_t G, int64_t D, int64_t H, int64_t R);
P3TOK_API int p3tok_apf_vit_forward_x3(float* x, int64_t B, int64_t G, int64_t D, int64_t heads, int64_t H, int64_t R,
                             const p3tok_vit_layer* layers, int64_t n_layers, const float* final_norm_w,
                             const float* final_norm_b, float ln_eps, float* pooled_out, void* workspace,
                             int64_t workspace_bytes, void* stream);
P3TOK_API int p3tok_vit_forward_x3(float* x, int64_t B, int64_t S, int64_t D, int64_t heads, int64_t H,
                         const p3tok_vit_layer* layers, int64_t n_layers, const float* pos, const float* final_norm_w,
                         const float* final_norm_b, float ln_eps, float* out_norm, float* pooled_out, int64_t pool_skip,
                         void* workspace, int64_t workspace_bytes, void* stream);

/* Building blocks of the above, exported for tests.
 * p3tok_layernorm_bf16: out = bf16(LN(x; w, b)) over the rows of x (M,D) f32; w = b = NULL: normalisation only.
 * p3tok_attention_bf16: qkv (B*G, 3D) bf16 laid out as AttentionLayer's reshape(B,N,3,heads,hd) -> out (B*G, D) bf16. */
P3TOK_API int p3tok_layernorm_bf16(const float* x, int64_t M, int64_t D, float eps, const float* w, const float* b,
                         void* out, void* stream);
P3TOK_API int p3tok_attention_bf16(const void* qkv, int64_t B, int64_t G, int64_t D, int64_t heads, void* out, void* stream);
/* Their split forms (the building blocks of the _x3 stacks), exported for tests:
 * p3tok_layernorm_split: out (M, 2D) bf16 = [hi | lo] of LN(x; w, b);
 * p3tok_attention_x3: qkv (B*G, 6D) bf16 = [hi | lo] of the qkv matrix above (lo of column c at column 3D + c) -> out
 * (B*G, 2D) bf16 = [hi | lo] of softmax(q k^T / sqrt(hd)) v. */
P3TOK_API int p3tok_layernorm_split(const float* x, int64_t M, int64_t D, float eps, const float* w, const float* b,
                          void* out, void* stream);
P3TOK_API int p3tok_attention_x3(const void* qkv, int64_t B, int64_t G, int64_t D, int64_t heads, void* out, void* stream);
/* p3tok_linear_bf16 with the ViT epilogues: act 0 none / 1 ReLU / 2 exact GELU / 3 GELU on columns < gelu_cols and ReLU on
 * the rest; then, if residual != NULL, out_f32 = res_mul * residual + out_scale * act(A W^T + bias) (residual may alias
 * out_f32).  N <= 2048 per call. */
P3TOK_API int p3tok_linear_bf16_ex(const void* A, int64_t M, int64_t K, const void* W, int64_t N, const float* bias, int act,
                         int64_t gelu_cols, const float* residual, float res_mul, float out_scale, void* out_bf16,
                         float* out_f32, void* stream);

/* ---- "next" row 4 (SURVEY 8f): training-mode building blocks ------------------------------------------------------
 * The reference trains the tokenizer (src/models/apf.py:335-346 keeps the "encoder" parameters trainable; Pix4Point
 * trains everything): nn.BatchNorm1d/2d in TRAIN mode (batch statistics, biased variance for the normalisation, running
 * estimates updated with the unbiased one; apf.py:129-143, pix4point.py:135-156) and autograd through Encoder.forward
 * (apf.py:145-181) / P3Embed.forward (pix4point.py:171-189).  fp32 on CUDA cores, fp64 accumulation of per-channel sums.
 * The host side (p3tok/train.py) strings these together as torch.autograd.Functions; dX = dY W reuses p3tok_linear_f32
 * with the transposed matrix.  All matrices row-major; "M" = rows (groups * k), "N" = channels. */
/* dW[N,K] (+)= dY[M,N]^T X[M,K]  (weight gradient of Y = X W^T); accumulate = 0 overwrites. */
P3TOK_API int p3tok_linear_tn_f32(const float* dY, const float* X, int64_t M, int64_t N, int64_t K, float* dW, int accumulate,
                        void* stream);
/* sum[c] = sum_m X[m,c], sumsq[c] = sum_m X[m,c]^2 (both overwritten): the batch statistics of a BatchNorm; a sharded
 * batch all-reduces these two vectors (and the row count) before the mean / variance are formed (SyncBN). */
P3TOK_API int p3tok_colstats_f32(const float* X, int64_t M, int64_t N, double* sum, double* sumsq, void* stream);
/* Y = act(gamma * (Z - mean) * rstd + beta), act = ReLU if relu else identity (nn.BatchNorm forward in train mode). */
P3TOK_API int p3tok_bn_act_f32(const float* Z, int64_t M, int64_t N, const float* mean, const float* rstd, const float* gamma,
                     const float* beta, int relu, float* Y, void* stream);
/* Backward of the above for dY = dL/dY: with dy' = dY * [Y > 0] (ReLU) and xhat = (Z - mean) rstd,
 *   stats: s1[c] = sum_m dy' (= dbeta), s2[c] = sum_m dy' xhat (= dgamma)   (overwritten; all-reduced when sharded)
 *   apply: dZ = gamma rstd (dy' - s1/count - xhat s2/count),  count = rows of the whole (global) batch. */
P3TOK_API int p3tok_bn_bwd_stats_f32(const float* dY, const float* Z, int64_t M, int64_t N, const float* mean, const float* rstd,
                           const float* gamma, const float* beta, int relu, double* s1, double* s2, void* stream);
P3TOK_API int p3tok_bn_bwd_apply_f32(const float* dY, const float* Z, int64_t M, int64_t N, int64_t count, const float* mean,
                           const float* rstd, const float* gamma, const float* beta, int relu, const double* s1,
                           const double* s2, float* dZ, void* stream);
/* torch.max over the k rows of a group with its index (first maximum): X [G*k, C] -> out [G, C], arg [G, C] in [0,k). */
P3TOK_API int p3tok_group_max_arg_f32(const float* X, int64_t G, int64_t k, int64_t C, float* out, int32_t* arg, void* stream);
/* its backward: dX[(g*k + r), c] (+)= (r == arg[g,c]) ? dOut[g,c] : 0  (accumulate = 0 overwrites every element). */
P3TOK_API int p3tok_group_max_bwd_f32(const float* dOut, const int32_t* arg, int64_t G, int64_t k, int64_t C, int accumulate,
                            float* dX, void* stream);
/* out[g,c] = sum over the k rows of group g (the gradient the expanded global feature collects, apf.py:162). */
P3TOK_API int p3tok_group_sum_f32(const float* X, int64_t G, int64_t k, int64_t C, float* out, void* stream);
/* Gradient of the kNN gather of group_knn (pix4point.py:92-102): dRows (B,G,k,3+D), idx (B,G,k) int32 ->
 * dP (B,N,3) += xyz part, dF (B,N,D) += feature part (atomic adds; either output may be NULL). */
P3TOK_API int p3tok_scatter_rows_add_f32(const float* dRows, const int32_t* idx, int64_t B, int64_t N, int64_t G, int64_t k,
                               int64_t D, float* dP, float* dF, void* stream);
/* The gathered row matrix a p3tok_rows descriptor (kind 0 or 1) stands for: X (B*G*k, cin) f32 - the training path's
 * input (the inference path never materialises it). */
P3TOK_API int p3tok_build_rows_f32(const p3tok_rows* rows, float* X, void* stream);

/* ---- gradients with respect to the input points (adversarial examples, saliency) -------------------------------------------
 * Both functions ACCUMULATE into dX (the caller zeroes it) with fp32 atomic adds, like p3tok_scatter_rows_add_f32 and torch's
 * own CUDA index backward: the result is reproducible to rounding, not bit for bit (the order of the adds varies; the *_det_f32
 * versions further down are bit-reproducible). */
/* Adjoint of p3tok_build_rows_f32 for kind 0 (APF): dRows (B*G*k, 2C) in the rows' output order (group j = input group
 * perm[b,j]) -> dX (B,N,C) += d rel at x[b,nbr] and sum over the group's k rows of (d ctr - d rel) at x[b,ctr].  rows->x is not
 * read; knn_idx is int64 or int32 (rows->idx_dtype). */
P3TOK_API int p3tok_apf_rows_bwd_f32(const p3tok_rows* rows, const float* dRows, float* dX, void* stream);
/* Adjoint of p3tok_gather_points: dOut (B,S,C), idx (B,S) int64 -> dX (B,N,C) += dOut at the gathered rows. */
P3TOK_API int p3tok_gather_points_bwd_f32(const float* dOut, int64_t B, int64_t N, int64_t C, const int64_t* idx, int64_t S,
                                          float* dX, void* stream);

/* ---- deterministic reductions (for torch.use_deterministic_algorithms) ----------------------------------------------------
 * The functions above that finish their sums with floating-point atomics (p3tok_linear_tn_f32, p3tok_colstats_f32,
 * p3tok_bn_bwd_stats_f32, p3tok_ln_param_grad_f32, p3tok_scatter_rows_add_f32, p3tok_apf_rows_bwd_f32,
 * p3tok_gather_points_bwd_f32) round in the order the CTAs arrive.  Each *_det_f32 below computes the same quantity with the same
 * arguments plus a caller-owned workspace (16-byte aligned, at least the matching *_workspace_bytes(); the library allocates
 * nothing), and its result is a function of the inputs and shapes only: bit-identical across calls, streams, concurrent load and
 * processes.  Launch geometry comes from the shapes, never from a device query.
 *
 * Ordered reductions.  p3tok_linear_tn_det_f32 splits M into the slices p3tok_linear_tn_f32 uses (rows per slice: a multiple of
 * 256 such that ceil(148*4 / (ceil(N/64) ceil(K/64))) slices cover M); slice z stores its fp32 partial dY_z^T X_z to
 * workspace[z][N][K], and dW = fp32(sum over z ascending, in fp64) (+ the old dW once when accumulate).  The three column-strip
 * reductions store the fp64 partials of strip y (the strips of the *_f32 versions) to workspace[0][y][N] (sum / s1 / dgamma) and
 * workspace[1][y][N] (sumsq / s2 / dbeta) and add the strips in ascending order in fp64.
 *
 * Fixed-point scatters.  Per cloud b, m_b = the largest finite |contribution| and K = a bound on the contributions one destination
 * receives (gather_points: S; apf_rows: G*(k+1); scatter_rows: G*k), s_b = 61 - ceil(log2 K) - e with m_b < 2^e (frexp; s_b = 0
 * when m_b = 0).  Each contribution v adds rint(v 2^s_b) to an int64 accumulator (one per call, shared by all of the call's
 * outputs; the APF centre term sum_n (d ctr - d rel), summed in fp32 in ascending n, is one contribution), and dX +=
 * fp32(sum) 2^-s_b.  Non-finite contributions follow IEEE addition per destination (any NaN or +inf with -inf: NaN; otherwise the
 * infinity).  A cloud's result does not depend on the other clouds of the batch. */
P3TOK_API int64_t p3tok_linear_tn_det_workspace_bytes(int64_t M, int64_t N, int64_t K);
P3TOK_API int p3tok_linear_tn_det_f32(const float* dY, const float* X, int64_t M, int64_t N, int64_t K, float* dW, int accumulate,
                                      void* workspace, int64_t workspace_bytes, void* stream);
/* workspace of p3tok_colstats_det_f32, p3tok_bn_bwd_stats_det_f32 and p3tok_ln_param_grad_det_f32 (N = D) */
P3TOK_API int64_t p3tok_colsum_det_workspace_bytes(int64_t M, int64_t N);
P3TOK_API int p3tok_colstats_det_f32(const float* X, int64_t M, int64_t N, double* sum, double* sumsq, void* workspace,
                                     int64_t workspace_bytes, void* stream);
P3TOK_API int p3tok_bn_bwd_stats_det_f32(const float* dY, const float* Z, int64_t M, int64_t N, const float* mean, const float* rstd,
                                         const float* gamma, const float* beta, int relu, double* s1, double* s2, void* workspace,
                                         int64_t workspace_bytes, void* stream);
P3TOK_API int p3tok_ln_param_grad_det_f32(const float* dY, const float* X, int64_t M, int64_t D, const float* mean, const float* rstd,
                                          double* dgamma, double* dbeta, void* workspace, int64_t workspace_bytes, void* stream);
/* workspace of the scatters for B clouds of N points with C channels (p3tok_scatter_rows_add_det_f32: C = 3 + D):
 * 12 bytes per (point, channel) + 4 per cloud */
P3TOK_API int64_t p3tok_scatter_det_workspace_bytes(int64_t B, int64_t N, int64_t C);
P3TOK_API int p3tok_scatter_rows_add_det_f32(const float* dRows, const int32_t* idx, int64_t B, int64_t N, int64_t G, int64_t k,
                                             int64_t D, float* dP, float* dF, void* workspace, int64_t workspace_bytes, void* stream);
P3TOK_API int p3tok_apf_rows_bwd_det_f32(const p3tok_rows* rows, const float* dRows, float* dX, void* workspace, int64_t workspace_bytes,
                                         void* stream);
P3TOK_API int p3tok_gather_points_bwd_det_f32(const float* dOut, int64_t B, int64_t N, int64_t C, const int64_t* idx, int64_t S,
                                              float* dX, void* workspace, int64_t workspace_bytes, void* stream);

/* ---- training through the ViT block stack (SURVEY 8f "next" #4 on top of #3) -------------------------------------------
 * The reference keeps the blocks frozen but trains point_encoder / encoder_norm / head (src/models/apf.py:335-346), so a
 * training step differentiates APFViTLayer x depth (src/models/apf_utils.py:268-293) -> encoder_norm -> max over tokens ->
 * ClassificationHead (apf.py:219-252, 358-371) with respect to the tokens.  GEMMs: p3tok_linear_f32 / p3tok_linear_tn_f32;
 * below are the pieces that are not GEMMs.  fp32 on CUDA cores; host side p3tok/train_vit.py. */
/* nn.LayerNorm over the last axis of X (M,D): Y = xhat * gamma + beta (gamma / beta may be NULL = no affine; Y may be NULL
 * when only the row statistics are wanted), mean[m], rstd[m] = 1/sqrt(biased variance + eps) kept for the backward. */
P3TOK_API int p3tok_ln_fwd_f32(const float* X, int64_t M, int64_t D, const float* gamma, const float* beta, float eps, float* Y,
                     float* mean, float* rstd, void* stream);
/* dX (+)= rstd (g dY - mean_c(g dY) - xhat mean_c(g dY xhat)), g = gamma (NULL = 1); accumulate = 0 overwrites. */
P3TOK_API int p3tok_ln_bwd_f32(const float* dY, const float* X, int64_t M, int64_t D, const float* mean, const float* rstd,
                     const float* gamma, int accumulate, float* dX, void* stream);
/* dgamma[c] = sum_m dY xhat, dbeta[c] = sum_m dY (fp64, overwritten). */
P3TOK_API int p3tok_ln_param_grad_f32(const float* dY, const float* X, int64_t M, int64_t D, const float* mean, const float* rstd,
                            double* dgamma, double* dbeta, void* stream);
/* AttentionLayer.forward between qkv and proj (apf_utils.py:141-153): qkv (B*G, 3*heads*hd) = [q | k | v] ->
 * O (B*G, heads*hd) = softmax(q k^T scale) v per (cloud, head); P (B*heads, G, G) = the probabilities, kept for the backward. */
P3TOK_API int p3tok_attn_fwd_f32(const float* qkv, int64_t B, int64_t G, int64_t heads, int64_t hd, float scale, float* O, float* P,
                       void* stream);
/* its backward: dO (B*G, heads*hd) -> dqkv (B*G, 3*heads*hd); scratch: 2 * B*heads*G*G floats. */
P3TOK_API int p3tok_attn_bwd_f32(const float* qkv, const float* P, const float* dO, int64_t B, int64_t G, int64_t heads, int64_t hd,
                       float scale, float* scratch, float* dqkv, void* stream);
/* out[e] = f(A[e], B[e]) over `total` elements (out may alias A or B):
 *   op 0  alpha A + beta B                   op 1  alpha A B[e / bdiv]  (dropout mask, bdiv = 1; DropPath per cloud, bdiv = G*D)
 *   op 2  gelu(A) (exact erf)                op 3  B gelu'(A)
 *   op 4  relu(A)                            op 5  B [A > 0] */
P3TOK_API int p3tok_ew_f32(int op, const float* A, const float* B, float alpha, float beta, int64_t total, int64_t bdiv, float* out,
                 void* stream);

/* out[g, c] = max over r < k of in[(g*k + r), c]   (torch.max(..., dim=k-axis)) */
P3TOK_API int p3tok_group_max(const float* in, int64_t ngroups, int64_t k, int64_t C, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* P3TOK_H_ */
