// embed_tc.cu - bf16 patch embedding on the 5th-generation tensor cores (tcgen05 + TMEM + TMA).
//
// Replaces Encoder.get_features (reference src/models/apf.py:145-169) and the conv1/conv2/pool
// half of a P3Embed stage (src/models/pix4point.py:179-188), eval-mode BatchNorm folded on the
// host, in the rtol-1e-2 precision mode: bf16 operands, fp32 accumulation in tensor memory.
//
// Kernels in this file
//   rows_first_layer_apf_warp_kernel / rows_first_layer_narrow_kernel
//                            gather + centre-subtract + first layer on CUDA cores when the input is narrow (cin <= 8: APF
//                            2C = 6/8, P3Embed stage 0 = 6): fp32 math from fp32 coordinates, bf16 out; one warp per
//                            32-row block, the next block's gather in flight while the current one is computed.  The APF
//                            variant folds the centre half of [nbr-ctr || ctr] into a per-block bias.
//                            (rows_first_layer_kernel / rows_first_layer_apf_kernel: the generic CTA-per-block forms.)
//   rows_gather_p4p_bf16_kernel / rows_gather_bf16_kernel
//                            wide inputs (P3Embed stage >= 1, cin = 131) are gathered to a zero-padded bf16 row matrix
//                            for the tensor cores.
//   tc_linear_kernel<PAIR, EW>  C = act(A W^T + bias + group_bias).  Persistent, warp-specialised:
//                              warp 0   TMA producer (warp-uniform loop, one elected lane issues)
//                              warp 1   tcgen05.mma issuer, descriptors in uniform registers
//                              warps 2..EW+1 epilogue, EW/4 per TMEM lane quarter;  last warp  A producer (A-resident mode)
//                            EW = 8 for the tokenizer's layers; EW = 16 with a lean epilogue (bf16 or TMA-stored fp32 only)
//                            for the small-M GEMMs of the ViT blocks (vit.cu), whose extra epilogues live here too: exact
//                            GELU (one MUFU), [gelu | relu] column split, fp32 residual as a TMA reduce-add, column-slice
//                            outputs (TcExtra, embed.cuh).
//                            PAIR = cta_group::2: two CTAs of a cluster share one 256 x BN tile - each holds its 128
//                            rows of A, HALF of the weight tile and its half of the accumulator; the leader issues the
//                            MMAs, TMA loads of both CTAs signal the leader's barrier, tcgen05.commit multicasts the slot
//                            release.  Two 128 x BN fp32 accumulators in TMEM overlap the epilogue of tile i with the
//                            MMAs of tile i+1; the epilogue works in 32-column tcgen05.ld pieces, fuses bias (smem) /
//                            per-group bias / ReLU (F2FP.RELU), packs bf16 into a swizzled 32x64 box for a TMA store; the
//                            fused patch max-pool is one redux.sync.max.f32 per column.
//   patch_embed_bf16         orchestration: which kernel runs which layers.  Default: first layer (CUDA cores) ->
//                            tc_fused_kernel (embed_fused.cu) for the two remaining per-point layers -> tc_linear for the
//                            pooled half of the concat layer (per-group bias) -> tc_fused_kernel for concat + output
//                            layer + pool; narrow P3Embed stages use tc_stage_kernel (embed_stage.cu) instead.
// What bounded tc_linear, in the order found (traces via P3TOK_TC_TRACE=1, ncu in profiles/): direct per-row global
// stores (620 GB/s) -> TMA stores; dependent bias loads in the epilogue -> smem staging; per-launch fixed
// cost -> large row chunks; the single-thread MMA loop -> warp-uniform loops + elect_one; weight-tile bytes per
// stage -> CTA pairs; then the epilogue itself (500-1000 cycles per 32x32 piece: ~140 dependent instructions in one
// warp) and the HBM round trip of every activation -> the fused kernels.  TMA multicast of the weight tile, L2
// prefetch of the next activation tile, 16 epilogue warps and a prefetched group-bias slice were measured neutral
// or worse.
// The concat layer W.[g||f] is evaluated as W_g.g (tensor-core GEMM over groups, becomes the per-group bias)
// + W_f.f, so no (rows, 2E) tensor exists.
#include <algorithm>
#include <vector>

#include <type_traits>

#include "tc_common.cuh"

namespace p3tok {

// ------------------------------------------------------------------------------------------------ GEMM
constexpr int TC_MAX_STAGES = 8;
constexpr int TC_EPI_WARPS = 8;                      // default epilogue-warp count: 2 warps per TMEM lane quarter (see TcCfg below)
constexpr int TC_MAX_KB = 8;                         // A-resident mode: K <= 512
constexpr int TC_A_STAGE = TC_BM * TC_BK * 2;        // 16 KB
constexpr int TC_STAGING = 32 * 128;                 // one 32-row x 64-column bf16 store box (4 KB, 128B-swizzled)
constexpr int TC_MAX_N = 2048;                       // bias vector staged in shared memory (8 KB)
// Shared memory: [pipeline stages][per-warp store staging 8 x 4 KB][bias 8 KB][barriers].  The TMA->MMA ring
// is sized at launch to fill what is left: a stage round trip (TMA latency ~1500 cycles + MMA drain) needs
// >= ingest_rate x latency bytes in flight, so the pair mode (32 KB stages) runs 5-6 stages deep.
constexpr int TC_SMEM = 227 * 1024;
constexpr int TC_EPI_BOXES = 2;                      // TMA-store boxes per epilogue warp (2 = double-buffered)
constexpr int TC_SGB_BYTES = 256;                    // per-warp 64-float group-bias slice
// The epilogue-warp count is a template parameter of the kernel: EW = TC_EPI_WARPS (8) for the tokenizer's layers, whose
// tiles are MMA-bound (16 warps measured -12 % there: registers), EW = 16 for the small-M bf16-output GEMMs of the ViT
// blocks (vit.cu), whose tile period is the epilogue's (two warps per scheduler issue ~1 instruction per 4-14 cycles).
template <int EW>
struct TcCfg {
  static constexpr int PER_Q = EW / 4;                   // epilogue warps per TMEM lane quarter, interleaved 64-column groups
  static constexpr int THREADS = 64 + EW * 32 + 32;      // warp 0 TMA, warp 1 MMA, epilogue warps, last warp = A producer (A-resident mode)
  static constexpr int ARES_WARP = 2 + EW;
  static constexpr int BOXES = EW > 8 ? 1 : TC_EPI_BOXES;
  static constexpr int WARP_SCRATCH = BOXES * TC_STAGING;   // 1024-aligned store boxes
  static constexpr int SMEM_FIXED = EW * (WARP_SCRATCH + TC_SGB_BYTES) + TC_MAX_N * 4 + 512 + 1024;
};

struct TcParams {
  int M, N, K, BN;
  int num_m_tiles, num_n_tiles;
  const float* bias;       // [N] or null
  const float* gbias;      // [ceil(M/rows_per_group), N] or null
  int rows_per_group;
  int relu;
  __nv_bfloat16* out_bf16; // [M,N] or null
  float* out_f32;          // [M,N] or null
  int f32_tma;             // out_f32 goes through swizzled 32x32 fp32 boxes + TMA stores (tmC is the fp32 map; no out_bf16)
  int res_add;             // f32_tma only: the boxes are ADDED to out_f32 by TMA reduce stores (cp.reduce.async.bulk.tensor .add)
                           // - the in-place residual x += out_scale * value with no load of x in the epilogue
  float* out_max;          // [ceil(M/32), N] max over each 32 consecutive rows, or null
  __nv_bfloat16* out_max_bf16;
  int max_relu;            // apply ReLU to the max (out_relu of the block)
  int gelu, gelu_cols;     // exact (erf) GELU after the bias on columns < gelu_cols (ViT mlp.fc1; ReLU, if set, applies to the
                           // columns from gelu_cols on: the adapter bottleneck rides in the same GEMM, embed.cuh TcExtra)
  const float* residual;   // [M,N] f32 or null: out_f32 = res_mul * residual + out_scale * value (may alias out_f32:
  float res_mul, out_scale; // every element is read by the thread that produces it, before its store box leaves)
  int stages, stage_bytes; // TMA->MMA ring depth and bytes per stage (A tile 16 KB + this CTA's part of the weight tile)
  int x3;                  // bf16x3 split mode (fp32-accurate on the tensor cores): A is [M, 2 Kp] = [hi | lo], W is [N, 3 Kp] =
                           // [W_hi | W_hi | W_lo], K = 3 Kp: k-blocks of the third segment re-read the hi half of A
  int out_split;           // out_bf16 is [M, 2 N] = [hi | lo] of the fp32 result (the next layer's split operand)
  int split_lo;            // out_split: column of the lo half relative to hi (N, or the full width when out_bf16 is a column slice)
  int ares;                // A-resident mode (pairs only): a pair walks ALL N tiles of its M group, the group's activation
                           // rows stay in shared memory and only weight boxes stream through the ring
  unsigned long long* trace;  // debug (P3TOK_TC_TRACE=1): per-CTA clock stamps, 16 words per tile per role
  unsigned long long* trace2; // debug: epilogue warp 0 of CTA 0, 8 stamps per (tile < 8, column group < 4)
};
// trace layout: trace[((cta * 64 + tile_it) * 3 + role) * 4 + {0..3}]
__device__ __forceinline__ void tc_trace(const TcParams& p, int it, int role, int slot, long long v) {
  if (p.trace && it < 64) p.trace[(((size_t)blockIdx.x * 64 + it) * 3 + role) * 4 + slot] = (unsigned long long)v;
}
// stamps of one column group: 0 start, 1 store box free, 2 first TMEM load back, 3 first half converted, 4 second load back,
// 5 second half converted, 6 store issued
__device__ __forceinline__ void tc_trace2(const TcParams& p, bool on, int it, int g, int slot) {
  if (on && it < 8 && g < 4) p.trace2[(it * 4 + g) * 8 + slot] = (unsigned long long)clock64();
}

// bias / per-group bias / ReLU on 32 accumulator columns starting at global column n0.  `sbias` is the
// bias vector staged in shared memory (zeros when the layer has none); all loads are issued before use.
__device__ __forceinline__ float4 lds128(uint32_t saddr) {   // explicit shared-space load (the generic form costs an LD + address check)
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
  return v;
}

// exact (erf) GELU without the erf: with q(t) = log2(erfc(t / sqrt 2) / 2), t = |x|,
//   gelu(x) = x Phi(x) = max(x, 0) - |x| * 2^q(|x|)
// (x < 0: x/2 erfc(|x|/sqrt 2); x > 0: x - x/2 erfc(x/sqrt 2)) - no cancellation in either tail.  q is smooth; its
// degree-7 least-squares Chebyshev fit on [0, 6.5] (fitted and checked against scipy in fp32 arithmetic: <= 7e-6 relative
// where |gelu| > 1e-6, absolute error at fp32 rounding level - 1/280 of a bf16 rounding) has a negative leading
// coefficient, so beyond the interval it only falls (q < -34 for t > 6.5, -inf for huge t: 2^q = 0, no clamp needed).
// 7 FMAs + ONE MUFU (EX2) + FMNMX + FFMA per element: the epilogue of the fc1 GEMM is issue- and MUFU-bound (erff():
// ~25 instructions; the A&S 7.1.26 form: 2 MUFUs).  Two elements per call: the Horner chain runs as packed FFMA2.
// (fma2: tc_common.cuh)
__device__ __forceinline__ void gelu_erf2(float& x0, float& x1) {
  const float t0 = fabsf(x0), t1 = fabsf(x1);
  float r0 = -1.808829734e-06f, r1 = -1.808829734e-06f;
  fma2(r0, r1, r0, r1, t0, t1, 6.107435026e-05f, 6.107435026e-05f);
  fma2(r0, r1, r0, r1, t0, t1, -9.264088059e-04f, -9.264088059e-04f);
  fma2(r0, r1, r0, r1, t0, t1, 8.492039891e-03f, 8.492039891e-03f);
  fma2(r0, r1, r0, r1, t0, t1, -5.392931550e-02f, -5.392931550e-02f);
  fma2(r0, r1, r0, r1, t0, t1, -4.584916519e-01f, -4.584916519e-01f);
  fma2(r0, r1, r0, r1, t0, t1, -1.151243301e+00f, -1.151243301e+00f);
  fma2(r0, r1, r0, r1, t0, t1, -9.999950370e-01f, -9.999950370e-01f);
  float e0, e1;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(r0));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(r1));
  x0 = fmaf(-t0, e0, fmaxf(x0, 0.f));
  x1 = fmaf(-t1, e1, fmaxf(x1, 0.f));
}

// `sbias` is staged zero-padded to a multiple of 64 columns, so the 32 columns starting at n0 are always readable.
__device__ __forceinline__ void epilogue_affine(float (&v)[32], const TcParams& p, const float* sbias, const float* gb, int n0,
                                                bool relu_now) {
  const int nmax = p.N - 4;                                  // N % 8 == 0: clamped float4 loads stay in range
  float4 g4[8];
  if (gb) {
#pragma unroll
    for (int j = 0; j < 8; ++j) g4[j] = __ldg(reinterpret_cast<const float4*>(gb + min(n0 + 4 * j, nmax)));
  }
  if (p.bias) {                                              // warp-uniform: layers whose bias rides in the group bias skip it
    const uint32_t sb = smem_u32(sbias + n0);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 b4 = lds128(sb + 16 * j);
      add2(v[4 * j], v[4 * j + 1], v[4 * j], v[4 * j + 1], b4.x, b4.y);
      add2(v[4 * j + 2], v[4 * j + 3], v[4 * j + 2], v[4 * j + 3], b4.z, b4.w);
    }
  }
  if (gb) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      add2(v[4 * j], v[4 * j + 1], v[4 * j], v[4 * j + 1], g4[j].x, g4[j].y);
      add2(v[4 * j + 2], v[4 * j + 3], v[4 * j + 2], v[4 * j + 3], g4[j].z, g4[j].w);
    }
  }
  if (relu_now) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
  }
}

// 32 accumulator columns (lane = row) starting at global column n0: bias / group bias / ReLU, then any of
//   - pack to bf16 into this warp's 32 x 128 B staging box (4 x 16-byte pieces, XOR-swizzled by row: conflict-free),
//   - fp32 store, - max over the warp's 32 rows.
template <bool LEAN>   // LEAN (16 epilogue warps, ~100 registers): bf16 output only - no fp32 / max / residual / per-row group-bias paths
__device__ __forceinline__ void epilogue_half(const TcParams& p, const float* sbias, const float* gb, const float* sgb,
                                              uint32_t sbox, int half, int row0, int row, bool row_ok, int lane, int n0,
                                              float (&v)[32]) {
  if (sgb) {   // this warp's group-bias slice (64 floats for the whole column group), staged in shared memory
    const uint32_t sg = smem_u32(sgb + 32 * half);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 g = lds128(sg + 16 * j);
      add2(v[4 * j], v[4 * j + 1], v[4 * j], v[4 * j + 1], g.x, g.y);
      add2(v[4 * j + 2], v[4 * j + 3], v[4 * j + 2], v[4 * j + 3], g.z, g.w);
    }
  }
  // bf16-only outputs take their ReLU from the conversion instruction (F2FP.RELU) instead of 32 FMNMX
  const bool gelu_here = p.gelu && n0 < p.gelu_cols;        // warp-uniform (gelu_cols is a multiple of 32)
  const bool relu_here = p.relu && !gelu_here;
  const bool relu_in_pack = relu_here && (LEAN || (!p.out_f32 && !p.out_max && !p.out_max_bf16 && !p.out_split));
  epilogue_affine(v, p, sbias, gb, n0, relu_here && !relu_in_pack);
  if (gelu_here) {
#pragma unroll
    for (int j = 0; j < 32; j += 2) gelu_erf2(v[j], v[j + 1]);
  }
  if (!LEAN && p.res_add && p.out_scale != 1.f) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] *= p.out_scale;
  }
  if (!LEAN && p.residual) {   // general residual (not in place): 128 contiguous bytes per lane; the load latency is exposed
    const int nmax = p.N - 4;
    const float* rr = p.residual + (size_t)(row_ok ? row : 0) * p.N;
    float4 r4[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) r4[j] = *reinterpret_cast<const float4*>(rr + min(n0 + 4 * j, nmax));
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      v[4 * j] = fmaf(p.res_mul, r4[j].x, p.out_scale * v[4 * j]);
      v[4 * j + 1] = fmaf(p.res_mul, r4[j].y, p.out_scale * v[4 * j + 1]);
      v[4 * j + 2] = fmaf(p.res_mul, r4[j].z, p.out_scale * v[4 * j + 2]);
      v[4 * j + 3] = fmaf(p.res_mul, r4[j].w, p.out_scale * v[4 * j + 3]);
    }
  }
  if (!LEAN && p.out_bf16 && p.out_split) {
    // bf16x3: the fp32 value leaves as hi = bf16(v) (box 0) and lo = bf16(v - hi) (box 1): hi + lo carries 16 mantissa bits
    const uint32_t rbase = sbox + lane * 128;
#pragma unroll
    for (int pc = 0; pc < 4; ++pc) {
      uint32_t hi[4], lo[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float a = v[pc * 8 + 2 * e], b = v[pc * 8 + 2 * e + 1];
        const __nv_bfloat16 ha = __float2bfloat16_rn(a), hb = __float2bfloat16_rn(b);
        hi[e] = (uint32_t)__bfloat16_as_ushort(ha) | ((uint32_t)__bfloat16_as_ushort(hb) << 16);
        lo[e] = pack_bf16x2(a - __bfloat162float(ha), b - __bfloat162float(hb));
      }
      const uint32_t a = rbase + (((uint32_t)(pc + 4 * half) ^ (lane & 7)) << 4);
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(hi[0]), "r"(hi[1]), "r"(hi[2]), "r"(hi[3]) : "memory");
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a + (uint32_t)TC_STAGING), "r"(lo[0]), "r"(lo[1]), "r"(lo[2]), "r"(lo[3])
                   : "memory");
    }
  } else if (p.out_bf16) {
    const uint32_t rbase = sbox + lane * 128;
    if (relu_in_pack) {
#pragma unroll
      for (int pc = 0; pc < 4; ++pc) {
        const uint32_t a = rbase + (((uint32_t)(pc + 4 * half) ^ (lane & 7)) << 4);
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(pack_bf16x2_relu(v[pc * 8], v[pc * 8 + 1])),
                     "r"(pack_bf16x2_relu(v[pc * 8 + 2], v[pc * 8 + 3])), "r"(pack_bf16x2_relu(v[pc * 8 + 4], v[pc * 8 + 5])),
                     "r"(pack_bf16x2_relu(v[pc * 8 + 6], v[pc * 8 + 7]))
                     : "memory");
      }
    } else {
#pragma unroll
      for (int pc = 0; pc < 4; ++pc) {
        const uint32_t a = rbase + (((uint32_t)(pc + 4 * half) ^ (lane & 7)) << 4);
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(pack_bf16x2(v[pc * 8], v[pc * 8 + 1])),
                     "r"(pack_bf16x2(v[pc * 8 + 2], v[pc * 8 + 3])), "r"(pack_bf16x2(v[pc * 8 + 4], v[pc * 8 + 5])),
                     "r"(pack_bf16x2(v[pc * 8 + 6], v[pc * 8 + 7]))
                     : "memory");
      }
    }
  }
  if (p.out_f32 && p.f32_tma) {
    // this half's 32 rows x 32 columns as one 4 KB box (rows of 128 B, 16-byte pieces XOR-swizzled by row): the direct
    // per-thread stores below touch 32 different cache lines per instruction (the group-bias GEMM spent most of its
    // 38 us in them)
    const uint32_t rbase = sbox + (LEAN ? 0u : (uint32_t)half * TC_STAGING) + lane * 128;   // LEAN: one box per warp, both halves
#pragma unroll
    for (int pc = 0; pc < 8; ++pc) {
      const uint32_t a = rbase + (((uint32_t)pc ^ (lane & 7)) << 4);
      asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v[4 * pc]), "f"(v[4 * pc + 1]), "f"(v[4 * pc + 2]),
                   "f"(v[4 * pc + 3])
                   : "memory");
    }
  } else if (!LEAN && p.out_f32 && row_ok) {
    float* o = p.out_f32 + (size_t)row * p.N + n0;
#pragma unroll
    for (int j = 0; j < 32; j += 4)
      if (n0 + j < p.N) *reinterpret_cast<float4*>(o + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
  }
  if (!LEAN && (p.out_max || p.out_max_bf16)) {
    if (!row_ok) {
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = -3.0e38f;
    }
    float m = warp_rows_max(v, lane);
    if (p.max_relu) m = fmaxf(m, 0.f);
    const size_t o = (size_t)(row0 >> 5) * p.N + n0 + lane;
    if (n0 + lane < p.N) {
      if (p.out_max) p.out_max[o] = m;
      if (p.out_max_bf16) p.out_max_bf16[o] = __float2bfloat16_rn(m);
    }
  }
}

template <bool PAIR, int EW>
__global__ void __launch_bounds__(TcCfg<EW>::THREADS, 1)
tc_linear_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ CUtensorMap tmC, const TcParams p) {
  using Cfg = TcCfg<EW>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int TC_STAGES = p.stages, STAGE_BYTES = p.stage_bytes;   // stage s starts at s*STAGE_BYTES: A tile (16 KB), then the weight rows
  const int num_kb = (p.K + TC_BK - 1) / TC_BK;
  const int ARES = PAIR ? p.ares : 0;
  const int ares_bytes = ARES ? num_kb * TC_A_STAGE : 0;   // resident activation K blocks in front of the ring
  uint8_t* sAres = smem;
  uint8_t* sA = smem + ares_bytes;
  uint8_t* sB = sA + (ARES ? 0 : TC_A_STAGE);
  uint8_t* sC = sA + TC_STAGES * p.stage_bytes;       // per-epilogue-warp store staging, 4 KB each
  float* sgb_all = reinterpret_cast<float*>(sC + EW * Cfg::WARP_SCRATCH);
  float* sbias = reinterpret_cast<float*>(sC + EW * (Cfg::WARP_SCRATCH + TC_SGB_BYTES));
  uint64_t* full = reinterpret_cast<uint64_t*>(sC + EW * (Cfg::WARP_SCRATCH + TC_SGB_BYTES) + TC_MAX_N * 4);
  uint64_t* empty = full + TC_MAX_STAGES;
  uint64_t* tfull = empty + TC_MAX_STAGES;
  uint64_t* tempty = tfull + 2;
  uint64_t* a_full = tempty + 2;                      // [TC_MAX_KB] leader (A-resident mode)
  uint64_t* a_empty = a_full + TC_MAX_KB;             // [TC_MAX_KB] local, multicast commit
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_empty + TC_MAX_KB);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);   // provably warp-uniform role index
  const int lane = threadIdx.x & 31;
  constexpr int CL = PAIR ? 2 : 1;                    // a pair's CTAs take consecutive M tiles and half the weight tile each
  const int rank = CL > 1 ? (int)cluster_ctarank() : 0;
  const int cluster_id = blockIdx.x / CL, num_clusters = gridDim.x / CL;
  const int num_mg = (p.num_m_tiles + CL - 1) / CL;
  const int num_items = num_mg * p.num_n_tiles;   // (group of CL M tiles) x N tile
  // local work list: entry li of this cluster is (M group mg, N tile nt).  Default: items round-robin over clusters;
  // A-resident: whole M groups round-robin, their N tiles back to back.
  auto decode = [&](int li, int& mg, int& nt) -> bool {
    if (ARES) {
      const int g = li / p.num_n_tiles;
      nt = li - g * p.num_n_tiles;
      mg = cluster_id + g * num_clusters;
      return mg < num_mg;
    }
    const int item = cluster_id + li * num_clusters;
    mg = item / p.num_n_tiles;
    nt = item - mg * p.num_n_tiles;
    return item < num_items;
  };

  if (threadIdx.x == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmB)) : "memory");
    for (int s = 0; s < TC_STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tfull[b], 1);
      mbar_init(&tempty[b], PAIR ? 2 * EW : EW);   // pair: both CTAs' epilogues report to the leader
    }
    for (int b = 0; b < TC_MAX_KB; ++b) {
      mbar_init(&a_full[b], 1);
      mbar_init(&a_empty[b], 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = threadIdx.x; i < ((p.N + 63) & ~63); i += Cfg::THREADS) sbias[i] = (p.bias && i < p.N) ? p.bias[i] : 0.f;   // zero-padded to 64
  if (warp == 1) {   // TMEM: 512 columns = two 128 x BN fp32 accumulators (this CTA's 128 rows)
    if (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::);
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (CL > 1) cluster_sync_all();   // peers' barriers are initialised before any pair load / remote arrive
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ---------------- TMA producer.  The whole warp runs the (warp-uniform) loop so that addresses and
    // counters live in uniform registers; one elected lane issues the asynchronous copies.
    const bool issuer = elect_one();
    int stage = 0;
    uint32_t phase = 0;
    // bytes landing on this CTA's (pair: the leader's) full barrier per stage
    const uint32_t tx = PAIR ? 2u * ((ARES ? 0u : (uint32_t)TC_A_STAGE) + (uint32_t)(p.BN / 2) * TC_BK * 2)
                             : TC_A_STAGE + (uint32_t)p.BN * TC_BK * 2;
    const int brows = p.BN / CL;     // rows of the weight tile this CTA fetches
    // A column of k-block kb: plain, or (bf16x3) [hi | lo | hi again] over the [hi | lo] operand
    const int kb_seg = p.x3 ? num_kb / 3 : num_kb;
    auto acol = [&](int kb) { return (p.x3 && kb >= 2 * kb_seg ? kb - 2 * kb_seg : kb) * TC_BK; };
    int mg, nt;
    for (int li = 0; decode(li, mg, nt); ++li) {
      const int mt = mg * CL + rank;   // may be a dummy tile past the end: TMA zero-fills, stores are clipped
      if (issuer && !ARES && !p.x3) {
        // pull the NEXT item's activation tile (streamed from HBM exactly once) into L2 ahead of its loads
        int nmg, nnt;
        if (decode(li + 1, nmg, nnt)) {
          const int nmt = nmg * CL + rank;
          if (nmt < p.num_m_tiles)
            for (int kb = 0; kb < num_kb; ++kb) tma_prefetch_2d(&tmA, kb * TC_BK, nmt * TC_BM);
        }
      }
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&empty[stage], phase ^ 1);
        if (issuer) {
          if (kb == 0) tc_trace(p, li, 0, 0, clock64());
          if (kb == num_kb - 1) tc_trace(p, li, 0, 1, clock64());
          uint8_t* a_dst = sA + stage * STAGE_BYTES;
          uint8_t* b_dst = sB + stage * STAGE_BYTES;
          if (PAIR) {
            if (rank == 0) mbar_expect_tx(&full[stage], tx);
            if (!ARES) tma_load_2d_pair(a_dst, &tmA, &full[stage], acol(kb), mt * TC_BM);
            tma_load_2d_pair(b_dst, &tmB, &full[stage], kb * TC_BK, nt * p.BN + rank * brows);
          } else {
            mbar_expect_tx(&full[stage], tx);
            tma_load_2d(a_dst, &tmA, &full[stage], acol(kb), mt * TC_BM);
            tma_load_2d(b_dst, &tmB, &full[stage], kb * TC_BK, nt * p.BN);
          }
        }
        __syncwarp();
        if (++stage == TC_STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == Cfg::ARES_WARP) {
    // ---------------- A producer (A-resident mode): the M group's activation rows, one 64-column K block at a time.
    // K block kb of the next group is fetched as soon as the last N tile of the current group has consumed it.
    if (ARES) {
      const bool issuer = elect_one();
      for (int g = 0, mg = cluster_id; mg < num_mg; mg += num_clusters, ++g) {
        const int mt = mg * CL + rank;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&a_empty[kb], ((uint32_t)g & 1) ^ 1);
          if (issuer) {
            if (rank == 0) mbar_expect_tx(&a_full[kb], 2u * (uint32_t)TC_A_STAGE);
            tma_load_2d_pair(sAres + kb * TC_A_STAGE, &tmA, &a_full[kb], kb * TC_BK, mt * TC_BM);
          }
          __syncwarp();
        }
      }
    }
  } else if (warp == 1) {
    if (!PAIR || rank == 0) {
      // ---------------- MMA issuer (pair: the leader issues for both SMs); warp-uniform loop, one elected lane
      const bool issuer = elect_one();
      // instruction descriptor: D=f32, A=B=bf16, both K-major, N = BN, M = 128 (256 across a pair)
      const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.BN >> 3) << 17) |
                             ((uint32_t)((PAIR ? 2 * TC_BM : TC_BM) >> 4) << 24);
      const uint64_t dconst = umma_desc_sw128(0);                 // everything but the start address
      const uint32_t a_base = smem_u32(sA) >> 4, b_base = smem_u32(sB) >> 4, stage_step = (uint32_t)STAGE_BYTES >> 4;
      const uint32_t ares_base = smem_u32(sAres) >> 4;
      int stage = 0;
      uint32_t phase = 0;
      int mg, nt;
      for (int it = 0; decode(it, mg, nt); ++it) {
        const int buf = it & 1;
        if (issuer) tc_trace(p, it, 1, 0, clock64());
        mbar_wait(&tempty[buf], ((uint32_t)(it >> 1) & 1) ^ 1);
        if (issuer) tc_trace(p, it, 1, 1, clock64());
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(buf * p.BN);
        const uint32_t gpar = ARES ? (uint32_t)(it / p.num_n_tiles) & 1 : 0;   // parity of this M group's A barriers
        for (int kb = 0; kb < num_kb; ++kb) {
          if (ARES && nt == 0) mbar_wait(&a_full[kb], gpar);      // this group's K block kb is resident (both CTAs)
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          if (issuer) {
            if (kb == 0) tc_trace(p, it, 1, 2, clock64());
            const uint64_t adesc = dconst | (uint64_t)(ARES ? ares_base + kb * (TC_A_STAGE >> 4) : a_base + stage * stage_step);
            const uint64_t bdesc = dconst | (uint64_t)(b_base + stage * stage_step);
#pragma unroll
            for (int k = 0; k < TC_BK / 16; ++k) {   // +32 bytes (2 x 16 B units) per 16-wide K step inside the swizzle atom
              if (PAIR) tc_mma_pair(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (uint32_t)((kb | k) != 0));
              else tc_mma(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (uint32_t)((kb | k) != 0));
            }
            if (PAIR) tc_commit_pair(&empty[stage]);      // frees the stage in both CTAs of the pair
            else tc_commit(&empty[stage]);                // frees the smem stage once these MMAs have read it
            if (PAIR && ARES && nt == p.num_n_tiles - 1) tc_commit_pair(&a_empty[kb]);   // last reader of this group's K block
          }
          __syncwarp();
          if (++stage == TC_STAGES) { stage = 0; phase ^= 1; }
        }
        if (issuer) {
          if (PAIR) tc_commit_pair(&tfull[buf]);   // accumulator halves complete in both CTAs
          else tc_commit(&tfull[buf]);             // accumulator complete
          tc_trace(p, it, 1, 3, clock64());
        }
        __syncwarp();
      }
    }
  } else {             // ---------------- epilogue warps: TMEM lane quarter q, column-group parity h
    const int ew = warp - 2;
    const int q = warp & 3, h = ew >> 2;
    uint8_t* stg = sC + ew * Cfg::WARP_SCRATCH;   // 1024-aligned: the TMA store un-swizzles by address bits
    int sbuf = 0;
    // (Fetching the per-warp group-bias slice one column group ahead was measured twice: the 384->768 layer went from
    // 338 to 376 us, the extra live registers and address arithmetic cost more than the hidden L2 round trip.)
    int mg, nt;
    for (int it = 0; decode(it, mg, nt); ++it) {
      const int mt = mg * CL + rank;
      const int buf = it & 1;
      if (ew == 0 && lane == 0) tc_trace(p, it, 2, 0, clock64());
      mbar_wait(&tfull[buf], (uint32_t)(it >> 1) & 1);
      if (ew == 0 && lane == 0) tc_trace(p, it, 2, 1, clock64());
      tc_fence_after();
      const int row0 = mt * TC_BM + q * 32;
      const int row = row0 + lane;
      const bool row_ok = row < p.M;
      const float* gb = (EW <= 8 && p.gbias && row_ok) ? p.gbias + (size_t)(row / p.rows_per_group) * p.N : nullptr;
      bool released = false;
      // per-warp group-bias slice: when a patch (rows_per_group rows) covers whole warps, all 32 rows of this
      // warp share one group-bias row, so the 64 values of a column group are fetched once, coalesced, BEFORE
      // the accumulator load (latency overlaps it) and re-read from shared memory as broadcasts
      const bool gb_shared = EW <= 8 && p.gbias && (p.rows_per_group % 32 == 0) && (row0 < p.M);
      const float* gb_row = gb_shared ? p.gbias + (size_t)(row0 / p.rows_per_group) * p.N : nullptr;
      float* sgb = sgb_all + ew * (TC_SGB_BYTES / 4);
      for (int gi = h; gi * 64 < p.BN; gi += Cfg::PER_Q) {
        const int n0 = nt * p.BN + gi * 64;
        if (n0 >= p.N || row0 >= p.M) break;     // warp-uniform
        const bool tr2 = p.trace2 && blockIdx.x == 0 && ew == 0 && lane == 0;
        const int g2 = (gi - h) / Cfg::PER_Q;
        tc_trace2(p, tr2, it, g2, 0);
        float2 gpre = make_float2(0.f, 0.f);
        if (gb_shared) {
          const int c = min(n0 + 2 * lane, p.N - 2);
          gpre = __ldg(reinterpret_cast<const float2*>(gb_row + c));
        }
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * p.BN + gi * 64);
        const bool f32_tma = p.out_f32 && p.f32_tma;   // fp32 output: box 0 / box 1 of this warp = the two 32-column halves
        const bool split = EW <= 8 && p.out_split;     // bf16x3: box 0 = hi, box 1 = lo of the same 64 columns (no double buffering)
        const uint32_t sbox = (f32_tma || split) ? smem_u32(stg) : smem_u32(stg + sbuf * TC_STAGING);
        if (p.out_bf16 || f32_tma) {   // the TMA store issued two groups (fp32: two halves) ago has finished reading this box
          if (lane == 0) {
            if (Cfg::BOXES == 2 && !split) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            else asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
          }
          __syncwarp();
        }
        tc_trace2(p, tr2, it, g2, 1);
        const bool last = (gi + Cfg::PER_Q >= (p.BN >> 6)) || (n0 + 64 * Cfg::PER_Q >= p.N);
        float v[32];
        tc_ld32_issue(taddr, v);
        if (gb_shared) {
          *reinterpret_cast<float2*>(sgb + 2 * lane) = gpre;
          __syncwarp();
        }
        tc_ld_wait();
        tc_trace2(p, tr2, it, g2, 2);
        epilogue_half<(EW > 8)>(p, sbias, gb_shared ? nullptr : gb, gb_shared ? sgb : nullptr, sbox, 0, row0, row, row_ok, lane, n0, v);
        tc_trace2(p, tr2, it, g2, 3);
        tc_ld32_issue(taddr + 32, v);
        if (f32_tma) {   // store half 0, then make sure box 1 (the previous group's half 1) has been read
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (lane == 0) {
            if (p.res_add)
              asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                               reinterpret_cast<uint64_t>(&tmC)),
                           "r"(sbox), "r"(n0), "r"(row0)
                           : "memory");
            else
              asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                               reinterpret_cast<uint64_t>(&tmC)),
                           "r"(sbox), "r"(n0), "r"(row0)
                           : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            if (Cfg::BOXES == 2) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            else asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // one box: half 1 overwrites what half 0 just sent
          }
          __syncwarp();
        }
        tc_ld_wait();
        tc_trace2(p, tr2, it, g2, 4);
        if (last) {
          // this warp has read its last accumulator columns of the tile: hand the TMEM buffer back to the MMA
          // warp now, before the remaining bias / convert / store work
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (PAIR) mbar_arrive_cta(&tempty[buf], 0);
            else mbar_arrive(&tempty[buf]);
          }
          released = true;
        }
        epilogue_half<(EW > 8)>(p, sbias, gb_shared ? nullptr : gb, gb_shared ? sgb : nullptr, sbox, 1, row0, row, row_ok, lane, n0 + 32, v);
        tc_trace2(p, tr2, it, g2, 5);
        if (p.out_bf16) {
          // one TMA store of the 32 x 64 bf16 box (clips rows >= M / columns >= N)
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (lane == 0) {
            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                             reinterpret_cast<uint64_t>(&tmC)),
                         "r"(sbox), "r"(n0), "r"(row0)
                         : "memory");
            if (split)      // the lo half of the split output: split_lo columns right of the hi half, same rows
              asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                               reinterpret_cast<uint64_t>(&tmC)),
                           "r"(sbox + (uint32_t)TC_STAGING), "r"(p.split_lo + n0), "r"(row0)
                           : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
          if (Cfg::BOXES == 2 && !split) sbuf ^= 1;
        } else if (f32_tma) {
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (lane == 0 && n0 + 32 < p.N) {
            if (p.res_add)
              asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                               reinterpret_cast<uint64_t>(&tmC)),
                           "r"(sbox + (Cfg::BOXES == 2 ? (uint32_t)TC_STAGING : 0u)), "r"(n0 + 32), "r"(row0)
                           : "memory");
            else
              asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                               reinterpret_cast<uint64_t>(&tmC)),
                           "r"(sbox + (Cfg::BOXES == 2 ? (uint32_t)TC_STAGING : 0u)), "r"(n0 + 32), "r"(row0)
                           : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        }
        tc_trace2(p, tr2, it, g2, 6);
        __syncwarp();   // group-bias slice is free for the next group
      }
      if (!released) {   // this warp had no group in the tile (narrow N tile or rows past M)
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (PAIR) mbar_arrive_cta(&tempty[buf], 0);
          else mbar_arrive(&tempty[buf]);
        }
      }
      if (ew == 0 && lane == 0) tc_trace(p, it, 2, 2, clock64());
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // this warp's stores are complete
  }
  tc_fence_before();
  __syncthreads();
  if (CL > 1) cluster_sync_all();   // no CTA leaves while a peer may still multicast into it or arrive on its barriers
  if (warp == 1) {
    tc_fence_after();
    if (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

static int pick_bn(int N) {
  // widest tile <= 256 (multiple of 64: the epilogue works in 64-column store boxes) with the least padding
  int best = 64, best_waste = 1 << 30;
  for (int bn = 256; bn >= 64; bn -= 64) {
    const int tiles = (N + bn - 1) / bn;
    const int waste = tiles * bn - N;
    if (waste < best_waste) { best_waste = waste; best = bn; }
  }
  return best;
}

// C = act(A[M,K] W[N,K]^T + bias + gbias), bf16 operands.  K % 8 == 0, N % 8 == 0.
static int tc_linear(const __nv_bfloat16* A, int64_t M, int K, const __nv_bfloat16* W, int N, const float* bias,
                     const float* gbias, int rows_per_group, int relu, __nv_bfloat16* out_bf16, float* out_f32,
                     float* out_max, __nv_bfloat16* out_max_bf16, int max_relu, cudaStream_t s, const TcExtra* ex = nullptr) {
  P3_REQUIRE(K % 8 == 0 && N % 8 == 0, P3TOK_ERR_UNSUPPORTED, "tc_linear: K=%d and N=%d must be multiples of 8", K, N);
  P3_REQUIRE(N <= TC_MAX_N, P3TOK_ERR_UNSUPPORTED, "tc_linear: N=%d > %d", N, TC_MAX_N);
  P3_REQUIRE(M < (1ll << 31) - 256, P3TOK_ERR_UNSUPPORTED, "tc_linear: too many rows");
  if (M == 0) return P3TOK_OK;
  TcParams p;
  p.M = (int)M; p.N = N; p.K = K; p.BN = pick_bn(N);
  if (ex && ex->bn > 0) {
    P3_REQUIRE(ex->bn % 64 == 0 && ex->bn <= 256, P3TOK_ERR_INVALID, "tc_linear: tile width %d", ex->bn);
    p.BN = ex->bn;
  }
  p.num_m_tiles = (int)((M + TC_BM - 1) / TC_BM);
  p.num_n_tiles = (N + p.BN - 1) / p.BN;
  // CTA pairs with cta_group::2 MMAs (M = 256 per pair, weight tile split) wherever there are two M tiles
  const bool pair = p.num_m_tiles >= 2;
  const int CL = pair ? 2 : 1;
  p.bias = bias; p.gbias = gbias; p.rows_per_group = rows_per_group > 0 ? rows_per_group : 1; p.relu = relu;
  p.out_bf16 = out_bf16; p.out_f32 = out_f32; p.out_max = out_max; p.out_max_bf16 = out_max_bf16; p.max_relu = max_relu;
  p.gelu = ex ? ex->gelu : 0;
  p.gelu_cols = (ex && ex->gelu_cols > 0) ? ex->gelu_cols : N;
  P3_REQUIRE(p.gelu_cols % 32 == 0 || p.gelu_cols == N, P3TOK_ERR_UNSUPPORTED, "tc_linear: gelu_cols must be a multiple of 32");
  p.residual = ex ? ex->residual : nullptr;
  p.res_mul = ex ? ex->res_mul : 0.f;
  p.out_scale = ex ? ex->out_scale : 1.f;
  p.x3 = ex ? ex->x3 : 0;
  p.out_split = ex ? ex->out_split : 0;
  if (p.x3) P3_REQUIRE(K % (3 * TC_BK) == 0, P3TOK_ERR_UNSUPPORTED, "tc_linear(x3): K=%d must be 3 x a multiple of 64", K);
  if (p.out_split) P3_REQUIRE(out_bf16 && N % 64 == 0 && !(ex && ex->epi16), P3TOK_ERR_UNSUPPORTED, "tc_linear(split): N=%d must be a multiple of 64", N);
  p.split_lo = (p.out_split && ex->split_n > 0) ? ex->split_n : N;
  P3_REQUIRE(p.split_lo >= N && p.split_lo % 8 == 0, P3TOK_ERR_UNSUPPORTED, "tc_linear(split): split width %d < N=%d", p.split_lo, N);
  const int64_t ldc = p.out_split ? 2 * (int64_t)p.split_lo : ((ex && ex->ldc > 0) ? ex->ldc : N);   // row pitch of out_bf16
  P3_REQUIRE(ldc == N || (out_bf16 && (!out_f32 || p.out_split) && ldc % 8 == 0), P3TOK_ERR_UNSUPPORTED, "tc_linear: ldc only for bf16 outputs");
  // 16 epilogue warps (lean epilogue: bf16 or TMA-stored / TMA-added fp32 outputs only), asked for by the ViT blocks
  const bool want16 = ex && ex->epi16 && !out_max && !out_max_bf16 && !gbias && !(out_bf16 && out_f32);
  CUtensorMap ta, tb, tc;
  int rc = make_map(&ta, A, M, p.x3 ? K / 3 * 2 : K, TC_BM);    // x3: the operand holds [hi | lo], 2/3 of the reduction length
  if (rc) return rc;
  rc = make_map(&tb, W, N, K, p.BN / CL);       // each CTA of a pair fetches half the rows of the weight tile
  if (rc) return rc;
  p.f32_tma = 0;
  p.res_add = 0;
  if (out_bf16) {
    rc = make_map(&tc, out_bf16, M, p.out_split ? p.split_lo + N : N, 32, ldc);     // store boxes: 64 columns x 32 rows
    if (rc) return rc;
  } else if (out_f32 && N % 4 == 0 && (reinterpret_cast<uintptr_t>(out_f32) & 15) == 0) {
    rc = make_map_f32(&tc, out_f32, M, N, 32);  // fp32 store boxes: 32 columns x 32 rows
    if (rc) return rc;
    p.f32_tma = 1;
    // in-place residual with unit multiplier: let the TMA unit add the boxes into x instead of loading x in the epilogue
    if (p.residual && p.residual == out_f32 && p.res_mul == 1.f) {
      p.res_add = 1;
      p.residual = nullptr;
    }
  } else {
    tc = ta;                                     // unused by the kernel
  }
  static thread_local bool configured[32] = {false};
  int dev = 0;
  P3_CUDA(cudaGetDevice(&dev));
  if (dev < 32 && !configured[dev]) {
    P3_CUDA(cudaFuncSetAttribute(tc_linear_kernel<false, TC_EPI_WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM));
    P3_CUDA(cudaFuncSetAttribute(tc_linear_kernel<true, TC_EPI_WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM));
    P3_CUDA(cudaFuncSetAttribute(tc_linear_kernel<false, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM));
    P3_CUDA(cudaFuncSetAttribute(tc_linear_kernel<true, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM));
    configured[dev] = true;
  }
  const bool ew16 = want16 && (out_bf16 || (p.f32_tma && !p.residual));
  const int smem_fixed = ew16 ? TcCfg<16>::SMEM_FIXED : TcCfg<TC_EPI_WARPS>::SMEM_FIXED;
  {
    const int wrows = pair ? p.BN / 2 : p.BN;
    // A-resident mode: with several N tiles per M group the default walk re-fetches the same
    // activation tile once per N tile, and at 128 rows per CTA the L2 -> shared-memory fill (activation tile + half a
    // weight tile per MMA group, ~62 B/cycle/SM at BN = 256) outruns what TMA delivers (~42 B/cycle/SM) before the
    // tensor pipe is busy.  Keeping the M group's rows resident halves the fill.
    const int num_kb = (K + TC_BK - 1) / TC_BK;
    p.ares = 0;
    if (pair && !p.x3 && p.num_n_tiles >= 2 && num_kb <= TC_MAX_KB) {
      const int ring = TC_SMEM - smem_fixed - num_kb * TC_A_STAGE;
      if (ring / (wrows * TC_BK * 2) >= 3) p.ares = 1;
    }
    p.stage_bytes = (p.ares ? 0 : TC_A_STAGE) + wrows * TC_BK * 2;
    p.stages = (TC_SMEM - smem_fixed - (p.ares ? num_kb * TC_A_STAGE : 0)) / p.stage_bytes;
    if (p.stages > TC_MAX_STAGES) p.stages = TC_MAX_STAGES;
  }
  static int trace_on = -1;
  if (trace_on < 0) trace_on = getenv("P3TOK_TC_TRACE") ? 1 : 0;
  p.trace = nullptr;
  const size_t trace_words = (size_t)num_sms() * 64 * 3 * 4;
  p.trace2 = nullptr;
  if (trace_on) {
    P3_CUDA(cudaMalloc(&p.trace, trace_words * 8));
    P3_CUDA(cudaMemsetAsync(p.trace, 0, trace_words * 8, s));
    P3_CUDA(cudaMalloc(&p.trace2, 8 * 4 * 8 * 8));
    P3_CUDA(cudaMemsetAsync(p.trace2, 0, 8 * 4 * 8 * 8, s));
  }
  const int items = p.ares ? (p.num_m_tiles + CL - 1) / CL : ((p.num_m_tiles + CL - 1) / CL) * p.num_n_tiles;
  const int max_clusters = num_sms() / CL;
  const int clusters = items < max_clusters ? items : max_clusters;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(clusters * CL));
  cfg.blockDim = dim3(ew16 ? TcCfg<16>::THREADS : TcCfg<TC_EPI_WARPS>::THREADS);
  cfg.dynamicSmemBytes = TC_SMEM;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)CL;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = CL > 1 ? 1 : 0;
  if (ew16) {
    if (pair) P3_CUDA(cudaLaunchKernelEx(&cfg, tc_linear_kernel<true, 16>, ta, tb, tc, p));
    else P3_CUDA(cudaLaunchKernelEx(&cfg, tc_linear_kernel<false, 16>, ta, tb, tc, p));
  } else {
    if (pair) P3_CUDA(cudaLaunchKernelEx(&cfg, tc_linear_kernel<true, TC_EPI_WARPS>, ta, tb, tc, p));
    else P3_CUDA(cudaLaunchKernelEx(&cfg, tc_linear_kernel<false, TC_EPI_WARPS>, ta, tb, tc, p));
  }
  count_launch();
  if (trace_on) {   // debug only: synchronises and prints CTA 0's per-tile timeline (cycles relative to its first stamp)
    std::vector<unsigned long long> h(trace_words);
    P3_CUDA(cudaStreamSynchronize(s));
    P3_CUDA(cudaMemcpy(h.data(), p.trace, trace_words * 8, cudaMemcpyDeviceToHost));
    P3_CUDA(cudaFree(p.trace));
    unsigned long long h2[8 * 4 * 8];
    P3_CUDA(cudaMemcpy(h2, p.trace2, sizeof(h2), cudaMemcpyDeviceToHost));
    P3_CUDA(cudaFree(p.trace2));
    for (int it = 2; it < 5; ++it)
      for (int g = 0; g < 4 && h2[(it * 4 + g) * 8]; ++g) {
        const unsigned long long* q = &h2[(it * 4 + g) * 8];
        fprintf(stderr, "[tc_trace2] tile%d group%d: box_free=+%lld ld0=+%lld conv0=+%lld ld1=+%lld conv1=+%lld store=+%lld\n", it, g,
                (long long)(q[1] - q[0]), (long long)(q[2] - q[1]), (long long)(q[3] - q[2]), (long long)(q[4] - q[3]),
                (long long)(q[5] - q[4]), (long long)(q[6] - q[5]));
      }
    fprintf(stderr, "[tc_trace] M=%d N=%d K=%d BN=%d CL=%d grid=%d ares=%d stages=%d\n", p.M, p.N, p.K, p.BN, CL, clusters * CL, p.ares, p.stages);
    for (int cta = 0; cta < 2; ++cta) {
      const unsigned long long t0 = h[(((size_t)cta * 64 + 0) * 3 + 1) * 4 + 0];
      for (int it = 0; it < 8; ++it) {
        const unsigned long long* q = &h[(((size_t)cta * 64 + it) * 3) * 4];
        if (!q[4]) break;
        auto rel = [&](unsigned long long v) { return v ? (long long)(v - t0) : -1ll; };
        fprintf(stderr, "[tc_trace] cta%d tile%d  tma[first=%lld last=%lld]  mma[start=%lld tempty_ok=%lld data_ok=%lld done_issue=%lld]  epi[wait=%lld tfull_ok=%lld released=%lld end=%lld]\n",
                cta, it, rel(q[0]), rel(q[1]), rel(q[4]), rel(q[5]), rel(q[6]), rel(q[7]), rel(q[8]), rel(q[9]), rel(q[10]), rel(q[11]));
      }
    }
  }
  return P3TOK_OK;
}

int tc_linear_ex(const __nv_bfloat16* A, int64_t M, int K, const __nv_bfloat16* W, int N, const float* bias, int relu,
                 const TcExtra& ex, __nv_bfloat16* out_bf16, float* out_f32, cudaStream_t s) {
  return tc_linear(A, M, K, W, N, bias, nullptr, 1, relu, out_bf16, out_f32, nullptr, nullptr, 0, s, &ex);
}

// ------------------------------------------------------------------------------------------------ first layer
// Narrow input: one CTA = 32 rows (one k=32 patch when aligned), 128 threads x 2 output channels per pass.
template <typename IdxT, int CP>   // CP = padded input width (8 or 16)
__global__ void __launch_bounds__(128)
rows_first_layer_kernel(p3tok_rows R, int64_t g_begin, int64_t nrows, const __nv_bfloat16* __restrict__ W,
                        const float* __restrict__ bias, int cin, int nout, int relu, __nv_bfloat16* __restrict__ out,
                        __nv_bfloat16* __restrict__ gmax32) {   // gmax32: optional max over each block of 32 rows
  __shared__ __align__(16) float xin[32][CP];
  const int64_t r0 = (int64_t)blockIdx.x * 32;
  const IdxT* knn = reinterpret_cast<const IdxT*>(R.knn_idx);
  for (int e = threadIdx.x; e < 32 * CP; e += 128) {
    const int rr = e / CP, c = e % CP;
    const int64_t r = r0 + rr;
    float v = 0.f;          // columns >= cin and rows >= nrows stay zero
    if (r < nrows && c < cin) {
      if (R.kind == 2) {
        v = R.x[(g_begin * R.k + r) * cin + c];
      } else {
        const int n = (int)(r % R.k);
        const int64_t bj = g_begin + r / R.k;
        const int64_t b = bj / R.G;
        const int64_t g = R.perm ? R.perm[bj] : (bj - b * R.G);
        const int64_t ni = (int64_t)knn[(b * R.G + g) * R.k + n];
        if (R.kind == 0) {
          const float* crow = R.x + (b * R.N + R.ctr_idx[b * R.G + g]) * R.C;
          v = c < R.C ? __fsub_rn(R.x[(b * R.N + ni) * R.C + c], crow[c]) : crow[c - R.C];
        } else {
          v = c < 3 ? R.x[(b * R.N + ni) * 3 + c] : R.feats[(b * R.N + ni) * R.D + (c - 3)];
        }
      }
    }
    xin[rr][c] = v;
  }
  __syncthreads();
  for (int n0 = threadIdx.x * 2; n0 < nout; n0 += 256) {
    float w0[CP], w1[CP];
#pragma unroll
    for (int c = 0; c < CP; ++c) {
      w0[c] = c < cin ? __bfloat162float(W[(size_t)n0 * cin + c]) : 0.f;
      w1[c] = (c < cin && n0 + 1 < nout) ? __bfloat162float(W[(size_t)(n0 + 1) * cin + c]) : 0.f;
    }
    const float b0 = bias ? bias[n0] : 0.f, b1 = (bias && n0 + 1 < nout) ? bias[n0 + 1] : 0.f;
    float m0 = -3.0e38f, m1 = -3.0e38f;
    for (int rr = 0; rr < 32; ++rr) {
      const int64_t r = r0 + rr;
      if (r >= nrows) break;
      float a0 = b0, a1 = b1;
#pragma unroll
      for (int c4 = 0; c4 < CP; c4 += 4) {
        const float4 xv = *reinterpret_cast<const float4*>(&xin[rr][c4]);   // warp-wide broadcast
        a0 = fmaf(w0[c4], xv.x, a0); a1 = fmaf(w1[c4], xv.x, a1);
        a0 = fmaf(w0[c4 + 1], xv.y, a0); a1 = fmaf(w1[c4 + 1], xv.y, a1);
        a0 = fmaf(w0[c4 + 2], xv.z, a0); a1 = fmaf(w1[c4 + 2], xv.z, a1);
        a0 = fmaf(w0[c4 + 3], xv.w, a0); a1 = fmaf(w1[c4 + 3], xv.w, a1);
      }
      if (relu) { a0 = fmaxf(a0, 0.f); a1 = fmaxf(a1, 0.f); }
      m0 = fmaxf(m0, a0); m1 = fmaxf(m1, a1);
      *reinterpret_cast<__nv_bfloat162*>(out + r * nout + n0) = __floats2bfloat162_rn(a0, a1);
    }
    // the block is one k = 32 patch: its max-pool is thread-local (bf16 rounding is monotonic, so rounding the
    // fp32 max equals the max of the rounded activations the next GEMM reads)
    if (gmax32) *reinterpret_cast<__nv_bfloat162*>(gmax32 + (r0 >> 5) * nout + n0) = __floats2bfloat162_rn(m0, m1);
  }
}

// Narrow P3Embed / direct rows (kind 1 or 2, cin <= 8) with nout = 32 * NPL.  One WARP owns a 32-row block at a time
// (lane = row for the gather, lane = NPL consecutive output channels for the layer), walks several blocks and has the
// next block's gathered inputs in registers while it computes the current one: no block-level barrier, the two
// dependent global loads (neighbour index -> point) of block i+1 overlap the FMAs of block i.  The generic kernel above
// left half of its threads idle at nout = 128, paid three 64-bit divisions per gathered element and exposed the gather
// latency once per CTA (133 us per 2^20 rows).
template <typename IdxT, int NPL>
__global__ void __launch_bounds__(128)
rows_first_layer_narrow_kernel(p3tok_rows R, int64_t g_begin, int64_t nrows, const __nv_bfloat16* __restrict__ W,
                               const float* __restrict__ bias, int cin, int relu, __nv_bfloat16* __restrict__ out,
                               __nv_bfloat16* __restrict__ gmax32) {
  constexpr int NOUT = 32 * NPL;
  __shared__ __align__(16) float xin_all[4][32][8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float (*xin)[8] = xin_all[warp];
  const int64_t nblocks = (nrows + 31) >> 5;
  const int64_t wstride = (int64_t)gridDim.x * 4;
  // gathered input of row (blk*32 + lane): 8 floats, zero beyond cin / nrows
  auto gather = [&](int64_t blk, float (&v)[8]) {
#pragma unroll
    for (int c = 0; c < 8; ++c) v[c] = 0.f;
    const int64_t r = blk * 32 + lane;
    if (blk >= nblocks || r >= nrows) return;
    if (R.kind == 2) {
      const float* src = R.x + (g_begin * R.k + r) * cin;
#pragma unroll
      for (int c = 0; c < 8; ++c) if (c < cin) v[c] = src[c];
    } else {
      const int64_t gq = r / R.k;
      const int n = (int)(r - gq * R.k);
      const int64_t bj = g_begin + gq;
      const int64_t b = bj / R.G;
      const int64_t ni = (int64_t)reinterpret_cast<const IdxT*>(R.knn_idx)[bj * R.k + n];
      const float* pr = R.x + (b * R.N + ni) * 3;
      const float* fr = R.feats + (b * R.N + ni) * R.D;
      v[0] = pr[0]; v[1] = pr[1]; v[2] = pr[2];
#pragma unroll
      for (int c = 3; c < 8; ++c) if (c < cin) v[c] = fr[c - 3];
    }
  };
  float w[NPL][8], b[NPL];
#pragma unroll
  for (int j = 0; j < NPL; ++j) {
    const int n = lane * NPL + j;
    b[j] = bias ? bias[n] : 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) w[j][c] = c < cin ? __bfloat162float(W[(size_t)n * cin + c]) : 0.f;
  }
  int64_t blk = (int64_t)blockIdx.x * 4 + warp;
  float nxt[8];
  gather(blk, nxt);
  for (; blk < nblocks; blk += wstride) {
    __syncwarp();                                    // the previous block's broadcasts are done
    *reinterpret_cast<float4*>(&xin[lane][0]) = make_float4(nxt[0], nxt[1], nxt[2], nxt[3]);
    *reinterpret_cast<float4*>(&xin[lane][4]) = make_float4(nxt[4], nxt[5], nxt[6], nxt[7]);
    __syncwarp();
    gather(blk + wstride, nxt);                      // in flight during the loop below
    const int64_t r0 = blk * 32;
    const int nr = (int)((nrows - r0) < 32 ? (nrows - r0) : 32);
    float m[NPL];
#pragma unroll
    for (int j = 0; j < NPL; ++j) m[j] = -3.0e38f;
    // The kernel is ISSUE-bound (ncu: 71 % issue-active, DRAM 41 %; 54 warp instructions per row in round 1), so: two output
    // channels per FFMA2, only the cin channels that exist (the zero-padded ones added +0), ReLU folded into the bf16
    // conversion and applied to the patch max once per block (max relu = relu max).
    auto row_loop = [&](auto cin_tag) {
    constexpr int CIN = decltype(cin_tag)::value;
#pragma unroll 4
    for (int row = 0; row < nr; ++row) {
      const float4 x0 = *reinterpret_cast<const float4*>(&xin[row][0]);   // warp-wide broadcasts
      const float4 x1 = *reinterpret_cast<const float4*>(&xin[row][4]);
      const float xr[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
      float a[NPL];
#pragma unroll
      for (int j = 0; j < NPL; ++j) a[j] = b[j];
#pragma unroll
      for (int c = 0; c < CIN; ++c) {
#pragma unroll
        for (int j = 0; j < NPL; j += 2) fma2(a[j], a[j + 1], w[j][c], w[j + 1][c], xr[c], xr[c], a[j], a[j + 1]);
      }
#pragma unroll
      for (int j = 0; j < NPL; ++j) m[j] = fmaxf(m[j], a[j]);
      uint32_t pk[NPL / 2];
#pragma unroll
      for (int j = 0; j < NPL / 2; ++j) pk[j] = relu ? pack_bf16x2_relu(a[2 * j], a[2 * j + 1]) : pack_bf16x2(a[2 * j], a[2 * j + 1]);
      __nv_bfloat16* o = out + (r0 + row) * NOUT + lane * NPL;
      if (NPL == 2) *reinterpret_cast<uint32_t*>(o) = pk[0];
      else if (NPL == 4) *reinterpret_cast<uint2*>(o) = make_uint2(pk[0], pk[1 % (NPL / 2)]);
      else *reinterpret_cast<uint4*>(o) = make_uint4(pk[0], pk[1 % (NPL / 2)], pk[2 % (NPL / 2)], pk[3 % (NPL / 2)]);
    }
    };
    if (cin == 6) row_loop(std::integral_constant<int, 6>{});
    else if (cin <= 4) row_loop(std::integral_constant<int, 4>{});
    else row_loop(std::integral_constant<int, 8>{});
    if (gmax32) {
      // bf16 rounding is monotonic: rounding the fp32 max equals the max of the rounded activations the next GEMM reads
      uint32_t pm[NPL / 2];
#pragma unroll
      for (int j = 0; j < NPL / 2; ++j) pm[j] = relu ? pack_bf16x2_relu(m[2 * j], m[2 * j + 1]) : pack_bf16x2(m[2 * j], m[2 * j + 1]);
      __nv_bfloat16* o = gmax32 + blk * NOUT + lane * NPL;
      if (NPL == 2) *reinterpret_cast<uint32_t*>(o) = pm[0];
      else if (NPL == 4) *reinterpret_cast<uint2*>(o) = make_uint2(pm[0], pm[1 % (NPL / 2)]);
      else *reinterpret_cast<uint4*>(o) = make_uint4(pm[0], pm[1 % (NPL / 2)], pm[2 % (NPL / 2)], pm[3 % (NPL / 2)]);
    }
  }
}

// APF rows whose 32-row block lies inside one patch (k % 32 == 0): the input is [nbr - ctr || ctr], and the centre
// half is the same for all 32 rows, so its contribution W[:, C:2C].ctr + bias is formed once per block and each
// row costs C (3 or 4) FMAs per output channel instead of 2C (apf.py:83-95 feeding apf.py:130).
template <typename IdxT>
__global__ void __launch_bounds__(128)
rows_first_layer_apf_kernel(p3tok_rows R, int64_t g_begin, int64_t nrows, const __nv_bfloat16* __restrict__ W,
                            const float* __restrict__ bias, int nout, int relu, __nv_bfloat16* __restrict__ out) {
  __shared__ __align__(16) float rel[32][4];
  __shared__ float ctr[4];
  const int C = R.C, cin = 2 * C;
  const int64_t r0 = (int64_t)blockIdx.x * 32;
  const IdxT* knn = reinterpret_cast<const IdxT*>(R.knn_idx);
  const int64_t bj = g_begin + r0 / R.k;               // output group of the whole block
  const int64_t b = bj / R.G;
  const int64_t g = R.perm ? R.perm[bj] : (bj - b * R.G);
  const float* crow = R.x + (b * R.N + R.ctr_idx[b * R.G + g]) * C;
  if (threadIdx.x < 32) {
    const int64_t r = r0 + threadIdx.x;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r < nrows) {
      const int64_t ni = (int64_t)knn[(b * R.G + g) * R.k + (r % R.k)];
      const float* prow = R.x + (b * R.N + ni) * C;
      v.x = __fsub_rn(prow[0], crow[0]);
      v.y = __fsub_rn(prow[1], crow[1]);
      v.z = __fsub_rn(prow[2], crow[2]);
      if (C == 4) v.w = __fsub_rn(prow[3], crow[3]);
    }
    *reinterpret_cast<float4*>(&rel[threadIdx.x][0]) = v;
  } else if (threadIdx.x < 36) {
    const int c = threadIdx.x - 32;
    ctr[c] = c < C ? crow[c] : 0.f;
  }
  __syncthreads();
  for (int n0 = threadIdx.x * 2; n0 < nout; n0 += 256) {
    float w0[4], w1[4];
    float base0 = bias ? bias[n0] : 0.f, base1 = bias ? bias[n0 + 1] : 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const bool ok = c < C;
      w0[c] = ok ? __bfloat162float(W[(size_t)n0 * cin + c]) : 0.f;
      w1[c] = ok ? __bfloat162float(W[(size_t)(n0 + 1) * cin + c]) : 0.f;
      if (ok) {
        base0 = fmaf(__bfloat162float(W[(size_t)n0 * cin + C + c]), ctr[c], base0);
        base1 = fmaf(__bfloat162float(W[(size_t)(n0 + 1) * cin + C + c]), ctr[c], base1);
      }
    }
#pragma unroll 4
    for (int rr = 0; rr < 32; ++rr) {
      const int64_t r = r0 + rr;
      if (r >= nrows) break;
      const float4 xv = *reinterpret_cast<const float4*>(&rel[rr][0]);   // warp-wide broadcast
      float a0 = fmaf(w0[0], xv.x, base0), a1 = fmaf(w1[0], xv.x, base1);
      a0 = fmaf(w0[1], xv.y, a0); a1 = fmaf(w1[1], xv.y, a1);
      a0 = fmaf(w0[2], xv.z, a0); a1 = fmaf(w1[2], xv.z, a1);
      a0 = fmaf(w0[3], xv.w, a0); a1 = fmaf(w1[3], xv.w, a1);
      if (relu) { a0 = fmaxf(a0, 0.f); a1 = fmaxf(a1, 0.f); }
      *reinterpret_cast<__nv_bfloat162*>(out + r * nout + n0) = __floats2bfloat162_rn(a0, a1);
    }
  }
}

// Warp-persistent form of the kernel above for nout = 32 * NPL (APF: 256): one warp owns a 32-row block at a time (lane =
// row for the gather, lane = NPL consecutive output channels for the layer) and has the next block's gathered inputs in
// registers while it computes the current one, so the dependent loads perm -> centre index -> centre row and neighbour
// index -> neighbour row overlap the FMAs (82 us per 2^19 rows before, bound by that chain once per CTA).
template <typename IdxT, int NPL>
__global__ void __launch_bounds__(128)
rows_first_layer_apf_warp_kernel(p3tok_rows R, int64_t g_begin, int64_t nrows, const __nv_bfloat16* __restrict__ W,
                                 const float* __restrict__ bias, int relu, __nv_bfloat16* __restrict__ out) {
  constexpr int NOUT = 32 * NPL;
  __shared__ __align__(16) float rel_all[4][32][4];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float (*rel)[4] = rel_all[warp];
  const int C = R.C, cin = 2 * C;
  const IdxT* knn = reinterpret_cast<const IdxT*>(R.knn_idx);
  const int64_t nblocks = (nrows + 31) >> 5;
  const int64_t wstride = (int64_t)gridDim.x * 4;
  // row (blk*32 + lane): v = neighbour - centre (zero beyond C / nrows), c = the block's centre row (same in every lane)
  auto gather = [&](int64_t blk, float4& v, float4& c) {
    v = make_float4(0.f, 0.f, 0.f, 0.f);
    c = v;
    if (blk >= nblocks) return;
    const int64_t r0 = blk * 32;
    const int64_t bj = g_begin + r0 / R.k;               // output group of the whole block (k % 32 == 0)
    const int64_t b = bj / R.G;
    const int64_t g = R.perm ? R.perm[bj] : (bj - b * R.G);
    const float* crow = R.x + (b * R.N + R.ctr_idx[b * R.G + g]) * C;
    c.x = crow[0]; c.y = crow[1]; c.z = crow[2];
    if (C == 4) c.w = crow[3];
    const int64_t r = r0 + lane;
    if (r < nrows) {
      const int64_t ni = (int64_t)knn[(b * R.G + g) * R.k + (r % R.k)];
      const float* prow = R.x + (b * R.N + ni) * C;
      v.x = __fsub_rn(prow[0], c.x);
      v.y = __fsub_rn(prow[1], c.y);
      v.z = __fsub_rn(prow[2], c.z);
      if (C == 4) v.w = __fsub_rn(prow[3], c.w);
    }
  };
  float wr[NPL][4], wc[NPL][4], b0[NPL];
#pragma unroll
  for (int j = 0; j < NPL; ++j) {
    const int n = lane * NPL + j;
    b0[j] = bias ? bias[n] : 0.f;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      wr[j][c] = c < C ? __bfloat162float(W[(size_t)n * cin + c]) : 0.f;
      wc[j][c] = c < C ? __bfloat162float(W[(size_t)n * cin + C + c]) : 0.f;
    }
  }
  int64_t blk = (int64_t)blockIdx.x * 4 + warp;
  float4 nv, nc;
  gather(blk, nv, nc);
  for (; blk < nblocks; blk += wstride) {
    const float4 cc = nc;
    __syncwarp();                                    // the previous block's broadcasts are done
    *reinterpret_cast<float4*>(&rel[lane][0]) = nv;
    __syncwarp();
    gather(blk + wstride, nv, nc);                   // in flight during the loop below
    float base[NPL];
#pragma unroll
    for (int j = 0; j < NPL; ++j)
      base[j] = fmaf(wc[j][3], cc.w, fmaf(wc[j][2], cc.z, fmaf(wc[j][1], cc.y, fmaf(wc[j][0], cc.x, b0[j]))));
    const int64_t r0 = blk * 32;
    const int nr = (int)((nrows - r0) < 32 ? (nrows - r0) : 32);
#pragma unroll 2
    for (int row = 0; row < nr; ++row) {
      const float4 xv = *reinterpret_cast<const float4*>(&rel[row][0]);   // warp-wide broadcast
      uint32_t pk[NPL / 2];
#pragma unroll
      for (int j = 0; j < NPL; j += 2) {
        float a0 = fmaf(wr[j][0], xv.x, base[j]), a1 = fmaf(wr[j + 1][0], xv.x, base[j + 1]);
        a0 = fmaf(wr[j][1], xv.y, a0); a1 = fmaf(wr[j + 1][1], xv.y, a1);
        a0 = fmaf(wr[j][2], xv.z, a0); a1 = fmaf(wr[j + 1][2], xv.z, a1);
        a0 = fmaf(wr[j][3], xv.w, a0); a1 = fmaf(wr[j + 1][3], xv.w, a1);
        pk[j / 2] = relu ? pack_bf16x2_relu(a0, a1) : pack_bf16x2(a0, a1);
      }
      __nv_bfloat16* o = out + (r0 + row) * NOUT + lane * NPL;
      if (NPL == 2) *reinterpret_cast<uint32_t*>(o) = pk[0];
      else if (NPL == 4) *reinterpret_cast<uint2*>(o) = make_uint2(pk[0], pk[1 % (NPL / 2)]);
      else *reinterpret_cast<uint4*>(o) = make_uint4(pk[0], pk[1 % (NPL / 2)], pk[2 % (NPL / 2)], pk[3 % (NPL / 2)]);
    }
  }
}

// Inputs of the APF first layer when it runs INSIDE the pair kernel (embed_fused.cu, FusedL1): rel[r] = neighbour - centre
// (fp32, the reference's subtraction, apf.py:83-84) for every row of the chunk and the centre row of every 32-row block -
// 16 bytes per row instead of the 512-byte bf16 first-layer row.  Rows in [nrows, nrows_pad) are zero-filled (the pair
// kernel's last tile reads whole 128-row slices).
template <typename IdxT>
__global__ void __launch_bounds__(256)
apf_rel_rows_kernel(p3tok_rows R, int64_t g_begin, int64_t nrows, int64_t nrows_pad, float4* __restrict__ rel, float4* __restrict__ ctr) {
  const int C = R.C;
  const IdxT* knn = reinterpret_cast<const IdxT*>(R.knn_idx);
  for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < nrows_pad; r += (int64_t)gridDim.x * blockDim.x) {
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f), c = v;
    if (r < nrows) {
      const int64_t bj = g_begin + r / R.k;                // output group (k % 32 == 0: the same for a whole 32-row block)
      const int64_t b = bj / R.G;
      const int64_t g = R.perm ? R.perm[bj] : (bj - b * R.G);
      const float* crow = R.x + (b * R.N + R.ctr_idx[b * R.G + g]) * C;
      c.x = crow[0]; c.y = crow[1]; c.z = crow[2];
      if (C == 4) c.w = crow[3];
      const int64_t ni = (int64_t)knn[(b * R.G + g) * R.k + (r % R.k)];
      const float* prow = R.x + (b * R.N + ni) * C;
      v.x = __fsub_rn(prow[0], c.x);
      v.y = __fsub_rn(prow[1], c.y);
      v.z = __fsub_rn(prow[2], c.z);
      if (C == 4) v.w = __fsub_rn(prow[3], c.w);
    }
    rel[r] = v;
    if ((r & 31) == 0) ctr[r >> 5] = c;
  }
}

// Wide input: gather rows to bf16 [nrows, kpad], zero padded
template <typename IdxT>
__global__ void rows_gather_bf16_kernel(p3tok_rows R, int64_t g_begin, int64_t nrows, int cin, int kpad,
                                        __nv_bfloat16* __restrict__ out) {
  const IdxT* knn = reinterpret_cast<const IdxT*>(R.knn_idx);
  const int64_t total = nrows * kpad;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(e % kpad);
    const int64_t r = e / kpad;
    float v = 0.f;
    if (c < cin) {
      if (R.kind == 2) {
        v = R.x[(g_begin * R.k + r) * cin + c];
      } else {
        const int n = (int)(r % R.k);
        const int64_t bj = g_begin + r / R.k;
        const int64_t b = bj / R.G;
        const int64_t g = R.perm ? R.perm[bj] : (bj - b * R.G);
        const int64_t ni = (int64_t)knn[(b * R.G + g) * R.k + n];
        if (R.kind == 0) {
          const float* crow = R.x + (b * R.N + R.ctr_idx[b * R.G + g]) * R.C;
          v = c < R.C ? __fsub_rn(R.x[(b * R.N + ni) * R.C + c], crow[c]) : crow[c - R.C];
        } else {
          v = c < 3 ? R.x[(b * R.N + ni) * 3 + c] : R.feats[(b * R.N + ni) * R.D + (c - 3)];
        }
      }
    }
    out[e] = __float2bfloat16_rn(v);
  }
}

// P3Embed rows with D % 4 == 0 (stage >= 1: D = previous stage width): one warp per row, the feature row is one
// coalesced float4 sweep.  Column order is ROTATED to [feats (D) | xyz (3) | zero pad] so that the 8-byte bf16 stores
// stay aligned; pad_weight_kernel rotates the weight columns the same way (rot = 3).
template <typename IdxT>
__global__ void __launch_bounds__(256)
rows_gather_p4p_bf16_kernel(p3tok_rows R, int64_t g_begin, int64_t nrows, int kpad, __nv_bfloat16* __restrict__ out) {
  const IdxT* knn = reinterpret_cast<const IdxT*>(R.knn_idx);
  const int lane = threadIdx.x & 31;
  const int D = R.D, d4 = D >> 2, tail4 = (kpad - D) >> 2;       // kpad % 8 == 0, D % 4 == 0
  const int64_t warp0 = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  // four rows per warp iteration: the four neighbour indices, then the four feature rows, are independent loads in flight
  // together (one row per iteration was bound by two dependent round trips: 305 us per 2^20 rows)
  for (int64_t r4 = warp0 * 4; r4 < nrows; r4 += nwarps * 4) {
    const float4* src[4];
    const float* pr[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int64_t r = (r4 + u < nrows) ? r4 + u : nrows - 1;
      const int64_t gq = r / R.k;
      const int64_t bj = g_begin + gq;
      const int64_t b = bj / R.G;
      const int64_t ni = (int64_t)knn[bj * R.k + (r - gq * R.k)];
      src[u] = reinterpret_cast<const float4*>(R.feats + (b * R.N + ni) * D);
      pr[u] = R.x + (b * R.N + ni) * 3;
    }
    for (int c = lane; c < d4; c += 32) {
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = __ldg(src[u] + c);
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (r4 + u < nrows)
          reinterpret_cast<uint2*>(out + (r4 + u) * kpad)[c] = make_uint2(pack_bf16x2(v[u].x, v[u].y), pack_bf16x2(v[u].z, v[u].w));
    }
    if (lane < 4 * tail4) {                          // [xyz, 0 | zeros] tail of row u = lane / tail4
      const int u = lane / tail4, piece = lane - u * tail4;
      if (r4 + u < nrows) {
        uint2 t = make_uint2(0u, 0u);
        if (piece == 0) t = make_uint2(pack_bf16x2(pr[u][0], pr[u][1]), pack_bf16x2(pr[u][2], 0.f));
        reinterpret_cast<uint2*>(out + (r4 + u) * kpad)[d4 + piece] = t;
      }
    }
  }
}

// out[n][c] = W[n][(c + rot) % K] for c < K, zero padding up to kpad (rot = 3 with the rotated P3Embed row layout)
__global__ void pad_weight_kernel(const __nv_bfloat16* __restrict__ W, int N, int K, int kpad, int rot, __nv_bfloat16* __restrict__ out) {
  const int total = N * kpad;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    const int c = e % kpad, n = e / kpad;
    out[e] = c < K ? W[(size_t)n * K + (c + rot) % K] : __float2bfloat16_rn(0.f);
  }
}

// max over `parts` consecutive partial rows (k = 32*parts): in [ngroups*parts, C] -> out [ngroups, C]
__global__ void partial_max_kernel(const float* __restrict__ in, int64_t ngroups, int parts, int C, float* out_f32,
                                   __nv_bfloat16* out_bf16) {
  const int64_t total = ngroups * C;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g = e / C;
    const int c = (int)(e - g * C);
    float m = in[(g * parts) * C + c];
    for (int q = 1; q < parts; ++q) m = fmaxf(m, in[(g * parts + q) * C + c]);
    if (out_f32) out_f32[e] = m;
    if (out_bf16) out_bf16[e] = __float2bfloat16_rn(m);
  }
}

// the same for bf16 partial maxima (the fused "pre" pair emits its 32-row maxima in bf16, read back from its store boxes)
__global__ void partial_max_bf16_kernel(const __nv_bfloat16* __restrict__ in, int64_t ngroups, int parts, int C,
                                        __nv_bfloat16* __restrict__ out) {
  const int64_t total = ngroups * C;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g = e / C;
    const int c = (int)(e - g * C);
    float m = __bfloat162float(in[(g * parts) * C + c]);
    for (int q = 1; q < parts; ++q) m = fmaxf(m, __bfloat162float(in[(g * parts + q) * C + c]));
    out[e] = __float2bfloat16_rn(m);
  }
}

// generic group max for k not a multiple of 32: in fp32 [ngroups*k, C]
__global__ void group_max_f32_kernel(const float* __restrict__ in, int64_t ngroups, int k, int C, int relu, float* out_f32,
                                     __nv_bfloat16* out_bf16) {
  const int64_t total = ngroups * C;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g = e / C;
    const int c = (int)(e - g * C);
    const float* q = in + g * k * C + c;
    float m = q[0];
    for (int r = 1; r < k; ++r) m = fmaxf(m, q[(int64_t)r * C]);
    if (relu) m = fmaxf(m, 0.f);
    if (out_f32) out_f32[e] = m;
    if (out_bf16) out_bf16[e] = __float2bfloat16_rn(m);
  }
}

__global__ void group_max_bf16_kernel(const __nv_bfloat16* __restrict__ in, int64_t ngroups, int k, int C,
                                      __nv_bfloat16* __restrict__ out) {
  const int64_t total = ngroups * C;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g = e / C;
    const int c = (int)(e - g * C);
    const __nv_bfloat16* q = in + g * k * C + c;
    float m = __bfloat162float(q[0]);
    for (int r = 1; r < k; ++r) m = fmaxf(m, __bfloat162float(q[(int64_t)r * C]));
    out[e] = __float2bfloat16_rn(m);
  }
}

static inline unsigned grid_1d(int64_t total, int threads) {
  int64_t b = (total + threads - 1) / threads;
  const int64_t cap = 148 * 16;
  return (unsigned)(b < 1 ? 1 : (b > cap ? cap : b));
}

// ------------------------------------------------------------------------------------------------ orchestration
// Chunking: one chunk of rows goes through all layers before the next starts.  Measured on B200 (C2,
// 524288 rows): per-launch fixed cost (prologue, pipeline fill, last-tile epilogue) outweighs keeping a
// chunk's activations L2-resident - 2-wave chunks 1.91 ms, 16-wave chunks 1.35 ms - so chunks are as
// large as a bounded workspace allows (default 2^20 rows: <= 1.6 GB per bf16 activation buffer at 768
// columns).  P3TOK_CHUNK_ROWS overrides for experiments.
// `wmax` = widest bf16 activation of the block: the default chunk keeps one activation buffer at <= 1.6 GB (2^20 rows
// at 768 columns) but lets narrow blocks (P3Embed stage 0: 256 columns) run 3x larger chunks - fewer launches, fewer
// pipeline fills and tails per row.
static int64_t chunk_groups(int64_t ngroups, int64_t k, int64_t wmax) {
  static int64_t rows_env = -1;
  if (rows_env < 0) {
    const char* e = getenv("P3TOK_CHUNK_ROWS");
    rows_env = e ? atoll(e) : 0;
  }
  int64_t rows_target = rows_env;
  if (rows_target <= 0) {
    rows_target = (1ll << 20) * 768 / (wmax > 0 ? wmax : 768);
    if (rows_target < (1ll << 20)) rows_target = 1ll << 20;
    if (rows_target > (1ll << 22)) rows_target = 1ll << 22;
  }
  if (rows_target < 128) rows_target = 128;
  int64_t cg = rows_target / k;
  if (cg < 1) cg = 1;
  // equal chunks (the last one would otherwise be a short straggler)
  const int64_t nchunks = (ngroups + cg - 1) / cg;
  if (nchunks > 1) cg = ((ngroups + nchunks - 1) / nchunks + 7) / 8 * 8;   // whole 256-row pair tiles for k = 32
  return ngroups < cg ? ngroups : cg;
}

struct BfLayout {
  int64_t cg, rows, wmax, F, kpad0;
  int64_t off_act0, off_act1, off_gmax_f32, off_gmax_bf16, off_gbias, off_scratch_f32, off_wpad, off_l1, total;
  int64_t l1_rows_pad;              // rows of the chunk padded to whole 256-row pair tiles (0: no in-kernel first layer)
};

// the first layer can run inside the "pre" pair kernel: APF-shaped block (coordinates in, 256 -> N1 -> F per-point layers)
static bool l1_fusable_mlp(const p3tok_mlp* m, int64_t k) {
  return m->cin <= 8 && m->n_pre == 3 && m->pre_dim[0] == 256 && m->pre_relu[0] == 1 && k % 32 == 0;
}

static BfLayout bf_layout(const p3tok_mlp* m, int64_t ngroups, int64_t k) {
  BfLayout L;
  L.F = m->pre_dim[m->n_pre - 1];
  L.kpad0 = m->cin <= 16 ? 0 : align_up(m->cin, 8);
  int64_t w = L.kpad0;
  for (int i = 0; i < m->n_pre; ++i) w = w > m->pre_dim[i] ? w : m->pre_dim[i];
  w = w > m->mid_dim ? w : m->mid_dim;
  L.wmax = w;
  L.cg = chunk_groups(ngroups, k, w);
  L.rows = L.cg * k;
  const int64_t wide = L.F > m->out_dim ? L.F : m->out_dim;
  int64_t o = 0;
  L.off_act0 = o; o += align_up(L.rows * w * 2, 1024);
  L.off_act1 = o; o += align_up(L.rows * w * 2, 1024);
  L.off_gmax_f32 = o; o += align_up((L.rows / 32 + 1) * wide * 4, 1024);
  L.off_gmax_bf16 = o; o += align_up((L.cg + 1) * L.F * 2, 1024);
  L.off_gbias = o; o += align_up(L.cg * m->mid_dim * 4, 1024);
  // fp32 scratch for the unfused max (k not a multiple of 32): one [rows, max(F,out)] matrix
  L.off_scratch_f32 = o; o += (k % 32 == 0) ? 0 : align_up(L.rows * wide * 4, 1024);
  L.off_wpad = o; o += L.kpad0 ? align_up((int64_t)m->pre_dim[0] * align_up(L.kpad0, 64) * 2, 1024) : 0;   // also the 64-padded form
  L.l1_rows_pad = l1_fusable_mlp(m, k) ? align_up(L.rows, 256) : 0;
  L.off_l1 = o;                     // packed first-layer weights | rel rows | block centres
  o += L.l1_rows_pad ? align_up(fused_l1_pack_bytes(), 1024) + L.l1_rows_pad * 16 + align_up(L.l1_rows_pad / 32 * 16, 1024) : 0;
  L.total = o + 1024;
  return L;
}

int64_t patch_embed_bf16_workspace(const p3tok_mlp* m, int64_t ngroups, int64_t k) { return bf_layout(m, ngroups, k).total; }

int patch_embed_bf16(const p3tok_rows* R, const p3tok_mlp* m, void* ws, int64_t ws_bytes, void* tokens, int tokens_bf16,
                     cudaStream_t s) {
  const int64_t ngroups = R->B * R->G, k = R->k;
  const BfLayout L = bf_layout(m, ngroups, k);
  P3_REQUIRE(ws_bytes >= L.total, P3TOK_ERR_WORKSPACE, "patch_embed(bf16): workspace %lld < %lld bytes", (long long)ws_bytes,
             (long long)L.total);
  for (int i = 0; i < m->n_pre; ++i)
    P3_REQUIRE(m->pre_dim[i] % 8 == 0, P3TOK_ERR_UNSUPPORTED, "patch_embed(bf16): layer widths must be multiples of 8");
  P3_REQUIRE(m->mid_dim % 8 == 0 && m->out_dim % 8 == 0, P3TOK_ERR_UNSUPPORTED,
             "patch_embed(bf16): layer widths must be multiples of 8");
  char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 1023) / 1024 * 1024);
  __nv_bfloat16* act[2] = {reinterpret_cast<__nv_bfloat16*>(base + L.off_act0), reinterpret_cast<__nv_bfloat16*>(base + L.off_act1)};
  float* gmax_f32 = reinterpret_cast<float*>(base + L.off_gmax_f32);
  __nv_bfloat16* gmax_bf16 = reinterpret_cast<__nv_bfloat16*>(base + L.off_gmax_bf16);
  float* gbias = reinterpret_cast<float*>(base + L.off_gbias);
  float* scratch = reinterpret_cast<float*>(base + L.off_scratch_f32);
  __nv_bfloat16* wpad = reinterpret_cast<__nv_bfloat16*>(base + L.off_wpad);
  const bool fused_max = (k % 32 == 0);
  const int parts = fused_max ? (int)(k / 32) : 0;
  const bool i64 = (R->kind == 2) || R->idx_dtype == P3TOK_I64;

  // P3Embed rows with a float4-aligned feature width use the rotated [feats | xyz] column order
  const bool rot_rows = L.kpad0 && R->kind == 1 && R->D % 4 == 0 && R->D >= 4 &&
                        (reinterpret_cast<uintptr_t>(R->feats) & 15) == 0;
  // P3Embed stage >= 1 (a single wide per-point layer): the gather runs inside the GEMM's producer (embed_gather.cu) and the
  // row matrix never exists; other shapes gather to bf16 rows for tc_linear.
  const bool gather_fused = rot_rows && m->n_pre == 1 && m->pre_relu[0] == 1 && tc_gather_linear_supported(R, m->pre_dim[0], k);
  const int64_t kpadw = gather_fused ? align_up(L.kpad0, 64) : L.kpad0;
  if (L.kpad0) {
    pad_weight_kernel<<<grid_1d((int64_t)m->pre_dim[0] * kpadw, 256), 256, 0, s>>>(
        (const __nv_bfloat16*)m->w_pre[0], m->pre_dim[0], m->cin, (int)kpadw, rot_rows ? 3 : 0, wpad);
    P3_LAUNCH_CHECK("pad_weight_kernel");
  }

  for (int64_t g0 = 0; g0 < ngroups; g0 += L.cg) {
    const int64_t gc = (ngroups - g0) < L.cg ? (ngroups - g0) : L.cg;
    const int64_t rows = gc * k;
    int cur = 0;
    int rc;
    // ---- first layer: CUDA cores for narrow inputs, otherwise gather to bf16 rows for the tensor cores
    int first_tc = 0;
    int kin;
    // APF blocks: the first layer runs inside the "pre" pair kernel (embed_fused.cu, FusedL1) - its 512-byte bf16 rows are
    // never written; what the pair kernel reads instead is 16 bytes per row (neighbour - centre) + one centre per 32 rows.
    static int fuse_on0 = -1;
    if (fuse_on0 < 0) { const char* e = getenv("P3TOK_FUSED"); fuse_on0 = e ? atoi(e) : 1; }
    FusedL1 l1;
    const bool l1_fused = fuse_on0 && L.l1_rows_pad && !L.kpad0 && R->kind == 0 && (R->C == 3 || R->C == 4) && fused_max &&
                          m->pre_relu[1] == 1 && m->pre_relu[2] == 0 && tc_fused_l1_supported(m->pre_dim[1], m->pre_dim[2]);
    if (l1_fused) {
      char* l1b = base + L.off_l1;
      float* packed = reinterpret_cast<float*>(l1b);
      float4* rel = reinterpret_cast<float4*>(l1b + align_up(fused_l1_pack_bytes(), 1024));
      float4* ctr = rel + L.l1_rows_pad;
      if (g0 == 0) {
        rc = fused_l1_pack((const __nv_bfloat16*)m->w_pre[0], m->b_pre[0], R->C, packed, s);
        if (rc) return rc;
      }
      const int64_t rows_pad = align_up(rows, 256);
      if (i64) apf_rel_rows_kernel<int64_t><<<grid_1d(rows_pad, 256), 256, 0, s>>>(*R, g0, rows, rows_pad, rel, ctr);
      else apf_rel_rows_kernel<int32_t><<<grid_1d(rows_pad, 256), 256, 0, s>>>(*R, g0, rows, rows_pad, rel, ctr);
      P3_LAUNCH_CHECK("apf_rel_rows_kernel");
      l1.rel = rel; l1.ctr = ctr; l1.w = packed; l1.relu = 1;
      first_tc = 1;
      kin = m->pre_dim[0];
    } else if (!L.kpad0) {
      const unsigned blocks = (unsigned)((rows + 31) / 32);
      // single per-point layer (P3Embed stage 0) with k = 32: the first-layer kernel also emits the patch max
      __nv_bfloat16* l1_gmax = (m->n_pre == 1 && k == 32 && m->pre_dim[0] % 2 == 0) ? gmax_bf16 : nullptr;
#define P3_L1(IDX, CPV)                                                                                        \
  rows_first_layer_kernel<IDX, CPV><<<blocks, 128, 0, s>>>(*R, g0, rows, (const __nv_bfloat16*)m->w_pre[0],    \
                                                           m->b_pre[0], m->cin, m->pre_dim[0], m->pre_relu[0], act[cur], l1_gmax)
      if (R->kind == 0 && k % 32 == 0 && (R->C == 3 || R->C == 4) &&
          (m->pre_dim[0] == 64 || m->pre_dim[0] == 128 || m->pre_dim[0] == 256)) {
        const unsigned nb = (unsigned)std::min<int64_t>((blocks + 3) / 4, (int64_t)num_sms() * 10);
#define P3_L1A(IDX, NPL)                                                                                              \
  rows_first_layer_apf_warp_kernel<IDX, NPL><<<nb, 128, 0, s>>>(*R, g0, rows, (const __nv_bfloat16*)m->w_pre[0], m->b_pre[0], \
                                                                 m->pre_relu[0], act[cur])
        const int npl = m->pre_dim[0] / 32;
        if (i64) { if (npl == 2) P3_L1A(int64_t, 2); else if (npl == 4) P3_L1A(int64_t, 4); else P3_L1A(int64_t, 8); }
        else     { if (npl == 2) P3_L1A(int32_t, 2); else if (npl == 4) P3_L1A(int32_t, 4); else P3_L1A(int32_t, 8); }
#undef P3_L1A
      } else if (R->kind == 0 && k % 32 == 0 && (R->C == 3 || R->C == 4) && m->pre_dim[0] % 2 == 0) {
        if (i64) rows_first_layer_apf_kernel<int64_t><<<blocks, 128, 0, s>>>(*R, g0, rows, (const __nv_bfloat16*)m->w_pre[0],
                                                                          m->b_pre[0], m->pre_dim[0], m->pre_relu[0], act[cur]);
        else rows_first_layer_apf_kernel<int32_t><<<blocks, 128, 0, s>>>(*R, g0, rows, (const __nv_bfloat16*)m->w_pre[0],
                                                                         m->b_pre[0], m->pre_dim[0], m->pre_relu[0], act[cur]);
      } else if (R->kind != 0 && m->cin <= 8 && (m->pre_dim[0] == 64 || m->pre_dim[0] == 128 || m->pre_dim[0] == 256)) {
#define P3_L1N(IDX, NPL)                                                                                          \
  rows_first_layer_narrow_kernel<IDX, NPL><<<nblk_narrow, 128, 0, s>>>(*R, g0, rows, (const __nv_bfloat16*)m->w_pre[0], \
                                                                  m->b_pre[0], m->cin, m->pre_relu[0], act[cur], l1_gmax)
        const int npl = m->pre_dim[0] / 32;
        // ~6 row blocks per warp: enough to amortise the weight loads and to keep one gather in flight per warp
        const unsigned nblk_narrow = (unsigned)std::min<int64_t>((blocks + 3) / 4, (int64_t)num_sms() * 10);
        if (i64) { if (npl == 2) P3_L1N(int64_t, 2); else if (npl == 4) P3_L1N(int64_t, 4); else P3_L1N(int64_t, 8); }
        else     { if (npl == 2) P3_L1N(int32_t, 2); else if (npl == 4) P3_L1N(int32_t, 4); else P3_L1N(int32_t, 8); }
#undef P3_L1N
      } else if (m->cin <= 8) { if (i64) P3_L1(int64_t, 8); else P3_L1(int32_t, 8); }
      else             { if (i64) P3_L1(int64_t, 16); else P3_L1(int32_t, 16); }
#undef P3_L1
      P3_LAUNCH_CHECK("rows_first_layer_kernel");
      first_tc = 1;
      kin = m->pre_dim[0];
    } else if (gather_fused) {
      __nv_bfloat16* part_bf16 = reinterpret_cast<__nv_bfloat16*>(gmax_f32);
      rc = tc_gather_linear(R, g0, rows, wpad, m->pre_dim[0], m->b_pre[0], 1, act[cur], parts == 1 ? gmax_bf16 : part_bf16, s);
      if (rc) return rc;
      if (parts > 1) {
        partial_max_bf16_kernel<<<grid_1d(gc * L.F, 256), 256, 0, s>>>(part_bf16, gc, parts, (int)L.F, gmax_bf16);
        P3_LAUNCH_CHECK("partial_max_bf16_kernel");
      }
      first_tc = m->n_pre;            // the block's only per-point layer is done, its patch max too
      kin = m->pre_dim[0];
    } else if (rot_rows) {
      const unsigned blocks = grid_1d(rows * 32, 256);
      if (i64) rows_gather_p4p_bf16_kernel<int64_t><<<blocks, 256, 0, s>>>(*R, g0, rows, (int)L.kpad0, act[cur]);
      else rows_gather_p4p_bf16_kernel<int32_t><<<blocks, 256, 0, s>>>(*R, g0, rows, (int)L.kpad0, act[cur]);
      P3_LAUNCH_CHECK("rows_gather_p4p_bf16_kernel");
      kin = (int)L.kpad0;
    } else {
      if (i64)
        rows_gather_bf16_kernel<int64_t><<<grid_1d(rows * L.kpad0, 256), 256, 0, s>>>(*R, g0, rows, m->cin, (int)L.kpad0, act[cur]);
      else
        rows_gather_bf16_kernel<int32_t><<<grid_1d(rows * L.kpad0, 256), 256, 0, s>>>(*R, g0, rows, m->cin, (int)L.kpad0, act[cur]);
      P3_LAUNCH_CHECK("rows_gather_bf16_kernel");
      kin = (int)L.kpad0;
    }
    // ---- remaining per-point layers on the tensor cores; the last one also emits the patch max
    bool have_gmax = gather_fused;
    static int fuse_on = -1;
    // Layer pairs go through tc_fused_kernel (embed_fused.cu): the hidden activation of each pair never reaches HBM.
    // P3TOK_FUSED=0 selects the layer-by-layer path.  History (same-box A/B, bench.py, ms per step): with 64-column
    // chunks the fused path lost (c2 1.22 vs 1.10); with 128-column chunks - every MMA at its nominal rate - and rings
    // deep enough to cover a TMA round trip it wins: c2 1.017 vs 1.166, c4 10.11 vs 10.72, c5 2.31 vs 2.50, c3 11.99 vs 12.73.
    if (fuse_on < 0) { const char* e = getenv("P3TOK_FUSED"); fuse_on = e ? atoi(e) : 1; }
    const bool fuse_pre = fuse_on && fused_max && (m->n_pre - first_tc == 2) && m->pre_relu[m->n_pre - 2] == 1 &&
                          m->pre_relu[m->n_pre - 1] == 0 &&
                          tc_fused_supported(kin, m->pre_dim[m->n_pre - 2], m->pre_dim[m->n_pre - 1], k, false);
    P3_REQUIRE(fuse_pre || !l1_fused, P3TOK_ERR_UNSUPPORTED, "patch_embed(bf16): in-kernel first layer without the pair kernel");
    if (fuse_pre) {
      // both tensor-core per-point layers in one kernel: the (rows x pre_dim[n-2]) hidden activation stays on-chip
      const int i0 = m->n_pre - 2, i1 = m->n_pre - 1;
      // the pair's epilogue emits the max of every 32 rows in bf16 (read back from its store boxes); k = 32*parts rows
      // per patch: the partial maxima go through the (otherwise unused) fp32 scratch and are combined below
      __nv_bfloat16* part_bf16 = reinterpret_cast<__nv_bfloat16*>(gmax_f32);
      rc = tc_fused(act[cur], rows, kin, (const __nv_bfloat16*)m->w_pre[i0], m->pre_dim[i0], m->b_pre[i0], nullptr, 32,
                    (const __nv_bfloat16*)m->w_pre[i1], m->pre_dim[i1], m->b_pre[i1], act[cur ^ 1],
                    nullptr, parts == 1 ? gmax_bf16 : part_bf16, 0, s, l1_fused ? &l1 : nullptr);
      if (rc) return rc;
      if (parts > 1) {
        partial_max_bf16_kernel<<<grid_1d(gc * L.F, 256), 256, 0, s>>>(part_bf16, gc, parts, (int)L.F, gmax_bf16);
        P3_LAUNCH_CHECK("partial_max_bf16_kernel");
      }
      have_gmax = true;
      cur ^= 1;
      kin = m->pre_dim[i1];
    }
    for (int i = first_tc; i < m->n_pre && !fuse_pre; ++i) {
      const bool last = (i == m->n_pre - 1);
      const __nv_bfloat16* Wi = (i == 0 && L.kpad0) ? wpad : (const __nv_bfloat16*)m->w_pre[i];
      if (last && fused_max) {
        rc = tc_linear(act[cur], rows, kin, Wi, m->pre_dim[i], m->b_pre[i], nullptr, 1, m->pre_relu[i], act[cur ^ 1], nullptr,
                       parts == 1 ? nullptr : gmax_f32, parts == 1 ? gmax_bf16 : nullptr, 0, s);
        if (rc) return rc;
        if (parts > 1) {
          partial_max_kernel<<<grid_1d(gc * L.F, 256), 256, 0, s>>>(gmax_f32, gc, parts, (int)L.F, nullptr, gmax_bf16);
          P3_LAUNCH_CHECK("partial_max_kernel");
        }
        have_gmax = true;
      } else if (last) {
        rc = tc_linear(act[cur], rows, kin, Wi, m->pre_dim[i], m->b_pre[i], nullptr, 1, m->pre_relu[i], act[cur ^ 1], scratch,
                       nullptr, nullptr, 0, s);
        if (rc) return rc;
        group_max_f32_kernel<<<grid_1d(gc * L.F, 256), 256, 0, s>>>(scratch, gc, (int)k, (int)L.F, 0, nullptr, gmax_bf16);
        P3_LAUNCH_CHECK("group_max_f32_kernel");
        have_gmax = true;
      } else {
        rc = tc_linear(act[cur], rows, kin, Wi, m->pre_dim[i], m->b_pre[i], nullptr, 1, m->pre_relu[i], act[cur ^ 1], nullptr,
                       nullptr, nullptr, 0, s);
        if (rc) return rc;
      }
      cur ^= 1;
      kin = m->pre_dim[i];
    }
    if (!have_gmax && !L.kpad0 && m->n_pre == 1 && k == 32 && m->pre_dim[0] % 2 == 0) have_gmax = true;   // emitted by the first-layer kernel
    if (!have_gmax) {
      // the block's only per-point layer ran on CUDA cores (P3Embed stage 0): reduce its bf16 output
      group_max_bf16_kernel<<<grid_1d(gc * L.F, 256), 256, 0, s>>>(act[cur], gc, (int)k, (int)L.F, gmax_bf16);
      P3_LAUNCH_CHECK("group_max_bf16_kernel");
    }
    // ---- concat layer: per-group half (becomes a bias), then the per-point half
    rc = tc_linear(gmax_bf16, gc, (int)L.F, (const __nv_bfloat16*)m->w_mid_g, m->mid_dim, m->b_mid, nullptr, 1, 0, nullptr, gbias,
                   nullptr, nullptr, 0, s);
    if (rc) return rc;
    // the patch tokens leave as f32 (reference dtype) or bf16: rounded once, by the epilogue / reduction that produces them
    float* tok = tokens_bf16 ? nullptr : reinterpret_cast<float*>(tokens) + g0 * m->out_dim;
    __nv_bfloat16* tokb = tokens_bf16 ? reinterpret_cast<__nv_bfloat16*>(tokens) + g0 * m->out_dim : nullptr;
    // narrow blocks (P3Embed stage 0): concat layer + output layer + pool in one kernel with the weights resident in
    // shared memory (embed_stage.cu); the hidden activation never reaches HBM.  P3TOK_STAGE=0 disables it.
    static int stage_on = -1;
    if (stage_on < 0) { const char* e = getenv("P3TOK_STAGE"); stage_on = e ? atoi(e) : 1; }
    if (stage_on && fused_max && tc_stage_supported((int)L.F, m->mid_dim, m->out_dim, k)) {
      rc = tc_stage(act[cur], rows, (int)L.F, (const __nv_bfloat16*)m->w_mid_f, m->mid_dim, nullptr, gbias, (int)k,
                    (const __nv_bfloat16*)m->w_out, m->out_dim, m->b_out, parts == 1 ? tok : gmax_f32, parts == 1 ? tokb : nullptr,
                    parts == 1 ? m->out_relu : 0, s);
      if (rc) return rc;
      if (parts > 1) {
        group_max_f32_kernel<<<grid_1d(gc * m->out_dim, 256), 256, 0, s>>>(gmax_f32, gc, parts, m->out_dim, m->out_relu, tok, tokb);
        P3_LAUNCH_CHECK("group_max_f32_kernel");
      }
      continue;
    }
    if (fuse_on && fused_max && tc_fused_supported((int)L.F, m->mid_dim, m->out_dim, k, true)) {
      // concat layer (per-point half + group bias, ReLU) and output layer in one kernel; only the patch max is written
      rc = tc_fused(act[cur], rows, (int)L.F, (const __nv_bfloat16*)m->w_mid_f, m->mid_dim, nullptr, gbias, (int)k,
                    (const __nv_bfloat16*)m->w_out, m->out_dim, m->b_out, nullptr, parts == 1 ? tok : gmax_f32,
                    parts == 1 ? tokb : nullptr, parts == 1 ? m->out_relu : 0, s);
      if (rc) return rc;
      if (parts > 1) {
        group_max_f32_kernel<<<grid_1d(gc * m->out_dim, 256), 256, 0, s>>>(gmax_f32, gc, parts, m->out_dim, m->out_relu, tok, tokb);
        P3_LAUNCH_CHECK("group_max_f32_kernel");
      }
      continue;
    }
    rc = tc_linear(act[cur], rows, (int)L.F, (const __nv_bfloat16*)m->w_mid_f, m->mid_dim, nullptr, gbias, (int)k, 1, act[cur ^ 1],
                   nullptr, nullptr, nullptr, 0, s);
    if (rc) return rc;
    cur ^= 1;
    // ---- output layer + max over the patch
    if (fused_max) {
      rc = tc_linear(act[cur], rows, m->mid_dim, (const __nv_bfloat16*)m->w_out, m->out_dim, m->b_out, nullptr, 1, 0, nullptr, nullptr,
                     parts == 1 ? tok : gmax_f32, parts == 1 ? tokb : nullptr, parts == 1 ? m->out_relu : 0, s);
      if (rc) return rc;
      if (parts > 1) {
        // ReLU commutes with max: apply it after combining the partial maxima
        group_max_f32_kernel<<<grid_1d(gc * m->out_dim, 256), 256, 0, s>>>(gmax_f32, gc, parts, m->out_dim, m->out_relu, tok, tokb);
        P3_LAUNCH_CHECK("group_max_f32_kernel");
      }
    } else {
      rc = tc_linear(act[cur], rows, m->mid_dim, (const __nv_bfloat16*)m->w_out, m->out_dim, m->b_out, nullptr, 1, 0, nullptr, scratch,
                     nullptr, nullptr, 0, s);
      if (rc) return rc;
      group_max_f32_kernel<<<grid_1d(gc * m->out_dim, 256), 256, 0, s>>>(scratch, gc, (int)k, m->out_dim, m->out_relu, tok, tokb);
      P3_LAUNCH_CHECK("group_max_f32_kernel");
    }
  }
  return P3TOK_OK;
}

// ------------------------------------------------------------------------------------------------ bf16x3 (fp32-accurate) mode
// The rtol-1e-4 contract on the tensor cores: every fp32 operand is carried as hi = bf16(v), lo = bf16(v - hi) (16 mantissa
// bits) and a product a.w is evaluated as a_hi.w_hi + a_lo.w_hi + a_hi.w_lo with fp32 accumulation in tensor memory - ONE
// tcgen05 GEMM over a three-fold reduction length: activations are stored [rows, 2K] = [hi | lo], the host prepares
// W' = [W_hi | W_hi | W_lo] (p3tok/fold.py), and the k-blocks of the third segment re-read the hi half (tc_linear x3).  The
// epilogue splits its fp32 result into the next layer's [hi | lo].  Measured error against the float64 oracle ~7e-6 of max
// (emulation: same figure), against 3e-7 for the CUDA-core fp32 path and 4e-3 for plain bf16.
// Narrow first layers (cin <= 16: the coordinates) stay on CUDA cores in fp32, as in the bf16 mode.
template <typename IdxT>
__global__ void __launch_bounds__(128)
rows_first_layer_split_kernel(p3tok_rows R, int64_t g_begin, int64_t nrows, const float* __restrict__ W, const float* __restrict__ bias,
                              int cin, int nout, int relu, __nv_bfloat16* __restrict__ out, float* __restrict__ out_f32) {
  __shared__ __align__(16) float xin[32][16];
  const int64_t r0 = (int64_t)blockIdx.x * 32;
  const IdxT* knn = reinterpret_cast<const IdxT*>(R.knn_idx);
  for (int e = threadIdx.x; e < 32 * 16; e += 128) {
    const int rr = e >> 4, c = e & 15;
    const int64_t r = r0 + rr;
    float v = 0.f;
    if (r < nrows && c < cin) {
      if (R.kind == 2) {
        v = R.x[(g_begin * R.k + r) * cin + c];
      } else {
        const int n = (int)(r % R.k);
        const int64_t bj = g_begin + r / R.k;
        const int64_t b = bj / R.G;
        const int64_t g = R.perm ? R.perm[bj] : (bj - b * R.G);
        const int64_t ni = (int64_t)knn[(b * R.G + g) * R.k + n];
        if (R.kind == 0) {
          const float* crow = R.x + (b * R.N + R.ctr_idx[b * R.G + g]) * R.C;
          v = c < R.C ? __fsub_rn(R.x[(b * R.N + ni) * R.C + c], crow[c]) : crow[c - R.C];
        } else {
          v = c < 3 ? R.x[(b * R.N + ni) * 3 + c] : R.feats[(b * R.N + ni) * R.D + (c - 3)];
        }
      }
    }
    xin[rr][c] = v;
  }
  __syncthreads();
  for (int n0 = threadIdx.x; n0 < nout; n0 += 128) {
    float w[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) w[c] = c < cin ? W[(size_t)n0 * cin + c] : 0.f;
    const float b0 = bias ? bias[n0] : 0.f;
    for (int rr = 0; rr < 32; ++rr) {
      const int64_t r = r0 + rr;
      if (r >= nrows) break;
      float a = b0;
#pragma unroll
      for (int c = 0; c < 16; ++c) a = fmaf(w[c], xin[rr][c], a);
      if (relu) a = fmaxf(a, 0.f);
      const __nv_bfloat16 hi = __float2bfloat16_rn(a);
      out[r * 2 * nout + n0] = hi;
      out[r * 2 * nout + nout + n0] = __float2bfloat16_rn(a - __bfloat162float(hi));
      if (out_f32) out_f32[r * nout + n0] = a;
    }
  }
}

// wide inputs (P3Embed stage >= 1): gathered rows as split operands [rows, 2 kpad] = [hi | lo], zero padded
template <typename IdxT>
__global__ void rows_gather_split_kernel(p3tok_rows R, int64_t g_begin, int64_t nrows, int cin, int kpad, __nv_bfloat16* __restrict__ out) {
  const IdxT* knn = reinterpret_cast<const IdxT*>(R.knn_idx);
  const int64_t total = nrows * kpad;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(e % kpad);
    const int64_t r = e / kpad;
    float v = 0.f;
    if (c < cin) {
      if (R.kind == 2) {
        v = R.x[(g_begin * R.k + r) * cin + c];
      } else {
        const int n = (int)(r % R.k);
        const int64_t bj = g_begin + r / R.k;
        const int64_t b = bj / R.G;
        const int64_t g = R.perm ? R.perm[bj] : (bj - b * R.G);
        const int64_t ni = (int64_t)knn[(b * R.G + g) * R.k + n];
        if (R.kind == 0) {
          const float* crow = R.x + (b * R.N + R.ctr_idx[b * R.G + g]) * R.C;
          v = c < R.C ? __fsub_rn(R.x[(b * R.N + ni) * R.C + c], crow[c]) : crow[c - R.C];
        } else {
          v = c < 3 ? R.x[(b * R.N + ni) * 3 + c] : R.feats[(b * R.N + ni) * R.D + (c - 3)];
        }
      }
    }
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    out[r * 2 * kpad + c] = hi;
    out[r * 2 * kpad + kpad + c] = __float2bfloat16_rn(v - __bfloat162float(hi));
  }
}

// fp32 [R, C] -> split bf16 [R, 2 cpad] = [hi | lo], zero padded to cpad columns
__global__ void split_rows_kernel(const float* __restrict__ in, int64_t R_, int C, int cpad, __nv_bfloat16* __restrict__ out) {
  const int64_t total = R_ * cpad;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(e % cpad);
    const int64_t r = e / cpad;
    const float v = c < C ? in[r * C + c] : 0.f;
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    out[r * 2 * cpad + c] = hi;
    out[r * 2 * cpad + cpad + c] = __float2bfloat16_rn(v - __bfloat162float(hi));
  }
}

struct X3Layout {
  int64_t cg, rows, wmax, F, wide;
  int64_t off_act0, off_act1, off_max32, off_gmax, off_gsplit, off_gbias, off_scratch, total;
};
static inline int64_t pad64(int64_t v) { return (v + 63) / 64 * 64; }

static X3Layout x3_layout(const p3tok_mlp* m, int64_t ngroups, int64_t k) {
  X3Layout L;
  L.F = m->pre_dim[m->n_pre - 1];
  int64_t w = m->cin > 16 ? pad64(m->cin) : 0;
  for (int i = 0; i < m->n_pre; ++i) w = w > m->pre_dim[i] ? w : m->pre_dim[i];
  w = w > m->mid_dim ? w : m->mid_dim;
  L.wmax = w;
  L.cg = chunk_groups(ngroups, k, 2 * w);
  L.rows = L.cg * k;
  L.wide = L.F > m->out_dim ? L.F : m->out_dim;
  int64_t o = 0;
  L.off_act0 = o; o += align_up(L.rows * 2 * w * 2, 1024);
  L.off_act1 = o; o += align_up(L.rows * 2 * w * 2, 1024);
  L.off_max32 = o; o += align_up((L.rows / 32 + 1) * L.wide * 4, 1024);
  L.off_gmax = o; o += align_up((L.cg + 1) * L.F * 4, 1024);
  L.off_gsplit = o; o += align_up((L.cg + 1) * 2 * pad64(L.F) * 2, 1024);
  L.off_gbias = o; o += align_up(L.cg * m->mid_dim * 4, 1024);
  // fp32 scratch [rows, wide]: the unfused max (k not a multiple of 32) and the max of a CUDA-core-only pre stage
  L.off_scratch = o; o += align_up(L.rows * L.wide * 4, 1024);
  L.total = o + 1024;
  return L;
}

int64_t patch_embed_x3_workspace(const p3tok_mlp* m, int64_t ngroups, int64_t k) { return x3_layout(m, ngroups, k).total; }

// Weights (prepared by p3tok/fold.py, wdtype P3TOK_BF16X3): a first layer with cin <= 16 stays fp32 [N, cin]; every other
// matrix is bf16 [N, 3 pad64(K)] = [W_hi | W_hi | W_lo].
int patch_embed_x3(const p3tok_rows* R, const p3tok_mlp* m, void* ws, int64_t ws_bytes, float* tokens, cudaStream_t s) {
  const int64_t ngroups = R->B * R->G, k = R->k;
  const X3Layout L = x3_layout(m, ngroups, k);
  P3_REQUIRE(ws_bytes >= L.total, P3TOK_ERR_WORKSPACE, "patch_embed(bf16x3): workspace %lld < %lld bytes", (long long)ws_bytes,
             (long long)L.total);
  for (int i = 0; i < m->n_pre; ++i)
    P3_REQUIRE(m->pre_dim[i] % 64 == 0, P3TOK_ERR_UNSUPPORTED, "patch_embed(bf16x3): layer widths must be multiples of 64");
  P3_REQUIRE(m->mid_dim % 64 == 0 && m->out_dim % 64 == 0, P3TOK_ERR_UNSUPPORTED, "patch_embed(bf16x3): layer widths must be multiples of 64");
  char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 1023) / 1024 * 1024);
  __nv_bfloat16* act[2] = {reinterpret_cast<__nv_bfloat16*>(base + L.off_act0), reinterpret_cast<__nv_bfloat16*>(base + L.off_act1)};
  float* max32 = reinterpret_cast<float*>(base + L.off_max32);
  float* gmax = reinterpret_cast<float*>(base + L.off_gmax);
  __nv_bfloat16* gsplit = reinterpret_cast<__nv_bfloat16*>(base + L.off_gsplit);
  float* gbias = reinterpret_cast<float*>(base + L.off_gbias);
  float* scratch = reinterpret_cast<float*>(base + L.off_scratch);
  const bool fused_max = (k % 32 == 0);
  const int parts = fused_max ? (int)(k / 32) : 0;
  const bool i64 = (R->kind == 2) || R->idx_dtype == P3TOK_I64;
  TcExtra ex;
  ex.x3 = 1;
  TcExtra exs = ex;
  exs.out_split = 1;
  const int F = (int)L.F;
  for (int64_t g0 = 0; g0 < ngroups; g0 += L.cg) {
    const int64_t gc = (ngroups - g0) < L.cg ? (ngroups - g0) : L.cg;
    const int64_t rows = gc * k;
    int cur = 0, rc, first_tc, kin;
    bool have_gmax = false;
    if (m->cin <= 16) {
      const bool only = (m->n_pre == 1);                 // the block's only per-point layer: also keep fp32 values for its max
      const unsigned blocks = (unsigned)((rows + 31) / 32);
      if (i64) rows_first_layer_split_kernel<int64_t><<<blocks, 128, 0, s>>>(*R, g0, rows, (const float*)m->w_pre[0], m->b_pre[0], m->cin,
                                                                           m->pre_dim[0], m->pre_relu[0], act[cur], only ? scratch : nullptr);
      else rows_first_layer_split_kernel<int32_t><<<blocks, 128, 0, s>>>(*R, g0, rows, (const float*)m->w_pre[0], m->b_pre[0], m->cin,
                                                                         m->pre_dim[0], m->pre_relu[0], act[cur], only ? scratch : nullptr);
      P3_LAUNCH_CHECK("rows_first_layer_split_kernel");
      if (only) {
        group_max_f32_kernel<<<grid_1d(gc * L.F, 256), 256, 0, s>>>(scratch, gc, (int)k, F, 0, gmax, nullptr);
        P3_LAUNCH_CHECK("group_max_f32_kernel");
        have_gmax = true;
      }
      first_tc = 1;
      kin = m->pre_dim[0];
    } else {
      const int kp = (int)pad64(m->cin);
      if (i64) rows_gather_split_kernel<int64_t><<<grid_1d(rows * kp, 256), 256, 0, s>>>(*R, g0, rows, m->cin, kp, act[cur]);
      else rows_gather_split_kernel<int32_t><<<grid_1d(rows * kp, 256), 256, 0, s>>>(*R, g0, rows, m->cin, kp, act[cur]);
      P3_LAUNCH_CHECK("rows_gather_split_kernel");
      first_tc = 0;
      kin = kp;
    }
    for (int i = first_tc; i < m->n_pre; ++i) {
      const bool last = (i == m->n_pre - 1);
      rc = tc_linear(act[cur], rows, 3 * kin, (const __nv_bfloat16*)m->w_pre[i], m->pre_dim[i], m->b_pre[i], nullptr, 1, m->pre_relu[i],
                     act[cur ^ 1], (last && !fused_max) ? scratch : nullptr, (last && fused_max) ? max32 : nullptr, nullptr, 0, s, &exs);
      if (rc) return rc;
      cur ^= 1;
      kin = m->pre_dim[i];
      if (last) {
        if (fused_max) {
          partial_max_kernel<<<grid_1d(gc * L.F, 256), 256, 0, s>>>(max32, gc, parts, F, gmax, nullptr);
          P3_LAUNCH_CHECK("partial_max_kernel");
        } else {
          group_max_f32_kernel<<<grid_1d(gc * L.F, 256), 256, 0, s>>>(scratch, gc, (int)k, F, 0, gmax, nullptr);
          P3_LAUNCH_CHECK("group_max_f32_kernel");
        }
        have_gmax = true;
      }
    }
    P3_REQUIRE(have_gmax, P3TOK_ERR_INVALID, "patch_embed(bf16x3): no per-point layer");
    // ---- concat layer: pooled half once per group (fp32 group bias), then the per-point half
    split_rows_kernel<<<grid_1d(gc * L.F, 256), 256, 0, s>>>(gmax, gc, F, F, gsplit);
    P3_LAUNCH_CHECK("split_rows_kernel");
    rc = tc_linear(gsplit, gc, 3 * F, (const __nv_bfloat16*)m->w_mid_g, m->mid_dim, m->b_mid, nullptr, 1, 0, nullptr, gbias, nullptr, nullptr,
                   0, s, &ex);
    if (rc) return rc;
    rc = tc_linear(act[cur], rows, 3 * F, (const __nv_bfloat16*)m->w_mid_f, m->mid_dim, nullptr, gbias, (int)k, 1, act[cur ^ 1], nullptr, nullptr,
                   nullptr, 0, s, &exs);
    if (rc) return rc;
    cur ^= 1;
    float* tok = tokens + g0 * m->out_dim;
    if (fused_max) {
      rc = tc_linear(act[cur], rows, 3 * m->mid_dim, (const __nv_bfloat16*)m->w_out, m->out_dim, m->b_out, nullptr, 1, 0, nullptr, nullptr,
                     parts == 1 ? tok : max32, nullptr, parts == 1 ? m->out_relu : 0, s, &ex);
      if (rc) return rc;
      if (parts > 1) {
        group_max_f32_kernel<<<grid_1d(gc * m->out_dim, 256), 256, 0, s>>>(max32, gc, parts, m->out_dim, m->out_relu, tok, nullptr);
        P3_LAUNCH_CHECK("group_max_f32_kernel");
      }
    } else {
      rc = tc_linear(act[cur], rows, 3 * m->mid_dim, (const __nv_bfloat16*)m->w_out, m->out_dim, m->b_out, nullptr, 1, 0, nullptr, scratch,
                     nullptr, nullptr, 0, s, &ex);
      if (rc) return rc;
      group_max_f32_kernel<<<grid_1d(gc * m->out_dim, 256), 256, 0, s>>>(scratch, gc, (int)k, m->out_dim, m->out_relu, tok, nullptr);
      P3_LAUNCH_CHECK("group_max_f32_kernel");
    }
  }
  return P3TOK_OK;
}

// fp32 [R, C] -> bf16 [R, 3 cpad] = [hi | hi | lo], zero padded: the weight operand of the bf16x3 product
__global__ void split_w3_kernel(const float* __restrict__ in, int64_t R_, int C, int cpad, __nv_bfloat16* __restrict__ out) {
  const int64_t total = R_ * cpad;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(e % cpad);
    const int64_t r = e / cpad;
    const float v = c < C ? in[r * C + c] : 0.f;
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    __nv_bfloat16* o = out + r * 3 * cpad + c;
    o[0] = hi;
    o[cpad] = hi;
    o[2 * cpad] = __float2bfloat16_rn(v - __bfloat162float(hi));
  }
}

// C = act(A W^T + bias + gbias) for fp32 operands through the bf16x3 tensor-core product (the training path's GEMMs when
// P3TOK_TRAIN_TC=1): both operands are split on the fly into the caller's workspace.
int linear_x3_f32(const float* A, int64_t M, int K, const float* W, int N, const float* bias, const float* gbias, int rows_per_group,
                  int relu, float* C, void* ws, int64_t ws_bytes, cudaStream_t s) {
  const int64_t kp = pad64(K);
  const int64_t a_bytes = align_up(M * 2 * kp * 2, 1024), w_bytes = align_up((int64_t)N * 3 * kp * 2, 1024);
  P3_REQUIRE(ws_bytes >= a_bytes + w_bytes + 1024, P3TOK_ERR_WORKSPACE, "linear_x3_f32: workspace %lld < %lld bytes", (long long)ws_bytes,
             (long long)(a_bytes + w_bytes + 1024));
  char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 1023) / 1024 * 1024);
  __nv_bfloat16* sa = reinterpret_cast<__nv_bfloat16*>(base);
  __nv_bfloat16* sw = reinterpret_cast<__nv_bfloat16*>(base + a_bytes);
  split_rows_kernel<<<grid_1d(M * kp, 256), 256, 0, s>>>(A, M, K, (int)kp, sa);
  P3_LAUNCH_CHECK("split_rows_kernel");
  split_w3_kernel<<<grid_1d((int64_t)N * kp, 256), 256, 0, s>>>(W, N, K, (int)kp, sw);
  P3_LAUNCH_CHECK("split_w3_kernel");
  TcExtra ex;
  ex.x3 = 1;
  return tc_linear(sa, M, (int)(3 * kp), sw, N, bias, gbias, rows_per_group, relu, nullptr, C, nullptr, nullptr, 0, s, &ex);
}

}  // namespace p3tok

using namespace p3tok;

extern "C" int64_t p3tok_linear_x3_workspace_bytes(int64_t M, int64_t K, int64_t N) {
  if (M < 0 || K <= 0 || N <= 0) return -1;
  const int64_t kp = (K + 63) / 64 * 64;
  return align_up(M * 2 * kp * 2, 1024) + align_up(N * 3 * kp * 2, 1024) + 1024;
}

extern "C" int p3tok_linear_x3_f32(const float* A, int64_t M, int64_t K, const float* W, int64_t N, const float* bias, const float* gbias,
                                   int64_t rows_per_group, int relu, float* C, void* workspace, int64_t workspace_bytes, void* stream) {
  P3_REQUIRE(M >= 0 && K > 0 && N > 0 && K < (1 << 22) && N < (1 << 24), P3TOK_ERR_INVALID, "linear_x3_f32: bad shape");
  if (M == 0) return P3TOK_OK;
  P3_REQUIRE(A && W && C && workspace, P3TOK_ERR_INVALID, "linear_x3_f32: null pointer");
  P3_REQUIRE(relu == 0 || relu == 1, P3TOK_ERR_UNSUPPORTED, "linear_x3_f32: activation %d", relu);
  return linear_x3_f32(A, M, (int)K, W, (int)N, bias, gbias, (int)rows_per_group, relu, C, workspace, workspace_bytes, as_stream(stream));
}

extern "C" int p3tok_linear_bf16(const void* A, int64_t M, int64_t K, const void* W, int64_t N, const float* bias,
                                 const float* gbias, int64_t rows_per_group, int relu, void* out_bf16, float* out_f32,
                                 float* out_max32, void* stream) {
  P3_REQUIRE(M >= 0 && K > 0 && N > 0 && K < (1 << 24) && N < (1 << 24), P3TOK_ERR_INVALID, "linear_bf16: bad shape");
  if (M == 0) return P3TOK_OK;
  P3_REQUIRE(A && W && (out_bf16 || out_f32 || out_max32), P3TOK_ERR_INVALID, "linear_bf16: null pointer");
  P3_REQUIRE((reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(W) & 15) == 0, P3TOK_ERR_UNSUPPORTED,
             "linear_bf16: operands must be 16-byte aligned");
  return tc_linear((const __nv_bfloat16*)A, M, (int)K, (const __nv_bfloat16*)W, (int)N, bias, gbias, (int)rows_per_group, relu,
                   (__nv_bfloat16*)out_bf16, out_f32, out_max32, nullptr, 0, as_stream(stream));
}
