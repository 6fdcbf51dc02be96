// tc_common.cuh - PTX wrappers (mbarrier, TMA, tcgen05, clusters) and tensor-map helpers shared by the
// tensor-core kernels (embed_tc.cu, embed_fused.cu).  sm_100a only.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <stdlib.h>

#include "embed.cuh"

namespace p3tok {

constexpr int TC_BM = 128, TC_BK = 64;

// ------------------------------------------------------------------------------------------------ PTX
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a pipeline bug must surface as a trapped launch (reported through the C ABI), never as
// a hung GPU.  ~2 s at 2 GHz is orders of magnitude beyond any legitimate wait in these kernels.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000ll) {
      printf("p3tok: mbarrier wait timed out (block %d thread %d parity %u)\n", (int)blockIdx.x, (int)threadIdx.x, parity);
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// L2 prefetch of a tensor box (no shared memory, no barrier): turns the later TMA load into an L2 hit
__device__ __forceinline__ void tma_prefetch_2d(const CUtensorMap* map, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];" ::"l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1)
               : "memory");
}
// ---- CTA-pair (cta_group::2) forms: one MMA spans both SMs of the pair (M = 256), each CTA holds its 128
// rows of A, half of the weight tile and its half of the accumulator; barriers live in the leader (rank 0)
constexpr uint32_t PEER_BIT_MASK = 0xFEFFFFFFu;   // clears the CTA-rank bit of a shared::cluster address -> leader's copy
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* map, uint64_t* leader_bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(leader_bar) & PEER_BIT_MASK), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tc_mma_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// the same MMA with an A-operand collector hint: KEEP = 1 loads A from shared memory and keeps it in the collector
// (SASS .A_KEEP), KEEP = 0 re-uses the A operand of the previous MMA instead of re-reading it (.A_REUSE, last use).
// For back-to-back MMAs that differ only in B / D (the two N halves of a wide output).
template <int KEEP>
__device__ __forceinline__ void tc_mma_pair_a(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  if (KEEP)
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16.collector::a::fill [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
  else
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16.collector::a::lastuse [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tc_commit_pair(uint64_t* bar) {   // arrives on `bar` in BOTH CTAs of the pair
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive_cta(uint64_t* bar, uint32_t cta) {   // arrive on `bar` of CTA `cta` of the cluster
  asm volatile(
      "{\n\t"
      ".reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(cta)
      : "memory");
}
__device__ __forceinline__ bool elect_one() {   // one lane of the (converged) warp
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, kind::f16 (bf16 operands, fp32 accumulate)
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// issue only: the registers are valid after tc_ld_wait()
__device__ __forceinline__ void tc_ld32_issue(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tc_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// UMMA shared-memory descriptor: K-major operand, 128-byte swizzle, rows of 128 B, 8-row groups 1024 B apart
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3fffu);   // start address  [0,14)
  d |= (uint64_t)1 << 16;                    // leading byte offset (unused for swizzled K-major) [16,30)
  d |= (uint64_t)(1024 >> 4) << 32;          // stride byte offset [32,46)
  d |= (uint64_t)1 << 46;                    // descriptor version (Blackwell) [46,48)
  d |= (uint64_t)2 << 61;                    // SWIZZLE_128B [61,64)
  return d;
}

// max over the warp's 32 rows (lane = row), lane l returns column l.  One redux.sync.max.f32 per column (SASS
// CREDUX.MAX.F32, result in a uniform register) instead of the 31-shuffle lane-transpose reduction (kept below for
// warp_rows_max_shfl): a third of the instructions and nothing on the shuffle/shared-memory pipe.
// Measured (profiles/microbench/redux_bench.cu, one SM): redux 565 cycles per 32x32 block per warp and ~12 cycles per
// CREDUX per SM sub-partition however many warps; shuffle transpose 363 cycles per block per warp, 61 per block per SM
// with 8 warps.  redux wins where the shuffle/shared-memory pipe is the contended resource (tc_linear epilogues with
// swizzled stores), the shuffle version where one warp per sub-partition must finish several blocks per tile
// (embed_stage.cu output epilogue).
__device__ __forceinline__ float warp_rows_max(float (&v)[32], int lane) {
  float m = 0.f;
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    float r;
    asm volatile("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(v[j]));
    if (lane == j) m = r;
  }
  return m;
}
__device__ __forceinline__ float warp_rows_max_shfl(float (&v)[32], int lane) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    const bool hi = (lane & off) != 0;
#pragma unroll
    for (int j = 0; j < off; ++j) {
      const float send = hi ? v[j] : v[j + off];
      const float keep = hi ? v[j + off] : v[j];
      v[j] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, off));
    }
  }
  return v[0];
}

// ---- 32-row max straight from tensor memory --------------------------------------------------------------------------
// tcgen05.ld.16x256b hands a thread the m16n8 accumulator fragment: registers 4s+{0,1} = (lane t/4, columns 8s + 2(t%4) +
// {0,1}), registers 4s+{2,3} = (lane t/4 + 8, same columns) (mapping read back on a B200: profiles/microbench/
// rowmax_bench.cu).  Two such loads (lanes +0..15 and +16..31 of the warp's quarter) put rows r, r+8, r+16, r+24 of a column
// pair into ONE thread, so 24 thread-local FMNMX leave only 8 row classes to reduce across lanes: a halving butterfly of
// 4 + 2 + 1 = 7 shuffles per 32 columns, against 32 redux.sync (~13 cycles each on the shared CREDUX unit: the 4500-cycle
// tile epilogue of the fused pair, profiles/r02_fused_trace.txt) or 31 shuffles after a 32x32b load.
__device__ __forceinline__ void tc_ld16x256_x4_issue(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.16x256b.x4.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
// column (0..31) whose maximum lane t holds after rows_max_frag()
__device__ __forceinline__ int rows_max_frag_col(int lane) {
  return 8 * (2 * ((lane >> 4) & 1) + ((lane >> 3) & 1)) + 2 * (lane & 3) + ((lane >> 2) & 1);
}
// a = fragment of lanes +0..15, b = of lanes +16..31 (both already waited for); nvalid = rows of the 32 that exist (< 32 only
// in the last, ragged row block: the others are masked out).  Returns in lane t the max of column rows_max_frag_col(t).
__device__ __forceinline__ float rows_max_frag(float (&a)[16], float (&b)[16], int lane, int nvalid) {
  if (nvalid < 32) {                                   // warp-uniform
    const int r = lane >> 2;
#pragma unroll
    for (int s = 0; s < 4; ++s) {
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        if (r >= nvalid) a[4 * s + e] = -3.0e38f;
        if (r + 8 >= nvalid) a[4 * s + 2 + e] = -3.0e38f;
        if (r + 16 >= nvalid) b[4 * s + e] = -3.0e38f;
        if (r + 24 >= nvalid) b[4 * s + 2 + e] = -3.0e38f;
      }
    }
  }
  float m[8];                                          // m[2s+e]: column 8s + 2(t%4) + e over rows {t/4, +8, +16, +24}
#pragma unroll
  for (int s = 0; s < 4; ++s) {
#pragma unroll
    for (int e = 0; e < 2; ++e) m[2 * s + e] = fmaxf(fmaxf(a[4 * s + e], a[4 * s + 2 + e]), fmaxf(b[4 * s + e], b[4 * s + 2 + e]));
  }
  {
    const bool hi = (lane & 16) != 0;                  // keep column sub-blocks {2,3} if hi else {0,1}
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float send = hi ? m[j] : m[j + 4];
      const float keep = hi ? m[j + 4] : m[j];
      m[j] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 16));
    }
  }
  {
    const bool hi = (lane & 8) != 0;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const float send = hi ? m[j] : m[j + 2];
      const float keep = hi ? m[j + 2] : m[j];
      m[j] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 8));
    }
  }
  {
    const bool hi = (lane & 4) != 0;
    const float send = hi ? m[0] : m[1];
    const float keep = hi ? m[1] : m[0];
    m[0] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 4));
  }
  return m[0];
}
// max over `nvalid` (<= 32) rows of a 32-row x 64-column bf16 store box (rows of 128 B, 16-byte chunks XOR-swizzled by row,
// as the epilogues stage it for a TMA store): lane l reads its two columns (2l, 2l+1) of every row - 32 conflict-free
// LDS.32 + 31 HMNMX2, nothing on the CREDUX unit and no second accumulator read.  bf16 rounding is monotonic, so this equals
// the rounded fp32 max.  Returns bf16x2 {column 2l, column 2l+1}.
__device__ __forceinline__ uint32_t box_rows_max_bf16x2(uint32_t sbox, int lane, int nvalid) {
  const uint32_t chunk = (uint32_t)(lane >> 2), within = (uint32_t)(lane & 3) * 4u;
  uint32_t m = 0xff80ff80u;                            // {-inf, -inf}
#pragma unroll 8
  for (int r = 0; r < nvalid; ++r) {
    uint32_t v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(sbox + (uint32_t)r * 128u + ((chunk ^ (uint32_t)(r & 7)) << 4) + within));
    asm("max.bf16x2 %0, %0, %1;" : "+r"(m) : "r"(v));
  }
  return m;
}

// (o0, o1) = (a0 + b0, a1 + b1) as one packed FADD2
__device__ __forceinline__ void add2(float& o0, float& o1, float a0, float a1, float b0, float b1) {
  asm("{ .reg .b64 ra, rb, rd; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%5}; add.rn.f32x2 rd, ra, rb; mov.b64 {%0,%1}, rd; }"
      : "=f"(o0), "=f"(o1)
      : "f"(a0), "f"(a1), "f"(b0), "f"(b1));
}
// (o0, o1) = (fma(a0, b0, c0), fma(a1, b1, c1)) as one packed FFMA2 (each half rounded like fmaf)
__device__ __forceinline__ void fma2(float& o0, float& o1, float a0, float a1, float b0, float b1, float c0, float c1) {
  asm("{ .reg .b64 ra, rb, rc, rd; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%5}; mov.b64 rc, {%6,%7}; fma.rn.f32x2 rd, ra, rb, rc; "
      "mov.b64 {%0,%1}, rd; }"
      : "=f"(o0), "=f"(o1)
      : "f"(a0), "f"(a1), "f"(b0), "f"(b1), "f"(c0), "f"(c1));
}
// bf16x2 {lo = relu(a), hi = relu(b)}: ReLU fused into the conversion (F2FP.RELU.BF16.F32.PACK_AB)
__device__ __forceinline__ uint32_t pack_bf16x2_relu(float a, float b) {
  uint32_t d;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(b), "f"(a));
  return d;
}

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&t);
}

// ------------------------------------------------------------------------------------------------ host: TMA maps
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static inline EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// bf16 row-major [rows, cols] (row pitch = cols*2 bytes), box = 64 cols x box_rows, 128B swizzle, OOB -> 0
static inline int make_map(CUtensorMap* m, const void* base, int64_t rows, int64_t cols, int box_rows, int64_t ld = 0) {
  P3_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0, P3TOK_ERR_UNSUPPORTED, "tensor map: base must be 16-byte aligned");
  EncodeTiledFn fn = encode_fn();
  P3_REQUIRE(fn, P3TOK_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)(ld > 0 ? ld : cols) * 2};   // ld: row pitch in elements when the matrix is a column slice
  cuuint32_t box[2] = {(cuuint32_t)TC_BK, (cuuint32_t)box_rows};
  cuuint32_t es[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  P3_REQUIRE(r == CUDA_SUCCESS, P3TOK_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) rows=%lld cols=%lld box_rows=%d", (int)r,
             (long long)rows, (long long)cols, box_rows);
  return P3TOK_OK;
}

// fp32 row-major [rows, cols] (row pitch = cols*4 bytes), box = 32 cols (128 B) x box_rows, 128B swizzle
static inline int make_map_f32(CUtensorMap* m, const void* base, int64_t rows, int64_t cols, int box_rows) {
  P3_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0 && cols % 4 == 0, P3TOK_ERR_UNSUPPORTED,
             "tensor map (f32): base must be 16-byte aligned and the row pitch a multiple of 16 bytes");
  EncodeTiledFn fn = encode_fn();
  P3_REQUIRE(fn, P3TOK_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)cols * 4};
  cuuint32_t box[2] = {32u, (cuuint32_t)box_rows};
  cuuint32_t es[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, es,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  P3_REQUIRE(r == CUDA_SUCCESS, P3TOK_ERR_CUDA, "cuTensorMapEncodeTiled (f32) failed (%d) rows=%lld cols=%lld", (int)r,
             (long long)rows, (long long)cols);
  return P3TOK_OK;
}

static inline int num_sms() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}


// embed_fused.cu
bool tc_fused_supported(int K0, int N1, int N2, int64_t rows_per_group, bool has_gbias);
// l1 != null: A0 is not read - the kernel forms it from the APF first layer (K0 == 256; see FusedL1)
struct FusedL1 {
  const float4* rel;     // [rows padded to a multiple of 256] neighbour - centre per row (fp32; .w = height channel or 0)
  const float4* ctr;     // [padded rows / 32] centre row of every 32-row block
  const float* w;        // packed first-layer weights, fused_l1_pack()
  int relu;
};
bool tc_fused_l1_supported(int N1, int N2);   // "pre" pair 256 -> N1 -> N2 with the first layer in-kernel
int64_t fused_l1_pack_bytes();
// W [256, 2C] bf16 (columns [rel | ctr]), bias [256] or null -> packed fp32 per-lane layout
int fused_l1_pack(const __nv_bfloat16* W, const float* bias, int C, float* packed, cudaStream_t s);
int tc_fused(const __nv_bfloat16* A0, int64_t M, int K0, const __nv_bfloat16* Wa, int N1, const float* bias_a,
             const float* gbias, int rows_per_group, const __nv_bfloat16* Wb, int N2, const float* bias_b,
             __nv_bfloat16* out_bf16, float* out_max, __nv_bfloat16* out_max_bf16, int max_relu, cudaStream_t s,
             const FusedL1* l1 = nullptr);

// embed_stage.cu
bool tc_stage_supported(int K0, int N1, int N2, int64_t rows_per_group);
int tc_stage(const __nv_bfloat16* A0, int64_t M, int K0, const __nv_bfloat16* Wa, int N1, const float* bias_a,
             const float* gbias, int rows_per_group, const __nv_bfloat16* Wb, int N2, const float* bias_b, float* out_max,
             __nv_bfloat16* out_max_bf16, int max_relu, cudaStream_t s);

// embed_gather.cu
bool tc_gather_linear_supported(const p3tok_rows* R, int N1, int64_t k);
int tc_gather_linear(const p3tok_rows* R, int64_t g_begin, int64_t rows, const __nv_bfloat16* W, int N1, const float* bias, int relu,
                     __nv_bfloat16* out_bf16, __nv_bfloat16* out_max_bf16, cudaStream_t s);

}  // namespace p3tok
