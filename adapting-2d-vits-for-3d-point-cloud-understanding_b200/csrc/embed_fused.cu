// embed_fused.cu - two consecutive layers of the patch-embedding MLP in ONE tcgen05 kernel (CTA pairs).
//
//   out = W_b . relu(W_a . A0 + bias_a [+ group_bias]) + bias_b          (then bf16 store and/or 32-row max)
//
// used twice per patch-embedding block (reference src/models/apf.py:129-143, src/models/pix4point.py:147-156):
//   "pre"  pair  h1 -> 256->512 (ReLU) -> 512->E        emits f (bf16) and the per-patch max g
//   "post" pair  f  -> E->2E (+W_g.g as group bias, ReLU) -> 2E->E   emits the patch tokens (max over the patch)
// The hidden activation (rows x 512 / rows x 768, the widest tensors of the block) never leaves the SM:
// per row tile the first GEMM is evaluated in 128-column chunks into a TMEM chunk accumulator, epilogue warps
// turn each chunk into a bf16 K-major shared-memory operand (bias / group bias, ReLU), and the second GEMM consumes it
// at once, accumulating the tile's full output row block in TMEM (<= 384 columns).  128 columns is the narrowest N
// at which a tcgen05.mma runs at its nominal rate (65 cycles; N = 64 costs 56 instead of 32, profiles/microbench):
// the first version of this kernel used 64-column chunks and N2/4-column B-MMAs and lost to the layer-by-layer path.
//
// Two CTAs of a cluster work as a pair (tcgen05 cta_group::2): one MMA spans both SMs (M = 256 rows), each CTA
// keeps its own 128 rows of A0 / chunk operands / accumulators and only HALF of every weight box.
//
// Per CTA shared memory: A0 (K0/64 x 16 KB) | 1 or 2 chunk operands (32 KB each) | ring RA of 8 KB boxes [64 n x 64 k]
// of W_a | ring RB of boxes [nq_rows/2 n x 64 k] of W_b | 8 x 4 KB store staging ("pre" only) | biases.  A TMA round
// trip is 1000-1500 cycles and a 12 KB W_b box is consumed in ~390, so ring DEPTH decides whether the MMAs starve: when
// two chunk operands would leave fewer than 4 + 3 ring slots (E = 384: 3 + 2), the second operand buffer goes to the
// rings (5 + 4) and the chunk epilogue waits for the previous chunk's B-GEMM before it stores (measured: chunk period
// 5200 -> 4270 cycles against 3112 of MMA work; what is left is shared-memory bandwidth - MMA operand fetch 256 KB +
// ring fills 96 KB + operand stores 32 KB per chunk is ~3000 cycles at 128 B/cycle).
// TMEM (per CTA, its 128 rows): columns [0,N2) output accumulator; chunk accumulators in the last 128 (N2 > 256:
// single-buffered) or 256 columns.
// Warps: 0 = TMA producer (A0 + RA), 1 = MMA issuer (leader CTA only), 2..9 = chunk epilogue (row quarter q,
// 64-column half h of each chunk), 10..17 = tile epilogue (row quarter q, alternating 64-column output groups),
// 18 = TMA producer (RB).  Barriers that the leader's MMA warp waits on live in the leader CTA: TMA loads of
// both CTAs signal them (cta_group::2 loads), epilogue warps of the peer arrive remotely; barriers that
// producers / epilogue warps wait on are local and released by multicast tcgen05.commit.
#include <vector>

#include "tc_common.cuh"

namespace p3tok {

constexpr int FU_CH_WARPS = 8, FU_OUT_WARPS = 8;
constexpr int FU_THREADS = (3 + FU_CH_WARPS + FU_OUT_WARPS) * 32;
constexpr int FU_CHUNK = 128;                // hidden columns per chunk: the narrowest N at which a tcgen05.mma still runs at
                                             // its nominal rate (65 cycles; N = 64 costs 56 instead of 32: profiles/microbench)
constexpr int FU_CH_BYTES = 2 * 16384;       // one chunk operand: 128 rows x 128 columns bf16 = two 64-column K blocks
constexpr int FU_RA_BOX = 64 * 128;          // 8 KB: this CTA's 64 of the chunk's 128 rows of W_a x 64 k
constexpr int FU_MAX_RA = 32, FU_MAX_RB = 16;
constexpr int FU_SMEM = 227 * 1024;
constexpr int FU_L1_WSTRIDE = 76;            // floats per lane: 32 rel + 32 ctr weights + 8 biases, padded so LDS.128 is conflict-free
constexpr int FU_L1_STAGE = 128 * 16 + 4 * 16;   // per tile and CTA: 128 rel rows + 4 block centres (float4 each)
constexpr int FU_L1_BYTES = 2 * FU_L1_STAGE;      // (the packed weights, 9.5 KB, are read through L1 once per tile: the shared
                                                  //  memory they would take is a ring slot)

struct FusedParams {
  int M, K0, N1, N2;
  int num_pairs;                    // ceil(num_m_tiles / 2): one 256-row tile per CTA pair
  int ra_slots, rb_slots, rb_box;   // ring depths; rb_box = (nq_rows/2) * 128 bytes
  int nch;                          // chunk operand buffers in shared memory: 2, or 1 when the weight rings need the room
  int nacc;                         // chunk accumulators in TMEM: 2 when N2 <= 256, else 1 (384 output + 128 chunk columns = 512)
  int nq, nq_rows;                  // output columns per B-MMA: N2 (nq = 1) or N2/2 (nq = 2, N2 > 256)
  const float* bias_a;              // [N1] or null
  const float* gbias;               // [M / rows_per_group, N1] or null; rows_per_group % 32 == 0
  int rows_per_group;
  const float* bias_b;              // [N2] or null
  int store_out;                    // bf16 [M,N2] through tmC
  float* out_max;                   // [M/32, N2] or null
  __nv_bfloat16* out_max_bf16;      // same, bf16, or null
  int max_relu;
  unsigned long long* trace;        // debug (P3TOK_TC_TRACE=1): pair 0's timeline (leader MMA warp + one epilogue warp of each kind)
  // ---- APF first layer produced in-kernel (K0 == 256): A0 = relu(W_rel . (nbr - ctr) + (W_ctr . ctr + bias)) written by the
  // chunk-epilogue warps straight into the swizzled A0 tile; l1_rel == null: A0 comes from tmA as before
  const float4* l1_rel;             // [rows padded to 256] (nbr - ctr) per row, fp32 (apf_rel_rows_kernel)
  const float4* l1_ctr;             // [rows / 32] centre row of every 32-row block
  const float* l1_w;                // [32 lanes][FU_L1_WSTRIDE]: lane l's 8 output channels, pair-packed (fused_l1_pack_kernel)
  int l1_relu;
};
// trace[(it * 16 + j) * 16 + slot]; slots 0-7 MMA warp, 8-11 chunk-epilogue warp 2, 12-15 tile-epilogue warp 10 (leader CTA)
__device__ __forceinline__ void fu_trace(const FusedParams& p, int it, int j, int slot, long long v) {
  if (p.trace && blockIdx.x == 0 && it < 4 && j < 16) p.trace[((size_t)it * 16 + j) * 16 + slot] = (unsigned long long)v;
}

__global__ void __launch_bounds__(FU_THREADS, 1)
tc_fused_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmWa,
                const __grid_constant__ CUtensorMap tmWb, const __grid_constant__ CUtensorMap tmC, const FusedParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int KB0 = p.K0 / 64, NC = p.N1 / FU_CHUNK, NQ = p.nq;
  uint8_t* sA0 = smem;                                   // KB0 x 16 KB
  uint8_t* sCH = sA0 + KB0 * 16384;                      // 2 x 32 KB chunk operands
  uint8_t* sRA = sCH + p.nch * FU_CH_BYTES;              // ra_slots x 8 KB
  uint8_t* sRB = sRA + p.ra_slots * FU_RA_BOX;           // rb_slots x rb_box
  uint8_t* sST = sRB + p.rb_slots * p.rb_box;            // 8 x 4 KB store staging when store_out
  float* sba = reinterpret_cast<float*>(sST + (p.store_out ? FU_OUT_WARPS * 4096 : 0));   // N1 floats
  float* sbb = sba + p.N1;                               // N2 floats
  float* sgb = sbb + p.N2;                               // chunk warps x 64 floats (group-bias slices)
  const bool L1 = p.l1_rel != nullptr;
  uint8_t* sl1 = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(sgb + FU_CH_WARPS * 64) + 15) & ~(uintptr_t)15);   // 2 x FU_L1_STAGE: rel rows + block centres
  uint64_t* bars = reinterpret_cast<uint64_t*>((reinterpret_cast<uintptr_t>(sl1 + (L1 ? 2 * FU_L1_STAGE : 0)) + 7) & ~(uintptr_t)7);
  uint64_t* a0_full = bars;            // leader
  uint64_t* a0_empty = bars + 1;       // local, multicast commit
  uint64_t* acc3_full = bars + 2;      // local, multicast commit
  uint64_t* acc3_empty = bars + 3;     // leader, 2 x FU_OUT_WARPS arrivals
  uint64_t* acc2_full = bars + 4;      // [2] local, multicast commit
  uint64_t* acc2_empty = bars + 6;     // [2] leader, 2 x FU_CH_WARPS
  uint64_t* ch_full = bars + 8;        // [2] leader, 2 x FU_CH_WARPS
  uint64_t* ch_empty = bars + 10;      // [2] local, multicast commit
  uint64_t* ra_full = bars + 12;       // [32] leader
  uint64_t* ra_empty = bars + 44;      // [32] local
  uint64_t* rb_full = bars + 76;       // [16] leader
  uint64_t* rb_empty = bars + 92;      // [16] local
  uint64_t* l1_full = bars + 108;      // [2] local, TMA bulk copy (tx bytes)
  uint64_t* l1_empty = bars + 110;     // [2] local, FU_CH_WARPS arrivals
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 112);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const int rank = (int)cluster_ctarank();
  const int pair_id = blockIdx.x >> 1, pair_stride = gridDim.x >> 1;

  if (threadIdx.x == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmA)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmWa)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tmWb)) : "memory");
    mbar_init(a0_full, L1 ? 2 * FU_CH_WARPS : 1);      // L1: every chunk-epilogue warp of both CTAs publishes its 16 rows
    mbar_init(a0_empty, 1);
    for (int b = 0; b < 2; ++b) { mbar_init(&l1_full[b], 1); mbar_init(&l1_empty[b], FU_CH_WARPS); }
    mbar_init(acc3_full, 1);
    mbar_init(acc3_empty, 2 * FU_OUT_WARPS);
    for (int b = 0; b < 2; ++b) {
      mbar_init(&acc2_full[b], 1);
      mbar_init(&acc2_empty[b], 2 * FU_CH_WARPS);
      mbar_init(&ch_full[b], 2 * FU_CH_WARPS);
      mbar_init(&ch_empty[b], 1);
    }
    for (int s = 0; s < FU_MAX_RA; ++s) { mbar_init(&ra_full[s], 1); mbar_init(&ra_empty[s], 1); }
    for (int s = 0; s < FU_MAX_RB; ++s) { mbar_init(&rb_full[s], 1); mbar_init(&rb_empty[s], 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = threadIdx.x; i < p.N1; i += FU_THREADS) sba[i] = p.bias_a ? p.bias_a[i] : 0.f;
  int bb_nonzero = 0;
  for (int i = threadIdx.x; i < p.N2; i += FU_THREADS) {
    const float b = p.bias_b ? p.bias_b[i] : 0.f;
    sbb[i] = b;
    bb_nonzero |= (b != 0.f);
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::);
  }
  tc_fence_before();
  const bool has_bb = __syncthreads_or(bb_nonzero) != 0;   // an all-zero output bias (folded away on the host) is not added
  cluster_sync_all();                       // the peer's barriers exist before any remote arrive / multicast commit
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int nq_rows = p.nq_rows;            // output columns per B-MMA; each CTA holds nq_rows/2 rows of the W_b box
  const uint32_t acc_col0 = 512u - (uint32_t)p.nacc * FU_CHUNK;   // TMEM column of chunk accumulator 0

  if (warp == 0) {
    // ---------------- producer 0: this CTA's A0 rows, then its half of every W_a box, in consumption order
    const bool issuer = elect_one();
    int rs = 0;
    uint32_t rph = 0;
    int it = 0;
    // L1: the first-layer inputs of tile `t` (128 rel rows + 4 block centres of this CTA, 2112 bytes) as two 1-D bulk copies
    // into staging buffer t & 1; issued one tile ahead of the chunk-epilogue warps that turn them into A0
    auto l1_load = [&](int t, int tp_t) {
      const int sb = t & 1;
      mbar_wait(&l1_empty[sb], ((uint32_t)(t >> 1) & 1) ^ 1);
      if (issuer) {
        const int64_t mt_t = 2 * (int64_t)tp_t + rank;
        uint8_t* dst = sl1 + sb * FU_L1_STAGE;
        mbar_expect_tx(&l1_full[sb], (uint32_t)FU_L1_STAGE);
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                     "l"(reinterpret_cast<uint64_t>(p.l1_rel + mt_t * TC_BM)), "r"(128 * 16), "r"(smem_u32(&l1_full[sb]))
                     : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst + 128 * 16)),
                     "l"(reinterpret_cast<uint64_t>(p.l1_ctr + mt_t * (TC_BM / 32))), "r"(4 * 16), "r"(smem_u32(&l1_full[sb]))
                     : "memory");
      }
      __syncwarp();
    };
    if (L1 && pair_id < p.num_pairs) l1_load(0, pair_id);
    for (int tp = pair_id; tp < p.num_pairs; tp += pair_stride, ++it) {
      const int mt = 2 * tp + rank;         // may be a dummy tile past the end: TMA zero-fills, stores are clipped
      if (L1) {
        if (tp + pair_stride < p.num_pairs) l1_load(it + 1, tp + pair_stride);
      } else {
        mbar_wait(a0_empty, (uint32_t)(it & 1) ^ 1);
        if (issuer) {
          if (rank == 0) mbar_expect_tx(a0_full, 2u * (uint32_t)KB0 * 16384u);
          for (int kb = 0; kb < KB0; ++kb) tma_load_2d_pair(sA0 + kb * 16384, &tmA, a0_full, kb * 64, mt * TC_BM);
        }
      }
      __syncwarp();
      for (int j = 0; j < NC; ++j) {
        for (int kb = 0; kb < KB0; ++kb) {
          mbar_wait(&ra_empty[rs], rph ^ 1);
          if (issuer) {
            if (rank == 0) mbar_expect_tx(&ra_full[rs], 2u * FU_RA_BOX);
            tma_load_2d_pair(sRA + rs * FU_RA_BOX, &tmWa, &ra_full[rs], kb * 64, j * FU_CHUNK + rank * (FU_CHUNK / 2));
          }
          __syncwarp();
          if (++rs == p.ra_slots) { rs = 0; rph ^= 1; }
        }
      }
    }
  } else if (warp == 2 + FU_CH_WARPS + FU_OUT_WARPS) {
    // ---------------- producer 1: this CTA's half of every W_b box
    const bool issuer = elect_one();
    int rs = 0;
    uint32_t rph = 0;
    for (int tp = pair_id; tp < p.num_pairs; tp += pair_stride) {
      for (int j = 0; j < NC; ++j) {
        for (int kq = 0; kq < 2 * NQ; ++kq) {     // (64-column K block of the chunk) x (output column group)
          const int kb2 = kq / NQ, qd = kq - kb2 * NQ;
          mbar_wait(&rb_empty[rs], rph ^ 1);
          if (issuer) {
            if (rank == 0) mbar_expect_tx(&rb_full[rs], 2u * (uint32_t)p.rb_box);
            tma_load_2d_pair(sRB + rs * p.rb_box, &tmWb, &rb_full[rs], j * FU_CHUNK + kb2 * 64, qd * nq_rows + rank * (nq_rows / 2));
          }
          __syncwarp();
          if (++rs == p.rb_slots) { rs = 0; rph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (rank == 0) {
      // ---------------- MMA issuer (leader CTA, for both SMs of the pair)
      const bool issuer = elect_one();
      const uint64_t dconst = umma_desc_sw128(0);
      const uint32_t idesc_a = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(FU_CHUNK >> 3) << 17) | ((uint32_t)((2 * TC_BM) >> 4) << 24);
      const uint32_t idesc_b = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(nq_rows >> 3) << 17) | ((uint32_t)((2 * TC_BM) >> 4) << 24);
      const uint32_t a0_base = smem_u32(sA0) >> 4, ch_base = smem_u32(sCH) >> 4;
      const uint32_t ra_base = smem_u32(sRA) >> 4, rb_base = smem_u32(sRB) >> 4;
      int ras = 0, rbs = 0;
      uint32_t raph = 0, rbph = 0;
      uint32_t gc = 0;          // global chunk counter of the A-GEMM (selects the chunk accumulator and its parity)
      uint32_t gcb = 0;         // global chunk counter of the B-GEMM
      int it = 0;
      // A(j): chunk accumulator (gc & 1) = A0 . W_a[chunk j]^T
      auto issue_A = [&](bool last_of_tile) {
        const uint32_t b = p.nacc == 2 ? (gc & 1) : 0u;                   // chunk accumulator and how often it was used
        const uint32_t use = p.nacc == 2 ? (gc >> 1) : gc;
        mbar_wait(&acc2_empty[b], (use & 1) ^ 1);
        tc_fence_after();
        const uint32_t d = tmem_base + acc_col0 + b * FU_CHUNK;
        for (int kb = 0; kb < KB0; ++kb) {
          mbar_wait(&ra_full[ras], raph);
          tc_fence_after();
          if (issuer) {
            const uint64_t ad = dconst | (uint64_t)(a0_base + kb * (16384 >> 4));
            const uint64_t bd = dconst | (uint64_t)(ra_base + ras * (FU_RA_BOX >> 4));
#pragma unroll
            for (int k = 0; k < 4; ++k) tc_mma_pair(d, ad + 2 * k, bd + 2 * k, idesc_a, (uint32_t)((kb | k) != 0));
            tc_commit_pair(&ra_empty[ras]);
          }
          __syncwarp();
          if (++ras == p.ra_slots) { ras = 0; raph ^= 1; }
        }
        if (issuer) {
          tc_commit_pair(&acc2_full[b]);
          if (last_of_tile) tc_commit_pair(a0_empty);   // every MMA that reads this tile's A0 precedes this commit
        }
        __syncwarp();
        ++gc;
      };
      // Measured and dropped: the A-GEMM running one chunk ahead of the B-GEMM ACROSS tiles (chunk 0 of the next tile issued
      // before the last B-GEMM of this tile) to give the tensor pipe work while the tile epilogue drains the output
      // accumulator (~4600 of 24700 cycles per tile at E = 384).  Measured on the same box: c2 0.977 vs 0.947 ms per step
      // WITHOUT it - the early A(0) delays the last B-GEMM and with it the tile epilogue that the next B(0) waits for.
      // Also measured and dropped (round 2, last session): the issuing thread POLLING the A and B streams' barriers
      // (mbarrier.test_wait) and issuing whichever k-block / K step has its operands, instead of parking inside A(j+1) on
      // the weight box the 5-slot A ring cannot hold yet while B(j) is ready (the "Anext" stamps of
      // profiles/r02_fused_trace_after.txt).  Bit-identical tokens, no stall - and c2 0.91 -> 1.41 ms per step whichever
      // stream has priority: one thread walking a state machine with 4-6 barrier probes (a shared-memory round trip each)
      // per step needs longer per k-block than the 260 cycles its four MMAs take, so the tensor pipe starves on ISSUE.
      // The blocking walk costs ~15 instructions per k-block.
      for (int tp = pair_id; tp < p.num_pairs; tp += pair_stride, ++it) {
        if (issuer) fu_trace(p, it, 0, 4, clock64());        // tile start
        mbar_wait(a0_full, (uint32_t)(it & 1));
        if (issuer) fu_trace(p, it, 0, 5, clock64());        // A0 present
        tc_fence_after();
        issue_A(NC == 1);
        if (issuer) fu_trace(p, it, 0, 6, clock64());        // A(0) issued
        for (int j = 0; j < NC; ++j) {
          if (j + 1 < NC) issue_A(j + 1 == NC - 1);
          // B(j): output accumulator += chunk(j) . W_b[:, chunk j]^T, one MMA group per quarter of the output columns
          const uint32_t b = p.nch == 2 ? (gcb & 1) : 0u;          // chunk operand buffer and how often it was used
          const uint32_t cuse = p.nch == 2 ? (gcb >> 1) : gcb;
          if (issuer) fu_trace(p, it, j, 0, clock64());           // A(j+1) issued
          mbar_wait(&ch_full[b], cuse & 1);
          if (issuer) fu_trace(p, it, j, 1, clock64());           // chunk j operand ready
          if (j == 0) mbar_wait(acc3_empty, (uint32_t)(it & 1) ^ 1);
          tc_fence_after();
          if (NQ == 2) {
            // two output column groups: both MMAs of a K step read the same chunk operand - the second one takes it from
            // the A collector instead of shared memory (this kernel is bound by shared-memory bandwidth)
            for (int kb2 = 0; kb2 < 2; ++kb2) {
              const int s0 = rbs;
              const uint32_t ph0 = rbph;
              if (++rbs == p.rb_slots) { rbs = 0; rbph ^= 1; }
              const int s1 = rbs;
              const uint32_t ph1 = rbph;
              if (++rbs == p.rb_slots) { rbs = 0; rbph ^= 1; }
              mbar_wait(&rb_full[s0], ph0);
              if (issuer && kb2 == 0) fu_trace(p, it, j, 2, clock64());   // first W_b box present
              mbar_wait(&rb_full[s1], ph1);
              if (issuer && kb2 == 1) fu_trace(p, it, j, 3, clock64());   // last W_b box present
              tc_fence_after();
              if (issuer) {
                const uint64_t ad = dconst | (uint64_t)(ch_base + b * (FU_CH_BYTES >> 4) + kb2 * (16384 >> 4));
                const uint64_t bd0 = dconst | (uint64_t)(rb_base + s0 * (p.rb_box >> 4));
                const uint64_t bd1 = dconst | (uint64_t)(rb_base + s1 * (p.rb_box >> 4));
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const uint32_t acc = (uint32_t)((j | kb2 | k) != 0);
                  tc_mma_pair_a<1>(tmem_base, ad + 2 * k, bd0 + 2 * k, idesc_b, acc);
                  tc_mma_pair_a<0>(tmem_base + (uint32_t)nq_rows, ad + 2 * k, bd1 + 2 * k, idesc_b, acc);
                }
                tc_commit_pair(&rb_empty[s0]);
                tc_commit_pair(&rb_empty[s1]);
              }
              __syncwarp();
            }
          } else
          for (int kq = 0; kq < 2 * NQ; ++kq) {
            const int kb2 = kq / NQ, qd = kq - kb2 * NQ;
            mbar_wait(&rb_full[rbs], rbph);
            if (issuer && kq == 0) fu_trace(p, it, j, 2, clock64());            // first W_b box present
            if (issuer && kq == 2 * NQ - 1) fu_trace(p, it, j, 3, clock64());   // last W_b box present
            tc_fence_after();
            if (issuer) {
              const uint64_t ad = dconst | (uint64_t)(ch_base + b * (FU_CH_BYTES >> 4) + kb2 * (16384 >> 4));
              const uint64_t bd = dconst | (uint64_t)(rb_base + rbs * (p.rb_box >> 4));
              const uint32_t d = tmem_base + (uint32_t)(qd * nq_rows);
#pragma unroll
              for (int k = 0; k < 4; ++k) tc_mma_pair(d, ad + 2 * k, bd + 2 * k, idesc_b, (uint32_t)((j | kb2 | k) != 0));
              tc_commit_pair(&rb_empty[rbs]);
            }
            __syncwarp();
            if (++rbs == p.rb_slots) { rbs = 0; rbph ^= 1; }
          }
          if (issuer) {
            fu_trace(p, it, j, 7, clock64());                       // B(j) issued
            tc_commit_pair(&ch_empty[b]);
            if (j == NC - 1) tc_commit_pair(acc3_full);
          }
          __syncwarp();
          ++gcb;
        }
      }
    }
  } else if (warp < 2 + FU_CH_WARPS) {
    // ---------------- chunk epilogue warps: chunk accumulator -> bias (+group bias) -> ReLU -> bf16 K-major operand
    const int ew = warp - 2;
    const int q = warp & 3, h = ew >> 2;            // row quarter, 64-column half (= K block) of every chunk
    const uint32_t lane_field = (uint32_t)(q * 32) << 16;
    const int trow = q * 32 + lane;                 // row inside this CTA's 128-row tile
    float* my_sgb = sgb + ew * 64;
    uint32_t gc = 0;
    int itc = 0;
    const bool tr = (warp == 2 && lane == 0);
    for (int tp = pair_id; tp < p.num_pairs; tp += pair_stride, ++itc) {
      const int row0 = (2 * tp + rank) * TC_BM + q * 32;
      const float* gb_row = (p.gbias && row0 < p.M) ? p.gbias + (size_t)(row0 / p.rows_per_group) * p.N1 : nullptr;
      for (int j = 0; j < NC; ++j, ++gc) {
        const uint32_t ba = p.nacc == 2 ? (gc & 1) : 0u, use = p.nacc == 2 ? (gc >> 1) : gc;   // accumulator / its use count
        const uint32_t bc = p.nch == 2 ? (gc & 1) : 0u, cuse = p.nch == 2 ? (gc >> 1) : gc;      // chunk operand buffer / use count
        const int c0 = j * FU_CHUNK + h * 64;
        float2 gpre = make_float2(0.f, 0.f);
        if (gb_row) gpre = __ldg(reinterpret_cast<const float2*>(gb_row + c0) + lane);   // coalesced 256 B, overlaps the wait below
        if (tr) fu_trace(p, itc, j, 8, clock64());                // waiting for the chunk accumulator
        mbar_wait(&acc2_full[ba], use & 1);
        if (tr) fu_trace(p, itc, j, 9, clock64());                // accumulator ready
        tc_fence_after();
        const uint32_t taddr = tmem_base + lane_field + acc_col0 + ba * FU_CHUNK + h * 64;
        float v[32];
        uint32_t pk[32];
        tc_ld32_issue(taddr, v);
        if (gb_row) {
          *reinterpret_cast<float2*>(my_sgb + 2 * lane) = gpre;
          __syncwarp();
        }
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          tc_ld_wait();
          if (half == 1) {             // last TMEM read of this warp: hand the accumulator back before the conversion
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cta(&acc2_empty[ba], 0);
          }
          const uint32_t sb = smem_u32(sba + c0 + 32 * half), sg = smem_u32(my_sgb + 32 * half);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            if (p.bias_a) {      // (null when the layer's bias travels inside the group bias: the "post" pair)
              float4 b4;
              asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b4.x), "=f"(b4.y), "=f"(b4.z), "=f"(b4.w) : "r"(sb + 16 * i));
              add2(v[4 * i], v[4 * i + 1], v[4 * i], v[4 * i + 1], b4.x, b4.y);
              add2(v[4 * i + 2], v[4 * i + 3], v[4 * i + 2], v[4 * i + 3], b4.z, b4.w);
            }
            if (gb_row) {
              float4 g4;
              asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(g4.x), "=f"(g4.y), "=f"(g4.z), "=f"(g4.w) : "r"(sg + 16 * i));
              add2(v[4 * i], v[4 * i + 1], v[4 * i], v[4 * i + 1], g4.x, g4.y);
              add2(v[4 * i + 2], v[4 * i + 3], v[4 * i + 2], v[4 * i + 3], g4.z, g4.w);
            }
            pk[16 * half + 2 * i] = pack_bf16x2_relu(v[4 * i], v[4 * i + 1]);        // ReLU rides on the conversion
            pk[16 * half + 2 * i + 1] = pack_bf16x2_relu(v[4 * i + 2], v[4 * i + 3]);
          }
          if (half == 0) tc_ld32_issue(taddr + 32, v);
        }
        if (tr) fu_trace(p, itc, j, 10, clock64());               // converted, waiting for the operand buffer
        mbar_wait(&ch_empty[bc], (cuse & 1) ^ 1);          // the B-GEMM that last read this buffer is done
        const uint32_t rbase = smem_u32(sCH) + bc * FU_CH_BYTES + h * 16384 + trow * 128;
#pragma unroll
        for (int pc = 0; pc < 8; ++pc) {
          const uint32_t a = rbase + (((uint32_t)pc ^ (uint32_t)(trow & 7)) << 4);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(pk[4 * pc]), "r"(pk[4 * pc + 1]), "r"(pk[4 * pc + 2]),
                       "r"(pk[4 * pc + 3])
                       : "memory");
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the MMA (async proxy)
        __syncwarp();
        if (lane == 0) mbar_arrive_cta(&ch_full[bc], 0);
        if (tr) fu_trace(p, itc, j, 11, clock64());               // operand published
      }
    }
  } else {
    // ---------------- tile epilogue warps: output accumulator -> bias -> bf16 store and/or 32-row max.
    // The next tile's B-GEMM cannot start before these warps hand the accumulator back, so this epilogue is on the tile's
    // critical path (round 1: 32 redux.sync per 32 columns = ~4500 cycles per tile at E = 384, 18 % of the tile).  Round 2:
    //   "post" pair (only the patch max leaves): accumulator read as m16n8 fragments (tcgen05.ld.16x256b), 24 thread-local
    //          FMNMX + 7 shuffles per 32 columns, bias added AFTER the max (max(x + b) == max(x) + b in fp32: rounding is
    //          monotonic) - rows_max_frag, tc_common.cuh;
    //   "pre" pair (bf16 store of f + bf16 patch max g): the max is read back from the swizzled store box the TMA store
    //          reads anyway (32 LDS.32 + HMNMX2 per 64 columns) - box_rows_max_bf16x2.
    const int ew = warp - 2 - FU_CH_WARPS;
    const int q = warp & 3, h = ew >> 2;
    const uint32_t lane_field = (uint32_t)(q * 32) << 16;
    uint8_t* stg = sST + ew * 4096;
    const int ngroups = p.N2 / 64;
    const int fcol = rows_max_frag_col(lane);
    // L1: tile `t`'s A0 from the staged first-layer inputs, produced by THESE warps: they are idle from the end of their
    // epilogue until the tile's last B-GEMM retires, and a0_empty fires a whole chunk period before that (after the last
    // A-GEMM), so the next tile's first A-GEMM finds its operand waiting - like the TMA-loaded A0 (producing in the chunk-
    // epilogue warps after the last chunk put ~2000 cycles per tile on the critical path: pair kernel 314 -> 370 us at c2).
    // This warp owns rows ew*16 .. +15 of the CTA's 128 (half of one 32-row block, so one centre); lane l owns output
    // channels 8l .. 8l+7 = 16-byte chunk l & 7 of k-block l >> 3.  Same fp32 operation order as
    // rows_first_layer_apf_warp_kernel (base = bias + W_ctr.ctr, then the rel chain), two channels per FFMA2.
    auto produce_a0 = [&](int t) {
      const int sb = t & 1;
      const float4* wl = reinterpret_cast<const float4*>(p.l1_w + lane * FU_L1_WSTRIDE);
      float wr[32], base[8];
      {
        float wc[32];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          *reinterpret_cast<float4*>(&wr[4 * i]) = __ldg(wl + i);
          *reinterpret_cast<float4*>(&wc[4 * i]) = __ldg(wl + 8 + i);
        }
        *reinterpret_cast<float4*>(&base[0]) = __ldg(wl + 16);
        *reinterpret_cast<float4*>(&base[4]) = __ldg(wl + 17);
        mbar_wait(&l1_full[sb], (uint32_t)(t >> 1) & 1);
        const float4 cc = *reinterpret_cast<const float4*>(sl1 + sb * FU_L1_STAGE + 128 * 16 + (ew >> 1) * 16);
        const float cv[4] = {cc.x, cc.y, cc.z, cc.w};
#pragma unroll
        for (int c = 0; c < 4; ++c) {
#pragma unroll
          for (int j = 0; j < 8; j += 2) fma2(base[j], base[j + 1], wc[c * 8 + j], wc[c * 8 + j + 1], cv[c], cv[c], base[j], base[j + 1]);
        }
      }
      const float4* relp = reinterpret_cast<const float4*>(sl1 + sb * FU_L1_STAGE) + ew * 16;
      const uint32_t dst0 = smem_u32(sA0) + (uint32_t)(lane >> 3) * 16384u;
#pragma unroll
      for (int r4 = 0; r4 < 16; r4 += 4) {
        uint32_t pk[4][4];
#pragma unroll
        for (int rr = 0; rr < 4; ++rr) {
          const float4 xv = relp[r4 + rr];                 // warp-wide broadcast
          const float xr[4] = {xv.x, xv.y, xv.z, xv.w};
          float a[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) a[j] = base[j];
#pragma unroll
          for (int c = 0; c < 4; ++c) {
#pragma unroll
            for (int j = 0; j < 8; j += 2) fma2(a[j], a[j + 1], wr[c * 8 + j], wr[c * 8 + j + 1], xr[c], xr[c], a[j], a[j + 1]);
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) pk[rr][j] = p.l1_relu ? pack_bf16x2_relu(a[2 * j], a[2 * j + 1]) : pack_bf16x2(a[2 * j], a[2 * j + 1]);
        }
        if (r4 == 0) mbar_wait(a0_empty, (uint32_t)(t & 1) ^ 1);      // every MMA that read the previous tile's A0 is done
#pragma unroll
        for (int rr = 0; rr < 4; ++rr) {
          const uint32_t trow_ = (uint32_t)(ew * 16 + r4 + rr);
          const uint32_t dst = dst0 + trow_ * 128u + ((((uint32_t)lane & 7u) ^ (trow_ & 7u)) << 4);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(pk[rr][0]), "r"(pk[rr][1]), "r"(pk[rr][2]), "r"(pk[rr][3]) : "memory");
        }
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the MMA (async proxy)
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&l1_empty[sb]);
        mbar_arrive_cta(a0_full, 0);
      }
    };
    if (L1 && pair_id < p.num_pairs) produce_a0(0);
    int it = 0;
    for (int tp = pair_id; tp < p.num_pairs; tp += pair_stride, ++it) {
      if (L1 && tp + pair_stride < p.num_pairs) produce_a0(it + 1);   // gated by a0_empty: this tile's last A-GEMM has retired
      const int row0 = (2 * tp + rank) * TC_BM + q * 32;
      const int row = row0 + lane;
      const bool row_ok = row < p.M;
      const int nvalid = p.M - row0 >= 32 ? 32 : (p.M - row0 > 0 ? p.M - row0 : 0);
      const bool tr = (warp == 2 + FU_CH_WARPS && lane == 0);
      if (tr) fu_trace(p, it, 0, 12, clock64());
      mbar_wait(acc3_full, (uint32_t)(it & 1));
      if (tr) fu_trace(p, it, 0, 13, clock64());
      tc_fence_after();
      bool released = false;
      if (!p.store_out) {
        for (int gi = h; gi < ngroups; gi += 2) {
          const int n0 = gi * 64;
          const bool last = gi + 2 >= ngroups;
          float a0[16], b0[16], a1[16], b1[16];
          const uint32_t t0 = tmem_base + lane_field + (uint32_t)n0;
          tc_ld16x256_x4_issue(t0, a0);
          tc_ld16x256_x4_issue(t0 + (16u << 16), b0);
          tc_ld16x256_x4_issue(t0 + 32u, a1);
          tc_ld16x256_x4_issue(t0 + 32u + (16u << 16), b1);
          tc_ld_wait();
          if (last) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cta(acc3_empty, 0);      // the next tile's B-GEMM may overwrite the accumulator
            if (tr) fu_trace(p, it, 0, 14, clock64());
            released = true;
          }
          float m0 = rows_max_frag(a0, b0, lane, nvalid) + sbb[n0 + fcol];
          float m1 = rows_max_frag(a1, b1, lane, nvalid) + sbb[n0 + 32 + fcol];
          if (p.max_relu) { m0 = fmaxf(m0, 0.f); m1 = fmaxf(m1, 0.f); }
          if (row0 < p.M) {
            const size_t o = (size_t)(row0 >> 5) * p.N2 + n0 + fcol;
            if (p.out_max) { p.out_max[o] = m0; p.out_max[o + 32] = m1; }
            if (p.out_max_bf16) { p.out_max_bf16[o] = __float2bfloat16_rn(m0); p.out_max_bf16[o + 32] = __float2bfloat16_rn(m1); }
          }
        }
      } else {
        for (int gi = h; gi < ngroups; gi += 2) {
          const int n0 = gi * 64;
          const bool last = gi + 2 >= ngroups;
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            float v[32];
            tc_ld32_issue(tmem_base + lane_field + (uint32_t)(n0 + half * 32), v);
            tc_ld_wait();
            if (last && half == 1) {
              tc_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive_cta(acc3_empty, 0);
              if (tr) fu_trace(p, it, 0, 14, clock64());
              released = true;
            }
            if (has_bb) {
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const float4 b4 = *reinterpret_cast<const float4*>(sbb + n0 + half * 32 + 4 * i);
                v[4 * i] += b4.x; v[4 * i + 1] += b4.y; v[4 * i + 2] += b4.z; v[4 * i + 3] += b4.w;
              }
            }
            if (half == 0) {   // the previous box of this warp has left shared memory
              if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
              __syncwarp();
            }
            const uint32_t rbase = smem_u32(stg) + lane * 128;
#pragma unroll
            for (int pc = 0; pc < 4; ++pc) {
              const uint32_t a = rbase + (((uint32_t)(pc + 4 * half) ^ (lane & 7)) << 4);
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(pack_bf16x2(v[pc * 8], v[pc * 8 + 1])),
                           "r"(pack_bf16x2(v[pc * 8 + 2], v[pc * 8 + 3])), "r"(pack_bf16x2(v[pc * 8 + 4], v[pc * 8 + 5])),
                           "r"(pack_bf16x2(v[pc * 8 + 6], v[pc * 8 + 7]))
                           : "memory");
            }
            if (p.out_max) {   // fp32 patch max next to the bf16 store (not used by the tokenizer's orchestration)
              if (!row_ok) {
#pragma unroll
                for (int i = 0; i < 32; ++i) v[i] = -3.0e38f;
              }
              float m = warp_rows_max(v, lane);
              if (p.max_relu) m = fmaxf(m, 0.f);
              if (row0 < p.M) p.out_max[(size_t)(row0 >> 5) * p.N2 + n0 + half * 32 + lane] = m;
            }
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (lane == 0 && row0 < p.M) {
            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                             reinterpret_cast<uint64_t>(&tmC)),
                         "r"(smem_u32(stg)), "r"(n0), "r"(row0)
                         : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
          if (p.out_max_bf16 && row0 < p.M) {   // the patch max of the values just staged (what the next GEMM reads, rounded once)
            uint32_t m = box_rows_max_bf16x2(smem_u32(stg), lane, nvalid);
            if (p.max_relu) asm("max.bf16x2 %0, %0, %1;" : "+r"(m) : "r"(0u));
            *reinterpret_cast<uint32_t*>(p.out_max_bf16 + (size_t)(row0 >> 5) * p.N2 + n0 + 2 * lane) = m;
          }
          __syncwarp();
        }
      }
      if (tr) fu_trace(p, it, 0, 15, clock64());
      if (!released) {   // (N2 == 64: the h = 1 warps have no output group) still hand the accumulator back
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cta(acc3_empty, 0);
      }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // no CTA leaves while the peer may still signal it or read its operands
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

// ------------------------------------------------------------------------------------------------ host
// ring depths for these shapes: what is left of shared memory after the resident operands is split between the two weight
// rings in proportion to the bytes a chunk needs from each (a chunk = K0/64 RA boxes and 2*nq RB boxes)
static bool fused_rings_n(int K0, int N1, int N2, bool store_out, int nch, bool l1, int& ra_slots, int& rb_slots, int& rb_box) {
  const int nq = N2 > 256 ? 2 : 1;
  rb_box = (N2 / nq / 2) * 128;
  const int fixed = (K0 / 64) * 16384 + nch * FU_CH_BYTES + (store_out ? FU_OUT_WARPS * 4096 : 0) +
                    (N1 + N2 + FU_CH_WARPS * 64) * 4 + (l1 ? FU_L1_BYTES + 16 : 0) + 116 * 8 + 64 + 1024;
  const int left = FU_SMEM - fixed;
  if (left < 2 * FU_RA_BOX + 2 * rb_box) return false;
  // split in proportion to the bytes a chunk needs from each ring.  (Measured and dropped: "the smaller ring as large as
  // possible" - the pre pair at E = 384 with 5 + 3 instead of 3 + 4 slots: c2 0.943 -> 0.975 ms, c4 5.31 -> 5.48 ms; the
  // B-GEMM's paired W_b boxes need the depth more than the A-GEMM does.)
  const int chunk_a = (K0 / 64) * FU_RA_BOX, chunk_b = 2 * nq * rb_box;
  ra_slots = (int)((int64_t)left * chunk_a / (chunk_a + chunk_b)) / FU_RA_BOX;
  if (ra_slots < 2) ra_slots = 2;
  if (ra_slots > FU_MAX_RA) ra_slots = FU_MAX_RA;
  rb_slots = (left - ra_slots * FU_RA_BOX) / rb_box;
  if (rb_slots > FU_MAX_RB) rb_slots = FU_MAX_RB;
  return rb_slots >= 2;
}

// Two chunk operand buffers let the chunk epilogue of chunk j+1 store while the B-GEMM of chunk j still reads; but a TMA
// round trip is ~1000-1500 cycles and a 12 KB weight box is consumed in ~390, so rings of 2-3 slots starve the MMAs
// (measured: chunk period 5200 cycles against 3100 of MMA work at E = 384).  When the rings would be that shallow the
// second operand buffer (32 KB) goes to the rings instead.
static bool fused_rings(int K0, int N1, int N2, bool store_out, bool l1, int& nch, int& ra_slots, int& rb_slots, int& rb_box) {
  nch = 2;
  if (fused_rings_n(K0, N1, N2, store_out, 2, l1, ra_slots, rb_slots, rb_box) && ra_slots >= 4 && rb_slots >= 3) return true;
  nch = 1;
  return fused_rings_n(K0, N1, N2, store_out, 1, l1, ra_slots, rb_slots, rb_box);
}

bool tc_fused_supported(int K0, int N1, int N2, int64_t rows_per_group, bool has_gbias) {
  if (K0 % 64 || N1 % FU_CHUNK || N2 % 64) return false;
  if (K0 < 64 || K0 > 384 || N2 < 64 || N2 > 384 || N1 < FU_CHUNK || N1 > 2048) return false;
  if (N2 > 256 && (N2 / 2) % 16) return false;          // two B-MMAs of N2/2 columns each
  if (has_gbias && (rows_per_group % 32 != 0)) return false;
  int nch, ra, rb, box;
  return fused_rings(K0, N1, N2, !has_gbias, false, nch, ra, rb, box);   // the "pre" pair (no group bias) also stores its output
}

// ---- APF first layer inside the pair kernel: per-lane packed fp32 weights.  Lane l owns output channels 8l .. 8l+7:
// floats [8c + j] = W[8l + j][c] (rel half, c < 4, zero beyond C), [32 + 8c + j] = W[8l + j][C + c] (centre half), [64 + j] = bias
__global__ void fused_l1_pack_kernel(const __nv_bfloat16* __restrict__ W, const float* __restrict__ bias, int C, float* __restrict__ out) {
  const int lane = blockIdx.x, i = threadIdx.x;            // 32 blocks x FU_L1_WSTRIDE threads
  float v = 0.f;
  if (i < 64) {
    const int half = i >> 5, c = (i & 31) >> 3, j = i & 7;
    if (c < C) v = __bfloat162float(W[(size_t)(8 * lane + j) * (2 * C) + half * C + c]);
  } else if (i < 72) {
    v = bias ? bias[8 * lane + (i - 64)] : 0.f;
  }
  out[lane * FU_L1_WSTRIDE + i] = v;
}
bool tc_fused_l1_supported(int N1, int N2) {
  if (!tc_fused_supported(256, N1, N2, 32, false)) return false;
  int nch, ra, rb, box;
  return fused_rings(256, N1, N2, true, true, nch, ra, rb, box);
}
int64_t fused_l1_pack_bytes() { return 32 * FU_L1_WSTRIDE * 4; }
int fused_l1_pack(const __nv_bfloat16* W, const float* bias, int C, float* packed, cudaStream_t s) {
  P3_REQUIRE(C == 3 || C == 4, P3TOK_ERR_UNSUPPORTED, "fused_l1_pack: C must be 3 or 4");
  fused_l1_pack_kernel<<<32, FU_L1_WSTRIDE, 0, s>>>(W, bias, C, packed);
  P3_LAUNCH_CHECK("fused_l1_pack_kernel");
  return P3TOK_OK;
}

// out = W_b relu(W_a A0 + bias_a + gbias) + bias_b.  A0 [M,K0] bf16, W_a [N1,K0], W_b [N2,N1] bf16.
int tc_fused(const __nv_bfloat16* A0, int64_t M, int K0, const __nv_bfloat16* Wa, int N1, const float* bias_a,
             const float* gbias, int rows_per_group, const __nv_bfloat16* Wb, int N2, const float* bias_b,
             __nv_bfloat16* out_bf16, float* out_max, __nv_bfloat16* out_max_bf16, int max_relu, cudaStream_t s,
             const FusedL1* l1) {
  P3_REQUIRE(tc_fused_supported(K0, N1, N2, rows_per_group, gbias != nullptr), P3TOK_ERR_UNSUPPORTED,
             "tc_fused: unsupported shape K0=%d N1=%d N2=%d", K0, N1, N2);
  P3_REQUIRE(!l1 || (K0 == 256 && l1->rel && l1->ctr && l1->w), P3TOK_ERR_UNSUPPORTED, "tc_fused: the in-kernel first layer needs K0 == 256");
  P3_REQUIRE(M < (1ll << 31) - 512, P3TOK_ERR_UNSUPPORTED, "tc_fused: too many rows");
  if (M == 0) return P3TOK_OK;
  FusedParams p;
  p.M = (int)M; p.K0 = K0; p.N1 = N1; p.N2 = N2;
  const int num_m_tiles = (int)((M + TC_BM - 1) / TC_BM);
  p.num_pairs = (num_m_tiles + 1) / 2;
  p.bias_a = bias_a; p.gbias = gbias; p.rows_per_group = rows_per_group > 0 ? rows_per_group : 32; p.bias_b = bias_b;
  p.store_out = out_bf16 != nullptr; p.out_max = out_max; p.out_max_bf16 = out_max_bf16; p.max_relu = max_relu;
  p.nacc = N2 <= 256 ? 2 : 1;
  p.nq = N2 > 256 ? 2 : 1;
  p.nq_rows = N2 / p.nq;
  p.rb_box = (p.nq_rows / 2) * 128;
  P3_REQUIRE(fused_rings(K0, N1, N2, p.store_out != 0, l1 != nullptr, p.nch, p.ra_slots, p.rb_slots, p.rb_box), P3TOK_ERR_UNSUPPORTED,
             "tc_fused: shapes do not fit shared memory");
  p.l1_rel = l1 ? l1->rel : nullptr; p.l1_ctr = l1 ? l1->ctr : nullptr; p.l1_w = l1 ? l1->w : nullptr; p.l1_relu = l1 ? l1->relu : 0;
  CUtensorMap ta, twa, twb, tc;
  int rc = make_map(&twa, Wa, N1, K0, FU_CHUNK / 2);  // each CTA of the pair fetches 64 of a chunk's 128 rows
  if (rc) return rc;
  if (l1) {
    ta = twa;                                     // unused: A0 is produced in the kernel
  } else {
    rc = make_map(&ta, A0, M, K0, TC_BM);
    if (rc) return rc;
  }
  rc = make_map(&twb, Wb, N2, N1, p.nq_rows / 2); // ... and half of the output rows of one B-MMA of W_b
  if (rc) return rc;
  if (out_bf16) {
    rc = make_map(&tc, out_bf16, M, N2, 32);
    if (rc) return rc;
  } else {
    tc = twa;
  }
  static thread_local bool configured[32] = {false};
  int dev = 0;
  P3_CUDA(cudaGetDevice(&dev));
  if (dev < 32 && !configured[dev]) {
    P3_CUDA(cudaFuncSetAttribute(tc_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, FU_SMEM));
    configured[dev] = true;
  }
  static int trace_on = -1;
  if (trace_on < 0) trace_on = getenv("P3TOK_TC_TRACE") ? 1 : 0;
  p.trace = nullptr;
  const size_t tw = 4 * 16 * 16;
  if (trace_on) {
    P3_CUDA(cudaMalloc(&p.trace, tw * 8));
    P3_CUDA(cudaMemsetAsync(p.trace, 0, tw * 8, s));
  }
  const int max_pairs = num_sms() / 2;
  const int pairs = p.num_pairs < max_pairs ? p.num_pairs : max_pairs;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(pairs * 2));
  cfg.blockDim = dim3(FU_THREADS);
  cfg.dynamicSmemBytes = FU_SMEM;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  P3_CUDA(cudaLaunchKernelEx(&cfg, tc_fused_kernel, ta, twa, twb, tc, p));
  count_launch();
  if (trace_on) {   // debug only: synchronises and prints pair 0's timeline (cycles relative to its first stamp)
    std::vector<unsigned long long> h(tw);
    P3_CUDA(cudaStreamSynchronize(s));
    P3_CUDA(cudaMemcpy(h.data(), p.trace, tw * 8, cudaMemcpyDeviceToHost));
    P3_CUDA(cudaFree(p.trace));
    fprintf(stderr, "[fu_trace] M=%d K0=%d N1=%d N2=%d ra=%d rb=%d nch=%d nacc=%d\n", p.M, p.K0, p.N1, p.N2, p.ra_slots, p.rb_slots, p.nch, p.nacc);
    const unsigned long long t0 = h[4];
    auto rel = [&](unsigned long long v) { return v ? (long long)(v - t0) : -1ll; };
    for (int it = 1; it < 3; ++it) {
      const unsigned long long* q = &h[(size_t)it * 16 * 16];
      fprintf(stderr, "[fu_trace] tile%d mma: start=%lld a0_ok=%lld A0_issued=%lld | out-epi: wait=%lld acc3_ok=%lld released=%lld end=%lld\n", it,
              rel(q[4]), rel(q[5]), rel(q[6]), rel(q[12]), rel(q[13]), rel(q[14]), rel(q[15]));
      for (int j = 0; j < 16 && q[j * 16 + 7]; ++j)
        fprintf(stderr, "[fu_trace]   chunk%-2d mma: Anext=%lld ch_ok=%lld wb0=%lld wb3=%lld B=%lld | ch-epi: wait=%lld acc2_ok=%lld conv=%lld pub=%lld\n",
                j, rel(q[j * 16 + 0]), rel(q[j * 16 + 1]), rel(q[j * 16 + 2]), rel(q[j * 16 + 3]), rel(q[j * 16 + 7]),
                rel(q[j * 16 + 8]), rel(q[j * 16 + 9]), rel(q[j * 16 + 10]), rel(q[j * 16 + 11]));
    }
  }
  return P3TOK_OK;
}

}  // namespace p3tok
