// knn.cu - k nearest neighbours of each patch centre: register-tiled distance sweep with a
// warp-level top-k.
//
// Replaces _square_distance + knn_point (reference src/data/sampler.py:47-75; mode APF_SQ) and
// the cdist + topk inside group_knn (src/models/pix4point.py:79-89; mode P4P_CDIST).  The
// (B,G,N) distance matrix the reference materialises is never formed.
//
// One warp owns CPW centres.  The CTA streams the cloud through shared memory in tiles of
// float4 {x, y, z, |p|^2}; each lane takes one point per step and evaluates it against the
// warp's CPW centres (the point is loaded once, the centres live in registers).  Distances
// follow the reference's exact fp32 operation order (see oracle/p3tok_oracle.c header):
//   APF : d = ((-2*dot)+|c|^2)+|p|^2 with dot = fma(cz,pz, fma(cy,py, cx*px))
//   P4P : t = fma(1,|p|^2, fma(|c|^2,1, fma(-2cz,pz, fma(-2cy,py, (-2cx)*px)))), d = sqrt(max(t,0))
// Selection: each centre keeps its current k best as 32*KPL sorted 64-bit keys
// (ordered-distance << 32 | index) spread over the warp's lanes.  A point is a candidate only
// if its distance is strictly below the current k-th distance (points arrive in ascending index
// order, so an equal distance with a larger index can never win); candidates are appended to a
// small shared-memory queue by ballot/popc and merged 32 at a time with a warp bitonic sort +
// bitonic merges.  The result is ascending by (distance, index): the canonical instance of
// torch.topk's implementation-defined tie order.
// Measured and rejected: direct per-candidate insertion (0.196 vs 0.12 ms at C2); two points per lane with packed
// f32x2 distance arithmetic (FFMA2/FADD2: c3 6.1 -> 7.7 ms, c5 0.59 -> 0.97 ms - twice the votes per active step and a
// vote is true twice as often; the queue merges, not the distance arithmetic, are what the kernel spends its time on).
#include <stdlib.h>

#include "common.cuh"

namespace p3tok {

constexpr int KNN_WARPS = 8;
constexpr int KNN_CPW = 4;                 // centres per warp (register tile)
constexpr int KNN_TILE = 2048;             // points per shared-memory tile (32 KB)
constexpr uint64_t KNN_SENTINEL = 0xffffffffffffffffull;

__device__ __forceinline__ uint64_t shfl_xor_u64(uint64_t v, int m) {
  uint32_t lo = (uint32_t)v, hi = (uint32_t)(v >> 32);
  lo = __shfl_xor_sync(0xffffffffu, lo, m);
  hi = __shfl_xor_sync(0xffffffffu, hi, m);
  return ((uint64_t)hi << 32) | lo;
}
__device__ __forceinline__ uint64_t shfl_u64(uint64_t v, int src) {
  uint32_t lo = (uint32_t)v, hi = (uint32_t)(v >> 32);
  lo = __shfl_sync(0xffffffffu, lo, src);
  hi = __shfl_sync(0xffffffffu, hi, src);
  return ((uint64_t)hi << 32) | lo;
}
__device__ __forceinline__ uint64_t umin64(uint64_t a, uint64_t b) { return a < b ? a : b; }
__device__ __forceinline__ uint64_t umax64(uint64_t a, uint64_t b) { return a < b ? b : a; }

// ascending bitonic sort of one key per lane
__device__ __forceinline__ uint64_t warp_sort_asc(uint64_t v, int lane) {
#pragma unroll
  for (int k = 2; k <= 32; k <<= 1) {
#pragma unroll
    for (int j = k >> 1; j > 0; j >>= 1) {
      const uint64_t o = shfl_xor_u64(v, j);
      const bool up = ((lane & k) == 0);          // this k-block sorts ascending
      const bool lower = ((lane & j) == 0);
      v = (up == lower) ? umin64(v, o) : umax64(v, o);
    }
  }
  return v;
}
// input: bitonic sequence over lanes; output ascending
__device__ __forceinline__ uint64_t warp_bitonic_merge_asc(uint64_t v, int lane) {
#pragma unroll
  for (int j = 16; j > 0; j >>= 1) {
    const uint64_t o = shfl_xor_u64(v, j);
    v = ((lane & j) == 0) ? umin64(v, o) : umax64(v, o);
  }
  return v;
}

// Merge an ascending run `q` (one key per lane) into the ascending list L[0..KPL) (element
// j*32+lane), keeping the 32*KPL smallest.
template <int KPL>
__device__ __forceinline__ void list_insert_run(uint64_t (&L)[KPL], uint64_t q, int lane) {
#pragma unroll
  for (int j = 0; j < KPL; ++j) {
    const uint64_t r = shfl_u64(q, 31 - lane);     // reversed run -> L[j] ++ r is bitonic per lane pair
    const uint64_t lo = umin64(L[j], r);
    if (j + 1 < KPL) {
      const uint64_t hi = umax64(L[j], r);
      q = warp_bitonic_merge_asc(hi, lane);        // carry: the 32 largest, ascending
    }
    L[j] = warp_bitonic_merge_asc(lo, lane);
  }
}

template <int KPL, int MODE>
__global__ void __launch_bounds__(KNN_WARPS * 32)
knn_kernel(const float* __restrict__ x, int N, int pt_stride, const float* __restrict__ centres, int G,
           int k, void* __restrict__ idx_out, int idx_is_i64, float* __restrict__ dist_out) {
  __shared__ float4 tile[KNN_TILE];
  __shared__ uint64_t queue[KNN_WARPS * KNN_CPW][64];

  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int b = blockIdx.y;
  const int g0 = (blockIdx.x * KNN_WARPS + warp) * KNN_CPW;   // first centre of this warp
  const float* P = x + (size_t)b * N * pt_stride;

  // centre registers (warp-uniform)
  float c0[KNN_CPW], c1[KNN_CPW], c2[KNN_CPW], cn[KNN_CPW];
#pragma unroll
  for (int c = 0; c < KNN_CPW; ++c) {
    const int g = min(g0 + c, G - 1);
    const float* cp = centres + ((size_t)b * G + g) * 3;
    const float cx = cp[0], cy = cp[1], cz = cp[2];
    cn[c] = sq3(cx, cy, cz);
    if (MODE == P3TOK_KNN_APF_SQ) {
      c0[c] = cx; c1[c] = cy; c2[c] = cz;
    } else {
      c0[c] = __fmul_rn(-2.f, cx); c1[c] = __fmul_rn(-2.f, cy); c2[c] = __fmul_rn(-2.f, cz);
    }
  }

  uint64_t L[KNN_CPW][KPL];
  float thr[KNN_CPW];     // candidates need d < thr  (or, P4P: t <= thr as a cheap pre-filter)
  float thr_d[KNN_CPW];   // exact current k-th distance (P4P), +inf while the list is not full
  int qn[KNN_CPW];
#pragma unroll
  for (int c = 0; c < KNN_CPW; ++c) {
#pragma unroll
    for (int j = 0; j < KPL; ++j) L[c][j] = KNN_SENTINEL;
    thr[c] = __int_as_float(0x7f800000);
    thr_d[c] = __int_as_float(0x7f800000);
    qn[c] = 0;
  }
  const int kth_lane = (k - 1) & 31, kth_j = (k - 1) >> 5;

  auto merge_queue = [&](int c, uint64_t (&Lc)[KPL], int cnt) {
    uint64_t* q = queue[warp * KNN_CPW + c];
    uint64_t v = (lane < cnt) ? q[lane] : KNN_SENTINEL;
    v = warp_sort_asc(v, lane);
    list_insert_run<KPL>(Lc, v, lane);
    // new threshold = k-th smallest so far
    uint64_t kth = 0;
#pragma unroll
    for (int j = 0; j < KPL; ++j)
      if (j == kth_j) kth = shfl_u64(Lc[j], kth_lane);
    const uint32_t ko = (uint32_t)(kth >> 32);
    const float kd = (ko == 0xffffffffu) ? __int_as_float(0x7f800000) : ord2f(ko);
    return kd;
  };

  for (int base = 0; base < N; base += KNN_TILE) {
    __syncthreads();
    const int cnt = min(KNN_TILE, N - base);
    for (int i = t; i < cnt; i += KNN_WARPS * 32) {
      const float* pp = P + (size_t)(base + i) * pt_stride;
      const float px = pp[0], py = pp[1], pz = pp[2];
      tile[i] = make_float4(px, py, pz, sq3(px, py, pz));
    }
    __syncthreads();
    if (g0 >= G) continue;   // warp without centres still helps loading tiles
    for (int i0 = 0; i0 < cnt; i0 += 32) {
      const int i = i0 + lane;
      const bool valid = i < cnt;
      const float4 p = tile[valid ? i : 0];
      // all CPW distance chains first (independent: instruction-level parallelism), ONE vote for the common case
      // "no candidate for any of the warp's centres", then the per-centre handling
      float dc[KNN_CPW];
      bool pc[KNN_CPW];
      bool any = false;
#pragma unroll
      for (int c = 0; c < KNN_CPW; ++c) {
        if (MODE == P3TOK_KNN_APF_SQ) {
          const float dot = __fmaf_rn(c2[c], p.z, __fmaf_rn(c1[c], p.y, __fmul_rn(c0[c], p.x)));
          float tt = __fmul_rn(-2.f, dot);
          tt = __fadd_rn(tt, cn[c]);
          dc[c] = __fadd_rn(__fadd_rn(tt, p.w), 0.f);
          pc[c] = valid && (dc[c] < thr[c]);
        } else {
          float tt = __fmul_rn(c0[c], p.x);
          tt = __fmaf_rn(c1[c], p.y, tt);
          tt = __fmaf_rn(c2[c], p.z, tt);
          tt = __fadd_rn(tt, cn[c]);      // fma(|c|^2, 1, t)
          tt = __fadd_rn(tt, p.w);        // fma(1, |p|^2, t)
          dc[c] = tt;
          pc[c] = valid && (tt <= thr[c]); // conservative: exact sqrt test below
        }
        any = any || pc[c];
      }
      if (!__any_sync(0xffffffffu, any)) continue;
#pragma unroll
      for (int c = 0; c < KNN_CPW; ++c) {
        float d = dc[c];
        bool pass = pc[c];
        uint32_t ball = __ballot_sync(0xffffffffu, pass);
        if (ball == 0) continue;
        if (MODE == P3TOK_KNN_P4P_CDIST) {
          d = __fadd_rn(__fsqrt_rn(fmaxf(d, 0.f)), 0.f);
          pass = pass && (d < thr_d[c]);
          ball = __ballot_sync(0xffffffffu, pass);
          if (ball == 0) continue;
        }
        uint64_t* q = queue[warp * KNN_CPW + c];
        if (pass) {
          const int pos = qn[c] + __popc(ball & ((1u << lane) - 1u));
          q[pos] = ((uint64_t)f2ord(d) << 32) | (uint32_t)(base + i);
        }
        qn[c] += __popc(ball);
        __syncwarp();
        if (qn[c] >= 32) {
          const float kd = merge_queue(c, L[c], 32);
          __syncwarp();
          if (lane + 32 < qn[c]) q[lane] = q[lane + 32];
          qn[c] -= 32;
          __syncwarp();
          if (MODE == P3TOK_KNN_APF_SQ) {
            thr[c] = kd;
          } else {
            thr_d[c] = kd;
            // t > kd*kd*(1+2^-22) (rounded up) implies sqrt_rn(t) >= kd: safe to drop early
            thr[c] = (kd == __int_as_float(0x7f800000)) ? kd
                     : __fmul_ru(__fmul_ru(kd, kd), 1.0000002384185791f);
          }
        }
      }
    }
  }
  if (g0 >= G) return;
#pragma unroll
  for (int c = 0; c < KNN_CPW; ++c) {
    if (qn[c] > 0) (void)merge_queue(c, L[c], qn[c]);
    const int g = g0 + c;
    if (g >= G) continue;
    const size_t o = ((size_t)b * G + g) * k;
#pragma unroll
    for (int j = 0; j < KPL; ++j) {
      const int r = j * 32 + lane;
      if (r < k) {
        const uint32_t id = (uint32_t)L[c][j];
        if (idx_is_i64) reinterpret_cast<int64_t*>(idx_out)[o + r] = (int64_t)id;
        else reinterpret_cast<int32_t*>(idx_out)[o + r] = (int32_t)id;
        if (dist_out) dist_out[o + r] = ord2f((uint32_t)(L[c][j] >> 32));
      }
    }
  }
}

template <int KPL>
static int knn_launch(const float* x, int B, int N, int pt_stride, const float* centres, int G, int k,
                      int mode, void* idx_out, int i64, float* dist_out, cudaStream_t s) {
  dim3 grid((unsigned)((G + KNN_WARPS * KNN_CPW - 1) / (KNN_WARPS * KNN_CPW)), (unsigned)B);
  if (mode == P3TOK_KNN_APF_SQ)
    knn_kernel<KPL, P3TOK_KNN_APF_SQ><<<grid, KNN_WARPS * 32, 0, s>>>(x, N, pt_stride, centres, G, k, idx_out, i64, dist_out);
  else
    knn_kernel<KPL, P3TOK_KNN_P4P_CDIST><<<grid, KNN_WARPS * 32, 0, s>>>(x, N, pt_stride, centres, G, k, idx_out, i64, dist_out);
  P3_LAUNCH_CHECK("knn_kernel");
  return P3TOK_OK;
}


// ================================================================================================
// Spatially sorted variant (clouds of up to 8192 points): the sweep above evaluates every (centre, point) pair and its
// running threshold only tightens as fast as random-order points allow (~k(1+ln(N/k)) candidates, ~10 merges per centre
// at N = 8192).  Here a preparation kernel sorts each cloud along a Z-order curve once, so that 32 consecutive points
// are a compact block with a bounding box; a warp then owns ONE centre: it seeds its list from the blocks around the
// centre's own position on the curve (tight threshold after ~96 points), tests all block boxes against the threshold
// 32 at a time (one lane per block), and evaluates only the blocks that can still contribute.  Distances, keys and the
// result are exactly those of the sweep: a block is skipped only if a lower bound of the COMPUTED distance (geometric
// bound minus a margin far above the rounding error of the expansion formula) exceeds the current k-th distance, and
// because points no longer arrive in index order the filter is non-strict (<=): ties at the k-th distance reach the
// merge, which orders by (distance, index).
// Clouds beyond 8192 points (one CTA's shared-memory sort) are handled as S = ceil(N / 8192) SEGMENTS of consecutive points,
// each sorted on its own (its own Z-order frame, block boxes and cell table); a query walks the segments one after the
// other, seeding from each.  A segment is a random 1/S sample of the cloud, so its blocks are ~S^(1/3) times wider than a
// global sort's - at N = 65536 a centre still evaluates only ~2-3 % of the cloud instead of all of it (sweep kernel).
#ifndef KNS_MIN_BLOCKS
#define KNS_MIN_BLOCKS 5                       // k <= 32: 48 registers, 40 resident warps per SM (64 registers / 32 warps before)
#endif
constexpr int KNS_MAX_N = 8192;                // points per segment
constexpr int KNS_MAX_SEG = 16;                // N <= 131072
constexpr int KNS_CELLS = 512;                 // coarse Z-order cells (top 9 bits of the 30-bit code) for the start position

struct KnsLayout {
  int64_t S, seg, nblk_seg;                     // segments per cloud, points per segment (the last may be shorter), blocks per segment
  int64_t off_pts, off_ids, off_bb, off_lut, off_meta, total;
};
static KnsLayout kns_layout(int64_t B, int64_t N) {
  KnsLayout L;
  L.S = (N + KNS_MAX_N - 1) / KNS_MAX_N;
  L.seg = (N + L.S - 1) / L.S;
  L.nblk_seg = (L.seg + 31) / 32;
  const int64_t nblk = L.S * L.nblk_seg;
  int64_t o = 0;
  L.off_pts = o; o += B * nblk * 32 * 16;       // float4 {x,y,z,|p|^2}, sorted, padded to whole blocks
  L.off_ids = o; o += B * nblk * 32 * 4;        // int32 original index
  L.off_bb = o; o += B * nblk * 32;             // 8 floats per block: min xyz, max xyz, -, -
  L.off_lut = o; o += B * L.S * (KNS_CELLS + 1) * 4;  // int32 first sorted position of each coarse cell (per segment)
  L.off_meta = o; o += B * L.S * 32;            // 8 floats per segment: min xyz, 1/(max-min) * 1023 xyz, max |p|^2, -
  L.total = o + 256;
  return L;
}

__device__ __forceinline__ uint32_t kns_part1by2(uint32_t n) {
  n &= 0x000003ff;
  n = (n ^ (n << 16)) & 0xff0000ff;
  n = (n ^ (n << 8)) & 0x0300f00f;
  n = (n ^ (n << 4)) & 0x030c30c3;
  n = (n ^ (n << 2)) & 0x09249249;
  return n;
}
__device__ __forceinline__ uint32_t kns_code(float x, float y, float z, const float* meta) {
  const int qx = min(1023, max(0, (int)((x - meta[0]) * meta[3])));
  const int qy = min(1023, max(0, (int)((y - meta[1]) * meta[4])));
  const int qz = min(1023, max(0, (int)((z - meta[2]) * meta[5])));
  return (kns_part1by2((uint32_t)qz) << 2) | (kns_part1by2((uint32_t)qy) << 1) | kns_part1by2((uint32_t)qx);
}

// one CTA per cloud: bounding box, Z-order keys, bitonic sort in shared memory, sorted copies + block boxes + cell table
// (Ntot points per cloud in S segments of `seg` points; this CTA = segment blockIdx.x % S of cloud blockIdx.x / S;
//  b below numbers the (cloud, segment) pairs, N is THIS segment's point count, id0 its first original index)
__global__ void __launch_bounds__(1024)
knn_prep_kernel(const float* __restrict__ x, int Ntot, int S, int seg, int nblk, int pt_stride, int P2, float4* __restrict__ pts,
                int* __restrict__ ids, float* __restrict__ bb, int* __restrict__ lut, float* __restrict__ meta_out) {
  extern __shared__ uint64_t keys[];
  __shared__ float red[7][32];
  __shared__ float meta[8];
  __shared__ int slut[KNS_CELLS + 1];
  const int b = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5, nw = blockDim.x >> 5, T = blockDim.x;
  const int cloud = b / S, id0 = (b - cloud * S) * seg;
  const int N = min(seg, Ntot - id0);
  const float* P = x + ((size_t)cloud * Ntot + id0) * pt_stride;
  float mn[3] = {3.4e38f, 3.4e38f, 3.4e38f}, mx[3] = {-3.4e38f, -3.4e38f, -3.4e38f}, wmax = 0.f;
  for (int i = t; i < N; i += T) {
    const float px = P[(size_t)i * pt_stride], py = P[(size_t)i * pt_stride + 1], pz = P[(size_t)i * pt_stride + 2];
    mn[0] = fminf(mn[0], px); mx[0] = fmaxf(mx[0], px);
    mn[1] = fminf(mn[1], py); mx[1] = fmaxf(mx[1], py);
    mn[2] = fminf(mn[2], pz); mx[2] = fmaxf(mx[2], pz);
    wmax = fmaxf(wmax, sq3(px, py, pz));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      mn[a] = fminf(mn[a], __shfl_xor_sync(0xffffffffu, mn[a], o));
      mx[a] = fmaxf(mx[a], __shfl_xor_sync(0xffffffffu, mx[a], o));
    }
    wmax = fmaxf(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
  }
  if (lane == 0) {
#pragma unroll
    for (int a = 0; a < 3; ++a) { red[a][warp] = mn[a]; red[3 + a][warp] = mx[a]; }
    red[6][warp] = wmax;
  }
  __syncthreads();
  if (warp == 0) {
    float v[7];
#pragma unroll
    for (int a = 0; a < 7; ++a) v[a] = lane < nw ? red[a][lane] : (a < 3 ? 3.4e38f : (a < 6 ? -3.4e38f : 0.f));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
      for (int a = 0; a < 7; ++a) {
        const float u = __shfl_xor_sync(0xffffffffu, v[a], o);
        v[a] = a < 3 ? fminf(v[a], u) : fmaxf(v[a], u);
      }
    }
    if (lane == 0) {
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        meta[a] = v[a];
        const float ext = v[3 + a] - v[a];
        meta[3 + a] = ext > 0.f ? 1023.f / ext : 0.f;
      }
      meta[6] = v[6];
      meta[7] = 0.f;
    }
  }
  for (int c = t; c <= KNS_CELLS; c += T) slut[c] = N;
  __syncthreads();
  if (t < 8) meta_out[(size_t)b * 8 + t] = meta[t];
  for (int i = t; i < P2; i += T) {
    uint64_t key = 0xffffffffffffffffull;
    if (i < N) key = ((uint64_t)kns_code(P[(size_t)i * pt_stride], P[(size_t)i * pt_stride + 1], P[(size_t)i * pt_stride + 2], meta) << 32) | (uint32_t)i;
    keys[i] = key;
  }
  __syncthreads();
  // Thread t owns elements t, t + T, ...: a warp's elements are aligned 32-element blocks, and for strides j <= 16 the
  // partner i ^ j lies in the same block - those stages only need a warp barrier.  A block barrier is needed before a
  // stage that crosses blocks (j >= 32) and after one (its writes land in other warps' blocks): 27 instead of 66 block
  // barriers at 2048 elements.
  int prev_j = 32;
  for (int kk = 2; kk <= P2; kk <<= 1) {
    for (int j = kk >> 1; j > 0; j >>= 1) {
      if (j >= 32 || prev_j >= 32) __syncthreads();
      else __syncwarp();
      for (int i = t; i < P2; i += T) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const uint64_t a = keys[i], c = keys[ixj];
          const bool up = (i & kk) == 0;
          if ((a > c) == up) { keys[i] = c; keys[ixj] = a; }
        }
      }
      prev_j = j;
    }
  }
  __syncthreads();
  // sorted copies, block boxes (a warp = one block of 32 consecutive sorted points), coarse cell table
  for (int j0 = warp * 32; j0 < nblk * 32; j0 += nw * 32) {
    const int j = j0 + lane;
    float4 pt = make_float4(0.f, 0.f, 0.f, __int_as_float(0x7fc00000));   // padding: |p|^2 = NaN never passes a comparison
    int id = -1;
    float lo[3] = {3.4e38f, 3.4e38f, 3.4e38f}, hi[3] = {-3.4e38f, -3.4e38f, -3.4e38f};
    if (j < N) {
      const uint64_t key = keys[j];
      id = (int)(uint32_t)key;
      const float px = P[(size_t)id * pt_stride], py = P[(size_t)id * pt_stride + 1], pz = P[(size_t)id * pt_stride + 2];
      pt = make_float4(px, py, pz, sq3(px, py, pz));
      lo[0] = hi[0] = px; lo[1] = hi[1] = py; lo[2] = hi[2] = pz;
      const int cell = (int)(key >> (32 + 21));
      const int prev = j > 0 ? (int)(keys[j - 1] >> (32 + 21)) : -1;
      if (cell != prev) slut[cell] = j;
    }
    pts[((size_t)b * nblk) * 32 + j] = pt;
    ids[((size_t)b * nblk) * 32 + j] = id < 0 ? id : id + id0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
        hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
      }
    }
    if (lane < 8) {
      const float v = lane < 3 ? lo[lane] : (lane < 6 ? hi[lane - 3] : 0.f);
      bb[(((size_t)b * nblk) + (j0 >> 5)) * 8 + lane] = v;
    }
  }
  __syncthreads();
  if (t == 0) {   // empty cells inherit the start of the next non-empty one
    for (int c = KNS_CELLS - 1; c >= 0; --c) slut[c] = min(slut[c], slut[c + 1]);
  }
  __syncthreads();
  for (int c = t; c <= KNS_CELLS; c += T) lut[(size_t)b * (KNS_CELLS + 1) + c] = slut[c];
}

template <int KPL, int MODE>
__global__ void __launch_bounds__(KNN_WARPS * 32, KPL == 1 ? KNS_MIN_BLOCKS : 4)
knn_sorted_kernel(const float4* __restrict__ pts, const int* __restrict__ ids, const float* __restrict__ bb,
                  const int* __restrict__ lut, const float* __restrict__ meta_all, int S, int nblk, const float* __restrict__ centres,
                  int G, int64_t total, int k, void* __restrict__ idx_out, int idx_is_i64, float* __restrict__ dist_out) {
  __shared__ uint64_t queue[KNN_WARPS][64];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t cw = (int64_t)blockIdx.x * KNN_WARPS + warp;      // this warp's centre
  if (cw >= total) return;
  const int b = (int)(cw / G);
  const float* cp = centres + (size_t)cw * 3;
  const float cx = cp[0], cy = cp[1], cz = cp[2];
  const float cn = sq3(cx, cy, cz);
  float c0, c1, c2;
  if (MODE == P3TOK_KNN_APF_SQ) { c0 = cx; c1 = cy; c2 = cz; }
  else { c0 = __fmul_rn(-2.f, cx); c1 = __fmul_rn(-2.f, cy); c2 = __fmul_rn(-2.f, cz); }

  uint64_t L[KPL];
#pragma unroll
  for (int j = 0; j < KPL; ++j) L[j] = KNN_SENTINEL;
  float thr = __int_as_float(0x7f800000);      // candidates need d <= thr  (P4P: t <= thr as the cheap pre-filter)
  float thr_d = __int_as_float(0x7f800000);    // exact current k-th distance (P4P)
  int qn = 0;
  const int kth_lane = (k - 1) & 31, kth_j = (k - 1) >> 5;
  uint64_t* q = queue[warp];

  auto merge = [&](int cnt) {
    uint64_t v = (lane < cnt) ? q[lane] : KNN_SENTINEL;
    v = warp_sort_asc(v, lane);
    list_insert_run<KPL>(L, v, lane);
    uint64_t kth = 0;
#pragma unroll
    for (int j = 0; j < KPL; ++j)
      if (j == kth_j) kth = shfl_u64(L[j], kth_lane);
    const uint32_t ko = (uint32_t)(kth >> 32);
    const float kd = (ko == 0xffffffffu) ? __int_as_float(0x7f800000) : ord2f(ko);
    if (MODE == P3TOK_KNN_APF_SQ) {
      thr = kd;
    } else {
      thr_d = kd;
      thr = (kd == __int_as_float(0x7f800000)) ? kd : __fmul_ru(__fmul_ru(kd, kd), 1.0000002384185791f);
    }
  };
  // one block of 32 sorted points (p = this lane's point, id < 0 on padding)
  auto process = [&](const float4 p, const int id) {
    float d;
    bool pass;
    if (MODE == P3TOK_KNN_APF_SQ) {
      const float dot = __fmaf_rn(c2, p.z, __fmaf_rn(c1, p.y, __fmul_rn(c0, p.x)));
      float tt = __fmul_rn(-2.f, dot);
      tt = __fadd_rn(tt, cn);
      d = __fadd_rn(__fadd_rn(tt, p.w), 0.f);
      pass = (id >= 0) && (d <= thr);
    } else {
      float tt = __fmul_rn(c0, p.x);
      tt = __fmaf_rn(c1, p.y, tt);
      tt = __fmaf_rn(c2, p.z, tt);
      tt = __fadd_rn(tt, cn);
      tt = __fadd_rn(tt, p.w);
      d = tt;
      pass = (id >= 0) && (tt <= thr);
    }
    uint32_t ball = __ballot_sync(0xffffffffu, pass);
    if (ball == 0) return;
    if (MODE == P3TOK_KNN_P4P_CDIST) {
      d = __fadd_rn(__fsqrt_rn(fmaxf(d, 0.f)), 0.f);
      pass = pass && (d <= thr_d);
      ball = __ballot_sync(0xffffffffu, pass);
      if (ball == 0) return;
    }
    if (pass) q[qn + __popc(ball & ((1u << lane) - 1u))] = ((uint64_t)f2ord(d) << 32) | (uint32_t)id;
    qn += __popc(ball);
    __syncwarp();
    if (qn >= 32) {
      merge(32);
      __syncwarp();
      if (lane + 32 < qn) q[lane] = q[lane + 32];
      qn -= 32;
      __syncwarp();
    }
  };

  for (int sg = 0; sg < S; ++sg) {              // segments of the cloud (one for N <= 8192), each sorted on its own
  const size_t bs = (size_t)b * S + sg;
  const float* meta = meta_all + bs * 8;
  const float4* P4 = pts + bs * nblk * 32;
  const int* ID = ids + bs * nblk * 32;
  const float* BB = bb + bs * nblk * 8;
  // margin of the block test: the expansion formula's rounding error is a few ulp of (|c|^2 + |p|^2 + 2|c||p|) <= 2(|c|^2+|p|^2)
  const float margin = 1e-5f * (cn + meta[6]) + 1e-30f;
  // ---- best-first walk over the segment's blocks: every lane keeps the lower bounds of 8 blocks (256 blocks per round,
  // one round for a segment of 8192 points) as 32-bit keys (lower bound's float bits, low 8 bits replaced by the block's
  // number in the round - rounding the bound DOWN, which is the safe side); one redux.sync.min picks the nearest unvisited
  // block, and the walk stops as soon as that bound exceeds the running k-th distance.  Nearest-first means the threshold
  // is tight after the first 2-3 blocks (the genuinely nearest ~96 points), so far fewer candidates pass the filter and
  // reach the queue merges that bound this kernel than in curve order (round 1: seed from the curve position, then all
  // blocks in index order - ~10 merges per centre at N = 8192, k = 32).
  if (nblk >= 128) {     // (measured: neutral on uniform clouds, +6 % on clustered ones at N = 8192; below
                         //  4096 points the 8-keys-per-lane bookkeeping costs more than it saves)
    for (int r0 = 0; r0 < nblk; r0 += 256) {
      uint32_t key[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int blk = r0 + u * 32 + lane;
        key[u] = 0xffffffffu;
        if (blk < nblk) {
          const float4 lo = *reinterpret_cast<const float4*>(BB + (size_t)blk * 8);       // min x,y,z, max x
          const float4 hi = *reinterpret_cast<const float4*>(BB + (size_t)blk * 8 + 4);   // max y,z
          const float dx = fmaxf(fmaxf(lo.x - cx, cx - lo.w), 0.f);
          const float dy = fmaxf(fmaxf(lo.y - cy, cy - hi.x), 0.f);
          const float dz = fmaxf(fmaxf(lo.z - cz, cz - hi.y), 0.f);
          const float lb = fmaxf((dx * dx + dy * dy + dz * dz) * 0.999999f - margin, 0.f);
          if (lb <= thr) key[u] = (__float_as_uint(lb) & 0xffffff00u) | (uint32_t)(u * 32 + lane);   // (padding blocks: lb = +inf)
        }
      }
      while (true) {
        uint32_t m = key[0];
#pragma unroll
        for (int u = 1; u < 8; ++u) m = min(m, key[u]);
        const uint32_t w = __reduce_min_sync(0xffffffffu, m);
        if (w == 0xffffffffu) break;
        if (__uint_as_float(w & 0xffffff00u) > thr) break;       // every unvisited block of the round is farther still
        const int id = (int)(w & 0xffu);
#pragma unroll
        for (int u = 0; u < 8; ++u)
          if (u == (id >> 5) && lane == (id & 31)) key[u] = 0xffffffffu;
        const int bk = r0 + id;
        process(P4[bk * 32 + lane], ID[bk * 32 + lane]);
      }
    }
    continue;
  }
  // ---- seed: the blocks around the centre's own position on the segment's curve
  const int cell = (int)(kns_code(cx, cy, cz, meta) >> 21);
  const int pos = lut[bs * (KNS_CELLS + 1) + cell];
  int s0 = (pos >> 5) - 1;
  s0 = max(0, min(s0, nblk - 3));
  const int s1 = min(nblk, s0 + 3);
  {
    // all seed blocks' loads are issued before the first one is consumed (one L2 round trip instead of three)
    float4 sp[3];
    int si[3];
#pragma unroll
    for (int u = 0; u < 3; ++u) {
      const int blk = min(s0 + u, nblk - 1);
      sp[u] = P4[blk * 32 + lane];
      si[u] = ID[blk * 32 + lane];
    }
#pragma unroll
    for (int u = 0; u < 3; ++u)
      if (s0 + u < s1) process(sp[u], si[u]);
  }

  // ---- all other blocks: box test 32 blocks at a time, evaluate the survivors
  for (int r0 = 0; r0 < nblk; r0 += 32) {
    const int blk = r0 + lane;
    float lb = __int_as_float(0x7f800000);
    const bool mine = blk < nblk && (blk < s0 || blk >= s1);   // (thr may still be +inf: validity is not encoded in lb)
    if (mine) {
      const float4 lo = *reinterpret_cast<const float4*>(BB + (size_t)blk * 8);       // min x,y,z, max x
      const float4 hi = *reinterpret_cast<const float4*>(BB + (size_t)blk * 8 + 4);   // max y,z
      const float dx = fmaxf(fmaxf(lo.x - cx, cx - lo.w), 0.f);
      const float dy = fmaxf(fmaxf(lo.y - cy, cy - hi.x), 0.f);
      const float dz = fmaxf(fmaxf(lo.z - cz, cz - hi.y), 0.f);
      lb = (dx * dx + dy * dy + dz * dz) * 0.999999f - margin;
    }
    uint32_t todo = __ballot_sync(0xffffffffu, mine && lb <= thr);
    // (loading the next surviving block before evaluating the current one was measured neutral: with 32-40 resident
    // warps per SM the L2 round trips are already hidden; the kernel is bound by the queue merges)
    while (todo) {
      const int bit = __ffs(todo) - 1;
      todo &= todo - 1;
      const float lbb = __shfl_sync(0xffffffffu, lb, bit);
      if (lbb > thr) continue;                     // the threshold tightened since the vote
      const int bk = r0 + bit;
      process(P4[bk * 32 + lane], ID[bk * 32 + lane]);
    }
  }
  }   // segments
  if (qn > 0) merge(qn);
  const int g = (int)(cw - (int64_t)b * G);
  const size_t o = ((size_t)b * G + g) * k;
#pragma unroll
  for (int j = 0; j < KPL; ++j) {
    const int r = j * 32 + lane;
    if (r < k) {
      const uint32_t id = (uint32_t)L[j];
      if (idx_is_i64) reinterpret_cast<int64_t*>(idx_out)[o + r] = (int64_t)id;
      else reinterpret_cast<int32_t*>(idx_out)[o + r] = (int32_t)id;
      if (dist_out) dist_out[o + r] = ord2f((uint32_t)(L[j] >> 32));
    }
  }
}

template <int KPL>
static int knn_sorted_launch(const float4* pts, const int* ids, const float* bb, const int* lut, const float* meta, int S, int nblk,
                             const float* centres, int G, int64_t total, int k, int mode, void* idx_out, int i64, float* dist_out,
                             cudaStream_t s) {
  const unsigned grid = (unsigned)((total + KNN_WARPS - 1) / KNN_WARPS);
  if (mode == P3TOK_KNN_APF_SQ)
    knn_sorted_kernel<KPL, P3TOK_KNN_APF_SQ><<<grid, KNN_WARPS * 32, 0, s>>>(pts, ids, bb, lut, meta, S, nblk, centres, G, total, k, idx_out, i64, dist_out);
  else
    knn_sorted_kernel<KPL, P3TOK_KNN_P4P_CDIST><<<grid, KNN_WARPS * 32, 0, s>>>(pts, ids, bb, lut, meta, S, nblk, centres, G, total, k, idx_out, i64, dist_out);
  P3_LAUNCH_CHECK("knn_sorted_kernel");
  return P3TOK_OK;
}

}  // namespace p3tok

using namespace p3tok;

extern "C" int p3tok_knn(const float* x, int64_t B, int64_t N, int64_t pt_stride, const float* centres,
                         int64_t G, int64_t k, int mode, void* idx_out, int idx_dtype, float* dist_out,
                         void* stream) {
  P3_REQUIRE(B >= 0 && N > 0 && G >= 0 && pt_stride >= 3, P3TOK_ERR_INVALID, "knn: bad shape");
  P3_REQUIRE(mode == P3TOK_KNN_APF_SQ || mode == P3TOK_KNN_P4P_CDIST, P3TOK_ERR_INVALID, "knn: bad mode %d", mode);
  P3_REQUIRE(idx_dtype == P3TOK_I64 || idx_dtype == P3TOK_I32, P3TOK_ERR_INVALID, "knn: idx dtype must be i32/i64");
  // torch.topk raises when k > N (sampler.py:74); mirror it as an error code
  P3_REQUIRE(k >= 1 && k <= N, P3TOK_ERR_INVALID, "knn: k=%lld out of range for N=%lld", (long long)k, (long long)N);
  P3_REQUIRE(k <= 128, P3TOK_ERR_UNSUPPORTED, "knn: k=%lld > 128", (long long)k);
  P3_REQUIRE(N < (1ll << 31) && B < 65536, P3TOK_ERR_UNSUPPORTED, "knn: N or B too large");
  if (B == 0 || G == 0) return P3TOK_OK;
  P3_REQUIRE(x && centres && idx_out, P3TOK_ERR_INVALID, "knn: null pointer");
  cudaStream_t s = as_stream(stream);
  const int i64 = idx_dtype == P3TOK_I64;
  if (k <= 32) return knn_launch<1>(x, (int)B, (int)N, (int)pt_stride, centres, (int)G, (int)k, mode, idx_out, i64, dist_out, s);
  if (k <= 64) return knn_launch<2>(x, (int)B, (int)N, (int)pt_stride, centres, (int)G, (int)k, mode, idx_out, i64, dist_out, s);
  return knn_launch<4>(x, (int)B, (int)N, (int)pt_stride, centres, (int)G, (int)k, mode, idx_out, i64, dist_out, s);
}

extern "C" int64_t p3tok_knn_workspace_bytes(int64_t B, int64_t N) {
  if (B < 0 || N <= 0 || N > (int64_t)KNS_MAX_N * KNS_MAX_SEG) return 0;       // 0: the sorted variant does not apply, use p3tok_knn
  return kns_layout(B, N).total;
}

// workspace pieces of the sorted variant
struct KnsPtrs {
  float4* pts; int* ids; float* bb; int* lut; float* meta;
};
static KnsPtrs kns_ptrs(void* workspace, int64_t B, int64_t N) {
  const KnsLayout L = kns_layout(B, N);
  char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~(uintptr_t)255);
  KnsPtrs p;
  p.pts = reinterpret_cast<float4*>(base + L.off_pts);
  p.ids = reinterpret_cast<int*>(base + L.off_ids);
  p.bb = reinterpret_cast<float*>(base + L.off_bb);
  p.lut = reinterpret_cast<int*>(base + L.off_lut);
  p.meta = reinterpret_cast<float*>(base + L.off_meta);
  return p;
}

// The preparation half (depends on the clouds only, not on the centres) ...
extern "C" int p3tok_knn_prepare(const float* x, int64_t B, int64_t N, int64_t pt_stride, void* workspace, int64_t workspace_bytes,
                                 void* stream) {
  P3_REQUIRE(B >= 0 && N > 0 && pt_stride >= 3, P3TOK_ERR_INVALID, "knn_prepare: bad shape");
  P3_REQUIRE(N <= (int64_t)KNS_MAX_N * KNS_MAX_SEG, P3TOK_ERR_UNSUPPORTED, "knn_prepare: N=%lld > %d (use p3tok_knn)", (long long)N,
             KNS_MAX_N * KNS_MAX_SEG);
  P3_REQUIRE(B < 65536, P3TOK_ERR_UNSUPPORTED, "knn_prepare: B too large");
  if (B == 0) return P3TOK_OK;
  P3_REQUIRE(x && workspace, P3TOK_ERR_INVALID, "knn_prepare: null pointer");
  P3_REQUIRE(workspace_bytes >= kns_layout(B, N).total, P3TOK_ERR_WORKSPACE, "knn_prepare: workspace %lld < %lld bytes",
             (long long)workspace_bytes, (long long)kns_layout(B, N).total);
  const KnsPtrs w = kns_ptrs(workspace, B, N);
  const KnsLayout L = kns_layout(B, N);
  int P2 = 32;
  while (P2 < L.seg) P2 <<= 1;
  const int threads = P2 > 1024 ? 1024 : P2;
  const size_t smem = (size_t)P2 * 8;
  static thread_local bool configured[32] = {false};
  int dev = 0;
  P3_CUDA(cudaGetDevice(&dev));
  if (dev < 32 && !configured[dev]) {
    P3_CUDA(cudaFuncSetAttribute(knn_prep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, KNS_MAX_N * 8));
    configured[dev] = true;
  }
  knn_prep_kernel<<<(unsigned)(B * L.S), threads, smem, as_stream(stream)>>>(x, (int)N, (int)L.S, (int)L.seg, (int)L.nblk_seg, (int)pt_stride,
                                                                              P2, w.pts, w.ids, w.bb, w.lut, w.meta);
  P3_LAUNCH_CHECK("knn_prep_kernel");
  return P3TOK_OK;
}

// ... and the query half on a workspace p3tok_knn_prepare has filled for the same (B, N) clouds.
extern "C" int p3tok_knn_query(const void* workspace, int64_t workspace_bytes, int64_t B, int64_t N, const float* centres, int64_t G,
                               int64_t k, int mode, void* idx_out, int idx_dtype, float* dist_out, void* stream) {
  P3_REQUIRE(B >= 0 && N > 0 && G >= 0, P3TOK_ERR_INVALID, "knn_query: bad shape");
  P3_REQUIRE(mode == P3TOK_KNN_APF_SQ || mode == P3TOK_KNN_P4P_CDIST, P3TOK_ERR_INVALID, "knn_query: bad mode %d", mode);
  P3_REQUIRE(idx_dtype == P3TOK_I64 || idx_dtype == P3TOK_I32, P3TOK_ERR_INVALID, "knn_query: idx dtype must be i32/i64");
  P3_REQUIRE(k >= 1 && k <= N, P3TOK_ERR_INVALID, "knn_query: k=%lld out of range for N=%lld", (long long)k, (long long)N);
  P3_REQUIRE(k <= 128, P3TOK_ERR_UNSUPPORTED, "knn_query: k=%lld > 128", (long long)k);
  P3_REQUIRE(N <= (int64_t)KNS_MAX_N * KNS_MAX_SEG, P3TOK_ERR_UNSUPPORTED, "knn_query: N=%lld > %d (use p3tok_knn)", (long long)N,
             KNS_MAX_N * KNS_MAX_SEG);
  if (B == 0 || G == 0) return P3TOK_OK;
  P3_REQUIRE(centres && idx_out && workspace, P3TOK_ERR_INVALID, "knn_query: null pointer");
  P3_REQUIRE(workspace_bytes >= kns_layout(B, N).total, P3TOK_ERR_WORKSPACE, "knn_query: workspace %lld < %lld bytes",
             (long long)workspace_bytes, (long long)kns_layout(B, N).total);
  const KnsPtrs w = kns_ptrs(const_cast<void*>(workspace), B, N);
  cudaStream_t s = as_stream(stream);
  const int i64 = idx_dtype == P3TOK_I64;
  const int64_t total = B * G;
  const KnsLayout L = kns_layout(B, N);
  const int S = (int)L.S, nb = (int)L.nblk_seg;
  if (k <= 32) return knn_sorted_launch<1>(w.pts, w.ids, w.bb, w.lut, w.meta, S, nb, centres, (int)G, total, (int)k, mode, idx_out, i64, dist_out, s);
  if (k <= 64) return knn_sorted_launch<2>(w.pts, w.ids, w.bb, w.lut, w.meta, S, nb, centres, (int)G, total, (int)k, mode, idx_out, i64, dist_out, s);
  return knn_sorted_launch<4>(w.pts, w.ids, w.bb, w.lut, w.meta, S, nb, centres, (int)G, total, (int)k, mode, idx_out, i64, dist_out, s);
}

extern "C" int p3tok_knn_sorted(const float* x, int64_t B, int64_t N, int64_t pt_stride, const float* centres, int64_t G,
                                int64_t k, int mode, void* idx_out, int idx_dtype, float* dist_out, void* workspace,
                                int64_t workspace_bytes, void* stream) {
  P3_REQUIRE(k >= 1 && k <= N, P3TOK_ERR_INVALID, "knn_sorted: k=%lld out of range for N=%lld", (long long)k, (long long)N);
  if (B == 0 || G == 0) return P3TOK_OK;
  int rc = p3tok_knn_prepare(x, B, N, pt_stride, workspace, workspace_bytes, stream);
  if (rc) return rc;
  return p3tok_knn_query(workspace, workspace_bytes, B, N, centres, G, k, mode, idx_out, idx_dtype, dist_out, stream);
}
