// fps.cu - farthest point sampling, one CTA (or one thread-block cluster) per cloud.
//
// Replaces furthest_point_sample (reference src/data/sampler.py:4-30) and
// farthest_point_sampling (src/models/pix4point.py:8-53).
//
// Layout: the cloud's raw (N, pt_stride) fp32 rows are staged once into shared memory - with a
// 1-D TMA bulk copy (cp.async.bulk -> UBLKCP) when the slice is 16-byte aligned, plain loads
// otherwise - and each thread then keeps PPT=8 points (x,y,z) and their running min-distance
// in REGISTERS for the whole G-iteration chain.  Shared memory keeps the staged rows only so
// that the winner's coordinates can be broadcast with one LDS per iteration.
// Per iteration: 8 distance updates per thread in the reference's exact fp32 order
// ((dx*dx)+(dy*dy))+(dz*dz) (no FMA contraction), a thread-local strict-> argmax (lowest index
// wins), two redux.sync per warp (max of the distance bits, then min index among the maxima),
// one __syncthreads, a second redux over the per-warp winners.  Clouds larger than 8192 points
// use a cluster of 2..16 CTAs: each CTA owns a contiguous slice and pushes its candidate
// (distance, index, xyz) into every peer's shared memory through DSMEM (st.async + mbarrier).
// A cluster CTA may hold up to 12288 points ("wide slice": 24 points per thread x 512 threads), so the
// cluster size is not forced to a power of two - it is chosen so that ALL clouds of the launch are
// resident at once (cudaOccupancyMaxActiveClusters).  Found with profiles/microbench/
// fps_cluster_trace.cu: a B200 seats only 15 clusters of 8 (or 7) CTAs - a cluster must sit inside one
// GPC - so the 16 clouds of BASELINE configs[3] ran as TWO waves (3.9 ms); as clusters of 6 (10923
// points per CTA; 22 seats) they are one (2.3 ms).
#include <cooperative_groups.h>
#include <cuda/ptx>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace p3tok {

constexpr int FPS_PPT = 8;           // points per thread (registers)
constexpr int FPS_CL_PPT = 16;       // register points per thread of the cluster kernels (512 threads per 8192-point slice)
constexpr int FPS_WIDE_PPT = 24;     // "wide slice" cluster CTAs: 24 points per thread x 512 threads (126 registers)
constexpr int FPS_MAX_THREADS = 1024;
constexpr int FPS_SLICE = FPS_PPT * FPS_MAX_THREADS;  // 8192 points per CTA (single-CTA clouds, regular cluster slices)
constexpr int FPS_SLICE_X = FPS_WIDE_PPT * 512;       // 12288 points per wide-slice cluster CTA
constexpr int fps_max_threads(int ppt) { return ppt == FPS_WIDE_PPT ? 512 : FPS_SLICE / ppt; }

#ifdef P3TOK_FPS_TRACE     // profiles/microbench/fps_cluster_trace.cu: per-phase clock stamps of iteration 100 of cloud 0
__device__ long long fps_trace_buf[16 * 32];
#define FPS_T(slot)                                                                                       \
  do {                                                                                                    \
    if (g == 100 && cloud == 0 && lane == 0 && (warp == 0 || warp == 5))                                  \
      fps_trace_buf[rank * 32 + (warp ? 16 : 0) + (slot)] = clock64();                                    \
    if ((slot) == 0 && (g == 200 || g == 1200) && cloud == 0 && t == 0)                                   \
      fps_trace_buf[rank * 32 + (g == 200 ? 8 : 9)] = clock64();                                          \
  } while (0)
#else
#define FPS_T(slot) do { } while (0)
#endif

struct __align__(16) FpsCand {
  uint32_t key;   // float bits of the candidate's min-distance (>= 0 -> order preserving)
  uint32_t idx;   // global point index
  float x, y, z;
  uint32_t pad[3];
};

__device__ __forceinline__ void warp_argmax(uint32_t& key, uint32_t& idx) {
  const uint32_t m = __reduce_max_sync(0xffffffffu, key);
  const uint32_t cand = (key == m) ? idx : 0xffffffffu;
  idx = __reduce_min_sync(0xffffffffu, cand);
  key = m;
}

// ---- cluster candidate exchange without barrier.cluster: each CTA sends its 32-byte candidate into every peer's shared
// memory as two st.async (STAS.128) - a remote store that also counts its bytes on the peer's mbarrier (complete_tx), so
// data and signal travel as one message - and every CTA arms its own barrier with the CL*32 bytes it expects and waits
// (acquire, cluster scope) until all candidates of the iteration are in.  History: barrier.cluster per iteration 3.4 us at
// 8 x 1024 threads (C4); DSMEM store + separate remote mbarrier.arrive(release) 2.4 us; this form: see DESIGN.md.
__device__ __forceinline__ uint32_t fps_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void fps_push_cand(const FpsCand* local_slot, uint64_t* local_bar, uint32_t dst_cta, const FpsCand& c) {
  uint32_t ra, rb;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(fps_smem_u32(local_slot)), "r"(dst_cta));
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(rb) : "r"(fps_smem_u32(local_bar)), "r"(dst_cta));
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%2, %3, %4, %5}, [%1];" ::"r"(ra), "r"(rb),
               "r"(c.key), "r"(c.idx), "r"(__float_as_uint(c.x)), "r"(__float_as_uint(c.y))
               : "memory");
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%2, %3, %4, %5}, [%1];" ::"r"(ra + 16), "r"(rb),
               "r"(__float_as_uint(c.z)), "r"(0u), "r"(0u), "r"(0u)
               : "memory");
}
__device__ __forceinline__ void fps_expect_cands(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(fps_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void fps_wait_cands(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(ok)
        : "r"(fps_smem_u32(bar)), "r"(parity)
        : "memory");
  }
}

// packed fp32 pairs: one instruction, two independent IEEE operations (round-to-nearest each)
__device__ __forceinline__ void fps_add2(float& o0, float& o1, float a0, float a1, float b0, float b1) {
  asm("{ .reg .b64 ra, rb, rd; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%5}; add.rn.f32x2 rd, ra, rb; mov.b64 {%0,%1}, rd; }"
      : "=f"(o0), "=f"(o1)
      : "f"(a0), "f"(a1), "f"(b0), "f"(b1));
}
__device__ __forceinline__ void fps_mul2(float& o0, float& o1, float a0, float a1, float b0, float b1) {
  asm("{ .reg .b64 ra, rb, rd; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%5}; mul.rn.f32x2 rd, ra, rb; mov.b64 {%0,%1}, rd; }"
      : "=f"(o0), "=f"(o1)
      : "f"(a0), "f"(a1), "f"(b0), "f"(b1));
}

// CL = 1: one CTA per cloud.  CL > 1: a cluster of `ncta` <= CL CTAs per cloud (run-time size).
// PPT: register points per thread.  An iteration is ISSUE-bound (N = 8192: ~900 of 1270 cycles at 8 points per thread x 32
// warps): each warp pays ~55 instructions of reduction / tie resolution / loop on top of 6 per point, so more points per
// thread and fewer warps mean fewer instructions per iteration (measured: 16 beats 8 by 9-12 % from N = 1024 up, 32 is no
// better than 16).
// Measured and dropped: (a) a "two clouds per SM" form for 4096 < N <= 8192 (6 register + 10 shared-memory points per thread,
// 512 threads, 64 registers, two CTAs per SM so that one cloud's reduction chain hides behind the other's distance pass) - 256
// clouds x 8192 points: 2.54 ms against 2.56 ms for two waves of the register form, the SM is issue-bound either way;
// (b) shared-memory "extra" points for the wide slices (+~110 issue cycles per point and iteration; registers hold 24);
// (c) a flag-in-data candidate exchange (tagged 8-byte remote stores polled by warp 0, CTA-scope mbarriers instead of the
// two __syncthreads): 2640 against 2330 cycles per iteration for the st.async form below.
template <int CL, int PPT = FPS_PPT>
__global__ void __launch_bounds__(fps_max_threads(PPT), 1)
fps_kernel(const float* __restrict__ x, int N, int pt_stride, const int64_t* __restrict__ start_idx,
           int G, int64_t* __restrict__ out_idx, int slice, int ncta) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  // [rows: slice*pt_stride floats][mbarrier 8B][warp slots 2*32*8B][cluster cands 2*16*32B]
  float* rows = reinterpret_cast<float*>(smem_raw);
  const int rows_bytes = ((slice * pt_stride * 4 + 127) / 128) * 128;
  uint64_t* mbar = reinterpret_cast<uint64_t*>(smem_raw + rows_bytes);
  uint2* wslot = reinterpret_cast<uint2*>(smem_raw + rows_bytes + 16);
  FpsCand* ccand = reinterpret_cast<FpsCand*>(smem_raw + rows_bytes + 16 + 2 * 32 * sizeof(uint2));
  uint64_t* cbar = reinterpret_cast<uint64_t*>(ccand + 2 * 16);   // [2] candidate-exchange barriers (clusters only)
  FpsCand* cwin = reinterpret_cast<FpsCand*>(cbar + 2);           // [2] winner of the iteration, for the whole CTA

  const int T = blockDim.x;
  const int t = threadIdx.x;
  const int lane = t & 31, warp = t >> 5, nwarps = T >> 5;
  int cloud, rank;
  if constexpr (CL > 1) {
    rank = (int)cg::this_cluster().block_rank();
    cloud = blockIdx.x / ncta;
  } else {
    rank = 0;
    cloud = blockIdx.x;
  }
  const int p0 = rank * slice;                    // first point of this CTA's slice
  const int np = max(0, min(slice, N - p0));      // points in this slice
  const float* src = x + ((size_t)cloud * N + p0) * pt_stride;

  // ---- stage the slice into shared memory
  const size_t bytes = (size_t)np * pt_stride * 4;
  const bool tma_ok = (bytes > 0) && (bytes % 16 == 0) && ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
  if (tma_ok) {
    if (t == 0) {
      cuda::ptx::mbarrier_init(mbar, 1);
      cuda::ptx::fence_proxy_async(cuda::ptx::space_shared);
    }
    __syncthreads();
    if (t == 0) {
      cuda::ptx::mbarrier_arrive_expect_tx(cuda::ptx::sem_release, cuda::ptx::scope_cta,
                                           cuda::ptx::space_shared, mbar, (uint32_t)bytes);
      // bulk copies are limited by the mbarrier tx-count (2^20-1): our slice is <= 128 KiB
      cuda::ptx::cp_async_bulk(cuda::ptx::space_cluster, cuda::ptx::space_global, rows, src,
                               (uint32_t)bytes, mbar);
    }
    while (!cuda::ptx::mbarrier_try_wait_parity(mbar, 0)) {
    }
  } else {
    for (int i = t; i < np * pt_stride; i += T) rows[i] = src[i];
    __syncthreads();
  }

  // ---- registers: PPT points per thread, local index j*T + t (so j ascending == index ascending)
  float px[PPT], py[PPT], pz[PPT], md[PPT];
#pragma unroll
  for (int j = 0; j < PPT; ++j) {
    const int i = j * T + t;
    if (i < np) {
      px[j] = rows[i * pt_stride + 0];
      py[j] = rows[i * pt_stride + 1];
      pz[j] = rows[i * pt_stride + 2];
      md[j] = 1e10f;   // sampler.py:19
    } else {
      px[j] = py[j] = pz[j] = 0.f;
      md[j] = -2.f;    // padding: never the maximum, never updated (fminf keeps -2)
    }
  }
  int far = (int)start_idx[cloud];
  far = min(max(far, 0), N - 1);   // the C ABI cannot validate device data; an out-of-range start index is clamped
  float cx, cy, cz;
  if constexpr (CL > 1) {
    // the owner CTA publishes the start point's coordinates to every peer
    cg::cluster_group cluster = cg::this_cluster();
    if (t == 0) {
      cuda::ptx::mbarrier_init(&cbar[0], 1);   // one local arrive (expect_tx) per phase; the peers contribute bytes
      cuda::ptx::mbarrier_init(&cbar[1], 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (t == 0 && far >= p0 && far < p0 + np) {
      const int l = far - p0;
      FpsCand c;
      c.key = 0; c.idx = (uint32_t)far;
      c.x = rows[l * pt_stride]; c.y = rows[l * pt_stride + 1]; c.z = rows[l * pt_stride + 2];
      c.pad[0] = c.pad[1] = c.pad[2] = 0;
      for (int r = 0; r < ncta; ++r) *cluster.map_shared_rank(&ccand[0], r) = c;
    }
    cluster.sync();
    cx = ccand[0].x; cy = ccand[0].y; cz = ccand[0].z;
    cluster.sync();   // everyone has read slot 0 before iteration 0 may overwrite it
  } else {
    cx = rows[far * pt_stride]; cy = rows[far * pt_stride + 1]; cz = rows[far * pt_stride + 2];
  }

  for (int g = 0; g < G; ++g) {
    if (t == 0 && rank == 0) out_idx[(size_t)cloud * G + g] = far;
    if (g == G - 1) break;
    // Distance updates: the differences and the squares two points per instruction (FADD2 / FMUL2: each half is an IEEE
    // fp32 op; x - c is computed as x + (-c), bit-identical), the two sums as SCALAR add.rn.  Round 1 also packed the sums
    // (add.rn.f32x2): ptxas 12.9 contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2 despite the .rn (and -fmad=false) - a
    // fused square differs from the reference's ((dx*dx)+(dy*dy))+(dz*dz) in the last bit for ~19 % of the pairs
    // (profiles/microbench/f32x2_check.cu), which flips FPS picks on near-ties (found by the C3-shape parity test).  A
    // scalar add.rn is never contracted; build() checks that the kernel's SASS holds no FFMA2.
    FPS_T(0);
    const float ncx = -cx, ncy = -cy, ncz = -cz;
#pragma unroll
    for (int j = 0; j < PPT; j += 2) {
      float dx0, dx1, dy0, dy1, dz0, dz1;
      fps_add2(dx0, dx1, px[j], px[j + 1], ncx, ncx);
      fps_add2(dy0, dy1, py[j], py[j + 1], ncy, ncy);
      fps_add2(dz0, dz1, pz[j], pz[j + 1], ncz, ncz);
      fps_mul2(dx0, dx1, dx0, dx1, dx0, dx1);
      fps_mul2(dy0, dy1, dy0, dy1, dy0, dy1);
      fps_mul2(dz0, dz1, dz0, dz1, dz0, dz1);
      const float d0 = __fadd_rn(__fadd_rn(dx0, dy0), dz0);
      const float d1 = __fadd_rn(__fadd_rn(dx1, dy1), dz1);
      md[j] = fminf(md[j], d0);
      md[j + 1] = fminf(md[j + 1], d1);
    }
    // thread-local maximum first; the index of the maximum is only resolved by the threads that tie with the warp's
    // maximum (usually one): lowest j == lowest point index inside a thread, lowest index wins across threads
    float best = md[0];
#pragma unroll
    for (int j = 1; j < PPT; ++j) best = fmaxf(best, md[j]);
    uint32_t key = best >= 0.f ? __float_as_uint(best) : 0u;
    uint32_t idx = 0xffffffffu;
    {
      const uint32_t wmax = __reduce_max_sync(0xffffffffu, key);
      if (key == wmax && best >= 0.f) {
        int besti = PPT - 1;
#pragma unroll
        for (int j = PPT - 2; j >= 0; --j) besti = (md[j] == best) ? j : besti;
        idx = (uint32_t)(p0 + besti * T + t);
      }
      idx = __reduce_min_sync(0xffffffffu, idx);
      key = wmax;
    }
    const int buf = g & 1;
    FPS_T(1);
    if (lane == 0) wslot[buf * 32 + warp] = make_uint2(key, idx);
    __syncthreads();
    FPS_T(2);
    {
      const uint2 s = (lane < nwarps) ? wslot[buf * 32 + lane] : make_uint2(0u, 0xffffffffu);
      key = s.x; idx = s.y;
      warp_argmax(key, idx);
    }
    if constexpr (CL > 1) {
      // Only warp 0 talks to the cluster (a cluster-scope acquire by all 1024 threads costs an L1 invalidate each);
      // it reduces the CL candidates and publishes the winner to the CTA through shared memory.
      if (warp == 0) {
        if (lane < ncta) {
          FpsCand c;
          c.key = key; c.idx = idx;
          if (idx != 0xffffffffu) {
            const int l = (int)idx - p0;
            c.x = rows[l * pt_stride]; c.y = rows[l * pt_stride + 1]; c.z = rows[l * pt_stride + 2];
          } else {
            c.x = c.y = c.z = 0.f;
          }
          c.pad[0] = c.pad[1] = c.pad[2] = 0;
          if (lane == 0) fps_expect_cands(&cbar[buf], (uint32_t)ncta * 32u);
          fps_push_cand(&ccand[buf * 16 + rank], &cbar[buf], (uint32_t)lane, c);
        }
        // buffer `buf` is reused every second iteration; a peer can be at most one iteration ahead (it needs this
        // CTA's candidate to finish an iteration), so two buffers and the barrier's phase parity are enough
        FPS_T(3);
        fps_wait_cands(&cbar[buf], (uint32_t)(g >> 1) & 1);
        FPS_T(4);
        uint32_t k2 = lane < ncta ? ccand[buf * 16 + lane].key : 0u;
        uint32_t i2 = lane < ncta ? ccand[buf * 16 + lane].idx : 0xffffffffu;
        const uint32_t mine = i2;
        warp_argmax(k2, i2);                                   // max key, lowest index among the maxima
        const uint32_t src = __ffs(__ballot_sync(0xffffffffu, lane < ncta && mine == i2)) - 1;
        if (lane == (int)src) cwin[buf] = ccand[buf * 16 + lane];
        FPS_T(5);
      }
      __syncthreads();
      FPS_T(6);
      far = (int)min(cwin[buf].idx, (uint32_t)(N - 1));   // no candidate anywhere (cannot happen for finite input): stay in range
      cx = cwin[buf].x; cy = cwin[buf].y; cz = cwin[buf].z;
    } else {
      far = (int)min(idx, (uint32_t)(N - 1));             // idx = 0xffffffff only if no thread had a candidate: stay in range
      cx = rows[far * pt_stride]; cy = rows[far * pt_stride + 1]; cz = rows[far * pt_stride + 2];
    }
  }
  if constexpr (CL > 1) cg::this_cluster().sync();   // no CTA exits while peers may still write to it
}

static size_t fps_smem_bytes(int slice, int pt_stride) {
  const size_t rows_bytes = (((size_t)slice * pt_stride * 4 + 127) / 128) * 128;
  return rows_bytes + 16 + 2 * 32 * sizeof(uint2) + 2 * 16 * sizeof(FpsCand) + 16 + 2 * sizeof(FpsCand);
}

template <int CL, int PPT>
static int fps_configure() {
  static thread_local bool configured[32] = {false};   // per device (cudaFuncSetAttribute is per-device state)
  int dev = 0;
  P3_CUDA(cudaGetDevice(&dev));
  if (dev < 32 && !configured[dev]) {
    P3_CUDA((cudaFuncSetAttribute(fps_kernel<CL, PPT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024)));
    if (CL > 8) P3_CUDA((cudaFuncSetAttribute(fps_kernel<CL, PPT>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1)));
    configured[dev] = true;
  }
  return P3TOK_OK;
}

// clusters of `ncta` CTAs (threads each, smem bytes each) that can be resident at once on the current device; <= 0: unknown
template <int CL, int PPT>
static int fps_max_clusters(int ncta, int threads, size_t smem) {
  if (fps_configure<CL, PPT>() != P3TOK_OK) return -1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(ncta * 64));
  cfg.blockDim = dim3((unsigned)threads);
  cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)ncta;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int n = -1;
  if (cudaOccupancyMaxActiveClusters(&n, fps_kernel<CL, PPT>, &cfg) != cudaSuccess) {
    cudaGetLastError();
    return -1;
  }
  return n;
}

template <int CL, int PPT>
static int fps_launch(const float* x, int B, int N, int pt_stride, const int64_t* start, int G,
                      int64_t* out, int slice, int threads, int ncta, cudaStream_t stream) {
  const size_t smem = fps_smem_bytes(slice, pt_stride);
  int rc = fps_configure<CL, PPT>();
  if (rc) return rc;
  const int CLr = ncta;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(B * CLr));
  cfg.blockDim = dim3((unsigned)threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)CLr;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = CL > 1 ? 1 : 0;
  P3_CUDA((cudaLaunchKernelEx(&cfg, fps_kernel<CL, PPT>, x, N, pt_stride, start, G, out, slice, ncta)));
  count_launch();
  return P3TOK_OK;
}

}  // namespace p3tok

using namespace p3tok;

extern "C" int p3tok_fps(const float* x, int64_t B, int64_t N, int64_t pt_stride,
                         const int64_t* start_idx, int64_t G, int64_t* out_idx, void* stream) {
  P3_REQUIRE(B >= 0 && N > 0 && G >= 0 && pt_stride >= 3, P3TOK_ERR_INVALID,
             "fps: bad shape B=%lld N=%lld G=%lld stride=%lld", (long long)B, (long long)N, (long long)G,
             (long long)pt_stride);
  if (B == 0 || G == 0) return P3TOK_OK;
  P3_REQUIRE(x && start_idx && out_idx, P3TOK_ERR_INVALID, "fps: null pointer");
  P3_REQUIRE(pt_stride <= 4, P3TOK_ERR_UNSUPPORTED, "fps: pt_stride %lld > 4 (pass xyz or xyz+height rows)",
             (long long)pt_stride);
  P3_REQUIRE(N <= (int64_t)FPS_SLICE * 16, P3TOK_ERR_UNSUPPORTED, "fps: N=%lld exceeds 131072", (long long)N);
  P3_REQUIRE(B * 16 < (1ll << 31) && B * G < (1ll << 40), P3TOK_ERR_UNSUPPORTED, "fps: batch too large");
  cudaStream_t s = as_stream(stream);
  const int Bi = (int)B, Ni = (int)N, Gi = (int)G, ps = (int)pt_stride;
  if (N <= FPS_SLICE) {           // one CTA per cloud, every point in registers
    const int ppt = Ni >= 1024 ? 16 : 8;   // measured: 16 beats 8 by 9-12 % from N = 1024 up, 32 is no better
    int threads = ((Ni + ppt - 1) / ppt + 31) / 32 * 32;
    if (threads < 32) threads = 32;
    if (ppt == 16) return fps_launch<1, 16>(x, Bi, Ni, ps, start_idx, Gi, out_idx, Ni, threads, 1, s);
    return fps_launch<1, 8>(x, Bi, Ni, ps, start_idx, Gi, out_idx, Ni, threads, 1, s);
  }
  // A cluster per cloud.  Candidate sizes: from the smallest that holds the cloud (12288 points per CTA as wide slices)
  // up to 8 (16 beyond 8 x 8192 points).  How many clusters of a size the device seats at once is asked of
  // the driver (once per size) - a cluster must sit inside one GPC, so it is NOT #SMs / size: a B200 seats 15 clusters of 8
  // or 7, 22 of 6 - and the choice minimises  waves x cycles per iteration  (measured: ~1000 cycles of reduction / exchange
  // chain + ~0.11 per point of the slice; profiles/microbench/fps_cluster_trace.cu).
  const int lo = (Ni + FPS_SLICE_X - 1) / FPS_SLICE_X;
  const int hi = (Ni + FPS_SLICE - 1) / FPS_SLICE <= 8 ? 8 : 16;
  static thread_local int seats[32][17][33];  // [device][cluster size][warps per CTA]: 0 = not asked yet
  int dev = 0;
  P3_CUDA(cudaGetDevice(&dev));
  int best_cl = 0, best_threads = 0, best_slice = 0;
  double best_cost = 0;
  for (int cl = hi; cl >= lo && cl >= 1; --cl) {
    const int slice = (Ni + cl - 1) / cl;
    const bool wide = slice > FPS_SLICE;
    if (wide && cl > 8) continue;             // the 16-CTA instantiation holds regular slices only
    const int ppt = wide ? FPS_WIDE_PPT : FPS_CL_PPT;
    const int threads = ((slice + ppt - 1) / ppt + 31) / 32 * 32;
    if (threads > fps_max_threads(ppt)) continue;
    int n = dev < 32 ? seats[dev][cl][threads / 32] : 0;
    if (n == 0) {
      const size_t sm = fps_smem_bytes(slice, ps);
      n = cl > 8 ? fps_max_clusters<16, FPS_CL_PPT>(cl, threads, sm)
                 : wide ? fps_max_clusters<8, FPS_WIDE_PPT>(cl, threads, sm) : fps_max_clusters<8, FPS_CL_PPT>(cl, threads, sm);
      if (n <= 0) n = -1;
      if (dev < 32) seats[dev][cl][threads / 32] = n;
    }
    if (n < 0) n = 148 / cl;                  // the driver would not say: assume no placement loss
    const double cost = (double)((Bi + n - 1) / n) * (1000.0 + 0.11 * slice);
    if (best_cl == 0 || cost < best_cost) { best_cl = cl; best_cost = cost; best_threads = threads; best_slice = slice; }
  }
  P3_REQUIRE(best_cl > 0, P3TOK_ERR_UNSUPPORTED, "fps: no cluster size for N=%lld", (long long)N);
  if (best_cl > 8) return fps_launch<16, FPS_CL_PPT>(x, Bi, Ni, ps, start_idx, Gi, out_idx, best_slice, best_threads, best_cl, s);
  if (best_slice > FPS_SLICE)
    return fps_launch<8, FPS_WIDE_PPT>(x, Bi, Ni, ps, start_idx, Gi, out_idx, best_slice, best_threads, best_cl, s);
  return fps_launch<8, FPS_CL_PPT>(x, Bi, Ni, ps, start_idx, Gi, out_idx, best_slice, best_threads, best_cl, s);
}
