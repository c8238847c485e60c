// Decode-sized linear layers for 9 - 64 tokens (one per sequence of a batched decode step): the contract of
// aki_mma_skinny_linear (skinny_linear.cu) -- y = epi(pro(x) W^T), RMSNorm prologue, store / residual / SwiGLU epilogue,
// the same rounding points -- on tcgen05 tensor cores.  Past 8 tokens skinny's design stops working (all of x in shared
// memory, one token per mma.sync n8 column); here x streams through shared memory next to the weights.
//   tile     one cluster = 128 weight rows (x2: gate and up rows in the SwiGLU mode) x BPAD = roundup(B, 16) tokens,
//            fp32 in TMEM.  D[row][token] += W[row][k] x[token][k]: A = weights, B = activations, both K-major
//            SWIZZLE_64B (sm100_ptx.cuh sw64_offset), one M128 x N=BPAD x K16 UMMA per 16 K.
//   split    the K range of a tile is cut into S contiguous runs of 64-element chunks, one per CTA of a cluster of S
//            (dispatch rule: bl_split below).  The partial tiles are reduced through distributed shared memory, with no
//            atomics and no workspace: CTA j of the cluster owns rows [j R, (j + 1) R) of the tile (R = ceil(128 / S)),
//            every CTA writes those rows of its partial into CTA j, and CTA j adds the S partials in rank order and runs
//            the epilogue on them.  The sum order depends on S only, never on B.
//   CTA      warp 0      TMA: weight chunks into a ring of ST stages (the first ST requested before griddepcontrol.wait:
//                        no kernel writes the weights), then the x chunk of every stage (rows >= B load as zeros)
//            warp 1      TMEM allocation; one thread issues the UMMAs, a commit frees each stage
//            warps 2-9   RMSNorm prologue: sum of squares of this CTA's K run of x (4 threads per token), exchanged
//                        through DSMEM so every CTA of the cluster holds the same inverse RMS, then normalise each x
//                        chunk in place in shared memory; finally the K-split reduction and the epilogue
// HBM-bound: algorithmic bytes = N*K*2 (x2 in mode 2) per call; x is re-read from L2 by every row tile.
#include <cuda_bf16.h>
#include <math.h>
#include <mutex>
#include "api_common.cuh"
#include "sm100_ptx.cuh"

namespace aki {

namespace bl {
constexpr int ROWS = 128;                 // weight rows per tile (UMMA M)
constexpr int KC = 64;                    // K per ring stage: two SWIZZLE_64B atoms of 32 elements
constexpr int MAX_SPLIT = 8;              // portable cluster size
constexpr int MAX_B = 64;
constexpr int PWARPS = 8;                 // prologue / epilogue warps
constexpr int PTHREADS = 32 * PWARPS;
constexpr int THREADS = 64 + PTHREADS;
constexpr int SMEM_LIMIT = 220 * 1024;
constexpr int TMEM_COLS = 128;            // 2 accumulators x 64 tokens at most
__host__ __device__ constexpr int nacc(int mode) { return mode == 2 ? 2 : 1; }
__host__ __device__ constexpr int w_stage_bytes(int mode) { return nacc(mode) * ROWS * KC * 2; }
__host__ __device__ constexpr int x_stage_bytes(int bpad) { return bpad * KC * 2; }
__host__ __device__ constexpr int stage_bytes(int mode, int bpad) { return w_stage_bytes(mode) + x_stage_bytes(bpad); }
// reduction buffer [acc][rank][token][rows of this CTA]: S * ceil(128 / S) <= 128 + S - 1 rows
__host__ __device__ constexpr int red_bytes(int mode, int bpad) { return nacc(mode) * (ROWS + MAX_SPLIT) * bpad * 4; }
__host__ __device__ constexpr int stages(int mode, int bpad) {
  return (SMEM_LIMIT - red_bytes(mode, bpad)) / stage_bytes(mode, bpad) > 6
             ? 6 : (SMEM_LIMIT - red_bytes(mode, bpad)) / stage_bytes(mode, bpad);
}
__host__ __device__ constexpr int smem_bytes(int mode, int bpad) {
  return 1024 + stages(mode, bpad) * stage_bytes(mode, bpad) + red_bytes(mode, bpad);
}
static_assert(smem_bytes(2, 64) <= 227 * 1024 && stages(2, 64) >= 3, "SwiGLU at 64 tokens must fit 3 stages");
}  // namespace bl

template <int BPAD, int MODE>
__global__ void __launch_bounds__(bl::THREADS, 1)
batch_linear_kernel(const __grid_constant__ CUtensorMap map_w, const __grid_constant__ CUtensorMap map_x,
                    const __nv_bfloat16* __restrict__ x, int64_t x_stride, const __nv_bfloat16* __restrict__ gamma,
                    float eps, const __nv_bfloat16* __restrict__ residual, int64_t res_stride,
                    __nv_bfloat16* __restrict__ y, int64_t y_stride, int B, int N, int K) {
  using namespace bl;
  constexpr int NACC = nacc(MODE), ST = stages(MODE, BPAD), STAGE = stage_bytes(MODE, BPAD);
  constexpr int WB = w_stage_bytes(MODE), XB = x_stage_bytes(BPAD);
  extern __shared__ uint8_t bl_smem_raw[];
  enum { W_FULL = 0, X_FULL = W_FULL + ST, X_READY = X_FULL + ST, EMPTY = X_READY + ST, ACC_FULL = EMPTY + ST,
         SS_FULL = ACC_FULL + 1, RED_FULL = SS_FULL + 1, N_BARS = RED_FULL + 1 };
  __shared__ __align__(8) uint64_t bars[N_BARS];
  __shared__ float ss_part[MAX_SPLIT][MAX_B];   // [rank][token] sums of squares of each CTA's K run
  __shared__ float inv_rms[BPAD];
  __shared__ uint32_t tmem_base_s;
  const uint32_t raw = smem_u32(bl_smem_raw);
  const uint32_t ring = (raw + 1023u) & ~1023u;
  uint8_t* ring_ptr = bl_smem_raw + (ring - raw);
  const uint32_t red = ring + ST * STAGE;
  const float* red_ptr = reinterpret_cast<const float*>(ring_ptr + ST * STAGE);
  const uint32_t bar0 = smem_u32(bars);
  auto BAR = [&](int i) { return bar0 + 8u * i; };
  auto W_ADDR = [&](int s) { return ring + s * STAGE; };
  auto X_ADDR = [&](int s) { return ring + s * STAGE + WB; };

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int S = gridDim.x, rank = blockIdx.x;          // cluster = (S, 1, 1) = one row of the grid: rank == blockIdx.x
  const int n0 = blockIdx.y * ROWS;
  const int nch = K / KC, c_lo = rank * nch / S, nloc = (rank + 1) * nch / S - c_lo;   // S <= nch: nloc >= 1
  const int R = (ROWS + S - 1) / S;
  const int r_lo = rank * R, rows_me = min(ROWS, r_lo + R) - r_lo;

  auto load_w = [&](int c) {
    const int s = c % ST;
    mbar_arrive_expect_tx(BAR(W_FULL + s), WB);
#pragma unroll
    for (int a = 0; a < NACC; ++a)
#pragma unroll
      for (int h = 0; h < 2; ++h)
        tma_load_2d(W_ADDR(s) + a * (ROWS * KC * 2) + h * (ROWS * 64), &map_w, BAR(W_FULL + s), (c_lo + c) * KC + 32 * h,
                    n0 + a * N);
  };
  if (tid == 0) {
    for (int s = 0; s < ST; ++s) {
      mbar_init(BAR(W_FULL + s), 1); mbar_init(BAR(X_FULL + s), 1);
      mbar_init(BAR(X_READY + s), PTHREADS); mbar_init(BAR(EMPTY + s), 1);
    }
    mbar_init(BAR(ACC_FULL), 1);
    mbar_init(BAR(SS_FULL), S * B);                     // one arrival per token from every CTA of the cluster
    mbar_init(BAR(RED_FULL), 2 * S * rows_me);          // one per (row, column half) of every CTA
    fence_barrier_init();
    tma_prefetch_desc(&map_w); tma_prefetch_desc(&map_x);
    for (int c = 0; c < min(ST, nloc); ++c) load_w(c);
  }
  if (warp == 1) tmem_alloc<TMEM_COLS>(smem_u32(&tmem_base_s));
  tc_fence_before();
  cluster_sync();                 // barrier inits of every CTA precede any remote access; doubles as __syncthreads
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  pdl_wait();                     // x / residual come from the previous kernel
  pdl_trigger();

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (elect_one()) {
      for (int c = 0; c < nloc; ++c) {
        const int s = c % ST;
        if (c >= ST) {
          mbar_wait(BAR(EMPTY + s), ((c / ST) - 1) & 1);
          load_w(c);
        }
        mbar_arrive_expect_tx(BAR(X_FULL + s), XB);
        for (int h = 0; h < 2; ++h)
          tma_load_2d(X_ADDR(s) + h * (BPAD * 64), &map_x, BAR(X_FULL + s), (c_lo + c) * KC + 32 * h, 0);
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (elect_one()) {
      constexpr uint32_t IDESC = umma_idesc_bf16(ROWS, BPAD, 0, 0);
      for (int c = 0; c < nloc; ++c) {
        const int s = c % ST;
        const uint32_t par = (c / ST) & 1;
        mbar_wait(BAR(W_FULL + s), par);
        mbar_wait(BAR((gamma ? X_READY : X_FULL) + s), par);
        tc_fence_after();
#pragma unroll
        for (int k = 0; k < KC / 16; ++k) {
          const uint64_t bdesc = umma_smem_desc(X_ADDR(s) + (k >> 1) * (BPAD * 64) + (k & 1) * 32, 16, 512, UMMA_SW64);
#pragma unroll
          for (int a = 0; a < NACC; ++a) {
            const uint64_t adesc =
                umma_smem_desc(W_ADDR(s) + a * (ROWS * KC * 2) + (k >> 1) * (ROWS * 64) + (k & 1) * 32, 16, 512, UMMA_SW64);
            umma_ss(tmem + a * BPAD, adesc, bdesc, IDESC, (c > 0 || k > 0) ? 1u : 0u);
          }
        }
        umma_commit(BAR(EMPTY + s));
      }
      umma_commit(BAR(ACC_FULL));
    }
  } else {
    const int ptid = tid - 64;
    if (gamma) {
      // ---------------------------------------------------------------- RMSNorm prologue
      // sum of squares of this CTA's K run: token b = ptid / 4, thread j = ptid % 4 adds the squares of 16-byte pieces
      // j, j + 4, ... in order (one FMA each), then two xor-shuffle levels; CTA j adds the S runs in rank order
      {
        const int b = ptid >> 2, j = ptid & 3, np = nloc * (KC / 8);
        float ss = 0.f;
        if (b < B) {
          const __nv_bfloat16* xr = x + (size_t)b * x_stride + (size_t)c_lo * KC;
          for (int p0 = j; p0 < np; p0 += 4 * 8) {
            uint4 u[8];
#pragma unroll
            for (int i = 0; i < 8; ++i)
              if (p0 + 4 * i < np) u[i] = *reinterpret_cast<const uint4*>(xr + 8 * (p0 + 4 * i));
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              if (p0 + 4 * i < np) {
                const __nv_bfloat162* hv = reinterpret_cast<const __nv_bfloat162*>(&u[i]);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const float2 f = __bfloat1622float2(hv[e]);
                  ss = fmaf(f.x, f.x, ss);
                  ss = fmaf(f.y, f.y, ss);
                }
              }
            }
          }
        }
        ss += __shfl_xor_sync(0xffffffffu, ss, 1);
        ss += __shfl_xor_sync(0xffffffffu, ss, 2);
        if (b < B && j == 0) {
          const uint32_t local = smem_u32(&ss_part[rank][b]);
          for (int r = 0; r < S; ++r) {
            st_cluster_f32(mapa_shared(local, r), ss);
            mbar_arrive_cluster(mapa_shared(BAR(SS_FULL), r));
          }
        }
      }
      mbar_wait_cluster(BAR(SS_FULL), 0);
      if (ptid < BPAD) {
        float t = 0.f;
        if (ptid < B)
          for (int r = 0; r < S; ++r) t += ss_part[r][ptid];
        inv_rms[ptid] = ptid < B ? rsqrtf(t / (float)K + eps) : 0.f;
      }
      named_bar_sync(1, PTHREADS);
      // normalise every x chunk in place as it lands: 16-byte piece q of the stage is (atom, row, swizzled chunk)
      for (int c = 0; c < nloc; ++c) {
        const int s = c % ST;
        mbar_wait(BAR(X_FULL + s), (c / ST) & 1);
        for (int q = ptid; q < BPAD * 8; q += PTHREADS) {
          const int a = q / (BPAD * 4), rem = q % (BPAD * 4), row = rem >> 2;
          const int lc = (rem & 3) ^ ((row >> 1) & 3);
          const int k = (c_lo + c) * KC + a * 32 + lc * 8;
          uint4* p = reinterpret_cast<uint4*>(ring_ptr + s * STAGE + WB + q * 16);
          const uint4 gm = *reinterpret_cast<const uint4*>(gamma + k);
          const __nv_bfloat162* gw = reinterpret_cast<const __nv_bfloat162*>(&gm);
          uint4 u = *p;
          __nv_bfloat162* hv = reinterpret_cast<__nv_bfloat162*>(&u);
          const float r = inv_rms[row];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 f = __bfloat1622float2(hv[e]);
            // Phi3RMSNorm: weight * (x * rsqrt(mean(x^2) + eps)).to(bf16)   -- two roundings
            hv[e] = __hmul2(gw[e], __floats2bfloat162_rn(f.x * r, f.y * r));
          }
          *p = u;
        }
        fence_proxy_async_smem();
        mbar_arrive(BAR(X_READY + s));
      }
    }
    // ------------------------------------------------------------------ K-split reduction through DSMEM
    // thread = TMEM lane (weight row) of its warp's lane quarter, one half of the token columns
    {
      const int quarter = warp & 3, half = (warp - 2) >> 2;
      const int row = 32 * quarter + lane;
      const int jt = row / R, rows_t = min(ROWS, (jt + 1) * R) - jt * R, rr = row - jt * R;
      const uint32_t dst = mapa_shared(red, jt);
      mbar_wait(BAR(ACC_FULL), 0);
      tc_fence_after();
#pragma unroll
      for (int a = 0; a < NACC; ++a) {
#pragma unroll
        for (int c8 = 0; c8 < BPAD / 16; ++c8) {
          const int col = half * (BPAD / 2) + 8 * c8;
          uint32_t v[8];
          tmem_ld_x8(tmem + ((uint32_t)(32 * quarter) << 16) + a * BPAD + col, v);
          tmem_wait_ld();
#pragma unroll
          for (int e = 0; e < 8; ++e)
            st_cluster_f32(dst + 4u * (uint32_t)((((a * S + rank) * BPAD + col + e) * rows_t) + rr), __uint_as_float(v[e]));
        }
      }
      tc_fence_before();
      mbar_arrive_cluster(mapa_shared(BAR(RED_FULL), jt));
    }
    mbar_wait_cluster(BAR(RED_FULL), 0);
    for (int idx = ptid; idx < rows_me * B; idx += PTHREADS) {
      const int b = idx / rows_me, rr = idx - b * rows_me, n = n0 + r_lo + rr;
      float s = 0.f, s2 = 0.f;
      for (int r = 0; r < S; ++r) {
        s += red_ptr[((size_t)r * BPAD + b) * rows_me + rr];
        if (MODE == 2) s2 += red_ptr[((size_t)(S + r) * BPAD + b) * rows_me + rr];
      }
      if (n < N) {
        float out = s;
        if (MODE == 2) {
          // Phi3MLP: down_proj(up * silu(gate)) with gate / up rounded to bf16 by gate_up_proj first
          const float gq = __bfloat162float(__float2bfloat16(s)), uq = __bfloat162float(__float2bfloat16(s2));
          const float act = __bfloat162float(__float2bfloat16(gq / (1.f + __expf(-gq))));
          out = uq * act;
        } else if (MODE == 1) {
          out = __bfloat162float(__float2bfloat16(s)) + __bfloat162float(residual[(size_t)b * res_stride + n]);
        }
        y[(size_t)b * y_stride + n] = __float2bfloat16(out);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc<TMEM_COLS>(tmem);
}

// ------------------------------------------------------------------------------------------------ host side
namespace bl {
constexpr int BPADS[4] = {16, 32, 48, 64};
using KernFn = void (*)(CUtensorMap, CUtensorMap, const __nv_bfloat16*, int64_t, const __nv_bfloat16*, float,
                        const __nv_bfloat16*, int64_t, __nv_bfloat16*, int64_t, int, int, int);
static KernFn kernel_table(int mode, int bi) {
#define AKI_BL_K(P) (mode == 0 ? (KernFn)batch_linear_kernel<P, 0> : mode == 1 ? (KernFn)batch_linear_kernel<P, 1> \
                                                                                : (KernFn)batch_linear_kernel<P, 2>)
  return bi == 0 ? AKI_BL_K(16) : bi == 1 ? AKI_BL_K(32) : bi == 2 ? AKI_BL_K(48) : AKI_BL_K(64);
#undef AKI_BL_K
}
static int smem_of(int mode, int bi) {
  const int p = BPADS[bi];
  return mode == 2 ? smem_bytes(2, p) : smem_bytes(0, p);
}

// Per-device one-time setup: shared-memory attribute of every instantiation, SM count, and for every cluster size s the
// number of clusters of s CTAs that can be resident at once (a cluster lives inside one GPC, so s-CTA clusters of
// one-CTA-per-SM kernels cannot always fill every SM).
struct DeviceState {
  std::once_flag once;
  cudaError_t err = cudaSuccess;
  int sm_count = 0;
  int max_clusters[3][4][MAX_SPLIT + 1] = {};
};
static DeviceState g_dev[64];

static int device_state(DeviceState** out) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { set_last_cuda_error("cudaGetDevice failed"); return AKI_ERR_CUDA; }
  DeviceState& d = g_dev[dev];
  std::call_once(d.once, [&]() {
    d.err = cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, dev);
    for (int m = 0; m < 3 && d.err == cudaSuccess; ++m)
      for (int bi = 0; bi < 4 && d.err == cudaSuccess; ++bi) {
        KernFn k = kernel_table(m, bi);
        d.err = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_of(m, bi));
        for (int s = 1; s <= MAX_SPLIT && d.err == cudaSuccess; ++s) {
          cudaLaunchConfig_t cfg = {};
          cfg.gridDim = dim3(s, 1, 1);
          cfg.blockDim = dim3(THREADS);
          cfg.dynamicSmemBytes = smem_of(m, bi);
          cudaLaunchAttribute attr[1];
          attr[0].id = cudaLaunchAttributeClusterDimension;
          attr[0].val.clusterDim.x = s; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
          cfg.attrs = attr;
          cfg.numAttrs = 1;
          int n = 0;
          d.err = cudaOccupancyMaxActiveClusters(&n, k, &cfg);
          d.max_clusters[m][bi][s] = n;
        }
      }
  });
  if (d.err != cudaSuccess) { set_last_cuda_error(cudaGetErrorString(d.err)); return AKI_ERR_CUDA; }
  *out = &d;
  return AKI_OK;
}

// THE DISPATCH RULE.  tiles = ceil(N / 128) row tiles, nch = K / 64 chunks.  Split S = the largest s in
// [1, min(8, nch)] such that the tiles x s CTAs fit in one wave: tiles * s <= SMs and tiles <= the number of s-CTA
// clusters the device can hold at once (DeviceState::max_clusters, per mode and token padding).  S = 1 when none does
// (the lm_head's 251 tiles: every CTA streams a whole tile).  aki_mma_batch_linear_split() reports it.
static int bl_split(const DeviceState& d, int mode, int bi, int N, int K) {
  const int tiles = (N + ROWS - 1) / ROWS, nch = K / KC;
  for (int s = nch < MAX_SPLIT ? nch : MAX_SPLIT; s > 1; --s)
    if ((long long)tiles * s <= d.sm_count && tiles <= d.max_clusters[mode][bi][s]) return s;
  return 1;
}
}  // namespace bl

}  // namespace aki

using namespace aki;

static int batch_linear_check(const void* x, int64_t x_stride, const void* w, const void* rms_weight,
                              const void* residual, const void* y, int B, int N, int K, int mode) {
  AKI_REQUIRE(x && w && y, AKI_ERR_NULL);
  AKI_REQUIRE(B >= 1 && B <= bl::MAX_B && N > 0 && K > 0 && mode >= 0 && mode <= 2, AKI_ERR_BAD_SHAPE);
  AKI_REQUIRE(N % 16 == 0 && K % bl::KC == 0, AKI_ERR_UNSUPPORTED);
  AKI_REQUIRE((mode == 1) == (residual != nullptr), AKI_ERR_NULL);
  AKI_REQUIRE(x_stride % 8 == 0 && (B == 1 || x_stride >= K), AKI_ERR_UNSUPPORTED);
  AKI_REQUIRE(aligned16(x) && aligned16(w) && (!rms_weight || aligned16(rms_weight)), AKI_ERR_MISALIGNED);
  return AKI_OK;
}

extern "C" int aki_mma_batch_linear_split(int B, int N, int K, int mode) {
  AKI_REQUIRE(B >= 1 && B <= bl::MAX_B && N > 0 && K > 0 && mode >= 0 && mode <= 2, AKI_ERR_BAD_SHAPE);
  AKI_REQUIRE(N % 16 == 0 && K % bl::KC == 0, AKI_ERR_UNSUPPORTED);
  bl::DeviceState* d = nullptr;
  int rc = bl::device_state(&d);
  if (rc) return rc;
  return bl::bl_split(*d, mode, (B - 1) / 16, N, K);
}

extern "C" int aki_mma_batch_linear(const void* x, int64_t x_stride, const void* w, const void* rms_weight, float rms_eps,
                                    const void* residual, int64_t residual_stride, void* y, int64_t y_stride, int B, int N,
                                    int K, int mode, aki_stream_t stream) {
  int rc = batch_linear_check(x, x_stride, w, rms_weight, residual, y, B, N, K, mode);
  if (rc) return rc;
  bl::DeviceState* d = nullptr;
  if ((rc = bl::device_state(&d))) return rc;
  const int bi = (B - 1) / 16;
  const int S = bl::bl_split(*d, mode, bi, N, K);
  CUtensorMap mw, mx;
  if ((rc = make_bf16_map_2d(&mw, w, K, mode == 2 ? 2 * N : N, K, bl::ROWS))) return rc;
  if ((rc = make_bf16_map_2d(&mx, x, K, B, B == 1 ? K : x_stride, bl::BPADS[bi]))) return rc;
  const int tiles = (N + bl::ROWS - 1) / bl::ROWS;
  // programmatic dependent launch (api_common.cuh): the CTAs start, and request their first weight chunks, while the
  // previous kernel of the stream drains
  launch_pdl_cluster(bl::kernel_table(mode, bi), dim3(S, tiles), dim3(bl::THREADS), bl::smem_of(mode, bi),
                     static_cast<cudaStream_t>(stream), (unsigned)S, mw, mx, static_cast<const __nv_bfloat16*>(x),
                     x_stride, static_cast<const __nv_bfloat16*>(rms_weight),
                     rms_eps, static_cast<const __nv_bfloat16*>(residual), residual_stride,
                     static_cast<__nv_bfloat16*>(y), y_stride, B, N, K);
  return check_launch();
}
