// Optimizer step of the SFT loop (include/aki_mma.h section (10)): the gradient clipping and the AdamW update of the
// reference's train_utils.py:143-158 (clip_grad_norm_ + AdamW.step) as two HBM-bound passes over a list of fp32 tensors.
//   grad_sq_norm  sum of g^2 over every tensor: per-chunk fp32 partials in HBM, then one CTA adds them in chunk order in
//                 fp64 (no float atomics: the same inputs give the same bits on every run and for any launch split).
//   adamw_step    g * min(1, max_norm / (sqrt(sq_norm) + 1e-6)), then torch.optim.AdamW's fused update (ATen
//                 fused_adam_utils.cuh adam_math, ADAMW mode) in the same fp32 operations and order, and the bf16 copy
//                 of the new parameter that the forward's Linears read instead of autocast's weight cast.
// The tensor list travels in the kernel's parameter space (__grid_constant__, up to OPT_MAX_ENTRIES = 256 entries per
// launch): no device table and no host-to-device copy.  A tensor is cut into chunks of OPT_CHUNK elements; chunk c of a
// launch belongs to the last entry whose first chunk is <= c.  16-byte accesses, scalar tail for numel % 4 != 0.
#include <cuda_bf16.h>
#include <math.h>
#include <string.h>
#include "api_common.cuh"

namespace aki {

constexpr int OPT_THREADS = 256;
constexpr int64_t OPT_CHUNK = OPT_THREADS * 4 * 16;   // 16384 elements: 16 float4 per thread
constexpr int OPT_MAX_ENTRIES = 256;                   // 256 x 56 B = 14 KB of the 32 KB parameter space

struct OptEntry {
  float* p;
  const float* g;
  float* m;
  float* v;
  __nv_bfloat16* p16;
  int64_t numel;
  int64_t chunk0;    // first chunk of this entry within the launch
};
struct OptList {
  int n;
  int64_t n_chunks;
  OptEntry e[OPT_MAX_ENTRIES];
};
struct AdamWHyper {
  float lr, beta1, beta2, eps, weight_decay, max_norm, step;
  const float* sq_norm;   // NULL: no clipping
};

__device__ __forceinline__ int opt_entry_of(const OptList& L, int64_t c) {
  int lo = 0, hi = L.n - 1;                 // largest i with chunk0 <= c (an empty entry shares chunk0 with the next)
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (L.e[mid].chunk0 <= c) lo = mid; else hi = mid - 1;
  }
  return lo;
}

__global__ void __launch_bounds__(OPT_THREADS)
grad_sq_norm_kernel(const __grid_constant__ OptList L, float* __restrict__ partial) {
  __shared__ float red[OPT_THREADS / 32];
  pdl_wait();
  pdl_trigger();
  for (int64_t c = blockIdx.x; c < L.n_chunks; c += gridDim.x) {
    const OptEntry& E = L.e[opt_entry_of(L, c)];
    const int64_t begin = (c - E.chunk0) * OPT_CHUNK;
    const int64_t end = min(begin + OPT_CHUNK, E.numel);
    const int64_t vend = begin + ((end - begin) & ~int64_t(3));
    float s = 0.f;
#pragma unroll 4
    for (int64_t k = begin + threadIdx.x * 4; k < vend; k += OPT_THREADS * 4) {
      const float4 g = *reinterpret_cast<const float4*>(E.g + k);
      s = fmaf(g.x, g.x, s); s = fmaf(g.y, g.y, s); s = fmaf(g.z, g.z, s); s = fmaf(g.w, g.w, s);
    }
    for (int64_t k = vend + threadIdx.x; k < end; k += OPT_THREADS) s = fmaf(E.g[k], E.g[k], s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = red[0];
#pragma unroll
      for (int w = 1; w < OPT_THREADS / 32; ++w) t += red[w];
      partial[c] = t;
    }
    __syncthreads();
  }
}

constexpr int OPT_FINISH_THREADS = 1024;

__global__ void __launch_bounds__(OPT_FINISH_THREADS)
grad_sq_norm_finish_kernel(const float* __restrict__ partial, int64_t n, float* __restrict__ sq_norm) {
  __shared__ double red[OPT_FINISH_THREADS / 32];
  pdl_wait();
  pdl_trigger();
  double s = 0.0;
#pragma unroll 8
  for (int64_t k = threadIdx.x; k < n; k += OPT_FINISH_THREADS) s += (double)partial[k];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = red[0];
    for (int w = 1; w < OPT_FINISH_THREADS / 32; ++w) t += red[w];
    sq_norm[0] = (float)t;
  }
}

// torch.optim.AdamW(fused=True) per element, written as ATen's adam_math writes it so that nvcc forms the same fp32
// operations (the same fma contractions and IEEE divisions / square roots).
__device__ __forceinline__ void adamw_elem(float& p, float g, float& m, float& v, float lr, float beta1, float beta2,
                                           float eps, float weight_decay, float step_size, float bc2_sqrt) {
  if (weight_decay != 0) p -= lr * weight_decay * p;
  m = fmaf(beta1, m, fmaf(-beta1, g, g));
  v = fmaf(beta2, v, fmaf(-beta2, g * g, g * g));
  const float denom = (sqrtf(v) / bc2_sqrt) + eps;
  p -= step_size * m / denom;
}

__global__ void __launch_bounds__(OPT_THREADS, 4)
adamw_kernel(const __grid_constant__ OptList L, const AdamWHyper h) {
  // bias corrections as torch computes them: float pow of the float step count
  const float bc1 = 1 - powf(h.beta1, h.step);
  const float bc2_sqrt = sqrtf(1 - powf(h.beta2, h.step));
  const float step_size = h.lr / bc1;
  pdl_wait();
  pdl_trigger();
  float clip = 1.f;
  if (h.sq_norm) {
    // clip_grads_with_norm_: max_norm / (total_norm + 1e-6), i.e. reciprocal(total_norm + 1e-6) * max_norm, clamped to
    // 1; a NaN passes through the clamp as torch.clamp passes it
    const float c = __fdiv_rn(1.f, sqrtf(h.sq_norm[0]) + 1e-6f) * h.max_norm;
    clip = c > 1.f ? 1.f : c;
  }
  const bool scale = h.sq_norm != nullptr;
  for (int64_t c = blockIdx.x; c < L.n_chunks; c += gridDim.x) {
    const OptEntry& E = L.e[opt_entry_of(L, c)];
    const int64_t begin = (c - E.chunk0) * OPT_CHUNK;
    const int64_t end = min(begin + OPT_CHUNK, E.numel);
    const int64_t vend = begin + ((end - begin) & ~int64_t(3));
#pragma unroll 2
    for (int64_t k = begin + threadIdx.x * 4; k < vend; k += OPT_THREADS * 4) {
      float4 p = *reinterpret_cast<const float4*>(E.p + k);
      float4 g = *reinterpret_cast<const float4*>(E.g + k);
      float4 m = *reinterpret_cast<const float4*>(E.m + k);
      float4 v = *reinterpret_cast<const float4*>(E.v + k);
      if (scale) { g.x *= clip; g.y *= clip; g.z *= clip; g.w *= clip; }
      adamw_elem(p.x, g.x, m.x, v.x, h.lr, h.beta1, h.beta2, h.eps, h.weight_decay, step_size, bc2_sqrt);
      adamw_elem(p.y, g.y, m.y, v.y, h.lr, h.beta1, h.beta2, h.eps, h.weight_decay, step_size, bc2_sqrt);
      adamw_elem(p.z, g.z, m.z, v.z, h.lr, h.beta1, h.beta2, h.eps, h.weight_decay, step_size, bc2_sqrt);
      adamw_elem(p.w, g.w, m.w, v.w, h.lr, h.beta1, h.beta2, h.eps, h.weight_decay, step_size, bc2_sqrt);
      *reinterpret_cast<float4*>(E.p + k) = p;
      *reinterpret_cast<float4*>(E.m + k) = m;
      *reinterpret_cast<float4*>(E.v + k) = v;
      if (E.p16) {
        __nv_bfloat162 lo = __floats2bfloat162_rn(p.x, p.y), hi = __floats2bfloat162_rn(p.z, p.w);
        uint2 u;
        memcpy(&u.x, &lo, 4);
        memcpy(&u.y, &hi, 4);
        *reinterpret_cast<uint2*>(E.p16 + k) = u;
      }
    }
    for (int64_t k = vend + threadIdx.x; k < end; k += OPT_THREADS) {
      float p = E.p[k], g = E.g[k], m = E.m[k], v = E.v[k];
      if (scale) g *= clip;
      adamw_elem(p, g, m, v, h.lr, h.beta1, h.beta2, h.eps, h.weight_decay, step_size, bc2_sqrt);
      E.p[k] = p; E.m[k] = m; E.v[k] = v;
      if (E.p16) E.p16[k] = __float2bfloat16_rn(p);
    }
  }
}

static int64_t chunks_of(int64_t numel) { return (numel + OPT_CHUNK - 1) / OPT_CHUNK; }

// Host checks shared by both entry points; `full` = the update's pointers too (the norm reads grad only).
static int check_entries(const AkiAdamWTensor* t, int n, bool full) {
  AKI_REQUIRE(t != nullptr, AKI_ERR_NULL);
  AKI_REQUIRE(n > 0, AKI_ERR_BAD_SHAPE);
  for (int i = 0; i < n; ++i) {   // an empty tensor may have NULL pointers (torch gives empty CUDA tensors no storage)
    AKI_REQUIRE(t[i].grad || t[i].numel == 0, AKI_ERR_NULL);
    AKI_REQUIRE(!full || t[i].numel == 0 || (t[i].param && t[i].exp_avg && t[i].exp_avg_sq), AKI_ERR_NULL);
  }
  for (int i = 0; i < n; ++i) AKI_REQUIRE(t[i].numel >= 0, AKI_ERR_BAD_SHAPE);
  for (int i = 0; i < n; ++i) {
    AKI_REQUIRE(aligned16(t[i].grad), AKI_ERR_MISALIGNED);
    AKI_REQUIRE(!full || (aligned16(t[i].param) && aligned16(t[i].exp_avg) && aligned16(t[i].exp_avg_sq) &&
                          aligned16(t[i].param_bf16)),
                AKI_ERR_MISALIGNED);
  }
  return AKI_OK;
}

static int64_t total_chunks(const AkiAdamWTensor* t, int n) {
  int64_t c = 0;
  for (int i = 0; i < n; ++i) c += chunks_of(t[i].numel);
  return c;
}

// Fills `L` with entries [first, first + count) of `t`; returns the launch's chunk count.
static int64_t fill_list(OptList& L, const AkiAdamWTensor* t, int first, int count) {
  L.n = count;
  int64_t c = 0;
  for (int i = 0; i < count; ++i) {
    const AkiAdamWTensor& s = t[first + i];
    L.e[i] = {s.param, s.grad, s.exp_avg, s.exp_avg_sq, static_cast<__nv_bfloat16*>(s.param_bf16), s.numel, c};
    c += chunks_of(s.numel);
  }
  L.n_chunks = c;
  return c;
}

// Persistent grid: `per_sm` resident CTAs per SM (adamw: 54 registers -> 4; norm: 8), chunks taken grid-stride.
static int grid_for(int64_t n_chunks, int per_sm) {
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  cudaGetLastError();
  const int64_t cap = (int64_t)sms * per_sm;
  return (int)(n_chunks < cap ? n_chunks : cap);
}

}  // namespace aki

extern "C" size_t aki_mma_grad_sq_norm_workspace_bytes(const AkiAdamWTensor* t, int n) {
  if (aki::check_entries(t, n, false) != AKI_OK) return 0;
  const int64_t c = aki::total_chunks(t, n);
  return (size_t)((c * 4 + 15) / 16 * 16 + 16);
}

extern "C" int aki_mma_grad_sq_norm(const AkiAdamWTensor* t, int n, void* workspace, size_t workspace_bytes,
                                    float* sq_norm, aki_stream_t stream) {
  const int st = aki::check_entries(t, n, false);
  if (st != AKI_OK) return st;
  AKI_REQUIRE(workspace && sq_norm, AKI_ERR_NULL);
  AKI_REQUIRE(aki::aligned16(workspace), AKI_ERR_MISALIGNED);
  AKI_REQUIRE(workspace_bytes >= aki_mma_grad_sq_norm_workspace_bytes(t, n), AKI_ERR_BAD_SHAPE);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  float* partial = static_cast<float*>(workspace);
  int64_t done = 0;
  static thread_local aki::OptList L;
  for (int first = 0; first < n; first += aki::OPT_MAX_ENTRIES) {
    const int count = n - first < aki::OPT_MAX_ENTRIES ? n - first : aki::OPT_MAX_ENTRIES;
    const int64_t c = aki::fill_list(L, t, first, count);
    if (c == 0) continue;
    aki::launch_pdl(aki::grad_sq_norm_kernel, dim3(aki::grid_for(c, 8)), dim3(aki::OPT_THREADS), 0, s, L, partial + done);
    const int e = aki::check_launch();
    if (e != AKI_OK) return e;
    done += c;
  }
  aki::launch_pdl(aki::grad_sq_norm_finish_kernel, dim3(1), dim3(aki::OPT_FINISH_THREADS), 0, s,
                  static_cast<const float*>(partial), done, sq_norm);
  return aki::check_launch();
}

extern "C" int aki_mma_adamw_step(const AkiAdamWTensor* t, int n, const float* sq_norm, float max_norm, float lr,
                                  float beta1, float beta2, float eps, float weight_decay, int64_t step,
                                  aki_stream_t stream) {
  const int st = aki::check_entries(t, n, true);
  if (st != AKI_OK) return st;
  AKI_REQUIRE(isfinite(lr) && lr >= 0.f, AKI_ERR_BAD_SHAPE);
  AKI_REQUIRE(beta1 >= 0.f && beta1 < 1.f && beta2 >= 0.f && beta2 < 1.f, AKI_ERR_BAD_SHAPE);   // false for NaN
  AKI_REQUIRE(isfinite(eps) && eps >= 0.f, AKI_ERR_BAD_SHAPE);
  AKI_REQUIRE(isfinite(weight_decay) && weight_decay >= 0.f, AKI_ERR_BAD_SHAPE);
  AKI_REQUIRE(step >= 1, AKI_ERR_BAD_SHAPE);
  AKI_REQUIRE(!sq_norm || (isfinite(max_norm) && max_norm > 0.f), AKI_ERR_BAD_SHAPE);
  const aki::AdamWHyper h = {lr, beta1, beta2, eps, weight_decay, max_norm, (float)step, sq_norm};
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  static thread_local aki::OptList L;
  for (int first = 0; first < n; first += aki::OPT_MAX_ENTRIES) {
    const int count = n - first < aki::OPT_MAX_ENTRIES ? n - first : aki::OPT_MAX_ENTRIES;
    const int64_t c = aki::fill_list(L, t, first, count);
    if (c == 0) continue;
    aki::launch_pdl(aki::adamw_kernel, dim3(aki::grid_for(c, 4)), dim3(aki::OPT_THREADS), 0, s, L, h);
    const int e = aki::check_launch();
    if (e != AKI_OK) return e;
  }
  return AKI_OK;
}
