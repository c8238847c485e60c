// Decode attention: one query per sequence against the whole KV cache (the reference's generate loop after
// prefill replaces the 4-D mask by a 2-D all-ones mask, codes/open_flamingo/src/aki_generation.py:56-84, so
// there is no MMA term).  HBM-bound: every K and V byte is read exactly once with 16-byte loads; split over
// the key axis so B*H*splits CTAs fill the 148 SMs, then a tiny combine kernel merges the partial softmaxes.
// Algorithmic bytes per call = 2 * B * H * kv_len * 96 * 2.
#include <cuda_bf16.h>
#include <math.h>
#include "api_common.cuh"

namespace aki {

constexpr int DEC_THREADS = 128;
constexpr int DEC_CHUNK = 512;  // keys per CTA
constexpr int DEC_D = 96;

__device__ __forceinline__ void bf8_to_f(const uint4& u, float* f) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t = __bfloat1622float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ uint4 ldg_nc_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

// lane = (g, s): g = lane>>2 in [0,8) picks the key, s = lane&3 owns 16-byte chunks {s, s+4, s+8} of the 96-wide row
__global__ void __launch_bounds__(DEC_THREADS)
decode_partial_kernel(const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ k_cache,
                      const __nv_bfloat16* __restrict__ v_cache, int64_t cache_stride_b, int64_t cache_stride_h,
                      const int32_t* __restrict__ kv_len, const int32_t* __restrict__ kv_start,
                      const uint32_t* __restrict__ kv_valid_bits, int bits_pitch, int H, float scale_log2, int n_splits,
                      float* __restrict__ ws_m, float* __restrict__ ws_l, float* __restrict__ ws_acc) {
  const int split = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, s = lane & 3;
  pdl_wait();          // q and the newest K / V row come from the previous kernel of a decode step
  pdl_trigger();
  const int len = kv_len[b];
  // keys [kv_start[b], kv_len[b]) are visible: left-padded prompts (padding_side="left" in AKI.generate) keep their pad
  // rows at the front of the cache
  const int j0 = max(split * DEC_CHUNK, kv_start ? kv_start[b] : 0), j1 = min(split * DEC_CHUNK + DEC_CHUNK, len);
  const size_t part = ((size_t)b * H + h) * n_splits + split;
  // interior invalid rows (the left padding of a follow-up turn's prompt): one bit per key
  const uint32_t* vbits = kv_valid_bits ? kv_valid_bits + (size_t)b * bits_pitch : nullptr;

  float qf[24];
  {
    const __nv_bfloat16* qp = q + ((size_t)b * H + h) * DEC_D;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      uint4 u = *reinterpret_cast<const uint4*>(qp + (s + 4 * i) * 8);
      bf8_to_f(u, qf + 8 * i);
    }
#pragma unroll
    for (int i = 0; i < 24; ++i) qf[i] *= scale_log2;
  }
  float m = -INFINITY, l = 0.f, acc[24];
#pragma unroll
  for (int i = 0; i < 24; ++i) acc[i] = 0.f;

  const __nv_bfloat16* kb = k_cache + (size_t)b * cache_stride_b + (size_t)h * cache_stride_h;
  const __nv_bfloat16* vb = v_cache + (size_t)b * cache_stride_b + (size_t)h * cache_stride_h;
  for (int jb = j0 + warp * 8; jb < j1; jb += (DEC_THREADS / 32) * 8 * 2) {
    // two keys per lane in flight
    uint4 ku[2][3], vu[2][3];
    bool ok[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int j = jb + u * (DEC_THREADS / 32) * 8 + g;
      ok[u] = j < j1;
      const int jj = ok[u] ? j : j0;
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        ku[u][i] = ldg_nc_v4(kb + (size_t)jj * DEC_D + (s + 4 * i) * 8);
        vu[u][i] = ldg_nc_v4(vb + (size_t)jj * DEC_D + (s + 4 * i) * 8);
      }
    }
    // the validity bit is folded in after the K / V loads are issued: their addresses must not wait on it
    if (vbits) {
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int j = jb + u * (DEC_THREADS / 32) * 8 + g;
        if (ok[u]) ok[u] = (__ldg(vbits + (j >> 5)) >> (j & 31)) & 1u;
      }
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      float kf[8], dot = 0.f;
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        bf8_to_f(ku[u][i], kf);
#pragma unroll
        for (int e = 0; e < 8; ++e) dot = fmaf(qf[8 * i + e], kf[e], dot);
      }
      dot += __shfl_xor_sync(0xffffffffu, dot, 1);
      dot += __shfl_xor_sync(0xffffffffu, dot, 2);
      if (ok[u]) {
        const float m_new = fmaxf(m, dot);
        const float alpha = exp2f(m - m_new);
        const float p = exp2f(dot - m_new);
        l = l * alpha + p;
        m = m_new;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          bf8_to_f(vu[u][i], kf);
#pragma unroll
          for (int e = 0; e < 8; ++e) acc[8 * i + e] = fmaf(p, kf[e], acc[8 * i + e] * alpha);
        }
      }
    }
  }
  // merge the 8 key groups of the warp
#pragma unroll
  for (int o = 4; o < 32; o <<= 1) {
    const float m_o = __shfl_xor_sync(0xffffffffu, m, o);
    const float l_o = __shfl_xor_sync(0xffffffffu, l, o);
    const float m_new = fmaxf(m, m_o);
    const float a = (m == -INFINITY) ? 0.f : exp2f(m - m_new);
    const float bsc = (m_o == -INFINITY) ? 0.f : exp2f(m_o - m_new);
    l = l * a + l_o * bsc;
#pragma unroll
    for (int i = 0; i < 24; ++i) {
      const float other = __shfl_xor_sync(0xffffffffu, acc[i], o);
      acc[i] = acc[i] * a + other * bsc;
    }
    m = m_new;
  }
  __shared__ float sm_m[4], sm_l[4], sm_acc[4][DEC_D];
  if (g == 0) {
    if (s == 0) { sm_m[warp] = m; sm_l[warp] = l; }
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int e = 0; e < 8; ++e) sm_acc[warp][(s + 4 * i) * 8 + e] = acc[8 * i + e];
  }
  __syncthreads();
  if (tid < DEC_D) {
    float M = fmaxf(fmaxf(sm_m[0], sm_m[1]), fmaxf(sm_m[2], sm_m[3]));
    float L = 0.f, A = 0.f;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
      const float sc = (sm_m[w] == -INFINITY) ? 0.f : exp2f(sm_m[w] - M);
      L += sm_l[w] * sc;
      A += sm_acc[w][tid] * sc;
    }
    ws_acc[part * DEC_D + tid] = A;
    if (tid == 0) { ws_m[part] = M; ws_l[part] = L; }
  }
}

__global__ void __launch_bounds__(DEC_D)
decode_combine_kernel(const float* __restrict__ ws_m, const float* __restrict__ ws_l, const float* __restrict__ ws_acc,
                      int H, int n_splits, __nv_bfloat16* __restrict__ out) {
  const int h = blockIdx.x, b = blockIdx.y, d = threadIdx.x;
  pdl_wait();
  pdl_trigger();
  const size_t base = ((size_t)b * H + h) * n_splits;
  float M = -INFINITY;
  for (int s = 0; s < n_splits; ++s) M = fmaxf(M, ws_m[base + s]);
  float L = 0.f, A = 0.f;
  for (int s = 0; s < n_splits; ++s) {
    const float ms = ws_m[base + s];
    if (ms == -INFINITY) continue;
    const float sc = exp2f(ms - M);
    L += ws_l[base + s] * sc;
    A += ws_acc[(base + s) * DEC_D + d] * sc;
  }
  out[((size_t)b * H + h) * DEC_D + d] = __float2bfloat16(L > 0.f ? A / L : 0.f);
}

}  // namespace aki

using namespace aki;

extern "C" size_t aki_mma_decode_workspace_bytes(int B, int H, int D, int max_kv_len) {
  if (B <= 0 || H <= 0 || D != DEC_D || max_kv_len <= 0) return 0;
  const size_t splits = (max_kv_len + DEC_CHUNK - 1) / DEC_CHUNK;
  return (size_t)B * H * splits * (DEC_D + 2) * sizeof(float);
}

extern "C" int aki_mma_decode_masked(const void* q, const void* k_cache, const void* v_cache, int64_t cache_stride_b,
                                     int64_t cache_stride_h, const int32_t* kv_len, const int32_t* kv_start,
                                     const uint32_t* kv_valid_bits, int bits_pitch, int max_kv_len, int B, int H, int D,
                                     float scale, void* out, void* workspace, size_t workspace_bytes,
                                     aki_stream_t stream) {
  AKI_REQUIRE(q && k_cache && v_cache && kv_len && out && workspace, AKI_ERR_NULL);
  AKI_REQUIRE(B > 0 && H > 0 && max_kv_len > 0 && B <= 65535 && H <= 65535, AKI_ERR_BAD_SHAPE);
  AKI_REQUIRE(!kv_valid_bits || (long long)bits_pitch * 32 >= max_kv_len, AKI_ERR_BAD_SHAPE);
  AKI_REQUIRE(D == DEC_D, AKI_ERR_UNSUPPORTED);
  AKI_REQUIRE(cache_stride_b % 8 == 0 && cache_stride_h % 8 == 0, AKI_ERR_UNSUPPORTED);
  AKI_REQUIRE(aligned16(q) && aligned16(k_cache) && aligned16(v_cache) && aligned16(workspace), AKI_ERR_MISALIGNED);
  AKI_REQUIRE(workspace_bytes >= aki_mma_decode_workspace_bytes(B, H, D, max_kv_len), AKI_ERR_BAD_SHAPE);
  const int n_splits = (max_kv_len + DEC_CHUNK - 1) / DEC_CHUNK;
  float* ws_m = static_cast<float*>(workspace);
  float* ws_l = ws_m + (size_t)B * H * n_splits;
  float* ws_acc = ws_l + (size_t)B * H * n_splits;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const float scale_log2 = scale * 1.4426950408889634f;
  launch_pdl(decode_partial_kernel, dim3(n_splits, H, B), dim3(DEC_THREADS), 0, st,
             static_cast<const __nv_bfloat16*>(q), static_cast<const __nv_bfloat16*>(k_cache),
             static_cast<const __nv_bfloat16*>(v_cache), cache_stride_b, cache_stride_h, kv_len, kv_start, kv_valid_bits,
             bits_pitch, H, scale_log2, n_splits, ws_m, ws_l, ws_acc);
  int rc = check_launch();
  if (rc != AKI_OK) return rc;
  launch_pdl(decode_combine_kernel, dim3(H, B), dim3(DEC_D), 0, st, ws_m, ws_l, ws_acc, H, n_splits,
             static_cast<__nv_bfloat16*>(out));
  return check_launch();
}

extern "C" int aki_mma_decode(const void* q, const void* k_cache, const void* v_cache, int64_t cache_stride_b,
                              int64_t cache_stride_h, const int32_t* kv_len, const int32_t* kv_start, int max_kv_len,
                              int B, int H, int D, float scale, void* out, void* workspace, size_t workspace_bytes,
                              aki_stream_t stream) {
  return aki_mma_decode_masked(q, k_cache, v_cache, cache_stride_b, cache_stride_h, kv_len, kv_start, nullptr, 0,
                               max_kv_len, B, H, D, scale, out, workspace, workspace_bytes, stream);
}
