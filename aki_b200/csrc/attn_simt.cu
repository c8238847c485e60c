// Verification kernels + backward pre/post-processing.
//   * aki_mma_attn_fwd_simt / aki_mma_attn_bwd_simt: the maths of Phi3Attention's eager core
//     (softmax_fp32(QK^T*scale + mask) V, installed equivalent models/phi3/modeling_phi3.py:153-175) and its
//     gradient as straightforward SIMT CUDA, fp32 throughout, no tensor cores.  TESTS ONLY: they cross-check
//     the tcgen05 kernels on-device at sizes the CPU oracle cannot reach.  Not a product path.
//   * bwd_preprocess / dq_finalize: small HBM-bound kernels used by the product backward.
#include <math.h>
#include <stdint.h>
#include "attn_aux.cuh"

namespace aki {

__device__ __forceinline__ float bf(const __nv_bfloat16 x) { return __bfloat162float(x); }
__device__ __forceinline__ float round_bf(float x) { return __bfloat162float(__float2bfloat16(x)); }

__device__ __forceinline__ float block_reduce(float v, float* red, bool is_max) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    float n = __shfl_xor_sync(0xffffffffu, v, o);
    v = is_max ? fmaxf(v, n) : v + n;
  }
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float r = red[0];
  for (int w = 1; w < nw; ++w) r = is_max ? fmaxf(r, red[w]) : r + red[w];
  __syncthreads();
  return r;
}

// ------------------------------------------------------------------------------------------------ forward
__global__ void __launch_bounds__(128)
attn_fwd_simt_kernel(TensorView q, TensorView k, TensorView v, TensorView o, float* __restrict__ lse,
                     const float* __restrict__ rope_cos, const float* __restrict__ rope_sin, int64_t rope_stride_b,
                     MaskMeta mm, int T, int q_off, int H, float scale) {
  extern __shared__ float sc[];  // q_off + T scores
  __shared__ float qs[96], red[4];
  // i: query row of q / o / lse / the RoPE tables; ia: its row in key (mask) coordinates
  const int i = blockIdx.x, ia = q_off + i, h = blockIdx.y, b = blockIdx.z, tid = threadIdx.x;
  const int len = meta_len(mm, b, q_off + T);
  __nv_bfloat16* orow = o.row(b, i, h);
  if (tid < 96) {
    float x = bf(q.row(b, i, h)[tid]);
    if (rope_cos) {
      const int d = tid % 48;
      const float c = rope_cos[(size_t)b * rope_stride_b + (size_t)i * 48 + d];
      const float s = rope_sin[(size_t)b * rope_stride_b + (size_t)i * 48 + d];
      const float other = bf(q.row(b, i, h)[tid < 48 ? tid + 48 : tid - 48]);
      x = (tid < 48) ? x * c - other * s : x * c + other * s;
      x = round_bf(x);  // the tensor-core path keeps rotated Q in bf16
    }
    qs[tid] = x;
  }
  __syncthreads();
  const int row_end = (ia < len) ? mma_row_end(mm, b, ia, len) : 0;
  float mx = -INFINITY;
  for (int j = tid; j < row_end; j += 128) {
    float s = -INFINITY;
    if (mma_allowed(mm, b, ia, j, len)) {
      const __nv_bfloat16* kr = k.row(b, j, h);
      float acc = 0.f;
#pragma unroll 8
      for (int d = 0; d < 96; ++d) acc = fmaf(qs[d], bf(kr[d]), acc);
      s = acc * scale;
    }
    sc[j] = s;
    mx = fmaxf(mx, s);
  }
  mx = block_reduce(mx, red, true);
  if (mx == -INFINITY) {  // no visible key: zeros (see DESIGN.md, fully masked rows)
    if (tid < 96) orow[tid] = __float2bfloat16(0.f);
    if (lse && tid == 0) lse[((size_t)b * H + h) * T + i] = INFINITY;
    return;
  }
  float sum = 0.f;
  for (int j = tid; j < row_end; j += 128) {
    const float p = __expf(sc[j] - mx);
    sc[j] = p;
    sum += p;
  }
  sum = block_reduce(sum, red, false);
  if (tid < 96) {
    float acc = 0.f;
    for (int j = 0; j < row_end; ++j) acc = fmaf(sc[j], bf(v.row(b, j, h)[tid]), acc);
    orow[tid] = __float2bfloat16(acc / sum);
  }
  if (lse && tid == 0) lse[((size_t)b * H + h) * T + i] = mx + logf(sum);
}

// ------------------------------------------------------------------------------------------------ preprocess
// Per (b,t,h) row: delta = sum_d O*dO ; q_rot = RoPE(q) (plain copy without tables) ; and the two [8] bf16
// row-statistics operand of the tcgen05 backward: [-LSE/scale x3, 0, -delta x3, 0], each value split into
// hi + mid + lo bf16 terms (rows that see nothing, and the padding rows t in [T, t_pad), get -1e30 / 0 so that
// their P^T is exactly 0).  HBM-bound: 6 lanes per row (lane l owns the 16-byte chunks l and l+6, i.e. the RoPE
// pair d <-> d+48), 5 rows per warp, every access a 16-byte vector.
__device__ __forceinline__ void split3_bf16(float v, __nv_bfloat16& a0, __nv_bfloat16& a1, __nv_bfloat16& a2) {
  a0 = __float2bfloat16(v);
  const float r1 = v - __bfloat162float(a0);
  a1 = __float2bfloat16(r1);
  a2 = __float2bfloat16(r1 - __bfloat162float(a1));
}

__global__ void __launch_bounds__(128)
bwd_preprocess_kernel(TensorView q, TensorView o, TensorView d_o, const float* __restrict__ lse,
                      const float* __restrict__ rope_cos, const float* __restrict__ rope_sin, int64_t rope_stride_b,
                      int B, int T, int t_pad, int H, float inv_scale, __nv_bfloat16* __restrict__ q_rot,
                      float* __restrict__ delta, __nv_bfloat16* __restrict__ row_stats) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane / 6, l = lane - 6 * g;
  const long long n_rows = (long long)B * t_pad * H;
  const long long row = ((long long)blockIdx.x * 4 + warp) * 5 + g;
  const bool active = (lane < 30) && (row < n_rows);
  int h = 0, t = 0, b = 0;
  if (active) {
    h = (int)(row % H);
    const long long bt = row / H;
    t = (int)(bt % t_pad);
    b = (int)(bt / t_pad);
  }
  const bool live = active && (t < T);
  float part = 0.f;
  if (live) {
    const uint4 q_lo = *reinterpret_cast<const uint4*>(q.row(b, t, h) + 8 * l);
    const uint4 q_hi = *reinterpret_cast<const uint4*>(q.row(b, t, h) + 48 + 8 * l);
    const uint4 o_lo = *reinterpret_cast<const uint4*>(o.row(b, t, h) + 8 * l);
    const uint4 o_hi = *reinterpret_cast<const uint4*>(o.row(b, t, h) + 48 + 8 * l);
    const uint4 g_lo = *reinterpret_cast<const uint4*>(d_o.row(b, t, h) + 8 * l);
    const uint4 g_hi = *reinterpret_cast<const uint4*>(d_o.row(b, t, h) + 48 + 8 * l);
    const __nv_bfloat162* ol = reinterpret_cast<const __nv_bfloat162*>(&o_lo);
    const __nv_bfloat162* oh = reinterpret_cast<const __nv_bfloat162*>(&o_hi);
    const __nv_bfloat162* gl = reinterpret_cast<const __nv_bfloat162*>(&g_lo);
    const __nv_bfloat162* gh = reinterpret_cast<const __nv_bfloat162*>(&g_hi);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 a = __bfloat1622float2(ol[e]), c = __bfloat1622float2(gl[e]);
      const float2 d = __bfloat1622float2(oh[e]), f = __bfloat1622float2(gh[e]);
      part = fmaf(a.x, c.x, part); part = fmaf(a.y, c.y, part);
      part = fmaf(d.x, f.x, part); part = fmaf(d.y, f.y, part);
    }
    uint4 r_lo = q_lo, r_hi = q_hi;
    if (rope_cos) {
      float cs[8], sn[8];
      const float* cr = rope_cos + (size_t)b * rope_stride_b + (size_t)t * 48 + 8 * l;
      const float* sr = rope_sin + (size_t)b * rope_stride_b + (size_t)t * 48 + 8 * l;
      *reinterpret_cast<float4*>(cs) = __ldg(reinterpret_cast<const float4*>(cr));
      *reinterpret_cast<float4*>(cs + 4) = __ldg(reinterpret_cast<const float4*>(cr + 4));
      *reinterpret_cast<float4*>(sn) = __ldg(reinterpret_cast<const float4*>(sr));
      *reinterpret_cast<float4*>(sn + 4) = __ldg(reinterpret_cast<const float4*>(sr + 4));
      const __nv_bfloat162* ql = reinterpret_cast<const __nv_bfloat162*>(&q_lo);
      const __nv_bfloat162* qh = reinterpret_cast<const __nv_bfloat162*>(&q_hi);
      __nv_bfloat162* rl = reinterpret_cast<__nv_bfloat162*>(&r_lo);
      __nv_bfloat162* rh = reinterpret_cast<__nv_bfloat162*>(&r_hi);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 lo = __bfloat1622float2(ql[e]), hi = __bfloat1622float2(qh[e]);
        rl[e] = __floats2bfloat162_rn(lo.x * cs[2 * e] - hi.x * sn[2 * e], lo.y * cs[2 * e + 1] - hi.y * sn[2 * e + 1]);
        rh[e] = __floats2bfloat162_rn(hi.x * cs[2 * e] + lo.x * sn[2 * e], hi.y * cs[2 * e + 1] + lo.y * sn[2 * e + 1]);
      }
    }
    __nv_bfloat16* dst = q_rot + (((size_t)b * H + h) * T + t) * 96;
    *reinterpret_cast<uint4*>(dst + 8 * l) = r_lo;
    *reinterpret_cast<uint4*>(dst + 48 + 8 * l) = r_hi;
  }
  // delta: sum of the 6 lane partials of the row (every lane of the warp takes part in the shuffles)
  float dl = 0.f;
#pragma unroll
  for (int k = 0; k < 6; ++k) dl += __shfl_sync(0xffffffffu, part, min(6 * g + k, 31));
  if (active && l == 0) {
    __nv_bfloat16 st[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) st[e] = __float2bfloat16(0.f);
    float v = -1e30f;
    if (live) {
      const size_t idx = ((size_t)b * H + h) * T + t;
      delta[idx] = dl;
      const float L = lse[idx];
      if (L < 3.0e38f) {
        v = -L * inv_scale;
        split3_bf16(v, st[0], st[1], st[2]);
      } else {
        st[0] = __float2bfloat16(v);
      }
      split3_bf16(-dl, st[4], st[5], st[6]);
    } else {
      st[0] = __float2bfloat16(v);
    }
    *reinterpret_cast<uint4*>(row_stats + (((size_t)b * H + h) * t_pad + t) * 8) = *reinterpret_cast<const uint4*>(st);
  }
}

// dq_accum (B,H,T,D) fp32 -> inverse RoPE -> bf16 strided d_q.   g = R^T g' :  lo = lo'*c + hi'*s ; hi = hi'*c - lo'*s
__global__ void __launch_bounds__(128)
dq_finalize_kernel(const float* __restrict__ dq_accum, TensorView d_q, const float* __restrict__ rope_cos,
                   const float* __restrict__ rope_sin, int64_t rope_stride_b, int T, int H, float scale) {
  const int t = blockIdx.x, b = blockIdx.y;
  for (int idx = threadIdx.x; idx < H * 48; idx += 128) {
    const int h = idx / 48, d = idx - h * 48;
    const float* src = dq_accum + (((size_t)b * H + h) * T + t) * 96;
    float lo = src[d] * scale, hi = src[d + 48] * scale;
    if (rope_cos) {
      const float c = rope_cos[(size_t)b * rope_stride_b + (size_t)t * 48 + d];
      const float s = rope_sin[(size_t)b * rope_stride_b + (size_t)t * 48 + d];
      const float lo2 = lo * c + hi * s, hi2 = hi * c - lo * s;
      lo = lo2; hi = hi2;
    }
    __nv_bfloat16* dst = d_q.row(b, t, h);
    dst[d] = __float2bfloat16(lo);
    dst[d + 48] = __float2bfloat16(hi);
  }
}

// ------------------------------------------------------------------------------------------------ backward (SIMT)
// one CTA per query row: dQ
__global__ void __launch_bounds__(128)
attn_bwd_simt_dq_kernel(const __nv_bfloat16* __restrict__ q_rot, TensorView k, TensorView v, TensorView d_o,
                        const float* __restrict__ lse, const float* __restrict__ delta, float* __restrict__ dq_accum,
                        MaskMeta mm, int T, int H, float scale) {
  extern __shared__ float sc[];
  __shared__ float qs[96], dos[96];
  const int i = blockIdx.x, h = blockIdx.y, b = blockIdx.z, tid = threadIdx.x;
  const int len = meta_len(mm, b, T);
  const size_t bh = (size_t)b * H + h;
  float* dst = dq_accum + (bh * T + i) * 96;
  const int row_end = (i < len) ? mma_row_end(mm, b, i, len) : 0;
  if (tid < 96) {
    qs[tid] = bf(q_rot[(bh * T + i) * 96 + tid]);
    dos[tid] = bf(d_o.row(b, i, h)[tid]);
  }
  __syncthreads();
  const float L = lse[bh * T + i], dl = delta[bh * T + i];
  for (int j = tid; j < row_end; j += 128) {
    float ds = 0.f;
    if (mma_allowed(mm, b, i, j, len)) {
      const __nv_bfloat16* kr = k.row(b, j, h);
      const __nv_bfloat16* vr = v.row(b, j, h);
      float s = 0.f, dp = 0.f;
#pragma unroll 8
      for (int d = 0; d < 96; ++d) {
        s = fmaf(qs[d], bf(kr[d]), s);
        dp = fmaf(dos[d], bf(vr[d]), dp);
      }
      const float p = __expf(s * scale - L);
      ds = p * (dp - dl) * scale;
    }
    sc[j] = ds;
  }
  __syncthreads();
  if (tid < 96) {
    float acc = 0.f;
    for (int j = 0; j < row_end; ++j) acc = fmaf(sc[j], bf(k.row(b, j, h)[tid]), acc);
    dst[tid] = acc;
  }
}

// one CTA per key: dK (w.r.t. pre-RoPE k when tables are given) and dV
__global__ void __launch_bounds__(128)
attn_bwd_simt_dkv_kernel(const __nv_bfloat16* __restrict__ q_rot, TensorView k, TensorView v, TensorView d_o,
                         const float* __restrict__ lse, const float* __restrict__ delta, TensorView d_k, TensorView d_v,
                         const float* __restrict__ rope_cos, const float* __restrict__ rope_sin, int64_t rope_stride_b,
                         MaskMeta mm, int T, int H, float scale) {
  extern __shared__ float sm[];  // [T] p, [T] ds
  float* sp = sm;
  float* sds = sm + T;
  __shared__ float ks[96], vs[96], dks[96];
  const int j = blockIdx.x, h = blockIdx.y, b = blockIdx.z, tid = threadIdx.x;
  const int len = meta_len(mm, b, T);
  const size_t bh = (size_t)b * H + h;
  if (tid < 96) {
    ks[tid] = bf(k.row(b, j, h)[tid]);
    vs[tid] = bf(v.row(b, j, h)[tid]);
  }
  __syncthreads();
  for (int i = tid; i < len; i += 128) {
    float p = 0.f, ds = 0.f;
    if (mma_allowed(mm, b, i, j, len)) {
      const __nv_bfloat16* qr = q_rot + (bh * T + i) * 96;
      const __nv_bfloat16* dr = d_o.row(b, i, h);
      float s = 0.f, dp = 0.f;
#pragma unroll 8
      for (int d = 0; d < 96; ++d) {
        s = fmaf(bf(qr[d]), ks[d], s);
        dp = fmaf(bf(dr[d]), vs[d], dp);
      }
      p = __expf(s * scale - lse[bh * T + i]);
      ds = p * (dp - delta[bh * T + i]) * scale;
    }
    sp[i] = p;
    sds[i] = ds;
  }
  __syncthreads();
  if (tid < 96) {
    float dv = 0.f, dk = 0.f;
    for (int i = 0; i < len; ++i) {
      dv = fmaf(sp[i], bf(d_o.row(b, i, h)[tid]), dv);
      dk = fmaf(sds[i], bf(q_rot[(bh * T + i) * 96 + tid]), dk);
    }
    d_v.row(b, j, h)[tid] = __float2bfloat16(j < len ? dv : 0.f);
    dks[tid] = (j < len) ? dk : 0.f;
  }
  __syncthreads();
  if (tid < 48) {
    float lo = dks[tid], hi = dks[tid + 48];
    if (rope_cos) {
      const float c = rope_cos[(size_t)b * rope_stride_b + (size_t)j * 48 + tid];
      const float s = rope_sin[(size_t)b * rope_stride_b + (size_t)j * 48 + tid];
      const float lo2 = lo * c + hi * s, hi2 = hi * c - lo * s;
      lo = lo2; hi = hi2;
    }
    d_k.row(b, j, h)[tid] = __float2bfloat16(lo);
    d_k.row(b, j, h)[tid + 48] = __float2bfloat16(hi);
  }
}

int check_attn_params(const AkiMmaAttnParams& p) {
  if (p.B <= 0 || p.H <= 0 || p.T <= 0 || p.B > 65535 || p.H > 65535) return AKI_ERR_BAD_SHAPE;
  if (p.q_offset < 0 || (int64_t)p.q_offset + p.T > INT32_MAX) return AKI_ERR_BAD_SHAPE;
  const int64_t n_keys = (int64_t)p.q_offset + p.T;
  if (p.D != AKI_MMA_HEAD_DIM) return AKI_ERR_UNSUPPORTED;
  int rc;
  if ((rc = check_tensor(p.q)) || (rc = check_tensor(p.k)) || (rc = check_tensor(p.v)) || (rc = check_tensor(p.o)))
    return rc;
  if ((p.rope_cos == nullptr) != (p.rope_sin == nullptr)) return AKI_ERR_NULL;
  if (p.rope_cos && (!aligned16(p.rope_cos) || !aligned16(p.rope_sin))) return AKI_ERR_MISALIGNED;
  if ((p.row_lo == nullptr) != (p.row_hi == nullptr)) return AKI_ERR_NULL;
  if (p.row_lo && p.meta_pitch < n_keys) return AKI_ERR_BAD_SHAPE;
  if ((p.kv_valid_bits || p.kv_mutual_bits) && (int64_t)p.bits_pitch * 32 < n_keys) return AKI_ERR_BAD_SHAPE;
  return AKI_OK;
}

int launch_bwd_preprocess(const AkiMmaAttnBwdParams& p, const BwdWorkspace& w, cudaStream_t st) {
  const AkiMmaAttnParams& f = p.fwd;
  const long long n_rows = (long long)f.B * w.t_pad * f.H;
  const long long blocks = (n_rows + 19) / 20;
  if (blocks <= 0 || blocks >= (1ll << 31)) return AKI_ERR_BAD_SHAPE;
  bwd_preprocess_kernel<<<(unsigned)blocks, 128, 0, st>>>(view_of(f.q), view_of(f.o), view_of(p.d_o), f.lse, f.rope_cos,
                                                           f.rope_sin, f.rope_stride_b, f.B, f.T, w.t_pad, f.H,
                                                           1.0f / f.scale, w.q_rot, w.delta, w.row_stats);
  return check_launch();
}

int launch_dq_finalize(const AkiMmaAttnBwdParams& p, const BwdWorkspace& w, float scale, cudaStream_t st) {
  const AkiMmaAttnParams& f = p.fwd;
  dq_finalize_kernel<<<dim3(f.T, f.B), 128, 0, st>>>(w.dq_accum, view_of(p.d_q), f.rope_cos, f.rope_sin,
                                                      f.rope_stride_b, f.T, f.H, scale);
  return check_launch();
}

}  // namespace aki

using namespace aki;

extern "C" size_t aki_mma_attn_bwd_workspace_bytes(int B, int H, int T, int D) {
  if (B <= 0 || H <= 0 || T <= 0 || D != AKI_MMA_HEAD_DIM) return 0;
  return carve_bwd_workspace(nullptr, B, H, T, D).bytes;
}

extern "C" int aki_mma_attn_fwd_simt(const AkiMmaAttnParams* p, aki_stream_t stream) {
  AKI_REQUIRE(p, AKI_ERR_NULL);
  int rc = check_attn_params(*p);
  if (rc) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const size_t smem = ((size_t)p->q_offset + p->T) * 4;
  if (smem > 48 * 1024) {
    if (cudaFuncSetAttribute(attn_fwd_simt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) !=
        cudaSuccess) {
      cudaGetLastError();
      return AKI_ERR_UNSUPPORTED;
    }
  }
  attn_fwd_simt_kernel<<<dim3(p->T, p->H, p->B), 128, smem, st>>>(view_of(p->q), view_of(p->k), view_of(p->v),
                                                                   view_of(p->o), p->lse, p->rope_cos, p->rope_sin,
                                                                   p->rope_stride_b, mask_meta_from(*p), p->T,
                                                                   p->q_offset, p->H, p->scale);
  return check_launch();
}

extern "C" int aki_mma_attn_bwd_simt(const AkiMmaAttnBwdParams* p, aki_stream_t stream) {
  AKI_REQUIRE(p, AKI_ERR_NULL);
  const AkiMmaAttnParams& f = p->fwd;
  AKI_REQUIRE(f.q_offset == 0, AKI_ERR_UNSUPPORTED);   // no backward for a continuation chunk
  int rc = check_attn_params(f);
  if (rc) return rc;
  if ((rc = check_tensor(p->d_o)) || (rc = check_tensor(p->d_q)) || (rc = check_tensor(p->d_k)) ||
      (rc = check_tensor(p->d_v)))
    return rc;
  AKI_REQUIRE(f.lse && p->workspace, AKI_ERR_NULL);
  AKI_REQUIRE(p->workspace_bytes >= aki_mma_attn_bwd_workspace_bytes(f.B, f.H, f.T, f.D), AKI_ERR_BAD_SHAPE);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  BwdWorkspace w = carve_bwd_workspace(p->workspace, f.B, f.H, f.T, f.D);
  if ((rc = launch_bwd_preprocess(*p, w, st))) return rc;
  const size_t smem1 = (size_t)f.T * 4, smem2 = (size_t)f.T * 8;
  if (smem2 > 48 * 1024) {
    if (cudaFuncSetAttribute(attn_bwd_simt_dq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1) !=
            cudaSuccess ||
        cudaFuncSetAttribute(attn_bwd_simt_dkv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2) !=
            cudaSuccess) {
      cudaGetLastError();
      return AKI_ERR_UNSUPPORTED;
    }
  }
  MaskMeta mm = mask_meta_from(f);
  attn_bwd_simt_dq_kernel<<<dim3(f.T, f.H, f.B), 128, smem1, st>>>(w.q_rot, view_of(f.k), view_of(f.v),
                                                                    view_of(p->d_o), f.lse, w.delta, w.dq_accum, mm, f.T,
                                                                    f.H, f.scale);
  if ((rc = check_launch())) return rc;
  attn_bwd_simt_dkv_kernel<<<dim3(f.T, f.H, f.B), 128, smem2, st>>>(w.q_rot, view_of(f.k), view_of(f.v),
                                                                     view_of(p->d_o), f.lse, w.delta, view_of(p->d_k),
                                                                     view_of(p->d_v), f.rope_cos, f.rope_sin,
                                                                     f.rope_stride_b, mm, f.T, f.H, f.scale);
  if ((rc = check_launch())) return rc;
  return launch_dq_finalize(*p, w, 1.0f, st);   // the SIMT kernels already folded scale into dS
}
