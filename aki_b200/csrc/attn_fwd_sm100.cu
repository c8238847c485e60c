// Modality-mutual attention forward for sm_100a: QK^T, online softmax and PV on tcgen05 tensor cores with
// TMEM accumulators, operands staged by TMA, mbarrier pipelines, warp-specialised roles, persistent CTAs fed by the
// hardware work queue (cluster launch control).
//
// Replaces the eager core of Phi3Attention.forward (softmax_fp32(QK^T/sqrt(96) + mask) V; installed
// equivalent transformers/models/phi3/modeling_phi3.py:153-175) fed by the reference's materialised
// (B,1,T,T) mask (codes/open_flamingo/src/vlm.py:410-443).  No mask is read from HBM: the predicate
//   allowed(i,j) = (j<=i & valid[j]) | (row_lo[i]<=j<row_hi[i] & mutual_ok[j])
// is evaluated in registers on the few key tiles that are not fully visible, and key tiles beyond a query tile's
// reach are never visited.  RoPE is applied to Q in shared memory right after the TMA load.
//
// WORK ITEM = one (batch, head) x one PAIR of query tiles from the forward plan (meta.cu, aki_mma_fwd_plan): query
// tiles of <= 128 rows that start at every image span, ranked by the number of 128-key tiles they visit and paired
// (both tiles of a pair consume one stream of K/V tiles).  Items are numbered heaviest-first inside groups of 32
// (batch, head) slices: the group size trades DRAM re-reads of K/V against L2 hot spots (many CTAs streaming the
// same K/V lines at the same moment) -- same box, T=8192, 4 images: groups of 16 / 32 / 64 -> 1.066 / 1.013 / 0.990 ms
// with 0.59 / 1.19 / 2.47 GB read from DRAM per launch (algorithmic: 0.3 GB);
// a CTA keeps asking the hardware queue for the next item
// (clusterlaunchcontrol.try_cancel) until the grid is exhausted.
//
// CTA = 16 warps:
//   warp 0       TMA producer: Q of the NEXT item while the current one runs (2 Q buffers), K ring (2 x 128 keys),
//                V ring (3 x 128 keys)
//   warp 1       scheduler: next item id from the hardware queue -> plan entry -> item ring (4 slots) in shared memory
//   warp 2 / 3   MMA issuer of query tile 0 / 1 (+ TMEM allocation): S_t = Q_t K_j^T (one N=128 group per 128 keys),
//                O_t += P_t V_j as two TS groups of 64 keys (P read from TMEM)
//   warps 4-7 / 8-11   softmax of tile 0 / 1: ONE THREAD PER SCORE ROW, 128 keys per pass -- no cross-warp exchange,
//                no block barrier in the loop: tcgen05.ld of the whole row, S buffer handed back at once (the next
//                QK^T runs under the exponentials), mask (only tiles that are not fully visible), row maximum, lazy
//                rescale of O (only when the maximum grew by more than 2^8; done in place by the same thread),
//                exp2 of keys 0-63 -> P -> PV, exp2 of keys 64-127 -> P -> PV.  Packed FFMA2 / FADD2 / FMNMX3.
//   warps 12-15  RoPE of the next item's Q tiles in shared memory, then the epilogue of the current item
//                (O / l -> bf16 -> global, LSE) while the softmax warps already run the next item
// TMEM columns: S0 [0,128) S1 [128,256) | O0 [256,352) O1 [352,448) | P0 [448,480) P1 [480,512) (64 keys of bf16 pairs).
// Shared memory: Q 2 buffers x 2 tiles x 24 KB; K ring 2 x 24 KB; V ring 3 x 24 KB.  Every tile is 3 SWIZZLE_64B atoms
// [128 rows][64 B] (head_dim 96 = 3 x 32), the layout both the TMA boxes and the UMMA descriptors use.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <mutex>
#include "attn_aux.cuh"
#include "sm100_ptx.cuh"

#ifndef AKI_FWD_POLY
#define AKI_FWD_POLY 0         // of every 4 score pairs, how many take the polynomial exp2 (FMA pipe) instead of MUFU.EX2
#endif                         // (same box, causal / 4 images: 0 -> 0.88 / 1.06 ms, 1 -> 0.87-0.99 / 1.04-1.19 depending on
                               // code placement, 2 -> 0.96 / 1.14, 3 -> 1.03 / 1.24: the softmax warps are bound by their
                               // own instruction stream, not by the MUFU pipe -- tools/mufu_bench.cu)


namespace aki {

namespace fwd {
constexpr int BM = 128, BN = 128, HD = 96;
constexpr int ATOM = 128 * 64, TILE_BYTES = 3 * ATOM;     // 24576
constexpr int K_STAGES = 2, V_STAGES = 3, SLOTS = 4;
constexpr int THREADS = 512;
constexpr int SMEM_Q = 0;                                  // [buffer][tile]
constexpr int SMEM_K = SMEM_Q + 4 * TILE_BYTES;
constexpr int SMEM_V = SMEM_K + K_STAGES * TILE_BYTES;
constexpr int SMEM_TOTAL = SMEM_V + V_STAGES * TILE_BYTES; // 221184
constexpr int SMEM_ALLOC = SMEM_TOTAL + 1024;              // slack for 1024-byte alignment
constexpr uint32_t TM_S = 0, TM_O = 256, TM_P = 448;       // S: 128 t; O: 96 t; P: 32 t
constexpr int REGS_CTRL = 56, REGS_SOFTMAX = 192, REGS_EPI = 72;   // 128*56 + 256*192 + 128*72 = 65536 = 512 x 128
constexpr float RESCALE_THRESHOLD = 8.0f;  // log2 units: P may grow to 2^8 before O is rescaled
#ifndef AKI_FWD_HEADS_PER_GROUP
#define AKI_FWD_HEADS_PER_GROUP 32
#endif
constexpr int HEADS_PER_GROUP = AKI_FWD_HEADS_PER_GROUP;
}  // namespace fwd

struct FwdKernelParams {
  TensorView q, o;
  float* lse;
  const float* rope_cos;
  const float* rope_sin;
  int64_t rope_stride_b;
  MaskMeta mm;
  const int4* plan;      // (B, 1 + plan_pairs) or nullptr
  int plan_pairs;
  int B, H, T;
  int q_off;             // queries are key rows [q_off, q_off + T) (AkiMmaAttnParams.q_offset)
  int ranks, group, n_items, use_clc;   // items: ((g * ranks + r) * group + slice)
  float scale_log2, scale;
  unsigned long long* trace;  // debug build (make TRACE=1, tools/fwd_trace.py): clock64 stamps of one CTA's first item
  int trace_cta;
};

#ifdef AKI_FWD_TRACE
#define TR(slot, j, k) do { if (tracing && (j) < 64) P.trace[((slot) * 64 + (j)) * 12 + (k)] = clock64(); } while (0)
#else
#define TR(slot, j, k) do { } while (0)
#endif

__device__ __forceinline__ uint32_t low_mask(int n) {  // n low bits set, n clamped to [0,32]
  return n <= 0 ? 0u : (n >= 32 ? 0xffffffffu : ((1u << n) - 1u));
}

// D[tmem] (+)= A[smem] * B[smem] with descriptors given as (low word, shared high word)
__device__ __forceinline__ void umma_ss_lh(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t desc_hi,
                                           uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 da, {%1, %3};\n\tmov.b64 db, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n\t}\n" ::"r"(d_tmem),
      "r"(a_lo), "r"(b_lo), "r"(desc_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_ts_lh(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_lo, uint32_t desc_hi,
                                           uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 db;\n\tsetp.ne.b32 p, %5, 0;\n\t"
      "mov.b64 db, {%2, %3};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], db, %4, p;\n\t}\n" ::"r"(d_tmem),
      "r"(a_tmem), "r"(b_lo), "r"(desc_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}

// exp2 of two scores on the FMA pipe (Cody-Waite split + degree-3 minimax polynomial, relative error 7.5e-5 -- far
// below the bf16 rounding of P): x = n + f with n = round(x) taken from the mantissa of x + 1.5*2^23, 2^f from the
// polynomial on [-0.5, 0.5], 2^n by adding n to the exponent field.  The MUFU unit (4 lanes per sub-partition) is the
// scarcest pipe of this kernel (16 384 exponentials per 128 x 128 tile = 1024 cycles against ~1000 of tensor time), so
// a share of the scores goes this way.  Inputs below -126 (masked scores are -inf) are clamped: they come out as
// 2^-126 ~ 1e-38 instead of 0, which vanishes against the row maximum's 2^0.
__device__ __forceinline__ void exp2_poly_x2(uint64_t a2, float& p0, float& p1) {
  float a0, a1;
  f32x2_unpack(a2, a0, a1);
  a0 = fmaxf(a0, -126.f); a1 = fmaxf(a1, -126.f);
  a2 = f32x2_pack(a0, a1);
  const uint64_t t2 = f32x2_add(a2, f32x2_pack(12582912.f, 12582912.f));
  const uint64_t n2 = f32x2_add(t2, f32x2_pack(-12582912.f, -12582912.f));
  const uint64_t f2 = f32x2_fma(n2, f32x2_pack(-1.f, -1.f), a2);
  uint64_t q = f32x2_fma(f2, f32x2_pack(0.0551716685f, 0.0551716685f), f32x2_pack(0.242611125f, 0.242611125f));
  q = f32x2_fma(q, f2, f32x2_pack(0.693260968f, 0.693260968f));
  q = f32x2_fma(q, f2, f32x2_pack(0.999928057f, 0.999928057f));
  float q0, q1, t0, t1;
  f32x2_unpack(q, q0, q1);
  f32x2_unpack(t2, t0, t1);
  p0 = __uint_as_float(__float_as_uint(q0) + (__float_as_uint(t0) << 23));
  p1 = __uint_as_float(__float_as_uint(q1) + (__float_as_uint(t1) << 23));
}

// Rare path of the online softmax: the running max grew by more than the threshold, this thread's row of O_t is
// rescaled by alpha.  Kept out of line so that the per-pass loop stays compact.
__device__ __noinline__ void rescale_o96(uint32_t tm_o, float alpha) {
#pragma unroll 1
  for (int c = 0; c < 6; ++c) {
    uint32_t o[16];
    tmem_ld_x16(tm_o + 16 * c, o);
    tmem_wait_ld();
#pragma unroll
    for (int x = 0; x < 16; ++x) o[x] = __float_as_uint(__uint_as_float(o[x]) * alpha);
    tmem_st_x16(tm_o + 16 * c, o);
  }
  tmem_wait_st();
}

template <bool ROPE>
__global__ void __launch_bounds__(fwd::THREADS, 1)
attn_fwd_sm100_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                      const __grid_constant__ CUtensorMap map_v, const FwdKernelParams P) {
  using namespace fwd;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  // barrier indices
  constexpr int Q_FULL = 0 /* [buf][tile] */, Q_READY = Q_FULL + 4 /* [buf] */, Q_EMPTY = Q_READY + 2 /* [buf] */,
                K_FULL = Q_EMPTY + 2, K_EMPTY = K_FULL + K_STAGES, V_FULL = K_EMPTY + K_STAGES,
                V_EMPTY = V_FULL + V_STAGES, S_FULL = V_EMPTY + V_STAGES /* [tile] */, S_FREE = S_FULL + 2,
                P_FULL = S_FREE + 2, PV_DONE = P_FULL + 2, O_DONE = PV_DONE + 2, O_FREE = O_DONE + 2,
                L_READY = O_FREE + 2, ITEM_FULL = L_READY + 2, ITEM_EMPTY = ITEM_FULL + SLOTS,
                CLC_BAR = ITEM_EMPTY + SLOTS, N_BARS = CLC_BAR + 1;
  __shared__ __align__(8) uint64_t bars[N_BARS];
  __shared__ __align__(16) int4 item_ring[SLOTS][3];   // {valid,b,h,len} {start0,start1,rows0,rows1} {nkv0,nkv1,nfull0,nfull1}
  __shared__ __align__(16) uint4 clc_resp;
  __shared__ float2 lm_s[2][128];                      // per tile, per row: (row sum, running max) of the finished item
  __shared__ uint32_t tmem_base_s;
  const uint32_t bar0 = smem_u32(bars);
  auto BAR = [&](int i) { return bar0 + 8u * i; };

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid == 0) {
    for (int i = 0; i < 4; ++i) mbar_init(BAR(Q_FULL + i), 1);
    for (int i = 0; i < 2; ++i) { mbar_init(BAR(Q_READY + i), 128); mbar_init(BAR(Q_EMPTY + i), 2); }
    for (int i = 0; i < K_STAGES; ++i) { mbar_init(BAR(K_FULL + i), 1); mbar_init(BAR(K_EMPTY + i), 2); }   // one release per query tile
    for (int i = 0; i < V_STAGES; ++i) { mbar_init(BAR(V_FULL + i), 1); mbar_init(BAR(V_EMPTY + i), 2); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(BAR(S_FULL + i), 1); mbar_init(BAR(S_FREE + i), 128);
      mbar_init(BAR(P_FULL + i), 128); mbar_init(BAR(PV_DONE + i), 1);
      mbar_init(BAR(O_DONE + i), 1); mbar_init(BAR(O_FREE + i), 128);
      mbar_init(BAR(L_READY + i), 128);
    }
    for (int i = 0; i < SLOTS; ++i) { mbar_init(BAR(ITEM_FULL + i), 1); mbar_init(BAR(ITEM_EMPTY + i), 15); }
    mbar_init(BAR(CLC_BAR), 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<512>(smem_u32(&tmem_base_s));
  if (warp == 0 && elect_one()) { tma_prefetch_desc(&map_q); tma_prefetch_desc(&map_k); tma_prefetch_desc(&map_v); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;

  // every role walks the same sequence of items through the ring; n = running item count of the caller
  auto item_wait = [&](uint32_t n, int4& v0, int4& v1, int4& v2) {
    const int slot = n % SLOTS;
    mbar_wait(BAR(ITEM_FULL + slot), (n / SLOTS) & 1);
    v0 = item_ring[slot][0]; v1 = item_ring[slot][1]; v2 = item_ring[slot][2];
  };

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    setmaxnreg_dec<REGS_CTRL>();
    if (elect_one()) {
      uint32_t n_it = 0, n_q = 0, kc = 0, vc = 0;
      bool q_end = false;
      auto issue_q = [&](uint32_t n, const int4& v0, const int4& v1, const int4& v2) {
        const int buf = n & 1;
        for (int t = 0; t < 2; ++t) {
          const uint32_t bar = BAR(Q_FULL + 2 * buf + t);
          if ((t ? v2.y : v2.x) > 0) {
            mbar_arrive_expect_tx(bar, TILE_BYTES);
            for (int a = 0; a < 3; ++a)
              tma_load_4d(smem_base + SMEM_Q + (2 * buf + t) * TILE_BYTES + a * ATOM, &map_q, bar, a * 32, t ? v1.y : v1.x, v0.z, v0.y);
          } else {
            mbar_arrive(bar);
          }
        }
      };
      for (;;) {
        int4 v0, v1, v2;
        item_wait(n_it, v0, v1, v2);
        if (!v0.x) break;
        if (n_q == n_it) {
          mbar_wait(BAR(Q_EMPTY + (n_q & 1)), ((n_q >> 1) & 1) ^ 1);
          issue_q(n_q, v0, v1, v2);
          ++n_q;
        }
        const int b = v0.y, h = v0.z, n_max = max(v2.x, v2.y);
        // Q of the next item as soon as its descriptor and its buffer are there (never blocks the K/V stream)
        auto try_next_q = [&]() {
          if (q_end || n_q != n_it + 1) return;
          const int slot = n_q % SLOTS;
          if (!mbar_test(BAR(ITEM_FULL + slot), (n_q / SLOTS) & 1)) return;
          const int4 w0 = item_ring[slot][0];
          if (!w0.x) { q_end = true; return; }
          if (!mbar_test(BAR(Q_EMPTY + (n_q & 1)), ((n_q >> 1) & 1) ^ 1)) return;
          issue_q(n_q, w0, item_ring[slot][1], item_ring[slot][2]);
          ++n_q;
        };
        auto load_k = [&](int j) {                 // 128 keys (rows beyond T are zero-filled)
          const uint32_t c = kc + j, s = c % K_STAGES;
          mbar_wait(BAR(K_EMPTY + s), ((c / K_STAGES) & 1) ^ 1);
          mbar_arrive_expect_tx(BAR(K_FULL + s), TILE_BYTES);
          for (int a = 0; a < 3; ++a)
            tma_load_4d(smem_base + SMEM_K + s * TILE_BYTES + a * ATOM, &map_k, BAR(K_FULL + s), a * 32, j * BN, h, b);
        };
        auto load_v = [&](int j) {
          const uint32_t c = vc + j, s = c % V_STAGES;
          mbar_wait(BAR(V_EMPTY + s), ((c / V_STAGES) & 1) ^ 1);
          mbar_arrive_expect_tx(BAR(V_FULL + s), TILE_BYTES);
          for (int a = 0; a < 3; ++a)
            tma_load_4d(smem_base + SMEM_V + s * TILE_BYTES + a * ATOM, &map_v, BAR(V_FULL + s), a * 32, j * BN, h, b);
        };
        // consumption order of the MMA warps: K0 | K1 V0 | K2 V1 | ...
        if (n_max > 0) load_k(0);
        for (int j = 0; j < n_max; ++j) {
          try_next_q();
          if (j + 1 < n_max) load_k(j + 1);
          load_v(j);
        }
        kc += n_max; vc += n_max;
        mbar_arrive(BAR(ITEM_EMPTY + n_it % SLOTS));
        ++n_it;
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ scheduler
    setmaxnreg_dec<REGS_CTRL>();
    if (lane == 0) {
      uint32_t n_pub = 0, n_clc = 0;
      long long id = blockIdx.x;
      const int n_keys = P.q_off + P.T, n_kt = (n_keys + BN - 1) / BN;
      auto publish = [&](const int4& v0, const int4& v1, const int4& v2) {
        const int slot = n_pub % SLOTS;
        mbar_wait(BAR(ITEM_EMPTY + slot), ((n_pub / SLOTS) & 1) ^ 1);
        item_ring[slot][0] = v0; item_ring[slot][1] = v1; item_ring[slot][2] = v2;
        mbar_arrive(BAR(ITEM_FULL + slot));
        ++n_pub;
      };
      for (;;) {
        // item id -> (group of slices, rank inside the plan, slice)
        const int per_group = P.ranks * P.group;
        const int g = (int)(id / per_group), rem = (int)(id % per_group);
        const int r = rem / P.group, bh = g * P.group + rem % P.group;
        if (bh < P.B * P.H) {
          const int b = bh / P.H, h = bh % P.H;
          const int len = meta_len(P.mm, b, n_keys);
          int4 e = make_int4(0, 0, 0, 0);
          int first_bad = 0;
          bool ok = false;
          if (P.plan) {
            const int4* row = P.plan + (size_t)b * (1 + P.plan_pairs);
            const int4 hdr = __ldg(row);
            if (r < hdr.x) { e = __ldg(row + 1 + r); first_bad = hdr.y; ok = true; }
          } else {
            // no plan: aligned tiles (2p, 2p+1) of the query rows, heaviest pair first
            const int n_qt = (P.T + BM - 1) / BM, p = P.ranks - 1 - r;
            if (p >= 0 && 2 * p < n_qt) {
              ok = true;
              for (int t = 0; t < 2; ++t) {
                const int qt = 2 * p + t;
                int nk = 0, rows = 0;
                if (qt < n_qt) {
                  rows = min(BM, P.T - qt * BM);
                  nk = min(P.mm.q_tile_kv_end ? __ldg(P.mm.q_tile_kv_end + (size_t)b * n_qt + qt)
                                              : (P.q_off + qt * BM + rows + BN - 1) / BN, n_kt);
                }
                if (t == 0) { e.x = qt * BM; e.z = nk | (rows << 16); }
                else { e.y = (qt < n_qt) ? qt * BM : 0; e.w = nk | (rows << 16); }
              }
              // without a plan nobody scanned the key bit-vectors: every tile is evaluated against the predicate
              first_bad = (P.mm.seq_len || P.mm.vbits) ? 0 : n_keys / BN;
            }
          }
          if (ok) {
            const int nk0 = e.z & 0xffff, nk1 = e.w & 0xffff;
            publish(make_int4(1, b, h, len), make_int4(e.x, e.y, e.z >> 16, e.w >> 16),
                    make_int4(nk0, nk1, min(first_bad, (P.q_off + e.x + 1) / BN), min(first_bad, (P.q_off + e.y + 1) / BN)));
          }
        }
        if (!P.use_clc) {
          id += gridDim.x;
          if (id >= P.n_items) break;
          continue;
        }
        mbar_arrive_expect_tx(BAR(CLC_BAR), 16);
        clc_try_cancel(smem_u32(&clc_resp), BAR(CLC_BAR));
        mbar_wait(BAR(CLC_BAR), n_clc & 1);
        ++n_clc;
        uint32_t next;
        const bool got = clc_query(smem_u32(&clc_resp), next);
        fence_proxy_async_smem();     // the response buffer is rewritten by the next (async-proxy) query
        if (!got) break;
        id = next;
      }
      publish(make_int4(0, 0, 0, 0), make_int4(0, 0, 0, 0), make_int4(0, 0, 0, 0));
    }
  } else if (warp == 2 || warp == 3) {
    // ------------------------------------------------------------------ MMA issuer of query tile t
    // Per pass j of this tile: QK^T(j+1) as soon as the softmax has taken S(j) out of TMEM, then PV(j) in two halves
    // as the softmax publishes them -- the program order of the softmax threads, so plain blocking waits suffice.
    // K / V stages and the Q buffer are released by one arrival per query tile: a commit behind the MMAs that read
    // them, or a plain arrive when this tile does not visit those keys.
    setmaxnreg_dec<REGS_CTRL>();
    const int t = warp - 2;
    if (elect_one()) {
      constexpr uint32_t IDESC_QK = umma_idesc_bf16(BM, BN, 0, 0), IDESC_PV = umma_idesc_bf16(BM, HD, 0, 1);
      const uint64_t DESC_KMAJ = umma_smem_desc(0, 16, 512, UMMA_SW64);
      const uint64_t DESC_V = umma_smem_desc(0, ATOM, 512, UMMA_SW64);     // MN-major: LBO = atom stride
      const uint32_t HI_K = (uint32_t)(DESC_KMAJ >> 32), KMAJ_LO = (uint32_t)DESC_KMAJ;
      const uint32_t HI_V = (uint32_t)(DESC_V >> 32), v_lo = (uint32_t)DESC_V + ((smem_base + SMEM_V) >> 4);
      const uint32_t k_lo = KMAJ_LO + ((smem_base + SMEM_K) >> 4);
      const uint32_t d_s = tmem + TM_S + 128 * t, d_o = tmem + TM_O + 96 * t, a_p = tmem + TM_P + 32 * t;
      uint32_t n_it = 0, kc = 0, vc = 0, n_qk = 0, n_ph = 0;
      for (;;) {
        int4 v0, v1, v2;
        item_wait(n_it, v0, v1, v2);
        if (!v0.x) break;
        const int nk = t ? v2.y : v2.x, n_max = max(v2.x, v2.y), buf = n_it & 1;

        const uint32_t qa = KMAJ_LO + ((smem_base + SMEM_Q + (2 * buf + t) * TILE_BYTES) >> 4);
#ifdef AKI_FWD_TRACE
        const bool tracing = P.trace && (int)blockIdx.x == P.trace_cta && n_it == 0;
#endif
        // Every barrier this warp ever waits on is waited on for EVERY item, whether or not its tile exists in the item:
        // a wait that is skipped for one phase lets the warp arrive at the next one a whole phase early, and a parity
        // wait cannot tell "phase p+1 complete" from "phase p not yet complete" (found by tools/stress.py: with RoPE the
        // epilogue warps lag by the rotation of the next item's Q, this warp skipped O_FREE on an item without its tile
        // and overwrote an O accumulator that was still being read).
        mbar_wait(ROPE ? BAR(Q_READY + buf) : BAR(Q_FULL + 2 * buf + t), (n_it >> 1) & 1);
        if (nk == 0) {
          // this tile does not exist in the item: release the Q buffer (the wait above also guarantees that the producer
          // has armed it for THIS item, so this warp cannot complete a Q_EMPTY phase with two arrivals of its own while
          // the other tile still reads Q)
          mbar_arrive(BAR(Q_EMPTY + buf));
        }
        auto handle_k = [&](int j) {
          const uint32_t c = kc + j, s = c % K_STAGES;
          // waited for even when this tile skips the keys: it keeps the tile from running a whole ring ahead and
          // arriving twice in one K_EMPTY phase
          mbar_wait(BAR(K_FULL + s), (c / K_STAGES) & 1);
          if (j < nk) {
            TR(2 + t, j, 0);
            if (n_qk > 0) mbar_wait(BAR(S_FREE + t), (n_qk - 1) & 1);   // the softmax holds the previous S in registers
            tc_fence_after();
            TR(2 + t, j, 1);
            const uint32_t ka = k_lo + s * (TILE_BYTES >> 4);
#pragma unroll
            for (int k = 0; k < 6; ++k)
              umma_ss_lh(d_s, qa + (((k >> 1) * ATOM + (k & 1) * 32) >> 4), ka + (((k >> 1) * ATOM + (k & 1) * 32) >> 4), HI_K,
                         IDESC_QK, k > 0);
            umma_commit(BAR(S_FULL + t));
            umma_commit(BAR(K_EMPTY + s));
            if (j == nk - 1) umma_commit(BAR(Q_EMPTY + buf));
            ++n_qk;
          } else {
            mbar_arrive(BAR(K_EMPTY + s));
          }
        };
        if (n_max > 0) handle_k(0);
        for (int j = 0; j < n_max; ++j) {
          if (j + 1 < n_max) handle_k(j + 1);
          const uint32_t c = vc + j, s = c % V_STAGES;
          mbar_wait(BAR(V_FULL + s), (c / V_STAGES) & 1);
          if (j < nk) {
            if (j == 0 && n_it > 0) mbar_wait(BAR(O_FREE + t), (n_it - 1) & 1);   // the epilogue has read the previous O_t
            const uint32_t va = v_lo + s * (TILE_BYTES >> 4);
#pragma unroll
            for (int half = 0; half < 2; ++half) {
              TR(2 + t, j, 2 + 2 * half);
              mbar_wait(BAR(P_FULL + t), n_ph & 1);
              ++n_ph;
              tc_fence_after();
              TR(2 + t, j, 3 + 2 * half);
#pragma unroll
              for (int k = 0; k < 4; ++k)
                umma_ts_lh(d_o, a_p + 8 * k, va + (4 * half + k) * 64, HI_V, IDESC_PV, (j > 0 || half > 0 || k > 0));
              umma_commit(BAR(PV_DONE + t));
            }
            umma_commit(BAR(V_EMPTY + s));
            if (j == nk - 1) umma_commit(BAR(O_DONE + t));
          } else {
            mbar_arrive(BAR(V_EMPTY + s));
          }
        }
        if (nk == 0 && n_it > 0) mbar_wait(BAR(O_FREE + t), (n_it - 1) & 1);   // observed every item (see above)
        kc += n_max; vc += n_max;
        mbar_arrive(BAR(ITEM_EMPTY + n_it % SLOTS));
        ++n_it;
      }
    }
  } else if (warp < 12) {
    // ------------------------------------------------------------------ softmax: one thread per score row
    setmaxnreg_inc<REGS_SOFTMAX>();
    const int t = (warp - 4) >> 2, g = warp & 3;
    const int r = 32 * g + lane;                  // row within the tile == TMEM lane
    const uint32_t lane_base = (uint32_t)(g * 32) << 16;
    const uint32_t tm_s = tmem + TM_S + 128 * t + lane_base;
    const uint32_t tm_o = tmem + TM_O + 96 * t + lane_base;
    const uint32_t tm_p = tmem + TM_P + 32 * t + lane_base;
    uint32_t n_it = 0, n_s = 0, n_pvh = 0;
    for (;;) {
      int4 v0, v1, v2;
      item_wait(n_it, v0, v1, v2);
      __syncwarp();
      if (lane == 0) mbar_arrive(BAR(ITEM_EMPTY + n_it % SLOTS));
      if (!v0.x) break;
      const int b = v0.y, len = v0.w;
      const int nk = t ? v2.y : v2.x, n_full = t ? v2.w : v2.z;
      const int i = P.q_off + (t ? v1.y : v1.x) + r;   // query index in mask (key) coordinates
      const bool row_live = (i < len);
      int row_lo = 0, row_hi = 0;
      if (row_live && P.mm.row_lo && nk > 0) {
        row_lo = __ldg(P.mm.row_lo + (size_t)b * P.mm.meta_pitch + i);
        row_hi = __ldg(P.mm.row_hi + (size_t)b * P.mm.meta_pitch + i);
      }
      float m_used = -INFINITY;  // running max (raw score units) the accumulators are expressed against
      float l = 0.f;             // row sum
#ifdef AKI_FWD_TRACE
      const bool tracing = P.trace && (int)blockIdx.x == P.trace_cta && n_it == 0 && r == 0;
#endif
      for (int j = 0; j < nk; ++j) {
        TR(t, j, 0);
        const bool partial = (j >= n_full);            // warp-uniform (CTA-uniform)
        uint32_t vw[4] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
        uint32_t mw[4] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
        if (partial) {                                 // one 32-bit word of each bit-vector covers 32 keys
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            const int wi = 4 * j + w;
            if (P.mm.vbits) vw[w] = (wi < P.mm.bits_pitch) ? __ldg(P.mm.vbits + (size_t)b * P.mm.bits_pitch + wi) : 0u;
            if (P.mm.mbits) mw[w] = (wi < P.mm.bits_pitch) ? __ldg(P.mm.mbits + (size_t)b * P.mm.bits_pitch + wi) : 0u;
          }
        }
        float s[128];
        mbar_wait(BAR(S_FULL + t), n_s & 1);
        ++n_s;
        tc_fence_after();
        TR(t, j, 1);
        tmem_ld_x32(tm_s, reinterpret_cast<uint32_t*>(s));
        tmem_ld_x32(tm_s + 32, reinterpret_cast<uint32_t*>(s) + 32);
        tmem_ld_x32(tm_s + 64, reinterpret_cast<uint32_t*>(s) + 64);
        tmem_ld_x32(tm_s + 96, reinterpret_cast<uint32_t*>(s) + 96);
        tmem_wait_ld();
        tc_fence_before();
        mbar_arrive(BAR(S_FREE + t));                  // QK^T of the next pass runs under the exponentials
        TR(t, j, 2);
        if (partial) {
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            const int col0 = j * BN + 32 * w;
            const int d = row_live ? (i - col0) : -1;             // causal: column c visible iff c <= d
            const int a = row_lo - col0, e = row_hi - col0;       // mutual: a <= c < e
            const uint32_t in_len = low_mask(len - col0);
            const uint32_t causal = low_mask(d + 1) & vw[w] & in_len;
            const uint32_t mutual = row_live ? (low_mask(e) & ~low_mask(a) & mw[w] & in_len) : 0u;
            const uint32_t ok = causal | mutual;
            // a word whose 32 keys are visible to every row of this warp costs one vote
            if (!__all_sync(0xffffffffu, ok == 0xffffffffu)) {
#pragma unroll
              for (int c = 0; c < 32; ++c)
                if (!((ok >> c) & 1u)) s[32 * w + c] = -INFINITY;
            }
          }
        }
        // ---- row maximum: three-input maxima (FMNMX3), four independent chains
        float mx[4] = {fmax3(s[0], s[1], s[2]), fmax3(s[3], s[4], s[5]), fmax3(s[6], s[7], s[8]), fmax3(s[9], s[10], s[11])};
#pragma unroll
        for (int c = 12; c < 124; c += 8) {
          mx[0] = fmax3(mx[0], s[c], s[c + 1]); mx[1] = fmax3(mx[1], s[c + 2], s[c + 3]);
          mx[2] = fmax3(mx[2], s[c + 4], s[c + 5]); mx[3] = fmax3(mx[3], s[c + 6], s[c + 7]);
        }
        mx[0] = fmax3(mx[0], s[124], s[125]); mx[1] = fmax3(mx[1], s[126], s[127]);
        const float m_new = fmaxf(m_used, fmaxf(fmax3(mx[0], mx[1], mx[2]), mx[3]));
        // ---- lazy rescale: O and l stay expressed against m_used until the maximum has grown by more than 2^8
        const bool need = (m_new - m_used) * P.scale_log2 > RESCALE_THRESHOLD || (m_used == -INFINITY && m_new > -INFINITY);
        if (__any_sync(0xffffffffu, need)) {
          if (j > 0) {
            const float alpha = need ? ((m_used == -INFINITY) ? 0.f : ex2_approx((m_used - m_new) * P.scale_log2)) : 1.f;
            mbar_wait(BAR(PV_DONE + t), (n_pvh - 1) & 1);    // every PV of this tile issued so far has landed
            tc_fence_after();
            rescale_o96(tm_o, alpha);
            l *= alpha;
          }
          if (need) m_used = m_new;
        }
        const float neg_m = (m_used == -INFINITY) ? 0.f : -m_used * P.scale_log2;
        const uint64_t sc2 = f32x2_pack(P.scale_log2, P.scale_log2), nm2 = f32x2_pack(neg_m, neg_m);
        // exp2((S - m_used) * scale*log2e) of 64 scores starting at `off`, packed IN PLACE into s[off .. off+32)
        auto exps = [&](int off) {
          uint64_t sum_a = f32x2_pack(0.f, 0.f), sum_b = sum_a;
#pragma unroll
          for (int x = 0; x < 32; ++x) {
            const uint64_t a2 = f32x2_fma(f32x2_pack(s[off + 2 * x], s[off + 2 * x + 1]), sc2, nm2);
            float p0, p1;
            if ((x & 3) >= 4 - AKI_FWD_POLY) {
              exp2_poly_x2(a2, p0, p1);
            } else {
              float a0, a1;
              f32x2_unpack(a2, a0, a1);
              p0 = ex2_approx(a0); p1 = ex2_approx(a1);
            }
            if (x & 1) sum_b = f32x2_add(sum_b, f32x2_pack(p0, p1));
            else sum_a = f32x2_add(sum_a, f32x2_pack(p0, p1));
            s[off + x] = __uint_as_float(pack_bf16x2(p0, p1));
          }
          float t0, t1;
          f32x2_unpack(f32x2_add(sum_a, sum_b), t0, t1);
          return t0 + t1;
        };
        // ---- keys 0-63 -> P -> PV(j, first half)
        TR(t, j, 3);
        l += exps(0);
        TR(t, j, 4);
        if (n_pvh > 0) mbar_wait(BAR(PV_DONE + t), (n_pvh - 1) & 1);   // the previous PV half has consumed P
        tc_fence_after();
        tmem_st_x32(tm_p, reinterpret_cast<const uint32_t*>(s));
        tmem_wait_st();
        tc_fence_before();
        mbar_arrive(BAR(P_FULL + t));
        ++n_pvh;
        TR(t, j, 6);
        // ---- keys 64-127 while PV(first half) runs
        l += exps(64);
        TR(t, j, 7);
        mbar_wait(BAR(PV_DONE + t), (n_pvh - 1) & 1);
        tc_fence_after();
        TR(t, j, 8);
        tmem_st_x32(tm_p, reinterpret_cast<const uint32_t*>(s) + 64);
        tmem_wait_st();
        tc_fence_before();
        mbar_arrive(BAR(P_FULL + t));
        ++n_pvh;
      }
      // ---- hand the row statistics to the epilogue warps and move on to the next item
      if (n_it > 0) mbar_wait(BAR(O_FREE + t), (n_it - 1) & 1);   // they have read the previous item's statistics
      lm_s[t][r] = make_float2(row_live ? l : 0.f, m_used);
      mbar_arrive(BAR(L_READY + t));
      ++n_it;
    }
  } else {
    // ------------------------------------------------------------------ RoPE of the next item's Q, epilogue of this one
    setmaxnreg_dec<REGS_EPI>();
    const int g = warp & 3;
    const int r = 32 * g + lane;
    const uint32_t lane_base = (uint32_t)(g * 32) << 16;
    auto rope_item = [&](uint32_t n, const int4& v0, const int4& v1, const int4& v2) {
      const int buf = n & 1, b = v0.y;
#pragma unroll 1
      for (int t = 0; t < 2; ++t) {
        mbar_wait(BAR(Q_FULL + 2 * buf + t), (n >> 1) & 1);
        const int i = (t ? v1.y : v1.x) + r;
        if ((t ? v2.y : v2.x) > 0 && i < P.T) {
          const uint32_t qa = smem_base + SMEM_Q + (2 * buf + t) * TILE_BYTES;
          const float* cr = P.rope_cos + (size_t)b * P.rope_stride_b + (size_t)i * 48;
          const float* sr = P.rope_sin + (size_t)b * P.rope_stride_b + (size_t)i * 48;
#pragma unroll 2
          for (int c = 0; c < 6; ++c) {          // 16-byte chunk c pairs with chunk c+6 (d <-> d+48)
            const uint32_t a_lo = qa + (c >> 2) * ATOM + sw64_offset(r, c & 3);
            const uint32_t a_hi = qa + ((c + 6) >> 2) * ATOM + sw64_offset(r, (c + 6) & 3);
            uint4 lo, hi;
            asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(lo.x), "=r"(lo.y), "=r"(lo.z), "=r"(lo.w) : "r"(a_lo));
            asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(hi.x), "=r"(hi.y), "=r"(hi.z), "=r"(hi.w) : "r"(a_hi));
            float cs[8], sn[8];
            *reinterpret_cast<float4*>(cs) = __ldg(reinterpret_cast<const float4*>(cr + c * 8));
            *reinterpret_cast<float4*>(cs + 4) = __ldg(reinterpret_cast<const float4*>(cr + c * 8 + 4));
            *reinterpret_cast<float4*>(sn) = __ldg(reinterpret_cast<const float4*>(sr + c * 8));
            *reinterpret_cast<float4*>(sn + 4) = __ldg(reinterpret_cast<const float4*>(sr + c * 8 + 4));
            const __nv_bfloat162* l2 = reinterpret_cast<const __nv_bfloat162*>(&lo);
            const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&hi);
            uint32_t lo_w[4], hi_w[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 lf = __bfloat1622float2(l2[e]), hf2 = __bfloat1622float2(h2[e]);
              lo_w[e] = pack_bf16x2(lf.x * cs[2 * e] - hf2.x * sn[2 * e], lf.y * cs[2 * e + 1] - hf2.y * sn[2 * e + 1]);
              hi_w[e] = pack_bf16x2(hf2.x * cs[2 * e] + lf.x * sn[2 * e], hf2.y * cs[2 * e + 1] + lf.y * sn[2 * e + 1]);
            }
            asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(a_lo), "r"(lo_w[0]), "r"(lo_w[1]), "r"(lo_w[2]), "r"(lo_w[3]) : "memory");
            asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(a_hi), "r"(hi_w[0]), "r"(hi_w[1]), "r"(hi_w[2]), "r"(hi_w[3]) : "memory");
          }
        }
      }
      fence_proxy_async_smem();
      mbar_arrive(BAR(Q_READY + buf));
    };
    uint32_t n_it = 0, n_od[2] = {0, 0};
    int4 v0, v1, v2;
    item_wait(0, v0, v1, v2);
    if (ROPE && v0.x) rope_item(0, v0, v1, v2);
    while (v0.x) {
      int4 w0, w1, w2;
      item_wait(n_it + 1, w0, w1, w2);
      if (ROPE && w0.x) rope_item(n_it + 1, w0, w1, w2);
      const int b = v0.y, h = v0.z, len = v0.w;
#pragma unroll 1
      for (int t = 0; t < 2; ++t) {
        const int nk = t ? v2.y : v2.x, rows = t ? v1.w : v1.z;
        const int ql = (t ? v1.y : v1.x) + r, i = P.q_off + ql;   // query row of q / o / lse, its key coordinate
        mbar_wait(BAR(L_READY + t), n_it & 1);
        const float2 lm = lm_s[t][r];
        if (nk > 0) {
          mbar_wait(BAR(O_DONE + t), n_od[t] & 1);
          ++n_od[t];
          tc_fence_after();
        }
        // rows with no visible key (batch padding, keys all invalid): zeros (DESIGN.md).  Their maximum never left -inf;
        // the row sum alone does not tell (the polynomial exp2 returns 2^-126, not 0, for a masked score)
        const float inv_l = (nk > 0 && i < len && lm.x > 0.f && lm.y > -INFINITY) ? 1.f / lm.x : 0.f;
        const bool store_row = (r < rows) && (ql < P.T);
        __nv_bfloat16* orow = P.o.row(b, store_row ? ql : 0, h);
        // tcgen05.ld is warp-collective (.sync.aligned): load unconditionally, predicate only the global stores
#pragma unroll 1
        for (int c = 0; c < 3; ++c) {
          uint32_t o[32];
          if (nk > 0) {
            tmem_ld_x32(tmem + TM_O + 96 * t + lane_base + 32 * c, o);
            tmem_wait_ld();
          }
#pragma unroll
          for (int x = 0; x < 4; ++x) {
            uint4 u;
            uint32_t* w = reinterpret_cast<uint32_t*>(&u);
#pragma unroll
            for (int e = 0; e < 4; ++e)
              w[e] = (inv_l > 0.f) ? pack_bf16x2(__uint_as_float(o[8 * x + 2 * e]) * inv_l,
                                                   __uint_as_float(o[8 * x + 2 * e + 1]) * inv_l)
                                   : 0u;
            if (store_row) *reinterpret_cast<uint4*>(orow + 32 * c + 8 * x) = u;
          }
        }
        if (P.lse && store_row)
          P.lse[((size_t)b * P.H + h) * P.T + ql] = (inv_l > 0.f) ? (lm.y * P.scale + __logf(lm.x)) : INFINITY;
        tc_fence_before();
        mbar_arrive(BAR(O_FREE + t));
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(BAR(ITEM_EMPTY + n_it % SLOTS));
      v0 = w0; v1 = w1; v2 = w2;
      ++n_it;
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(BAR(ITEM_EMPTY + n_it % SLOTS));   // the terminator's slot
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<512>(tmem);
}

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = []() -> EncodeTiledFn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess) return nullptr;
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}

// (D=96, T, H, B) bf16 view -> tensor map with [32 x 128 x 1 x 1] SWIZZLE_64B boxes
int make_tile_map(CUtensorMap* m, const AkiMmaTensor4& t, int B, int H, int T, int box_rows) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) { set_last_cuda_error("cuTensorMapEncodeTiled entry point not found"); return AKI_ERR_CUDA; }
  cuuint64_t dims[4] = {96, (cuuint64_t)T, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)t.stride_t * 2, (cuuint64_t)t.stride_h * 2, (cuuint64_t)t.stride_b * 2};
  cuuint32_t box[4] = {32, (cuuint32_t)box_rows, 1, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, t.ptr, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_last_cuda_error("cuTensorMapEncodeTiled failed"); return AKI_ERR_CUDA; }
  return AKI_OK;
}

// dQ accumulator (B,H,T,96) fp32 contiguous -> [32 x 128 x 1 x 1] fp32 SWIZZLE_128B boxes for TMA reductions
int make_dq_accum_map(CUtensorMap* m, float* dq_accum, int B, int H, int T) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) { set_last_cuda_error("cuTensorMapEncodeTiled entry point not found"); return AKI_ERR_CUDA; }
  cuuint64_t dims[4] = {96, (cuuint64_t)T, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t strides[3] = {96 * 4, (cuuint64_t)T * 96 * 4, (cuuint64_t)H * T * 96 * 4};
  cuuint32_t box[4] = {32, 128, 1, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, dq_accum, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_last_cuda_error("cuTensorMapEncodeTiled(dq) failed"); return AKI_ERR_CUDA; }
  return AKI_OK;
}

// row statistics (B,H,t_pad,8) bf16 contiguous -> [8 x 128 x 1 x 1] boxes, no swizzle: one box is the K-major
// SWIZZLE_NONE operand [16 row groups][8 rows][16 B] of the backward's statistics k-step
int make_row_stats_map(CUtensorMap* m, void* base, int B, int H, int t_pad) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) { set_last_cuda_error("cuTensorMapEncodeTiled entry point not found"); return AKI_ERR_CUDA; }
  cuuint64_t dims[4] = {8, (cuuint64_t)t_pad, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t strides[3] = {16, (cuuint64_t)t_pad * 16, (cuuint64_t)H * t_pad * 16};
  cuuint32_t box[4] = {8, 128, 1, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_last_cuda_error("cuTensorMapEncodeTiled(row stats) failed"); return AKI_ERR_CUDA; }
  return AKI_OK;
}

// Per-device one-time setup (kernel attribute, SM count): the library may drive several GPUs from one process.
struct FwdDeviceState {
  std::once_flag once;
  int sm_count = 0;
  cudaError_t err = cudaSuccess;
};
static FwdDeviceState g_fwd_dev[64];

static int fwd_device_setup(int* sm_count) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { set_last_cuda_error("cudaGetDevice failed"); return AKI_ERR_CUDA; }
  FwdDeviceState& s = g_fwd_dev[dev];
  std::call_once(s.once, [&]() {
    s.err = cudaFuncSetAttribute(attn_fwd_sm100_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, fwd::SMEM_ALLOC);
    if (s.err == cudaSuccess)
      s.err = cudaFuncSetAttribute(attn_fwd_sm100_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, fwd::SMEM_ALLOC);
    if (s.err == cudaSuccess) s.err = cudaDeviceGetAttribute(&s.sm_count, cudaDevAttrMultiProcessorCount, dev);
  });
  if (s.err != cudaSuccess) { set_last_cuda_error(cudaGetErrorString(s.err)); return AKI_ERR_CUDA; }
  *sm_count = s.sm_count;
  return AKI_OK;
}

}  // namespace aki

using namespace aki;

extern "C" int aki_mma_attn_fwd(const AkiMmaAttnParams* p, aki_stream_t stream) {
  AKI_REQUIRE(p, AKI_ERR_NULL);
  int rc = check_attn_params(*p);
  if (rc) return rc;
  AKI_REQUIRE(!p->fwd_plan || p->plan_pairs >= ((p->T + fwd::BM - 1) / fwd::BM + 1) / 2, AKI_ERR_BAD_SHAPE);
  CUtensorMap mq, mk, mv;
  if ((rc = make_tile_map(&mq, p->q, p->B, p->H, p->T, fwd::BM))) return rc;
  const int n_keys = p->q_offset + p->T;   // check_attn_params: no overflow
  if ((rc = make_tile_map(&mk, p->k, p->B, p->H, n_keys, fwd::BN))) return rc;
  if ((rc = make_tile_map(&mv, p->v, p->B, p->H, n_keys, fwd::BN))) return rc;
  FwdKernelParams kp;
  kp.q = view_of(p->q); kp.o = view_of(p->o);
  kp.lse = p->lse; kp.rope_cos = p->rope_cos; kp.rope_sin = p->rope_sin; kp.rope_stride_b = p->rope_stride_b;
  kp.mm = mask_meta_from(*p);
  kp.plan = reinterpret_cast<const int4*>(p->fwd_plan);
  kp.plan_pairs = p->plan_pairs;
  kp.B = p->B; kp.H = p->H; kp.T = p->T;
  kp.q_off = p->q_offset;
  const int n_qt = (p->T + fwd::BM - 1) / fwd::BM;
  kp.ranks = p->fwd_plan ? p->plan_pairs : (n_qt + 1) / 2;
  const long long slices = (long long)p->B * p->H;
  kp.group = (int)(slices < fwd::HEADS_PER_GROUP ? slices : fwd::HEADS_PER_GROUP);
  const long long n_groups = (slices + kp.group - 1) / kp.group;
  const long long n_items = n_groups * kp.ranks * kp.group;
  AKI_REQUIRE(n_items > 0 && n_items < (1ll << 31), AKI_ERR_BAD_SHAPE);
  kp.n_items = (int)n_items;
  kp.scale = p->scale;
  kp.scale_log2 = p->scale * 1.4426950408889634f;
  kp.trace = nullptr; kp.trace_cta = -1;
#ifdef AKI_FWD_TRACE
  // Debug build only (make TRACE=1; tools/fwd_trace.py): dumps clock64 stamps of one CTA's first item and SYNCHRONISES.
  const char* trace_env = getenv("AKI_MMA_FWD_TRACE");
  const size_t trace_bytes = 4 * 64 * 12 * sizeof(unsigned long long);
  if (trace_env) {
    kp.trace_cta = atoi(trace_env);
    cudaMalloc(&kp.trace, trace_bytes);
    cudaMemset(kp.trace, 0, trace_bytes);
  }
#endif
  int sm_count = 0;
  if ((rc = fwd_device_setup(&sm_count))) return rc;
  // AKI_MMA_FWD_SCHED=static: persistent CTAs walk the items with a fixed stride instead of the hardware queue (A/B only)
  static const bool use_static = []() { const char* e = getenv("AKI_MMA_FWD_SCHED"); return e && e[0] == 's'; }();
  kp.use_clc = use_static ? 0 : 1;
  const unsigned grid = kp.use_clc ? (unsigned)n_items : (unsigned)(n_items < sm_count ? n_items : sm_count);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  timing_hook_begin(st);
  if (p->rope_cos)
    attn_fwd_sm100_kernel<true><<<grid, fwd::THREADS, fwd::SMEM_ALLOC, st>>>(mq, mk, mv, kp);
  else
    attn_fwd_sm100_kernel<false><<<grid, fwd::THREADS, fwd::SMEM_ALLOC, st>>>(mq, mk, mv, kp);
  timing_hook_end(st);
#ifdef AKI_FWD_TRACE
  if (trace_env) {
    cudaDeviceSynchronize();
    static unsigned long long host[4 * 64 * 12];
    cudaMemcpy(host, kp.trace, trace_bytes, cudaMemcpyDeviceToHost);
    cudaFree(kp.trace);
    unsigned long long t0 = ~0ull;
    for (size_t i = 0; i < 4 * 64 * 12; ++i) if (host[i] && host[i] < t0) t0 = host[i];
    const char* names[4] = {"sm_t0", "sm_t1", "mma_t0", "mma_t1"};
    for (int slot = 0; slot < 4; ++slot)
      for (int j = 0; j < 64; ++j) {
        if (!host[(slot * 64 + j) * 12] && !host[(slot * 64 + j) * 12 + 2]) continue;
        fprintf(stderr, "TRACE %s j=%d:", names[slot], j);
        for (int k = 0; k < 10; ++k) fprintf(stderr, " %llu", host[(slot * 64 + j) * 12 + k] ? host[(slot * 64 + j) * 12 + k] - t0 : 0ull);
        fprintf(stderr, "\n");
      }
  }
#endif
  return check_launch();
}
