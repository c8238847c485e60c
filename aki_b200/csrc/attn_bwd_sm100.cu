// Modality-mutual attention backward for sm_100a (tcgen05 / TMEM / TMA).
//
// Gradient of softmax_fp32(QK^T*scale + mask) V (the eager core of Phi3Attention.forward; installed equivalent
// transformers/models/phi3/modeling_phi3.py:153-175; the reference obtains it from autograd over five passes
// on a (B,32,T,T) tensor).  One CTA owns one 128-key tile of one (batch, head) and walks exactly the query tiles
// that can see it (kv_tile_q_mask: with MMA that set is the image-row tiles before the diagonal plus everything
// from the diagonal on), with everything transposed so that keys sit on TMEM lanes:
//     S^T  = K Q_i^T  - LSE_i/scale       (SS)        P^T = exp2(S^T * scale*log2e)   -> TMEM (bf16, own columns)
//     dP^T = V dO_i^T - delta_i           (SS)        dS^T = P^T o dP^T               -> smem (bf16)
//     dV  += P^T dO_i                     (TS)
//     dQ_i = dS K                         (SS, A MN-major = the dS^T smem buffer, B MN-major = K)
//     dK  += dS^T Q_i                     (SS, A K-major = dS^T, B MN-major = Q_i)       (x scale in the epilogue)
// (A variant that wrote P^T in place over S^T and kept dS^T in TMEM for a TS dK was no faster and showed a rare
// dV mismatch -- S^T(i+1) overwriting columns that dV(i) still reads as its A operand -- so every TMEM region that
// an MMA reads is only ever rewritten after an explicit mbarrier round trip.)
// The per-query statistics are folded INTO the two score MMAs: a 7th k-step multiplies a constant "ones" operand
// [1,1,1,0..] on the key side with a [128][8] bf16 row-statistics operand on the query side that holds -LSE/scale
// (resp. -delta) split into three bf16 terms (hi + mid + lo: 2^-24 relative).  In this transposed layout LSE and
// delta vary along the TMEM COLUMNS, so without the fold every element would need a shared-memory broadcast read
// and an FFMA/FADD; with it the element-wise work per score is one multiply (packed f32x2), one ex2 and one
// bf16 pack for P, and one multiply and one pack for dS (ncu before the fold: the compute warps, not the tensor
// pipe, bounded the kernel at 35% tensor-active).  Rows beyond the sequence get -1e30 there, so P is exactly 0.
// dK / dV accumulate in TMEM over the whole loop; dQ_i is drained by a dedicated warpgroup: TMEM -> registers ->
// fp32 SWIZZLE_128B staging in shared memory -> TMA tensor reduction (cp.reduce.async.bulk.tensor .add) into a
// fp32 accumulator in HBM; aki_mma_attn_bwd's finalize kernel applies scale, the inverse RoPE and the bf16 cast.
//
// PERSISTENT CTAs on the hardware work queue (cluster launch control, as in the forward): an item is one
// (batch, head, key tile); items are numbered heaviest key tile first inside groups of 8 (batch, head) slices (their
// Q / dO stay in L2) and a CTA keeps asking for the next one.  The next item's query-tile list, its first Q / dO tiles
// and -- as soon as the last MMAs of the current item have read K / V -- its K / V tiles are fetched under the current
// item's tail; the dK / dV epilogue of item n overlaps S^T / dP^T of item n+1.
// 16 warps: 0 TMA producer | 1, 2 MMA issuers (streams A / B; 2 also allocates TMEM) | 3 scheduler: next item id, list of
// the query tiles to visit | 4-11 compute (thread <-> key row r; the two warpgroups split the 128 query columns of a
// tile in halves; on the few tiles that are not fully visible they read the query rows' mutual intervals from
// global memory) | 12-15 dQ drain.  Tensor-pipe order per query tile: dV(i) S(i+1) dQ(i) dK(i) dP(i+1) -- the dQ drain overlaps dK, the
// exponentials of tile i+1 overlap dQ/dK/dP.
// TMEM columns: S^T [0,128)  dP^T/dQ [128,256)  dV [256,352)  dK [352,448)  P^T (bf16 pairs) [448,512).
// Shared memory: K, V 24 KB each (resident), Q ring 2x(24+2) KB (the [128][8] row statistics travel with Q), dO ring
// 2x24 KB, dS^T 32 KB, dQ staging 2x16 KB, ones/zero core matrices, mask statistics, query-tile list.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <mutex>
#include "attn_aux.cuh"
#include "sm100_ptx.cuh"

namespace aki {

namespace bwd {
constexpr int BN = 128, BM = 128;
constexpr int ATOM_BYTES = 128 * 64;          // bf16 operand atom [128 rows][64 B], SWIZZLE_64B
constexpr int TILE_BYTES = 3 * ATOM_BYTES;
constexpr int AUG_BYTES = 128 * 16;           // row-statistics operand [16 groups][8 rows][16 B], no swizzle
constexpr int DQ_ATOM_BYTES = 128 * 128;      // fp32 staging atom [128 rows][32 floats], SWIZZLE_128B
// Q(it) lives from S^T(it) to dK(it), ~1.5 steps plus the TMA latency: a third Q stage removes the ~700-cycle wait of
// stream A for Q(it+1) (clock64 trace), but only fits next to 2 x 8 KB of dQ staging, and the drain then becomes the
// bottleneck (6 proxy-fenced rounds per tile; measured 2.67 ms vs 2.57 ms) -- kept at 2 stages + 2 x 16 KB staging.
constexpr int Q_STAGES = 2, DO_STAGES = 2;
constexpr int THREADS = 512;
constexpr int MAX_TILES = 512;                // T <= 65536
constexpr int SMEM_K = 0;
constexpr int SMEM_V = SMEM_K + TILE_BYTES;
constexpr int SMEM_Q = SMEM_V + TILE_BYTES;
constexpr int SMEM_DO = SMEM_Q + Q_STAGES * TILE_BYTES;
constexpr int SMEM_DS = SMEM_DO + DO_STAGES * TILE_BYTES;   // 4 atoms [128][64 B]
constexpr int SMEM_DQ = SMEM_DS + 4 * ATOM_BYTES;           // 2 staging atoms
constexpr int SMEM_QAUG = SMEM_DQ + 2 * DQ_ATOM_BYTES;      // Q_STAGES x AUG_BYTES: [-LSE/scale x3, 0, -delta x3, 0] per query row
constexpr int SMEM_ONES = SMEM_QAUG + Q_STAGES * AUG_BYTES; // core matrix [8][16 B] of [1,1,1,0,0,0,0,0] rows (selects -LSE/scale)
constexpr int SMEM_ONES_D = SMEM_ONES + 128;                // core matrix of [0,0,0,0,1,1,1,0] rows (selects -delta)
constexpr int SMEM_ZERO = SMEM_ONES_D + 128;                // one all-zero core matrix
constexpr int SLOTS = 2;                      // item ring: the current item and the next one
constexpr int SMEM_QLIST = SMEM_ZERO + 128;                 // SLOTS x uint16[MAX_TILES]
constexpr int SMEM_TOTAL = SMEM_QLIST + SLOTS * MAX_TILES * 2;
#ifndef AKI_BWD_SLICES_PER_GROUP
#define AKI_BWD_SLICES_PER_GROUP 8
#endif
constexpr int SMEM_ALLOC = SMEM_TOTAL + 1024;
static_assert(SMEM_ALLOC + 256 <= 232448, "shared memory budget");
constexpr uint32_t TM_S = 0, TM_DP = 128, TM_DV = 256, TM_DK = 352, TM_P = 448;
constexpr int REGS_CTRL = 64, REGS_COMPUTE = 168, REGS_DRAIN = 112;   // 128*64 + 256*168 + 128*112 = 65536
}  // namespace bwd

struct BwdKernelParams {
  TensorView d_k, d_v;
  const float* rope_cos;
  const float* rope_sin;
  int64_t rope_stride_b;
  MaskMeta mm;
  int B, H, T, n_t, n_words;
  int group, n_items, use_clc;   // items: ((g * n_t + kt) * group + slice)
  float scale_log2, scale;
  unsigned long long* trace;  // debug build (make TRACE=1, tools/bwd_trace.py): clock64 stamps of one CTA
  int trace_cta;
};

// -DKO_x (tools/build_bwd_ko.sh) are timing-only knockout builds: each removes one component -- an MMA group (KO_S KO_DP
// KO_DV KO_DQ KO_DK), the ex2 (KO_EXP), the dS compute + store + proxy fence (KO_DS; KO_FENCE only the fence), the dQ
// drain (KO_DRAIN; KO_RED only its reductions), the Q/dO loads after the first ring fill (KO_TMA).  Results are wrong by
// construction; the shipped build defines none of them.
#ifdef AKI_FWD_TRACE
#define TRB(slot, j, k) do { if (tracing && (j) < 64) P.trace[((slot) * 64 + (j)) * 8 + (k)] = clock64(); } while (0)
#else
#define TRB(slot, j, k) do { } while (0)
#endif

__device__ __forceinline__ void f32x2_mul(float& lo, float& hi, float a_lo, float a_hi, float b_lo, float b_hi) {
  uint64_t r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(f32x2_pack(a_lo, a_hi)), "l"(f32x2_pack(b_lo, b_hi)));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(r));
}

__global__ void __launch_bounds__(bwd::THREADS, 1)
attn_bwd_sm100_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                      const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_do,
                      const __grid_constant__ CUtensorMap map_dq, const __grid_constant__ CUtensorMap map_qaug,
                      const BwdKernelParams P) {
  using namespace bwd;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* const smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));   // generic pointer to the aligned base
  constexpr int KV_FULL = 0, KV_EMPTY = 1, Q_FULL = 2, Q_EMPTY = Q_FULL + Q_STAGES, DO_FULL = Q_EMPTY + Q_STAGES,
                DO_EMPTY = DO_FULL + DO_STAGES, S_FULL = DO_EMPTY + DO_STAGES, P_READY = S_FULL + 1,
                DP_FULL = P_READY + 1, DS_READY = DP_FULL + 1, DQ_FULL = DS_READY + 1, DQ_DRAINED = DQ_FULL + 1,
                ALL_DONE = DQ_DRAINED + 1, ACC_FREE = ALL_DONE + 1,
                ITEM_FULL = ACC_FREE + 1, ITEM_EMPTY = ITEM_FULL + SLOTS, CLC_BAR = ITEM_EMPTY + SLOTS, N_BARS = CLC_BAR + 1;
  __shared__ __align__(8) uint64_t bars[N_BARS];
  __shared__ __align__(16) int4 item_ring[SLOTS][2];   // {valid, b, h, kt} {n_q, keys_all_valid, len, 0}
  __shared__ __align__(16) uint4 clc_resp;
  __shared__ uint32_t tmem_base_s;
  const uint32_t bar0 = smem_u32(bars);
  auto BAR = [&](int i) { return bar0 + 8u * i; };

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  uint16_t* const qlist_all = reinterpret_cast<uint16_t*>(smem_gen + SMEM_QLIST);

  if (tid == 0) {
    mbar_init(BAR(KV_FULL), 1); mbar_init(BAR(KV_EMPTY), 2);
    // every Q / dO stage is read by both MMA warps: two commits free it
    for (int i = 0; i < Q_STAGES; ++i) { mbar_init(BAR(Q_FULL + i), 1); mbar_init(BAR(Q_EMPTY + i), 2); }
    for (int i = 0; i < DO_STAGES; ++i) { mbar_init(BAR(DO_FULL + i), 1); mbar_init(BAR(DO_EMPTY + i), 2); }
    mbar_init(BAR(S_FULL), 1); mbar_init(BAR(P_READY), 256); mbar_init(BAR(DP_FULL), 1);
    mbar_init(BAR(DS_READY), 256); mbar_init(BAR(DQ_FULL), 1); mbar_init(BAR(DQ_DRAINED), 128);
    mbar_init(BAR(ALL_DONE), 2); mbar_init(BAR(ACC_FREE), 256);
    for (int i = 0; i < SLOTS; ++i) { mbar_init(BAR(ITEM_FULL + i), 1); mbar_init(BAR(ITEM_EMPTY + i), 15); }
    mbar_init(BAR(CLC_BAR), 1);
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc<512>(smem_u32(&tmem_base_s));
    // constant operands of the statistics k-step: one core matrix of [1,1,1,0,0,0,0,0] rows, one of zeros
    if (lane < 8) *reinterpret_cast<uint4*>(smem_gen + SMEM_ONES + lane * 16) = make_uint4(0x3f803f80u, 0x00003f80u, 0u, 0u);
    else if (lane < 16) *reinterpret_cast<uint4*>(smem_gen + SMEM_ONES_D + (lane - 8) * 16) = make_uint4(0u, 0u, 0x3f803f80u, 0x00003f80u);
    else if (lane < 24) *reinterpret_cast<uint4*>(smem_gen + SMEM_ZERO + (lane - 16) * 16) = make_uint4(0u, 0u, 0u, 0u);
    fence_proxy_async_smem();
  }
  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&map_q); tma_prefetch_desc(&map_k); tma_prefetch_desc(&map_v); tma_prefetch_desc(&map_do);
    tma_prefetch_desc(&map_dq); tma_prefetch_desc(&map_qaug);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;

  // every role walks the same sequence of items through the ring; n = running item count of the caller
  auto item_wait = [&](uint32_t n, int4& v0, int4& v1) {
    const int slot = n % SLOTS;
    mbar_wait(BAR(ITEM_FULL + slot), (n / SLOTS) & 1);
    v0 = item_ring[slot][0]; v1 = item_ring[slot][1];
  };

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    setmaxnreg_dec<REGS_CTRL>();
    if (elect_one()) {
      uint32_t n_it = 0, n_work = 0, qc = 0;   // items seen, items with work, Q / dO tiles loaded so far
      for (;;) {
        int4 v0, v1;
        item_wait(n_it, v0, v1);
        if (!v0.x) break;
        const int b = v0.y, h = v0.z, j0 = v0.w * BN, n_q = v1.x;
        const uint16_t* qlist = qlist_all + (n_it % SLOTS) * MAX_TILES;
        auto load_tile = [&](int it) {
          const int i0 = (int)qlist[it];
          const uint32_t c = qc + it, sq = c % Q_STAGES, sd = c % DO_STAGES;
          mbar_wait(BAR(Q_EMPTY + sq), ((c / Q_STAGES) & 1) ^ 1);
#ifdef KO_TMA
          if (c >= Q_STAGES) { mbar_arrive(BAR(Q_FULL + sq)); mbar_wait(BAR(DO_EMPTY + sd), ((c / DO_STAGES) & 1) ^ 1); mbar_arrive(BAR(DO_FULL + sd)); return; }
#endif
          mbar_arrive_expect_tx(BAR(Q_FULL + sq), TILE_BYTES + AUG_BYTES);
          for (int a = 0; a < 3; ++a)
            tma_load_4d(smem_base + SMEM_Q + sq * TILE_BYTES + a * ATOM_BYTES, &map_q, BAR(Q_FULL + sq), a * 32, i0, h, b);
          tma_load_4d(smem_base + SMEM_QAUG + sq * AUG_BYTES, &map_qaug, BAR(Q_FULL + sq), 0, i0, h, b);
          mbar_wait(BAR(DO_EMPTY + sd), ((c / DO_STAGES) & 1) ^ 1);
          mbar_arrive_expect_tx(BAR(DO_FULL + sd), TILE_BYTES);
          for (int a = 0; a < 3; ++a)
            tma_load_4d(smem_base + SMEM_DO + sd * TILE_BYTES + a * ATOM_BYTES, &map_do, BAR(DO_FULL + sd), a * 32, i0, h, b);
        };
        if (n_q > 0) {
          // the first Q / dO tiles go out as soon as their stages are free (the previous item's last steps), K / V once
          // its last MMAs have read the resident tiles
          const int pre = min(n_q, Q_STAGES);
          for (int it = 0; it < pre; ++it) load_tile(it);
          if (n_work > 0) mbar_wait(BAR(KV_EMPTY), (n_work - 1) & 1);
          mbar_arrive_expect_tx(BAR(KV_FULL), 2 * TILE_BYTES);
          for (int a = 0; a < 3; ++a) {
            tma_load_4d(smem_base + SMEM_K + a * ATOM_BYTES, &map_k, BAR(KV_FULL), a * 32, j0, h, b);
            tma_load_4d(smem_base + SMEM_V + a * ATOM_BYTES, &map_v, BAR(KV_FULL), a * 32, j0, h, b);
          }
          for (int it = pre; it < n_q; ++it) load_tile(it);
          qc += n_q;
          ++n_work;
        }
        mbar_arrive(BAR(ITEM_EMPTY + n_it % SLOTS));
        ++n_it;
      }
    }
  } else if (warp == 1 || warp == 2) {
    // ------------------------------------------------------------------ MMA issuers
    // TWO issuing warps: an M=128, K=16 tcgen05.mma costs ~64-70 cycles whatever N is when a single thread
    // streams them (tools/mma_mix_bench.cu: this step takes 2337 cycles from one thread, ~1650-2050 from two), so
    // the step is split into two independent in-order streams that the barrier protocol already separates:
    //   warp 1 (A): dV(i) += P^T dO_i ; S^T(i+1)           warp 2 (B): dQ_i ; dK += dS^T Q_i ; dP^T(i+1)
    // Every TMEM / smem region an MMA reads is rewritten only after an mbarrier round trip: S^T(i+1) after P_READY(i)
    // (A); dQ_i over dP^T(i) after DS_READY, dP^T(i+1) over dQ_i after DQ_DRAINED, and dP^T(i+1) sits behind dK(i), so
    // the dS^T buffer is consumed before the compute warps can see DP_FULL(i+1) (B).  Q / dO stages are freed by one
    // commit from each stream, K / V (per item) likewise; the dK / dV accumulators of the next item wait for ACC_FREE.
    setmaxnreg_dec<REGS_CTRL>();
    if (elect_one()) {
      constexpr uint32_t IDESC_SS_KK = umma_idesc_bf16(128, 128, 0, 0);       // S^T, dP^T
      constexpr uint32_t IDESC_N96_BMN = umma_idesc_bf16(128, 96, 0, 1);      // dV (TS), dK (SS)
      constexpr uint32_t IDESC_N96_AMN_BMN = umma_idesc_bf16(128, 96, 1, 1);  // dQ
      const uint32_t sK = smem_base + SMEM_K, sV = smem_base + SMEM_V, sDS = smem_base + SMEM_DS;
      // descriptors differ only in the 14-bit start-address field: build the constant parts once
      const uint64_t DESC_KMAJ = umma_smem_desc(0, 16, 512, UMMA_SW64);
      const uint64_t DESC_MNMAJ = umma_smem_desc(0, ATOM_BYTES, 512, UMMA_SW64);
      // statistics k-step (no swizzle, K-major): ones = one core matrix shared by every row group (SBO 0), its
      // second K chunk = the zero core matrix (LBO); row statistics = [16 groups][128 B], second K chunk aliases
      // the first (LBO 0) and meets the zero chunk of the ones operand.  Validated in tools/umma_probe.cu (5-7).
      const uint64_t DESC_ONES = umma_smem_desc(smem_base + SMEM_ONES, SMEM_ZERO - SMEM_ONES, 0, UMMA_SW_NONE);
      const uint64_t DESC_ONES_D = umma_smem_desc(smem_base + SMEM_ONES_D, SMEM_ZERO - SMEM_ONES_D, 0, UMMA_SW_NONE);
      const uint64_t DESC_AUG = umma_smem_desc(0, 0, 128, UMMA_SW_NONE);
      auto kmajor = [&](uint32_t base, int k) {   // 16-element K step k of a [rows][96|128] K-major SW64 tile
        return DESC_KMAJ | (uint64_t)(((base + (k >> 1) * ATOM_BYTES + (k & 1) * 32) >> 4) & 0x3FFFu);
      };
      auto mnmajor = [&](uint32_t base, int k) {  // 16-row K step k of a tile read as MN-major
        return DESC_MNMAJ | (uint64_t)(((base + k * 1024) >> 4) & 0x3FFFu);
      };
      uint32_t n_it = 0, n_work = 0, gs = 0;   // items seen, items with work, query-tile steps so far (== Q / dO tile count)
      if (warp == 1) {
        for (;;) {
          int4 v0, v1;
          item_wait(n_it, v0, v1);
          if (!v0.x) break;
          const int n_q = v1.x;
#ifdef AKI_FWD_TRACE
          const bool tracing = P.trace && (int)blockIdx.x == P.trace_cta && n_it == 0;
#endif
          if (n_q > 0) {
          // ---------------- stream A
          auto issue_s = [&](int it) {
            const uint32_t c = gs + it;
            const uint32_t sQ = smem_base + SMEM_Q + (c % Q_STAGES) * TILE_BYTES;
            const uint32_t sA = smem_base + SMEM_QAUG + (c % Q_STAGES) * AUG_BYTES;
#ifndef KO_S
#pragma unroll
            for (int k = 0; k < 6; ++k) umma_ss(tmem + TM_S, kmajor(sK, k), kmajor(sQ, k), IDESC_SS_KK, k > 0);
            umma_ss(tmem + TM_S, DESC_ONES, DESC_AUG | (uint64_t)((sA >> 4) & 0x3FFFu), IDESC_SS_KK, 1);
#endif
            umma_commit(BAR(S_FULL));
            umma_commit(BAR(Q_EMPTY + c % Q_STAGES));   // this stream's half of the release (the other: dK on B)
          };
          mbar_wait(BAR(KV_FULL), n_work & 1);
          mbar_wait(BAR(Q_FULL + gs % Q_STAGES), (gs / Q_STAGES) & 1);
          tc_fence_after();
          issue_s(0);     // the S region is ours: P_READY of the previous item's last tile was waited for below
          for (int it = 0; it < n_q; ++it) {
            const uint32_t c = gs + it;
            const uint32_t sDO = smem_base + SMEM_DO + (c % DO_STAGES) * TILE_BYTES;
            // dV += P^T dO_it
            TRB(2, it, 0);
            mbar_wait(BAR(DO_FULL + c % DO_STAGES), (c / DO_STAGES) & 1);   // dO_it has landed (stream B waits for it too)
            mbar_wait(BAR(P_READY), c & 1);
            if (it == 0 && n_work > 0) mbar_wait(BAR(ACC_FREE), (n_work - 1) & 1);   // the epilogue has read the previous dV
            tc_fence_after();
            TRB(2, it, 1);
#ifndef KO_DV
#pragma unroll
            for (int k = 0; k < 8; ++k)
              umma_ts(tmem + TM_DV, tmem + TM_P + 8 * k, mnmajor(sDO, k), IDESC_N96_BMN, (it > 0 || k > 0));
#endif
            umma_commit(BAR(DO_EMPTY + c % DO_STAGES));
            TRB(2, it, 2);
            // S^T of the next query tile (the S region is free once P^T(it) has been written to its own columns)
            if (it + 1 < n_q) {
              mbar_wait(BAR(Q_FULL + (c + 1) % Q_STAGES), ((c + 1) / Q_STAGES) & 1);
              tc_fence_after();
              TRB(2, it, 3);
              issue_s(it + 1);
              TRB(2, it, 4);
            }
          }
          umma_commit(BAR(ALL_DONE));
          umma_commit(BAR(KV_EMPTY));
            gs += n_q; ++n_work;
          }
          mbar_arrive(BAR(ITEM_EMPTY + n_it % SLOTS));
          ++n_it;
        }
      } else {
        for (;;) {
          int4 v0, v1;
          item_wait(n_it, v0, v1);
          if (!v0.x) break;
          const int n_q = v1.x;
#ifdef AKI_FWD_TRACE
          const bool tracing = P.trace && (int)blockIdx.x == P.trace_cta && n_it == 0;
#endif
          if (n_q > 0) {
          // ---------------- stream B
          auto issue_dp = [&](int it) {
            const uint32_t c = gs + it;
            const uint32_t sDO = smem_base + SMEM_DO + (c % DO_STAGES) * TILE_BYTES;
            const uint32_t sA = smem_base + SMEM_QAUG + (c % Q_STAGES) * AUG_BYTES;   // row statistics travel with Q(it)
#ifndef KO_DP
#pragma unroll
            for (int k = 0; k < 6; ++k) umma_ss(tmem + TM_DP, kmajor(sV, k), kmajor(sDO, k), IDESC_SS_KK, k > 0);
            umma_ss(tmem + TM_DP, DESC_ONES_D, DESC_AUG | (uint64_t)((sA >> 4) & 0x3FFFu), IDESC_SS_KK, 1);
#endif
            umma_commit(BAR(DP_FULL));
            umma_commit(BAR(DO_EMPTY + c % DO_STAGES));
          };
          mbar_wait(BAR(KV_FULL), n_work & 1);
          mbar_wait(BAR(DO_FULL + gs % DO_STAGES), (gs / DO_STAGES) & 1);
          mbar_wait(BAR(Q_FULL + gs % Q_STAGES), (gs / Q_STAGES) & 1);
          if (gs > 0) mbar_wait(BAR(DQ_DRAINED), (gs - 1) & 1);   // dQ of the previous item's last tile has left the dP region
          tc_fence_after();
          issue_dp(0);
          for (int it = 0; it < n_q; ++it) {
            const uint32_t c = gs + it;
            const uint32_t sQ = smem_base + SMEM_Q + (c % Q_STAGES) * TILE_BYTES;
            // dQ_it = dS K first (its drain then overlaps dK), dK += dS^T Q_it
            TRB(3, it, 0);
            mbar_wait(BAR(DS_READY), c & 1);
            tc_fence_after();
            TRB(3, it, 1);
#ifndef KO_DQ
#pragma unroll
            for (int k = 0; k < 8; ++k)
              umma_ss(tmem + TM_DP, mnmajor(sDS, k), mnmajor(sK, k), IDESC_N96_AMN_BMN, k > 0);
#endif
            umma_commit(BAR(DQ_FULL));
            if (it == 0 && n_work > 0) { mbar_wait(BAR(ACC_FREE), (n_work - 1) & 1); tc_fence_after(); }   // previous dK read
#ifndef KO_DK
#pragma unroll
            for (int k = 0; k < 8; ++k)
              umma_ss(tmem + TM_DK, kmajor(sDS, k), mnmajor(sQ, k), IDESC_N96_BMN, (it > 0 || k > 0));
#endif
            umma_commit(BAR(Q_EMPTY + c % Q_STAGES));
            TRB(3, it, 2);
            // dP^T of the next query tile overwrites the dQ region: wait until it has been drained
            if (it + 1 < n_q) {
              mbar_wait(BAR(DO_FULL + (c + 1) % DO_STAGES), ((c + 1) / DO_STAGES) & 1);
              mbar_wait(BAR(Q_FULL + (c + 1) % Q_STAGES), ((c + 1) / Q_STAGES) & 1);   // -delta sits in the Q stage
              TRB(3, it, 3);
              mbar_wait(BAR(DQ_DRAINED), c & 1);
              tc_fence_after();
              TRB(3, it, 4);
              issue_dp(it + 1);
              TRB(3, it, 5);
            }
          }
          umma_commit(BAR(ALL_DONE));
          umma_commit(BAR(KV_EMPTY));
            gs += n_q; ++n_work;
          }
          mbar_arrive(BAR(ITEM_EMPTY + n_it % SLOTS));
          ++n_it;
        }
      }
    }
  } else if (warp == 3) {
    // ------------------------------------------------------------------ scheduler: next item, its query-tile list
    setmaxnreg_dec<REGS_CTRL>();
    uint32_t n_pub = 0, n_clc = 0;
    long long id = blockIdx.x;
    for (;;) {
      // item id -> (group of slices, key tile, slice): key tiles ascending = heaviest first inside a group
      const int per_group = P.n_t * P.group;
      const int g = (int)(id / per_group), rem = (int)(id % per_group);
      const int kt = rem / P.group, bh = g * P.group + rem % P.group;
      if (bh < P.B * P.H) {
        const int b = bh / P.H, h = bh % P.H;
        const int len = meta_len(P.mm, b, P.T);
        const int j0 = kt * BN;
        const int slot = n_pub % SLOTS;
        mbar_wait(BAR(ITEM_EMPTY + slot), ((n_pub / SLOTS) & 1) ^ 1);
        uint16_t* const qlist = qlist_all + slot * MAX_TILES;
        // list of query tiles to visit (first query row of each, ascending)
        const int n_live = (len + BM - 1) / BM;
        int n = 0;
        if (j0 < len) {
          if (P.mm.kv_tile_q_mask) {
            const uint32_t* mrow = P.mm.kv_tile_q_mask + ((size_t)b * P.n_t + kt) * P.n_words;
            for (int w0 = 0; w0 < P.n_words; w0 += 32) {
              const int w = w0 + lane;
              uint32_t word = (w < P.n_words) ? mrow[w] : 0u;
              if (w * 32 >= n_live) word = 0u;                                        // keep only live tiles
              else if (w * 32 + 32 > n_live) word &= (1u << (n_live - w * 32)) - 1u;
              const int cnt = __popc(word);
              int incl = cnt;
#pragma unroll
              for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += t;
              }
              int pos = n + incl - cnt;
              while (word) {
                const int bit = __ffs(word) - 1;
                word &= word - 1;
                qlist[pos++] = (uint16_t)((w * 32 + bit) * BM);
              }
              n += __shfl_sync(0xffffffffu, incl, 31);
            }
            // Visits before the diagonal exist only for image rows (their interval reaches this key tile).  An image span
            // that straddles two 128-row tiles would cost two visits per key tile; the query tile is only a TMA coordinate,
            // so such a pair becomes ONE visit of the unaligned tile that starts at the span's first relevant row.
            __syncwarp();
            int n_pre = 0;
            for (int e = lane; e < n; e += 32) n_pre += ((int)qlist[e] < j0) ? 1 : 0;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) n_pre += __shfl_xor_sync(0xffffffffu, n_pre, o);
            if (n_pre >= 2 && P.mm.row_lo) {
              auto relevant = [&](int i) {
                if (i >= len) return false;
                const int lo = __ldg(P.mm.row_lo + (size_t)b * P.mm.meta_pitch + i);
                const int hi = __ldg(P.mm.row_hi + (size_t)b * P.mm.meta_pitch + i);
                return hi > lo && lo < j0 + BN && hi > j0;
              };
              int out = 0, e = 0;
              while (e < n_pre) {
                const int a = (int)qlist[e];
                int i0 = a, step = 1;
                if (e + 1 < n_pre && (int)qlist[e + 1] == a + BM) {
                  int first = 1 << 30, last = -1;
#pragma unroll
                  for (int k = 0; k < 4; ++k) {
                    const int row = 32 * k + lane;
                    if (relevant(a + row)) first = min(first, row);
                    if (relevant(a + BM + row)) last = max(last, row);
                  }
#pragma unroll
                  for (int o = 16; o > 0; o >>= 1) {
                    first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
                    last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
                  }
                  if (first > 0 && first < BM && last < first) { i0 = a + first; step = 2; }
                }
                __syncwarp();
                if (lane == 0) qlist[out] = (uint16_t)i0;
                ++out;
                e += step;
              }
              const int shift = n_pre - out;
              if (shift > 0) {
                for (int base = n_pre; base < n; base += 32) {
                  const int idx = base + lane;
                  const uint16_t v = (idx < n) ? qlist[idx] : (uint16_t)0;
                  __syncwarp();
                  if (idx < n) qlist[idx - shift] = v;
                  __syncwarp();
                }
                n -= shift;
              }
            }
          } else {
            for (int qt = kt + lane; qt < n_live; qt += 32) qlist[qt - kt] = (uint16_t)(qt * BM);
            n = max(0, n_live - kt);
          }
        }
        // are all 128 keys of this tile inside the sequence and causally visible (no padding)?
        bool ok = true;
        if (lane < 4) {
          const int jw = j0 + 32 * lane;
          ok = (jw + 32 <= len);
          if (ok && P.mm.vbits) ok = (P.mm.vbits[(size_t)b * P.mm.bits_pitch + (jw >> 5)] == 0xffffffffu);
        }
        ok = __all_sync(0xffffffffu, ok);
        __syncwarp();
        if (lane == 0) {
          item_ring[slot][0] = make_int4(1, b, h, kt);
          item_ring[slot][1] = make_int4(n, ok ? 1 : 0, len, 0);
          mbar_arrive(BAR(ITEM_FULL + slot));
        }
        ++n_pub;
      }
      // next item: the hardware queue, or a fixed stride (A/B builds)
      int more = 0;
      long long next = 0;
      if (lane == 0) {
        if (!P.use_clc) {
          next = id + gridDim.x;
          more = next < P.n_items;
        } else {
          mbar_arrive_expect_tx(BAR(CLC_BAR), 16);
          clc_try_cancel(smem_u32(&clc_resp), BAR(CLC_BAR));
          mbar_wait(BAR(CLC_BAR), n_clc & 1);
          uint32_t x;
          more = clc_query(smem_u32(&clc_resp), x) ? 1 : 0;
          next = x;
          fence_proxy_async_smem();     // the response buffer is rewritten by the next (async-proxy) query
        }
      }
      ++n_clc;
      more = __shfl_sync(0xffffffffu, more, 0);
      next = __shfl_sync(0xffffffffu, next, 0);
      if (!more) break;
      id = next;
    }
    {
      const int slot = n_pub % SLOTS;
      mbar_wait(BAR(ITEM_EMPTY + slot), ((n_pub / SLOTS) & 1) ^ 1);
      if (lane == 0) {
        item_ring[slot][0] = make_int4(0, 0, 0, 0);
        item_ring[slot][1] = make_int4(0, 0, 0, 0);
        mbar_arrive(BAR(ITEM_FULL + slot));
      }
    }
  } else if (warp < 12) {
    // ------------------------------------------------------------------ compute warps: P^T and dS^T
    setmaxnreg_inc<REGS_COMPUTE>();
    const int ct = tid - 128;                 // 0..255
    const int r = ct & 127;                   // key row within the tile == TMEM lane
    const int hq = ct >> 7;                   // which half of the query columns
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    uint32_t n_it = 0, n_work = 0, gs = 0;
    for (;;) {
      int4 v0, v1;
      item_wait(n_it, v0, v1);
      if (!v0.x) break;
      const int b = v0.y, h = v0.z, j0 = v0.w * BN, n_q = v1.x, len = v1.z;
      const bool keys_all_valid = v1.y != 0;
      const uint16_t* qlist = qlist_all + (n_it % SLOTS) * MAX_TILES;
      const int j = j0 + r;                     // key index

      // key-side predicate bits
      bool k_valid = (j < len), k_mutual = (j < len);
      if (j < len && P.mm.vbits) k_valid = (P.mm.vbits[(size_t)b * P.mm.bits_pitch + (j >> 5)] >> (j & 31)) & 1u;
      if (j < len && P.mm.mbits) k_mutual = (P.mm.mbits[(size_t)b * P.mm.bits_pitch + (j >> 5)] >> (j & 31)) & 1u;

      float p[64];   // P^T row half, kept from phase a to phase b
#ifdef AKI_FWD_TRACE
      const bool tracing = P.trace && (int)blockIdx.x == P.trace_cta && (tid & 127) == 0 && n_it == 0;   // warps 4 and 8 (same SMSP)
      const int slot = hq;
#endif

      auto phase_a = [&](int it) {
        const uint32_t c = gs + it;
        const int i0 = (int)qlist[it];
        const bool full = (i0 >= j0 + BN) && keys_all_valid;     // every query row lies after every key; CTA-uniform
        TRB(slot, it, 0);
        mbar_wait(BAR(S_FULL), c & 1);
        tc_fence_after();
        TRB(slot, it, 1);
        uint32_t sraw[64];
        tmem_ld_x32(tmem + TM_S + lane_base + 64 * hq, sraw);
        tmem_ld_x32(tmem + TM_S + lane_base + 64 * hq + 32, sraw + 32);
        tmem_wait_ld();
#pragma unroll
        for (int c2 = 0; c2 < 64; c2 += 2) {
          float x0, x1;
          f32x2_mul(x0, x1, __uint_as_float(sraw[c2]), __uint_as_float(sraw[c2 + 1]), P.scale_log2, P.scale_log2);
#ifdef KO_EXP
          p[c2] = x0; p[c2 + 1] = x1;
#else
          p[c2] = ex2_approx(x0);
          p[c2 + 1] = ex2_approx(x1);
#endif
        }
        if (!full) {
          // c visible iff (c >= cmin, causal) or (row c of the tile is an image row whose interval holds key j).  The
          // intervals of this half's 64 query rows come straight from global memory (warp-uniform addresses: one
          // broadcast transaction per load, L1-resident); only tiles that are not fully visible get here -- the diagonal,
          // key tiles with padding and the image-row visits before the diagonal.  (They used to travel through a
          // 2-stage shared-memory ring filled by another warp; releasing a stage of that ring without having waited
          // for it -- fully visible tiles skip the wait -- let the consumer overtake the producer by a whole phase.)
          const int cmin = k_valid ? (j - i0 - 64 * hq) : (1 << 30);
          if (P.mm.row_lo && k_mutual) {
            const int32_t* lo_p = P.mm.row_lo + (size_t)b * P.mm.meta_pitch + i0 + 64 * hq;
            const int32_t* hi_p = P.mm.row_hi + (size_t)b * P.mm.meta_pitch + i0 + 64 * hq;
            const int n_live = len - (i0 + 64 * hq);       // rows c >= n_live lie beyond the sequence
#pragma unroll
            for (int cc = 0; cc < 64; ++cc) {
              int lo = 0, wd = 0;
              if (cc < n_live) { lo = __ldg(lo_p + cc); wd = max(__ldg(hi_p + cc) - lo, 0); }
              const bool ok = (cc >= cmin) || ((unsigned)(j - lo) < (unsigned)wd);
              p[cc] = ok ? p[cc] : 0.f;
            }
          } else {
#pragma unroll
            for (int cc = 0; cc < 64; ++cc) p[cc] = (cc >= cmin) ? p[cc] : 0.f;
          }
        }
        uint32_t pk[32];
#pragma unroll
        for (int x = 0; x < 32; ++x) pk[x] = pack_bf16x2(p[2 * x], p[2 * x + 1]);
        TRB(slot, it, 2);
        tmem_st_x32(tmem + TM_P + lane_base + 32 * hq, pk);   // own columns: the other half may still be reading S^T
        tmem_wait_st();
        tc_fence_before();
        mbar_arrive(BAR(P_READY));
        TRB(slot, it, 3);
      };

      auto phase_b = [&](int it) {
        const uint32_t c = gs + it;
        TRB(slot, it, 4);
        mbar_wait(BAR(DP_FULL), c & 1);
        tc_fence_after();
        TRB(slot, it, 5);
        uint32_t draw[64];
        tmem_ld_x32(tmem + TM_DP + lane_base + 64 * hq, draw);
        tmem_ld_x32(tmem + TM_DP + lane_base + 64 * hq + 32, draw + 32);
        tmem_wait_ld();
        const uint32_t ds_base = smem_base + SMEM_DS;
        uint32_t dsw[32];
#pragma unroll
        for (int c8 = 0; c8 < 8; ++c8) {   // 8 query columns -> one 16-byte chunk of the dS^T row
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int cc = 8 * c8 + 2 * e;
            float d0, d1;
            f32x2_mul(d0, d1, p[cc], p[cc + 1], __uint_as_float(draw[cc]), __uint_as_float(draw[cc + 1]));
            dsw[4 * c8 + e] = pack_bf16x2(d0, d1);
          }
          const int col = 64 * hq + 8 * c8;          // query column of this chunk
          const uint32_t addr = ds_base + (col >> 5) * ATOM_BYTES + sw64_offset(r, (col & 31) >> 3);
#ifndef KO_DS
          asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(dsw[4 * c8]), "r"(dsw[4 * c8 + 1]),
                       "r"(dsw[4 * c8 + 2]), "r"(dsw[4 * c8 + 3]));
#endif
        }
#if !defined(KO_DS) && !defined(KO_FENCE)
        fence_proxy_async_smem();
#endif
        tc_fence_before();
        mbar_arrive(BAR(DS_READY));
        TRB(slot, it, 6);
      };

      // a(0) | b(0) a(1) | b(1) a(2) | ... | b(n_q-1)   (one instance of each phase in the instruction stream)
      for (int step = 0; step <= n_q && n_q > 0; ++step) {
        if (step > 0) phase_b(step - 1);
        if (step < n_q) phase_a(step);
      }

      // ---- epilogue: dV, dK (x scale, inverse RoPE) -> bf16 -> global.  tcgen05.ld is warp-collective: the loads
      // are unconditional, only the global stores are predicated on the row being inside the tensor.
      {
        const bool store_row = (j < P.T);
        const int js = store_row ? j : 0;
        __nv_bfloat16* dvrow = P.d_v.row(b, js, h) + 48 * hq;
        __nv_bfloat16* dkrow = P.d_k.row(b, js, h);
        if (n_q > 0) {
          // RoPE tables of this key row: fetched before the wait so that their latency hides behind the last MMAs
          float cs[24], sn[24];
          if (P.rope_cos) {
            const float4* c4 = reinterpret_cast<const float4*>(P.rope_cos + (size_t)b * P.rope_stride_b + (size_t)js * 48 + 24 * hq);
            const float4* s4 = reinterpret_cast<const float4*>(P.rope_sin + (size_t)b * P.rope_stride_b + (size_t)js * 48 + 24 * hq);
#pragma unroll
            for (int x = 0; x < 6; ++x) {
              *reinterpret_cast<float4*>(cs + 4 * x) = __ldg(c4 + x);
              *reinterpret_cast<float4*>(sn + 4 * x) = __ldg(s4 + x);
            }
          }
          mbar_wait(BAR(ALL_DONE), n_work & 1);
          tc_fence_after();
          uint32_t acc[48];
          tmem_ld_x32(tmem + TM_DV + lane_base + 48 * hq, acc);
          tmem_ld_x16(tmem + TM_DV + lane_base + 48 * hq + 32, acc + 32);
          // dK: this half owns columns [24hq, 24hq+24) and their RoPE partners [48+24hq, 48+24hq+24)
          uint32_t lo[24], hi[24];
          tmem_ld_x16(tmem + TM_DK + lane_base + 24 * hq, lo);
          tmem_ld_x8(tmem + TM_DK + lane_base + 24 * hq + 16, *reinterpret_cast<uint32_t(*)[8]>(lo + 16));
          tmem_ld_x16(tmem + TM_DK + lane_base + 48 + 24 * hq, hi);
          tmem_ld_x8(tmem + TM_DK + lane_base + 48 + 24 * hq + 16, *reinterpret_cast<uint32_t(*)[8]>(hi + 16));
          tmem_wait_ld();
          tc_fence_before();
          mbar_arrive(BAR(ACC_FREE));      // the accumulators may be overwritten by the next item's first dV / dK
#pragma unroll
          for (int x = 0; x < 6; ++x) {
            uint4 u;
            u.x = pack_bf16x2(__uint_as_float(acc[8 * x]), __uint_as_float(acc[8 * x + 1]));
            u.y = pack_bf16x2(__uint_as_float(acc[8 * x + 2]), __uint_as_float(acc[8 * x + 3]));
            u.z = pack_bf16x2(__uint_as_float(acc[8 * x + 4]), __uint_as_float(acc[8 * x + 5]));
            u.w = pack_bf16x2(__uint_as_float(acc[8 * x + 6]), __uint_as_float(acc[8 * x + 7]));
            if (store_row) *reinterpret_cast<uint4*>(dvrow + 8 * x) = u;
          }
          float flo[24], fhi[24];
#pragma unroll
          for (int x = 0; x < 24; ++x) {
            float a = __uint_as_float(lo[x]) * P.scale, e = __uint_as_float(hi[x]) * P.scale;
            if (P.rope_cos) {   // g = R^T g'
              const float a2 = a * cs[x] + e * sn[x], e2 = e * cs[x] - a * sn[x];
              a = a2; e = e2;
            }
            flo[x] = a; fhi[x] = e;
          }
#pragma unroll
          for (int x = 0; x < 3; ++x) {
            uint4 u, w;
            u.x = pack_bf16x2(flo[8 * x], flo[8 * x + 1]); u.y = pack_bf16x2(flo[8 * x + 2], flo[8 * x + 3]);
            u.z = pack_bf16x2(flo[8 * x + 4], flo[8 * x + 5]); u.w = pack_bf16x2(flo[8 * x + 6], flo[8 * x + 7]);
            w.x = pack_bf16x2(fhi[8 * x], fhi[8 * x + 1]); w.y = pack_bf16x2(fhi[8 * x + 2], fhi[8 * x + 3]);
            w.z = pack_bf16x2(fhi[8 * x + 4], fhi[8 * x + 5]); w.w = pack_bf16x2(fhi[8 * x + 6], fhi[8 * x + 7]);
            if (store_row) {
              *reinterpret_cast<uint4*>(dkrow + 24 * hq + 8 * x) = u;
              *reinterpret_cast<uint4*>(dkrow + 48 + 24 * hq + 8 * x) = w;
            }
          }
        } else if (store_row) {
          const uint4 z = make_uint4(0, 0, 0, 0);
#pragma unroll
          for (int x = 0; x < 6; ++x) *reinterpret_cast<uint4*>(dvrow + 8 * x) = z;
#pragma unroll
          for (int x = 0; x < 3; ++x) {
            *reinterpret_cast<uint4*>(dkrow + 24 * hq + 8 * x) = z;
            *reinterpret_cast<uint4*>(dkrow + 48 + 24 * hq + 8 * x) = z;
          }
        }
      }
      if (n_q > 0) { gs += n_q; ++n_work; }
      __syncwarp();
      if (lane == 0) mbar_arrive(BAR(ITEM_EMPTY + n_it % SLOTS));
      ++n_it;
    }
  } else {
    // ------------------------------------------------------------------ dQ drain warps (lane r <-> QUERY row r)
    setmaxnreg_dec<REGS_DRAIN>();
    const int r = tid - 384;
    const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
    uint32_t n_it = 0, gs = 0;
    for (;;) {
      int4 v0, v1;
      item_wait(n_it, v0, v1);
      if (!v0.x) break;
      const int b = v0.y, h = v0.z, n_q = v1.x;
      const uint16_t* qlist = qlist_all + (n_it % SLOTS) * MAX_TILES;
#ifdef AKI_FWD_TRACE
      const bool tracing = P.trace && (int)blockIdx.x == P.trace_cta && r == 0 && n_it == 0;
#endif
      for (int it = 0; it < n_q; ++it) {
        const uint32_t c = gs + it;
        const int i0 = (int)qlist[it];
        TRB(4, it, 0);
        mbar_wait(BAR(DQ_FULL), c & 1);
        tc_fence_after();
        TRB(4, it, 1);
#ifdef KO_DRAIN
        mbar_arrive(BAR(DQ_DRAINED));
        continue;
#endif
        uint32_t dq[96];
        tmem_ld_x32(tmem + TM_DP + lane_base, dq);
        tmem_ld_x32(tmem + TM_DP + lane_base + 32, dq + 32);
        tmem_ld_x32(tmem + TM_DP + lane_base + 64, dq + 64);
        tmem_wait_ld();
        tc_fence_before();
        mbar_arrive(BAR(DQ_DRAINED));
        TRB(4, it, 2);
        // three [128][32 x fp32] SWIZZLE_128B atoms through two staging buffers
#pragma unroll
        for (int a = 0; a < 3; ++a) {
          const int buf = (c * 3 + a) & 1;
          const uint32_t abase = smem_base + SMEM_DQ + buf * DQ_ATOM_BYTES;
          if (r == 0) tma_store_wait_read<1>();       // the reduction that last read this buffer has finished reading
          named_bar_sync(2, 128);
#pragma unroll
          for (int x = 0; x < 8; ++x) {
            const uint32_t addr = abase + r * 128 + ((x ^ (r & 7)) << 4);
            asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(dq[32 * a + 4 * x]),
                         "r"(dq[32 * a + 4 * x + 1]), "r"(dq[32 * a + 4 * x + 2]), "r"(dq[32 * a + 4 * x + 3]) : "memory");
          }
          fence_proxy_async_smem();
          named_bar_sync(3, 128);
#ifndef KO_RED
          if (r == 0) {
            tma_reduce_add_4d(&map_dq, abase, 32 * a, i0, h, b);
            tma_store_commit();
          }
#endif
        }
      }
      gs += n_q;
      __syncwarp();
      if (lane == 0) mbar_arrive(BAR(ITEM_EMPTY + n_it % SLOTS));
      ++n_it;
    }
    // the reductions still in flight only have to finish READING the staging buffers before the CTA retires its shared
    // memory; their global writes complete with the grid
    if (r == 0) tma_store_wait_read<0>();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<512>(tmem);
}

// Per-device one-time setup (kernel attribute, SM count): the library may drive several GPUs from one process.
struct BwdDeviceState {
  std::once_flag once;
  int sm_count = 0;
  cudaError_t err = cudaSuccess;
};
static BwdDeviceState g_bwd_dev[64];

static int bwd_device_setup(int* sm_count) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { set_last_cuda_error("cudaGetDevice failed"); return AKI_ERR_CUDA; }
  BwdDeviceState& s = g_bwd_dev[dev];
  std::call_once(s.once, [&]() {
    s.err = cudaFuncSetAttribute(attn_bwd_sm100_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bwd::SMEM_ALLOC);
    if (s.err == cudaSuccess) s.err = cudaDeviceGetAttribute(&s.sm_count, cudaDevAttrMultiProcessorCount, dev);
  });
  if (s.err != cudaSuccess) { set_last_cuda_error(cudaGetErrorString(s.err)); return AKI_ERR_CUDA; }
  *sm_count = s.sm_count;
  return AKI_OK;
}

}  // namespace aki

using namespace aki;

extern "C" int aki_mma_attn_bwd(const AkiMmaAttnBwdParams* p, aki_stream_t stream) {
  AKI_REQUIRE(p, AKI_ERR_NULL);
  const AkiMmaAttnParams& f = p->fwd;
  AKI_REQUIRE(f.q_offset == 0, AKI_ERR_UNSUPPORTED);   // no backward for a continuation chunk
  int rc = check_attn_params(f);
  if (rc) return rc;
  if ((rc = check_tensor(p->d_o)) || (rc = check_tensor(p->d_q)) || (rc = check_tensor(p->d_k)) ||
      (rc = check_tensor(p->d_v)))
    return rc;
  AKI_REQUIRE(f.lse && p->workspace, AKI_ERR_NULL);
  AKI_REQUIRE(p->deterministic == 0, AKI_ERR_UNSUPPORTED);
  AKI_REQUIRE(p->workspace_bytes >= aki_mma_attn_bwd_workspace_bytes(f.B, f.H, f.T, f.D), AKI_ERR_BAD_SHAPE);
  AKI_REQUIRE((reinterpret_cast<uintptr_t>(p->workspace) & 255u) == 0, AKI_ERR_MISALIGNED);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  BwdWorkspace w = carve_bwd_workspace(p->workspace, f.B, f.H, f.T, f.D);
  if ((rc = launch_bwd_preprocess(*p, w, st))) return rc;
  if (cudaMemsetAsync(w.dq_accum, 0, (size_t)f.B * f.H * f.T * f.D * sizeof(float), st) != cudaSuccess) {
    set_last_cuda_error(cudaGetErrorString(cudaGetLastError()));
    return AKI_ERR_CUDA;
  }
  AkiMmaTensor4 qrot{w.q_rot, (int64_t)f.H * f.T * f.D, (int64_t)f.D, (int64_t)f.T * f.D};
  CUtensorMap mq, mk, mv, mdo, mdq, mqa;
  if ((rc = make_tile_map(&mq, qrot, f.B, f.H, f.T, bwd::BM))) return rc;
  if ((rc = make_tile_map(&mk, f.k, f.B, f.H, f.T, bwd::BN))) return rc;
  if ((rc = make_tile_map(&mv, f.v, f.B, f.H, f.T, bwd::BN))) return rc;
  if ((rc = make_tile_map(&mdo, p->d_o, f.B, f.H, f.T, bwd::BM))) return rc;
  if ((rc = make_dq_accum_map(&mdq, w.dq_accum, f.B, f.H, f.T))) return rc;
  if ((rc = make_row_stats_map(&mqa, w.row_stats, f.B, f.H, w.t_pad))) return rc;
  BwdKernelParams kp;
  kp.d_k = view_of(p->d_k); kp.d_v = view_of(p->d_v);
  kp.rope_cos = f.rope_cos; kp.rope_sin = f.rope_sin; kp.rope_stride_b = f.rope_stride_b;
  kp.mm = mask_meta_from(f);
  kp.B = f.B; kp.H = f.H; kp.T = f.T;
  kp.n_t = (f.T + bwd::BN - 1) / bwd::BN;
  kp.n_words = (kp.n_t + 31) / 32;
  AKI_REQUIRE(kp.n_t <= bwd::MAX_TILES, AKI_ERR_UNSUPPORTED);
  kp.scale = f.scale;
  kp.scale_log2 = f.scale * 1.4426950408889634f;
  kp.trace = nullptr; kp.trace_cta = -1;
#ifdef AKI_FWD_TRACE
  const char* trace_env = getenv("AKI_MMA_BWD_TRACE");
  const size_t trace_bytes = 5 * 64 * 8 * sizeof(unsigned long long);
  if (trace_env) {
    kp.trace_cta = atoi(trace_env);
    cudaMalloc(&kp.trace, trace_bytes);
    cudaMemset(kp.trace, 0, trace_bytes);
  }
#endif
  const long long slices = (long long)f.B * f.H;
  kp.group = (int)(slices < AKI_BWD_SLICES_PER_GROUP ? slices : AKI_BWD_SLICES_PER_GROUP);
  const long long n_groups = (slices + kp.group - 1) / kp.group;
  const long long n_items = n_groups * kp.n_t * kp.group;
  AKI_REQUIRE(n_items > 0 && n_items < (1ll << 31), AKI_ERR_BAD_SHAPE);
  kp.n_items = (int)n_items;
  int sm_count = 0;
  if ((rc = bwd_device_setup(&sm_count))) return rc;
  // AKI_MMA_BWD_SCHED=static: persistent CTAs walk the items with a fixed stride instead of the hardware queue (A/B only)
  static const bool use_static = []() { const char* e = getenv("AKI_MMA_BWD_SCHED"); return e && e[0] == 's'; }();
  kp.use_clc = use_static ? 0 : 1;
  const long long grid = kp.use_clc ? n_items : (n_items < sm_count ? n_items : sm_count);
  timing_hook_begin(st);
  attn_bwd_sm100_kernel<<<(unsigned)grid, bwd::THREADS, bwd::SMEM_ALLOC, st>>>(mq, mk, mv, mdo, mdq, mqa, kp);
  timing_hook_end(st);
#ifdef AKI_FWD_TRACE
  if (trace_env) {
    cudaDeviceSynchronize();
    static unsigned long long host[5 * 64 * 8];
    cudaMemcpy(host, kp.trace, trace_bytes, cudaMemcpyDeviceToHost);
    cudaFree(kp.trace);
    unsigned long long t0 = ~0ull;
    for (size_t i = 0; i < 5 * 64 * 8; ++i) if (host[i] && host[i] < t0) t0 = host[i];
    const char* names[5] = {"cmp_h0", "cmp_h1", "mma_A", "mma_B", "drain"};
    for (int slot = 0; slot < 5; ++slot)
      for (int j = 0; j < 64; ++j) {
        bool any = false;
        for (int k = 0; k < 8; ++k) any = any || host[(slot * 64 + j) * 8 + k];
        if (!any) continue;
        fprintf(stderr, "TRACE %s it=%d:", names[slot], j);
        for (int k = 0; k < 7; ++k) fprintf(stderr, " %llu", host[(slot * 64 + j) * 8 + k] ? host[(slot * 64 + j) * 8 + k] - t0 : 0ull);
        fprintf(stderr, "\n");
      }
  }
#endif
  if ((rc = check_launch())) return rc;
  return launch_dq_finalize(*p, w, f.scale, st);   // dS^T is kept unscaled inside the kernel
}
