// Integer kernels around the attention core: segment metadata (replaces the reference's Python mask loop,
// codes/open_flamingo/src/vlm.py:410-443, :486-577), per-tile loop bounds, the debug expansion to the
// reference's (B,1,T,T) int64 tensor, and the splice gather (vlm.py:516-588, utils.py:62-96).
// All HBM-bound; O(B*T) integers instead of O(B*T^2).
#include <cuda_bf16.h>
#include <limits.h>
#include <string.h>
#include "api_common.cuh"

namespace aki {

constexpr int SEG_THREADS = 256;

__device__ __forceinline__ int block_exclusive_scan(int v, int* warp_sums, int& block_total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int n = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += n;
  }
  if (lane == 31) warp_sums[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int w = (lane < SEG_THREADS / 32) ? warp_sums[lane] : 0;
    int wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int n = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += n;
    }
    if (lane < SEG_THREADS / 32) warp_sums[lane] = wi - w;  // exclusive warp offsets
    if (lane == 31) warp_sums[32] = wi;                      // block total
  }
  __syncthreads();
  int excl = incl - v + warp_sums[warp];
  block_total = warp_sums[32];
  __syncthreads();
  return excl;
}

__global__ void __launch_bounds__(SEG_THREADS)
segments_kernel(const int64_t* __restrict__ lang_x, const int64_t* __restrict__ attention_mask, int L, int N,
                int64_t media_id, int64_t asst_id, int t_cap, int text_only, int32_t* __restrict__ seq_len,
                int32_t* __restrict__ q_end_out, int32_t* __restrict__ seg, int32_t* __restrict__ row_lo,
                int32_t* __restrict__ row_hi, int32_t* __restrict__ src, uint32_t* __restrict__ kv_valid_bits,
                uint32_t* __restrict__ kv_mutual_bits, int32_t* __restrict__ status) {
  const int b = blockIdx.x, tid = threadIdx.x;
  const int64_t* ids = lang_x + (size_t)b * L;
  const int64_t* am = attention_mask + (size_t)b * L;
  const int words = (t_cap + 31) / 32;
  __shared__ int s_first_asst, s_nimg, s_nimg_before;
  __shared__ int warp_sums[33];
  if (tid == 0) { s_first_asst = INT_MAX; s_nimg = 0; s_nimg_before = 0; }
  __syncthreads();
  // pass 1: first <|assistant|> (only the first occurrence counts, vlm.py:492-494) and #images
  int first = INT_MAX, nimg = 0;
  for (int l = tid; l < L; l += SEG_THREADS) {
    int64_t t = ids[l];
    if (t == asst_id) first = min(first, l);
    nimg += (t == media_id);
  }
  atomicMin(&s_first_asst, first);
  atomicAdd(&s_nimg, nimg);
  __syncthreads();
  const int l0 = s_first_asst;
  const int total_img = s_nimg;
  // pass 2: images before the <|assistant|> token -> its post-splice index
  if (l0 != INT_MAX) {
    int c = 0;
    for (int l = tid; l < l0; l += SEG_THREADS) c += (ids[l] == media_id);
    atomicAdd(&s_nimg_before, c);
  }
  __syncthreads();
  const int q_end = (l0 == INT_MAX) ? 0 : l0 + s_nimg_before * (N - 1) + 1;
  const int T_b = L + total_img * (N - 1);
  if (tid == 0) {
    seq_len[b] = T_b;
    if (q_end_out) q_end_out[b] = q_end;
    if (status && T_b > t_cap) atomicExch(status, 1);
  }
  if (!(seg || row_lo || row_hi || src || kv_valid_bits || kv_mutual_bits)) return;  // size pass only
  // clear bit vectors, fill padding tail
  for (int w = tid; w < words; w += SEG_THREADS) {
    if (kv_valid_bits) kv_valid_bits[(size_t)b * words + w] = 0u;
    if (kv_mutual_bits) kv_mutual_bits[(size_t)b * words + w] = 0u;
  }
  for (int t = T_b + tid; t < t_cap; t += SEG_THREADS) {
    size_t o = (size_t)b * t_cap + t;
    if (seg) seg[o] = -1;
    if (row_lo) row_lo[o] = 0;
    if (row_hi) row_hi[o] = 0;
    if (src) src[o] = INT_MIN;
  }
  __syncthreads();
  // pass 3: scatter every token to its spliced position
  int carry = 0;
  for (int c0 = 0; c0 < L; c0 += SEG_THREADS) {
    const int l = c0 + tid;
    const int64_t tok = (l < L) ? ids[l] : 0;
    const int is_img = (l < L) && (tok == media_id);
    int chunk_total;
    const int k = carry + block_exclusive_scan(is_img, warp_sums, chunk_total);
    carry += chunk_total;
    if (l >= L) continue;
    const int pos = l + k * (N - 1);
    if (!is_img) {
      if (pos < t_cap) {
        size_t o = (size_t)b * t_cap + pos;
        if (seg) seg[o] = 0;
        if (row_lo) row_lo[o] = 0;
        if (row_hi) row_hi[o] = 0;
        if (src) src[o] = l;
        // the reference drops key j where (1 - mask[j]).bool(), i.e. mask[j] != 1   (vlm.py:434-438)
        if (am[l] == 1) {
          if (kv_valid_bits) atomicOr(&kv_valid_bits[(size_t)b * words + (pos >> 5)], 1u << (pos & 31));
          if (kv_mutual_bits) atomicOr(&kv_mutual_bits[(size_t)b * words + (pos >> 5)], 1u << (pos & 31));
        }
      }
    } else {
      const int span_end = pos + N;
      const int lo = (q_end > span_end) ? span_end : 0;
      const int hi = (q_end > span_end) ? q_end : 0;
      for (int v = 0; v < N; ++v) {
        const int t = pos + v;
        if (t >= t_cap) break;
        size_t o = (size_t)b * t_cap + t;
        if (seg) seg[o] = k + 1;
        if (row_lo) row_lo[o] = lo;
        if (row_hi) row_hi[o] = hi;
        if (src) src[o] = -1 - (k * N + v);
        if (kv_valid_bits) atomicOr(&kv_valid_bits[(size_t)b * words + (t >> 5)], 1u << (t & 31));
        if (kv_mutual_bits && !text_only) atomicOr(&kv_mutual_bits[(size_t)b * words + (t >> 5)], 1u << (t & 31));
      }
    }
  }
}

__global__ void __launch_bounds__(128)
tile_bounds_kernel(const int32_t* __restrict__ seq_len, const int32_t* __restrict__ row_lo,
                   const int32_t* __restrict__ row_hi, int T, int q_off, int t_cap, int n_tiles, int n_words,
                   int32_t* __restrict__ q_tile_kv_end, uint32_t* __restrict__ kv_tile_q_mask) {
  const int tile = blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
  const int len = min(seq_len[b], q_off + T);     // key coordinates; the query rows are [q_off, q_off + T)
  const int32_t* lo = row_lo + (size_t)b * t_cap;
  const int32_t* hi = row_hi + (size_t)b * t_cap;
  __shared__ int s_max;
  __shared__ uint32_t s_mask[64];   // up to 2048 tiles (T <= 262144)
  if (tid == 0) s_max = 0;
  for (int w = tid; w < n_words; w += 128) s_mask[w] = 0u;
  __syncthreads();
  const int r0 = tile * AKI_MMA_TILE;
  // query tile: how far right do its rows look
  int need = 0;
  const int i = q_off + r0 + tid;
  if (i < len) {
    need = i + 1;
    const int a = lo[i], e = hi[i];
    if (e > a) need = max(need, min(e, len));
  }
  atomicMax(&s_max, need);
  // key tile: which query tiles hold a row that sees any of its keys (q_off == 0: the host refuses the mask otherwise)
  if (kv_tile_q_mask && r0 < len) {
    const int j1 = min(r0 + AKI_MMA_TILE, len);
    const int n_live = (len + AKI_MMA_TILE - 1) / AKI_MMA_TILE;
    for (int qt = tile + tid; qt < n_live; qt += 128) atomicOr(&s_mask[qt >> 5], 1u << (qt & 31));  // causal part
    for (int r = tid; r < r0; r += 128) {                                                         // mutual part
      const int a = lo[r], e = hi[r];
      if (e > a && e > r0 && a < j1) atomicOr(&s_mask[(r / AKI_MMA_TILE) >> 5], 1u << ((r / AKI_MMA_TILE) & 31));
    }
  }
  __syncthreads();
  if (tid == 0 && q_tile_kv_end) q_tile_kv_end[(size_t)b * n_tiles + tile] = (s_max + AKI_MMA_TILE - 1) / AKI_MMA_TILE;
  if (kv_tile_q_mask)
    for (int w = tid; w < n_words; w += 128) kv_tile_q_mask[((size_t)b * n_tiles + tile) * n_words + w] = s_mask[w];
}

// Forward work plan (include/aki_mma.h, aki_mma_fwd_plan): one block per sample.  Query rows are cut into tiles of
// <= 128 rows that start at every image span (rows whose mutual interval [row_lo,row_hi) is non-empty and differs
// from the previous row's), each tile gets the number of 128-key tiles its rows can see, tiles are ranked by that
// count and paired.  O(T) integer work per sample; the result is shared by all heads and all layers.
constexpr int PLAN_THREADS = 256;
constexpr int PLAN_MAX_TILES = 1280;   // T <= 65536: 512 aligned tiles + span cuts
constexpr int PLAN_MAX_CUTS = 256;

__global__ void __launch_bounds__(PLAN_THREADS)
fwd_plan_kernel(const int32_t* __restrict__ seq_len, const int32_t* __restrict__ row_lo,
                const int32_t* __restrict__ row_hi, const uint32_t* __restrict__ vbits, int T, int q_off,
                int meta_pitch, int bits_pitch, int max_pairs, int flags, int4* __restrict__ plan) {
  // Rows are in key coordinates throughout: the query rows are [q_off, q_off + T) of q_off + T keys; the plan stores
  // tile starts relative to q_off.
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n_keys = q_off + T;
  const int len = seq_len ? min(seq_len[b], n_keys) : n_keys;
  const int32_t* lo = row_lo ? row_lo + (size_t)b * meta_pitch : nullptr;
  const int32_t* hi = row_hi ? row_hi + (size_t)b * meta_pitch : nullptr;
  __shared__ int s_first_bad, s_ncut, s_ntiles;
  __shared__ int s_cut[PLAN_MAX_CUTS + 2];
  __shared__ int s_cut_sorted[PLAN_MAX_CUTS + 2];
  __shared__ int s_seg_tile0[PLAN_MAX_CUTS + 2];
  __shared__ int s_start[PLAN_MAX_TILES], s_rows[PLAN_MAX_TILES], s_nkv[PLAN_MAX_TILES];
  __shared__ uint16_t s_order[PLAN_MAX_TILES];
  const int n_kt = (n_keys + AKI_MMA_TILE - 1) / AKI_MMA_TILE;
  if (tid == 0) { s_first_bad = n_kt; s_ncut = 0; }
  __syncthreads();
  // first 128-key tile that is not entirely inside the sequence and causally valid
  for (int kt = tid; kt < n_kt; kt += PLAN_THREADS) {
    bool bad = (kt * AKI_MMA_TILE + AKI_MMA_TILE > len);
    if (!bad && vbits) {
      const uint32_t* w = vbits + (size_t)b * bits_pitch + 4 * kt;
      bad = (w[0] & w[1] & w[2] & w[3]) != 0xffffffffu;
    }
    if (bad) atomicMin(&s_first_bad, kt);
  }
  // change points of the rows' mutual interval: a span STARTS where a row with a non-empty interval follows a row with
  // a different (or no) interval, and ENDS where a row without one follows
  const int n_aligned = (T + AKI_MMA_TILE - 1) / AKI_MMA_TILE;
  const int budget = min(max(2 * max_pairs - n_aligned - 1, 0), PLAN_MAX_CUTS);
  if ((flags & 1) && lo && budget > 0) {
    for (int i = q_off + 1 + tid; i < len; i += PLAN_THREADS) {
      const int a = lo[i], e = hi[i], a0 = lo[i - 1], e0 = hi[i - 1];
      const int id = (e > a) ? a : -1, id0 = (e0 > a0) ? a0 : -1;     // identity of the span a row belongs to
      if (id != id0) {
        const int k = atomicAdd(&s_ncut, 1);
        if (k < PLAN_MAX_CUTS) s_cut[k] = i;
      }
    }
  }
  __syncthreads();
  const int nchg = min(s_ncut, PLAN_MAX_CUTS);
  // rank sort of the change points (ascending) into s_seg_tile0 (scratch until the walk below)
  for (int k = tid; k < nchg; k += PLAN_THREADS) {
    const int v = s_cut[k];
    int rank = 0;
    for (int m = 0; m < nchg; ++m) rank += (s_cut[m] < v) ? 1 : 0;
    s_seg_tile0[rank] = v;
  }
  __syncthreads();
  if (tid == 0) {
    // Walk the change points and decide where the 128-row grid is cut.  Cutting at a span start p makes the span its
    // own query tile (only ONE tile walks the keys up to <|assistant|>) but leaves a short tile in front of p and puts
    // the following tiles off the 128-key grid (each then straddles one more key tile on its diagonal); cutting again
    // at the next multiple of 128 behind the span puts them back.  Each cut is taken only when the key-tile visits it
    // adds (unused rows of a short tile x the key tiles that tile visits) are fewer than those it saves.
    int nb = 0, prev = q_off;                  // boundaries so far (excluding q_off), last boundary
    s_cut_sorted[0] = q_off;
    if ((flags & 1) && prev % AKI_MMA_TILE != 0 && nb < budget) {
      // a continuation chunk that starts off the key-tile grid: a short first tile puts the following ones back on it
      const int G = (prev + AKI_MMA_TILE - 1) / AKI_MMA_TILE * AKI_MMA_TILE;
      const int next_chg = (nchg > 0) ? s_seg_tile0[0] : len;
      if (G < next_chg && G < len) {
        const int waste_realign = (AKI_MMA_TILE - (G - prev)) * (G / AKI_MMA_TILE);   // x 1/128, as below
        const int waste_stay = min(next_chg, len) - G;
        if (waste_realign < waste_stay) { s_cut_sorted[++nb] = G; prev = G; }
      }
    }
    for (int k = 0; k < nchg && nb < budget; ++k) {
      const int c = s_seg_tile0[k];
      const int a = lo[c], e = hi[c];
      const int off = (c - prev) % AKI_MMA_TILE;               // rows of the short tile a cut at c would leave behind
      if (e > a) {                                             // span start
        if (off != 0) {
          const int waste_cut = (AKI_MMA_TILE - off) * ((c + AKI_MMA_TILE - 1) / AKI_MMA_TILE);          // x 1/128
          const int waste_nocut = ((min(e, len) + AKI_MMA_TILE - 1) / AKI_MMA_TILE - (c + AKI_MMA_TILE - 1) / AKI_MMA_TILE) * AKI_MMA_TILE;
          if (waste_cut <= waste_nocut) { s_cut_sorted[++nb] = c; prev = c; }
        }
      } else if (prev % AKI_MMA_TILE != 0) {                   // span end on a grid that is off the key tiles: realign?
        const int G = (c + AKI_MMA_TILE - 1) / AKI_MMA_TILE * AKI_MMA_TILE;
        const int next_chg = (k + 1 < nchg) ? s_seg_tile0[k + 1] : len;
        if (G > c && G < next_chg && G < len) {
          const int r = (G - prev) % AKI_MMA_TILE;             // rows of the short tile in front of G
          const int waste_realign = (r == 0) ? 0 : (AKI_MMA_TILE - r) * (G / AKI_MMA_TILE);              // x 1/128
          const int waste_stay = (min(next_chg, len) - G);     // one more key tile for every later tile: x 1/128 too
          if (waste_realign < waste_stay) { s_cut_sorted[++nb] = G; prev = G; }
        }
      }
    }
    s_ncut = nb;
    s_cut_sorted[1 + nb] = n_keys;
    int n = 0;
    for (int k = 0; k <= nb; ++k) {
      s_seg_tile0[k] = n;
      n += (s_cut_sorted[k + 1] - s_cut_sorted[k] + AKI_MMA_TILE - 1) / AKI_MMA_TILE;
    }
    s_seg_tile0[nb + 1] = n;
    s_ntiles = n;
  }
  __syncthreads();
  const int ncut = s_ncut;
  const int n_tiles = s_ntiles;   // <= n_aligned + ncut <= 2 * max_pairs - 1
  // tiles of each segment
  for (int k = warp; k <= ncut; k += PLAN_THREADS / 32) {
    const int t0 = s_seg_tile0[k], cnt = s_seg_tile0[k + 1] - t0, r0 = s_cut_sorted[k], r1 = s_cut_sorted[k + 1];
    for (int x = lane; x < cnt; x += 32) {
      s_start[t0 + x] = r0 + x * AKI_MMA_TILE;
      s_rows[t0 + x] = min(AKI_MMA_TILE, r1 - (r0 + x * AKI_MMA_TILE));
    }
  }
  __syncthreads();
  // key tiles each query tile must visit: its rows look right up to max(i + 1, row_hi[i]) (clipped to the sequence)
  for (int x = warp; x < n_tiles; x += PLAN_THREADS / 32) {
    const int r0 = s_start[x], nr = s_rows[x];
    int need = 0;
    for (int r = lane; r < nr; r += 32) {
      const int i = r0 + r;
      if (i < len) {
        need = max(need, i + 1);
        if (lo) {
          const int a = lo[i], e = hi[i];
          if (e > a) need = max(need, min(e, len));
        }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) need = max(need, __shfl_xor_sync(0xffffffffu, need, o));
    if (lane == 0) s_nkv[x] = (need + AKI_MMA_TILE - 1) / AKI_MMA_TILE;
  }
  __syncthreads();
  // rank by key-tile count (descending; ties by start) -- or plain descending start (the causal order) without bit 1
  for (int x = tid; x < n_tiles; x += PLAN_THREADS) {
    int rank = 0;
    if (flags & 2) {
      const int nk = s_nkv[x], st = s_start[x];
      for (int y = 0; y < n_tiles; ++y) {
        const int nky = s_nkv[y];
        rank += (nky > nk || (nky == nk && s_start[y] < st)) ? 1 : 0;
      }
    } else {
      rank = n_tiles - 1 - x;
    }
    s_order[rank] = (uint16_t)x;
  }
  __syncthreads();
  const int n_pairs = (n_tiles + 1) / 2;
  int4* out = plan + (size_t)b * (1 + max_pairs);
  if (tid == 0) out[0] = make_int4(n_pairs, s_first_bad, n_tiles, 0);
  for (int p = tid; p < max_pairs; p += PLAN_THREADS) {
    int4 e = make_int4(0, 0, 0, 0);
    if (p < n_pairs) {
      const int x0 = s_order[2 * p];
      e.x = s_start[x0] - q_off; e.z = s_nkv[x0] | (s_rows[x0] << 16);
      if (2 * p + 1 < n_tiles) {
        const int x1 = s_order[2 * p + 1];
        e.y = s_start[x1] - q_off; e.w = s_nkv[x1] | (s_rows[x1] << 16);
      }
    }
    out[1 + p] = e;
  }
}

__global__ void __launch_bounds__(256)
expand_mask_kernel(const int32_t* __restrict__ seq_len, const int32_t* __restrict__ row_lo,
                   const int32_t* __restrict__ row_hi, const uint32_t* __restrict__ vbits,
                   const uint32_t* __restrict__ mbits, int T, int t_cap, int64_t* __restrict__ out) {
  const int b = blockIdx.z, i = blockIdx.y;
  const int j = blockIdx.x * 256 + threadIdx.x;
  if (j >= T) return;
  const int len = seq_len[b];
  const int words = (t_cap + 31) / 32;
  int64_t ok = 0;
  if (i < len && j < len) {
    const uint32_t vb = (vbits[(size_t)b * words + (j >> 5)] >> (j & 31)) & 1u;
    const uint32_t mb = (mbits[(size_t)b * words + (j >> 5)] >> (j & 31)) & 1u;
    const int lo = row_lo[(size_t)b * t_cap + i], hi = row_hi[(size_t)b * t_cap + i];
    ok = ((j <= i) && vb) || (j >= lo && j < hi && mb);
  }
  out[((size_t)b * T + i) * T + j] = ok;
}

__global__ void __launch_bounds__(128)
splice_kernel(const uint4* __restrict__ lang_embeds, const uint4* __restrict__ vision_tokens,
              const int64_t* __restrict__ labels_in, const int32_t* __restrict__ src,
              const int32_t* __restrict__ seq_len, int L, int N, int n_img_max, int E8, int T, int t_cap,
              uint32_t pad_pair, int pad_left, uint4* __restrict__ out, int64_t* __restrict__ labels_out) {
  const int t = blockIdx.x, b = blockIdx.y;
  const int len = min(seq_len[b], T);
  const int shift = pad_left ? (T - len) : 0;
  const int ts = t - shift;  // position in mask coordinates
  uint4* dst = out + ((size_t)b * T + t) * E8;
  const bool pad = (ts < 0 || ts >= len);
  const int s = pad ? INT_MIN : src[(size_t)b * t_cap + ts];
  if (s == INT_MIN) {
    const uint4 pv = make_uint4(pad_pair, pad_pair, pad_pair, pad_pair);
    for (int e = threadIdx.x; e < E8; e += 128) dst[e] = pv;
    if (labels_out && threadIdx.x == 0) labels_out[(size_t)b * T + t] = -100;
    return;
  }
  const uint4* from = (s >= 0) ? lang_embeds + ((size_t)b * L + s) * E8
                               : vision_tokens + ((size_t)b * n_img_max * N + (size_t)(-1 - s)) * E8;
  for (int e = threadIdx.x; e < E8; e += 128) dst[e] = from[e];
  if (labels_out && threadIdx.x == 0)
    labels_out[(size_t)b * T + t] = (s >= 0 && labels_in) ? labels_in[(size_t)b * L + s] : -100;
}

}  // namespace aki

using namespace aki;

extern "C" int aki_mma_segments(const int64_t* lang_x, const int64_t* attention_mask, int B, int L, int N,
                                int64_t media_token_id, int64_t assistant_token_id, int t_cap, int text_only,
                                int32_t* seq_len, int32_t* q_end, int32_t* seg, int32_t* row_lo, int32_t* row_hi,
                                int32_t* src, uint32_t* kv_valid_bits, uint32_t* kv_mutual_bits, int32_t* status,
                                aki_stream_t stream) {
  AKI_REQUIRE(lang_x && attention_mask && seq_len, AKI_ERR_NULL);
  AKI_REQUIRE(B > 0 && L > 0 && N > 0 && t_cap > 0, AKI_ERR_BAD_SHAPE);
  segments_kernel<<<B, SEG_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      lang_x, attention_mask, L, N, media_token_id, assistant_token_id, t_cap, text_only, seq_len, q_end, seg, row_lo,
      row_hi, src, kv_valid_bits, kv_mutual_bits, status);
  return check_launch();
}

extern "C" int aki_mma_tile_bounds_at(const int32_t* seq_len, const int32_t* row_lo, const int32_t* row_hi, int B,
                                      int T, int q_offset, int t_cap, int32_t* q_tile_kv_end, uint32_t* kv_tile_q_mask,
                                      aki_stream_t stream) {
  AKI_REQUIRE(seq_len && row_lo && row_hi, AKI_ERR_NULL);
  AKI_REQUIRE(B > 0 && T > 0 && q_offset >= 0 && (long long)q_offset + T <= INT_MAX, AKI_ERR_BAD_SHAPE);
  AKI_REQUIRE(t_cap >= q_offset + T, AKI_ERR_BAD_SHAPE);
  AKI_REQUIRE(q_offset == 0 || !kv_tile_q_mask, AKI_ERR_UNSUPPORTED);   // backward-only data: no continuation backward
  const int n_tiles = (T + AKI_MMA_TILE - 1) / AKI_MMA_TILE;
  const int n_words = (n_tiles + 31) / 32;
  AKI_REQUIRE(n_words <= 64, AKI_ERR_UNSUPPORTED);
  tile_bounds_kernel<<<dim3(n_tiles, B), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      seq_len, row_lo, row_hi, T, q_offset, t_cap, n_tiles, n_words, q_tile_kv_end, kv_tile_q_mask);
  return check_launch();
}

extern "C" int aki_mma_tile_bounds(const int32_t* seq_len, const int32_t* row_lo, const int32_t* row_hi, int B, int T,
                                   int t_cap, int32_t* q_tile_kv_end, uint32_t* kv_tile_q_mask, aki_stream_t stream) {
  return aki_mma_tile_bounds_at(seq_len, row_lo, row_hi, B, T, 0, t_cap, q_tile_kv_end, kv_tile_q_mask, stream);
}

extern "C" int aki_mma_fwd_plan_at(const int32_t* seq_len, const int32_t* row_lo, const int32_t* row_hi,
                                   const uint32_t* kv_valid_bits, int B, int T, int q_offset, int meta_pitch,
                                   int bits_pitch, int max_pairs, int flags, int32_t* plan, aki_stream_t stream) {
  AKI_REQUIRE(plan, AKI_ERR_NULL);
  AKI_REQUIRE((row_lo == nullptr) == (row_hi == nullptr), AKI_ERR_NULL);
  AKI_REQUIRE(B > 0 && T > 0 && q_offset >= 0 && (long long)q_offset + T <= INT_MAX, AKI_ERR_BAD_SHAPE);
  const int n_keys = q_offset + T;
  const int n_aligned = (T + AKI_MMA_TILE - 1) / AKI_MMA_TILE;
  AKI_REQUIRE(max_pairs >= (n_aligned + 1) / 2, AKI_ERR_BAD_SHAPE);
  AKI_REQUIRE(2 * max_pairs <= PLAN_MAX_TILES, AKI_ERR_UNSUPPORTED);
  AKI_REQUIRE(!row_lo || meta_pitch >= n_keys, AKI_ERR_BAD_SHAPE);
  AKI_REQUIRE(!kv_valid_bits || (long long)bits_pitch * 32 >= n_keys, AKI_ERR_BAD_SHAPE);
  AKI_REQUIRE(aligned16(plan), AKI_ERR_MISALIGNED);
  fwd_plan_kernel<<<B, PLAN_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      seq_len, row_lo, row_hi, kv_valid_bits, T, q_offset, meta_pitch, bits_pitch, max_pairs, flags,
      reinterpret_cast<int4*>(plan));
  return check_launch();
}

extern "C" int aki_mma_fwd_plan(const int32_t* seq_len, const int32_t* row_lo, const int32_t* row_hi,
                                const uint32_t* kv_valid_bits, int B, int T, int meta_pitch, int bits_pitch,
                                int max_pairs, int flags, int32_t* plan, aki_stream_t stream) {
  return aki_mma_fwd_plan_at(seq_len, row_lo, row_hi, kv_valid_bits, B, T, 0, meta_pitch, bits_pitch, max_pairs, flags,
                             plan, stream);
}

extern "C" int aki_mma_expand_mask(const int32_t* seq_len, const int32_t* row_lo, const int32_t* row_hi,
                                   const uint32_t* kv_valid_bits, const uint32_t* kv_mutual_bits, int B, int T,
                                   int t_cap, int64_t* mask4d, aki_stream_t stream) {
  AKI_REQUIRE(seq_len && row_lo && row_hi && kv_valid_bits && kv_mutual_bits && mask4d, AKI_ERR_NULL);
  AKI_REQUIRE(B > 0 && T > 0 && t_cap >= T && T <= 65535, AKI_ERR_BAD_SHAPE);
  expand_mask_kernel<<<dim3((T + 255) / 256, T, B), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      seq_len, row_lo, row_hi, kv_valid_bits, kv_mutual_bits, T, t_cap, mask4d);
  return check_launch();
}

extern "C" int aki_mma_splice(const void* lang_embeds, const void* vision_tokens, const int64_t* labels_in,
                              const int32_t* src, const int32_t* seq_len, int B, int L, int N, int n_img_max, int E,
                              int T, int t_cap, float pad_value, int pad_left, void* out_embeds, int64_t* labels_out,
                              aki_stream_t stream) {
  AKI_REQUIRE(lang_embeds && src && seq_len && out_embeds, AKI_ERR_NULL);
  AKI_REQUIRE(B > 0 && L > 0 && N > 0 && T > 0 && t_cap >= T && E > 0, AKI_ERR_BAD_SHAPE);
  AKI_REQUIRE(E % 8 == 0, AKI_ERR_UNSUPPORTED);
  AKI_REQUIRE(aligned16(lang_embeds) && aligned16(out_embeds) && (!vision_tokens || aligned16(vision_tokens)),
              AKI_ERR_MISALIGNED);
  __nv_bfloat16 pb = __float2bfloat16(pad_value);
  uint16_t bits;
  memcpy(&bits, &pb, 2);
  const uint32_t pair = (uint32_t)bits | ((uint32_t)bits << 16);
  splice_kernel<<<dim3(T, B), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint4*>(lang_embeds), static_cast<const uint4*>(vision_tokens), labels_in, src, seq_len, L, N,
      n_img_max, E / 8, T, t_cap, pair, pad_left, static_cast<uint4*>(out_embeds), labels_out);
  return check_launch();
}
