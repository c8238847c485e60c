/* aki_mma.h -- C ABI of libaki_mma.so: B200 (sm_100a) kernels for AKI's modality-mutual attention (MMA).
 *
 * This is the drop-in boundary for the one hot path of sony/aki: the attention inside the Phi-3.5-mini
 * decoder layers, where the reference materialises a (B,1,T,T) int64 0/1 mask
 * (codes/open_flamingo/src/vlm.py:410-443, :445-603; utils.py:99-108), has transformers 4.41.2 turn it into
 * an additive fp32 mask and runs eager softmax(QK^T/sqrt(96) + mask) V (Phi-3 remote code).  Every entry
 * point below names the reference interface it replaces.
 *
 * Conventions
 *   - plain pointers + sizes; every pointer is a DEVICE pointer unless stated otherwise.
 *   - the caller allocates every buffer (outputs, workspace); the library never allocates or frees device
 *     memory and never synchronises the device.  All work is enqueued on `stream` (a cudaStream_t).
 *   - return value: AKI_OK (0) or a negative AkiStatus; no exceptions, no abort, no stdout.
 *   - stateless and re-entrant; one process per GPU.
 *   - bf16 tensors have a contiguous last dimension; strides are in ELEMENTS.
 *   - head_dim must be 96 (Phi-3.5-mini: 32 heads x 96); anything else returns AKI_ERR_UNSUPPORTED.
 */
#ifndef AKI_MMA_H_
#define AKI_MMA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AKI_MMA_ABI_VERSION 2
#define AKI_MMA_HEAD_DIM 96
#define AKI_MMA_TILE 128 /* query / key tile edge used by the attention kernels and by tile_bounds */

typedef void* aki_stream_t; /* cudaStream_t */

typedef enum AkiStatus {
  AKI_OK = 0,
  AKI_ERR_NULL = -1,        /* a required pointer is NULL */
  AKI_ERR_BAD_SHAPE = -2,   /* negative / zero / inconsistent sizes */
  AKI_ERR_UNSUPPORTED = -3, /* head_dim != 96, stride not a multiple of 8 elements, ... */
  AKI_ERR_MISALIGNED = -4,  /* pointer not 16-byte aligned */
  AKI_ERR_CUDA = -5,        /* CUDA runtime / driver error (launch, tensor-map encode) */
  AKI_ERR_NO_DEVICE = -6    /* no sm_100 device visible */
} AkiStatus;

int aki_mma_abi_version(void);
const char* aki_mma_strerror(int status);
/* Last CUDA error string seen by this thread (diagnostics for AKI_ERR_CUDA). Host pointer, never NULL. */
const char* aki_mma_last_cuda_error(void);

/* ------------------------------------------------------------------------------------------------------
 * (1) Segment metadata  -- replaces the per-sample Python loop of
 *     VLMWithLanguageStream._prepare_inputs_for_forward (vlm.py:486-577: torch.where for <image> and the
 *     first <|assistant|> id 32001, splice bookkeeping) and _make_modality_mutual_mask (vlm.py:410-443).
 *     Instead of a (B,1,T,T) int64 tensor it emits O(B*T) integers from which
 *        allowed(i,j) = i<len & j<len & ( (j<=i & valid[j]) | (row_lo[i]<=j<row_hi[i] & mutual_ok[j]) )
 *     reproduces the reference mask bit-for-bit (single image) and defines >=2 images per sample, which the
 *     reference cannot run (vlm.py:547-554 raises).  Mask coordinates are top-left aligned as in
 *     stack_with_padding_2D_attention (utils.py:99-108).
 *
 *     lang_x, attention_mask : (B, L) int64.   N = vision tokens per <image> (AKI: 144, aki.py:20).
 *     t_cap                  : row pitch of the (B, t_cap) outputs; must be >= max_b T_b
 *                              (T_b = L + n_img_b*(N-1)); entries t >= T_b are filled as padding.
 *     text_only              : 0 = "contiguous" (an image span sees every later key of another segment up to
 *                              and including <|assistant|>; == reference for one image), 1 = later TEXT keys only.
 *     outputs: seq_len (B) int32 = T_b | q_end (B) int32 = post-splice index of first <|assistant|> + 1, else 0
 *              seg (B,t_cap) int32: 0 text, k>=1 vision tokens of the k-th image, -1 padding
 *              row_lo,row_hi (B,t_cap) int32 | src (B,t_cap) int32: l>=0 text token, -1-(k*N+v) vision, INT32_MIN pad
 *              kv_valid_bits, kv_mutual_bits (B, ceil(t_cap/32)) uint32: bit j = key j visible causally /
 *              through the mutual block.   Any output pointer except seq_len may be NULL (skipped).
 *     status (1) int32, optional: set to 1 on device if some T_b > t_cap (outputs truncated). */
int aki_mma_segments(const int64_t* lang_x, const int64_t* attention_mask, int B, int L, int N,
                     int64_t media_token_id, int64_t assistant_token_id, int t_cap, int text_only,
                     int32_t* seq_len, int32_t* q_end, int32_t* seg, int32_t* row_lo, int32_t* row_hi,
                     int32_t* src, uint32_t* kv_valid_bits, uint32_t* kv_mutual_bits, int32_t* status,
                     aki_stream_t stream);

/* Per-tile visit lists for AKI_MMA_TILE-row tiles (derived data the attention kernels consume so that fully
 * masked tiles are never visited).  n_t = ceil(T/128), W = ceil(n_t/32):
 *   q_tile_kv_end  (B, n_t)    : number of key tiles query tile qt must visit (0 = tile is all padding); the
 *                                visible key tiles of a query tile are always the contiguous range [0, end)
 *   kv_tile_q_mask (B, n_t, W) : bit qt of row kt is set iff some live row of query tile qt sees some key of
 *                                key tile kt (backward: with MMA this set is NOT contiguous -- the image-row
 *                                tiles before the diagonal plus everything from the diagonal on) */
int aki_mma_tile_bounds(const int32_t* seq_len, const int32_t* row_lo, const int32_t* row_hi, int B, int T,
                        int t_cap, int32_t* q_tile_kv_end, uint32_t* kv_tile_q_mask, aki_stream_t stream);
/* Same for the T query rows [q_offset, q_offset + T) of a continuation (see AkiMmaAttnParams.q_offset): query tile qt
 * holds rows q_offset + [128 qt, 128 qt + 128) and q_tile_kv_end (B, ceil(T/128)) counts key tiles over
 * [0, q_offset + T).  t_cap >= q_offset + T.  kv_tile_q_mask (backward only) must be NULL when q_offset != 0.
 * aki_mma_tile_bounds(...) == aki_mma_tile_bounds_at(..., 0, ...). */
int aki_mma_tile_bounds_at(const int32_t* seq_len, const int32_t* row_lo, const int32_t* row_hi, int B, int T,
                           int q_offset, int t_cap, int32_t* q_tile_kv_end, uint32_t* kv_tile_q_mask,
                           aki_stream_t stream);

/* Forward work plan (ABI 2): the query rows of every sample cut into tiles of <= 128 rows that START at each image span
 * (so that a span of <= 128 vision tokens is ONE query tile instead of straddling two aligned ones -- with the
 * reference's 128/144-token spans an aligned tiling makes two tiles per span walk all keys up to <|assistant|>), each
 * with the number of 128-key tiles it must visit; tiles are ranked by that count and paired (two query tiles share
 * one stream of K/V tiles in the forward kernel), heaviest pair first -- the order the persistent forward CTAs consume.
 *   plan (B, 1 + max_pairs, 4) int32: row 0 = {n_pairs, first key tile that holds a padded / invalid key, n_tiles, 0};
 *   row 1+p = {start0, start1, n_kv0 | rows0 << 16, n_kv1 | rows1 << 16}.
 *   max_pairs >= ceil(ceil(T/128) / 2); every pair above that minimum lets two more spans start a tile of their own
 *   (spans beyond the budget keep the aligned cut: same results, more masked work).
 *   flags: bit 0 = cut at span starts, bit 1 = rank and pair by key-tile count (0: index order).  Default 3.
 * No reference counterpart: the reference materialises the (B,1,T,T) mask instead (vlm.py:410-443). */
int aki_mma_fwd_plan(const int32_t* seq_len, const int32_t* row_lo, const int32_t* row_hi,
                     const uint32_t* kv_valid_bits, int B, int T, int meta_pitch, int bits_pitch, int max_pairs,
                     int flags, int32_t* plan, aki_stream_t stream);
/* Plan of a continuation chunk (AkiMmaAttnParams.q_offset): cuts and pairs the T query rows [q_offset, q_offset + T)
 * and counts key tiles over [0, q_offset + T); the tile starts it stores are chunk rows (0 = first query).  When the
 * chunk starts off the 128-key grid, a first short tile realigns the following ones if that saves key-tile visits.
 * meta_pitch >= q_offset + T, bits_pitch >= ceil((q_offset + T) / 32); row 0's first-bad key tile is absolute.
 * aki_mma_fwd_plan(...) == aki_mma_fwd_plan_at(..., 0, ...). */
int aki_mma_fwd_plan_at(const int32_t* seq_len, const int32_t* row_lo, const int32_t* row_hi,
                        const uint32_t* kv_valid_bits, int B, int T, int q_offset, int meta_pitch, int bits_pitch,
                        int max_pairs, int flags, int32_t* plan, aki_stream_t stream);

/* Debug / parity helper: expand the compact description to the reference's (B,1,T,T) int64 0/1 tensor
 * (what _prepare_inputs_for_forward returns under "attention_mask", vlm.py:589-603). */
int aki_mma_expand_mask(const int32_t* seq_len, const int32_t* row_lo, const int32_t* row_hi,
                        const uint32_t* kv_valid_bits, const uint32_t* kv_mutual_bits, int B, int T, int t_cap,
                        int64_t* mask4d, aki_stream_t stream);

/* Splice ("next" row f-2): inputs_embeds / labels of vlm.py:516-588 as one gather driven by `src`.
 *   lang_embeds (B,L,E) bf16, vision_tokens (B,n_img_max,N,E) bf16, labels_in (B,L) int64 or NULL
 *   out_embeds (B,T,E) bf16, labels_out (B,T) int64 or NULL.  Padding rows: embeds = pad_value (the reference
 *   fills embedding rows with the scalar pad_token_id, vlm.py:584-588), labels = -100.
 *   pad_left != 0 shifts every sample right by T - T_b (padding_side="left", utils.py:62-96). */
int aki_mma_splice(const void* lang_embeds, const void* vision_tokens, const int64_t* labels_in,
                   const int32_t* src, const int32_t* seq_len, int B, int L, int N, int n_img_max, int E, int T,
                   int t_cap, float pad_value, int pad_left, void* out_embeds, int64_t* labels_out,
                   aki_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * (2) Phi-3 longrope tables -- replaces Phi3RotaryEmbedding.forward (remote code; installed equivalent
 *     models/phi3/modeling_phi3.py:118-131): cos/sin(pos * inv_freq) * attention_factor, fp32.
 *     position_ids (B,T) int64; inv_freq (D/2) fp32 (= 1/(ext_factor * theta^(2k/D)), the caller picks
 *     short/long factors as modeling_rope_utils.py:47-80 does); outputs cos,sin (B,T,D/2) fp32. */
int aki_mma_rope_table(const int64_t* position_ids, const float* inv_freq, float attention_factor, int B, int T,
                       int half_dim, float* cos_out, float* sin_out, aki_stream_t stream);

/* (3) RoPE + KV-cache write -- replaces apply_rotary_pos_emb on K and DynamicCache.update's torch.cat
 *     (modeling_phi3.py:248-251; KV contract vlm.py:463-468, aki_generation.py:45-47,80).
 *     Reads the packed projection qkv (B,T,3*H*D) bf16 (strides given), rotates K, and writes K (post-RoPE)
 *     and V into caches laid out (B,H,t_cap,D) at rows [past_len, past_len+T).  v_cache may be NULL (training:
 *     V is consumed in place).  q_rot (B,H,T,D) bf16 may be non-NULL to also emit rotated Q (decode path).
 *     cos/sin: (B or 1, T, D/2) fp32, rope_stride_b = 0 broadcasts over batch.
 *     t_cap (ABI 2) = rows per (b,h) of the caches: past_len + T > t_cap is AKI_ERR_BAD_SHAPE; with the device-resident
 *     length (_dev) a row at or beyond t_cap is dropped instead of landing in the next head's rows. */
int aki_mma_rope_kv_write(const void* qkv, int64_t qkv_stride_b, int64_t qkv_stride_t, const float* cos,
                          const float* sin, int64_t rope_stride_b, int B, int T, int H, int D, void* k_cache,
                          void* v_cache, int64_t cache_stride_b, int64_t cache_stride_h, int past_len, int t_cap,
                          void* q_rot, aki_stream_t stream);
/* Same, with the past length read from DEVICE memory (past_len_dev (B) int32, one per sequence): the decode step can
 * then be captured in a CUDA graph and replayed while the cache grows (aki_generation.py:72-84 derives the position
 * from past_key_values[0][0].shape[2] on the host every step). */
int aki_mma_rope_kv_write_dev(const void* qkv, int64_t qkv_stride_b, int64_t qkv_stride_t, const float* cos,
                              const float* sin, int64_t rope_stride_b, int B, int T, int H, int D, void* k_cache,
                              void* v_cache, int64_t cache_stride_b, int64_t cache_stride_h,
                              const int32_t* past_len_dev, int t_cap, void* q_rot, aki_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * (4) Attention core -- replaces the eager path of Phi3Attention.forward: QK^T/sqrt(D) + additive mask,
 *     softmax in fp32, P V (modeling_phi3.py:153-175) together with the 4-D mask inversion of transformers
 *     4.41.2 (_prepare_4d_causal_attention_mask) -- no mask is read from HBM, the predicate is evaluated per
 *     128x128 tile from row_lo/row_hi and the two key bit-vectors.
 *     Rows with no visible key (batch padding) produce zeros (the reference produces a uniform average over
 *     all keys; see DESIGN.md "fully masked rows"). */
typedef struct AkiMmaTensor4 { /* logical (B, T, H, D) bf16 view, last dim contiguous */
  void* ptr;
  int64_t stride_b, stride_t, stride_h; /* elements; multiples of 8 */
} AkiMmaTensor4;

typedef struct AkiMmaAttnParams {
  int32_t B, H, T, D; /* T queries against q_offset + T keys (q_offset = 0: prefill / training); D == 96 */
  float scale;        /* softmax scale, 1/sqrt(96) */
  AkiMmaTensor4 q;    /* (B,T,H,D); pre-RoPE if rope_cos != NULL, else used as is */
  AkiMmaTensor4 k;    /* (B,q_offset+T,H,D) post-RoPE keys (cache layout or any strided view) */
  AkiMmaTensor4 v;    /* (B,q_offset+T,H,D) */
  AkiMmaTensor4 o;    /* output, (B,T,H,D) view */
  float* lse;         /* (B,H,T) fp32 natural-log sum-exp of scaled scores; may be NULL (inference) */
  const float* rope_cos; /* (B or 1, T, D/2) fp32 or NULL: rotate Q while loading it (row r of the table = query r) */
  const float* rope_sin;
  int64_t rope_stride_b;
  /* MMA description in KEY coordinates (row i of the metadata = absolute row i of the q_offset + T key sequence; query r
   * is absolute row q_offset + r; rows below q_offset are never read); all NULL => plain causal over the keys.
   * seq_len <= q_offset + T, meta_pitch >= q_offset + T, bits_pitch >= ceil((q_offset + T) / 32). */
  const int32_t* seq_len;          /* (B) */
  const int32_t* row_lo;           /* (B, meta_pitch) */
  const int32_t* row_hi;           /* (B, meta_pitch) */
  const uint32_t* kv_valid_bits;   /* (B, bits_pitch) */
  const uint32_t* kv_mutual_bits;  /* (B, bits_pitch) */
  const int32_t* q_tile_kv_end;    /* (B, ceil(T/128)): key tiles of each 128-row QUERY tile (aki_mma_tile_bounds_at) */
  const uint32_t* kv_tile_q_mask;  /* (B, ceil(T/128), ceil(ceil(T/128)/32)); backward only */
  int32_t meta_pitch, bits_pitch;
  /* ABI 2: forward work plan from aki_mma_fwd_plan ((B, 1 + plan_pairs) x 4 int32), or NULL: aligned 128-row query
   * tiles in index order (and, when seq_len / kv_valid_bits are given without a plan, every key tile is evaluated
   * against the predicate -- correct, slower). */
  const int32_t* fwd_plan;
  int32_t plan_pairs;
  /* Continuation onto a KV cache (follow-up turn, chunked prefill): the T queries are rows [q_offset, q_offset + T) of
   * the key sequence.  q, o, lse and the RoPE tables have T rows; k, v and the metadata above cover q_offset + T rows
   * (a plan from aki_mma_fwd_plan_at, kv ends from aki_mma_tile_bounds_at with the same q_offset).  0 = prefill.
   * q_offset < 0 or q_offset + T > INT32_MAX: AKI_ERR_BAD_SHAPE.  The backward refuses q_offset != 0
   * (AKI_ERR_UNSUPPORTED): training never continues onto a cache. */
  int32_t q_offset;
} AkiMmaAttnParams;

int aki_mma_attn_fwd(const AkiMmaAttnParams* p, aki_stream_t stream);

typedef struct AkiMmaAttnBwdParams {
  AkiMmaAttnParams fwd;   /* same q/k/v/o/lse/metadata as the forward call (lse required) */
  AkiMmaTensor4 d_o;      /* (B,T,H,D) bf16 */
  AkiMmaTensor4 d_q;      /* outputs; gradients w.r.t. the PRE-RoPE q / k when rope tables are given */
  AkiMmaTensor4 d_k;
  AkiMmaTensor4 d_v;
  void* workspace;        /* aki_mma_attn_bwd_workspace_bytes() bytes, 256-byte aligned */
  size_t workspace_bytes;
  int32_t deterministic;  /* must be 0: dQ partial sums of the key tiles are added with fp32 reductions in L2 (order varies
                             from run to run, last-bit differences in dQ); anything else returns AKI_ERR_UNSUPPORTED */
} AkiMmaAttnBwdParams;

size_t aki_mma_attn_bwd_workspace_bytes(int B, int H, int T, int D);
int aki_mma_attn_bwd(const AkiMmaAttnBwdParams* p, aki_stream_t stream);

/* (5) Decode -- the generate loop after prefill (aki_generation.py:56-84): a 2-D all-ones mask, i.e. one
 *     query per sequence sees every cached key [0, kv_len[b]).  Memory-bound split-KV kernel.
 *     q (B,H,D) bf16 post-RoPE; caches (B,H,t_cap,D); out (B,H,D) bf16; workspace from
 *     aki_mma_decode_workspace_bytes(). kv_len (B) int32 device array.  kv_start (B) int32 device array or NULL (ABI 2):
 *     first visible key of each sequence -- the leading pad rows of a left-padded prompt (padding_side="left",
 *     aki.py:172-182) stay in the cache and must not be attended (the reference's 2-D mask zeroes them). */
size_t aki_mma_decode_workspace_bytes(int B, int H, int D, int max_kv_len);
int aki_mma_decode(const void* q, const void* k_cache, const void* v_cache, int64_t cache_stride_b,
                   int64_t cache_stride_h, const int32_t* kv_len, const int32_t* kv_start, int max_kv_len, int B, int H,
                   int D, float scale, void* out, void* workspace, size_t workspace_bytes, aki_stream_t stream);
/* Same, skipping every key whose bit in kv_valid_bits (B, bits_pitch) uint32 is 0 (bit j of word j/32 = key j): a
 * batched follow-up turn appends left-padded prompts, so the cache holds invalid rows in its interior, which kv_start
 * cannot describe.  bits_pitch * 32 >= max_kv_len.  kv_valid_bits = NULL: aki_mma_decode. */
int aki_mma_decode_masked(const void* q, const void* k_cache, const void* v_cache, int64_t cache_stride_b,
                          int64_t cache_stride_h, const int32_t* kv_len, const int32_t* kv_start,
                          const uint32_t* kv_valid_bits, int bits_pitch, int max_kv_len, int B, int H, int D, float scale,
                          void* out, void* workspace, size_t workspace_bytes, aki_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * (6) Decode-sized linear layers around the attention op (SURVEY 8 f-1, ABI 2) -- for B <= 8 tokens (one per sequence of
 *     a decode step) replaces Phi3RMSNorm.forward + nn.Linear + the SiLU gate of Phi3MLP + the residual adds of
 *     Phi3DecoderLayer.forward (transformers/models/phi3/modeling_phi3.py:49-64, 295-335):
 *        y (B,N) = epilogue( prologue(x) (B,K) . W (N,K)^T )         bf16 in / out, fp32 accumulation, W row-major
 *     rms_weight (K) bf16 or NULL: RMSNorm prologue with HF's rounding points ((x * rsqrt(mean x^2 + eps)).bf16 * weight)
 *     mode 0: store | 1: y = residual + (.) (residual (B,N) bf16) | 2: SwiGLU, W has 2N rows (gate rows [0,N), up rows
 *     [N,2N) as gate_up_proj stores them), y = up * silu(gate).
 *     N % 16 == 0; K % 1024 == 0; strides in elements.  HBM-bound: N*K*2 bytes per call. */
int aki_mma_skinny_linear(const void* x, int64_t x_stride, const void* w, const void* rms_weight, float rms_eps,
                          const void* residual, int64_t residual_stride, void* y, int64_t y_stride, int B, int N, int K,
                          int mode, aki_stream_t stream);
/* Same contract, argument for argument, for 1 <= B <= 64 tokens (a batched decode step), on tcgen05 tensor cores: the
 * weights stream through a TMA ring, the K range of each 128-row tile is split over a cluster of CTAs and reduced in a
 * fixed order through distributed shared memory (deterministic, no workspace).  N % 16 == 0; K % 64 == 0; x_stride
 * % 8 == 0 and x_stride >= K when B > 1; strides in elements.  Same status codes as aki_mma_skinny_linear.  Row b of the
 * output depends on B only through roundup(B, 16).  HBM-bound: N*K*2 bytes per call (x2 in mode 2).
 * aki_mma_batch_linear_split: the number of CTAs (1 - 8) a call with these arguments splits K over, or a negative
 * status; needs a current device. */
int aki_mma_batch_linear(const void* x, int64_t x_stride, const void* w, const void* rms_weight, float rms_eps,
                         const void* residual, int64_t residual_stride, void* y, int64_t y_stride, int B, int N, int K,
                         int mode, aki_stream_t stream);
int aki_mma_batch_linear_split(int B, int N, int K, int mode);

/* ------------------------------------------------------------------------------------------------------
 * (7) Element-wise work of the decoder layer at PREFILL size (SURVEY 8 f-1, ABI 2) -- one pass over HBM each, replacing
 *     the ATen kernels of Phi3RMSNorm.forward, the residual adds of Phi3DecoderLayer.forward and the SiLU gate of
 *     Phi3MLP.forward (transformers/models/phi3/modeling_phi3.py:49-64, 295-306, 317-335); the GEMMs between them stay
 *     with the caller.  bf16 in / out, HF's rounding points; strides in elements (rows of M tokens).
 *     aki_mma_add_rmsnorm: h = residual + x (skipped when residual is NULL; written to h_out when non-NULL, h_out may
 *     alias residual), y = weight * (h * rsqrt(mean(h^2) + eps)).bf16.  K % 256 == 0, K <= 4096.
 *     aki_mma_swiglu: y (M,N) = up * silu(gate) with gate = gate_up[:, :N], up = gate_up[:, N:2N].  N % 8 == 0. */
int aki_mma_add_rmsnorm(const void* x, int64_t x_stride, const void* residual, int64_t residual_stride, const void* weight,
                        float eps, void* h_out, int64_t h_stride, void* y, int64_t y_stride, int M, int K,
                        aki_stream_t stream);
int aki_mma_swiglu(const void* gate_up, int64_t gate_up_stride, void* y, int64_t y_stride, int M, int N,
                   aki_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * (8) Next-token cross-entropy over the LM head's logits (SURVEY 8 f-2, ABI 2) -- the loss Phi3ForCausalLM(labels=...)
 *     hands AKI.forward (codes/open_flamingo/src/aki.py:125-130; HF: logits.float(), shift by one, CrossEntropyLoss with
 *     ignore_index): logits (B,T,V) bf16 (strides in elements), labels (B,T) int64.  Row (b,t) pairs with
 *     labels[b,t+1]; rows whose target is ignore_index (or t = T-1) contribute 0.
 *     fwd: row_loss, row_lse (B,T) fp32 = logsumexp - target logit, computed in fp32 from the bf16 logits.
 *     bwd: dlogits (B,T,V) bf16 = (softmax - onehot) * *scale_dev (device scalar: dloss / number of valid targets).
 *     V % 8 == 0.  HBM-bound: V*2 bytes per row forward, 2*V*2 backward. */
int aki_mma_cross_entropy_fwd(const void* logits, int64_t stride_b, int64_t stride_t, const int64_t* labels,
                              int64_t labels_stride_b, int B, int T, int V, long long ignore_index, float* row_loss,
                              float* row_lse, aki_stream_t stream);
int aki_mma_cross_entropy_bwd(const void* logits, int64_t stride_b, int64_t stride_t, const int64_t* labels,
                              int64_t labels_stride_b, int B, int T, int V, long long ignore_index, const float* row_lse,
                              const float* scale_dev, void* dlogits, int64_t d_stride_b, int64_t d_stride_t,
                              aki_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * (9) The element-wise work of (7) in the TRAINING layout of the reference's amp_bf16 precision (configs/sft.yaml:55;
 *     SURVEY 8 f-1 for the SFT step): fp32 residual stream and norm weights, bf16 GEMM operands; forward and backward.
 *     add_rmsnorm_amp_fwd: h_out = h_in + float(a) (a (M,K) bf16 = o_proj / down_proj output; a and h_out both NULL:
 *       no add), r_out (M) = rsqrt(mean(h^2) + eps), x (M,K) bf16 = bf16(weight * (h * r)) -- the residual add, the fp32
 *       Phi3RMSNorm and the autocast cast of the next Linear's input in one pass.  All rows contiguous.  K % 256 == 0,
 *       K <= 3072.
 *     rmsnorm_amp_bwd: dh (M,K) fp32 = dh_out (NULL = 0) + gradient of the norm w.r.t. h given dx (M,K) bf16;
 *       dw_partial (aki_mma_rmsnorm_amp_bwd_partials(M), K) fp32: per-warp partial sums of the weight gradient, to be
 *       summed over dim 0 by the caller (no atomics: deterministic).
 *     swiglu_bwd: d_gate_up (M,2N) bf16 from d_out (M,N) bf16 and gate_up (M,2N) bf16, with eager autograd's rounding
 *       points. */
int aki_mma_add_rmsnorm_amp_fwd(const float* h_in, const void* a, const float* weight, float eps, float* h_out, void* x,
                                float* r_out, int M, int K, aki_stream_t stream);
int aki_mma_rmsnorm_amp_bwd_partials(int M);
int aki_mma_rmsnorm_amp_bwd(const void* dx, const float* dh_out, const float* h, const float* r, const float* weight,
                            float* dh, float* dw_partial, int M, int K, aki_stream_t stream);
int aki_mma_swiglu_bwd(const void* d_out, const void* gate_up, void* d_gate_up, int M, int N, aki_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * (10) Optimizer step of the SFT loop -- replaces torch.nn.utils.clip_grad_norm_ + torch.optim.AdamW.step of the
 *      reference's training step (train_utils.py:143-158) and, through the bf16 parameter copy it writes, autocast's
 *      fp32 -> bf16 weight cast in every forward (configs/sft.yaml:55 amp_bf16).  Two HBM-bound passes over a list of
 *      fp32 tensors, given as a HOST array of entries (copied into the kernels' parameter space: no device table; longer
 *      lists than one launch takes are split into several launches by the library).  Every pointer is 16-byte aligned.
 *   aki_mma_grad_sq_norm: *sq_norm (device, 1 float) = sum of grad^2 over every entry.  Reads `grad` and `numel` only.
 *     Fixed-order reduction (fp32 partials of 16384 elements, added in fp64 in chunk order): the same inputs give the
 *     same bits on every run.  workspace: aki_mma_grad_sq_norm_workspace_bytes(t, n) bytes (0 for an invalid list).
 *   aki_mma_adamw_step: per element, with c = min(1, max_norm / (sqrt(*sq_norm) + 1e-6)) (c = 1 when sq_norm is NULL;
 *     a NaN norm gives c = NaN, an infinite one c = 0, as clip_grad_norm_ does):
 *       g = grad * c;  param -= lr * weight_decay * param;  exp_avg = lerp(exp_avg, g, 1 - beta1);
 *       exp_avg_sq = lerp(exp_avg_sq, g^2, 1 - beta2);
 *       param -= lr / (1 - beta1^step) * exp_avg / (sqrt(exp_avg_sq) / sqrt(1 - beta2^step) + eps)
 *     in the fp32 operations of torch.optim.AdamW(fused=True); then param_bf16 (when non-NULL) = bf16(param), rounded to
 *     nearest even like param.to(torch.bfloat16).  `grad` is NOT rescaled in place (clip_grad_norm_ rescales it).
 *     step >= 1 is the step count after this update; 0 <= beta < 1, lr, eps, weight_decay finite and >= 0, max_norm
 *     finite and > 0 when sq_norm is given; otherwise AKI_ERR_BAD_SHAPE.
 *   All status codes are returned before any launch: AKI_ERR_NULL (t, a required pointer of a non-empty entry,
 *   workspace, sq_norm), AKI_ERR_BAD_SHAPE (n <= 0, numel < 0, hyperparameters, workspace too small), AKI_ERR_MISALIGNED. */
typedef struct AkiAdamWTensor {
  float* param;
  const float* grad;
  float* exp_avg;
  float* exp_avg_sq;
  void* param_bf16;   /* bf16 copy written after the update, or NULL */
  int64_t numel;
} AkiAdamWTensor;

size_t aki_mma_grad_sq_norm_workspace_bytes(const AkiAdamWTensor* t, int n);
int aki_mma_grad_sq_norm(const AkiAdamWTensor* t, int n, void* workspace, size_t workspace_bytes, float* sq_norm,
                         aki_stream_t stream);
int aki_mma_adamw_step(const AkiAdamWTensor* t, int n, const float* sq_norm, float max_norm, float lr, float beta1,
                       float beta2, float eps, float weight_decay, int64_t step, aki_stream_t stream);

/* Measurement hook (bench.py roofline): the NEXT aki_mma_attn_fwd / aki_mma_attn_bwd call of this host thread
 * records `ev_begin` right before and `ev_end` right after its tcgen05 attention kernel on the call's stream (the
 * preprocess / memset / finalize launches of the backward stay outside), then the hook clears itself.
 * Both are cudaEvent_t created by the caller with timing enabled; pass NULL, NULL to cancel.  No reference
 * counterpart (the reference has no profiling hooks, SURVEY section 5). */
int aki_mma_set_timing_events(void* ev_begin, void* ev_end);
/* Number of CUDA kernels this library has enqueued since it was loaded (process-wide, all threads): bench.py reports
 * the difference over its timed region as "gpu_launches".  cudaMemsetAsync of the backward workspace is not a kernel of
 * this library and is not counted.  No reference counterpart. */
unsigned long long aki_mma_launch_count(void);

/* ------------------------------------------------------------------------------------------------------
 * Verification kernels (tests only): the same maths as (4) written as plain SIMT CUDA with no tensor cores,
 * used to cross-check the tcgen05 kernels on-device at sizes the CPU oracle cannot reach.  The forward honours
 * q_offset like aki_mma_attn_fwd; the backward refuses it. */
int aki_mma_attn_fwd_simt(const AkiMmaAttnParams* p, aki_stream_t stream);
int aki_mma_attn_bwd_simt(const AkiMmaAttnBwdParams* p, aki_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* AKI_MMA_H_ */
