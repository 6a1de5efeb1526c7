/*
 * b2l.h - C ABI of libb200llama.so: the B200 (sm_100a) quantized-decode path for
 * Lightning-AI/lit-llama.
 *
 * The reference has no native boundary of its own: its "operator API" for this path
 * is a set of Python nn.Module classes that lit_llama/utils.py:141-162 swaps in for
 * torch.nn.Linear, plus the model-level modules of lit_llama/model.py.  Each entry
 * point below states the reference forward it replaces (file:line relative to the
 * reference checkout).  INTEGRATION.md shows the ctypes binding a maintainer adds.
 *
 * Conventions
 *  - Every pointer is a DEVICE pointer owned by the caller (PyTorch).  The library
 *    never allocates or frees device memory on the call path and never synchronises;
 *    every call only enqueues work on `stream` and is CUDA-graph capturable.
 *  - Return value: 0 = ok, <0 = bad argument / unsupported shape (B2L_E_*),
 *    >0 = a cudaError_t.  b2l_last_error() returns a thread-local message.
 *  - There is no CPU fallback.
 *  - Activations are bf16 (B2L_BF16).  Scales/zeros may be bf16 or f32 (the
 *    reference creates them in the default dtype, quantization.py:360-369).
 */
#ifndef B2L_H_
#define B2L_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* b2l_stream_t; /* == cudaStream_t */

enum { B2L_BF16 = 0, B2L_F32 = 1 };

enum {
  B2L_E_ARG = -1,         /* null pointer / negative size / misaligned pointer      */
  B2L_E_UNSUPPORTED = -2, /* shape or mode outside what the kernels implement        */
  B2L_E_STATE = -3        /* call sequence error (e.g. model not finalised)          */
};

int b2l_version(void);
const char* b2l_last_error(void);
/* Device facts the host side sizes grids with (SM count etc.).  0 on success. */
int b2l_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ------------------------------------------------------------------------------
 * ColBlockQuantizedLinear  (lit_llama/quantization.py:340-423)
 *
 * Reference storage (quantization.py:350-369, 386-390): quant_weight is uint8, logical
 * (out, in/epb) with strides (1, out) - i.e. memory is row-major (in/epb, out) - and
 * entry nr of byte [o, j] holds column epb*j+nr at bit nr*bits.  scales/zeros are
 * (out, n_groups) row-major, n_groups = ceil(in / tile_cols).
 * ---------------------------------------------------------------------------- */

/* get_weight(): dense (out, in) row-major weight, (level - zero) * scale evaluated in
 * out_dtype like quantization.py:392-411 (bit-exact with the reference). */
int b2l_q_dequant(const void* qw, const void* scales, const void* zeros, int sz_dtype,
                  void* w_out, int out_dtype, int out_features, int in_features, int bits,
                  int tile_cols, b2l_stream_t stream);

/* forward(): y[M,N] = x[M,K] @ dequant(W)^T (+ bias).  Generic kernel: any bits in
 * {4,8}, any tile_cols, any M; reads the reference layout directly.  Replaces both
 * branches of quantization.py:413-423 (the Triton kernel :187-333 and the dense
 * fallback).  x, y bf16 row-major with leading dimensions ldx, ldy (elements). */
int b2l_q_linear(const void* x, int ldx, const void* qw, const void* scales, const void* zeros,
                 int sz_dtype, const void* bias, void* y, int ldy, int M, int N, int K, int bits,
                 int tile_cols, b2l_stream_t stream);

/* One-time (load-time) re-tiling of a 4-bit, one-group-per-row weight for the
 * tcgen05 kernel: [N/128 tiles][K/32 slabs][128 rows][16 B].  N is padded up to a
 * multiple of 128 with zero levels.  Pure permutation of nibbles (bit-exact,
 * invertible: b2l_q4_untile).  Precedent for load-time transforms in the
 * reference: Linear8bitLt._load_from_state_dict, quantization.py:52-67. */
size_t b2l_q4_tiled_bytes(int N, int K);
int b2l_q4_tile(const void* qw, void* qw_tiled, int N, int K, b2l_stream_t stream);
int b2l_q4_untile(const void* qw_tiled, void* qw, int N, int K, b2l_stream_t stream);

/* Prologue / epilogue selectors of the fused tcgen05 linear. */
enum { B2L_PRO_NONE = 0, B2L_PRO_RMSNORM = 1 };
enum {
  B2L_EPI_STORE = 0,    /* y = bf16(acc)                                              */
  B2L_EPI_RESIDUAL = 1, /* y = bf16(bf16(acc) + res)            model.py:166-167       */
  B2L_EPI_SWIGLU = 2    /* rows interleaved [64 of c_fc1 | 64 of c_fc2] per tile:
                           y = bf16(bf16(silu(bf16(a))) * bf16(b))   model.py:252     */
};

#define B2L_PF_SEGMENTS 4
typedef struct b2l_q4_linear_args {
  const void* x;        /* bf16 [M, K], leading dim ldx                               */
  int ldx;
  const void* qw_tiled; /* from b2l_q4_tile                                           */
  const void* scales;   /* [N] per-row                                                */
  const void* zeros;    /* [N]                                                        */
  int sz_dtype;
  void* y;              /* bf16 [M, N_out], leading dim ldy (N_out = N/2 for SWIGLU)  */
  int ldy;
  int M, N, K;          /* M <= 16; N % 128 == 0 after padding; K % 32 == 0           */
  int prologue;         /* B2L_PRO_*                                                  */
  const void* norm_scale; /* bf16 [K] RMSNorm scale when prologue == RMSNORM          */
  float eps;
  int epilogue;         /* B2L_EPI_*                                                  */
  const void* res;      /* bf16 [M, N] residual (leading dim ldres) for RESIDUAL      */
  int ldres;
  int split_k;          /* cluster size along K: 1..8 (0 = library picks)             */
  int flags;            /* B2L_F_*                                                    */
  void* trace;          /* debug: device uint64[256] receiving clock64() stamps of CTA 0
                           (NULL = off); see tools/diag.py `trace`                     */
  void* workspace;      /* b2l_q4_gemv_batch only: b2l_q4_gemv_batch_workspace_bytes(K) bytes of device
                           scratch, 16-byte aligned (activation fragments; may be shared by all
                           launches of one stream)                                       */
  const void* pf_ptr[B2L_PF_SEGMENTS];          /* b2l_q4_gemv only, L2 prefetch hint: byte ranges (16-byte aligned,
                           multiples of 16; NULL / 0 = unused) that LATER launches will stream - typically the
                           weights of the next linears.  The CTAs ask the L2 for them as soon as their own
                           weight ring is full, so HBM keeps streaming while this launch waits for its
                           activations, reduces and writes its result (the reference has no counterpart:
                           quantization.py:284-333 launches one Triton kernel per linear)          */
  unsigned long long pf_bytes[B2L_PF_SEGMENTS];
  /* strided form of the same hint - the KV-cache rows a later b2l_attention launch reads (model.py:211-222):
     pf_nseg ranges, pf_seg_stride bytes apart, at each of pf_kv[0] and pf_kv[1]; every range is
     rows * pf_row_bytes bytes long, rows = min(*pf_rows, pf_rows_max) read ON THE DEVICE when the launch runs
     (pf_rows = the step's input_pos).  pf_kv[0] == NULL: unused                                           */
  const void* pf_kv[2];
  const long long* pf_rows;
  int pf_rows_max, pf_nseg, pf_row_bytes;
  unsigned long long pf_seg_stride;
} b2l_q4_linear_args;

enum {
  B2L_F_PDL = 1,        /* launch with programmatic dependent launch                   */
  B2L_F_NO_ALIAS_N = 2, /* debug: do not alias B operand rows 8..15 onto rows 0..7     */
  B2L_F_ROPE_ROWS = 4,  /* b2l_attention: `rope` holds the T rows already selected by
                           input_pos (the reference's call convention, model.py:93)    */
  B2L_F_ATTN_UNFUSED = 8, /* debug: force the three-kernel attention path for T == 1   */
  B2L_F_DEBUG_NOCOMPUTE = 16 /* debug: b2l_q4_gemv streams the weights but skips the math */
};

/* Fused [RMSNorm ->] int4 linear [-> residual | SwiGLU] on tcgen05.  Replaces
 * RMSNorm.forward (model.py:270-277) + ColBlockQuantizedLinear.forward
 * (quantization.py:413-423) + the residual add / silu*mul of Block/MLP.forward
 * (model.py:166-167, 252). */
int b2l_q4_linear_tc(const b2l_q4_linear_args* args, b2l_stream_t stream);

/* Prefill-shaped linear (any M; meant for M > 16): y[M, N] = x[M, K] . dequant(W)^T on tcgen05 (csrc/q4_gemm.cu):
 * 256 x 256 output tile per CTA, both operands from shared memory (producer warps dequantise the packed levels with
 * the reference's own bf16 roundings, so the tensor core multiplies exactly get_weight()'s matrix), fp32 accumulators
 * in tensor memory.  Same argument block as b2l_q4_linear_tc; qw_tiled from b2l_q4_tile; prologue / epilogue must be
 * NONE / STORE; K % 64 == 0; ldx % 8 == 0.  Replaces quantization.py:187-333 (Triton tile kernel) / :413-423. */
int b2l_q4_gemm(const b2l_q4_linear_args* args, b2l_stream_t stream);

/* Batch-1 decode variant of the fused linear (M == 1): TMA-staged packed weights, PDL prefetch, persistent CTAs
 * that own 16-row blocks over the full K (no cross-CTA reduction), and an EXACT integer contraction on the legacy
 * tensor pipe: the activation row is scaled by a power of two and split into balanced base-256 digits, digit plane j
 * is column j of mma.sync.m16n8k32 (u8 x s8 -> s32), a packed byte feeds two weight rows (csrc/q4_gemv.cu).
 * Same argument block as b2l_q4_linear_tc (ldx/ldy/ldres unused; split_k > 0 overrides the grid size);
 * qw_tiled must come from b2l_q4_tile_i8: [N/16 row blocks][K/64 k blocks][32 lanes][16 B], byte = level of row g
 * (low nibble) and of row g + 8 (high nibble).  For B2L_EPI_SWIGLU the rows of a 16-row block are
 * [8 of c_fc1 | 8 of c_fc2].  K % 64 == 0, K <= 24576. */
size_t b2l_q4_tiled_i8_bytes(int N, int K);
int b2l_q4_tile_i8(const void* qw, void* qw_tiled, int N, int K, b2l_stream_t stream);
int b2l_q4_untile_i8(const void* qw_tiled, void* qw, int N, int K, b2l_stream_t stream);
int b2l_q4_gemv(const b2l_q4_linear_args* args, b2l_stream_t stream);

/* The same fused linear for 1..8 activation rows (batched decode) on mma.sync.m16n8k16 (f16), weight tiling
 * b2l_q4_tile_mma ([N/16 row blocks][K/64 k blocks][32 lanes][16 B] in m16n8k16 A-fragment order), argument block of
 * b2l_q4_gemv plus `workspace`; x [M, K] with leading dimension ldx (ldx % 8 == 0), y / res
 * with ldy / ldres.  An mma.m16n8k16 tile has 8 columns: activation row n is column n, so 8 rows cost the MMAs
 * of one.  Two launches: the rows are normalised and converted to MMA fragment order once
 * (q4_batch_prep_kernel), then streamed stage by stage next to the weights (q4_gemv_batch_kernel).
 * Replaces the same reference code as b2l_q4_gemv for B > 1 (model.py:76-122 accepts any batch). */
size_t b2l_q4_gemv_batch_workspace_bytes(int K);
size_t b2l_q4_tiled_mma_bytes(int N, int K);
int b2l_q4_tile_mma(const void* qw, void* qw_tiled, int N, int K, b2l_stream_t stream);
int b2l_q4_untile_mma(const void* qw_tiled, void* qw, int N, int K, b2l_stream_t stream);
int b2l_q4_gemv_batch(const b2l_q4_linear_args* args, b2l_stream_t stream);

/* ------------------------------------------------------------------------------
 * model.py element-wise pieces (used by the module-level drop-ins and by prefill)
 * ---------------------------------------------------------------------------- */

/* RMSNorm.forward, model.py:270-277, evaluated with the reference's bf16 rounding
 * points.  x, y bf16 [rows, C]. */
int b2l_rmsnorm(const void* x, const void* scale, void* y, int rows, int C, float eps,
                b2l_stream_t stream);

/* transformer.wte(idx), model.py:102.  idx int32 or int64 [n]; out bf16 [n, C]. */
int b2l_embedding(const void* idx, int idx_is_i64, const void* wte, void* out, int n, int C,
                  int vocab, b2l_stream_t stream);

/* silu(a) * b with the reference's bf16 rounding points, model.py:252. */
int b2l_silu_mul(const void* a, const void* b, void* y, size_t n, b2l_stream_t stream);

/* x + h, model.py:166-167. */
int b2l_add(const void* a, const void* b, void* y, size_t n, b2l_stream_t stream);

/* ------------------------------------------------------------------------------
 * Linear8bitLt  (lit_llama/quantization.py:38-77; forward inherited from bitsandbytes:
 * LLM.int8() with has_fp16_weights=False, threshold=6.0).  CB int8 (out, in) row-major,
 * SCB fp32 (out) as produced by quantization.py:69-77.
 * ---------------------------------------------------------------------------- */
/* load-time re-tiling of CB into mma.m16n8k32 fragment order: [N/16][K/128][4][32 lanes][16 B] */
size_t b2l_q8_tiled_bytes(int N, int K);
int b2l_q8_tile(const void* cb, void* tiled, int N, int K, b2l_stream_t stream);
/* y[N] (bf16) for ONE activation row x[K] (bf16): fp16 cast, outlier columns (|a| >= threshold)
 * in fp16 against CB*SCB/127, the rest row-absmax-quantised to int8 and contracted on the tensor
 * cores, dequantised by SCA*SCB/127^2.  outlier_mask: optional K-bit mask shared by a batch
 * (b2l_q8_outlier_mask); NULL = derive it from this row. */
int b2l_q8_gemv(const void* x, const void* w_tiled, const void* cb, const void* scb,
                const void* outlier_mask, void* y, int N, int K, float threshold, int flags,
                b2l_stream_t stream);
int b2l_q8_outlier_mask(const void* x, int ldx, int M, int K, float threshold, void* mask,
                        b2l_stream_t stream);

/* generate.py:68-75 up to the probabilities: probs = softmax(where(l < kth, -inf, l)) with
 * l = logits / temperature (bf16, rounded like ATen does on the GPU) and kth the top_k-th
 * largest l (top_k == 0: no filtering).  logits, probs bf16 [V].  One launch; the caller draws
 * with torch.multinomial so the RNG stream is the reference's. */
int b2l_topk_softmax(const void* logits, float temperature, int top_k, void* probs, int V,
                     b2l_stream_t stream);

/* generate.py:68-76 in one launch: the probabilities above AND the draw of generate.py:76
 * (torch.multinomial(probs, num_samples=1)).  For one draw ATen computes argmax(probs / q), q ~ Exp(1)
 * (ATen/native/Distributions.cpp, ties to the lower index); `noise` is that q, bf16 [V], drawn by the caller with
 * torch (`torch.empty_like(probs).exponential_(1)`: the RNG consumption of multinomial), so `*token` (device
 * int64) equals the reference's sample for the same generator state.  probs may be NULL. */
int b2l_topk_softmax_sample(const void* logits, float temperature, int top_k, const void* noise, void* probs,
                            int64_t* token, int V, b2l_stream_t stream);

/* ------------------------------------------------------------------------------
 * CausalSelfAttention.forward without the two linears, model.py:197-232:
 * split qkv, apply_rope(q), apply_rope(k) (model.py:306-323), append k,v to the
 * cache at input_pos (roll-when-full branch model.py:214-218 handled on the device
 * with a ring offset), causal softmax(q k^T / sqrt(hs)) v.
 *
 * qkv   bf16 [B, T, 3*C]   (q | k | v thirds, each [nh, hs])
 * k/v cache bf16 [B, nh, S, hs]; physical slot = (logical slot + *ring_start) % S
 * rope  f32 [block_size, hs/2, 2] (cos, sin) - build_rope_cache, model.py:280-303
 * input_pos int64 [T] on the device (never read by the host).  Query t writes its
 *            k,v at logical slot min(input_pos[t], S-1) and attends slots <= that.
 * ring_start int32 [1] on the device, read-only here; b2l_ring_advance moves it
 * y     bf16 [B, T, C]
 * work  scratch of b2l_attn_workspace_bytes(...) bytes (split-S partials + tickets);
 *       the caller zero-fills it ONCE after allocating it
 * ---------------------------------------------------------------------------- */
size_t b2l_attn_workspace_bytes(int B, int n_head, int head_size, int T, int S);
int b2l_attention(void* qkv, void* k_cache, void* v_cache, const void* rope,
                  const int64_t* input_pos, const int32_t* ring_start, void* y, void* work, int B,
                  int T, int n_head, int head_size, int S, int block_size, int flags,
                  b2l_stream_t stream);

/* ------------------------------------------------------------------------------
 * Tensor-parallel decode (new capability: every reference script is Fabric(devices=1); the split dims are the ones
 * scripts/convert_checkpoint.py:56-64 records).  One-shot all-reduce (sum, fp32 accumulation in rank order, one
 * rounding) of a bf16 row of n elements over the GPUs of one node, through peer memory: every rank pushes
 * {2 values, epoch} words into its slot of every peer's exchange buffer (NVLink stores) and polls its own buffer
 * (csrc/tp_allreduce.cu).  `out` may alias `partial`.  All ranks must issue the same sequence of calls.
 * peer_buf[r]: rank r's buffer of b2l_tp_buffer_bytes(world, max_elems) bytes as mapped into this process
 * (peer_buf[rank] = the local one), zero-filled once before the first call; epoch: 16 local device words, status:
 * one, zero-filled once.  status becomes 1 if a bounded wait timed out (the result is then undefined).
 * ---------------------------------------------------------------------------- */
typedef struct b2l_tp_comm {
  void* peer_buf[8];
  int rank, world;
  int max_elems;
  unsigned int* epoch;
  int* status;
} b2l_tp_comm;
size_t b2l_tp_buffer_bytes(int world, int max_elems);
int b2l_tp_allreduce(const b2l_tp_comm* comm, const void* partial, void* out, int n, int flags,
                     b2l_stream_t stream);

/* The roll branch of model.py:214-218 as a ring: if input_pos[T-1] >= S the ring start
 * advances by one slot (the oldest entry is dropped, exactly what torch.roll(-1) +
 * overwrite of slot S-1 does).  Call once per forward, before the layers. */
int b2l_ring_advance(const int64_t* input_pos, int T, int32_t* ring_start, int S,
                     b2l_stream_t stream);

/* Same without a cache (input_pos is None, model.py:104-106): positions 0..T-1.
 * qkv is rotated in place; work as for b2l_attention with S = T. */
int b2l_attention_nocache(void* qkv, const void* rope, void* y, void* work, int B, int T,
                          int n_head, int head_size, int block_size, b2l_stream_t stream);

/* kv_caches as the reference would hold them (logical order): un-rotates the ring
 * into `out` [B, nh, S, hs]. */
int b2l_kv_unroll(const void* cache, const int32_t* ring_start, void* out, int B, int n_head,
                  int S, int head_size, b2l_stream_t stream);

/* ------------------------------------------------------------------------------
 * Whole decode step: LLaMA.forward for T == 1 with a KV cache (model.py:76-122),
 * every kernel of the step enqueued by one call.
 * ---------------------------------------------------------------------------- */
typedef struct b2l_q4_weight {
  const void* qw_tiled;   /* b2l_q4_tile layout (tcgen05 kernel), used when B > 1; may be NULL if B == 1 */
  const void* qw_mma;     /* mma.sync kernels: b2l_q4_tile_i8 layout when B == 1 (b2l_q4_gemv), b2l_q4_tile_mma
                             layout when B in 2..8 (b2l_q4_gemv_batch); may be NULL if B > 8 */
  const void* scales;
  const void* zeros;
  int N, K;
} b2l_q4_weight;

typedef struct b2l_layer {
  const void* rms_1;       /* bf16 [C] */
  const void* rms_2;       /* bf16 [C] */
  b2l_q4_weight c_attn;    /* [3C, C]                                                */
  b2l_q4_weight c_proj;    /* [C, C]                                                 */
  b2l_q4_weight c_fc12;    /* [2*n_hidden, C]; qw_tiled rows interleaved 64/64 per 128-row tile,
                              qw_mma rows interleaved 8/8 per 16-row block (scales/zeros in the
                              order of the layout in use)                               */
  b2l_q4_weight mlp_proj;  /* [C, n_hidden]                                          */
  void* k_cache;           /* bf16 [B, nh, S, hs]                                    */
  void* v_cache;
} b2l_layer;

typedef struct b2l_decode_args {
  int n_layer, n_head, n_embd, n_hidden, vocab; /* vocab = padded_vocab_size          */
  int B, S;                                     /* batch, max_seq_length              */
  int sz_dtype;
  float eps;
  const b2l_layer* layers;   /* HOST array [n_layer]                                  */
  const void* wte;           /* bf16 [vocab, C]                                       */
  const void* ln_f;          /* bf16 [C]                                              */
  b2l_q4_weight lm_head;     /* [vocab, C]                                            */
  const void* rope;          /* f32 [block_size, hs/2, 2]                             */
  const void* idx;           /* int32/int64 [B] tokens of this step                   */
  int idx_is_i64;
  const int64_t* input_pos;  /* int64 [1]                                             */
  int32_t* ring_start;       /* int32 [1]; advanced by the step when the cache is full */
  int block_size;            /* rows of the rope table                                */
  void* x;                   /* bf16 [B, C]   residual stream scratch                 */
  void* qkv;                 /* bf16 [B, 3C]                                          */
  void* att;                 /* bf16 [B, C]                                           */
  void* hid;                 /* bf16 [B, n_hidden]                                    */
  void* attn_work;           /* f32, b2l_attn_workspace_bytes                         */
  void* logits;              /* bf16 [B, vocab]                                       */
  int flags;                 /* B2L_F_*                                               */
  void* timeline;            /* debug: device uint64[(5*n_layer+1)*64] of %globaltimer stamps per
                                launch (NULL = off); tools/diag.py `timeline`               */
  void* batch_work;          /* B in 2..8: scratch of b2l_q4_gemv_batch_workspace_bytes(max K) bytes; the
                                linears then run on the mma.sync batch kernel (weights need qw_mma).
                                NULL: tcgen05 kernel (weights need qw_tiled)              */
} b2l_decode_args;

int b2l_decode_step(const b2l_decode_args* args, b2l_stream_t stream);
/* Number of kernels one b2l_decode_step enqueues (for bench.py's gpu_launches). */
int b2l_decode_step_launches(const b2l_decode_args* args);

#ifdef __cplusplus
}
#endif
#endif /* B2L_H_ */
