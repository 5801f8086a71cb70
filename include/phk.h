/*
 * phk.h -- C ABI of the B200-native phenaki hot path (libphk.so).
 *
 * The reference (lucidrains/phenaki-pytorch @ 9415d4e) has no FFI: the path sits behind
 * torch.nn.Module classes (phenaki_pytorch/__init__.py:1-4).  This header is the boundary a
 * maintainer would bind instead (ctypes stub in INTEGRATION.md): plain pointers, sizes and a
 * cudaStream_t; no torch types.  Every entry point cites the reference code it replaces
 * (paths relative to /root/reference/phenaki_pytorch/).
 *
 * Conventions
 *   - every function returns int: 0 ok, <0 argument/shape error (PHK_E_*), >0 a cudaError_t.
 *     Nothing throws or aborts.  phk_last_error() returns a static description of the last <0.
 *   - all device pointers are BORROWED for the duration of the call; the library allocates
 *     nothing on the device: scratch comes from a caller-owned workspace
 *     (phk_*_workspace_bytes()).  Work is enqueued on the caller's stream, no host sync,
 *     except the *_host entry points which copy from/to host memory and synchronise.
 *   - residual stream / LayerNorm / softmax are fp32.  `prec` selects the contraction type:
 *     PHK_PREC_F32  fp32 FFMA GEMMs (parity mode, token ids identical to the fp32 reference);
 *     PHK_PREC_BF16 bf16 operands on tcgen05 tensor cores with fp32 TMEM accumulation (the
 *                   dtype flow of the reference under torch.autocast(bfloat16), SURVEY H2).
 *     PHK_PREC_BF16X3 fp32-grade products ON the tensor cores: every nn.Linear operand is split into two bf16 terms
 *                   (x = hi + lo, |x - hi - lo| <= 2^-17 |x|) and C = A_hi W_hi + A_hi W_lo + A_lo W_hi is ONE tcgen05
 *                   GEMM over the concatenated K' = 3K ([hi | hi | lo] x [hi | lo | hi], fp32 TMEM accumulation);
 *                   everything else (LayerNorm, attention core, GEGLU, PEG, fp32 activations) is the parity mode's.
 *                   Token ids equal the fp32 reference's at the bars of tests/test_gpu_parity_at_size.py without
 *                   the FFMA GEMMs' cost.  Inference only (the training step treats it as PHK_PREC_F32).
 *   - token ids are int64 (reference dtype), masks are uint8 (0/1).
 */
#ifndef PHK_H_
#define PHK_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* phk_stream_t; /* == cudaStream_t */

enum { PHK_PREC_F32 = 0, PHK_PREC_BF16 = 1, PHK_PREC_BF16X3 = 2 };
enum {
  PHK_E_ARG = -1,      /* null pointer / non-positive size            */
  PHK_E_SHAPE = -2,    /* shape contract violated (reference asserts) */
  PHK_E_UNSUPPORTED = -3,
  PHK_E_WORKSPACE = -4 /* workspace too small                         */
};

int phk_version(void);
const char* phk_last_error(void);
/* number of kernels this library has launched in this process (bench.py gpu_launches) */
int64_t phk_launch_count(void);

/* Per-kernel-family timing (CUDA events on the launching stream) for bench.py's roofline and
 * share-of-step numbers.  Families, in order: patchify_ln, layernorm, gemm_f32, gemm_bf16,
 * attention, peg, geglu, lfq, embed, cpb, sample_tokens, topk_mask, critic, cfg_combine.
 * work_by_family = algorithmic FLOPs (gemm, attention) or bytes (memory-bound kernels). */
#define PHK_NUM_FAMILIES 14
int phk_prof_enable(int32_t on);
int phk_prof_collect(double* ms_by_family, int64_t* calls_by_family, double* work_by_family, int32_t n);

/* ------------------------------------------------------------------------------------------ */
/* Weight tables (filled by the host-side modules from the reference state_dict layout)        */
/* ------------------------------------------------------------------------------------------ */

/* attention.py:89-126 Attention.  *_h are optional bf16 copies of the same matrices, padded so
 * every leading dimension is a multiple of 8 elements (16 B, TMA requirement). */
typedef struct {
  const float* norm_g;  const float* norm_b;      /* norm.gamma / norm.beta [dim]              */
  const float* ctx_g;   const float* ctx_b;       /* context_norm.* [dim_context]              */
  const float* null_kv;                           /* [heads, 2*num_null_kv, dim_head]          */
  const float* q_scale; const float* k_scale;     /* [dim_head]                                */
  const float* wq; const float* wkv; const float* wo; /* [I,dim] [2I,dim_context] [dim,I]      */
  const void* wq_h; const void* wkv_h; const void* wo_h;
  int32_t num_null_kv; int32_t dim_context;
} phk_attn_t;

/* attention.py:45-53 FeedForward: LN(affine) -> Linear(dim,2*inner) -> GEGLU -> Linear(inner,dim) */
typedef struct {
  const float* ln_g; const float* ln_b;
  const float* w1; const float* w2;               /* [2*inner, dim], [dim, inner]               */
  const void* w1_h; const void* w2_h;             /* bf16: w1 rows interleaved val/gate per 64, */
  int32_t inner; int32_t inner_pad;               /* w2 K padded to inner_pad (multiple of 64)  */
} phk_ff_t;

/* attention.py:57-85 PEG: depthwise Conv3d(dim,dim,3,groups=dim); w tap-major [27, dim]
 * (= dsconv.weight[dim,1,3,3,3].reshape(dim,27).t(), packed by the host module) */
typedef struct { const float* w; const float* b; int32_t causal; int32_t _pad; } phk_peg_t;

/* one entry of Transformer.layers (attention.py:300-306): .0 PEG .1 self .2 cross .3 FF */
typedef struct {
  int32_t has_peg; int32_t has_cross;
  phk_peg_t peg; phk_attn_t self_attn; phk_attn_t cross_attn; phk_ff_t ff;
} phk_layer_t;

/* attention.py:279-332 Transformer */
typedef struct {
  int32_t dim; int32_t heads; int32_t dim_head; int32_t depth; int32_t causal; int32_t _pad;
  const phk_layer_t* layers;
  const float* out_g; const float* out_b;         /* norm_out.gamma / beta                      */
  const float* alibi_slopes;                      /* [heads] when causal (attention.py:201-212) */
} phk_transformer_t;

/* attention.py:229-275 ContinuousPositionBias with the default 2 hidden layers */
typedef struct {
  const float* w0; const float* b0;               /* [hidden, num_dims]                         */
  const float* w1; const float* b1;               /* [hidden, hidden]                           */
  const float* w2; const float* b2;               /* [heads, hidden]                            */
  int32_t num_dims; int32_t hidden; int32_t heads; int32_t _pad;
} phk_cpb_t;

/* cvivit.py:226-335 CViViT, encode-side members only */
typedef struct {
  int32_t dim, heads, dim_head, channels;
  int32_t image_h, image_w, patch_h, patch_w, patch_t;
  int32_t codebook_bits; int32_t _pad0, _pad1;
  /* to_patch_emb_first_frame.{1,2,3} / to_patch_emb.{1,2,3} (cvivit.py:273-285) */
  const float* pf_ln1_g; const float* pf_ln1_b; const float* pf_w; const float* pf_b;
  const float* pf_ln2_g; const float* pf_ln2_b; const void* pf_w_h;
  const float* pr_ln1_g; const float* pr_ln1_b; const float* pr_w; const float* pr_b;
  const float* pr_ln2_g; const float* pr_ln2_b; const void* pr_w_h;
  phk_cpb_t spatial_bias;                         /* spatial_rel_pos_bias                       */
  phk_transformer_t spatial;                      /* enc_spatial_transformer                    */
  phk_transformer_t temporal;                     /* enc_temporal_transformer                   */
  const float* vq_w; const float* vq_b;           /* vq.project_in [bits, dim], [bits]          */
  /* lookup_free_quantization=False (cvivit.py:321): the cosine-sim codebook vq._codebook.embed[0] [codebook_size, dim]
   * (unit rows); vq_w / vq_b are then NULL and codebook_bits 0 */
  const float* codebook; const void* codebook_h;
  int32_t codebook_size; int32_t _pad2;
} phk_cvivit_t;

/* cvivit.py:323-335 the decoder half of CViViT (vq.project_out, dec_* transformers, to_pixels*) */
typedef struct {
  int32_t dim, heads, dim_head, channels;
  int32_t image_h, image_w, patch_h, patch_w;
  int32_t patch_t, codebook_bits;
  const float* vq_out_w; const float* vq_out_b;   /* vq.project_out [dim, bits], [dim]          */
  phk_cpb_t spatial_bias;                         /* spatial_rel_pos_bias (shared with encode)  */
  phk_transformer_t temporal;                     /* dec_temporal_transformer                   */
  phk_transformer_t spatial;                      /* dec_spatial_transformer                    */
  const float* px_first_w; const float* px_first_b; const void* px_first_w_h; /* to_pixels_first_frame.0 [C*p1*p2, dim] */
  const float* px_w; const float* px_b; const void* px_w_h;                   /* to_pixels.0 [C*pt*p1*p2, dim]          */
} phk_cvivit_dec_t;

/* phenaki_pytorch.py:105-147 MaskGit / :217-249 TokenCritic (is_critic: no bias, Linear(dim,1)) */
typedef struct {
  int32_t dim, heads, dim_head, num_tokens, max_seq_len, is_critic, has_bias, _pad;
  float shrink_alpha; float _padf;
  const float* token_emb; const float* pos_emb;   /* [num_tokens+1, dim], [max_seq_len, dim]    */
  phk_cpb_t pos_bias;                             /* continuous_pos_bias (MaskGit only)         */
  phk_transformer_t transformer;
  const float* head_w; const float* head_b;       /* to_logits: [V,dim],[V]  | critic [1,dim],[1]*/
  const void* head_w_h;
} phk_maskgit_t;

/* ------------------------------------------------------------------------------------------ */
/* Building blocks (each is one kernel launch unless noted; used directly by the unit tests)   */
/* ------------------------------------------------------------------------------------------ */

/* F.layer_norm over the last dim, eps 1e-5 (attention.py:35-36, :48, :308).
 * out_bf16!=0 writes __nv_bfloat16 instead of float.  raw_bf16 (optional, bf16 mode) also
 * receives the un-normalised row converted to bf16 (self-attention projects k,v from raw x,
 * attention.py:140-144).  Row map as in phk_gemm_f32: seg_len>0 places the OUTPUT row (scatter), seg_len<0 picks
 * the INPUT row with |seg_len| (gather; `rows` then counts output rows), seg_len==0: identity. */
int phk_layernorm(const float* x, const float* gamma, const float* beta, void* out, void* raw_bf16,
                  int64_t rows, int32_t dim, int32_t out_bf16, int64_t seg_len, int64_t seg_stride,
                  int64_t seg_off, phk_stream_t s);

/* Rearrange 'b c (t pt)(h p1)(w p2) -> b t h w (c pt p1 p2)' + LayerNorm(K) of
 * to_patch_emb* (cvivit.py:273-275, 280-282): frames [f0, f0+nt*pt) of video (B,C,F,H,W) fp32
 * -> A[(b,t,h,w), K] (fp32 or bf16), K = C*pt*p1*p2. */
int phk_patchify_ln(const float* video, int32_t B, int32_t C, int32_t F, int32_t H, int32_t W,
                    int32_t f0, int32_t nt, int32_t pt, int32_t p1, int32_t p2,
                    const float* ln_g, const float* ln_b, void* out, int32_t out_bf16, phk_stream_t s);

/* C[map(m), n] = sum_k A[m,k] * W[n,k] (+bias[n]) (+residual[map(m), n]); nn.Linear semantics.
 * Row map: map(m) = (m / seg_len) * seg_stride + seg_off + m % seg_len (seg_len<=0: identity).
 * fp32 FFMA kernel (parity mode). */
int phk_gemm_f32(const float* A, int64_t lda, const float* W, int64_t ldw, float* C, int64_t ldc,
                 int64_t M, int32_t N, int32_t K, const float* bias, const float* residual,
                 int64_t seg_len, int64_t seg_stride, int64_t seg_off, phk_stream_t s);

/* Same contract on tcgen05 tensor cores: A,W bf16 (K-major, lda/ldw multiples of 8), fp32 TMEM
 * accumulators, TMA-fed, warp-specialised.  epilogue: 0 store fp32 (+bias,+residual),
 * 1 store bf16 (+bias), 2 GEGLU on val/gate-interleaved W rows -> bf16 [M, N/2]. */
int phk_gemm_bf16(const void* A, int64_t lda, const void* W, int64_t ldw, void* C, int64_t ldc,
                  int64_t M, int32_t N, int32_t K, const float* bias, const float* residual,
                  int64_t seg_len, int64_t seg_stride, int64_t seg_off, int32_t epilogue,
                  phk_stream_t s);

/* Two independent products C1 = A1 W1^T (+bias1) [M1,N1] and C2 = A2 W2^T (+bias2) [M2,N2] (bf16 operands, fp32
 * outputs) in ONE launch: the q and k,v projections of a self-attention block read different inputs (LayerNorm(x) vs
 * raw x, attention.py:140-146) and are each a single wave of tiles; the first-frame and rest-frames patch embeddings
 * (cvivit.py:542-549) are 16 + 128 tiles.  Launched together their tiles pipeline / fill the machine. */
int phk_gemm_bf16_x2(const void* A1, int64_t lda1, const void* W1, int64_t ldw1, float* C1, int64_t ldc1,
                     int64_t M1, int32_t N1, int32_t K1, const float* bias1, const void* A2, int64_t lda2,
                     const void* W2, int64_t ldw2, float* C2, int64_t ldc2, int64_t M2, int32_t N2, int32_t K2,
                     const float* bias2, phk_stream_t s);

/* The q and k,v projections of one self-attention block (attention.py:140-146: q from LayerNorm(x), k,v from the raw x)
 * in ONE launch whose epilogue writes the bf16 OPERANDS of the attention core (attention.py:153-157) instead of fp32
 * projections: Qn[M, I] = F.normalize(q, per 64-wide head) * q_scale * sim_scale, KVn[M, 2I] = [F.normalize(k) * k_scale |
 * v].  xn / xraw bf16 [M, lda], Wq bf16 [I, ldw], Wkv bf16 [2I, ldw]; dim_head 64, I % 128 == 0.  Consumed by
 * phk_attention_tc_bf16 / phk_attention_small_bf16. */
int phk_gemm_bf16_qkv(const void* xn, const void* xraw, int64_t lda, const void* Wq, const void* Wkv, int64_t ldw,
                      void* Qn, void* KVn, int64_t M, int32_t I, int32_t K, const float* q_scale, const float* k_scale,
                      float sim_scale, phk_stream_t s);

/* x = A W^T (+bias) + x IN PLACE (C is the fp32 residual stream, nn.Linear + residual of attention.py:322-330) and, from
 * the same epilogue, the LayerNorm the NEXT sub-block applies to x: ln_out[M, ln_ld] = bf16(LayerNorm(x) * ln_g + ln_b)
 * (ln_b may be NULL), raw_out (optional) = bf16(x).  N = row width in {128, 256, 512, 1024}: the N / 128 CTAs of a
 * 128-row tile form a cluster and sum their row statistics through distributed shared memory. */
int phk_gemm_bf16_ln(const void* A, int64_t lda, const void* W, int64_t ldw, float* C, int64_t ldc, int64_t M, int32_t N,
                     int32_t K, const float* bias, const float* ln_g, const float* ln_b, float ln_eps, void* ln_out,
                     void* raw_out, int64_t ln_ld, phk_stream_t s);

/* The same product with the row statistics exchanged through global memory instead of a cluster (the N / 128 CTAs of a
 * 128-row tile are ordinary CTAs of a grid of at most one CTA per SM, all resident; no GPC-local cluster placement).
 *   stat_ws : PHK_LN_STAT_BYTES bytes of device scratch, 16-byte aligned, any content;
 *   counters: PHK_LN_COUNTERS zero-initialised 32-bit device words, consumed by the call (left non-zero) -- give every
 *             call of a stream-ordered sequence its own words and clear them together once per sequence. */
#define PHK_LN_STAT_BYTES (2 * 148 * 128 * 8)
#define PHK_LN_COUNTERS 160
int phk_gemm_bf16_ln_ws(const void* A, int64_t lda, const void* W, int64_t ldw, float* C, int64_t ldc, int64_t M,
                        int32_t N, int32_t K, const float* bias, const float* ln_g, const float* ln_b, float ln_eps,
                        void* ln_out, void* raw_out, int64_t ln_ld, void* stat_ws, uint32_t* counters, phk_stream_t s);

/* PHK_PREC_BF16X3 operand split: x fp32 [rows, ld] (K valid columns) -> bf16 [rows, 3 * Kp], Kp = K rounded up to 8:
 * [hi | hi | lo] (weights == 0: the activation side) or [hi | lo | hi] (weights != 0), hi = bf16(x), lo = bf16(x - hi),
 * zero in the padding columns.  With both sides split this way a plain bf16 GEMM over K' = 3 Kp computes
 * A_hi W_hi + A_hi W_lo + A_lo W_hi. */
int phk_split3(const float* x, int64_t ld, void* out, int64_t rows, int32_t K, int32_t weights, phk_stream_t s);

/* debug aid: per-CTA clock64 phase stamps of phk_gemm_bf16 (16 x int64 per CTA); NULL disables */
int phk_debug_gemm_trace(long long* device_buffer);
/* tests / A-B measurements: force the tcgen05 GEMM variant: 0 automatic, 1 one CTA per 128x128 tile, 2 CTA pairs
 * (cta_group::2) with 256x128 tiles, 3 CTA pairs with 256x256 tiles (2 and 3 apply when M > 128); < 0 restores the
 * PHK_GEMM_MODE environment default. */
int phk_debug_gemm_mode(int32_t mode);
/* tests / A-B measurements: declare (1) or withdraw (0), for the calling thread, that the W operands of the following
 * phk_gemm_bf16* calls are not written by earlier kernels of the stream -- the kernel then requests their first tiles before
 * its programmatic-dependent-launch wait.  The forward drivers (phk_cvivit_*, phk_maskgit_*) set this themselves. */
int phk_debug_static_weights(int32_t on);
/* tests / A-B measurements: phk_attention_tc* variant -- 0 probabilities through a shared-memory tile (two CTAs per SM),
 * 1 probabilities in tensor memory as the TMEM A operand of P.V (three CTAs per SM); < 0 restores the default. */
int phk_debug_attention_tc_variant(int32_t variant);

/* GEGLU (attention.py:40-43): out[r, j] = gelu_erf(h[r, inner + j]) * h[r, j] */
int phk_geglu(const float* h, float* out, int64_t rows, int32_t inner, phk_stream_t s);

/* Cosine-sim attention core (attention.py:146-181) for all four uses (spatial, temporal
 * causal+ALiBi, MaskGit self with bias/mask, cross with null-kv/mask).  q fp32 [.., I],
 * kv fp32 [.., 2I] (k at column h*dh, v at column I + h*dh), I = heads*dim_head.
 * Sequence s = (so, si), so < n_outer, si < n_inner: query token i lives at element offset
 * so*q_outer + si*q_inner + i*q_tok (+ h*dh); keys likewise with the k_* strides of sequence
 * (so % kv_outer_mod, si); outputs with the o_* strides.  All strides are in ELEMENTS.
 * bias fp32 [heads, n_q, n_k] or NULL (never covers the null keys, attention.py:162);
 * key_mask uint8 [*, n_k] or NULL, row = so % mask_outer_mod (0: so); sequences with
 * so >= mask_off_from (>=0) see an all-False mask = the cond_drop_prob=1 half of a
 * classifier-free-guidance pair (phenaki_pytorch.py:188-190).
 * alibi_slopes fp32 [heads] (attention.py:201-212), required when causal. */
typedef struct {
  int32_t n_outer, n_inner, n_q, n_k, heads, dim_head, num_null_kv, causal;
  int64_t q_outer, q_inner, q_tok;
  int64_t k_outer, k_inner, k_tok;
  int64_t o_outer, o_inner, o_tok;
  int32_t kv_outer_mod, mask_outer_mod, mask_off_from, out_bf16;
  float scale;                 /* 8 (attention.py:100) */
  int32_t _pad;
} phk_attn_geom_t;
int phk_attention(const float* q, const float* kv, const float* null_kv, const float* q_scale,
                  const float* k_scale, const float* bias, const uint8_t* key_mask,
                  const float* alibi_slopes, void* out, const phk_attn_geom_t* g, phk_stream_t s);

/* Tensor-core (tcgen05) attention core for self-attention sequences of n >= 64 tokens, dim_head 64, no null-kv / key
 * mask / causal (those take phk_attention): S = QK^T and O = PV on tcgen05, S and P never leave the SM.
 * phk_attention_tc_bf16: operands as phk_gemm_bf16_qkv writes them -- Qn bf16 [n_seq*n, ld_q], KVn bf16 [n_seq*n, ld_kv]
 *   (token-major; 4-D tensor maps pick one head's tile, V is an MN-major operand: no head-major or transposed copy);
 *   bias fp32 [heads, n, n] or NULL -> out bf16 [n_seq*n, heads*64].
 * phk_attention_tc: the same from fp32 projections q [n_seq*n, heads*64], kv [n_seq*n, 2*heads*64]: a small kernel first
 *   writes the normalised bf16 operands into `scratch` (>= phk_attention_tc_scratch_bytes). */
int phk_attention_tc_bf16(const void* Qn, int64_t ld_q, const void* KVn, int64_t ld_kv, const float* bias,
                          void* out_bf16, int32_t n_seq, int32_t n, int32_t heads, phk_stream_t s);
/* Small sequences (n <= 16: the temporal transformer, causal + ALiBi) on the same bf16 operands, one warp per (sequence,
 * head); geometry strides in elements as for phk_attention. */
int phk_attention_small_bf16(const void* Qn, const void* KVn, const float* alibi_slopes, void* out,
                             const phk_attn_geom_t* g, phk_stream_t s);
/* The same core for 16 < n <= 64 tokens per sequence (the spatial transformer's frames) on warp-level MMAs: one CTA per
 * (sequence, head), all resident at once; arguments as phk_attention_tc_bf16. */
int phk_attention_mid_bf16(const void* Qn, int64_t ld_q, const void* KVn, int64_t ld_kv, const float* bias, void* out_bf16,
                           int32_t n_seq, int32_t n, int32_t heads, phk_stream_t s);
int64_t phk_attention_tc_scratch_bytes(int32_t n_seq, int32_t n, int32_t heads);
int phk_attention_tc(const float* q, const float* kv, const float* q_scale, const float* k_scale,
                     const float* bias, void* out_bf16, int32_t n_seq, int32_t n, int32_t heads, float scale,
                     void* scratch, int64_t scratch_bytes, phk_stream_t s);

/* PEG (attention.py:64-85) + residual: y = x + conv3d_depthwise(pad(x)) + b on a logical
 * (B,T,H,W,D) channels-last view.  layout 0: row = logical flat index (MaskGit, (b,n,d)).
 * layout 1: the C-ViViT temporal quirk -- the caller's physical rows are (b,t,h,w) but the
 * reference conv sees the '(b h w) t d' buffer REINTERPRETED as (b,t,h,w,d) (attention.py:71
 * with cvivit.py:468-470); the kernel composes both index maps. */
int phk_peg3d(const float* x, const float* w, const float* b, float* y, int32_t B, int32_t T,
              int32_t H, int32_t W, int32_t D, int32_t causal, int32_t layout, phk_stream_t s);

/* ContinuousPositionBias (attention.py:257-275) -> out[heads, n, n], n = d0*d1*d2 (d2=1 for 2-D).
 * The MLP runs once per distinct coordinate delta (prod(2*d_i-1) rows) and is expanded.
 * scratch: >= phk_cpb_scratch_floats() floats. */
int64_t phk_cpb_scratch_floats(const phk_cpb_t* c, int32_t d0, int32_t d1, int32_t d2);
int phk_cpb_bias(const phk_cpb_t* c, int32_t d0, int32_t d1, int32_t d2, float* scratch,
                 float* out, phk_stream_t s);

/* LFQ ids (cvivit.py:570 -> vector_quantize_pytorch.LFQ.forward, restated in oracle/lfq.py):
 * proj = x @ Wp^T + bp ; id = sum_d (proj_d > 0) << (bits-1-d).  proj_out optional [rows,bits]. */
int phk_lfq_ids(const float* x, const float* wp, const float* bp, int64_t* ids, float* proj_out,
                int64_t rows, int32_t dim, int32_t bits, phk_stream_t s);

/* LayerNorm (attention.py:308,332: the temporal transformer's norm_out) fused with phk_lfq_ids: the normalised row
 * stays in registers.  out_norm (optional fp32 [rows, dim]) and proj_out (optional [rows, bits]) receive the
 * intermediate values for the parity tests; shapes outside dim % 128 == 0, dim <= 1024, bits <= 16 fall back to
 * phk_layernorm + phk_lfq_ids and then need out_norm as the row buffer. */
int phk_layernorm_lfq(const float* x, const float* gamma, const float* beta, const float* wp, const float* bp,
                      int64_t* ids, float* out_norm, float* proj_out, int64_t rows, int32_t dim, int32_t bits,
                      phk_stream_t s);

/* Cosine-sim VectorQuantize ids (cvivit.py:321, :568-570 with lookup_free_quantization=False; oracle/lfq.py):
 * ids[r] = argmax_c l2norm(x[r]) . codebook[c] = argmax_c x[r] . codebook[c] (unit codebook rows), first maximum on ties.
 * PHK_PREC_F32: x fp32 [rows, dim], fp32 FFMA similarities strip by strip; PHK_PREC_BF16: x bf16 [rows, dim], the fused
 * tcgen05 head at temperature 0 (dim <= 512): the [rows, K] similarities are never stored. */
int64_t phk_vq_cosine_scratch_bytes(int64_t rows, int32_t K, int32_t prec);
int phk_vq_cosine_ids(const void* x, const float* codebook, const void* codebook_h, int64_t* ids, int64_t rows,
                      int32_t dim, int32_t K, void* scratch, int64_t scratch_bytes, int32_t prec, phk_stream_t s);

/* LFQ indices_to_codes + project_out (cvivit.py:437-439 -> LFQ.indices_to_codes, oracle/lfq.py):
 * out[r, :] = w_out @ (bit_j(id_r) ? +1 : -1)_j + b_out, bits MSB first; w_out [dim, bits]; out fp32 [rows, dim]. */
int phk_lfq_codes(const int64_t* ids, const float* w_out, const float* b_out, float* out,
                  int64_t rows, int32_t dim, int32_t bits, phk_stream_t s);

/* Rearrange 'b t h w (c pt p1 p2) -> b c (t pt) (h p1) (w p2)' (cvivit.py:286-295), the mirror of phk_patchify_ln:
 * P fp32 [B*nt*(H/p1)*(W/p2), ldp >= C*pt*p1*p2] -> frames [f0, f0 + nt*pt) of video (B,C,F,H,W) fp32. */
int phk_unpatchify(const float* P, int64_t ldp, float* video, int32_t B, int32_t C, int32_t F,
                   int32_t H, int32_t W, int32_t f0, int32_t nt, int32_t pt, int32_t p1, int32_t p2,
                   phk_stream_t s);

/* token_emb[id] + pos_emb[pos] then x*a + x*(1-a) (phenaki_pytorch.py:194-199); a<0 skips the
 * shrink (TokenCritic, :290-291). rows = b*n. */
int phk_token_embed(const int64_t* ids, const float* tok, const float* pos, float* out,
                    int32_t b, int32_t n, int32_t dim, int32_t vocab_rows, float alpha,
                    int32_t replicas /* 2: also emit the CFG null half */, phk_stream_t s);

/* CFG + gumbel argmax + confidence, one pass over the vocabulary
 * (phenaki_pytorch.py:161, 83-93, 506-509, 547-550):
 *   l = null + (cond-null)*cond_scale   (null==NULL or cond_scale==1: l = cond)
 *   pred = argmax_v( l/max(T,1e-10) - log(-log(u+1e-10)+1e-10) ), first index on ties
 *   ids = mask ? pred : ids ;  score = mask ? 1 - softmax(l)[pred] : -1e4
 * u: uniform draws [rows, V] (parity mode) or NULL -> in-kernel noise (seed, offset):
 *   Philox4x32 with 7 rounds (Random123 definition), key = (seed lo, seed hi), counter =
 *   (c lo, c hi, 0, 0) with c = offset + r * ceil(V/4) + v/4 (64-bit, wraps mod 2^64) for token
 *   row r; entry v takes output word v%4.  A row consumes ceil(V/4) counters.
 *   bits w -> uniform u = (2*(w >> 9) + 1) / 2^24 (exact, strictly inside (0, 1)) ->
 *   gumbel g = -ln(-ln u), both logarithms in base 2 on the fast-math unit;
 *   pred = argmax_v( fma(l, 1/max(T,1e-10), g) ), first index on ties.
 *   phk_noise_probe returns the words and the transform the kernels use.
 * seg_*: token row r reads logits row (r/seg_len)*seg_stride + seg_off + r%seg_len, i.e. the
 * `logits[:, prime_len:]` slice of a primed sample (:503-504); seg_len<=0: identity.  The noise
 * counters follow the token row r, not the logits row. */
int phk_sample_tokens(const float* cond, const float* null_logits, int64_t ld, const float* u,
                      uint64_t seed, uint64_t offset, float cond_scale, float temperature,
                      const uint8_t* mask, int64_t* ids, int64_t* pred_out, float* score_out,
                      int64_t rows, int32_t V, int64_t seg_len, int64_t seg_stride, int64_t seg_off,
                      phk_stream_t s);

/* Cosine-schedule re-masking (phenaki_pytorch.py:485-491): mask = scatter(topk(scores,k));
 * ids = where(mask, mask_id, ids).  n <= 4096; ties: lower index wins. */
int phk_topk_mask(const float* scores, int32_t b, int32_t n, int32_t k, uint8_t* mask,
                  int64_t* ids, int64_t mask_id, phk_stream_t s);

/* Cross-attention on packed operands (bf16 mode; attention.py:137-181 with null keys + at most 32 key slots, dim_head 64).
 * phk_cross_kv_pack: once per transformer call, for every layer l: pack[(l * ctx_b + b) * heads + h] = { K^ [32][64] bf16
 *   (null keys first, then the text keys; l2-normalised * k_scale; zero padding), V [32][64] bf16 }, dead[(l * ctx_b + b)][32]
 *   = 1 for a masked text key or a padding slot.  kv[l]: fp32 [ctx_b * L, 2 * heads * 64] (phk_maskgit_context_kv), null_kv[l]:
 *   [heads, 2 * nnull, 64], k_scale[l]: [64], key_mask [ctx_b, L] or NULL.  pack: depth * ctx_b * heads * 8192 bytes.
 * phk_gemm_bf16_qnorm: Qn[M, I] = normalize_per_head(xn Wq^T) * q_scale * sim_scale as bf16 (the q projection's epilogue).
 * phk_attention_cross_packed: one layer; sequence s uses the text s % ctx_b, sequences >= null_from (-1: none) attend to the
 *   null keys only (the null half of a CFG pair). */
int phk_cross_kv_pack(const float* const* kv, const float* const* null_kv, const float* const* k_scale, int32_t depth,
                      const uint8_t* key_mask, int32_t ctx_b, int32_t L, int32_t heads, int32_t nnull, void* pack, float* dead,
                      phk_stream_t s);
int phk_gemm_bf16_qnorm(const void* xn, int64_t lda, const void* Wq, int64_t ldw, void* Qn, int64_t M, int32_t I, int32_t K,
                        const float* q_scale, float sim_scale, phk_stream_t s);
int phk_attention_cross_packed(const void* Qn, int64_t ld_q, const void* pack, const float* dead, void* out, int64_t ld_o,
                               int32_t n_seq, int32_t n_q, int32_t heads, int32_t ctx_b, int32_t nnull, int32_t null_from,
                               phk_stream_t s);

/* critic score (phenaki_pytorch.py:246-249, 263, 544-545):
 *   sc = x @ w + b per row; out = null + (cond - null)*scale + noise_K*(u-0.5)*noise_mult  */
int phk_critic_scores(const float* x_cond, const float* x_null, const float* w, const float* b,
                      const float* u, float cond_scale, float noise_K, float noise_mult, float* out,
                      int64_t rows, int32_t dim, int64_t seg_len, int64_t seg_stride, int64_t seg_off,
                      phk_stream_t s);

/* forward_with_cond_scale tail (phenaki_pytorch.py:161): out = null + (cond - null) * scale */
int phk_cfg_combine(const float* cond, const float* null_out, float cond_scale, float* out,
                    int64_t n, phk_stream_t s);

/* ------------------------------------------------------------------------------------------ */
/* Fused drivers = the reference-facing operations                                             */
/* ------------------------------------------------------------------------------------------ */

/* CViViT.forward(video, return_only_codebook_ids=True) (cvivit.py:518-574).
 * video (B,C,F,H,W) fp32 device; ids (B,T',H',W') int64 device.
 * spatial_bias: cached phk_cpb_bias(spatial_bias, H', W') output [heads, H'W', H'W'] or NULL
 * (recomputed inside).  taps: optional fp32 device buffers for the parity tests:
 * tap_patch / tap_spatial / tap_temporal [B*T'*H'*W', dim] in (b,t,h,w) row order,
 * tap_proj [rows, bits] = LFQ pre-sign projection.
 * Launch cost: the ~75 launches of one call are a pure function of (table contents, buffers, shape, prec).  With
 * spatial_bias given and no taps, the second call with an identical key is captured into a CUDA graph on a
 * library-owned stream and later calls replay it on `s` (one cudaGraphLaunch; env PHK_GRAPH=0 keeps every call
 * eager).  The graph only bakes in addresses: new data in the same buffers (video, weights updated in place) is
 * honoured; a table with different pointers or dims is a different key. */
int64_t phk_cvivit_workspace_bytes(const phk_cvivit_t* m, int32_t B, int32_t F, int32_t prec);
int phk_cvivit_encode(const phk_cvivit_t* m, const float* video, int32_t B, int32_t F,
                      int64_t* ids, void* workspace, int64_t workspace_bytes, int32_t prec,
                      const float* spatial_bias, float* tap_patch, float* tap_spatial,
                      float* tap_temporal, float* tap_proj, phk_stream_t s);
/* same through HOST buffers (pinned or pageable): H2D of the video, encode, D2H of the ids,
 * stream synchronise.  dev_video / dev_ids are caller-owned staging buffers. */
int phk_cvivit_encode_host(const phk_cvivit_t* m, const float* host_video, int32_t B, int32_t F,
                           int64_t* host_ids, void* dev_video, int64_t* dev_ids, void* workspace,
                           int64_t workspace_bytes, int32_t prec, const float* spatial_bias,
                           phk_stream_t s);

/* Pipelined variant of phk_cvivit_encode_host for a stream of batches (what a tokenisation job over a dataset does):
 * submit() enqueues H2D on the pipe's own copy stream, encode + D2H of the ids on the caller's stream `s`, and
 * returns at once; the copy of batch i+1 overlaps the encode of batch i.  The caller owns `depth` staging slots:
 * dev_video_slots = depth x (B,C,F,H,W) floats, dev_ids_slots = depth x B*T'*H'*W' int64 (slot = ticket % depth), and
 * must keep B, F fixed while tickets are in flight.  host_video should be pinned and must stay untouched until
 * wait(ticket) returns.  wait(ticket) blocks until that
 * batch's host_ids are valid; at most `depth` tickets may be in flight.  Host-side objects only (one stream, 3*depth
 * events); no device memory is allocated. */
typedef struct phk_encode_pipe phk_encode_pipe_t;
int phk_encode_pipe_create(phk_encode_pipe_t** pipe, int32_t depth);
int phk_encode_pipe_destroy(phk_encode_pipe_t* pipe);
int phk_encode_pipe_submit(phk_encode_pipe_t* pipe, const phk_cvivit_t* m, const float* host_video, int32_t B,
                           int32_t F, int64_t* host_ids, void* dev_video_slots, int64_t* dev_ids_slots,
                           void* workspace, int64_t workspace_bytes, int32_t prec, const float* spatial_bias,
                           phk_stream_t s, int64_t* ticket);
int phk_encode_pipe_wait(phk_encode_pipe_t* pipe, int64_t ticket);

/* CViViT.decode_from_codebook_indices(ids) / CViViT.decode(tokens) (cvivit.py:437-443, 476-516):
 * LFQ indices_to_codes -> dec_temporal_transformer -> dec_spatial_transformer -> to_pixels un-patchify.
 * ids (B, T'*H'*W') int64 device, or ids == NULL and tokens [B*T'*H'*W', dim] fp32 (decode of float tokens);
 * video (B, C, 1 + (T'-1)*pt, H, W) fp32 device.  taps: optional fp32 [B*T'*H'*W', dim] in (b,t,h,w) order. */
int64_t phk_cvivit_decode_workspace_bytes(const phk_cvivit_dec_t* m, int32_t B, int32_t Tp, int32_t prec);
int phk_cvivit_decode(const phk_cvivit_dec_t* m, const int64_t* ids, const float* tokens, int32_t B,
                      int32_t Tp, float* video, void* workspace, int64_t workspace_bytes, int32_t prec,
                      const float* spatial_bias, float* tap_codes, float* tap_temporal,
                      float* tap_spatial, phk_stream_t s);

/* context_norm + to_kv of every cross-attention layer (attention.py:137-144).  Depends only on
 * the text embedding, so Phenaki.sample computes it once per call instead of once per forward.
 * context (b,L,dim_context) fp32; out_kv [depth, b*L, 2*heads*dim_head] fp32;
 * scratch 3*b*L*dim_context floats (the normalised text rows; behind them, PHK_PREC_BF16X3 only, their split copy). */
int phk_maskgit_context_kv(const phk_maskgit_t* m, const float* context, int32_t b, int32_t L,
                           float* out_kv, float* scratch, int32_t prec, phk_stream_t s);

/* MaskGit.forward / TokenCritic.forward (phenaki_pytorch.py:163-213, 265-302), optionally for a
 * classifier-free-guidance pair (:149-161): ids (b,n) int64; sequences [0,b) are the conditional
 * pass and, when cfg_pair!=0, sequences [b,2b) replay the same ids with the text mask dropped
 * (cond_drop_prob = 1).  ctx_kv from phk_maskgit_context_kv or NULL (no context: cross-attention
 * skipped, attention.py:327); text_mask uint8 (b,L); video_mask uint8 (b,n) or NULL;
 * pos_bias: cached phk_cpb_bias(pos_bias, pt, ph, pw) [heads,n,n] or NULL (recomputed).
 * out: MaskGit logits fp32 [(1+cfg_pair)*b*n, num_tokens], or final embeds [.., dim] when
 * return_embeds!=0 or the model is a critic (its Linear(dim,1) head is phk_critic_scores). */
int64_t phk_maskgit_workspace_bytes(const phk_maskgit_t* m, int32_t b, int32_t n, int32_t L,
                                    int32_t cfg_pair, int32_t prec);
int phk_maskgit_forward(const phk_maskgit_t* m, const int64_t* ids, int32_t b, int32_t n,
                        int32_t pt, int32_t ph, int32_t pw, const float* ctx_kv, int32_t L,
                        const uint8_t* text_mask, const uint8_t* video_mask, int32_t cfg_pair,
                        int32_t return_embeds, const float* pos_bias, float* out, void* workspace,
                        int64_t workspace_bytes, int32_t prec, phk_stream_t s);

/* e_cfg = norm_out(x_null) + cond_scale * (norm_out(x_cond) - norm_out(x_null)) as bf16 [rows, dim]
 * (attention.py:308,332 + phenaki_pytorch.py:161).  to_logits is linear, so applying the classifier-free-guidance
 * combination to the final embeddings equals applying it to the two logits tensors; dim % 128 == 0, dim <= 1024. */
int phk_layernorm_cfg(const float* x_cond, const float* x_null, const float* gamma, const float* beta,
                      float cond_scale, void* out_bf16, int64_t rows, int32_t dim, phk_stream_t s);

/* Fused logits head for the sampling loop (phenaki_pytorch.py:213 + 83-93 + 506-509 + 547-550): a tcgen05 GEMM whose
 * epilogue applies bias and gumbel noise (in-kernel Philox, same counter layout as phk_sample_tokens with u == NULL)
 * and reduces argmax / online softmax over the vocabulary straight out of TMEM, so the (b, n, V) logits never exist
 * in memory.  emb bf16 [emb_rows >= n_tokens, dim <= 512] = guided embeddings (phk_layernorm_cfg, or plain norm_out
 * rows when there is no guidance); the 128-token A panel stays resident in shared memory, W streams through TMA.
 * Noise as phk_sample_tokens with u == NULL, token t of the call being row r = t: counter offset + t * ceil(V/4) + v/4,
 * word v%4, the same uniform and gumbel transform.  Outputs as phk_sample_tokens. */
int64_t phk_head_sample_scratch_bytes(int32_t n_tokens);
int phk_head_sample(const void* emb, int64_t ld_emb, int64_t emb_rows, const void* W, int64_t ldw, const float* bias,
                    int32_t n_tokens, int32_t V, int32_t dim, float temperature, uint64_t seed, uint64_t offset,
                    const uint8_t* mask, int64_t* ids, int64_t* pred_out, float* score_out, void* scratch,
                    int64_t scratch_bytes, phk_stream_t s);

/* phk_head_sample with the noise key in DEVICE memory: rng_state = uint64[2] {seed, offset} (NULL: the by-value pair).
 * A CUDA graph that captured the call bakes the pointer, not the values, so every replay can draw fresh noise. */
int phk_head_sample_rng(const void* emb, int64_t ld_emb, int64_t emb_rows, const void* W, int64_t ldw, const float* bias,
                        int32_t n_tokens, int32_t V, int32_t dim, float temperature, uint64_t seed, uint64_t offset,
                        const uint64_t* rng_state, const uint8_t* mask, int64_t* ids, int64_t* pred_out, float* score_out,
                        void* scratch, int64_t scratch_bytes, phk_stream_t s);

/* The tail of one demasking iteration restricted to the tokens that are still masked.  Rows do not interact after the
 * last attention, and the reference keeps the prediction and the confidence only where the mask is set
 * (`ids = where(mask, pred, ids)`, phenaki_pytorch.py:509; `where(mask, 1 - p, -1e4)`, :547-550), so the final LayerNorm,
 * the guidance combination and the logits head are computed for the masked rows only: positions are compacted (exactly
 * k per sequence -- the count phk_topk_mask was given, known on the host), norm_out + CFG are gathered into a bf16
 * [b*k, dim] operand, phk_head_sample runs on those rows and the results are scattered back.
 * x_cond / x_null fp32 [b*n, dim]: the residual stream BEFORE norm_out of the two halves; head_w bf16 [V, ldw];
 * mask / ids / pred_out / score_out as phk_sample_tokens, with score = -1e4 and pred = id at unmasked positions;
 * rng_state as phk_head_sample_rng.  The noise counters follow the COMPACT row: the j-th masked position (in position
 * order) of sequence i draws from counters offset + (i * k + j) * ceil(V/4) + v/4, whatever its position. */
int64_t phk_sample_tail_scratch_bytes(int32_t b, int32_t k, int32_t dim);
int phk_sample_tail(const float* x_cond, const float* x_null, const float* gamma, const float* beta, float cond_scale,
                    const void* head_w, int64_t ldw, const float* head_b, int32_t b, int32_t n, int32_t k, int32_t V,
                    int32_t dim, float temperature, uint64_t seed, uint64_t offset, const uint64_t* rng_state,
                    const uint8_t* mask, int64_t* ids, int64_t* pred_out, float* score_out, void* scratch,
                    int64_t scratch_bytes, phk_stream_t s);
/* The same when the residual stream carries a prime prefix: the row of sampled token t of sequence i is
 * i * src_stride + src_off + t (src_stride = prime_len + n, src_off = prime_len; phenaki_pytorch.py:493, 503-504). */
int phk_sample_tail_rows(const float* x_cond, const float* x_null, const float* gamma, const float* beta, float cond_scale,
                         const void* head_w, int64_t ldw, const float* head_b, int32_t b, int32_t n, int32_t k, int32_t V,
                         int32_t dim, float temperature, uint64_t seed, uint64_t offset, const uint64_t* rng_state,
                         const uint8_t* mask, int64_t* ids, int64_t* pred_out, float* score_out, int32_t src_stride,
                         int32_t src_off, void* scratch, int64_t scratch_bytes, phk_stream_t s);

/* One demasking iteration's network half for the sampling loop (phenaki_pytorch.py:495-509, 547-550): MaskGit forward
 * of the CFG pair (as phk_maskgit_forward with cfg_pair=1) + phk_head_sample.  bf16 weights required, cond_scale != 1,
 * no priming.  ids_in (b,n) = current (partly masked) ids; ids/pred_out/score_out/mask as phk_sample_tokens.
 * masked_per_seq: the number of set mask entries of EVERY sequence when the caller knows it (the k it gave
 * phk_topk_mask), else 0.  With 0 < masked_per_seq < n the final LayerNorm, the guidance and the logits head run on the
 * masked rows only (phk_sample_tail); pred_out is then the current id at unmasked positions. */
int64_t phk_maskgit_sample_workspace_bytes(const phk_maskgit_t* m, int32_t b, int32_t n, int32_t L);
int phk_maskgit_sample_step(const phk_maskgit_t* m, const int64_t* ids_in, int32_t b, int32_t n, int32_t pt,
                            int32_t ph, int32_t pw, const float* ctx_kv, int32_t L, const uint8_t* text_mask,
                            const uint8_t* video_mask, const float* pos_bias, float cond_scale, float temperature,
                            uint64_t seed, uint64_t offset, const uint8_t* mask, int64_t* ids, int64_t* pred_out,
                            float* score_out, int32_t masked_per_seq, void* workspace, int64_t workspace_bytes,
                            phk_stream_t s);
/* With a prime prefix (Phenaki.sample(prime_frames=...), the scene chains of make_video): ids_in (b, n) = prime ids
 * followed by the tokens being sampled, n = prime_len + sampled tokens; mask / ids / pred_out / score_out
 * (b, n - prime_len) cover the sampled tokens; masked_per_seq > 0 is required (the head runs on the masked rows only). */
int phk_maskgit_sample_step_primed(const phk_maskgit_t* m, const int64_t* ids_in, int32_t b, int32_t n, int32_t pt,
                                   int32_t ph, int32_t pw, const float* ctx_kv, int32_t L, const uint8_t* text_mask,
                                   const float* pos_bias, float cond_scale, float temperature, uint64_t seed,
                                   uint64_t offset, const uint8_t* mask, int64_t* ids, int64_t* pred_out, float* score_out,
                                   int32_t masked_per_seq, int32_t prime_len, void* workspace, int64_t workspace_bytes,
                                   phk_stream_t s);

/* rng_state[1] += stride on the stream (device-resident noise key, see phk_head_sample_rng) */
int phk_rng_advance(uint64_t* rng_state, uint64_t stride, phk_stream_t s);

/* Test hook of the in-kernel sampling noise (phk_sample_tokens with u == NULL): n device entries,
 * bits_out[i] = Philox word i%4 of counter offset + i/4 under key seed (bits_in == NULL) or bits_in[i];
 * gumbel_out[i] = the sampling kernels' gumbel transform of that word. */
int phk_noise_probe(const uint32_t* bits_in, uint64_t seed, uint64_t offset, int64_t n, uint32_t* bits_out,
                    float* gumbel_out, phk_stream_t s);

/* One WHOLE demasking iteration (phenaki_pytorch.py:485-509, 547-550) as one call:
 *   [k_remask > 0:  mask = scatter(topk(scores, k_remask)); ids = where(mask, mask_id, ids)]      (phk_topk_mask)
 *   -> MaskGit forward of the CFG pair on ids -> tail on the masked rows -> ids, pred, scores updated IN PLACE
 *   -> rng_state[1] += b*n*ceil(V/4) + 1 (the noise counters the iteration consumed).
 * k_remask == 0 is the first iteration (every token masked: mask must be all ones).  rng_state: device uint64[2]
 * {seed, offset}.  With PHK_STEP_GRAPH=1 the launch sequence is captured into a CUDA graph the second time the same
 * arguments are seen (same table contents, pointers, shape, scalars) and later calls are ONE cudaGraphLaunch -- the
 * noise key and the token state live in device memory, so nothing that changes between calls is baked in.  Buffers
 * must therefore be stable across calls.  bf16 weights, cond_scale != 1, no priming (as phk_maskgit_sample_step). */
int phk_maskgit_demask_iteration(const phk_maskgit_t* m, int64_t* ids, uint8_t* mask, float* scores, int64_t* pred,
                                 int32_t b, int32_t n, int32_t pt, int32_t ph, int32_t pw, const float* ctx_kv, int32_t L,
                                 const uint8_t* text_mask, const float* pos_bias, float cond_scale, float temperature,
                                 uint64_t* rng_state, int32_t k_remask, void* workspace, int64_t workspace_bytes,
                                 phk_stream_t s);

/* The iteration of a sample WITH a critic and / or a prime prefix (phenaki_pytorch.py:478-550; make_video's scene chains),
 * one call, replayed as a CUDA graph like phk_maskgit_demask_iteration:
 *   [k_remask > 0: phk_topk_mask on `scores`] -> ids copied behind the prime ids in token_in -> MaskGit forward of the CFG
 *   pair + tail on the masked rows: ids / pred / scores updated in place -> rng_state[1] += stride
 *   -> unless `last`: ids -> token_in, critic forward of the CFG pair, scores = head(cond, null, cond_scale) +
 *      noise_K * (u - 0.5) * noise_mult (:534-545).
 * token_in [b, prime_len + n] int64: prime ids in the first prime_len columns (written once by the caller); with
 * prime_len == 0 pass token_in == ids.  pt*ph*pw == prime_len + n.  critic: a TokenCritic table (is_critic), ctx via
 * critic_ctx_kv (or NULL: no cross attention); critic == NULL: SelfCritic -- the MaskGit's own embeddings under head_w /
 * head_b (fp32 [dim], [1]).  critic_noise: [b, n] uniform draws the caller refreshes before every call (device buffer at a
 * stable address), or NULL.  Same buffer-stability rule as phk_maskgit_demask_iteration; bf16 weights, cond_scale != 1. */
int64_t phk_maskgit_demask_iteration_critic_workspace_bytes(const phk_maskgit_t* m, const phk_maskgit_t* critic, int32_t b,
                                                            int32_t n_total, int32_t L);
int phk_maskgit_demask_iteration_critic(const phk_maskgit_t* m, const phk_maskgit_t* critic, const float* head_w,
                                        const float* head_b, int64_t* token_in, int64_t* ids, uint8_t* mask, float* scores,
                                        int64_t* pred, int32_t b, int32_t n, int32_t prime_len, int32_t pt, int32_t ph,
                                        int32_t pw, const float* ctx_kv, const float* critic_ctx_kv, int32_t L,
                                        const uint8_t* text_mask, const float* pos_bias, float cond_scale, float temperature,
                                        uint64_t* rng_state, int32_t k_remask, const float* critic_noise, float noise_K,
                                        float noise_mult, int32_t last, void* workspace, int64_t workspace_bytes,
                                        phk_stream_t s);

/* tests / A-B runs: 1 = phk_maskgit_demask_iteration replays a CUDA graph, 0 = eager, < 0 = the PHK_STEP_GRAPH default */
int phk_debug_step_graph(int32_t on);

/* ------------------------------------------------------------------------------------------ */
/* Training step (SURVEY 8f-2): Phenaki.forward (phenaki_pytorch.py:562-687)                   */
/* ------------------------------------------------------------------------------------------ */

/* One forward + loss + backward of MaskGit (masked cross entropy, :620-640) or of a critic (BCE with logits,
 * :652-675) in fp32: what `loss = phenaki(...); loss.backward()` computes for that network under torch autograd.
 * The head follows the arguments: `labels` given -> head_w [1, dim], head_b [1] + BCE (a TokenCritic table, or a
 * MaskGit table whose head members point at SelfCritic.to_pred, :307-336); otherwise to_logits + cross entropy.
 *   ids_in  (b,n) int64   network input: ids with the mask id at the masked positions (MaskGit) or with the sampled
 *                         predictions at the masked positions (critic)
 *   targets (b,n) int64 + token_mask (b,n) uint8   MaskGit: loss = mean over masked rows of CE(logits, target)
 *   labels  (b,n) float 0/1                        critic : loss = mean over all rows of BCE_with_logits(score, label)
 *   context (b,L,dim_context) fp32 raw text embeddings or NULL; text_mask (b,L) uint8; video_mask (b,n) uint8 or NULL
 *   grads   a table of the SAME layout as `m` whose float pointers address ZERO-FILLED gradient buffers of the
 *           parameters' shapes (peg.w in the parameter's own [dim, 1, 3, 3, 3] layout; bf16 members and scalars unused);
 *           d(loss_scale * loss)/d(parameter) is ACCUMULATED into it.  Parameters without a gradient in the reference
 *           (beta buffers, the self-attention context_norm) are not touched.
 *   loss_out device float: the UNSCALED loss.  logits_out: optional fp32 [b*n, num_tokens] that receives the MaskGit
 *           logits (the critic branch samples its input from them, :646).
 * The gradient-shrink trick (:199) scales the embedding gradients by shrink_alpha, as autograd does.  cond_drop_prob is
 * 0 in the reference's training forward (:594 overwrites the argument), so there is no text dropout.
 * prec: PHK_PREC_F32 = fp32 FFMA products (parity with the fp32 reference); PHK_PREC_BF16 = the forward, dgrad and
 * wgrad product of every nn.Linear on the tcgen05 GEMM (phk_gemm_bf16) with operands converted on the fly from the
 * fp32 activations / master weights (the dtype flow of torch.autocast(bfloat16)); LayerNorm, softmax, GEGLU, the
 * attention core and all gradients of non-matrix parameters stay fp32 in both modes. */
int64_t phk_maskgit_train_workspace_bytes(const phk_maskgit_t* m, int32_t b, int32_t n, int32_t L, int32_t bce_head,
                                          int32_t prec);
int phk_maskgit_train_step(const phk_maskgit_t* m, const phk_maskgit_t* grads, const int64_t* ids_in,
                           const int64_t* targets, const uint8_t* token_mask, const float* labels, int32_t b, int32_t n,
                           int32_t pt, int32_t ph, int32_t pw, const float* context, int32_t L,
                           const uint8_t* text_mask, const uint8_t* video_mask, float loss_scale, float* loss_out,
                           float* logits_out, void* workspace, int64_t workspace_bytes, int32_t prec, phk_stream_t s);
/* Data-parallel overlap: `events` (cudaEvent_t handles, count >= depth + 2) are recorded by the NEXT phk_maskgit_train_step
 * call of the calling thread, on its stream, as gradient groups become final: events[0] head + norm_out, events[1 + k]
 * transformer layer depth-1-k, events[depth + 1] embeddings + position-bias MLP (= all).  One-shot; NULL clears. */
int phk_train_set_progress_events(void** events, int32_t count);

#ifdef __cplusplus
}
#endif
#endif /* PHK_H_ */
