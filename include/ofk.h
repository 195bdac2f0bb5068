/*
 * ofk.h -- C ABI of libofk.so: the B200 (sm_100a) kernels behind the OpenFlamingo dense hot path.
 *
 * The reference (mlfoundations/open_flamingo) is pure eager PyTorch and has NO native interface; each
 * entry point below names the reference Python it replaces (paths relative to the reference repo root,
 * open_flamingo/src/...).  INTEGRATION.md shows the ctypes binding a maintainer would add.
 *
 * Conventions
 *  - All pointers are DEVICE pointers unless stated; no torch types cross this boundary.
 *  - `stream` is a cudaStream_t passed as void*.  Kernels are enqueued on it and never synchronise.
 *  - Nothing here allocates device memory: the caller owns outputs and workspaces.
 *  - Return value: 0 on success, negative OFK_ERR_* otherwise; ofk_last_error() gives the message.
 *    Nothing throws across the ABI.
 *  - bf16 tensors are raw uint16 storage (__nv_bfloat16); "f32" is IEEE float.
 *  - Row-major everywhere; `ld*` are row strides in ELEMENTS.
 */
#ifndef OFK_H_
#define OFK_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OFK_ABI_VERSION 2

enum {
  OFK_OK = 0,
  OFK_ERR_ARG = -1,    /* bad argument (shape / null / unsupported combination) */
  OFK_ERR_ALIGN = -2,  /* pointer or stride alignment violates the TMA / vector-access contract */
  OFK_ERR_CUDA = -3,   /* CUDA runtime error at launch */
  OFK_ERR_DRIVER = -4  /* driver entry point (tensor-map encode) unavailable or failed */
};

/* GEMM epilogues (fused into the tcgen05 kernel's TMEM->global stage). */
enum {
  OFK_EPI_STORE_BF16 = 0,      /* out(bf16) = acc                                            nn.Linear, helpers.py:35-37,153-155 */
  OFK_EPI_STORE_F32 = 1,       /* out(f32)  = acc                                                                               */
  OFK_EPI_ATOMIC_F32 = 2,      /* out(f32) += acc  (red.global.add; wgrad / split-K / dmedia accumulation over layers)          */
  OFK_EPI_BIAS_BF16 = 3,       /* out(bf16) = acc + bias[n]                                  ViT in_proj / out_proj (open_clip) */
  OFK_EPI_BIAS_QGELU_BF16 = 4, /* out(bf16) = quick_gelu(acc + bias[n])                      ViT mlp.c_fc + QuickGELU           */
  OFK_EPI_GELU_DUAL = 5,       /* out(bf16) = z = acc ; out2(bf16) = gelu_erf(z)             FeedForward helpers.py:19-20        */
  OFK_EPI_GATE_RESID_F32 = 6,  /* out(f32) = bf16(acc)*tanh(*gate) + aux(f32); out2(bf16)=acc (optional; gate NULL => 1)
                                  helpers.py:267-277 (x = branch * gate.tanh() + x), helpers.py:130-131 (Perceiver residuals)   */
  OFK_EPI_DGELU_BF16 = 7,      /* out(bf16) = acc * gelu_erf'(aux(bf16) = z)                 autograd of helpers.py:20           */
  OFK_EPI_BIAS_RESID_F32 = 8,  /* out(f32) = bf16(acc + bias[n]) + aux(f32)  (out may alias aux)  ViT residual adds            */
  OFK_EPI_BIAS_GELU_BF16 = 9,  /* out(bf16) = gelu_erf(acc + bias[n])                        ViT mlp.c_fc + nn.GELU (non-openai) */
  OFK_EPI_SWIGLU_DUAL = 10     /* B = packed [gate; up] weight (OFK_SWIGLU_GROUP layout below), N = 2 * I:
                                  out(bf16) [M, I] = h = bf16(bf16(silu(g)) * u), g / u = bf16(acc) of the gate / up rows;
                                  out2(bf16) [M, 2I] = raw bf16(acc) in the packed column order (optional, for the backward).
                                  A and B K-major only, N % 32 == 0.   HF LlamaMLP: act_fn(gate_proj(x)) * up_proj(x)      */
};

/* Packed SwiGLU weight: gate_proj and up_proj ([I, D] each, I % 16 == 0) interleaved in groups of OFK_SWIGLU_GROUP rows,
 *   packed row 32 j + i      = gate row 16 j + i   (i < 16)
 *   packed row 32 j + 16 + i = up   row 16 j + i
 * so each 32-column round of the GEMM epilogue holds 16 gate columns and the 16 matching up columns.  The GEMM's raw
 * output `out2` and the gradient ofk_swiglu_bwd writes use the same column order; a dgrad GEMM of that gradient against
 * the packed weight gives the gradient of the MLP input in one pass. */
#define OFK_SWIGLU_GROUP 16

const char* ofk_last_error(void);
int ofk_abi_version(void);
/* Number of kernels this library has launched since load (bench.py's `gpu_launches`). */
long long ofk_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * GEMM  out[m,n] = epi( sum_k A(m,k) * B(n,k) ), bf16 operands, fp32 accumulate in TMEM (tcgen05).
 *   a_mn_major = 0: A stored [M,K] (K contiguous).  = 1: A stored [K,M] (M contiguous).
 *   b_mn_major = 0: B stored [N,K] (K contiguous).  = 1: B stored [K,N] (N contiguous).
 *   forward  y = x W^T       : A=x [R,in]  (0), B=W [out,in] (0)         nn.Linear (helpers.py:18-21,35-37,153-155)
 *   dgrad    dx = dy W       : A=dy [R,out](0), B=W [out,in] (1), K=out  autograd of the above
 *   wgrad    dW += dy^T x    : A=dy [R,out](1), B=x [R,in]   (1), K=R    autograd of the above (ATOMIC_F32)
 *   splits  : split-K factor (ATOMIC_F32 only).  block_n: 0 = auto, else 128 or 256.
 * Requirements: N % 16 == 0; operand base pointers 16-byte aligned, lda/ldb % 8 == 0.
 */
int ofk_gemm_bf16(int epi, int a_mn_major, int b_mn_major, const void* A, long long lda, const void* B,
                  long long ldb, int M, int N, int K, int splits, int block_n, void* out, long long ldo,
                  void* out2, long long ldo2, const void* aux, long long ldaux, const float* bias,
                  const float* gate, void* stream);

/* Same GEMM with a caller-owned scratch buffer that enables the "tail split": when the last round of the persistent
 * 256 x 256-tile grid would be at most half full (e.g. the N = 2048 projections of MPT-1B: 256 tiles on 74 SM pairs =
 * 3.46 rounds), its tiles are cut into 2-4 k-slices that run on the otherwise idle SM pairs; the slices exchange fp32
 * partial accumulators through `workspace` (L2-resident) and the last slice applies the fused epilogue, so results
 * do not depend on whether the split is taken beyond fp32 summation order.  `workspace` must hold at least
 * ofk_gemm_workspace_bytes() bytes, be 16-byte aligned, have its first 16384 bytes zeroed once before first use, and
 * must not be shared by GEMMs that may run concurrently (one buffer per stream).  NULL = plain ofk_gemm_bf16.
 * Replaces the same reference lines as ofk_gemm_bf16. */
long long ofk_gemm_workspace_bytes(void);
int ofk_gemm_bf16_ws(int epi, int a_mn_major, int b_mn_major, const void* A, long long lda, const void* B,
                     long long ldb, int M, int N, int K, int splits, int block_n, void* out, long long ldo,
                     void* out2, long long ldo2, const void* aux, long long ldaux, const float* bias,
                     const float* gate, void* workspace, long long workspace_bytes, void* stream);

/* Leave `n` SMs (rounded down to whole pairs, at most 64) out of every persistent GEMM grid launched from now on; returns
 * the previous value.  The data-parallel step uses it while gradient-chunk all-reduces are in flight (train.GradBucket):
 * a persistent grid that owns all 148 SMs lets NCCL's CTAs in only at kernel boundaries, which serialises the
 * "overlapped" reduction behind each GEMM.  0 restores the full grid. */
int ofk_gemm_reserve_sms(int n);

/* Same GEMM with grouped row maps (logical row r -> (r / rows_per_group) * group_stride + group_offset + r % rpg):
 *   out_*  : where the rows of `out` go inside a larger interleaved buffer (STORE_BF16 / BIAS_BF16 / STORE_F32);
 *   a_k_*  : which physical rows of an MN-major A form the reduction dimension (rows_per_group % 64 == 0).
 * Lets PerceiverAttention's k/v for the media tokens and for the latents (helpers.py:53-54: to_kv(cat(x, latents)))
 * be produced by two GEMMs that write straight into the concatenated [b*T, v+n, 2*inner] layout, and lets the
 * wgrads reduce over only the media (or only the latent) rows of the concatenated gradient.  0 = identity. */
int ofk_gemm_bf16_grouped(int epi, int a_mn_major, int b_mn_major, const void* A, long long lda, const void* B,
                          long long ldb, int M, int N, int K, int splits, int block_n, void* out, long long ldo,
                          const float* bias, int out_rows_per_group, int out_group_stride, int out_group_offset,
                          int a_k_rows_per_group, int a_k_group_stride, int a_k_group_offset, void* stream);

/* ------------------------------------------------------------------------------------------------
 * LayerNorm over the last dim (eps inside sqrt, affine), fp32 statistics.  nn.LayerNorm at
 * helpers.py:17,32-33,47-48,105,132,151,184.
 *   x: [rows, D] f32 (ldx).  y: bf16 (y_is_f32 = 0) or f32, written at
 *   row index  (r / rows_per_group) * group_stride + group_offset + r % rows_per_group  of y (ldy) --
 *   this lets two LayerNorms write the two halves of PerceiverAttention's cat((x, latents), -2)
 *   (helpers.py:53) in place (rows_per_group <= 0: identity mapping).  mean/rstd: [rows] f32 outputs (may be
 *   NULL).  D % 4 == 0, D <= 4096.
 */
int ofk_layernorm_fwd(const float* x, long long ldx, const float* gamma, const float* beta,
                      float eps, int rows, int D, void* y, int y_is_f32, long long ldy, int rows_per_group,
                      int group_stride, int group_offset, float* mean, float* rstd, void* stream);

/* LayerNorm backward.  dy: [rows, D] bf16 or f32 (same row mapping as fwd via dy_* group args);
 * x: f32 [rows, D]; dx(f32) = LN'(dy) (+ dx_add if non-NULL; dx_add may alias dx); dx NULL = parameter
 * gradients only (PerceiverAttention.norm_media: its input, the frozen ViT features, needs no gradient).
 * dgamma/dbeta (f32 [D]) are ACCUMULATED (+=).  workspace: >= ofk_layernorm_bwd_workspace(rows, D) bytes. */
long long ofk_layernorm_bwd_workspace(int rows, int D);
int ofk_layernorm_bwd(const void* dy, int dy_is_f32, long long lddy, int rows_per_group, int group_stride,
                      int group_offset, const float* x, long long ldx, const float* gamma, const float* mean,
                      const float* rstd, int rows, int D, float* dx, long long lddx, const float* dx_add,
                      long long ldadd, float* dgamma, float* dbeta, void* workspace, void* stream);

/* RMSNorm over the last dim, fp32 statistics: y(bf16) = bf16(gamma * (x * rsqrt(mean(x^2) + eps))).  The variant of
 * the LayerNorm kernels above without centring and without beta.  HF LlamaRMSNorm.forward (input_layernorm /
 * post_attention_layernorm of LlamaDecoderLayer) followed by the autocast cast in front of the next Linear.
 *   x: [rows, D] f32 (ldx); y: bf16 (ldy); rstd: [rows] f32 output (may be NULL).  D % 4 == 0, D <= 4096. */
int ofk_rmsnorm_fwd(const float* x, long long ldx, const float* gamma, float eps, int rows, int D, void* y,
                    long long ldy, float* rstd, void* stream);

/* RMSNorm backward, input gradient only (frozen gamma): dx(f32) = RMSNorm'(dy) (+ dx_add if non-NULL; may alias dx).
 * dy: [rows, D] bf16 (dy_is_f32 = 0) or f32.  Autograd of HF LlamaRMSNorm.forward. */
int ofk_rmsnorm_bwd(const void* dy, int dy_is_f32, long long lddy, const float* x, long long ldx, const float* gamma,
                    const float* rstd, int rows, int D, float* dx, long long lddx, const float* dx_add, long long ldadd,
                    void* stream);

/* Rotary position embedding, in place on bf16 rows: x is [batch * T, ldx]; its first nheads * head_dim columns are
 * nheads heads (q and k of a fused [q | k | v] row: nheads = 2 * heads).  Row r = b * T + t uses
 * cos / sin[b * cs_bstride + t * head_dim + i] (f32, cs_bstride 0 or T * head_dim).
 *   inverse = 0: x = bf16(x * cos + rotate_half(x) * sin), products and sum in f32 (HF apply_rotary_pos_emb under
 *                autocast: bf16 q/k times f32 cos/sin, cast to bf16 by SDPA).
 *   inverse = 1: the transposed rotation with autograd's rounding (each branch's gradient rounded to bf16, then
 *                summed): turns dq / dk of the rotated tensors into gradients of the projection outputs.
 * head_dim % 16 == 0, ldx % 8 == 0, x 16-byte aligned. */
int ofk_rope(void* x, long long ldx, int batch, int T, int nheads, int head_dim, const float* cos, const float* sin,
             long long cs_bstride, int inverse, void* stream);

/* SwiGLU backward (autograd of HF LlamaMLP's act_fn(gate_proj(x)) * up_proj(x) under autocast):
 *   a = bf16(silu(g)),  du = bf16(dh * a),  dg = bf16(bf16(dh * u) * silu'(g))
 * dh: [rows, I] bf16; gu: [rows, 2I] bf16 packed g / u (out2 of OFK_EPI_SWIGLU_DUAL); dgu: [rows, 2I] bf16 in the same
 * packed order.  I % 16 == 0, row strides % 8 == 0. */
int ofk_swiglu_bwd(const void* dh, long long lddh, const void* gu, long long ldgu, int rows, int I, void* dgu,
                   long long lddgu, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Attention core  O = softmax(scale * Q K^T + mask) V  per (batch, head), head_dim = 64, bf16 in/out,
 * fp32 softmax, online (flash-style).
 * Default implementation (csrc/attention_tc.cu): Q/K/V (and dO) tiles staged by TMA (cp.async.bulk.tensor, 128-byte
 * swizzle), QK^T / PV and the five backward contractions as tcgen05.mma with TMEM accumulators, lane-per-row softmax
 * on the TMEM read-out, P / dS through swizzled shared memory.  It needs batch strides == rows * row stride and
 * 16-byte aligned bases; any other layout runs the mma.sync kernels of csrc/attention.cu (same results).
 *   q: [batch, nq, heads*64] (ldq row stride), k/v: [batch, nk, heads*64] (ldk/ldv), o like q (ldo).
 *   q_bstride/k_bstride...: batch strides in elements.  lse: [batch, heads, nq] f32 (log2 domain, for bwd).
 *   mask_mode: 0 = none                                              PerceiverAttention helpers.py:58-63, ViT MHA
 *              1 = media mask, text_time == block+1  (torch.eq)       MaskedCrossAttention helpers.py:196-229
 *              2 = media mask, text_time >= block+1  (torch.ge)       only_attend_immediate_media=False
 *   text_time: [batch, nq] int32 (cumsum of media_locations, helpers.py:199-208); keys are grouped in
 *   blocks of `keys_per_media` (= 64 latents).  Rows with no allowed key (and, for mode 1, text_time == 0,
 *   helpers.py:223-229) produce exact zeros.
 */
int ofk_attn_fwd(const void* q, const void* k, const void* v, void* o, float* lse, int batch, int heads, int nq,
                 int nk, long long q_bstride, long long ldq, long long k_bstride, long long ldk,
                 long long v_bstride, long long ldv, long long o_bstride, long long ldo, float scale,
                 int mask_mode, const int* text_time, int keys_per_media, void* stream);

/* Scratch the tensor-core backward needs: an fp32 dQ accumulator [batch*nq, heads*head_dim] whenever more than one
 * 128-key tile contributes to a query row (0 bytes when nk <= 128).  Caller-owned, 16-byte aligned, need not be
 * initialised.  Without it (NULL / too small) the backward runs the mma.sync kernels. */
long long ofk_attn_bwd_workspace_bytes(int batch, int heads, int head_dim, int nq, int nk);

/* Backward of the above.  delta: [batch, heads, nq] f32 scratch.  dq like q; dk/dv like k/v (bf16).
 * dq/dk/dv are fully overwritten.  */
int ofk_attn_bwd(const void* q, const void* k, const void* v, const void* o, const void* d_o, const float* lse,
                 float* delta, void* dq, void* dk, void* dv, int batch, int heads, int nq, int nk,
                 long long q_bstride, long long ldq, long long k_bstride, long long ldk, long long v_bstride,
                 long long ldv, long long o_bstride, long long ldo, long long dq_bstride, long long lddq,
                 long long dk_bstride, long long lddk, long long dv_bstride, long long lddv, float scale,
                 int mask_mode, const int* text_time, int keys_per_media, void* workspace, long long workspace_bytes,
                 void* stream);

/* ------------------------------------------------------------------------------------------------
 * Dense self-attention core of the frozen LM's decoder blocks (HF MptAttention; reached via
 * flamingo_lm.py:63-65 -- SURVEY.md section 8f rank 1).  head_dim 64 or 128.  Same TMA + tcgen05 implementation
 * (and the same mma.sync path for other layouts) as ofk_attn_fwd / ofk_attn_bwd.
 *   S = scale * Q K^T + slopes[h] * key_index  (ALiBi; slopes NULL = no bias)
 *   masked (mask[b, q, k] != 0, mask: [batch, nq, nk] bytes or NULL; and/or causal: key > query + nk - nq)
 *   scores take "finfo.min" exactly like masked_fill: a fully masked row attends uniformly.
 *   pure_causal_flag: optional DEVICE int; nonzero means "the mask is exactly the causal rule" (all-ones HF
 *   attention_mask): the kernel then ignores `mask`, applies the causal rule and skips key tiles above the
 *   diagonal -- a device-side decision, so no host synchronisation is needed to pick the fast path.
 *   lse: [batch, heads, nq] f32, log2 domain (consumed only by ofk_attn_dense_bwd).
 * Backward is dgrad only (the LM is frozen): dq/dk/dv bf16, fully overwritten; workspace as for ofk_attn_bwd.
 */
int ofk_attn_dense_fwd(const void* q, const void* k, const void* v, void* o, float* lse, int batch, int heads,
                       int head_dim, int nq, int nk, long long q_bstride, long long ldq, long long k_bstride,
                       long long ldk, long long v_bstride, long long ldv, long long o_bstride, long long ldo,
                       float scale, int causal, const unsigned char* mask, const float* slopes,
                       const int* pure_causal_flag, void* stream);
int ofk_attn_dense_bwd(const void* q, const void* k, const void* v, const void* o, const void* d_o,
                       const float* lse, float* delta, void* dq, void* dk, void* dv, int batch, int heads,
                       int head_dim, int nq, int nk, long long q_bstride, long long ldq, long long k_bstride,
                       long long ldk, long long v_bstride, long long ldv, long long o_bstride, long long ldo,
                       long long dq_bstride, long long lddq, long long dk_bstride, long long lddk,
                       long long dv_bstride, long long lddv, float scale, int causal, const unsigned char* mask,
                       const float* slopes, const int* pure_causal_flag, void* workspace, long long workspace_bytes,
                       void* stream);

/* Attention implementation switch, for A/B measurements and for the parity tests that compare the two paths:
 * nonzero = always use the mma.sync kernels; 0 = tensor-core path whenever the layout allows (the default, unless
 * the environment variable OFK_ATTN_LEGACY=1 is set when the library is loaded).  Returns the previous setting.
 * ofk_attn_tc_launch_count(): how many tcgen05 attention kernels (forward or backward) have been launched. */
int ofk_attn_force_legacy(int on);
long long ofk_attn_tc_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * Small fused elementwise / reduction kernels.
 */
/* text_time[b, t] = inclusive cumsum over t of (ids[b,t] == media_id)   (helpers.py:208; flamingo.py:310)
 * or, cached-media mode, count_nonzero(media_locations[b,:]) broadcast (helpers.py:199-205). */
int ofk_text_time(const long long* input_ids, long long media_token_id, int batch, int t_txt, int n_loc,
                  const unsigned char* media_locations, int use_cached_media, int* text_time, void* stream);

/* Training labels on the device (train_utils.py:102-106 for image-text pairs, :126-149 for interleaved MMC4 rows):
 * labels = input_ids with pad_token_id and media_token_id replaced by -100; with interleaved != 0 also every token
 * before the row's first <image> and every token after an <|endofchunk|> up to the next <image> (the
 * <|endofchunk|> keeps its label).  Replaces the reference's per-row Python while-loops; int64 in / out,
 * row strides in elements, rows independent; bit-exact. */
int ofk_make_labels(const long long* input_ids, long long ld_ids, int batch, int t_txt, long long pad_token_id,
                    long long media_token_id, long long endofchunk_token_id, int interleaved, long long* labels,
                    long long ld_labels, void* stream);

/* dst(bf16) = src(f32), n elements (n % 8 == 0 fast path). */
int ofk_cast_f32_bf16(const float* src, void* dst, long long n, void* stream);

/* Gate backward (autograd of helpers.py:274,277):
 *   dbranch(bf16)[i] = dout(f32)[i] * tanh(*gate);  dgate[0] += (1 - tanh(*gate)^2) * sum_i dout[i]*branch(bf16)[i]
 * gate NULL => multiplier 1 and no dgate (plain residual branch, helpers.py:130-131). */
int ofk_gate_bwd(const float* dout, const void* branch, const float* gate, void* dbranch, float* dgate,
                 long long n, void* stream);

/* dst(f32) += src(f32) */
int ofk_add_f32(float* dst, const float* src, long long n, void* stream);

/* ViT patch extraction: images [n, 3, H, W] f32 NCHW -> patches [n * (H/P)*(W/P), ldp] bf16 with the
 * (c, ph, pw) ordering of a conv weight [out, 3, P, P] flattened; columns >= 3*P*P are zero.  Replaces the
 * stride-P conv of open_clip VisionTransformer.conv1 (third party; call site flamingo.py:195). */
int ofk_patchify(const float* images, int n, int H, int W, int P, void* patches, long long ldp, void* stream);

/* tokens[n, 1 + g, D] f32 = cat(class_emb, patch_emb(bf16)[n, g, D]) + pos_emb[1+g, D]   (open_clip ViT) */
int ofk_vit_assemble(const void* patch_emb, const float* class_emb, const float* pos_emb, int n, int g, int D,
                     float* tokens, void* stream);

/* Shifted causal-LM cross-entropy on the LM-head logits (the loss Flamingo.forward returns with labels,
 * flamingo.py:111-117 -> HF ForCausalLMLoss: float logits, labels shifted by one, mean over non-ignored).
 *   logits: [rows = B*T, vocab] bf16 or f32 (ld); labels: [B, T] int64 (host-unshifted when shift_labels = 1).
 *   fwd: lse[rows]; *loss_sum += sum(lse - logit[target]); *count += #non-ignored rows.  (caller zeroes them)
 *   bwd: dlogits = (softmax - onehot) * (*grad_scale) / max(*count, 1) for non-ignored rows, 0 otherwise. */
int ofk_ce_fwd(const void* logits, int logits_is_f32, long long ld, long long rows, int vocab,
               const long long* labels, int T, int shift_labels, long long ignore_index, float* lse,
               float* loss_sum, float* count, void* stream);
int ofk_ce_bwd(const void* logits, int logits_is_f32, long long ld, long long rows, int vocab,
               const long long* labels, int T, int shift_labels, long long ignore_index, const float* lse,
               const float* grad_scale, const float* count, void* dlogits, long long ldd, void* stream);

/* Fused AdamW over a flat f32 parameter / gradient buffer (train.py:392-415, train_utils.py:208-216):
 * grads are first scaled by clip_scale (global-norm clip), decoupled weight decay `wd`.
 * Also emits the bf16 operand copy for the next step's GEMMs (w_bf16 may be NULL).
 * step_dev / lr_dev (optional DEVICE floats) override bias_corr1/2 (= 1 - beta^step) and lr, so that a captured
 * CUDA graph of the training step stays valid as the step count and learning-rate schedule advance. */
int ofk_adamw(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, void* w_bf16, long long n,
              float lr, float beta1, float beta2, float eps, float wd, float bias_corr1, float bias_corr2,
              const float* clip_scale, const float* step_dev, const float* lr_dev, void* stream);

/* out[0] += sum_i x[i]^2   (global grad norm, train_utils.py:208) */
int ofk_sumsq(const float* x, long long n, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* OFK_H_ */
