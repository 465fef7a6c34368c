/* vitk — C ABI of the B200 (sm_100a) kernel library behind the ViT-B/16 fine-tuning hot path.
 *
 * This is the drop-in boundary.  The reference (/root/reference/ViT-Training.py:83-90,120-132)
 * reaches the hot path through PyTorch modules of HuggingFace transformers
 * (HF = transformers/models/vit/modeling_vit.py, v5.5.0), which dispatch to ATen operators.
 * Each entry point below replaces the ATen operator(s) named in its comment; the Python side
 * (chest-x-ray-vit_b200/ops.py) binds them with ctypes and exposes them as torch custom ops.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only.  All pointers are DEVICE pointers unless
 *     named host_*.  bf16 buffers are passed as void* / uint16_t*.
 *   - every call is asynchronous on `stream` (a cudaStream_t); nothing synchronises the host,
 *     nothing allocates or frees device memory.  Workspaces are caller-provided.
 *   - return 0 on success, >0 = cudaError_t, <0 = argument/shape error (VITK_E*).
 *     vitk_last_error() returns a thread-local message for the last non-zero return.
 *   - thread-safe / re-entrant (PyTorch calls backward from its autograd thread).
 */
#ifndef VITK_H_
#define VITK_H_

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define VITK_API __attribute__((visibility("default")))
#else
#define VITK_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define VITK_VERSION 100

#define VITK_EINVAL (-1)   /* bad argument / unsupported shape */
#define VITK_EALIGN (-2)   /* pointer or leading dimension not aligned as required */
#define VITK_EDEVICE (-3)  /* not an sm_100 device */
#define VITK_EDRIVER (-4)  /* cuTensorMapEncodeTiled unavailable / failed */

typedef void* vitk_stream_t; /* cudaStream_t */

VITK_API int vitk_version(void);
/* 0 iff device `dev` has compute capability 10.x; the library refuses to run elsewhere. */
VITK_API int vitk_check_device(int dev);
VITK_API const char* vitk_last_error(void);

/* ------------------------------------------------------------------ input normalisation
 * Replaces ToTensor+Normalize on img.convert("RGB") (ViT-Training.py:60-66) fused with the
 * im2col of Conv2d(k=s=patch) (HF:151,166).  gray u8 [B,H,W] → bf16 [B*(H/p)*(W/p), 3*p*p],
 * column k = c*p*p + ky*p + kx, value (g/255 - mean[c]) / std[c].  host_mean/std: 3 floats. */
VITK_API int vitk_patchify_u8(const uint8_t* gray, int64_t B, int64_t H, int64_t W, int64_t patch,
                     const float* host_mean, const float* host_std, void* out_bf16, vitk_stream_t stream);
/* Same im2col for the drop-in fp32 NCHW input [B,3,H,W] (collate_fn, ViT-Training.py:77-80). */
VITK_API int vitk_patchify_f32(const float* pixel_values, int64_t B, int64_t H, int64_t W, int64_t patch,
                      void* out_bf16, vitk_stream_t stream);

/* RandomHorizontalFlip of the training transform (ViT-Training.py:61), on the device: image b of gray u8 [B,H,W] is
 * mirrored in place along W iff mask[b] != 0 (the caller draws the mask, p = 0.5 in torchvision).  A pure permutation of
 * bytes: identical to flipping before ToTensor+Normalize.  W % 16 == 0. */
VITK_API int vitk_hflip_u8(uint8_t* gray, const uint8_t* mask, int64_t B, int64_t H, int64_t W, vitk_stream_t stream);

/* ------------------------------------------------------------------ LayerNorm
 * Replaces aten::native_layer_norm / native_layer_norm_backward (HF:325-326,333,340,455).
 * x fp32 [M,D] (row stride ldx elements) → y bf16 [M,D]; mean/rstd fp32 [M] saved for backward. */
/* (_rows: logical row r is written to physical row r·row_stride of y / mean / rstd — row_stride = T normalises the CLS
 * rows of a [B,T,D] tensor in place, as vitk_layernorm_bwd_rows reads them.) */
VITK_API int vitk_layernorm_fwd_rows(const float* x, int64_t ldx, const float* gamma, const float* beta, float eps, int64_t M,
                  int64_t D, int64_t row_stride, void* y_bf16, float* mean, float* rstd, vitk_stream_t stream);
VITK_API int vitk_layernorm_fwd(const float* x, int64_t ldx, const float* gamma, const float* beta, float eps,
                       int64_t M, int64_t D, void* y_bf16, float* mean, float* rstd, vitk_stream_t stream);
/* dx = dres + LNbwd(dy) (bf16 [M,D]; dres may be NULL); dgamma/dbeta fp32 [D] are ACCUMULATED
 * (+=) with atomics, so zero them first for a plain gradient.  dxsum (optional, fp32 [D]) += Σ_rows dx:
 * dx is also the output gradient of the Linear that fed this residual stream, so this is that layer's
 * bias gradient (aten::sum in HF's AddmmBackward) without another pass over dx. */
VITK_API int vitk_layernorm_bwd(const void* dy_bf16, const float* x, int64_t ldx, const float* mean, const float* rstd,
                       const float* gamma, const void* dres_bf16, int64_t M, int64_t D, void* dx_bf16,
                       float* dgamma, float* dbeta, float* dxsum, vitk_stream_t stream);
/* Same over a strided subset of rows: logical row r is physical row r·row_stride of dy / dres / dx / mean / rstd
 * (x uses ldx).  With row_stride = T and ldx = T·D it touches only the B CLS rows of [B,T,D] tensors — all that
 * carries gradient in the top encoder layer (HF modeling_vit.py:641 selects sequence_output[:, 0]). */
VITK_API int vitk_layernorm_bwd_rows(const void* dy_bf16, const float* x, int64_t ldx, const float* mean, const float* rstd,
                       const float* gamma, const void* dres_bf16, int64_t M, int64_t D, int64_t row_stride,
                       void* dx_bf16, float* dgamma, float* dbeta, float* dxsum, vitk_stream_t stream);

/* ------------------------------------------------------------------ dense contraction
 * Replaces aten::addmm / aten::mm (+ fused bias/GELU/residual elementwise ops) for the patch
 * embedding, QKV, attention-output and MLP projections and their dgrad/wgrad (HF:166,228-230,
 * 266,297-298,309-311).  D[M,N] = A·Bᵀ with logical A [M,K], logical B [N,K], bf16 in, fp32
 * accumulate in TMEM (tcgen05.mma), operands staged by TMA.
 *   a_mn_major = 0: A stored [M,K] with K contiguous, lda = row stride (elements)
 *   a_mn_major = 1: A stored [K,M] with M contiguous, lda = stride between k-rows
 *   (same for B with N).  lda/ldb multiples of 8, base pointers 16-byte aligned.
 * N must be a multiple of 128.  Two kernels sit behind this entry point: a CTA-pair kernel
 * (tcgen05 cta_group::2, 256×{128,192,256} tiles, epilogue through swizzled shared memory and TMA
 * stores / TMA reduce-add) used whenever it applies, and a single-CTA kernel (128×N tiles) that
 * also handles the row-remapping patch-embedding epilogue. */
enum vitk_epilogue {
  VITK_EPI_STORE_BF16 = 0,      /* d bf16 = acc                                  (dgrad)   */
  VITK_EPI_BIAS_BF16 = 1,       /* d bf16 = acc + bias[n]                        (QKV)     */
  VITK_EPI_BIAS_GELU_BF16 = 2,  /* d bf16 = u = acc + bias; d2 bf16 = gelu_erf(u) (fc1)    */
  VITK_EPI_BIAS_RESID_F32 = 3,  /* d f32 = acc + bias[n] + aux_f32[m,n]          (out, fc2)*/
  VITK_EPI_PATCH_F32 = 4,       /* d f32[(m/rows_in)*rows_out + row_off + m%rows_in, n] =
                                   acc + bias[n] + aux_f32[row_off + m%rows_in, n] (patch+pos) */
  VITK_EPI_DGELU_BF16 = 5,      /* d bf16 = acc * gelu'(aux_bf16[m,n])           (fc2 dgrad)*/
  VITK_EPI_ACCUM_F32 = 6,       /* d f32 += acc (red.global.add; split-K allowed) (wgrad)  */
  VITK_EPI_STORE_F32 = 7,       /* d f32 = acc                                             */
  VITK_EPI_BIAS_GELUG_BF16 = 8, /* u = acc + bias; d bf16 = gelu_erf(u); d2 bf16 (optional) = gelu_erf'(u)  (fc1, training) */
  VITK_EPI_MUL_BF16 = 9,        /* d bf16 = acc * aux_bf16[m,n]                  (fc2 dgrad with saved gelu') */
  VITK_EPI_UNPATCH_F32 = 10     /* inverse of PATCH_F32 (input gradient, col2im of dh·Wp): row m is token
                                   t = m % rows_out of image g = m / rows_out; rows with t < row_off are dropped, patch
                                   q = t − row_off sits at (q / G, q % G) with G² = rows_out − row_off; column
                                   n = c·256 + ky·16 + kx goes to d f32 [g, c, 16·(q/G) + ky, 16·(q%G) + kx] of the NCHW
                                   image [M/rows_out, 3, 16G, 16G].  N = 768, ldd = 16G (the image width),
                                   M % rows_out == 0; no bias, no aux; every element of d written exactly once.
                                   rows_in = 0: a square grid, as above.  rows_in > 0: a rectangular grid of rows_in
                                   patches per image row (G = rows_in, (rows_out − row_off) / rows_in patch rows), so d is
                                   [M/rows_out, 3, 16·(rows_out − row_off)/rows_in, 16·rows_in] and ldd = 16·rows_in */
};

typedef struct vitk_gemm_args {
  const void* a;
  const void* b;
  int64_t M, N, K;
  int64_t lda, ldb;
  int32_t a_mn_major, b_mn_major;
  int32_t epilogue;      /* enum vitk_epilogue */
  int32_t split_k;       /* >=1; >1 only with VITK_EPI_ACCUM_F32; 0 = library chooses */
  void* d;
  int64_t ldd;
  void* d2;              /* second output (same ldd), VITK_EPI_BIAS_GELU_BF16 only */
  const float* bias;     /* [N] or NULL */
  const void* aux;       /* residual f32 / pos f32 / pre-activation bf16, row stride ld_aux */
  int64_t ld_aux;
  int64_t rows_in, rows_out, row_off; /* VITK_EPI_PATCH_F32 row remap; VITK_EPI_UNPATCH_F32 grid (rows_in: patches per
                                         image row, 0 = square) */
  int32_t tile_n;        /* 0 = library chooses; else 128, 192 or 256 */
  int32_t max_ctas;      /* 0 = all SMs; else cap on the persistent grid, leaving SMs to a concurrent collective */
  int32_t variant;       /* 0 = library chooses; 1 = single-CTA 128×N tiles (gemm.cu); 2 = CTA pair,
                            256×N tiles, TMA-store epilogue (gemm2.cu; not for VITK_EPI_PATCH_F32 / UNPATCH_F32); 3 = as 2 but
                            always with 8 epilogue warps (the A/B reference of the 16-warp heavy-epilogue
                            instantiations, which produce the same bits) */
} vitk_gemm_args;

VITK_API int vitk_gemm_bf16(const vitk_gemm_args* args, vitk_stream_t stream);

/* Column sums (bias gradients, aten::sum over rows): out f32 [N] += Σ_m x_bf16[m,n]. */
VITK_API int vitk_colsum_bf16(const void* x_bf16, int64_t M, int64_t N, int64_t ldx, float* out, vitk_stream_t stream);

/* ------------------------------------------------------------------ attention
 * Replaces aten::scaled_dot_product_attention fwd/bwd (HF:232-246, sdpa_attention.py:92-102):
 * softmax(Q·Kᵀ·scale)·V per (batch, head), no mask, no dropout, head_dim 64.
 * qkv bf16 [B,T,3,H,64] (the fused QKV projection output, row stride 3*H*64);
 * o bf16 [B,T,H*64]; lse fp32 [B,H,T] (natural-log sum-exp of the scaled scores). */
VITK_API int vitk_attn_fwd(const void* qkv_bf16, int64_t B, int64_t T, int64_t H, float scale, void* o_bf16, float* lse,
                  vitk_stream_t stream);
/* p[b,h,i,j] = exp(scale·q_i·k_j − lse[b,h,i]) as fp32 [B,H,T,T] (contiguous), from the qkv buffer and the lse that
 * vitk_attn_fwd wrote — HF eager_attention_forward's attn_weights (modeling_vit.py:185-190).  Writes exactly B·H·T²
 * floats and nothing else.  qkv 16-byte aligned; lse and probs 4-byte aligned. */
VITK_API int vitk_attn_probs(const void* qkv_bf16, const float* lse, int64_t B, int64_t T, int64_t H, float scale,
                             float* probs, vitk_stream_t stream);
/* dqkv bf16 [B,T,3,H,64].  workspace: vitk_attn_bwd_workspace_bytes(B,T,H) bytes. */
VITK_API size_t vitk_attn_bwd_workspace_bytes(int64_t B, int64_t T, int64_t H);
VITK_API int vitk_attn_bwd(const void* qkv_bf16, const void* o_bf16, const void* do_bf16, const float* lse, int64_t B,
                  int64_t T, int64_t H, float scale, void* dqkv_bf16, void* workspace, vitk_stream_t stream);

/* ------------------------------------------------------------------ embeddings glue
 * CLS rows of the embedding output (HF:117-124): h[b,0,:] = cls + pos[0]. */
VITK_API int vitk_embed_cls(const float* cls, const float* pos, int64_t B, int64_t T, int64_t D, float* h, vitk_stream_t stream);
/* Backward of cat(cls,patches)+pos: dpos[t] += Σ_b dh[b,t]; dcls += Σ_b dh[b,0];
 * dbias += Σ_{b,t>=1} dh[b,t]; dpatch bf16 [B*(T-1), D] = dh[b,1+p] (compact, for the wgrad GEMM). */
VITK_API int vitk_embed_bwd(const void* dh_bf16, int64_t B, int64_t T, int64_t D, float* dpos, float* dcls, float* dbias,
                   void* dpatch_bf16, vitk_stream_t stream);

/* Position embeddings at another patch grid (HF ViTEmbeddings.interpolate_pos_encoding, modeling_vit.py:60-99): replaces
 * the cat(pos[:, :1], F.interpolate(pos[:, 1:].reshape(1, s, s, D).permute(0, 3, 1, 2), size=(gh, gw), mode="bicubic",
 * align_corners=False).permute(0, 2, 3, 1).view(1, -1, D)) of HF:79-99 and its autograd backward.
 * vitk_pos_interp: pos fp32 [1 + gh0·gw0, D] → out fp32 [1 + gh·gw, D]; out[0] = pos[0], rows 1.. the gh0×gw0 grid
 *   resized to gh×gw: out = Wy · pos · Wxᵀ per channel, with Wy [gh, gh0] and Wx [gw, gw0] torch's bicubic matrices
 *   (cubic convolution, A = −0.75, source coordinate (o + 0.5)·in/out − 0.5, taps clamped to the grid).
 * vitk_pos_interp_bwd: the exact adjoint, ACCUMULATED: dpos[0] += dout[0], dpos[1..] += Wyᵀ · dout[1..] · Wx per channel;
 *   every dpos element is summed by one thread in a fixed order (no atomics: two runs give the same bits).
 * Both: grids 1..4096 per side, D a multiple of 4 up to 4096, buffers 16-byte aligned and not overlapping. */
VITK_API int vitk_pos_interp(const float* pos, int64_t gh0, int64_t gw0, int64_t gh, int64_t gw, int64_t D, float* out,
                             vitk_stream_t stream);
VITK_API int vitk_pos_interp_bwd(const float* dout, int64_t gh, int64_t gw, int64_t gh0, int64_t gw0, int64_t D, float* dpos,
                                 vitk_stream_t stream);

/* ------------------------------------------------------------------ head + loss
 * Replaces final LayerNorm on the CLS rows, classifier Linear(D→C) and BCEWithLogitsLoss (mean)
 * with their gradients (HF:455,641-646; loss_utils.py:110-112; Trainer call site trainer.py:1978).
 * vitk_head_fwd:  h f32 [B,T,D] (only rows t=0 are read) → logits f32 [B,C]; when labels f32
 *   [B,C] != NULL also loss f32 [1] (mean over B·C) and, when dlogits != NULL, the fused loss
 *   gradient dlogits f32 [B,C] = (σ(logit) − y)/(B·C).  mean/rstd f32 [B] (optional) are the
 *   LayerNorm statistics the backward reuses.  Both head entry points take C <= 64 and D <= 8192. */
VITK_API int vitk_head_fwd(const float* h, int64_t B, int64_t T, int64_t D, int64_t C, const float* gamma,
                  const float* beta, float eps, const float* Wc, const float* bc, const float* labels, float* logits,
                  float* loss, float* dlogits, float* mean, float* rstd, vitk_stream_t stream);
/* vitk_head_bwd: chains dlogits·(*dloss) (dloss = device pointer to the upstream scalar gradient,
 *   NULL = 1) through the classifier and the LayerNorm of the CLS rows.  dh bf16 [B,T,D]: rows
 *   t=0 are written, all other rows are NOT touched (their gradient is zero — clear them once).
 *   dWc [C,D], dbc [C], dgamma [D], dbeta [D] are ACCUMULATED (+=). */
VITK_API int vitk_head_bwd(const float* h, const float* mean, const float* rstd, const float* gamma, const float* beta,
                  const float* Wc, int64_t B, int64_t T, int64_t D, int64_t C, const float* dlogits,
                  const float* dloss, void* dh_bf16, float* dWc, float* dbc, float* dgamma, float* dbeta,
                  vitk_stream_t stream);

/* CLS-row attention for the top encoder layer of a classifier: HF reads only sequence_output[:, 0]
 * (modeling_vit.py:641), so of the last layer's attention only query 0 is consumed and only its row carries a gradient.
 * Same buffers as vitk_attn_fwd / vitk_attn_bwd; o / lse / do are touched at token 0 only; dqkv gets dense dK and dV
 * (rank one per key), dQ at token 0 and zeros elsewhere.  T <= 4096. */
VITK_API int vitk_attn_cls_fwd(const void* qkv_bf16, int64_t B, int64_t T, int64_t H, float scale, void* o_bf16, float* lse,
                  vitk_stream_t stream);
VITK_API int vitk_attn_cls_bwd(const void* qkv_bf16, const void* o_bf16, const void* do_bf16, const float* lse, int64_t B,
                  int64_t T, int64_t H, float scale, void* dqkv_bf16, vitk_stream_t stream);

/* ------------------------------------------------------------------ evaluation counters
 * Replaces compute_metrics / the final report of /root/reference/ViT-Training.py:112-118,139-146
 * (sigmoid → >= threshold → sklearn f1_score(average="micro") / classification_report): accumulates, per class c,
 * counts[c][0..3] += {TP, FP, FN, TN} over B×C fp32 logits and {0,1} fp32 labels.  counts: int64 [C,4], caller-zeroed
 * before the first batch of an evaluation loop; sigmoid = 1/(1+exp(−x)) in fp32 as in ATen.  C <= 4096. */
VITK_API int vitk_multilabel_counts(const float* logits, const float* labels, int64_t B, int64_t C, float threshold,
               int64_t* counts, vitk_stream_t stream);

/* ------------------------------------------------------------------ optimizer (flat buffers)
 * torch.optim.AdamW semantics as HF Trainer configures it (trainer.py:1143-1217,1760):
 *   g' = g·(*grad_scale)   (grad_scale: device pointer, NULL = 1; see vitk_clip_scale)
 *   p ← p·(1 − lr·wd);  m ← m + (1−β1)(g' − m);  v ← v + (1−β2)(g'² − v);
 *   p ← p − lr/bias_corr1 · m / (√v/√bias_corr2 + eps);   p_bf16 ← bf16(p) when p_bf16 != NULL;
 *   g ← 0 when zero_grad != 0 (optimizer.zero_grad() folded into the same pass).
 * bias_corr_dev != NULL: device pointer to {1 − β1^t, 1/√(1 − β2^t)} written by vitk_adamw_tick; the two scalar
 * corrections are then ignored (a captured CUDA graph replays with fixed kernel arguments, so the step count must
 * live on the device).  n multiple of 4; all buffers 16-byte aligned. */
VITK_API int vitk_adamw(float* p, float* g, float* m, float* v, void* p_bf16, int64_t n, float lr, float beta1,
               float beta2, float eps, float weight_decay, float bias_corr1, float bias_corr2,
               const float* grad_scale, int zero_grad, const float* bias_corr_dev, vitk_stream_t stream);
/* Optimizer step counter on the device (the `step` entry of torch.optim.AdamW's state, torch/optim/adamw.py):
 * *step_dev += increment (0 or 1); bias_corr_dev[0] = 1 − β1^t, bias_corr_dev[1] = 1/√(1 − β2^t). */
VITK_API int vitk_adamw_tick(int64_t* step_dev, int increment, float beta1, float beta2, float* bias_corr_dev,
               vitk_stream_t stream);
/* out[0] += Σ x²  (global gradient norm, trainer.py:2489-2493), summed in a fixed order: replicas holding identical
 * gradients get bit-identical norms (torch.nn.utils.clip_grad_norm_ is deterministic too).  scratch: device buffer of
 * vitk_sumsq_scratch_floats() floats, zero-initialised once by the caller (the kernel leaves its ticket word at zero);
 * calls sharing a scratch buffer must be stream-ordered. */
VITK_API int64_t vitk_sumsq_scratch_floats(void);
VITK_API int vitk_sumsq_f32(const float* x, int64_t n, float* out, float* scratch, vitk_stream_t stream);
/* Data-parallel gradient mean, owner's step (replaces the XLA-implicit cross-replica gradient reduction of
 * /root/reference/ViT-Training.py:106,170; used by parallel.PeerGradSync after the copy engines pulled this rank's shard
 * of a bucket from every peer over NVLink): own[i] = (own[i] + Σ_{p<n_peers} peers[p·peer_stride + i]) · inv_world,
 * fixed summation order.  n, peer_stride multiples of 4; max_ctas caps the grid (0 = 2 per SM). */
VITK_API int vitk_shard_mean(float* own, const float* peers, int64_t n, int64_t peer_stride, int n_peers, float inv_world,
               int max_ctas, vitk_stream_t stream);
/* scale[0] = min(1, max_norm / (sqrt(sumsq[0]) + 1e-6))  (torch.nn.utils.clip_grad_norm_). */
VITK_API int vitk_clip_scale(const float* sumsq, float max_norm, float* scale, vitk_stream_t stream);

/* ------------------------------------------------------------------ parameter shadow / misc
 * bf16 shadow refresh after optimizer.step(): dst_bf16[i] = bf16(src[i]). n multiple of 8. */
VITK_API int vitk_cast_f32_bf16(const float* src, void* dst_bf16, int64_t n, vitk_stream_t stream);
VITK_API int vitk_fill_zero(void* ptr, size_t bytes, vitk_stream_t stream);
/* Host-only: the launch vitk_gemm_bf16 makes for these arguments on a GPU with `sms` SMs, decided by the same code
 * and rejected with the same error where vitk_gemm_bf16 would reject them (operand pointers are checked for NULL and
 * alignment, never dereferenced).  kernel: 1 = single-CTA, 2 = CTA pair, 3 = CTA pair with 16 epilogue warps; tile
 * width (128 / 192 / 256 columns), split-K factor, half-width tiles per 256-row band (mixed 256+128 schedule of the
 * pair kernel; 0 for the single-CTA kernel), work items dealt round-robin over the grid, and the grid in CTAs.
 * Needs no device; used by the CPU tests of the schedule. */
VITK_API int vitk_gemm_plan(const vitk_gemm_args* args, int sms, int* tile_n, int* split_k, int* n_half, int* work_items,
                            int* kernel, int* ctas);
/* Diagnostics: when device_buf is non-NULL, CTA (0,0,0) of vitk_attn_bwd records clock64() stamps of its pipeline
 * phases into it (>= 1024 int64; slot = 16·query_block + phase) and the CTA-pair GEMM records per-K-block / per-tile /
 * per-CTA stamps (>= 8192 int64; layout in csrc/gemm2.cu); NULL (default) disables. */
VITK_API int vitk_debug_timeline(void* device_buf);
/* Diagnostics: a one-thread kernel that writes %globaltimer (ns) to slot `slot` of the vitk_debug_timeline buffer, in
 * stream order — brackets another launch with device-side time stamps. */
VITK_API int vitk_debug_stamp(int64_t slot, vitk_stream_t stream);
/* Number of kernels this library has launched in this process (all threads); bench.py reads it
 * around the timed region to report gpu_launches. */
VITK_API int64_t vitk_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* VITK_H_ */
