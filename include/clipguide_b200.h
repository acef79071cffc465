/*
 * clipguide_b200 -- C ABI of the B200-native CLIP-guidance hot path.
 *
 * The reference (Penguin-jpg/clip-diffusion) has no FFI/plugin registry: its "operator API"
 * for this path is a handful of Python functions plus torch autograd (SURVEY.md section 8(b)).
 * Each entry point below is the device-side replacement of one of those functions; the
 * reference file:line it replaces is cited per function.  The Python mirror of the reference
 * interface lives in clip_diffusion_b200/ and binds this library with ctypes (INTEGRATION.md).
 *
 * Conventions
 *   - plain C: device pointers + sizes, no torch types.  Pointers are DEVICE pointers unless the
 *     name ends in _h (host).  `stream` is a cudaStream_t passed as void* (NULL = default stream).
 *   - every function returns 0 on success, a negative CG_E* code on bad arguments, or a positive
 *     cudaError_t; cg_last_error() gives a human readable message for the calling thread.
 *   - nothing allocates: callers own all buffers (workspace sizes are queried first).
 *   - all kernels are compiled for sm_100a only; there is no CPU fallback.
 */
#ifndef CLIPGUIDE_B200_H
#define CLIPGUIDE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CG_EINVAL (-1)
#define CG_ENOSPC (-2)
#define CG_EARCH (-3)

const char* cg_last_error(void);
/* ABI version of this header; bumps when a signature changes. */
int cg_abi_version(void);
/* 0 if the current device is sm_100; CG_EARCH otherwise. */
int cg_check_device(void);

/* ------------------------------------------------------------------ losses ---------------- */

/* total_variational_loss, clip_diffusion/losses.py:20-28 -- value and analytic gradient in one pass.
 *   x [B,C,H,W] fp32.  loss[b] = mean_{c,h,w}(dx^2 + dy^2) (replicate pad => last col/row differences 0).
 *   grad (may be NULL) [B,C,H,W]: grad = (accumulate ? grad : 0) + grad_scale * d loss[b] / d x.
 *   loss (may be NULL) [B] is overwritten. */
int cg_tv_loss_fwd_bwd(const float* x, int B, int C, int H, int W, float grad_scale, int accumulate,
                       float* loss, float* grad, void* stream);

/* rgb_range_loss, clip_diffusion/losses.py:31-35.  Same calling convention as cg_tv_loss_fwd_bwd. */
int cg_range_loss_fwd_bwd(const float* x, int B, int C, int H, int W, float grad_scale, int accumulate,
                          float* loss, float* grad, void* stream);
/* structural_dissimilarity_loss, clip_diffusion/losses.py:48-54 (init-image branch of conditon_function, sample.py:220-225): 1 - MS-SSIM of
 * x and y, both [C,H,W] fp32 in [-1,1] (mapped to [0,1] inside, image_utils.py:40-42), with pytorch_msssim.MS_SSIM(win_size=11,
 * win_sigma=1.5, data_range=1, size_average=True) semantics (5 scales; the package itself is not vendored by the reference: restated from
 * its published algorithm, oracle/ms_ssim.py).  loss (optional) = the value; grad (optional) (+)= grad_scale * d loss / d x.  H, W
 * multiples of 16, smaller side > 160.  workspace: cg_ms_ssim_workspace_bytes. */
size_t cg_ms_ssim_workspace_bytes(int C, int H, int W);
int cg_ms_ssim_dissimilarity_fwd_bwd(const float* x, const float* y, int C, int H, int W, float grad_scale, int accumulate, float* loss,
                                     float* grad, void* workspace, void* stream);
/* The image-space tail of conditon_function in ONE pass (clip_diffusion/sample.py:217-228): grad (+)= d(tv_scale * TV(x) + range_scale *
 * range(x))/dx, nan_flag[0] = 1 if the finished grad holds a NaN (what `torch.isnan(grad_tensor).any()` tests; nan_flag has 2 floats),
 * loss2 (optional) = [B][2] values (TV, range).  Needs W % 128 == 0; values are deterministic (no float atomics). */
int cg_image_losses_fwd_bwd(const float* x, int B, int C, int H, int W, float tv_scale, float range_scale, int accumulate,
                            float* loss2, float* grad, float* nan_flag, void* stream);

/* square_spherical_distance_loss, clip_diffusion/losses.py:10-16 (with L2_norm, utils/functional.py:74-76).
 *   emb [N,E], txt [P,E] fp32 (un-normalised).  dist [N,P] = 2*asin(||emb^ - txt^||/2)^2. */
int cg_spherical_dist_fwd(const float* emb, const float* txt, int N, int P, int E, float* dist, void* stream);
/* gradient of sum_{n,p} gdist[n,p]*dist[n,p] with respect to emb -> demb [N,E]. */
int cg_spherical_dist_bwd(const float* emb, const float* txt, const float* gdist, int N, int P, int E,
                          float* demb, void* stream);
/* Fused form used by the fast cond_fn (sample.py:179-198): loss_out[0] (+)= coef * sum_n sum_p w[p]*dist[n,p],
 * demb [N,E] = d(that)/d emb, one pass.  w may be NULL (all ones).  loss_out may be NULL. */
int cg_spherical_loss_fwd_bwd(const float* emb, const float* txt, const float* w, int N, int P, int E, float coef,
                              float* loss_out, float* demb, void* stream);

/* ------------------------------------------------------------------ cutouts --------------- */

/* flag bits of cg_cut_t.flags */
#define CG_CUT_GRAY_PRE 1  /* grayscale the source crop before resampling (inner cuts, cutouts.py:102-103) */
#define CG_CUT_GRAY_POST 2 /* grayscale after resampling (overview variants, cutouts.py:72,76)           */
#define CG_CUT_HFLIP 4     /* horizontal flip after resampling (overview variants, cutouts.py:74,76)     */
#define CG_CUT_OVERVIEW 8  /* informational: source is the zero-padded square (cutouts.py:54-64)         */

/* One cutout: the square crop [y0,y0+size) x [x0,x0+size) of the image (coordinates may lie outside
 * the image: those pixels are zero, cutouts.py:54-62), resampled to cut_size^2 with ResizeRight's
 * antialiased cubic (cutouts.py:64,105). */
typedef struct {
  int32_t y0, x0, size, flags;
} cg_cut_t;

/* The per-call augmentation parameters of cutouts.py:31-45 (one set for the whole batch) plus the
 * epilogue (CLIP_NORMALIZE, utils/functional.py:16-18,100). */
typedef struct {
  int32_t flip;        /* RandomHorizontalFlip coin */
  int32_t gray;        /* RandomGrayscale coin */
  int32_t perm[4];     /* ColorJitter op order: 0 brightness, 1 contrast, 2 saturation, 3 hue */
  float theta[6];      /* torchvision inverse affine matrix (output -> input), row major 2x3 */
  float theta_fwd[6];  /* its inverse (input -> output), used by the backward gather */
  float brightness, contrast, saturation, hue;
  int32_t augment;     /* 0: skip the whole augmentation chain (base cutouts only) */
  int32_t normalize;   /* 1: apply (x-mean)/std at the end */
  float mean[3], stdv[3];
  uint64_t noise_seed; /* Philox key when `noise` is NULL */
  uint64_t cut_index0; /* global index of cutout 0 of this call (shards of one record draw the same noise) */
  float noise_std;     /* 0.01 in the reference (cutouts.py:34,40,42) */
  int32_t input01;     /* 1: x_in is already in [0,1] (Cutouts.forward, cutouts.py:47); 0: [-1,1] and the
                          kernel applies denormalize_image_zero_to_one (image_utils.py:40-42) on load */
  /* In-kernel noise that reproduces the reference ON CUDA bit for bit: the three `torch.randn_like(input)` calls of cutouts.py:34,40,42
   * draw from torch's CUDA generator (Philox4x32-10, curand_normal4, the thread/element mapping of ATen's distribution_nullary_kernel).
   * noise_mode 1: noise_seed = the generator's seed, noise_offset[s] = its Philox offset at the s-th call, noise_total = cutouts of
   * the WHOLE batch (shards generate their slice of the same stream; cut_index0 is the slice start), noise_threads = grid * 256 of
   * torch's launch for that tensor (cg_randn_like_torch_geometry).  noise_mode 0: the library's own counter-based keying. */
  int32_t noise_mode;
  uint32_t noise_threads;
  uint64_t noise_offset[3];
  uint64_t noise_total;
} cg_aug_t;

/* output formats of cg_cutouts_fwd / input format of cg_cutouts_bwd */
#define CG_FMT_F32_NCHW 0   /* [N,3,cs,cs] fp32 -- what make_cutouts returns */
#define CG_FMT_BF16_PATCH 1 /* [N, g*g, kpad] bf16, k = c*p*p + py*p + px: the im2col rows of CLIP's conv1 */
#define CG_FMT_F32_PATCH 2  /* same layout in fp32: the conv1 dgrad GEMM's output, accepted by cg_cutouts_bwd as `dout` */

size_t cg_cutouts_workspace_bytes(int N, int cs, int max_size);

/* torch.randn / torch.randn_like for a float32 CUDA tensor of `numel` elements, reproduced from the generator state (seed, Philox offset
 * at the call): out[i] equals what torch writes, bit for bit (cutouts.py:34,40,42 on a CUDA device).  cg_randn_like_torch_geometry
 * returns the thread count of torch's launch (grid * 256, host only: device properties) and, through *offset_increment, by how much
 * the call advances the generator's offset. */
uint32_t cg_randn_like_torch_geometry(int64_t numel, uint64_t* offset_increment);
int cg_randn_like_torch(float* out, int64_t numel, uint64_t seed, uint64_t offset, void* stream);

/* make_cutouts, clip_diffusion/cutouts.py:117-134 (+ CLIP_NORMALIZE) as fused kernels.
 *   x_in [3,H,W] fp32 in [-1,1]; cuts_h/aug_h are HOST structs (copied asynchronously);
 *   noise: NULL (generated in-kernel, Philox) or 3 stacked tensors [3][N,3,cs,cs] fp32 of N(0,1) draws;
 *   out: format `fmt`; for CG_FMT_BF16_PATCH, `patch` divides cs and kpad >= 3*patch*patch (pad is zeroed).
 *   workspace (cg_cutouts_workspace_bytes) keeps what the backward needs until cg_cutouts_bwd. */
int cg_cutouts_fwd(const float* x_in, int H, int W, const cg_cut_t* cuts_h, int N, int cs, const cg_aug_t* aug_h,
                   const float* noise, void* out, int fmt, int patch, int kpad, void* workspace, void* stream);

/* Backward of the above: dout (same format as out) -> dx_in [3,H,W] fp32:
 *   dx_in = (accumulate ? dx_in : 0) + coef * d<dout,out>/d x_in.   Deterministic (gather form, no atomics).
 *   input01 must equal the forward's aug_h->input01. */
int cg_cutouts_bwd(const void* dout, int H, int W, int N, int cs, int fmt, int patch, int kpad, float coef,
                   int accumulate, int input01, float* dx_in, void* workspace, void* stream);

/* ------------------------------------------------------------------ CLIP ViT -------------- */
/* The OpenAI CLIP VisionTransformer reached through embed_image (utils/functional.py:97-102,
 * models.py:76-80): building blocks.  Activations are bf16 row-major [M, D]; the residual stream
 * and its gradient are fp32. */

/* LayerNorm forward (eps 1e-5) over M rows of D fp32 values, row r at x + r*row_stride:
 *   y = LN(x) * gamma + beta, written as bf16 (y_bf16, contiguous [M,D], GEMM operand) and/or fp32
 *   (y_f32, contiguous [M,D]; ln_pre / ln_post feed fp32 consumers).  Saves mean/rstd [M]. */
int cg_layernorm_fwd(const float* x, const float* gamma, const float* beta, int M, int D, int64_t row_stride,
                     void* y_bf16, float* y_f32, float* mean, float* rstd, void* stream);
/* LayerNorm backward (frozen gamma/beta => input gradient only).  dy contiguous [M,D] fp32; x, dx and
 * dx_bf16 (optional bf16 copy of the updated dx) use row_stride:  dx = (accumulate ? dx : 0) + LN'(dy). */
int cg_layernorm_bwd(const float* dy, const float* x, const float* gamma, const float* mean, const float* rstd,
                     int M, int D, int64_t row_stride, int accumulate, float* dx, void* dx_bf16, void* stream);

/* GEMM epilogues (all: acc[M,N] = A[M,K] . B[N,K]^T, bf16 operands K-major, fp32 accumulation in TMEM) */
#define CG_EPI_BIAS_BF16 0        /* out_bf16 = acc + bias                                     (QKV)          */
#define CG_EPI_BIAS_RESID_F32 1   /* out_f32 = aux_f32 + acc + bias  (aux may alias out)      (out-proj, c_proj) */
#define CG_EPI_BIAS_QGELU_BF16 2  /* aux_bf16 = u = acc + bias ; out_bf16 = u*sigmoid(1.702u)  (c_fc)         */
#define CG_EPI_DQGELU_BF16 3      /* out_bf16 = acc * QuickGELU'(aux_bf16)                     (c_proj dgrad) */
#define CG_EPI_F32 4              /* out_f32 = acc                                             (dgrad into LN) */
#define CG_EPI_BF16 5             /* out_bf16 = acc                                            (out-proj dgrad) */
#define CG_EPI_PATCH_POS_F32 6    /* out_f32[(m/g2)*(g2+1)+1+m%g2, :] = acc + pos[1+m%g2, :]   (conv1 patch embed) */

/* tcgen05/TMEM/TMA GEMM.  A [M,K] bf16 row-major (lda elements), B [N,K] bf16 row-major (ldb); K % 64 == 0,
 * N % 128 == 0.  out/aux/bias/pos as the epilogue needs (others NULL); ldo = leading dimension of out/aux
 * in elements; g2 = patches per image for CG_EPI_PATCH_POS_F32. */
int cg_gemm_bf16_tn(const void* A, const void* B, int M, int N, int K, int64_t lda, int64_t ldb, int epilogue,
                    const float* bias, void* out, void* aux, int64_t ldo, const float* pos, int g2, void* stream);

/* Tile variant cg_gemm_bf16_tn runs a problem on (host only, no launch): the per-problem choice, including the
 * CG_GEMM_PAIR / CG_GEMM_BN overrides read from the environment at the first call.  Negative on bad sizes. */
#define CG_GEMM_TILE_128x256 0
#define CG_GEMM_TILE_128x128 1
#define CG_GEMM_TILE_PAIR_256x256 2 /* two CTAs of a cluster share one 256 x 256 tile */
int cg_gemm_tile_variant(int M, int N, int K, int epilogue);

/* ------------------------------------------------------------------ CLIP ModifiedResNet ---- */
/* The OpenAI CLIP ModifiedResNet image tower (clip/model.py ModifiedResNet: the RN101 of chosen_clip_models, config.py:41, reached
 * through embed_image like the ViTs) on NHWC bf16 activations, rows [N*H*W, C].  BatchNorm (eval) is folded into the convolution
 * weights and biases at load, so each convolution is a GEMM plus bias: a 1x1 convolution reads the activation rows as its A operand,
 * a 3x3 convolution reads the rows cg_im2col3x3_nhwc builds.  The input gradient of a stride-1 3x3 convolution is the same convolution
 * of the output gradient with the flipped, transposed weights W'[cin, (ky*3 + kx)*Cout + cout] = W[cout, cin, 2 - ky, 2 - kx]. */

/* The GEMM epilogues of a ReLU network (cg_gemm_bf16_tn_relu; the mask tests follow torch's threshold_backward: 0 where the saved
 * output is <= 0): */
#define CG_EPI_BIAS_RELU_BF16 7        /* out_bf16 = relu(acc + bias)                           (stem convs, Bottleneck conv1/conv2) */
#define CG_EPI_BIAS_RESID_RELU_BF16 8  /* out_bf16 = relu(acc + bias + resid_bf16)              (Bottleneck conv3 + identity)  */
#define CG_EPI_DRELU_BF16 9            /* out_bf16 = acc * [mask_bf16 > 0]                      (dgrads into a ReLU output)     */
#define CG_EPI_RESID_DRELU 10          /* out_f32 = (acc + resid_f32) * [mask_bf16 > 0] (no mask: 1; resid may alias out_f32),
                                          out_bf16 = bf16(out_f32)                              (conv1 dgrad + identity gradient) */
/* cg_gemm_bf16_tn with one of the epilogues 7-10: same operands, sizes and tile variants.  resid, mask and out_bf16 are addressed with
 * ldo like out; bias (7, 8), resid (8, 10), mask (9; optional for 10) and out_bf16 (10) are given exactly when the epilogue reads or
 * writes them, NULL otherwise.  out is fp32 for RESID_DRELU and bf16 otherwise. */
int cg_gemm_bf16_tn_relu(const void* A, const void* B, int M, int N, int K, int64_t lda, int64_t ldb, int epilogue, const float* bias,
                         const void* resid, const void* mask, void* out, void* out_bf16, int64_t ldo, void* stream);

/* nn.Conv2d(C, *, 3, stride, padding=1)'s im2col rows: x [N,H,W] pixels of ldx bf16 values (the first C are the channels) ->
 * out [N*Ho*Wo, kpad] bf16, column (ky*3 + kx)*C + c, zero for taps outside the image and for columns >= 9C.  Ho = (H-1)/stride + 1;
 * stride 1 or 2; kpad a multiple of 64 and >= 9C; ldx % 8 == 0.  A pure copy. */
int cg_im2col3x3_nhwc(const void* x, int N, int H, int W, int C, int64_t ldx, int stride, int kpad, void* out, void* stream);
/* Input gradient of the stem's conv1 (3x3, stride 2, padding 1, no bias; the flip above needs stride 1): dy [N, Ho, Wo] pixels of lddy
 * bf16 values (the first Cout are the channels), w [Cout, Cin, 3, 3] fp32 -> dx [N, H, W, kpad] fp32 (columns >= Cin zero): the
 * CG_FMT_F32_PATCH layout with patch 1 that cg_cutouts_bwd and cg_patchify_bwd read.  Each pixel sums its (at most 4) output positions
 * x Cout channels in a fixed order.  Cin <= 8, Cout <= 256. */
int cg_conv3x3s2_dgrad(const void* dy, int N, int H, int W, int Cout, int64_t lddy, const float* w, int Cin, int kpad, float* dx, void* stream);
/* nn.AvgPool2d(2) on NHWC bf16 rows (Bottleneck.avgpool, downsample[-1], the stem's pool): x [N,H,W,C] -> y [N,H/2,W/2,C], fp32 sums.
 * H, W even, C % 8 == 0. */
int cg_avgpool2x2_nhwc_fwd(const void* x, int N, int H, int W, int C, void* y, void* stream);
/* Its gradient: dx [N,H,W,C] = 0.25 dy[n, y/2, x/2, c], times [mask > 0] when the bf16 mask [N,H,W,C] (a saved ReLU output) is given.
 * dy fp32 (dy_f32) or bf16, dx fp32 (dx_f32) or bf16. */
int cg_avgpool2x2_nhwc_bwd(const void* dy, int dy_f32, const void* mask, int N, int H, int W, int C, void* dx, int dx_f32, void* stream);
/* AttentionPool2d's tokens: x [N*S, C] bf16 (the last stage's output, S = H*W), pos [S+1, C] fp32 ->
 * tok [N*(S+1), C] bf16, tok[n,0] = mean_s x[n,s] + pos[0], tok[n,1+s] = x[n,s] + pos[1+s] (the A operand of the packed q|k|v
 * projection; attention is cg_attention_fwd / _bwd with T = S+1).  C % 8 == 0. */
int cg_resnet_attnpool_fwd(const void* x, const float* pos, int N, int S, int C, void* tok, void* stream);
/* Its gradient through the last stage's ReLU: dtok [N*(S+1), C] fp32 -> g[n,s] = (dtok[n,1+s] + dtok[n,0]/S) * [x[n,s] > 0], fp32 g and
 * its bf16 copy g_bf16, both [N*S, C]. */
int cg_resnet_attnpool_bwd(const float* dtok, const void* x, int N, int S, int C, float* g, void* g_bf16, void* stream);
/* The pool's output is attention row 0 only: dctx [N*T, C] bf16 = dy[n] (fp32 [N, C]) in row n*T, zero in every other row. */
int cg_resnet_attnpool_dctx(const float* dy, int N, int T, int C, void* dctx, void* stream);

/* Fused multi-head attention over packed qkv [Nimg*T, 3*D] bf16 (q | k | v, head h at column h*64), head_dim 64,
 * softmax scale 1/8.  ctx [Nimg*T, D] bf16, lse [Nimg, heads, T] fp32. */
int cg_attention_fwd(const void* qkv, int Nimg, int T, int heads, void* ctx, float* lse, void* stream);
/* dgrad: dctx [Nimg*T, D] bf16 -> dqkv [Nimg*T, 3*D] bf16 (recomputes P from q,k,lse).  delta_ws [Nimg, heads, T] fp32 is scratch for
 * rowsum(dO * O): written by the T > 272 (mma.sync) path only; the tcgen05 path (T <= 272) keeps those sums on chip. */
int cg_attention_bwd(const void* qkv, const void* ctx, const void* dctx, const float* lse, int Nimg, int T, int heads,
                     void* dqkv, float* delta_ws, void* stream);

/* Small helpers of the tower. */
/* x[n*T + 0, :] = cls + pos[0]  (class token rows of the residual stream). */
int cg_vit_set_cls_rows(const float* cls, const float* pos, int Nimg, int T, int D, float* x, void* stream);
/* emb[N,E] = y[N,D] @ proj[D,E] (fp32)  and its dgrad dy[N,D] = demb[N,E] @ proj^T. */
int cg_vit_proj_fwd(const float* y, const float* proj, int N, int D, int E, float* emb, void* stream);
int cg_vit_proj_bwd(const float* demb, const float* proj, int N, int D, int E, float* dy, void* stream);
/* fp32 -> bf16 copy of token rows; drop_cls=1 skips the class-token row of every image:
 * out[n*(T-1)+j, :] = x[n*T+1+j, :]  (A operand of the conv1 dgrad GEMM). */
int cg_vit_tokens_to_bf16(const float* x, int Nimg, int T, int D, int drop_cls, void* out_bf16, void* stream);
/* embed_image's front end for an arbitrary image batch (utils/functional.py:97-101): optional CLIP_NORMALIZE,
 * then conv1's im2col rows:  img [N,3,cs,cs] fp32 -> out [N, (cs/patch)^2, kpad] bf16 (pad zeroed); and its
 * backward dpatch -> dimg. */
int cg_patchify_fwd(const float* img, int N, int cs, int patch, int kpad, int normalize, void* out_bf16, void* stream);
int cg_patchify_bwd(const void* dpatch, int dpatch_is_f32, int N, int cs, int patch, int kpad, int normalize, float* dimg, void* stream);

/* The OpenAI CLIP text transformer (CLIP.encode_text, reached through embed_text, utils/functional.py:91-94; the reference encodes
 * its prompts with it once per job, preprocessing.py:11-24).  Forward only: the text side is a constant of the guidance step.
 *   x = token_embedding[tokens] + positional_embedding;  L x {x += MHA_causal(ln_1 x); x += c_proj(QuickGELU(c_fc(ln_2 x)))};
 *   out = ln_final(x)[n, argmax_t tokens[n, t]] @ text_projection
 * The blocks use cg_layernorm_fwd, cg_gemm_bf16_tn and the causal attention below; the projection is cg_vit_proj_fwd. */
/* cg_attention_fwd with a causal mask (key j > query i is -inf): same layout, scale and outputs; lse [Nseq, heads, T] is the
 * log-sum-exp over the keys j <= i.  tcgen05 kernel only: T <= 272 (CG_EINVAL beyond; OpenAI's context length is 77). */
int cg_attention_causal_fwd(const void* qkv, int Nseq, int T, int heads, void* ctx, float* lse, void* stream);
/* x[n*T + t, :] = token_embedding[tokens[n, t], :] + pos[t, :].  tokens [N, T] int32, token_embedding [V, D] fp32, pos [T, D] fp32,
 * x [N*T, D] fp32 (residual stream); D % 4 == 0.  The table is never read outside [0, V): a row whose id lies outside gets NaN. */
int cg_text_embed_fwd(const int* tokens, const float* token_embedding, const float* pos, int N, int T, int D, int V, float* x, void* stream);
/* End-of-text pooling + ln_final: e_n = the first t with tokens[n, t] maximal (torch.argmax; the end-of-text id 49407 is the largest),
 * y[n, :] = LayerNorm(x[n*T + e_n, :]) * gamma + beta (eps 1e-5).  x [N*T, D], y [N, D] fp32; D % 4 == 0. */
int cg_text_pool_fwd(const float* x, const int* tokens, int N, int T, int D, const float* gamma, const float* beta, float* y, void* stream);

/* ------------------------------------------------------------------ cond_fn tail ---------- */
/* sample.py:228-238: NaN guard + RMS-normalised clamp, on device (no host sync):
 *   if (bad) out = 0 else { m = sqrt(mean(g^2)); out = sign * g * clamp(m,-thr,thr)/m }
 * where bad = bad_flag[0] != 0 when bad_flag is given (the reference tests the PRE-VJP gradient, sample.py:228,
 * see cg_any_nan) and any(isnan(g)) otherwise.  `scratch` is 2 floats of device memory. */
int cg_grad_finalize(const float* g, int64_t n, float sign, float thr, const float* bad_flag, float* out, float* scratch,
                     void* stream);
/* any(isnan(g)) -> flag[0] (1.0f/0.0f), device side; flag must have room for 2 floats. */
int cg_any_nan(const float* g, int64_t n, float* flag, void* stream);

/* ------------------------------------------------------------------ sampler side (next row N2) ---- */
/* denoised_function, clip_diffusion/sample.py:116-132 (Imagen dynamic thresholding of the x0 prediction):
 *   thr[b] = max(quantile(|x[b,:]|, q) , min_thr)  with torch.quantile's "linear" interpolation;  out = clamp(x,-thr,thr)/thr.
 * x, out [B, n] fp32 (may alias); thr_out [B] optional.  Exact radix select instead of torch.quantile's sort. */
size_t cg_dynamic_threshold_workspace_bytes(int B);
int cg_dynamic_threshold(const float* x, int B, int64_t n, float q, float min_thr, float* out, float* thr_out, void* workspace,
                         void* stream);

/* ------------------------------------------------------------------ replicated UNet (next row N1) ---- */
/* GroupNorm32 (+ timestep scale-shift) (+ SiLU) of the guided-diffusion UNet blocks (built at clip_diffusion/models.py:87-131;
 * ResBlock / AttentionBlock of the un-vendored crowsonkb/guided-diffusion, SURVEY.md App. A.3), for NHWC fp16 activations:
 *   y[n,p,c] = act( (gamma_c * (x - mean_{n,g}) * rstd_{n,g} + beta_c) * (1 + scale[n,c]) + shift[n,c] )
 * x [N,HW,C] fp16 (channels_last), C % 8 == 0, C <= 2048, C % G == 0; gamma, beta [C] fp32; scale_shift [N,2C] fp32 (scale | shift)
 * or NULL; act = SiLU if silu != 0; y [N,HW,C] fp16 (out_f32 == 0) or fp32.  Statistics in fp32/fp64 like GroupNorm32's x.float().
 * stats [N,G,2] (mean, rstd) and coef [2,N,C] (the folded per-channel affine a_c, b_c) are outputs kept for the backward.
 * pre_bias [C] fp32 or NULL: bias of the convolution that produced x, deferred into this op -- the normalised tensor is x + pre_bias_c
 * (folded into the per-group statistics and the per-channel affine; costs no memory pass).
 * input_partial or NULL: per-chunk channel sums of x already produced by the kernel that wrote x (cg_bias_residual_add_stats_nhwc /
 * cg_concat2_stats_nhwc, same N, HW, C): the statistics pass over x is skipped.
 * workspace: cg_groupnorm_nhwc_workspace_bytes(N,HW,C) bytes, 16-byte aligned. */
size_t cg_groupnorm_nhwc_workspace_bytes(int N, int HW, int C);
/* Host-only: the launch geometry the normalisation kernels (and the *_stats producers) use for a [N,HW,C] tensor --
 * out5 = {channel octets per row, rows per CTA iteration, threads per CTA, row chunks per sample (gridDim.x), rows per chunk}.
 * Exposed so that the chunking invariants can be tested without a GPU. */
int cg_groupnorm_nhwc_geometry(int N, int HW, int C, int* out5);
int cg_groupnorm_nhwc_fwd(const void* x, int N, int HW, int C, int G, const float* gamma, const float* beta, const float* scale_shift,
                          const float* pre_bias, const void* input_partial, float eps, int silu, int out_f32, void* y, float* stats, float* coef,
                          void* workspace, void* stream);
/* input gradient of the above (weights are frozen, models.py:67-71 / :120-127): dy [N,HW,C] fp16 (dy_f32 == 0) or fp32,
 * x / stats / coef as given to / produced by the forward -> dx [N,HW,C] fp16.  dres [N,HW,C] fp16 or NULL is added to dx: the
 * gradient that reaches x through its other consumer (the block's residual / skip path), saving autograd's separate accumulation pass. */
int cg_groupnorm_nhwc_bwd(const void* dy, int dy_f32, const void* x, int N, int HW, int C, int G, const float* stats, const float* coef,
                          const float* pre_bias, int silu, const void* dres, void* dx, void* workspace, void* stream);
/* ResBlock tail `skip(x) + out_conv(h)` with the convolution biases deferred: out[r,c] = a[r,c] + b[r,c] + bias[c].
 * a, b, out [rows, C] fp16 (NHWC rows = N*H*W), bias [C] fp32, C % 8 == 0.  Its gradient is the identity on a and b. */
int cg_bias_residual_add_nhwc(const void* a, const void* b, const float* bias, int64_t rows, int C, void* out, void* stream);
/* The resblock_updown resamplers on NHWC fp16 (guided-diffusion Upsample / Downsample without conv, App. A.3):
 *   up == 0: y [N,H/2,W/2,C] = scale * (sum of each 2x2 window of x [N,H,W,C])   (avg_pool2d: scale 0.25)
 *   up != 0: y [N,2H,2W,C]   = scale * x[n, i/2, j/2, c]                         (nearest upsampling: scale 1)
 * Each is the other's gradient (d avg_pool = up with 0.25, d upsample = down with 1).  fp32 accumulation. */
int cg_resample2x_nhwc(const void* x, int N, int H, int W, int C, int up, float scale, void* y, void* stream);
/* The UNet's skip connections, `torch.cat([h, hs.pop()], dim=1)` on NHWC fp16 rows (guided-diffusion UNetModel.forward):
 *   split == 0: cat[r, 0:Ca] = a[r, :], cat[r, Ca:Ca+Cb] = b[r, :]     (a, b are read)
 *   split != 0: the inverse -- a and b are WRITTEN from cat             (the concatenation's gradient)
 * a [rows,Ca], b [rows,Cb], cat [rows,Ca+Cb] fp16; Ca, Cb multiples of 8. */
int cg_concat2_nhwc(void* a, int Ca, void* b, int Cb, int64_t rows, void* cat, int split, void* stream);
/* The same two producers, additionally writing the chunk partials (sum, sum of squares per channel and row chunk, of the fp16 values
 * they store) that a following cg_groupnorm_nhwc_fwd over [N,HW,C] accepts as input_partial.  partial: cg_groupnorm_nhwc_workspace_bytes
 * (N,HW,C) bytes.  out / cat [N,HW,C] fp16 with C = Ca + Cb for the concatenation. */
int cg_bias_residual_add_stats_nhwc(const void* a, const void* b, const float* bias, int N, int HW, int C, void* out, void* partial, void* stream);
int cg_concat2_stats_nhwc(const void* a, int Ca, const void* b, int Cb, int N, int HW, void* cat, void* partial, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CLIPGUIDE_B200_H */
