/*
 * vtp_b200.h — C ABI of the B200-native (sm_100a) VTP hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8b): the reference (MiniMax-AI/VTP) is pure Python/PyTorch and has no
 * FFI of its own, so the boundary is the set of fused stages that the reference's L1 layers dispatch to ATen for.
 * Every entry point takes raw device pointers, sizes and a CUDA stream, returns an int status (0 = ok, <0 = error,
 * message via vtp_last_error()), never throws, never allocates, never synchronises. The Python host
 * (vtp_b200/model.py, mirroring vtp/models/vtp_hf/modeling_vtp.py) binds these with ctypes.
 *
 * Each declaration cites the reference call site (relative to the reference root) that it replaces.
 */
#ifndef VTP_B200_H
#define VTP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* vtp_stream_t; /* cudaStream_t */

enum {
    VTP_OK = 0,
    VTP_ERR_ARG = -1,   /* bad argument / unsupported shape */
    VTP_ERR_CUDA = -2,  /* CUDA runtime / driver error */
    VTP_ERR_ARCH = -3,  /* device is not sm_100 */
};
enum { VTP_F32 = 0, VTP_BF16 = 1 };
enum { VTP_ACT_NONE = 0, VTP_ACT_GELU = 1, VTP_ACT_SWIGLU8 = 2, VTP_ACT_ROPE = 3, VTP_ACT_RELU = 4 };

const char* vtp_last_error(void);
int vtp_version(void);
/* 0 if the current device is compute capability 10.x, VTP_ERR_ARCH otherwise */
int vtp_check_device(void);

/* ------------------------------------------------------------------------------------------------------------
 * tcgen05 / TMA GEMM with fused epilogue:  out = epi( A · Bᵀ ),  bf16 operands, fp32 accumulation in TMEM.
 * Replaces every nn.Linear / 1x1 nn.Conv2d / 16x16-stride-16 nn.Conv2d on the path:
 *   layers/attention.py:62,64,92,94 (qkv, proj)   layers/ffn.py:73-81 (w1,w2,w3)   layers/embeddings.py:58,64
 *   encoders/vision_transformer_bottleneck.py:30,66-79   decoders/pixel_decoder.py:108,138,157,160
 *   vtp_hf/modeling_vtp.py:274,308,329   heads/dino_head.py:65-89   layers/block.py:387-412 (text tower linears)
 * and their dgrad / wgrad in the training step (operand major-ness flags select the transposes).
 * ------------------------------------------------------------------------------------------------------------ */
typedef struct {
    int M, N, K;            /* out is [M,N]; reduction length K */
    const void* A;          /* bf16. a_mn_major=0: A[M][lda] (K contiguous); =1: A[K][lda] (M contiguous) */
    int lda, a_mn_major;
    const void* B;          /* bf16. b_mn_major=0: B[N][ldb] (K contiguous, nn.Linear.weight); =1: B[K][ldb] */
    int ldb, b_mn_major;
    void* out;              /* [M][ldo] (after row remap / pixel shuffle) */
    int ldo, out_dtype;     /* VTP_F32 | VTP_BF16 */
    const float* bias;      /* [N] fp32 or NULL */
    int act;                /* VTP_ACT_* */
    int round_bf16;         /* round (acc+bias) to bf16 first (autocast nn.Linear output semantics) */
    const void* resid;      /* residual added after activation, same indexing as out; NULL = none */
    int ldr, resid_dtype;
    int accumulate;         /* 1: atomic fp32 add into out (required when split_k > 1) */
    int split_k;            /* >=1: split the reduction across CTAs; -1: chosen by the library (with accumulate=1) */
    int rr_group, rr_skip;  /* rr_skip>0: out_row = (row/rr_group)*(rr_group+rr_skip) + rr_skip + row%rr_group (cls slot);
                             * rr_skip<0: drop the first -rr_skip rows of every rr_group rows (compaction); 0 = identity */
    const void* rope_sin;   /* VTP_ACT_ROPE: bf16 [rope_tokens-rope_prefix][64] tables (layers/embeddings.py:131-180) */
    const void* rope_cos;
    int rope_tokens, rope_prefix, rope_cols; /* tokens/sequence, un-rotated prefix tokens, leading columns rotated (2*D) */
    int ps_r, ps_gh, ps_gw, ps_cout;         /* ps_r>0: PixelShuffle(ps_r) NCHW store, grid gh x gw, cout channels */
    void* out2;             /* optional bf16 copy of (acc+bias) before activation (saved for backward), [M][ldo2] */
    int ldo2;
    /* implicit 3x3 / pad-1 convolution (utils/lpips.py:127-167 VGG16 features and their dgrad): conv_C > 0 makes A an
     * NHWC bf16 activation [B][conv_H][conv_W][conv_C] loaded by 4-D TMA (OOB zero fill = padding); then M = B*H*W,
     * K = 9*conv_C with k = (3*dy+dx)*conv_C + c, B = weights [N][9*conv_C], out = NHWC [B*H*W][ldo] */
    int conv_C, conv_H, conv_W;
    const void* mask_pos;   /* optional bf16 [M][ldm]: out *= (mask_pos > 0) — ReLU backward fused in the epilogue */
    int ldm;
} vtp_gemm_args;

int vtp_gemm_bf16(const vtp_gemm_args* args, vtp_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * HBM-bound stages around the GEMMs (vtp_b200/csrc/elementwise.cu)
 * ------------------------------------------------------------------------------------------------------------ */
/* layers/embeddings.py:58,61-70 — input side of PatchEmbed's Conv2d(C,D,p,p): NCHW fp32 image -> bf16 im2col rows
 * (or fp32 for the accurate mode) [B*(H/p)*(W/p)][C*p*p], k = c*p*p + i*p + j (== conv weight.flatten(1)); the conv
 * itself is vtp_gemm_bf16. */
int vtp_patchify(const float* img, void* out, int out_dtype, int B, int C, int H, int W, int p, vtp_stream_t stream);
/* encoders/vision_transformer.py:198-217 — x[b, t, :] = vec[t, :] for t < nprefix (cls / storage tokens) */
int vtp_fill_prefix_tokens(void* x, int x_dtype, const float* vec, int B, int tokens, int nprefix, int D,
                           vtp_stream_t stream);
/* encoders/vision_transformer.py:195 — torch.where(masks, mask_token, x): idx = flat indices into [B*HW] */
int vtp_apply_mask_tokens(void* x, int x_dtype, const float* mask_token, const int64_t* idx, int n, int HW, int tokens,
                          int prefix, int D, vtp_stream_t stream);
/* layers/normalization.py:17-22 (RMSNorm, b == NULL) and nn.LayerNorm (encoders/vision_transformer.py:30-34,
 * layers/normalization.py:25-40).  x [M][ldx] fp32|bf16; y_mode: 0 fp32 [M][D], 1 bf16 [M][D], 2 bf16x3 split [M][3D]
 * (hi|hi|lo, operand of the fp32-accurate GEMM).  rstd_out/mean_out [M] optional (saved for backward). */
int vtp_norm_fwd(const void* x, int x_dtype, long ldx, void* y, int y_mode, const float* w, const float* b, float eps,
                 int M, int D, float* rstd_out, float* mean_out, vtp_stream_t stream);
/* fp32 [M][ldx] -> bf16 [M][3K]: A side (b_side=0) hi|hi|lo, B side (b_side=1) hi|lo|hi;  A'·B'^T = fp32-accurate */
int vtp_split3(const float* x, long ldx, void* out_bf16, long M, int K, int b_side, vtp_stream_t stream);
/* in [B][R][C] -> out [B][C][R] with dtype conversion and element batch strides (vtp_hf/modeling_vtp.py:395,
 * decoders/pixel_decoder.py:141) */
int vtp_transpose_batched(const void* in, int in_dtype, long in_bstride, void* out, int out_dtype, long out_bstride,
                          int B, int R, int C, vtp_stream_t stream);
/* out[i,:] = in[idx[i],:] (vtp.py:432-439,470-473 iBOT gather; encoders/text_transformer.py:224 argmax pool) */
int vtp_gather_rows(const void* in, int in_dtype, long ld_in, void* out, int out_dtype, long ld_out, const int64_t* idx,
                    int n, int D, vtp_stream_t stream);
/* batch-subset stochastic depth (layers/block.py:201-233): out[i*T + t, :] = alpha * x[img_idx[i]*T + t, :]  (= x[indices];
 * alpha = 1 forward, = b/keep for the gradient of the scaled residual) and its dual
 * dst[img_idx[i]*T + t, :] += alpha * src[i*T + t, :]  (= torch.index_add(x, 0, residual, indices, alpha)); indices distinct */
int vtp_gather_images(const float* x, float* out, const int64_t* img_idx, int n_img, int T, int D, float alpha,
                      vtp_stream_t stream);
int vtp_scatter_add_images(const void* src, int src_dtype, float* dst, const int64_t* img_idx, int n_img, int T, int D,
                           float alpha, vtp_stream_t stream);
/* stand-alone SwiGLU gate (layers/ffn.py:77-81) on the 8-interleaved pre-activation: hid = round(round(silu(x1))*x2) */
int vtp_swiglu_fwd(const void* pre, void* hid, long M, int Hs, vtp_stream_t stream);
/* stand-alone in-place axial RoPE (layers/attention.py:12-23,70-89, bf16 arithmetic) on the q,k parts of bf16 qkv */
int vtp_rope_fwd(void* qkv, const void* sin, const void* cos, long rows, int T, int prefix, int D, vtp_stream_t stream);
/* vtp_hf/modeling_vtp.py:297-298 — out[b*L+l] = token_embedding[ids[b,l]] + positional_embedding[l] (fp32) */
int vtp_embed_tokens(const int64_t* ids, const float* emb, const float* pos, float* out, long BL, int L, int D,
                     vtp_stream_t stream);
/* F.normalize(x, dim=-1, eps) (vtp_hf/modeling_vtp.py:276,310; heads/dino_head.py:83-84); norm_out [M] optional */
int vtp_l2norm_fwd(const void* x, int x_dtype, void* y, int y_dtype, float* norm_out, int M, int D, float eps,
                   vtp_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Attention (vtp_b200/csrc/attention.cu)
 * ------------------------------------------------------------------------------------------------------------ */
/* layers/attention.py:110-126 after RoPE (F.scaled_dot_product_attention, scale 1/8, head_dim 64) and the causal
 * nn.MultiheadAttention of layers/block.py:387-412.  qkv bf16 [B*T][3*H*64] packed [q|k|v] x [H][64]; out bf16
 * [B*T][H*64]; lse fp32 [B][H][T] optional (saved for backward).  `prefix` (<= 4) leading tokens (cls) are computed
 * on CUDA cores, the other HW = T-prefix tokens on tcgen05: HW <= 256 by the single-pass kernels (attention.cu,
 * attention_pipe.cu; causal allowed), HW > 256 by the key-streaming online-softmax kernel (attention_long.cu;
 * non-causal only, a causal call returns VTP_ERR_ARG). */
int vtp_attention_fwd(const void* qkv, void* out, float* lse, int B, int T, int H, int prefix, int causal,
                      vtp_stream_t stream);
/* same op on fp32 tensors (CUDA cores) for the fp32-accurate inference mode */
int vtp_attention_fwd_f32(const float* qkv, float* out, int B, int T, int H, int causal, vtp_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Training step (the reference releases no training loop — SURVEY.md M3/a21; these are the autograd duals of the
 * forward stages above plus restated losses and a fused optimiser)
 * ------------------------------------------------------------------------------------------------------------ */
/* dual of vtp_attention_fwd incl. the RoPE rotation (layers/attention.py:70-89,110-126): dqkv = d/d(pre-RoPE qkv) */
int vtp_attention_bwd(const void* qkv, const void* o, const void* dout, const float* lse, void* dqkv,
                      const void* rope_sin, const void* rope_cos, int B, int T, int H, int prefix, int causal,
                      vtp_stream_t stream);
/* dual of vtp_norm_fwd: g[M][D] (fp32 stream gradient) += dx ; dw[D] += ; db[D] += (LayerNorm).  Optional fused
 * by-products of the updated g: g_bf16_out [M][D] (the dY operand of the preceding sub-layer) and g_colsum[D] += Σ_m g
 * (that sub-layer's bias gradient) */
int vtp_norm_bwd(const void* x, int x_dtype, const float* rstd, const float* mean, const float* w, const void* dy_bf16,
                 float* g, float* dw, float* db, int M, int D, int is_ln, void* g_bf16_out, float* g_colsum,
                 vtp_stream_t stream);
/* dual of the SwiGLU gate epilogue (layers/ffn.py:77-81): pre [M][2Hs] 8-interleaved, dhid [M][Hs] -> dpre, dbias */
int vtp_swiglu_bwd(const void* pre, const void* dhid, void* dpre, float* dbias, int M, int Hs, vtp_stream_t stream);
/* dual of the GELU epilogue (text MLP layers/block.py:399-403, DINO head heads/dino_head.py:92-126) */
int vtp_gelu_bwd(const void* pre, const void* dhid, void* dpre, float* dbias, int M, int N, vtp_stream_t stream);
/* y_bf16[M][N] = cast(x[M][ldx]) (optional) ; colsum[N] += column sums (bias gradients) (optional) */
int vtp_cast_colsum(const void* x, int x_dtype, long ldx, void* y_bf16, float* colsum, int M, int N, vtp_stream_t stream);
/* dual of vtp_l2norm_fwd */
int vtp_l2norm_bwd(const void* y, int y_dtype, const float* nrm, const float* dy, void* dx, int dx_dtype, int M, int D,
                   float eps, vtp_stream_t stream);
/* dst[idx[i]][:] += src[i][:] (fp32 atomics): dual of vtp_gather_rows / vtp_embed_tokens */
int vtp_scatter_add_rows(const void* src, int src_dtype, long ld_src, float* dst, long ld_dst, const int64_t* idx, int n,
                         int D, vtp_stream_t stream);
/* g fp32 [B*T][D] -> bf16 [B*(T-prefix)][D] without the prefix rows (+ dcls[prefix][D] += their sum): dual of the
 * cls concat (encoders/vision_transformer.py:198-217), operand of the patch-embed wgrad */
int vtp_strip_prefix(const float* g, void* out_bf16, float* dcls, int B, int T, int prefix, int D, vtp_stream_t stream);
/* fused multi-tensor AdamW on a flat fp32 master buffer: also zeroes grad, refreshes the bf16 compute copy and the EMA
 * teacher (vtp.py:388-401: teacher = m*teacher + (1-m)*student) in the same pass */
int vtp_adamw_step(float* p, float* g, float* m, float* v, void* p_bf16, float* teacher, void* teacher_bf16, long n,
                   float lr, float beta1, float beta2, float eps, float weight_decay, int step, float grad_scale,
                   float ema_momentum, const float* hyper, vtp_stream_t stream);
/* device-resident step state `hyper` float[8] = {step, 1-b1^step, 1-b2^step, lr, weight decay, EMA momentum, -, -}: advances
 * the step and looks the scheduled lr / wd / teacher momentum up in device tables (restating the reference's
 * CosineScheduler, models/utils/text_utils.py:160-207, which is a precomputed table as well; null table = keep the value).
 * vtp_adamw_step reads it when `hyper` is non-null, so a CUDA graph of the whole training step carries no host scalars. */
int vtp_hyper_tick(float* hyper, float beta1, float beta2, const float* lr_table, const float* wd_table,
                   const float* momentum_table, int table_len, vtp_stream_t stream);
int vtp_cast_f32_to_bf16(const float* x, void* y, long n, vtp_stream_t stream);
int vtp_axpby(float* y, const float* x, float a, float b, long n, vtp_stream_t stream);
/* OpenCLIP ClipLoss row-wise softmax-CE on a similarity block sim = I·Tᵀ with logits = exp(*log_scale)·sim
 * (vtp_hf/modeling_vtp.py:329): loss, d(log_scale) and G = dL/dsim (bf16) */
int vtp_softmax_ce(const float* sim, long ld, int R, int C, int label0, const float* log_scale, void* G_bf16, long ldg,
                   float coef, float* loss_acc, float* dscale_acc, vtp_stream_t stream);
/* DINOv2 centred+sharpened teacher softmax, in place on bf16 logits [R][K] */
int vtp_dino_teacher_probs(void* t_bf16, const float* center, int R, int K, float temp, vtp_stream_t stream);
/* DINOv2 DINOLoss/iBOTPatchLoss cross-entropy of student logits [R][K] vs up to two teacher rows: loss + in-place grad */
int vtp_dino_student_ce(void* s_bf16, const void* tprobs_bf16, const int* t0, const int* t1, const float* w, int R, int K,
                        float temp, float* loss_acc, vtp_stream_t stream);
/* pixel L1 loss + gradient (+ optional extra NCHW gradient, e.g. LPIPS), written pixel-unshuffled as the bf16 dY of
 * proj_out (decoders/pixel_decoder.py:157-160) */
int vtp_recon_l1_grad(const void* rec, int rec_dtype, const float* tgt, const float* dlp, void* out_bf16, float* loss_acc,
                      int B, int C, int gh, int gw, int r, float coef, vtp_stream_t stream);
/* heads/dino_head.py:48-49 weight_norm(dim=0): W[k,:] = g[k] v[k,:]/||v[k,:]|| (bf16) and its dual */
int vtp_weight_norm_fwd(const float* v, const float* g, void* w_bf16, float* vnorm, int K, int D, vtp_stream_t stream);
int vtp_weight_norm_bwd(const float* v, const float* g, const float* vnorm, const float* dW, float* dv, float* dg, int K,
                        int D, vtp_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * LPIPS perceptual loss (utils/lpips.py:61-171); the VGG16 convolutions run on vtp_gemm_bf16 (conv_C > 0)
 * ------------------------------------------------------------------------------------------------------------ */
/* ScalingLayer (lpips.py:103-114) + 3x3 im2col of the 3-channel image: NCHW (fp32|bf16) -> bf16 [B*H*W][32], k=tap*3+c */
int vtp_lpips_prep(const void* img, int img_dtype, void* out_bf16, int B, int H, int W, vtp_stream_t stream);
/* nn.MaxPool2d(2,2) on NHWC bf16 (lpips.py:127-149 via torchvision vgg16.features) */
int vtp_maxpool2_fwd(const void* x, void* y, int B, int H, int W, int C, vtp_stream_t stream);
/* dual of MaxPool2d(2,2) fused with the tap-gradient add and the ReLU mask: dz = (gtap + route(dpool)) * (y > 0) */
int vtp_pool_relu_bwd(const void* y, const void* dpool, const void* gtap, void* dz, int B, int H, int W, int C,
                      vtp_stream_t stream);
/* one LPIPS tap (lpips.py:88-100,169-175): normalize_tensor, squared diff, lin 1x1, spatial mean: loss += and gradient
 * w.r.t. the reconstruction features f0 (bf16 [P][C]) */
int vtp_lpips_tap(const void* f0, const void* f1, const float* w, void* g0, long P, int C, float coef, float* loss_acc,
                  vtp_stream_t stream);
/* col2im of the conv1_1 input gradient + ScalingLayer backward: bf16 [B*H*W][32] -> fp32 NCHW d(image) */
int vtp_lpips_img_grad(const void* dcol, float* dimg, int B, int H, int W, vtp_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Contrastive exchange over NVLink peer memory (vtp_b200/csrc/clip.cu): collective C2 of SURVEY.md §8e — the feature
 * all-gather that OpenCLIP's ClipLoss performs before vtp_hf/modeling_vtp.py:329's logits — fused with the logits, the
 * logit-scale softmax-CE and the gradient matrices.  No backward collective is needed (every rank holds the full
 * Bg x Bg similarity matrix).
 * ------------------------------------------------------------------------------------------------------------ */
/* img_ptrs/txt_ptrs: HOST arrays of `world` device pointers (own + IPC-mapped peers) to L2-normalised bf16 features
 * [B][E].  One kernel: gather through peer memory + S = I_all·T_allᵀ fp32 [world*B][ld] and St = Sᵀ; fi_all/ft_all bf16
 * [world*B][E] receive the gathered features. */
int vtp_clip_gather_logits(const void* const* img_ptrs, const void* const* txt_ptrs, int world, int B, int E, float* S,
                           float* St, long ld, void* fi_all, void* ft_all, vtp_stream_t stream);
/* lse[0][r] / lse[1][r] = logsumexp_c exp(*log_scale)·S[r][c] / ·St[r][c] for all Bg rows; rows [row0,row0+B) add
 * coef·(lse − logit[r][r]) to *loss_acc and Σ_c g·logit to *dscale_acc (g = coef (softmax − onehot)) */
int vtp_clip_lse(const float* S, const float* St, long ld, int Bg, int row0, int B, const float* log_scale, float coef,
                 float* lse, float* loss_acc, float* dscale_acc, vtp_stream_t stream);
/* dMi / dMt bf16 [B][Bgp]: d(Σ_ranks L_local)/dS (resp. /dSt) rows [row0,row0+B): row-direction softmax term +
 * column-direction softmax term − 2·onehot, times coef·exp(*log_scale); columns [Bg,Bgp) zero.
 * Then dI_local = dMi·T_all and dT_local = dMt·I_all (vtp_gemm_bf16, b_mn_major). */
int vtp_clip_grad(const float* S, const float* St, long ld, int Bg, int Bgp, int row0, int B, const float* log_scale,
                  float coef, const float* lse, void* dMi, void* dMt, vtp_stream_t stream);
/* Peer-memory plumbing (set-up time only; the ONLY entry points that allocate / synchronise): a zeroed cudaMalloc
 * buffer, its 64-byte CUDA IPC handle, mapping of a peer's handle, and a flag barrier over the ranks' signal pads
 * (pad_ptrs: HOST array of `world` device pointers to uint64[world] pads; epoch strictly increasing; *err_flag = 1 if
 * a peer did not arrive within ~20 s). */
int vtp_comm_alloc(long bytes, void** ptr);
int vtp_comm_free(void* ptr);
int vtp_comm_get_handle(void* ptr, unsigned char* handle64);
int vtp_comm_open_handle(const unsigned char* handle64, void** peer_ptr);
int vtp_comm_close_handle(void* peer_ptr);
/* flag barrier; on time-out (~20 s) *err_flag = 1 and, if given, *poison = NaN (the caller's loss slot: the failure
 * then travels with the step's result instead of needing its own host read) */
int vtp_comm_barrier(const void* const* pad_ptrs, int world, int rank, long epoch, int* err_flag, float* poison,
                     vtp_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Data formats either side of the encode / decode path (vtp_b200/csrc/latents_io.cu; SURVEY.md §8f ranks 1-2)
 * ------------------------------------------------------------------------------------------------------------ */
/* generation/tokenizer/vtp_tokenizer.py:106-119 (decode_to_images) and tools/test_reconstruction_hf.py:371-372,
 * 401-402: torchvision Normalize(inv_mean, inv_std) = (x - sub3[c]) / div3[c], x255, clamp [0,255], truncation to
 * uint8, NCHW (fp32|bf16) -> NHWC, in one pass.  Bit-exact with the torch expression. */
int vtp_image_to_u8(const void* img, int img_dtype, const float* sub3, const float* div3, uint8_t* out_nhwc, int B, int H,
                    int W, vtp_stream_t stream);
/* latents_stats.pt of generation/tools/extract_features_vtp.py:128-131: sum[c] += sum x, sumsq[c] += sum x^2 (fp64)
 * over latents [B][C][HW] (fp32|bf16) */
int vtp_latent_stats(const void* lat, int dtype, int B, int C, int HW, double* sum, double* sumsq, vtp_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Input side of the training step (vtp_b200/csrc/data.cu; SURVEY.md §8f rank 4 — the reference releases no training
 * data loader, README.md:245 points at DINOv2 / OpenCLIP): every crop of the step in one pass.
 * ------------------------------------------------------------------------------------------------------------ */
/* out[n] (fp32 NCHW [N][3][S][S]) = normalise(bilinear_resize(crop(src[src_idx[n]], boxes[n] = x0,y0,w,h), S x S, half-pixel
 * centres), optional horizontal flip); src uint8 NHWC [B][H][W][3]; mean3 / std3 are HOST pointers (3 floats each). */
int vtp_crop_resize_norm(const uint8_t* src_nhwc, int B, int H, int W, const int* src_idx, const float* boxes_xywh,
                         const uint8_t* flips, float* out_nchw, int N, int S, const float* mean3, const float* std3,
                         vtp_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* VTP_B200_H */
