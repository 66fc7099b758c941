/*
 * pfd_b200 — C ABI of the B200 (sm_100a) kernel library behind the Prompt-Free-Diffusion hot path.
 *
 * The reference (SHI-Labs/Prompt-Free-Diffusion) has NO native boundary: every op on the path is a
 * torch/ATen library call made from lib/model_zoo/*.py.  This header is therefore the boundary a
 * maintainer would bind (via ctypes, see INTEGRATION.md) to replace those call sites.  Each entry
 * point cites the reference call site(s) it replaces.
 *
 * Conventions
 *   - plain C types only: device pointers as void*, sizes as int32/int64, cudaStream_t as void*.
 *   - every function returns 0 on success; non-zero = error, text via pfd_last_error().
 *   - no ownership transfer: the caller allocates every buffer (e.g. through torch) and keeps it
 *     alive until the stream has executed the call.
 *   - all activations are fp16, channel-last ("NHWC" / token-major [B, N, C]); all reductions and
 *     accumulations are fp32.
 *   - thread safety: calls on distinct streams are independent; pfd_last_error is thread-local.
 */
#ifndef PFD_B200_H_
#define PFD_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PFD_ABI_VERSION 2
#if defined(__GNUC__)
#define PFD_API __attribute__((visibility("default")))
#else
#define PFD_API
#endif
#define PFD_MAX_SEG 3

/* activation codes for pfd_gemm_desc.act */
enum {
  PFD_ACT_NONE = 0,
  PFD_ACT_SILU = 1,   /* x*sigmoid(x)          (openaimodel.py:203 nn.SiLU, autokl_modules.py:33) */
  PFD_ACT_GELU = 2,   /* exact erf GELU        (swin.py:84 nn.GELU)                               */
  PFD_ACT_RELU = 3,   /* F.relu, NaN kept (seecoder.py:24, controlnet_annotator/hed/__init__.py:37) */
  PFD_ACT_GEGLU = 4   /* value*gelu(gate), weights packed [value|gate] per N tile (attention.py:44-51) */
};

PFD_API int pfd_version(void);
PFD_API const char* pfd_last_error(void);
/* number of kernels launched by this library in this process so far (bench.py: gpu_launches) */
PFD_API int64_t pfd_launch_count(void);
/* Run-time tuning switches, so that variants can be A/B-timed inside one process (tools/ab_unet.py); name == NULL
 * resets all of them to the built-in defaults.  Unknown names are stored and ignored.  Known names (default):
 *   gemm_tma_epi (1)   TMA-store epilogue of pfd_gemm_f16 for plain channel-last outputs (0 = register epilogue)
 *   gemm_pair (0)      1 = CTA-pair kernel (cta_group::2) for long-K contractions, 2 = wherever applicable
 *   gemm_streamk (0)   stream-K tail of the persistent GEMM
 *   xattn_short (1)    persistent single-score-tile kernel of pfd_flash_attn_* for Nk <= 160, d <= 48
 *   flash_poly_mod (0) exponent path of the attention softmax: 1 = packed-half MUFU, n > 1 = every n-th pair on the FMA pipe */
PFD_API int pfd_set_option(const char* name, int32_t value);

/*
 * pfd_gemm_f16 — the tcgen05 tensor-core contraction used for every Linear, 1x1 conv, 3x3 conv
 * (implicit GEMM, TMA does the im2col) and batched QK^T / PV product on the path.
 *
 *   out[n, y, x, :] = act( alpha * sum_seg sum_tap sum_c A_seg[n, y*s+dy-1+o, x*s+dx-1+o, c] * Wt[:, k(seg,tap,c)]
 *                          + bias + rowadd[n, :] ) + residual[n, y, x, :]
 *
 * Replaces: torch.nn.functional.conv2d / F.linear / torch.einsum / torch.bmm at
 *   openaimodel.py:203,229,240 (ResBlock convs + skip), :150 (Downsample), :105 (Upsample conv),
 *   attention.py:169-176,186-201 (to_q/k/v/out, QK^T, PV), :47,67 (GEGLU proj, ff out),
 *   attention.py:329,343 (proj_in/out), openaimodel.py:217-223,2629-2633 (emb_layers, time_embed),
 *   controlnet.py:165-181,299, autokl_modules.py:92-106,162-202,487,529, autokl.py:27,
 *   swin.py:88-90,171-173,322, seecoder.py:70-76,111,161,215-217,358,381.
 *
 * A operand: up to PFD_MAX_SEG channel-last fp16 tensors sharing the output raster (W,H,NB);
 *   segment s contributes taps[s] (1 or 9) x a_c[s] entries of K, in that order, so the weight
 *   matrix Wt is [N, K] row-major with K = sum_s taps[s]*a_c[s] (k = base_s + tap*a_c[s] + c).
 *   A plain [M,K] GEMM is W=M, H=1, NB=1 (or NB=batch for a batched GEMM with b_batch_stride!=0).
 * Requirements: a_c[s] % 8 == 0, K % 8 == 0, N % 8 == 0, all pointers 16-byte aligned.
 */
typedef struct pfd_gemm_desc {
  int32_t nseg;
  int32_t taps[PFD_MAX_SEG];
  int32_t a_c[PFD_MAX_SEG];
  const void* a_ptr[PFD_MAX_SEG];
  int64_t a_sx[PFD_MAX_SEG]; /* element strides of A: pixel, row, image */
  int64_t a_sy[PFD_MAX_SEG];
  int64_t a_sn[PFD_MAX_SEG];
  int32_t in_w, in_h;        /* extent of the A raster (== W,H for stride 1; ~2W,2H for stride 2) */
  int32_t stride;            /* 1 or 2 (3x3 stride-2 conv, openaimodel.py:150) */
  int32_t W, H, NB;          /* output raster: width, height, images (or rows, 1, batches) */

  const void* b_ptr;         /* weights [N, K] fp16 (K contiguous) */
  int32_t N;
  int64_t K;                 /* row pitch of b in elements (>= sum of segment K) */
  int64_t b_batch_stride;    /* 0: weights shared; else elements between per-image B matrices */

  float alpha;
  int32_t act;
  const void* bias;          /* [N] fp16 or NULL */
  const void* rowadd;        /* [NB, >=N] fp16 or NULL: per-image broadcast add (time embedding) */
  int64_t rowadd_ld;         /* row pitch of rowadd in elements (0 = N) */
  const void* residual;      /* same addressing as out, or NULL */

  void* out;                 /* fp16 */
  /* out offset (elements) = (n/ndiv)*so_n1 + (n%ndiv)*so_n0 + y*so_y + x*so_x
   *                         + (c/cdiv)*so_c1 + (c%cdiv)*so_c0                     */
  int64_t so_n1, so_n0, so_y, so_x, so_c1, so_c0;
  int32_t ndiv, cdiv;
  int32_t bn_force;          /* 0 = library picks the N tile; else one of 64/128/160/192/256 (GEGLU packing) */
  int32_t tap_off;           /* 3x3 taps read A at (y*s + dy - 1 + tap_off): 0 = symmetric padding 1; 1 = the VAE
                                encoder's F.pad(x,(0,1,0,1)) + stride-2 conv with padding 0 (autokl_modules.py:69-76) */
  void* stream;
} pfd_gemm_desc;

PFD_API int pfd_gemm_f16(const pfd_gemm_desc* d);
/*
 * GroupNorm(32 groups) [+ SiLU] over channel-last fp16, optionally over the channel-concatenation
 * of two tensors (the UNet skip concat, pfd.py:356,519) — writes one contiguous [NB,H,W,C1+C2].
 * Replaces: diffusion_utils.py:175-191 (GroupNorm32, eps 1e-5) + nn.SiLU (openaimodel.py:201-203,
 *   224-229, 2732-2734), attention.py:83-84 (eps 1e-6), autokl_modules.py:33-39,
 *   seecoder.py:359,383.
 * ws: scratch of at least NB*groups*16 + NB*4 bytes (fp64 sum / sum-of-squares per (image, group), then one
 *     32-bit arrival counter per image for the single-pass kernel),
 *     16-byte aligned.  zero_ws != 0: the call zeroes it first (one extra memset node); zero_ws == 0: the
 *     caller guarantees it is already zero (e.g. one bulk memset of many slots per network evaluation).
 */
PFD_API int pfd_groupnorm_f16(const void* x1, int32_t c1, const void* x2, int32_t c2, int32_t NB,
                      int64_t HW, int32_t groups, const void* gamma, const void* beta, float eps,
                      int32_t silu, void* out, float* ws, int32_t zero_ws, void* stream);

/* LayerNorm over the last dim of [rows, C] fp16 (attention.py:294-296, swin.py norms, seecoder.py norms).
 * Optional fused residual: out = LN(x + res) (post-norm layers of seecoder.py:85-90,135-136). */
PFD_API int pfd_layernorm_f16(const void* x, const void* res, int64_t rows, int32_t C, const void* gamma,
                      const void* beta, float eps, void* out, void* stream);

/*
 * Row softmax over fp16 scores [batch, rows, cols] (row pitch ld), in place or to out:
 *   p = softmax( round_fp16(s) * scale + bias[(b % bias_mod_h)...] + mask[...] )
 * reproducing the reference's fp16 score rounding (attention.py:188-197, autokl_modules.py:188-192,
 * swin.py:187-203).  bias: [nheads, rows, cols] fp16 or NULL, selected by (b % nheads);
 * mask: [nwin, rows, cols] fp16 or NULL, selected by ((b / nheads) % nwin).
 */
PFD_API int pfd_softmax_f16(void* s, int64_t batch, int32_t rows, int32_t cols, int64_t ld, float scale,
                    const void* bias, int32_t nheads, const void* mask, int32_t nwin, void* stream);

/* sinusoidal timestep embedding [cos | sin], fp32 math, fp16 out (diffusion_utils.py:131-151). */
PFD_API int pfd_timestep_embedding_f16(const int64_t* t, int32_t n, int32_t dim, float max_period,
                               void* out, void* stream);

/* nearest-neighbour 2x upsample, channel-last (openaimodel.py:114, autokl_modules.py:54). */
PFD_API int pfd_upsample2x_f16(const void* x, int32_t NB, int32_t H, int32_t W, int32_t C, void* out,
                       void* stream);

/* layout converts at the pipeline edges: NCHW fp16/fp32 <-> channel-last fp16 (with channel pad):
 * out[n,y,x,c] = x[n,c,y,x]*mul + add for c < C, 0 for the pad channels (autokl.py:34: x*2-1). */
PFD_API int pfd_nchw_to_nhwc_f16(const void* x, int32_t src_is_f32, int32_t NB, int32_t C, int32_t H,
                         int32_t W, int32_t Cpad, float mul, float add, void* out, void* stream);
/* out_nchw[n,c,y,x] = clamp(x[n,y,x,c]*mul + add, lo, hi) for c < C (autokl.py:47,53: (dec+1)/2, clamp) */
PFD_API int pfd_nhwc_to_nchw_f16(const void* x, int32_t NB, int32_t C, int32_t H, int32_t W, int32_t Cpad,
                         float mul, float add, float lo, float hi, void* out, void* stream);

/* explicit im2col for 3x3 convs whose Cin is too small for the TMA path (Cin<8: UNet/VAE conv_in,
 * ControlNet hint stem): out[n,y,x, tap*Cin + c] (K padded to Kpad with zeros). */
PFD_API int pfd_im2col3x3_f16(const void* x, int32_t NB, int32_t H, int32_t W, int32_t C, int32_t stride,
                      int32_t Kpad, void* out, void* stream);

/* out = a*sa + b*sb (elementwise fp16, fp32 math); b may be NULL. */
PFD_API int pfd_axpby_f16(const void* a, float sa, const void* b, float sb, int64_t n, void* out,
                  void* stream);
/* out[n, :] = a[n, :] + row[:]  (level/position embeddings, seecoder.py:402,513) */
PFD_API int pfd_add_rowvec_f16(const void* a, const void* row, int64_t rows, int32_t C, void* out,
                       void* stream);

/*
 * Fused classifier-free-guidance combine + DDIM update (ddim.py:150-151,159-171), fp16 in/out with
 * the reference's fp16 rounding points reproduced:
 *   e = e_u + s*(e_c - e_u); pred_x0 = (x - sqrt(1-a_t)*e)/sqrt(a_t);
 *   x_prev = sqrt(a_prev)*pred_x0 + sqrt(1-a_prev-sigma^2)*e   (eta = 0 path; sigma*noise added by caller)
 * eps: [2*B, ...] as [uncond | cond] halves of `half_n` elements each; coefficients are read from a
 * device table coef[step*4 + {0..3}] = {a_t, a_prev, sigma_t, sqrt_one_minus_at} (fp32) indexed by
 * the device-side int *step so that a captured CUDA graph can be replayed for every step.
 * noise (optional, eta > 0, ddim.py:168-170): x_prev += sigma_t * noise * temperature with the reference's fp16
 * rounding order.  log_tab (optional): int32 slot per schedule index (-1 = none); the step's x_prev / pred_x0
 * are also stored at log_xt / log_x0 + slot*half_n (the `intermediates` lists, ddim.py:122-124).
 */
PFD_API int pfd_ddim_step_f16(const void* eps, const void* x, int64_t half_n, float guidance,
                      const float* coef, const int32_t* step, void* x_prev, void* pred_x0,
                      const void* noise, float temperature, const int32_t* log_tab, void* log_xt,
                      void* log_x0, void* stream);

/* VAE encoder posterior (distributions.py:24-37, autokl.py:33-42, pfd.py:266-273): moments = channel-last
 * [B,H,W,cpad] quant_conv output (mean | logvar in the first 2*zc channels); logvar clamped to [-30,20],
 * std = exp(logvar/2), sample = scale*(mean + std*noise) with caller-drawn fp32 noise [B,zc,H,W] (NULL: mode).
 * Outputs NCHW fp16 [B,zc,H,W]; each may be NULL. */
PFD_API int pfd_vae_posterior_f16(const void* moments, int32_t B, int32_t zc, int32_t H, int32_t W, int32_t cpad,
                                  const float* noise, float scale, void* mean, void* logvar, void* stdv,
                                  void* sample, void* stream);

/* Device-side loop header of one DDIM step (ddim.py:108-113): *step -= 1; t_out[0..nb) = ttab[*step].
 * Lets one CUDA graph hold several (or all) steps of the sampling loop with no host work in between. */
PFD_API int pfd_ddim_begin_step(int32_t* step, const int64_t* ttab, int64_t* t_out, int32_t nb, void* stream);

/* Swin window plumbing on channel-last [B,H,W,C] (swin.py:269-304): pad + cyclic shift + window
 * partition in one gather (fwd) and the inverse scatter + crop (bwd). */
PFD_API int pfd_window_gather_f16(const void* x, int32_t B, int32_t H, int32_t W, int32_t C, int32_t ws,
                          int32_t shift, void* out, void* stream);
PFD_API int pfd_window_scatter_f16(const void* win, int32_t B, int32_t H, int32_t W, int32_t C,
                           int32_t ws, int32_t shift, const void* residual, void* out,
                           void* stream);
/* PatchMerging 2x2 gather -> [B, H/2*W/2, 4C] in the reference's x0,x1,x2,x3 order (swin.py:341-346). */
PFD_API int pfd_patch_merge_gather_f16(const void* x, int32_t B, int32_t H, int32_t W, int32_t C,
                               void* out, void* stream);

/*
 * Fused flash attention (tcgen05): out[b, i, h*d + :] = softmax_j( fp16(q_i . k_j) * scale ) @ v  per (b, h),
 * scores never leave the SM.  Replaces attention.py:186-201 (einsum -> softmax -> einsum) for the UNet /
 * ControlNet self- and cross-attention.
 *   q  [B*heads, q_rows, d]   (first Nq rows valid)      k [B*heads, k_rows, d] (first Nk rows valid)
 *   vt [B*heads, d, vt_pitch] (V transposed, first Nk columns valid)
 *   out element (b, i, h, c) at  b*o_sb + i*o_sq + h*d + c.       d % 8 == 0, d <= 192.
 * Nk <= 160 with d <= 48 (the cross-attention against the 148 SeeCoder context tokens at the UNet's d = 40 level,
 * attention.py:178-201 with `context`) runs a persistent kernel whose single score tile holds every key (exact row
 * maximum, no online softmax); everything else the 64-key-block flash kernel.
 */
PFD_API int pfd_flash_attn_f16(const void* q, const void* k, const void* vt, void* out, int32_t B,
                               int32_t heads, int32_t Nq, int32_t Nk, int32_t d, int32_t q_rows,
                               int32_t k_rows, float scale, int64_t vt_pitch, int64_t o_sb, int64_t o_sq,
                               int32_t reserved, void* stream);

/* Same kernel with arbitrary 4-D strided operands: q, k as [B, heads, N, d] views and vt as [B, heads, d, Nk]
 * views, strides {batch, head, row} in elements (rows contiguous).  Lets a fused q|k projection GEMM and a
 * "swapped" V^T = Wv . X^T GEMM ([C, B*N] row-major) feed the kernel without any re-layout. */
PFD_API int pfd_flash_attn_strided_f16(const void* q, const void* k, const void* vt, void* out, int32_t B,
                                       int32_t heads, int32_t Nq, int32_t Nk, int32_t d,
                                       const int64_t* q_strides, const int64_t* k_strides,
                                       const int64_t* vt_strides, float scale, int64_t o_sb, int64_t o_sq,
                                       void* stream);

/* PatchEmbed gather (swin.py:479-489): NCHW image (fp16/fp32) -> [B, ceil(H/P), ceil(W/P), Kpad] rows in
 * the K order of the flattened conv weight [O, C*P*P]; zero padding for ragged H/W and K..Kpad. */
PFD_API int pfd_patchify_f16(const void* x, int32_t src_is_f32, int32_t B, int32_t C, int32_t H,
                             int32_t W, int32_t P, int32_t Kpad, void* out, void* stream);

/*
 * ControlNet.preprocess(type='canny') on the GPU (controlnet.py:332-360 -> controlnet_annotator/canny/__init__.py:4-5,
 * i.e. cv2.Canny(rgb_u8, low, high) with aperture 3 / L1 gradient, bit-exact): x is an NCHW [B,3,H,W] image in
 * [0,1] (fp16 or fp32), quantised like ToPILImage (x.mul(255).byte()); out is float32 [B,3,H,W] with 1.0 on edge
 * pixels (ToTensor + repeat(1,3,1,1)).  workspace: pfd_canny_workspace_bytes(B,H,W) bytes of device memory.
 * The call synchronises `stream` (hysteresis runs until a host-visible fixed point): not graph-capturable.
 * sweeps_out (optional, host): number of hysteresis sweeps that were needed.
 */
PFD_API int64_t pfd_canny_workspace_bytes(int32_t B, int32_t H, int32_t W);
PFD_API int pfd_canny_f32(const void* x, int32_t src_is_f32, int32_t B, int32_t H, int32_t W, int32_t low,
                          int32_t high, void* workspace, float* out, int32_t* sweeps_out, void* stream);
/* ToTensor(ToPILImage(x)) = floor(x*255)/255 as float32 (controlnet.py:345-348, preprocess type 'input'). */
PFD_API int pfd_image_u8_roundtrip_f32(const void* x, int32_t src_is_f32, int64_t n, float* out, void* stream);

/*
 * ControlNet.preprocess(type='hed' / 'softedge_v11p') on the GPU (controlnet.py:370-376 ->
 * controlnet_annotator/hed/__init__.py:102-128).  The network's 3x3 convs (+ ReLU) run on pfd_gemm_f16 with every
 * conv bias multiplied by a power-of-two activation scale s (ReLU and max-pool commute with it, so every activation
 * is exactly s times the reference's; s keeps the raw 0-255 input's activations inside fp16).  Stream-ordered and
 * capturable.
 */
#define PFD_HED_MAPS 5
/* Network input (hed/__init__.py:111-113,52): x NCHW [B,3,H,W] fp16/fp32 in [0,1], quantised like ToPILImage,
 * out[n,y,x,c] = fp16((u8 - norm[c]) * scale), channel-last [B,H,W,3].  norm: device fp32 [3].  The subtraction comes
 * before the first conv's zero padding, as in the reference. */
PFD_API int pfd_hed_input_f16(const void* x, int32_t src_is_f32, int32_t B, int32_t H, int32_t W, const float* norm,
                              float scale, void* out, void* stream);
/* 2x2 / stride-2 max-pool, channel-last [NB,H,W,C] -> [NB,H/2,W/2,C] (floor; hed/__init__.py:34 F.max_pool2d).
 * C % 8 == 0. */
PFD_API int pfd_maxpool2x2_f16(const void* x, int32_t NB, int32_t H, int32_t W, int32_t C, void* out, void* stream);
/* 1x1 conv to one channel (DoubleConvBlock.projection, hed/__init__.py:30,38) with fp32 accumulation and output:
 * out[m] = dot(x[m,:], w) * inv_scale + b[0] for channel-last fp16 x [M,C]; w device fp32 [C], b device fp32 [1].
 * inv_scale = 1/s undoes the activation scale.  C % 8 == 0. */
PFD_API int pfd_hed_project_f32(const void* x, int64_t M, int32_t C, const float* w, const float* b, float inv_scale,
                                float* out, void* stream);
/* The host tail of apply_hed (hed/__init__.py:118-128) + ToTensor / repeat (controlnet.py:373-375):
 * maps[k] is a device fp32 [B, map_h[k], map_w[k]] logit map (host arrays of PFD_HED_MAPS entries, each map no
 * larger than HxW); each is resized to HxW like cv2.resize(INTER_LINEAR) on float32, the maps are averaged in fp32,
 * e = sigmoid(mean) in fp64, u8 = (uint8)clip(e*255, 0, 255); out float32 [B,3,H,W] = u8/255 in all three channels.
 * *nonfinite (device int32, zeroed by the call) counts pixels whose mean logit is not finite. */
PFD_API int pfd_hed_fuse_f32(const float* const* maps, const int32_t* map_h, const int32_t* map_w, int32_t B,
                             int32_t H, int32_t W, float* out, int32_t* nonfinite, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PFD_B200_H_ */
