/* libimagharmony_sm100.so -- C ABI of the B200-native SDXL / IMAGHarmony denoise hot path.
 *
 * The reference (muzishen/IMAGHarmony) has no FFI of its own: its operator boundary is the diffusers
 * attention-processor protocol (ip_adapter/attention_processor.py:364-371) and the nn.Module calls inside the
 * diffusers UNet it drives from ip_adapter/custom_pipelines.py:338-345.  Each entry point below names the reference
 * call site(s) whose arithmetic it replaces.  The Python host (imagharmony_b200/ops.py) binds these with ctypes.
 *
 * Conventions
 *   - all tensors are fp16 ("__half") device pointers unless stated; activations are NHWC / [rows, channels].
 *   - `stream` is a cudaStream_t passed as void*; nothing here allocates, synchronises or keeps state except an
 *     internally locked TMA-descriptor cache.
 *   - return 0 on success, <0 on error; ih_last_error() returns a thread-local description.
 */
#ifndef IH_API_H
#define IH_API_H

#ifdef __cplusplus
extern "C" {
#endif

#define IH_API_VERSION 1

/* epilogue flags for ih_gemm_f16 */
#define IH_EPI_NONE 0
#define IH_EPI_GEGLU 1 /* out[:, j] = (acc[:, j] + b[j]) * gelu_erf(acc[:, F + j] + b[F + j]),  N = 2F */
#define IH_EPI_SILU 2  /* out = silu(acc + bias) */
#define IH_EPI_GELU 4  /* out = gelu_erf(acc + bias) */
#define IH_EPI_QUICK_GELU 8 /* out = x * sigmoid(1.702 x), x = acc + bias  (CLIP-L text tower MLP, scope row f2) */

const char* ih_last_error(void);
int ih_version(void);
long long ih_launch_count(void); /* kernels launched by this library since the last reset */
void ih_launch_count_reset(void);

/* out[M,N] = epi(A[M,K] @ W[N,K]^T + bias[N] + rowbias[row / rows_per_group, N]) + residual[M,N]
 * Replaces nn.Linear: attention_processor.py:292,299-300,320 (AttnProcessor2_0 to_q/to_k/to_v/to_out),
 * :396,410-411,432-433,453 (IPAttnProcessor2_0 incl. to_k_ip/to_v_ip), and the diffusers proj_in/proj_out/FF/1x1
 * conv layers reached through custom_pipelines.py:338-345.  tile_n: 0 = auto, else 64/128/256. */
int ih_gemm_f16(const void* a, long long lda, const void* w, const void* bias, const void* rowbias,
                int rows_per_group, long long ld_rowbias, const void* residual, long long ldr, void* out,
                long long ldo, int M, int N, int K, int epilogue, int tile_n, void* stream);

/* ih_gemm_f16 with LayerNorm folded in (BasicTransformerBlock norm1/2/3 -> attn / FF projections).
 *   stats_out != NULL : additionally write, per output row and 64-column slab, (sum, sum of squares) of the fp16 values
 *                       stored: float [ceil(N/64), M, 2] (one writer per slot; deterministic).
 *   ln_stats  != NULL : `a` holds the RAW (un-normalised) rows; `w` is the weight pre-multiplied by the LayerNorm gamma
 *                       with every row centred (w[n,k] = W[n,k] gamma[k] - mean_k(W[n,:] gamma)), so that
 *                       a w^T = (a - mean(a)) (W gamma)^T; `bias` = W beta + b.  The epilogue applies
 *                       out = rstd[m] * acc + bias[n], rstd rebuilt from the producer's slabs
 *                       ln_stats [ln_slabs, M, 2] over the K features with epsilon ln_eps. */
int ih_gemm_ln_f16(const void* a, long long lda, const void* w, const void* bias, const void* rowbias,
                   int rows_per_group, long long ld_rowbias, const void* residual, long long ldr, void* out,
                   long long ldo, int M, int N, int K, int epilogue, int tile_n, const void* ln_stats, int ln_slabs,
                   float ln_eps, void* stats_out, void* stream);

/* out = epi(alpha * (A W^T) + bias) + residual: ih_gemm_f16 with an output scale.  Used by the VAE decoder's SCALED
 * RESIDUAL STREAM (scope row f1): the reference upcasts the SDXL VAE to fp32 because its activations overflow fp16
 * (custom_pipelines.py:366-371); here the residual stream is stored as 2^-k * x (GroupNorm is scale-invariant, every
 * conv / linear that writes the stream scales its output and bias by 2^-k), which is exact in real arithmetic. */
int ih_gemm_scaled_f16(const void* a, long long lda, const void* w, const void* bias, const void* residual,
                       long long ldr, void* out, long long ldo, int M, int N, int K, int epilogue, float alpha,
                       void* stream);

/* One-shot hint for the NEXT ih_gemm_* / ih_conv2d_* launch of the calling thread: while it runs, an idle warp of every
 * CTA prefetches a slice of `weights` (the weight matrix of the kernel that will follow it) into L2
 * (cp.async.bulk.prefetch.L2).  Inside a denoise step every layer's weights come from HBM; this hides the first round
 * trips of the following launch.  A pure performance hint: results never depend on it. */
void ih_gemm_prefetch_next(const void* weights, long long bytes);

/* Debug aid: CTA 0 of later GEMM / conv launches writes %globaltimer stamps into this device buffer (>= 16 uint64);
 * NULL disables.  Not used on the product path. */
void ih_gemm_set_trace(void* device_buffer);

/* 3x3 convolution, padding 1, stride 1|2, NHWC activations, weight [Cout, 9*Cin] (tap-major: (ky*3+kx)*Cin + c).
 * out = conv(x) + bias[Cout] + rowbias[b*ld_rowbias + c] + residual.  Replaces diffusers ResnetBlock2D / Downsample2D /
 * Upsample2D nn.Conv2d (custom_pipelines.py:338-345 -> unet forward). */
int ih_conv2d_f16(const void* x, const void* w, const void* bias, const void* rowbias, long long ld_rowbias,
                  const void* residual, void* out, int B, int Hin, int Win, int Cin, int Cout, int ksize, int stride,
                  int tile_n, void* stream);
/* 3x3 conv (stride 1, pad 1) with a FUSED 1x1 shortcut convolution over one or two further NHWC sources:
 *   out = conv3x3(x) + [sc0 | sc1] Wsc^T + bias + rowbias        w = [Cout, 9*Cin + Csc0 + Csc1] (3x3 taps, then Wsc)
 * i.e. diffusers ResnetBlock2D `conv2(h) + conv_shortcut(cat(hidden, skip))` as ONE launch: the shortcut's K blocks
 * accumulate into the same TMEM tile and the channel concat of the up-blocks is never materialised.  Csc0, Csc1 % 64 == 0;
 * sc1 may be NULL. */
int ih_conv2d_shortcut_f16(const void* x, const void* w, const void* bias, const void* rowbias, long long ld_rowbias,
                           const void* sc0, int Csc0, const void* sc1, int Csc1, void* out, int B, int H, int W, int Cin,
                           int Cout, void* stream);
/* out = alpha * conv(x) + bias + residual (3x3, pad 1): the VAE decoder's scaled residual stream, see ih_gemm_scaled_f16. */
int ih_conv2d_scaled_f16(const void* x, const void* w, const void* bias, const void* residual, void* out, int B, int Hin,
                         int Win, int Cin, int Cout, int stride, float alpha, void* stream);

/* 3x3 conv, stride 2, padding on the bottom and right only: conv(F.pad(x, (0, 1, 0, 1)), stride=2), input row
 * 2*oy + dy (the other stride-2 convs read 2*oy + dy - 1).  Replaces the VAE encoder's Downsample2D(padding=0)
 * ([3P] diffusers AutoencoderKL.encode, img2img).  Weight layout as ih_conv2d_f16; even H, W; Cin % 64 == 0.
 * out = conv(x) + bias: linear in the scaled residual stream, so the caller scales only the bias. */
int ih_conv2d_s2_padbr_f16(const void* x, const void* w, const void* bias, void* out, int B, int Hin, int Win, int Cin,
                           int Cout, void* stream);

/* Multi-head attention, head_dim 64, softmax scale 1/8, no mask.
 *   q: [B, Nq, *] rows with ldq elements per row, head h at columns [h*64, h*64+64) (same for k, v, out).
 *   Self attention (n_ip == 0): out = softmax(q k^T / 8) v over Nk keys.
 *   Decoupled IP cross attention (n_ip > 0): keys/values are the concatenation [text (Nk - n_ip) ; ip (n_ip)];
 *     out = softmax_text(q k_t^T/8) v_t + ip_scale * softmax_ip(q k_ip^T/8) v_ip   (two separate softmaxes).
 * Replaces F.scaled_dot_product_attention at attention_processor.py:312-314 (self), :423-425 (text branch),
 * :440-442 + :450 (IP branch and the scale*ip axpy).  Nk <= 128 uses the single-block path. */
int ih_attention_f16(const void* q, long long ldq, const void* k, long long ldk, const void* v, long long ldv,
                     void* out, long long ldo, int B, int H, int Nq, int Nk, int n_ip, float ip_scale,
                     void* stream);

/* ih_attention_f16 with a caller-owned scratch buffer (>= ih_attention_workspace_bytes(...) bytes, ZERO-FILLED once
 * by the caller; the kernels leave its arrival counters at zero).  With it the long self-attention shapes (Nk > 96,
 * n_ip == 0) cut the query tiles that would otherwise form a nearly empty last wave into KV parts that share one wave
 * and are merged by a second small kernel (flash-decoding style, fixed merge order: deterministic; IH_ATTN_FUSED_MERGE=1
 * merges inside the attention kernel instead, which measured slower).  workspace == NULL behaves like ih_attention_f16. */
long long ih_attention_workspace_bytes(int B, int H, int Nq, int Nk, int n_ip);
/* Fused front half of a cross-attention layer: out = CrossAttn(LayerNorm(h) Wq^T, k, v) for short key axes (Nk <= 96,
 * Nq % 128 == 0): the q projection (K input channels -> H*64) runs as a tcgen05 GEMM whose epilogue performs the
 * (decoupled) attention per head, so q never goes to HBM.  h: [B*Nq, K] raw rows; wq: [H*64, K]; bias: [H*64] or NULL;
 * ln_stats/ln_slabs/ln_eps as in ih_gemm_ln_f16 (NULL: no folded LayerNorm); k, v, n_ip, ip_scale, out as in
 * ih_attention_f16.  Replaces attention_processor.py:396 (to_q) + :423-425, :440-442, :450 (IPAttnProcessor2_0) and
 * :292, :312-314 (AttnProcessor2_0 with encoder_hidden_states). */
int ih_xattn_q_fused_f16(const void* h, long long ldh, const void* wq, const void* bias, const void* ln_stats,
                         int ln_slabs, float ln_eps, const void* k, long long ldk, const void* v, long long ldv,
                         void* out, long long ldo, int B, int H, int Nq, int Nk, int n_ip, float ip_scale, int K,
                         void* stream);

/* Test aid: 0 (default) = split only when the cost model predicts a gain, 1 = split whenever a plan exists. */
void ih_attention_set_split_policy(int policy);
/* Debug aid (effective only in builds with -DIH_ATTN_TRACE=1): CTA 0 of later ping-pong attention launches writes
 * clock64 stamps of KV blocks 4..7 into this device buffer (>= 192 int64: softmax thread of tile 0 at [0,64), of tile
 * 1 at [64,128)); NULL disables.  See tools/attn_trace.py and profiles/r1_attn_trace.md. */
void ih_attention_set_trace(void* device_buffer);
int ih_attention_ws_f16(const void* q, long long ldq, const void* k, long long ldk, const void* v, long long ldv,
                        void* out, long long ldo, int B, int H, int Nq, int Nk, int n_ip, float ip_scale,
                        void* workspace, long long workspace_bytes, void* stream);

/* GroupNorm over NHWC [B, HW, C] (optionally the channel-concatenation of two tensors x0 [.., C0] and x1 [.., C1]),
 * fp32 partial sums reduced in double, optional fused SiLU.  stats_ws: ih_groupnorm_workspace_bytes(B, groups) bytes,
 * zero-initialised ONCE by the caller (the kernels leave its ticket counters at zero again) and not shared by
 * concurrently running calls.  Replaces nn.GroupNorm (+ nn.SiLU) in diffusers ResnetBlock2D / Transformer2DModel. */
long long ih_groupnorm_workspace_bytes(int B, int groups);
int ih_groupnorm_f16(const void* x0, int C0, const void* x1, int C1, const void* gamma, const void* beta, void* out,
                     void* stats_ws, int B, int HW, int groups, float eps, int silu, void* stream);

/* LayerNorm over the last dim of [rows, C], fp32 statistics. Replaces nn.LayerNorm in BasicTransformerBlock. */
int ih_layernorm_f16(const void* x, const void* gamma, const void* beta, void* out, int rows, int C, float eps,
                     void* stream);

/* Small-M linear (M <= 64 rows): out[m, n] = act_out(W[n,:] . act_in(x[m,:]) + b[n]) * out_scale + addend[m, n];
 * act: 0 none, 1 SiLU.
 * Time / added-condition embeddings and the 17 time_emb_proj layers (diffusers), ImageProjModel / HarmonyAttention
 * linears (ip_adapter.py:41-48, train.py:243-266). */
int ih_linear_small_f16(const void* x, long long ldx, const void* w, const void* bias, const void* addend,
                        long long ld_add, void* out, long long ldo, int M, int N, int K, int act_in, int act_out,
                        float out_scale, void* stream);

/* Small generic attention on CUDA cores: out = softmax(q k^T / scale) v, head dims dqk / dv <= 128, Nk <= 1024,
 * B*H*Nq a multiple of 4.  HarmonyAttention's Cross_Attention (attention_processor.py:35-56; head_dim 40, v_dim 64,
 * scale = sqrt(40) is a divisor as in the reference), once per generate(). */
int ih_attention_small_f16(const void* q, long long ldq, const void* k, long long ldk, const void* v, long long ldv,
                           void* out, long long ldo, int B, int H, int Nq, int Nk, int dqk, int dv, float scale,
                           void* stream);

/* Sinusoidal embedding (flip_sin_to_cos, shift 0): out[i, :] = [cos(t_i f), sin(t_i f)], f = 10000^(-j/half). t fp32.
 * step_i32 == NULL: t_i = t_f32[i]; else every row uses t_f32[*step_i32] (device-resident step counter, so the
 * timestep of custom_pipelines.py:325 can live inside a replayed CUDA graph). */
int ih_sinusoid_f16(const void* t_f32, const void* step_i32, void* out, long long ldo, int n, int dim, void* stream);

/* out[i] = a[i] + b[i % period]: residual / positional-embedding adds of the Resampler (resampler.py:128-131,143-144). */
int ih_add_bcast_f16(const void* a, const void* b, void* out, long long n, long long period, void* stream);
/* out[b, :] = mean_n x[b, n, :]  -- Resampler masked_mean with an all-ones mask (resampler.py:137-138,150-158). */
int ih_mean_tokens_f16(const void* x, void* out, int B, int n, int D, void* stream);

/* In-place row softmax of an fp16 matrix [rows, cols] (row stride ld elements, fp32 statistics), cols <= 32768.  With
 * two ih_gemm_f16 calls it forms the single-head, head_dim-512 attention of the VAE decoder mid block
 * ([3P] diffusers AutoencoderKL, called at custom_pipelines.py:373). */
int ih_softmax_rows_f16(void* x, long long ld, long long rows, int cols, void* stream);
/* same, with only the first valid_cols columns of every row taking part; the padding columns are written as 0. */
int ih_softmax_rows_masked_f16(void* x, long long ld, long long rows, int cols, int valid_cols, void* stream);

/* Nearest-neighbour 2x upsample NHWC [B,H,W,C] -> [B,2H,2W,C]. */
int ih_upsample2x_f16(const void* x, void* out, int B, int H, int W, int C, void* stream);

/* Channel concat of two NHWC tensors: out[.., :C0] = x0, out[.., C0:] = x1. rows = B*H*W. */
int ih_concat_f16(const void* x0, int C0, const void* x1, int C1, void* out, long long rows, void* stream);

/* conv_in: NCHW latent [B,4,H,W] -> NHWC [B,H,W,Cout], 3x3 pad 1 (weight OIHW [Cout,4,3,3]). */
int ih_conv_in_f16(const void* x_nchw, const void* w, const void* bias, void* out, int B, int H, int W, int Cin,
                   int Cout, void* stream);
/* conv_out: NHWC [B,H,W,Cin] -> NCHW [B,Cout,H,W], 3x3 pad 1 (weight OIHW [Cout,Cin,3,3]), Cout <= 8. */
int ih_conv_out_f16(const void* x, const void* w, const void* bias, void* out_nchw, int B, int H, int W, int Cin,
                    int Cout, void* stream);

/* conv_in on the tensor-core GEMM: im2col of the NCHW latent into A [B*H*W, Kpad] (k = ci*9 + ky*3 + kx, zero padded),
 * to be multiplied with the OIHW weight flattened (and zero padded) to [Cout, Kpad] by ih_gemm_f16. */
int ih_im2col3x3_nchw_f16(const void* x_nchw, void* out, int B, int Cin, int H, int W, int Kpad, void* stream);
/* VAE encoder conv_in on the tensor-core GEMM, straight from the PIL pixels: uint8 RGB NHWC [B,H,W,3] -> im2col rows
 * [B*H*W, Kpad] (k = ci*9 + ky*3 + kx, zero padding 1, K padding zero) of fp16(2 * (v / 255) - 1), the fp32 rounding
 * points of [3P] diffusers VaeImageProcessor (pil_to_numpy, normalize).  Kpad % 8 == 0, Kpad >= 27. */
int ih_image_im2col3x3_u8(const void* rgb_u8, void* out, int B, int H, int W, int Kpad, void* stream);
/* img2img initial latents from the encoder's moments (NHWC [Bm, h, w, ldm]: mean in channels [0, C), logvar in [C, 2C)):
 *   z = fp16(sf * fp16(mean + exp(0.5 clamp(logvar, -30, 20)) * eps))   ([3P] DiagonalGaussianDistribution.sample in fp32,
 *       cast, `scaling_factor * latents` in fp16);  eps == NULL: z = mean (latents passed as they are, Be ignored);
 *   out = fp16(z + fp16(noise * fp16(sigma)))   ([3P] EulerDiscreteScheduler.add_noise on fp16 tensors).
 * eps fp32 NCHW [Be, C, h, w], noise fp16 NCHW [B, C, h, w], out fp16 NCHW [B, C, h, w]; output image b reads moments
 * b % Bm and eps b % Be. */
int ih_vae_sample_add_noise_f16(const void* moments, long long ldm, int Bm, const void* eps_f32, int Be, const void* noise,
                                void* out_nchw, int B, int C, int h, int w, float scaling_factor, float sigma,
                                void* stream);
/* Inpainting start latents: as ih_vae_sample_add_noise_f16, and z0_nchw receives z (fp16 NCHW [B, C, h, w], the
 * blend's clean latents).  pure_noise = 1 (strength 1): latents = fp16(noise * sigma), sigma = init_noise_sigma, not
 * rounded to fp16. */
int ih_vae_sample_inpaint_f16(const void* moments, long long ldm, int Bm, const void* eps_f32, int Be, const void* noise,
                              void* latents_nchw, void* z0_nchw, int B, int C, int h, int w, float scaling_factor,
                              float sigma, int pure_noise, void* stream);
/* Inpainting latent mask: uint8 grayscale [Bm, H, W] (H, W multiples of 8) -> uint8 {0, 1} [Bm, H/8, W/8], latent
 * (y, x) = pixel (8y, 8x) >= 128 ([3P] VaeImageProcessor binarize at 0.5, then F.interpolate nearest). */
int ih_latent_mask_u8(const void* mask_u8, void* out_u8, int Bm, int H, int W, void* stream);
/* conv_out on ih_conv2d_f16 with Cout padded to 16: gather NHWC [B, HW, ldc] channels [0, C) into NCHW [B, C, HW]. */
int ih_nhwc_to_nchw_f16(const void* x, long long ldc, void* out, int B, long long HW, int C, void* stream);

/* One scheduler transition (custom_pipelines.py:332-334,348-357):
 *   eps = u + g (c - u)  (fp16 tensor arithmetic, rounded like the reference's);
 *   x <- fp16( x + ((x - (x - sigma_i eps)) / sigma_i) (sigma_{i+1} - sigma_i) )   (fp32 inside, Euler, [3P] diffusers);
 *   model_in <- cat([x, x]) / sqrt(sigma_{i+1}^2 + 1)  (next step's scaled CFG input); step counter i += 1.
 * noise_pred: [2n,4,H,W] fp16 (uncond half first), latents: [n,4,H,W] fp16, model_in: [2n,4,H,W] fp16.
 * sigmas: device fp32 [T+1]; step: device int32 (read, then incremented). n_per_image = 4*H*W. */
int ih_euler_cfg_step(const void* noise_pred, void* latents, void* model_in, const void* sigmas, void* step,
                      float guidance, long long n_per_image, int n_images, void* stream);

/* ---- scope row f2: conditioning encoders (CLIP towers the reference loads at ip_adapter.py:81-84 and calls at
 * :163-164 (image) and through encode_prompt :292-319 (text)); arithmetic = [3P] transformers CLIPEncoderLayer. ---- */

/* softmax(q k^T * scale (+ causal mask)) v, any head dims that are multiples of 8 (<= 256), fp32 softmax.
 * q [B*Nq, >= H*dqk], k [B*Nk, >= H*dqk], v [B*Nk, >= H*dv], out [B*Nq, >= H*dv]; causal: key j visible iff j <= i.
 * Replaces CLIPAttention (text: causal, head_dim 64; ViT-bigG vision: head_dim 104). */
int ih_attention_generic_f16(const void* q, long long ldq, const void* k, long long ldk, const void* v, long long ldv,
                             void* out, long long ldo, int B, int H, int Nq, int Nk, int dqk, int dv, float scale,
                             int causal, void* stream);

/* out[r, :] = tok_emb[ids[r], :] + pos_emb[r % T, :]   (CLIPTextEmbeddings); ids int32 device [rows]. */
int ih_embed_tokens_f16(const void* ids_i32, const void* tok_emb, const void* pos_emb, void* out, int rows, int T, int C,
                        int vocab, void* stream);

/* PNS judge front end: image NCHW fp16 in [-1, 1] (VAE output) -> area-averaged S x S -> [0, 1] -> CLIP mean / std
 * normalisation -> patch rows [B*(S/P)^2, Kpad], k = c*P*P + py*P + px (flattened patch_embedding conv weight layout).
 * mean3 / std3: HOST pointers to 3 floats. */
int ih_resize_patchify_f16(const void* img_nchw, void* out, int B, int C, int Hin, int Win, int S, int P, int Kpad,
                           const float* mean3, const float* std3, void* stream);

/* General scheduler transition: the loop options the reference accepts beyond the default CFG path.
 *   use_cfg = 0 : guidance_scale <= 1 (custom_pipelines.py:223 do_classifier_free_guidance False): noise_pred and
 *                 model_in are [n,4,H,W]; eps = noise_pred (:332,:348 skipped).
 *   guidance_rescale > 0 (:352-354, [3P] diffusers rescale_noise_cfg): eps <- r * eps * (std(c) / std(eps)) + (1 - r) * eps
 *                 with the per-image unbiased std over all non-batch elements, fp16 rounding points of the fp16 tensors.
 * Otherwise identical to ih_euler_cfg_step (which stays the fast path for the default call). */
int ih_euler_step_ex(const void* noise_pred, void* latents, void* model_in, const void* sigmas, void* step,
                     float guidance, float guidance_rescale, long long n_per_image, int n_images, int use_cfg,
                     void* stream);

/* Masked (inpainting) scheduler transition ([3P] diffusers StableDiffusionXLInpaintPipeline, 4-channel UNet): the
 * transition of ih_euler_cfg_step (use_cfg && guidance_rescale == 0) or ih_euler_step_ex (otherwise), then, with k the
 * step index read from `step`, before model_in is formed:
 *   proper  = z0 if k == *last_step, else fp16(z0 + fp16(noise * fp16(sigma_{k+1})))   (add_noise at the next sigma);
 *   latents = fp16(fp16(fp16(1 - m) * proper) + fp16(m * latents)).
 * mask_u8: uint8 {0, 1} [Bm, hw] (1 = regenerate), latent image b uses mask b % Bm; z0, noise: fp16 NCHW, the latents'
 * shape; last_step: device int32, the index of the last executed step.  Launches as many kernels as the plain step. */
int ih_euler_step_inpaint(const void* noise_pred, void* latents, void* model_in, const void* sigmas, void* step,
                          float guidance, float guidance_rescale, long long n_per_image, int n_images, int use_cfg,
                          const void* mask_u8, int Bm, long long hw, const void* z0, const void* noise,
                          const void* last_step, void* stream);

/* model_in = cat([latents, latents]) / sqrt(sigma[*step]^2 + 1)   (custom_pipelines.py:332-334, first step). */
int ih_scale_model_input(const void* latents, void* model_in, const void* sigmas, const void* step, long long total,
                         void* stream);
/* same with duplicate = 0: model_in = latents / sqrt(...) for the no-CFG loop (custom_pipelines.py:332 else-branch). */
int ih_scale_model_input_ex(const void* latents, void* model_in, const void* sigmas, const void* step, long long total,
                            int duplicate, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* IH_API_H */
