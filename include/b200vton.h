/* libb200vton.so — C ABI of the Blackwell-native IDM-VTON denoising engine.
 *
 * The reference (yisol/IDM-VTON) has no C/FFI plugin API; its seams are Python protocols (SURVEY.md 8b: pipeline
 * __call__, UNet2DConditionModel.forward, the diffusers attention-processor protocol). This header is the boundary the
 * Python host (idm-vton_b200/*.py, loaded with ctypes) binds instead of the ATen/cuDNN/cuBLAS/SDPA library calls the
 * reference issues. Every entry point cites the reference call site it replaces.
 *
 * Conventions
 *   - all pointers are DEVICE pointers to fp16 data unless stated; the caller (PyTorch) owns every buffer;
 *     the library never allocates or frees device memory;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream); launches are asynchronous and may be
 *     captured into a CUDA graph;
 *   - return value 0 = success, non-zero = error (1 invalid argument, 2 CUDA error, 3 unsupported shape);
 *     b200vton_last_error() returns the message for the calling thread. There is no CPU fallback.
 *   - activations are NHWC / token-major: a feature map [B,H,W,C] and a token matrix [B*H*W, C] are the same memory.
 */
#ifndef B200VTON_H_
#define B200VTON_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

int b200vton_version(void);
const char* b200vton_last_error(void);
/* kernels launched (or recorded into a capturing stream) by this library since it was loaded */
long long b200vton_launch_count(void);
/* library options: "gemm_2cta_auto" = 1 (default) lets gemm / conv3x3 pick the 2-CTA persistent kernel for large
 * problems when force_bn == 0; 0 keeps every launch on the 1-CTA kernel. "attention_pingpong" = 1 (default) runs
 * b200vton_attention on the pipelined kernel (attn6.cu: S issued one tile ahead, P in tensor memory) when Nq >= 256;
 * 0 keeps the one-tile kernel (attn.cu), which the tests use as an independent cross-check.
 * ("attention_q_tiles" = 1 | 2 pins the pipelined kernel's query tiles per CTA, 0 = chosen from the K/V length;
 * "attention_poly_exp" = 0 | 1 | 2 of every 4 exponentials evaluated by an FMA-pipe polynomial instead of the SFU,
 * default 0: measured slower).
 * "gemm_cluster4" = 1 runs large linear layers with 256-wide tiles in four-CTA clusters whose CTA pairs multicast the
 * shared A slabs; 0 (default: it measured slower on B200) keeps two-CTA clusters.
 * "programmatic_launch" = 1 launches the hot kernels with programmatic stream serialization (their set-up overlaps
 * the previous kernel's tail; they wait for it before allocating tensor memory or touching global memory);
 * 0 (default) = plain stream order. */
int b200vton_set_option(const char* name, int value);

/* out[M,N] = epi(A[M,K] . W[N,K]^T): nn.Linear on the hot path — attn to_q/to_k/to_v/to_out
 * (ip_adapter/attention_processor.py:240-268), Transformer2DModel.proj_in/proj_out
 * (src/transformerhacked_tryon.py:331-345,410-427), FeedForward GEGLU / net.2 (src/attentionhacked_tryon.py:621-679).
 * epi: v = fp16(acc + bias[n]); v = fp16(v + rowvec[m / rows_per_sample, n]); v = fp16(v + residual[m, n]).
 * flags & 1 (GEGLU): W/bias rows are tile-interleaved [value | gate] (see engine.pack_geglu) and
 *             out[M, N/2] = fp16(value) * fp16(gelu_erf(fp16(gate))).
 * flags & 2 (GELU): v = fp16(gelu_erf(fp16(acc + bias))) before the rowvec / residual terms (ip_adapter/resampler.py:13-20;
 *             the CLIP ViT-H / bigG MLPs). flags & 4 (quick-GELU): v = fp16(x * sigmoid(1.702 x)), x = fp16(acc + bias)
 *             (the CLIP ViT-L text encoder's MLP, src/tryon_pipeline.py:592).
 * K % 64 == 0; N, lda, ldw, ldo % 8 == 0. force_bn: 0 = automatic kernel and tile width; 64/128/160/256 = 1-CTA
 * kernel with that tile width; 1000 + {128,160,192,256} = 2-CTA persistent kernel (cta_group::2) with that width. */
int b200vton_gemm_f16(const void* A, int64_t lda, const void* W, int64_t ldw, void* out, int64_t ldo, int M, int N,
                      int K, const void* bias, const void* residual, int64_t ldr, const void* rowvec,
                      int64_t ld_rowvec, int rows_per_sample, int flags, int force_bn, void* stream);

/* NHWC 3x3 convolution, pad 1, stride 1 or 2, as implicit GEMM: diffusers ResnetBlock2D.conv1/conv2 (+conv_shortcut),
 * conv_in / conv_out (src/unet_hacked_tryon.py:416,755,1245,1386), the conv of Upsample2D, and (stride 2) the conv of
 * Downsample2D (src/unet_block_hacked_tryon.py:1113,1246): the A operand's tensor map then steps two input pixels per
 * output pixel (TMA traversal stride), so no im2col buffer exists.
 * x: [B,H,W,Cin] with channel stride ldx; w: [9][Cout][Cin] (tap = ky*3+kx); out: [B*Ho*Wo, ldo], Ho = (H-1)/stride+1.
 * epi: v = fp16(acc + bias); v = fp16(v + temb[b, n]) (time_emb_proj broadcast add);
 *      1x1 shortcut (w_sc [Cout, C0+C1] over the channel concat of sc0|sc1, accumulated in a second TMEM tile):
 *      s = fp16(acc_sc + bias_sc); v = fp16(s + v);   identity residual: v = fp16(v + residual[m, n]). */
int b200vton_conv3x3_nhwc(const void* x, int64_t ldx, int B, int H, int W, int Cin, const void* w, int Cout,
                          const void* bias, const void* temb, int64_t ld_temb, const void* sc0, int C0,
                          const void* sc1, int C1, const void* w_sc, const void* bias_sc, const void* residual,
                          int64_t ldr, void* out, int64_t ldo, int force_bn, int stride, void* stream);

/* softmax(Q K^T * scale) V, head_dim 64, keys/values streamed from two segments without concatenation:
 * segment 0 = (k0, v0)[b]; segment 1 = (k1, v1)[base + (b - kv1_off) % mod] for b >= kv1_off, where mod = kv1_mod
 * (or B1 when kv1_mod == 0) and base = *kv1_base (a device int32, or 0 when NULL: lets one captured graph walk the
 * per-timestep slices of garment K/V precomputed for all denoise steps); for b < kv1_off the N1
 * tokens are all-zero K/V handled in closed form (CFG-uncond half, src/tryon_pipeline.py:1796).
 * Replaces cat + F.scaled_dot_product_attention of src/attentionhacked_tryon.py:334-348 /
 * ip_adapter/attention_processor.py:238-262 (attn1) and :1970-1995 (attn2: call once for the 77 text tokens, once for
 * the 16 IP tokens with accumulate = 1: out = fp16(out + fp16(result))). Also PerceiverAttention
 * (ip_adapter/resampler.py:49-78; segment 0 = image tokens, segment 1 = latents).
 * q: [B,Nq,*] row stride ldq, head h at columns [64h, 64h+64); same for k/v/out. */
int b200vton_attention(const void* q, int64_t ldq, const void* k0, const void* v0, int64_t ldkv0, const void* k1,
                       const void* v1, int64_t ldkv1, void* out, int64_t ldo, int B, int H, int Nq, int N0, int N1,
                       int B1, int kv1_off, int kv1_mod, const void* kv1_base, float scale, int accumulate,
                       void* stream);

/* Decoupled cross-attention (attn2 of every transformer block) in one launch:
 *   out = fp16( fp16(softmax(Q Kt^T * scale) Vt) + fp16(ip_scale * fp16(softmax(Q Ki^T * scale) Vi)) ),  head_dim 64,
 * Kt/Vt = [B, Nt <= 80, *] the text tokens (attn2.to_k / to_v), Ki/Vi = [B, Ni <= 16, *] the IP-Adapter image tokens
 * (processor to_k_ip / to_v_ip); Ni = 0 (ki = vi = NULL) is the plain text cross-attention of the garment UNet.
 * Replaces IPAttnProcessor2_0.__call__ (ip_adapter/attention_processor.py: two scaled_dot_product_attention calls and
 * hidden_states + self.scale * ip_hidden_states), called as attn2 at src/attentionhacked_tryon.py:368-380, and
 * AttnProcessor2_0 at src/attentionhacked_garmnet.py:371-383. Same result as two b200vton_attention calls
 * (the second with accumulate = 1), one kernel instead of two. Layouts as b200vton_attention. */
int b200vton_cross_attention(const void* q, int64_t ldq, const void* kt, const void* vt, int64_t ldkv_t, int Nt,
                             const void* ki, const void* vi, int64_t ldkv_i, int Ni, void* out, int64_t ldo, int B,
                             int H, int Nq, float scale, float ip_scale, void* stream);

/* fp32 3x3 convolution, stride 1, zero padding 1, on the TF32 tensor cores (TF32 products, fp32 accumulate, fp32 bias,
 * fp32 out — the arithmetic class PyTorch uses for fp32 cuDNN convolutions by default): the VAE's convolutions
 * (diffusers AutoencoderKL ResnetBlock2D.conv1/conv2, Upsample2D.conv; the reference runs the SDXL VAE in fp32,
 * src/tryon_pipeline.py:913-915,1076-1093). x: [B,H,W,Cin] dense NHWC (= channels_last memory), w: [9][Cout][Cin]
 * (tap-major), bias: [Cout] or NULL, residual: [B,H,W,Cout] fp32 NHWC or NULL — out = (acc + bias) + residual, the
 * ResnetBlock2D's `input_tensor + hidden_states` in the epilogue with torch's rounding; out: [B,H,W,Cout].
 * Cin, Cout multiples of 32, Cout >= 64, W divisible by 8. */
int b200vton_conv3x3_nhwc_f32(const void* x, int B, int H, int W, int Cin, const void* w, int Cout, const void* bias,
                               const void* residual, void* out, void* stream);

/* The same convolution with fp16 operands: x [B,H,W,Cin] fp16 NHWC (the fp16 output of b200vton_groupnorm_nhwc_f32), w
 * [9][Cout][Cin] fp16; fp32 accumulation, fp32 bias / residual / out. An fp16 operand carries the 10-bit mantissa the TF32
 * tensor core rounds an fp32 operand to (and GroupNorm(+SiLU) outputs are far inside fp16's range), so the arithmetic class is
 * that of the TF32 convolution at half the operand traffic and twice the MMA rate. Cin a multiple of 64. */
int b200vton_conv3x3_nhwc_f16in_f32(const void* x, int B, int H, int W, int Cin, const void* w, int Cout, const void* bias,
                                    const void* residual, void* out, void* stream);

/* Split operands for fp32-accurate products on the TF32 tensor cores (the VAE mid-block attention, diffusers AutoencoderKL
 * mid_block.attentions[0], exact fp32 in the reference: src/tryon_pipeline.py:913-915,1076-1093):
 * hi = tf32(x * scale), lo = tf32(x * scale - hi), both exactly representable in TF32 (10 mantissa bits, round half up).
 * x: B blocks of per_batch contiguous floats with batch stride stride_b (elements); hi / lo: dense [B, per_batch]. */
int b200vton_split_tf32(const void* x, int64_t stride_b, int B, int64_t per_batch, float scale, void* hi, void* lo,
                        void* stream);
/* Row softmax of fp32 scores [rows, N] (max-subtracted, expf, fp32 sum) written directly as the two TF32 parts of the
 * probabilities: p_hi = tf32(p), p_lo = tf32(p - p_hi); the fp32 probabilities themselves are never stored. N % 4 == 0. */
int b200vton_softmax_split_tf32(const void* scores, int64_t rows, int N, void* p_hi, void* p_lo, void* stream);

/* fp32 GroupNorm(32 groups)(+SiLU) over dense NHWC [B,HW,C] fp32 — the VAE's norms (diffusers AutoencoderKL
 * ResnetBlock2D.norm1/norm2 + SiLU, Attention.group_norm, conv_norm_out), deterministic two-stage statistics.
 * gamma/beta: [C] fp32 or NULL. stats_ws: scratch of stats_ws_doubles doubles, at least 64 * max(B, 1184) is always
 * enough. out: fp32, or — out_fp16 != 0 — fp16 of the same shape (one rounding of the fp32 result), the operand format of
 * b200vton_conv3x3_nhwc_f16in_f32. The VAE's default route (B200VTON_VAE_NHWC=0 restores the cuDNN NCHW path). */
int b200vton_groupnorm_nhwc_f32(const void* x, int B, int HW, int C, const void* gamma, const void* beta, float eps,
                                 int silu, void* stats_ws, int64_t stats_ws_doubles, void* out, int out_fp16, void* stream);

/* GroupNorm(32 groups) over NHWC [B,HW,C0+C1] read from up to two channel-concatenated sources (x1 may be NULL),
 * fp32 statistics (deterministic fixed-order reduction, no atomics on data), optional SiLU, fp16 out [B*HW, C0+C1].
 * ONE launch: statistics, a per-sample barrier between the CTAs of the launch, and the normalisation (the rows stay in
 * shared memory in between when they fit, so the tensor is read once). B <= 4096.
 * stats_ws: (max(B,296)*64 + 4096) doubles; the last 4096 doubles hold the barrier state and must be ZERO before the
 * first call that uses this workspace (the kernel leaves them reusable: no clearing between calls / graph replays).
 * One workspace must not be shared by launches that may run concurrently (different streams); more generally two
 * GroupNorm launches must not run CONCURRENTLY on one device (two streams, two processes): each sizes its grid to be
 * fully co-resident on an otherwise free device, and two half-resident grids would wait for each other at their
 * barriers (the spin is bounded: the kernel traps after 4 s instead of hanging). The engine launches everything on one
 * stream, like the reference pipeline.
 * diffusers ResnetBlock2D.norm1/norm2 (+nonlinearity), Transformer2DModel.norm
 * (src/transformerhacked_tryon.py:329), conv_norm_out + conv_act (src/unet_hacked_tryon.py:1384-1385). */
int b200vton_groupnorm(const void* x0, int C0, const void* x1, int C1, int B, int HW, const void* gamma,
                       const void* beta, float eps, int silu, void* stats_ws, void* out, void* stream);

/* LayerNorm over the last dim of [rows, C]: BasicTransformerBlock.norm1/2/3
 * (src/attentionhacked_tryon.py:310,365,390); the garment UNet's norm1 output is the exported garment feature
 * (src/attentionhacked_garmnet.py:321-322). */
int b200vton_layernorm(const void* x, int64_t ldx, int rows, int C, const void* gamma, const void* beta, float eps,
                       void* out, int64_t ldo, void* stream);

/* dst[s,y,x,c_off+c] = src[s % Bs, c, y, x]: NCHW module inputs -> NHWC engine buffer; implements the CFG
 * duplication and the 13-channel concat of src/tryon_pipeline.py:1769,1777 as batch/channel offsets. */
int b200vton_nchw_to_nhwc(const void* src, int Bs, int Cs, int H, int W, void* dst, int Bd, int ldc, int c_off,
                          void* stream);
/* dst NCHW [B,C,H,W] = src NHWC [B,H,W,ldc][..., :C] */
int b200vton_nhwc_to_nchw(const void* src, int B, int C, int H, int W, int ldc, void* dst, void* stream);
/* b200vton_nchw_to_nhwc with every value multiplied by *scale (one fp32 on the device), rounded once to fp16: the
 * latent scatter fused with `scheduler.scale_model_input` (sample / sqrt(sigma^2 + 1) of the Euler schedulers,
 * src/tryon_pipeline.py:1772). */
int b200vton_nchw_to_nhwc_scaled(const void* src, int Bs, int Cs, int H, int W, const void* scale, void* dst, int Bd,
                                 int ldc, int c_off, void* stream);

/* nearest-neighbour x2 (diffusers Upsample2D's F.interpolate), NHWC */
int b200vton_upsample2x_nhwc(const void* src, int B, int H, int W, int C, void* dst, void* stream);
/* patches of a 3x3 stride-2 pad-1 conv (diffusers Downsample2D) as A[B*Ho*Wo, 9*C], K ordered tap-major */
int b200vton_im2col3x3_s2_nhwc(const void* src, int B, int H, int W, int C, void* dst, void* stream);

/* diffusers Timesteps(dim, flip_sin_to_cos=True, freq_shift=0): out[r, :] = [cos | sin](values[r % n] * freq),
 * values: n fp32 on device; out: [n * rows_repeat, dim] fp16 (src/unet_hacked_tryon.py:1134-1139,1185). */
int b200vton_timestep_embedding(const void* values, int n, int dim, int rows_repeat, void* out, void* stream);

/* y = W x + b for M <= 16 rows (TimestepEmbedding, add_embedding, batched ResnetBlock2D.time_emb_proj):
 * x' = in_silu ? fp16(silu(x)) : x; y = fp16(W x' + b); y = out_silu ? fp16(silu(y)) : y; y = fp16(y + addend). */
int b200vton_skinny_linear(const void* x, int ldx, int M, int K, const void* W, int64_t ldw, int N, const void* bias,
                           int in_silu, int out_silu, const void* addend, int ld_add, void* out, int ldo,
                           void* stream);

/* Encoder self-attention for the CLIP towers around the loop (SURVEY.md 8f row 2): replaces transformers' CLIPAttention
 * inside `self.image_encoder(image, output_hidden_states=True)` (src/tryon_pipeline.py:468-470: ViT-H, 16 heads of 80,
 * 257 tokens, no mask) and inside `text_encoder(text_input_ids, output_hidden_states=True)` (src/tryon_pipeline.py:592-596:
 * heads of 64, 77 tokens, causal mask). q / k / v: [B, N, >= H*D] views with row strides ldq / ldkv (the three column
 * blocks of a fused QKV projection buffer); out: [B, N, H*D], row stride ldo. D = 16..96, multiple of 16.
 * out = softmax(scale * q k^T [+ causal mask]) v per head, fp32 softmax, fp16 probabilities, fp32 accumulation. */
int b200vton_encoder_attention(const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv, void* out,
                               int64_t ldo, int B, int H, int N, int D, float scale, int causal, void* stream);

/* CLIPVisionEmbeddings.patch_embedding as a GEMM operand (src/tryon_pipeline.py:468): x [B,C,Hi,Wi] fp16 ->
 * out [B*(Hi/P)*(Wi/P), ldk] fp16, row = (b, gy, gx), column = (c, ky, kx) = the flattened conv weight's K order;
 * columns >= C*P*P are written as zeros (ldk = K rounded up to a multiple of 64 for b200vton_gemm_f16). */
int b200vton_patchify(const void* x, int B, int C, int Hi, int Wi, int P, void* out, int ldk, void* stream);

/* CLIPTextEmbeddings (src/tryon_pipeline.py:592): out[r, :] = fp16(token_embedding[ids[r], :] + position_embedding[r % T, :]);
 * ids: int64 [rows] on the device (clamped to [0, vocab)); C % 8 == 0. */
int b200vton_token_embedding(const void* ids, int rows, int T, int C, int vocab, const void* token_embedding,
                             const void* position_embedding, void* out, void* stream);

/* CFG combine + DDPMScheduler.step (src/tryon_pipeline.py:1814-1823). eps NHWC [2B,HW,ldc] (uncond first) or [B,..]
 * when do_cfg == 0; latents/noise/out NCHW [B,C,H,W] (noise may be NULL); coef: 6 fp32 on device
 * {guidance_scale, sqrt(1-abar_t), 1/sqrt(abar_t), x0 coeff, x_t coeff, sigma_t}. */
int b200vton_cfg_ddpm_step(const void* eps, int ldc, int B, int C, int H, int W, const void* latents,
                           const void* noise, const void* coef, int do_cfg, void* out, void* stream);

/* CFG combine + the update of another scheduler (the pipeline's `scheduler.step` at src/tryon_pipeline.py:1823 with
 * DDIMScheduler, EulerDiscreteScheduler, EulerAncestralDiscreteScheduler or DPMSolverMultistepScheduler in its place).
 * family: 0 DDIM, 1 Euler, 2 Euler-ancestral, 3 DPM-Solver++ (orders 1 and 2). Layouts as b200vton_cfg_ddpm_step;
 * coef: 8 fp32 on device {guidance_scale, 6 per-family step scalars, model-input scale} (rounding points and row layout in
 * csrc/sched.cu). noise: [B,C,H,W] or NULL (required by family 2; DDIM adds it only when its std coefficient is
 * non-zero; ignored by families 1 and 3). hist: [B,C,H,W] fp16, the previous step's x0 prediction, read and then
 * overwritten in place (required by family 3, ignored otherwise). */
int b200vton_cfg_sched_step(const void* eps, int ldc, int B, int C, int H, int W, const void* latents,
                            const void* noise, void* hist, const void* coef, int family, int do_cfg, void* out,
                            void* stream);

/* Pre-processing of the inpainting inputs in one launch (diffusers VaeImageProcessor.preprocess for image and mask,
 * the masked image and the latent-resolution mask: src/tryon_pipeline.py:1588-1602, 940-943). image: [B,3,H,W] fp32;
 * mask: [B,mask_channels,H,W] fp32 (1, or 3 = RGB converted to grayscale); image_min: device scalar = min(image)
 * (values already in [-1,1], i.e. min < 0, are not normalised again — diffusers' rule, decided on the device);
 * outputs: init_image, masked_image [B,3,H,W] fp32, mask_bin [B,1,H,W] fp32 (0/1 at threshold 0.5),
 * mask_latent [B,1,H/vae_scale,W/vae_scale] fp16 (nearest). */
int b200vton_preprocess_inpaint(const void* image, const void* mask, int mask_channels, const void* image_min, int B,
                                int H, int W, int vae_scale, void* init_image, void* mask_bin, void* masked_image,
                                void* mask_latent, void* stream);

/* Post-processing of the VAE decoder output in one launch (VaeImageProcessor.postprocess, src/tryon_pipeline.py:1885):
 * x [B,3,H,W] fp32 in NCHW memory (nhwc = 0) or NHWC memory (nhwc = 1) -> clamp(x/2 + 0.5, 0, 1) written as fp32 NCHW
 * (out_pt, may be NULL) and/or uint8 NHWC round(255 y) (out_u8, may be NULL; what "np"/"pil" produce, 4x less D2H). */
int b200vton_postprocess_image(const void* x, int nhwc, int B, int H, int W, void* out_pt, void* out_u8, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200VTON_H_ */
