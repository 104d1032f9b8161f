// extern "C" surface of libb200vton.so (declared in include/b200vton.h). Thin forwarding only.
#include "../../include/b200vton.h"

#include "host.h"

namespace vton {
int gemm_f16_impl(const void* A, long long lda, const void* W, long long ldw, void* out, long long ldo, int M, int N,
                  int K, const void* bias, const void* residual, long long ldr, const void* rowvec, long long ld_rowvec,
                  int rows_per_sample, int flags, int force_bn, cudaStream_t stream);
int conv3x3_impl(const void* x, long long ldx, int B, int H, int W, int Cin, const void* w, int Cout, const void* bias,
                 const void* temb, long long ld_temb, const void* sc0, int C0, const void* sc1, int C1, const void* w_sc,
                 const void* bias_sc, const void* residual, long long ldr, void* out, long long ldo, int force_bn,
                 int stride, cudaStream_t stream);
int conv3x3_f32_impl(const void* x, int B, int H, int W, int Cin, const void* w, int Cout, const void* bias,
                     const void* residual, void* out, int in_fp16, cudaStream_t stream);
int split_tf32_impl(const void* x, long long stride_b, int B, long long per_batch, float scale, void* hi, void* lo,
                    cudaStream_t stream);
int softmax_split_tf32_impl(const void* s, long long rows, int N, void* phi, void* plo, cudaStream_t stream);
int groupnorm_f32_impl(const void* x, int B, int HW, int C, const void* gamma, const void* beta, float eps, int silu,
                       void* stats_ws, long long stats_ws_doubles, void* out, int out_fp16, cudaStream_t stream);
int cross_attn_impl(const void* q, long long ldq, const void* kt, const void* vt, long long ldkv_t, int Nt,
                    const void* ki, const void* vi, long long ldkv_i, int Ni, void* out, long long ldo, int B, int H,
                    int Nq, float scale, float ip_scale, cudaStream_t stream);
int attn_impl(const void* q, long long ldq, const void* k0, const void* v0, long long ldkv0, const void* k1,
              const void* v1, long long ldkv1, void* out, long long ldo, int B, int H, int Nq, int N0, int N1, int B1,
              int kv1_off, int kv1_mod, const void* kv1_base, float scale, int accumulate, cudaStream_t stream);
int groupnorm_impl(const void* x0, int C0, const void* x1, int C1, int B, int HW, const void* gamma, const void* beta,
                   float eps, int silu, void* stats_ws, void* out, cudaStream_t stream);
int layernorm_impl(const void* x, long long ldx, int rows, int C, const void* gamma, const void* beta, float eps,
                   void* out, long long ldo, cudaStream_t stream);
int nchw_to_nhwc_impl(const void* src, int Bs, int Cs, int H, int W, void* dst, int Bd, int ldc, int c_off,
                      cudaStream_t stream);
int nhwc_to_nchw_impl(const void* src, int B, int C, int H, int W, int ldc, void* dst, cudaStream_t stream);
int upsample2x_impl(const void* src, int B, int H, int W, int C, void* dst, cudaStream_t stream);
int im2col_s2_impl(const void* src, int B, int H, int W, int C, void* dst, cudaStream_t stream);
int timestep_embed_impl(const void* values, int n, int dim, int rows_repeat, void* out, cudaStream_t stream);
int skinny_linear_impl(const void* x, int ldx, int M, int K, const void* W, long long ldw, int N, const void* bias,
                       int in_silu, int out_silu, const void* addend, int ld_add, void* out, int ldo,
                       cudaStream_t stream);
int preprocess_impl(const void* image, const void* mask, int Cm, const void* img_min, int B, int H, int W, int scale,
                    void* init_image, void* mask_bin, void* masked_image, void* mask_latent, cudaStream_t stream);
int postprocess_impl(const void* x, int nhwc, int B, int H, int W, void* out_pt, void* out_u8, cudaStream_t stream);
int enc_attn_impl(const void* q, long long ldq, const void* k, const void* v, long long ldkv, void* out, long long ldo,
                  int B, int H, int N, int D, float scale, int causal, cudaStream_t stream);
int patchify_impl(const void* x, int B, int C, int Hi, int Wi, int P, void* out, int ldk, cudaStream_t stream);
int token_embed_impl(const void* ids, int rows, int T, int C, int vocab, const void* tok, const void* pos, void* out,
                     cudaStream_t stream);
void set_auto_v2(int on);
void set_cluster4(int on);
void set_attn_v2(int on);
void set_attn_qtiles(int n);
void set_attn_poly(int n);
int cfg_ddpm_impl(const void* eps, int ldc, int B, int C, int H, int W, const void* latents, const void* noise,
                  const void* coef, int do_cfg, void* out, cudaStream_t stream);
int cfg_sched_impl(const void* eps, int ldc, int B, int C, int H, int W, const void* latents, const void* noise,
                   void* hist, const void* coef, int family, int do_cfg, void* out, cudaStream_t stream);
int nchw_to_nhwc_scaled_impl(const void* src, int Bs, int Cs, int H, int W, const void* scale, void* dst, int Bd,
                             int ldc, int c_off, cudaStream_t stream);
}  // namespace vton

#define S(stream) static_cast<cudaStream_t>(stream)

extern "C" {

int b200vton_version(void) { return 107; }
const char* b200vton_last_error(void) { return vton::get_last_error(); }
long long b200vton_launch_count(void) { return vton::launch_count(); }
int b200vton_set_option(const char* name, int value) {
  if (name && strcmp(name, "gemm_2cta_auto") == 0) {
    vton::set_auto_v2(value);
    return 0;
  }
  if (name && strcmp(name, "gemm_cluster4") == 0) {
    vton::set_cluster4(value);
    return 0;
  }
  if (name && strcmp(name, "programmatic_launch") == 0) {
    vton::set_pdl(value);
    return 0;
  }
  if (name && strcmp(name, "attention_poly_exp") == 0) {
    vton::set_attn_poly(value);
    return 0;
  }
  if (name && strcmp(name, "attention_q_tiles") == 0) {
    vton::set_attn_qtiles(value);
    return 0;
  }
  if (name && strcmp(name, "attention_pingpong") == 0) {
    vton::set_attn_v2(value);
    return 0;
  }
  vton::set_last_error("unknown option %s", name ? name : "(null)");
  return vton::kErrInvalid;
}

int b200vton_gemm_f16(const void* A, int64_t lda, const void* W, int64_t ldw, void* out, int64_t ldo, int M, int N,
                      int K, const void* bias, const void* residual, int64_t ldr, const void* rowvec,
                      int64_t ld_rowvec, int rows_per_sample, int flags, int force_bn, void* stream) {
  return vton::gemm_f16_impl(A, lda, W, ldw, out, ldo, M, N, K, bias, residual, ldr, rowvec, ld_rowvec,
                             rows_per_sample, flags, force_bn, S(stream));
}

int b200vton_conv3x3_nhwc(const void* x, int64_t ldx, int B, int H, int W, int Cin, const void* w, int Cout,
                          const void* bias, const void* temb, int64_t ld_temb, const void* sc0, int C0,
                          const void* sc1, int C1, const void* w_sc, const void* bias_sc, const void* residual,
                          int64_t ldr, void* out, int64_t ldo, int force_bn, int stride, void* stream) {
  return vton::conv3x3_impl(x, ldx, B, H, W, Cin, w, Cout, bias, temb, ld_temb, sc0, C0, sc1, C1, w_sc, bias_sc,
                            residual, ldr, out, ldo, force_bn, stride, S(stream));
}

int b200vton_attention(const void* q, int64_t ldq, const void* k0, const void* v0, int64_t ldkv0, const void* k1,
                       const void* v1, int64_t ldkv1, void* out, int64_t ldo, int B, int H, int Nq, int N0, int N1,
                       int B1, int kv1_off, int kv1_mod, const void* kv1_base, float scale, int accumulate,
                       void* stream) {
  return vton::attn_impl(q, ldq, k0, v0, ldkv0, k1, v1, ldkv1, out, ldo, B, H, Nq, N0, N1, B1, kv1_off, kv1_mod, kv1_base, scale,
                         accumulate, S(stream));
}

int b200vton_encoder_attention(const void* q, int64_t ldq, const void* k, const void* v, int64_t ldkv, void* out,
                               int64_t ldo, int B, int H, int N, int D, float scale, int causal, void* stream) {
  return vton::enc_attn_impl(q, ldq, k, v, ldkv, out, ldo, B, H, N, D, scale, causal, S(stream));
}
int b200vton_patchify(const void* x, int B, int C, int Hi, int Wi, int P, void* out, int ldk, void* stream) {
  return vton::patchify_impl(x, B, C, Hi, Wi, P, out, ldk, S(stream));
}
int b200vton_token_embedding(const void* ids, int rows, int T, int C, int vocab, const void* token_embedding,
                             const void* position_embedding, void* out, void* stream) {
  return vton::token_embed_impl(ids, rows, T, C, vocab, token_embedding, position_embedding, out, S(stream));
}

int b200vton_cross_attention(const void* q, int64_t ldq, const void* kt, const void* vt, int64_t ldkv_t, int Nt,
                             const void* ki, const void* vi, int64_t ldkv_i, int Ni, void* out, int64_t ldo, int B,
                             int H, int Nq, float scale, float ip_scale, void* stream) {
  return vton::cross_attn_impl(q, ldq, kt, vt, ldkv_t, Nt, ki, vi, ldkv_i, Ni, out, ldo, B, H, Nq, scale, ip_scale,
                               S(stream));
}

int b200vton_conv3x3_nhwc_f32(const void* x, int B, int H, int W, int Cin, const void* w, int Cout, const void* bias,
                               const void* residual, void* out, void* stream) {
  return vton::conv3x3_f32_impl(x, B, H, W, Cin, w, Cout, bias, residual, out, 0, S(stream));
}
int b200vton_conv3x3_nhwc_f16in_f32(const void* x, int B, int H, int W, int Cin, const void* w, int Cout, const void* bias,
                                    const void* residual, void* out, void* stream) {
  return vton::conv3x3_f32_impl(x, B, H, W, Cin, w, Cout, bias, residual, out, 1, S(stream));
}
int b200vton_split_tf32(const void* x, int64_t stride_b, int B, int64_t per_batch, float scale, void* hi, void* lo,
                        void* stream) {
  return vton::split_tf32_impl(x, stride_b, B, per_batch, scale, hi, lo, S(stream));
}
int b200vton_softmax_split_tf32(const void* scores, int64_t rows, int N, void* p_hi, void* p_lo, void* stream) {
  return vton::softmax_split_tf32_impl(scores, rows, N, p_hi, p_lo, S(stream));
}

int b200vton_groupnorm_nhwc_f32(const void* x, int B, int HW, int C, const void* gamma, const void* beta, float eps,
                                 int silu, void* stats_ws, int64_t stats_ws_doubles, void* out, int out_fp16, void* stream) {
  return vton::groupnorm_f32_impl(x, B, HW, C, gamma, beta, eps, silu, stats_ws, stats_ws_doubles, out, out_fp16, S(stream));
}

int b200vton_groupnorm(const void* x0, int C0, const void* x1, int C1, int B, int HW, const void* gamma,
                       const void* beta, float eps, int silu, void* stats_ws, void* out, void* stream) {
  return vton::groupnorm_impl(x0, C0, x1, C1, B, HW, gamma, beta, eps, silu, stats_ws, out, S(stream));
}

int b200vton_layernorm(const void* x, int64_t ldx, int rows, int C, const void* gamma, const void* beta, float eps,
                       void* out, int64_t ldo, void* stream) {
  return vton::layernorm_impl(x, ldx, rows, C, gamma, beta, eps, out, ldo, S(stream));
}

int b200vton_nchw_to_nhwc(const void* src, int Bs, int Cs, int H, int W, void* dst, int Bd, int ldc, int c_off,
                          void* stream) {
  return vton::nchw_to_nhwc_impl(src, Bs, Cs, H, W, dst, Bd, ldc, c_off, S(stream));
}
int b200vton_nhwc_to_nchw(const void* src, int B, int C, int H, int W, int ldc, void* dst, void* stream) {
  return vton::nhwc_to_nchw_impl(src, B, C, H, W, ldc, dst, S(stream));
}
int b200vton_upsample2x_nhwc(const void* src, int B, int H, int W, int C, void* dst, void* stream) {
  return vton::upsample2x_impl(src, B, H, W, C, dst, S(stream));
}
int b200vton_im2col3x3_s2_nhwc(const void* src, int B, int H, int W, int C, void* dst, void* stream) {
  return vton::im2col_s2_impl(src, B, H, W, C, dst, S(stream));
}
int b200vton_timestep_embedding(const void* values, int n, int dim, int rows_repeat, void* out, void* stream) {
  return vton::timestep_embed_impl(values, n, dim, rows_repeat, out, S(stream));
}
int b200vton_skinny_linear(const void* x, int ldx, int M, int K, const void* W, int64_t ldw, int N, const void* bias,
                           int in_silu, int out_silu, const void* addend, int ld_add, void* out, int ldo,
                           void* stream) {
  return vton::skinny_linear_impl(x, ldx, M, K, W, ldw, N, bias, in_silu, out_silu, addend, ld_add, out, ldo,
                                  S(stream));
}
int b200vton_cfg_ddpm_step(const void* eps, int ldc, int B, int C, int H, int W, const void* latents,
                           const void* noise, const void* coef, int do_cfg, void* out, void* stream) {
  return vton::cfg_ddpm_impl(eps, ldc, B, C, H, W, latents, noise, coef, do_cfg, out, S(stream));
}
int b200vton_cfg_sched_step(const void* eps, int ldc, int B, int C, int H, int W, const void* latents,
                            const void* noise, void* hist, const void* coef, int family, int do_cfg, void* out,
                            void* stream) {
  return vton::cfg_sched_impl(eps, ldc, B, C, H, W, latents, noise, hist, coef, family, do_cfg, out, S(stream));
}
int b200vton_nchw_to_nhwc_scaled(const void* src, int Bs, int Cs, int H, int W, const void* scale, void* dst, int Bd,
                                 int ldc, int c_off, void* stream) {
  return vton::nchw_to_nhwc_scaled_impl(src, Bs, Cs, H, W, scale, dst, Bd, ldc, c_off, S(stream));
}

int b200vton_preprocess_inpaint(const void* image, const void* mask, int mask_channels, const void* image_min, int B,
                                int H, int W, int vae_scale, void* init_image, void* mask_bin, void* masked_image,
                                void* mask_latent, void* stream) {
  return vton::preprocess_impl(image, mask, mask_channels, image_min, B, H, W, vae_scale, init_image, mask_bin,
                               masked_image, mask_latent, S(stream));
}
int b200vton_postprocess_image(const void* x, int nhwc, int B, int H, int W, void* out_pt, void* out_u8, void* stream) {
  return vton::postprocess_impl(x, nhwc, B, H, W, out_pt, out_u8, S(stream));
}

}  // extern "C"
