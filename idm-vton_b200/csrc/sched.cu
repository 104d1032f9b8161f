// Fused classifier-free guidance + scheduler update for the non-DDPM schedulers the pipeline accepts
// (src/tryon_pipeline.py:1814-1823 with `pipe.scheduler` swapped for DDIM, Euler, Euler-ancestral or DPM-Solver++), and
// the latent scatter with the Euler families' input scaling (`scheduler.scale_model_input`, :1772).
// Restated from diffusers 0.25.0 (epsilon prediction); the per-step scalars are computed on the host by
// denoise.step_plan and live in a device row, so one captured CUDA graph serves every step of a request.
#include "common.cuh"
#include "host.h"

namespace vton {

// Scheduler families (b200vton_cfg_sched_step's `family`).
enum : int { kSchedDDIM = 0, kSchedEuler = 1, kSchedEulerAncestral = 2, kSchedDPMpp = 3 };

// ------------------------------------------------------------------------------------------------
// Coefficient row: 8 fp32 on the device. coef[0] = guidance scale, coef[7] = model-input scale (read by the scaled
// scatter below), coef[1..6] per family. A divisor d that torch applies as `fp16_tensor / cpu_scalar` is stored as d:
// ATen's CUDA division by a CPU scalar multiplies by the fp32 reciprocal 1/d, which the kernel recomputes (IEEE
// division, no fast-math) so the host-side step() run on the device and this kernel round identically.
// CFG (all families): g = u + fp16(gs * fp16(c - u)), or g = eps when do_cfg == 0.
//
// DDIM (DDIMScheduler.step, eta from the caller; every op rounds to fp16 like the reference's fp16 tensor arithmetic)
//   coef = {gs, sqrt(1-abar_t), sqrt(abar_t), sqrt(abar_prev), sqrt(1-abar_prev-std^2), std, -, in_scale}
//   x0 = fp16(fp16(x - fp16(sb * g)) * (1/sa));  prev = fp16(fp16(sap * x0) + fp16(cdir * g))
//   prev = fp16(prev + fp16(std * noise))   (only when std != 0: eta == 0 draws no noise)
// Euler (EulerDiscreteScheduler.step, s_churn = 0: the sample is upcast to fp32 inside step, the result cast back)
//   coef = {gs, sigma, sigma_next - sigma, -, -, -, -, in_scale}
//   x = fp32(x16);  x0 = x - fp16(sigma * g);  d = (x - x0) * (1/sigma);  prev = fp16(x + d * dt)   (fp32 ops,
//   each rounded: no FMA contraction, torch runs them as separate kernels)
// Euler-ancestral (EulerAncestralDiscreteScheduler.step; fp32 as Euler)
//   coef = {gs, sigma, sigma_down - sigma, sigma_up, -, -, -, in_scale}
//   as Euler, then prev = fp16(prev + fp16(sigma_up * noise))
// DPM-Solver++ (DPMSolverMultistepScheduler.step, algorithm_type "dpmsolver++", orders 1 and 2; no upcast in 0.25.0:
//   fp16 per-op). alpha_s = 1/sqrt(sigma_s^2+1), sig_s = sigma_s * alpha_s (same for t = the next sigma),
//   lambda = log(alpha) - log(sig), h = lambda_t - lambda_s, h0 = lambda_s - lambda_prev, r0 = h0 / h
//   coef = {gs, sig_s, alpha_s, sig_t/sig_s, alpha_t*(exp(-h)-1), c2, 1/r0, in_scale}
//   m0 = x0 = fp16(fp16(x - fp16(sig_s * g)) * (1/alpha_s));  m1 = hist (the previous step's x0)
//   prev = fp16(fp16(ratio * x) - fp16(c1 * m0))                               (first order: c2 == 0)
//   D1 = fp16(rr * fp16(m0 - m1));  prev = fp16(prev + fp16(c2 * D1))         (second order)
//   c2 = -0.5 * c1 (midpoint) or alpha_t*((exp(-h)-1)/h + 1) (heun); hist = m0 afterwards (each thread reads, then
//   writes, its own element, so the update is in place).
// eps: NHWC [2B, HW, ldc] (uncond rows first) or [B, ...] when do_cfg == 0; latents / noise / hist / out: NCHW [B,C,HW].
// ------------------------------------------------------------------------------------------------
template <int FAMILY>
__global__ void cfg_sched_kernel(const __half* eps, int ldc, int B, int C, int HW, const __half* latents,
                                 const __half* noise, __half* hist, const float* coef, int do_cfg, __half* out) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(B) * C * HW;
  if (i >= total) return;
  const int px = static_cast<int>(i % HW);
  const int c = static_cast<int>((i / HW) % C);
  const int b = static_cast<int>(i / (static_cast<long long>(HW) * C));
  const float gs = coef[0];
  float g;
  if (do_cfg) {
    const float u = h2f(eps[(static_cast<long long>(b) * HW + px) * ldc + c]);
    const float t = h2f(eps[(static_cast<long long>(b + B) * HW + px) * ldc + c]);
    g = round_h(u + round_h(gs * round_h(t - u)));
  } else {
    g = h2f(eps[(static_cast<long long>(b) * HW + px) * ldc + c]);
  }
  const float x = h2f(latents[i]);
  float prev;
  if (FAMILY == kSchedDDIM) {
    const float sb = coef[1], inv_sa = __fdiv_rn(1.f, coef[2]), sap = coef[3], cdir = coef[4], std_t = coef[5];
    const float x0 = round_h(round_h(x - round_h(sb * g)) * inv_sa);
    prev = round_h(round_h(sap * x0) + round_h(cdir * g));
    if (noise && std_t != 0.f) prev = round_h(prev + round_h(std_t * h2f(noise[i])));
  } else if (FAMILY == kSchedEuler || FAMILY == kSchedEulerAncestral) {
    const float sigma = coef[1], inv_sigma = __fdiv_rn(1.f, sigma), dt = coef[2];
    const float x0 = __fsub_rn(x, round_h(__fmul_rn(sigma, g)));
    const float d = __fmul_rn(__fsub_rn(x, x0), inv_sigma);
    prev = __fadd_rn(x, __fmul_rn(d, dt));
    if (FAMILY == kSchedEulerAncestral && noise) prev = __fadd_rn(prev, round_h(__fmul_rn(coef[3], h2f(noise[i]))));
  } else {
    const float sig_s = coef[1], inv_alpha_s = __fdiv_rn(1.f, coef[2]), ratio = coef[3], c1 = coef[4], c2 = coef[5],
                rr = coef[6];
    const float m0 = round_h(round_h(x - round_h(sig_s * g)) * inv_alpha_s);
    prev = round_h(round_h(ratio * x) - round_h(c1 * m0));
    if (c2 != 0.f) {
      const float d1 = round_h(rr * round_h(m0 - h2f(hist[i])));
      prev = round_h(prev + round_h(c2 * d1));
    }
    hist[i] = f2h(m0);
  }
  out[i] = f2h(prev);
}

int cfg_sched_impl(const void* eps, int ldc, int B, int C, int H, int W, const void* latents, const void* noise,
                   void* hist, const void* coef, int family, int do_cfg, void* out, cudaStream_t stream) {
  VTON_CHECK_ARG(B > 0 && C > 0 && C <= ldc && H > 0 && W > 0 && eps && latents && coef && out,
                 "cfg_sched_step: bad arguments");
  VTON_CHECK_ARG(family >= kSchedDDIM && family <= kSchedDPMpp, "cfg_sched_step: unknown scheduler family %d", family);
  VTON_CHECK_ARG(family != kSchedDPMpp || hist, "cfg_sched_step: DPM-Solver++ needs the history buffer");
  VTON_CHECK_ARG(family != kSchedEulerAncestral || noise, "cfg_sched_step: Euler-ancestral needs the noise buffer");
  const long long total = static_cast<long long>(B) * C * H * W;
  const unsigned grid = static_cast<unsigned>((total + 255) / 256);
  const __half* e = static_cast<const __half*>(eps);
  const __half* x = static_cast<const __half*>(latents);
  const __half* n = static_cast<const __half*>(noise);
  __half* hs = static_cast<__half*>(hist);
  const float* cf = static_cast<const float*>(coef);
  __half* o = static_cast<__half*>(out);
  switch (family) {
    case kSchedDDIM: cfg_sched_kernel<kSchedDDIM><<<grid, 256, 0, stream>>>(e, ldc, B, C, H * W, x, n, hs, cf, do_cfg, o); break;
    case kSchedEuler: cfg_sched_kernel<kSchedEuler><<<grid, 256, 0, stream>>>(e, ldc, B, C, H * W, x, n, hs, cf, do_cfg, o); break;
    case kSchedEulerAncestral:
      cfg_sched_kernel<kSchedEulerAncestral><<<grid, 256, 0, stream>>>(e, ldc, B, C, H * W, x, n, hs, cf, do_cfg, o);
      break;
    default: cfg_sched_kernel<kSchedDPMpp><<<grid, 256, 0, stream>>>(e, ldc, B, C, H * W, x, n, hs, cf, do_cfg, o); break;
  }
  count_launch();
  VTON_CUDA(cudaGetLastError());
  return kOk;
}

// ------------------------------------------------------------------------------------------------
// dst[s, y, x, c_off + c] = fp16(src[s % Bs, c, y, x] * scale[0]): the scatter of nchw_to_nhwc_kernel fused with
// `scheduler.scale_model_input` of the Euler families, sample / sqrt(sigma^2 + 1), which ATen runs as a multiply by the
// fp32 reciprocal (division by a CPU scalar). scale: one fp32 on the device (the coefficient row's in_scale), so the
// captured graph follows the per-step sigma.
// ------------------------------------------------------------------------------------------------
__global__ void nchw_to_nhwc_scaled_kernel(const __half* src, int Bs, int Cs, int HW, const float* scale, __half* dst,
                                           int Bd, int ldc, int c_off) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long total = static_cast<long long>(Bd) * HW;
  if (i >= total) return;
  const int s = static_cast<int>(i / HW);
  const int px = static_cast<int>(i % HW);
  const int sb = s % Bs;
  const float k = *scale;
  for (int c = 0; c < Cs; ++c)
    dst[i * ldc + c_off + c] = f2h(__fmul_rn(h2f(src[(static_cast<long long>(sb) * Cs + c) * HW + px]), k));
}

int nchw_to_nhwc_scaled_impl(const void* src, int Bs, int Cs, int H, int W, const void* scale, void* dst, int Bd,
                             int ldc, int c_off, cudaStream_t stream) {
  VTON_CHECK_ARG(Bs > 0 && Cs > 0 && H > 0 && W > 0 && Bd > 0 && c_off >= 0 && c_off + Cs <= ldc,
                 "nchw_to_nhwc_scaled: bad shape");
  VTON_CHECK_ARG(src && dst && scale, "nchw_to_nhwc_scaled: null pointer");
  const long long total = static_cast<long long>(Bd) * H * W;
  nchw_to_nhwc_scaled_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, stream>>>(
      static_cast<const __half*>(src), Bs, Cs, H * W, static_cast<const float*>(scale), static_cast<__half*>(dst), Bd,
      ldc, c_off);
  count_launch();
  VTON_CUDA(cudaGetLastError());
  return kOk;
}

}  // namespace vton
