"""ORACLE (test infrastructure, not product): the update rules of the four non-DDPM schedulers the engine runs, restated
independently of idm_vton_b200 from their papers, in float64 scalars:

  DDIM         Song et al. 2021, eq. 12: x' = sqrt(a') x0 + sqrt(1 - a' - s^2) eps + s z,
               x0 = (x - sqrt(1-a) eps) / sqrt(a),  s = eta sqrt((1-a')/(1-a)) sqrt(1 - a/a')
  Euler        Karras et al. 2022, Alg. 1 (deterministic Euler in sigma) on the VE variable x = x_vp sqrt(1 + sigma^2):
               the network sees x / sqrt(1 + sigma^2) (VP <-> VE scaling), D = x - sigma eps, x' = x + (sigma' - sigma)(x - D)/sigma
  Euler-a      the ancestral split sigma_up = min(sigma', sqrt(sigma'^2 (sigma^2 - sigma'^2) / sigma^2)),
               sigma_down = sqrt(sigma'^2 - sigma_up^2): x' = x + (sigma_down - sigma)(x - D)/sigma + sigma_up z
  DPM-Solver++ Lu et al. 2022, Alg. 2 (2M): alpha = 1/sqrt(1+sigma^2), s = sigma alpha, lambda = log(alpha/s),
               h = lambda' - lambda, r = h_prev / h, D = (1 + 1/(2r)) x0 - 1/(2r) x0_prev (first step, and the steps the
               solver's order schedule takes first order: D = x0), x' = (s'/s) x - alpha' (e^-h - 1) D; onto sigma' = 0
               (h = +inf) x' = x0. solver_type "heun": x' = (s'/s) x - alpha'(e^-h - 1) x0 + alpha'((e^-h - 1)/h + 1)(x0 - x0_prev)/r.

The schedule itself (timesteps, sigmas, alphas_cumprod) is taken from a configured scheduler object: only the step
rules are restated here. `denoise_loop` is loop_ref.denoise_loop's loop driven by such a scheduler, with the
`scale_model_input` call and the float timesteps the DDPM loop does not need. Only tests/ may import this module.
"""
import math

import torch


def _kind(sched):
    cfg = getattr(sched, "config", {})
    name = (cfg.get("_class_name") if isinstance(cfg, dict) else None) or type(sched).__name__
    return {"DDIMScheduler": "ddim", "EulerDiscreteScheduler": "euler", "EulerAncestralDiscreteScheduler": "euler_ancestral",
            "DPMSolverMultistepScheduler": "dpmsolver++"}[name]


class PaperScheduler:
    """Scheduler-shaped wrapper (set_timesteps / timesteps / scale_model_input / step(eps, t, x, noise=)) that steps by the
    paper forms above over the tables of `sched`. eta: DDIM's eta."""

    def __init__(self, sched, eta=0.0):
        self.sched, self.eta, self.kind = sched, float(eta), _kind(sched)
        cfg = sched.config
        self.cfg = (lambda k, d=None: cfg.get(k, d)) if isinstance(cfg, dict) else (lambda k, d=None: getattr(cfg, k, d))

    def set_timesteps(self, n):
        self.sched.set_timesteps(n)
        self.timesteps = self.sched.timesteps
        self.ac = [float(a) for a in self.sched.alphas_cumprod.double()]
        self.sigmas = [float(s) for s in self.sched.sigmas.double()] if self.kind != "ddim" else None
        self.i, self.x0_prev, self.lam_prev = 0, None, None
        return self.timesteps

    # --- the per-step scalars -------------------------------------------------------------------------------------
    def _ddim_alphas(self, t):
        n_train, n = int(self.cfg("num_train_timesteps", 1000)), len(self.timesteps)
        prev = int(t) - n_train // n
        final = 1.0 if self.cfg("set_alpha_to_one", True) else self.ac[0]
        return self.ac[int(t)], (self.ac[prev] if prev >= 0 else final)

    def scale_model_input(self, x, t):
        if self.kind in ("euler", "euler_ancestral"):
            return x / math.sqrt(self.sigmas[self.i] ** 2 + 1)
        return x

    def _dpm_order(self):
        n, i = len(self.timesteps), self.i
        if self.cfg("solver_order", 2) == 1 or i == 0 or self.sigmas[i + 1] in (0.0, self.sigmas[i]):
            return 1
        if i == n - 1 and (self.cfg("euler_at_final", False) or (self.cfg("lower_order_final", True) and n < 15)
                           or self.cfg("final_sigmas_type", "sigma_min") == "zero"):
            return 1
        return 2

    def step(self, eps, t, x, noise=None):
        i = self.i
        if self.kind == "ddim":
            a, a_prev = self._ddim_alphas(t)
            x0 = (x - math.sqrt(1 - a) * eps) / math.sqrt(a)
            s = self.eta * math.sqrt((1 - a_prev) / (1 - a)) * math.sqrt(1 - a / a_prev)
            out = math.sqrt(a_prev) * x0 + math.sqrt(max(1 - a_prev - s * s, 0.0)) * eps
            if s > 0:
                out = out + s * noise
        elif self.kind in ("euler", "euler_ancestral"):
            sig, sig_next = self.sigmas[i], self.sigmas[i + 1]
            D = x - sig * eps
            d = (x - D) / sig
            if self.kind == "euler":
                out = x + (sig_next - sig) * d
            else:
                up = min(sig_next, math.sqrt(sig_next ** 2 * (sig ** 2 - sig_next ** 2) / sig ** 2))
                down = math.sqrt(sig_next ** 2 - up ** 2)
                out = x + (down - sig) * d + up * noise
        else:
            sig_s, sig_t = self.sigmas[i], self.sigmas[i + 1]
            alpha_s = 1 / math.sqrt(1 + sig_s ** 2)
            s_s = sig_s * alpha_s
            x0 = (x - s_s * eps) / alpha_s
            lam_s = math.log(alpha_s / s_s)
            if sig_t == 0.0:
                out = x0
            else:
                alpha_t = 1 / math.sqrt(1 + sig_t ** 2)
                s_t = sig_t * alpha_t
                h = math.log(alpha_t / s_t) - lam_s
                phi = alpha_t * (math.exp(-h) - 1)
                if self._dpm_order() == 1:
                    out = (s_t / s_s) * x - phi * x0
                else:
                    r = (lam_s - self.lam_prev) / h
                    if self.cfg("solver_type", "midpoint") == "heun":
                        out = (s_t / s_s) * x - phi * x0 + alpha_t * ((math.exp(-h) - 1) / h + 1) * (x0 - self.x0_prev) / r
                    else:
                        D = (1 + 1 / (2 * r)) * x0 - (1 / (2 * r)) * self.x0_prev
                        out = (s_t / s_s) * x - phi * D
            self.x0_prev, self.lam_prev = x0, lam_s
        self.i += 1
        return out

    def draws_noise(self):
        return self.kind == "euler_ancestral" or (self.kind == "ddim" and self.eta > 0)


def denoise_loop(sd_t, cfg_t, sd_g, cfg_g, inp, num_steps, scheduler, guidance_scale=2.0, noises=None, max_steps=None):
    """The reference loop (src/tryon_pipeline.py:1765-1823, as restated by loop_ref.denoise_loop) driven by a
    PaperScheduler: the latent half of the UNet input goes through `scheduler.scale_model_input` (:1772) and both UNets see
    the float timestep (Euler's timesteps need not be integers). inp / noises as in loop_ref.denoise_loop; noises[i] is
    used by the steps that draw noise (DDIM with eta > 0, Euler-ancestral)."""
    from . import unet_ref as R
    sch = scheduler
    timesteps = sch.set_timesteps(num_steps)
    latents = inp["latents"]
    for i, t in enumerate(timesteps):
        if max_steps is not None and i >= max_steps:
            break
        latent_model_input = sch.scale_model_input(torch.cat([latents] * 2), t)                    # :1769-1772
        latent_model_input = torch.cat([latent_model_input, inp["mask"], inp["masked_image_latents"],
                                        inp["pose_latents"]], dim=1)                             # :1777
        tt = torch.as_tensor(float(t), device=latents.device)
        feats = R.unet_garment_forward(sd_g, cfg_g, inp["cloth_latents"], tt, inp["text_embeds_cloth"])  # :1787
        if feats[0].shape[0] != latents.shape[0]:
            feats = [f.expand(latents.shape[0], -1, -1) for f in feats]          # one shared garment
        feats = [torch.cat([torch.zeros_like(d), d]) for d in feats]                              # :1796
        added = {"text_embeds": inp["add_text_embeds"], "time_ids": inp["add_time_ids"],
                 "image_embeds": inp["image_embeds"]}
        noise_pred = R.unet_tryon_forward(sd_t, cfg_t, latent_model_input, tt, inp["prompt_embeds"], added, feats)
        u, c = noise_pred.chunk(2)
        noise_pred = u + guidance_scale * (c - u)                                                 # :1815-1816
        latents = sch.step(noise_pred, t, latents, noise=None if noises is None else noises[i])   # :1823
    return latents
