"""DDPM ancestral scheduler with the reference pipeline's configuration (host side, plain torch fp32).

Restates diffusers==0.25.0 DDPMScheduler as used by src/tryon_pipeline.py:1561,1823 (set_timesteps / step) for:
scaled_linear betas 0.00085..0.012, 1000 train steps, epsilon prediction, fixed_small variance, leading spacing with
steps_offset 1, optional zero-terminal-SNR rescale (train_xl.py:317). The per-step arithmetic itself runs in
b200vton_cfg_ddpm_step; this class only produces the timestep list and the per-step scalar coefficients.
"""
import torch


def _rescale_zero_terminal_snr(betas):
    alphas = 1.0 - betas
    alphas_cumprod = torch.cumprod(alphas, dim=0)
    alphas_bar_sqrt = alphas_cumprod.sqrt()
    a0 = alphas_bar_sqrt[0].clone()
    aT = alphas_bar_sqrt[-1].clone()
    alphas_bar_sqrt = alphas_bar_sqrt - aT
    alphas_bar_sqrt = alphas_bar_sqrt * (a0 / (a0 - aT))
    alphas_bar = alphas_bar_sqrt ** 2
    alphas = alphas_bar[1:] / alphas_bar[:-1]
    alphas = torch.cat([alphas_bar[0:1], alphas])
    return 1 - alphas


class DDPMScheduler:
    order = 1
    init_noise_sigma = 1.0

    def __init__(self, num_train_timesteps=1000, beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
                 timestep_spacing="leading", steps_offset=1, rescale_betas_zero_snr=False,
                 prediction_type="epsilon", variance_type="fixed_small", clip_sample=False):
        if beta_schedule != "scaled_linear" or prediction_type != "epsilon" or variance_type != "fixed_small" or clip_sample:
            raise NotImplementedError("only the IDM-VTON scheduler configuration is supported")
        if timestep_spacing not in ("leading", "trailing", "linspace"):
            raise ValueError(timestep_spacing)
        self.config = type("Cfg", (), dict(num_train_timesteps=num_train_timesteps, beta_start=beta_start,
                                           beta_end=beta_end, beta_schedule=beta_schedule,
                                           timestep_spacing=timestep_spacing, steps_offset=steps_offset,
                                           rescale_betas_zero_snr=rescale_betas_zero_snr,
                                           prediction_type=prediction_type, variance_type=variance_type,
                                           clip_sample=clip_sample))()
        betas = torch.linspace(beta_start ** 0.5, beta_end ** 0.5, num_train_timesteps, dtype=torch.float32) ** 2
        if rescale_betas_zero_snr:
            betas = _rescale_zero_terminal_snr(betas)
        self.betas = betas
        self.alphas = 1.0 - betas
        self.alphas_cumprod = torch.cumprod(self.alphas, dim=0)
        self.one = torch.tensor(1.0)
        self.num_inference_steps = None
        self.timesteps = torch.arange(num_train_timesteps - 1, -1, -1)

    def set_timesteps(self, num_inference_steps, device=None):
        n = self.config.num_train_timesteps
        if num_inference_steps > n:
            raise ValueError(f"num_inference_steps {num_inference_steps} > num_train_timesteps {n}")
        self.num_inference_steps = num_inference_steps
        sp = self.config.timestep_spacing
        if sp == "leading":
            ratio = n // num_inference_steps
            ts = (torch.arange(0, num_inference_steps, dtype=torch.float64) * ratio).round().flip(0).to(torch.int64)
            ts = ts + self.config.steps_offset
        elif sp == "trailing":
            ratio = n / num_inference_steps
            ts = (torch.arange(n, 0, -ratio, dtype=torch.float64)).round().to(torch.int64) - 1
        else:
            ts = torch.linspace(0, n - 1, num_inference_steps, dtype=torch.float64).round().flip(0).to(torch.int64)
        self.timesteps = ts.to(device) if device is not None else ts

    def scale_model_input(self, sample, timestep=None):
        return sample

    def previous_timestep(self, t):
        steps = self.num_inference_steps if self.num_inference_steps else self.config.num_train_timesteps
        return t - self.config.num_train_timesteps // steps

    def step(self, model_output, timestep, sample, generator=None, return_dict=True):
        """diffusers DDPMScheduler.step (epsilon prediction, fixed_small variance) on the host in plain torch — the
        arithmetic the reference loop runs at src/tryon_pipeline.py:1823. The engine does NOT call this (its per-step
        update is the fused `b200vton_cfg_ddpm_step` kernel fed by `step_coefficients`); it exists so this object is a
        complete scheduler for callers that step it themselves (e.g. the reference pipeline in oracle/make_golden_pipeline.py)."""
        t = int(timestep)
        prev_t = self.previous_timestep(t)
        a_t = self.alphas_cumprod[t]
        a_prev = self.alphas_cumprod[prev_t] if prev_t >= 0 else self.one
        b_t, b_prev = 1 - a_t, 1 - a_prev
        cur_a = a_t / a_prev
        cur_b = 1 - cur_a
        pred_original_sample = (sample - b_t ** 0.5 * model_output) / a_t ** 0.5
        pred_prev_sample = (a_prev ** 0.5 * cur_b) / b_t * pred_original_sample + cur_a ** 0.5 * b_prev / b_t * sample
        self._last_noise = None
        if t > 0:
            dev = model_output.device
            rand_dev = "cpu" if (generator is not None and generator.device.type == "cpu" and dev.type != "cpu") else dev
            noise = torch.randn(model_output.shape, generator=generator, device=rand_dev, dtype=model_output.dtype).to(dev)
            var = torch.clamp((1 - a_prev) / (1 - a_t) * cur_b, min=1e-20)
            pred_prev_sample = pred_prev_sample + (var ** 0.5) * noise
            self._last_noise = noise
        if not return_dict:
            return (pred_prev_sample,)
        return type("DDPMSchedulerOutput", (), dict(prev_sample=pred_prev_sample, pred_original_sample=pred_original_sample))()

    def step_coefficients(self, t):
        """(sqrt(1-abar_t), 1/sqrt(abar_t), x0 coeff, x_t coeff, sigma_t) as python floats, computed in fp32 torch
        exactly like DDPMScheduler.step / _get_variance."""
        t = int(t)
        prev_t = self.previous_timestep(t)
        a_t = self.alphas_cumprod[t]
        a_prev = self.alphas_cumprod[prev_t] if prev_t >= 0 else self.one
        b_t = 1 - a_t
        b_prev = 1 - a_prev
        cur_a = a_t / a_prev
        cur_b = 1 - cur_a
        c0 = (a_prev ** 0.5 * cur_b) / b_t
        c1 = cur_a ** 0.5 * b_prev / b_t
        var = torch.clamp((1 - a_prev) / (1 - a_t) * cur_b, min=1e-20)
        sigma = var ** 0.5 if t > 0 else torch.tensor(0.0)
        inv_sa = torch.tensor(1.0, dtype=torch.float32) / (a_t ** 0.5)
        return float(b_t ** 0.5), float(inv_sa), float(c0), float(c1), float(sigma)


# ---------------------------------------------------------------------------------------------------------------------
# Schedulers the pipeline can be switched to (`pipe.scheduler = DPMSolverMultistepScheduler.from_config(...)`), restated
# from diffusers==0.25.0 because diffusers is not a dependency of the engine. "Parity unpinned": these were written from
# the published 0.25.0 sources and papers and have not been run side by side with diffusers itself (tests/
# test_schedulers.py holds a check that runs when diffusers is importable). The engine never calls their step(): its
# per-step update is b200vton_cfg_sched_step fed by denoise.step_plan, which reads the tables these objects (or the
# caller's own diffusers objects) expose after set_timesteps. step() exists so each object is a complete scheduler and
# pins the plan on the host. Restated for epsilon prediction without clipping / thresholding; other settings raise.
# Tables follow diffusers: alphas_cumprod fp32, sigmas fp32 on the CPU (0-dim coefficients multiply fp16 tensors as
# fp32 scalars, and ATen divides a CUDA tensor by a CPU scalar as a multiply by its fp32 reciprocal).
# ---------------------------------------------------------------------------------------------------------------------
import inspect as _inspect
import math as _math

import numpy as _np


class _Config(dict):
    """diffusers' FrozenDict surface: keys readable as items and as attributes."""

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError:
            raise AttributeError(k) from None


def _config_items(config):
    if isinstance(config, dict):
        return dict(config)
    return {k: getattr(config, k) for k in dir(config) if not k.startswith("__") and not callable(getattr(config, k))}


class _FromConfig:
    @classmethod
    def from_config(cls, config=None, **kwargs):
        """diffusers' ConfigMixin.from_config: keys this class does not know (another scheduler's config) are ignored."""
        items = _config_items(config) if config is not None else {}
        items.update(kwargs)
        params = _inspect.signature(cls.__init__).parameters
        return cls(**{k: v for k, v in items.items() if k in params and k != "self"})

    def _register(self, **kw):
        self.config = _Config(_class_name=type(self).__name__, **kw)


def _betas(num_train_timesteps, beta_start, beta_end, beta_schedule, trained_betas, rescale_betas_zero_snr):
    if trained_betas is not None:
        betas = torch.tensor(trained_betas, dtype=torch.float32)
    elif beta_schedule == "linear":
        betas = torch.linspace(beta_start, beta_end, num_train_timesteps, dtype=torch.float32)
    elif beta_schedule == "scaled_linear":
        betas = torch.linspace(beta_start ** 0.5, beta_end ** 0.5, num_train_timesteps, dtype=torch.float32) ** 2
    else:
        raise NotImplementedError(f"beta_schedule {beta_schedule!r} is not restated here")
    if rescale_betas_zero_snr:
        betas = _rescale_zero_terminal_snr(betas)
    return betas


def _check_epsilon(name, prediction_type, thresholding=False, clip_sample=False):
    if prediction_type != "epsilon":
        raise NotImplementedError(f"{name}: prediction_type {prediction_type!r} is not supported (epsilon prediction only)")
    if thresholding or clip_sample:
        raise NotImplementedError(f"{name}: thresholding / clip_sample are not supported")


def _spaced_int_timesteps(n_train, n, spacing, steps_offset):
    """DDIMScheduler.set_timesteps (the same rule as DDPMScheduler.set_timesteps)."""
    if n > n_train:
        raise ValueError(f"num_inference_steps {n} > num_train_timesteps {n_train}")
    if spacing == "linspace":
        ts = _np.linspace(0, n_train - 1, n).round()[::-1].copy().astype(_np.int64)
    elif spacing == "leading":
        ratio = n_train // n
        ts = (_np.arange(0, n) * ratio).round()[::-1].copy().astype(_np.int64) + steps_offset
    elif spacing == "trailing":
        ratio = n_train / n
        ts = _np.round(_np.arange(n_train, 0, -ratio)).astype(_np.int64) - 1
    else:
        raise ValueError(f"timestep_spacing {spacing!r}")
    return torch.from_numpy(ts)


def _randn_like(x, generator):
    dev = x.device
    rand_dev = "cpu" if (generator is not None and generator.device.type == "cpu" and dev.type != "cpu") else dev
    return torch.randn(x.shape, generator=generator, device=rand_dev, dtype=x.dtype).to(dev)


def _upcast(x):
    """`sample.to(torch.float32)` of the Euler steps; float64 stays float64 so the step can be checked in fp64."""
    return x.to(torch.promote_types(x.dtype, torch.float32))


def _output(cls_name, return_dict, prev, x0):
    if not return_dict:
        return (prev,)
    return type(cls_name, (), dict(prev_sample=prev, pred_original_sample=x0))()


class DDIMScheduler(_FromConfig):
    """diffusers 0.25.0 DDIMScheduler: set_timesteps, step (DDIM eq. 12 with `eta`), _get_variance. Parity unpinned."""
    order = 1
    init_noise_sigma = 1.0

    def __init__(self, num_train_timesteps=1000, beta_start=0.0001, beta_end=0.02, beta_schedule="linear",
                 trained_betas=None, clip_sample=True, set_alpha_to_one=True, steps_offset=0, prediction_type="epsilon",
                 thresholding=False, dynamic_thresholding_ratio=0.995, clip_sample_range=1.0, sample_max_value=1.0,
                 timestep_spacing="leading", rescale_betas_zero_snr=False):
        self._register(num_train_timesteps=num_train_timesteps, beta_start=beta_start, beta_end=beta_end,
                       beta_schedule=beta_schedule, trained_betas=trained_betas, clip_sample=clip_sample,
                       set_alpha_to_one=set_alpha_to_one, steps_offset=steps_offset, prediction_type=prediction_type,
                       thresholding=thresholding, timestep_spacing=timestep_spacing,
                       rescale_betas_zero_snr=rescale_betas_zero_snr)
        self.betas = _betas(num_train_timesteps, beta_start, beta_end, beta_schedule, trained_betas, rescale_betas_zero_snr)
        self.alphas = 1.0 - self.betas
        self.alphas_cumprod = torch.cumprod(self.alphas, dim=0)
        self.final_alpha_cumprod = torch.tensor(1.0) if set_alpha_to_one else self.alphas_cumprod[0]
        self.num_inference_steps = None
        self.timesteps = torch.from_numpy(_np.arange(0, num_train_timesteps)[::-1].copy().astype(_np.int64))

    def scale_model_input(self, sample, timestep=None):
        return sample

    def set_timesteps(self, num_inference_steps, device=None):
        c = self.config
        self.num_inference_steps = num_inference_steps
        ts = _spaced_int_timesteps(c.num_train_timesteps, num_inference_steps, c.timestep_spacing, c.steps_offset)
        self.timesteps = ts.to(device) if device is not None else ts

    def _alphas(self, t):
        prev_t = t - self.config.num_train_timesteps // self.num_inference_steps
        a_t = self.alphas_cumprod[t]
        a_prev = self.alphas_cumprod[prev_t] if prev_t >= 0 else self.final_alpha_cumprod
        return a_t, a_prev

    def _get_variance(self, t):
        a_t, a_prev = self._alphas(t)
        b_t, b_prev = 1 - a_t, 1 - a_prev
        return (b_prev / b_t) * (1 - a_t / a_prev)

    def step(self, model_output, timestep, sample, eta=0.0, use_clipped_model_output=False, generator=None,
             variance_noise=None, return_dict=True):
        _check_epsilon("DDIMScheduler", self.config.prediction_type, self.config.thresholding, self.config.clip_sample)
        t = int(timestep)
        a_t, a_prev = self._alphas(t)
        b_t = 1 - a_t
        pred_original_sample = (sample - b_t ** 0.5 * model_output) / a_t ** 0.5
        std_dev_t = eta * self._get_variance(t) ** 0.5
        pred_sample_direction = (1 - a_prev - std_dev_t ** 2) ** 0.5 * model_output
        prev_sample = a_prev ** 0.5 * pred_original_sample + pred_sample_direction
        if eta > 0:
            if variance_noise is None:
                variance_noise = _randn_like(model_output, generator)
            prev_sample = prev_sample + std_dev_t * variance_noise
        return _output("DDIMSchedulerOutput", return_dict, prev_sample, pred_original_sample)


class _SigmaScheduler(_FromConfig):
    """Step-index bookkeeping shared by the sigma-parametrised schedulers (diffusers `_init_step_index`)."""
    _step_index = None

    @property
    def step_index(self):
        return self._step_index

    def _init_step_index(self, timestep):
        if torch.is_tensor(timestep):
            timestep = timestep.to(self.timesteps.device)
        cand = (self.timesteps == timestep).nonzero()
        self._step_index = int(cand[1 if len(cand) > 1 else 0])

    @staticmethod
    def _sigma_to_t(sigma, log_sigmas):
        log_sigma = _np.log(_np.maximum(sigma, 1e-10))
        dists = log_sigma - log_sigmas[:, _np.newaxis]
        low_idx = _np.cumsum((dists >= 0), axis=0).argmax(axis=0).clip(max=log_sigmas.shape[0] - 2)
        high_idx = low_idx + 1
        low, high = log_sigmas[low_idx], log_sigmas[high_idx]
        w = _np.clip((low - log_sigma) / (low - high), 0, 1)
        t = (1 - w) * low_idx + w * high_idx
        return t.reshape(sigma.shape)

    @staticmethod
    def _convert_to_karras(in_sigmas, num_inference_steps):
        sigma_min, sigma_max = in_sigmas[-1].item(), in_sigmas[0].item()
        rho = 7.0
        ramp = _np.linspace(0, 1, num_inference_steps)
        min_inv_rho, max_inv_rho = sigma_min ** (1 / rho), sigma_max ** (1 / rho)
        return (max_inv_rho + ramp * (min_inv_rho - max_inv_rho)) ** rho


class EulerDiscreteScheduler(_SigmaScheduler):
    """diffusers 0.25.0 EulerDiscreteScheduler: set_timesteps (leading / trailing / linspace, linear interpolation,
    optional Karras sigmas, final sigma 0), init_noise_sigma, scale_model_input, step with s_churn = 0 (Karras et al.
    Alg. 2 with gamma = 0; the noise is drawn every step, as the published step does, and unused). Parity unpinned."""
    order = 1

    def __init__(self, num_train_timesteps=1000, beta_start=0.0001, beta_end=0.02, beta_schedule="linear",
                 trained_betas=None, prediction_type="epsilon", interpolation_type="linear", use_karras_sigmas=False,
                 timestep_spacing="linspace", steps_offset=0, rescale_betas_zero_snr=False):
        if interpolation_type != "linear":
            raise NotImplementedError(f"EulerDiscreteScheduler: interpolation_type {interpolation_type!r} is not restated")
        self._register(num_train_timesteps=num_train_timesteps, beta_start=beta_start, beta_end=beta_end,
                       beta_schedule=beta_schedule, trained_betas=trained_betas, prediction_type=prediction_type,
                       interpolation_type=interpolation_type, use_karras_sigmas=use_karras_sigmas,
                       timestep_spacing=timestep_spacing, steps_offset=steps_offset,
                       rescale_betas_zero_snr=rescale_betas_zero_snr)
        self.betas = _betas(num_train_timesteps, beta_start, beta_end, beta_schedule, trained_betas, rescale_betas_zero_snr)
        self.alphas = 1.0 - self.betas
        self.alphas_cumprod = torch.cumprod(self.alphas, dim=0)
        self.num_inference_steps = None
        self.set_timesteps(num_train_timesteps)
        self.num_inference_steps = None

    @property
    def init_noise_sigma(self):
        max_sigma = self.sigmas.max()
        if self.config.timestep_spacing in ("linspace", "trailing"):
            return max_sigma
        return (max_sigma ** 2 + 1) ** 0.5

    def _float_timesteps(self, n):
        c = self.config
        if n > c.num_train_timesteps:
            raise ValueError(f"num_inference_steps {n} > num_train_timesteps {c.num_train_timesteps}")
        if c.timestep_spacing == "linspace":
            return _np.linspace(0, c.num_train_timesteps - 1, n, dtype=_np.float32)[::-1].copy()
        if c.timestep_spacing == "leading":
            ratio = c.num_train_timesteps // n
            ts = (_np.arange(0, n) * ratio).round()[::-1].copy().astype(_np.float32)
            return ts + c.steps_offset
        if c.timestep_spacing == "trailing":
            ratio = c.num_train_timesteps / n
            return _np.arange(c.num_train_timesteps, 0, -ratio).round().copy().astype(_np.float32) - 1
        raise ValueError(f"timestep_spacing {c.timestep_spacing!r}")

    def set_timesteps(self, num_inference_steps, device=None):
        self.num_inference_steps = num_inference_steps
        timesteps = self._float_timesteps(num_inference_steps)
        sigmas = (((1 - self.alphas_cumprod) / self.alphas_cumprod) ** 0.5).numpy()
        log_sigmas = _np.log(sigmas)
        sigmas = _np.interp(timesteps, _np.arange(0, len(sigmas)), sigmas)
        if self.config.use_karras_sigmas:
            sigmas = self._convert_to_karras(in_sigmas=sigmas, num_inference_steps=num_inference_steps)
            timesteps = _np.array([self._sigma_to_t(s, log_sigmas) for s in sigmas])
        sigmas = torch.from_numpy(sigmas).to(dtype=torch.float32)
        self.timesteps = torch.from_numpy(timesteps.astype(_np.float32))
        if device is not None:
            self.timesteps = self.timesteps.to(device)
        self.sigmas = torch.cat([sigmas, torch.zeros(1)])          # kept on the CPU, like diffusers
        self._step_index = None

    def scale_model_input(self, sample, timestep):
        if self.step_index is None:
            self._init_step_index(timestep)
        sigma = self.sigmas[self.step_index]
        return sample / ((sigma ** 2 + 1) ** 0.5)

    def step(self, model_output, timestep, sample, s_churn=0.0, s_tmin=0.0, s_tmax=float("inf"), s_noise=1.0,
             generator=None, return_dict=True):
        _check_epsilon("EulerDiscreteScheduler", self.config.prediction_type)
        if s_churn != 0.0:
            raise NotImplementedError("EulerDiscreteScheduler: s_churn > 0 is not restated (the pipeline never passes it)")
        if self.step_index is None:
            self._init_step_index(timestep)
        sample = _upcast(sample)
        sigma = self.sigmas[self.step_index]
        _randn_like(model_output, generator) * s_noise            # drawn and unused with gamma = 0
        sigma_hat = sigma * (0.0 + 1)
        pred_original_sample = sample - sigma_hat * model_output
        derivative = (sample - pred_original_sample) / sigma_hat
        dt = self.sigmas[self.step_index + 1] - sigma_hat
        prev_sample = sample + derivative * dt
        prev_sample = prev_sample.to(model_output.dtype)
        self._step_index += 1
        return _output("EulerDiscreteSchedulerOutput", return_dict, prev_sample, pred_original_sample)


class EulerAncestralDiscreteScheduler(EulerDiscreteScheduler):
    """diffusers 0.25.0 EulerAncestralDiscreteScheduler: the Euler tables (no Karras sigmas) and the ancestral step,
    sigma_up = sqrt(sigma_to^2 (sigma_from^2 - sigma_to^2) / sigma_from^2), sigma_down = sqrt(sigma_to^2 - sigma_up^2),
    noise drawn every step. Parity unpinned."""

    def __init__(self, num_train_timesteps=1000, beta_start=0.0001, beta_end=0.02, beta_schedule="linear",
                 trained_betas=None, prediction_type="epsilon", timestep_spacing="linspace", steps_offset=0,
                 rescale_betas_zero_snr=False):
        super().__init__(num_train_timesteps, beta_start, beta_end, beta_schedule, trained_betas, prediction_type,
                         timestep_spacing=timestep_spacing, steps_offset=steps_offset,
                         rescale_betas_zero_snr=rescale_betas_zero_snr)
        self.config["_class_name"] = type(self).__name__

    def step(self, model_output, timestep, sample, generator=None, return_dict=True):
        _check_epsilon("EulerAncestralDiscreteScheduler", self.config.prediction_type)
        if self.step_index is None:
            self._init_step_index(timestep)
        sample = _upcast(sample)
        sigma = self.sigmas[self.step_index]
        pred_original_sample = sample - sigma * model_output
        sigma_from, sigma_to = self.sigmas[self.step_index], self.sigmas[self.step_index + 1]
        sigma_up = (sigma_to ** 2 * (sigma_from ** 2 - sigma_to ** 2) / sigma_from ** 2) ** 0.5
        sigma_down = (sigma_to ** 2 - sigma_up ** 2) ** 0.5
        derivative = (sample - pred_original_sample) / sigma
        dt = sigma_down - sigma
        prev_sample = sample + derivative * dt
        noise = _randn_like(model_output, generator)
        prev_sample = prev_sample + noise * sigma_up
        prev_sample = prev_sample.to(model_output.dtype)
        self._step_index += 1
        return _output("EulerAncestralDiscreteSchedulerOutput", return_dict, prev_sample, pred_original_sample)


class DPMSolverMultistepScheduler(_SigmaScheduler):
    """diffusers 0.25.0 DPMSolverMultistepScheduler with algorithm_type "dpmsolver++" (Lu et al. 2022, DPM-Solver++(2M)
    Alg. 2): set_timesteps (leading / trailing / linspace, optional Karras sigmas), convert_model_output,
    dpm_solver_first_order_update, multistep_dpm_solver_second_order_update (midpoint / heun), lower_order_final,
    euler_at_final. `final_sigmas_type` ("sigma_min": sqrt((1-abar_0)/abar_0), or "zero") selects the sigma after the last
    timestep; "zero" makes the last step first order. solver_order 3, SDE variants and lu lambdas are not restated.
    No fp32 upcast inside step (fp16 tensors stay fp16). Parity unpinned."""

    def __init__(self, num_train_timesteps=1000, beta_start=0.0001, beta_end=0.02, beta_schedule="linear",
                 trained_betas=None, solver_order=2, prediction_type="epsilon", thresholding=False,
                 dynamic_thresholding_ratio=0.995, sample_max_value=1.0, algorithm_type="dpmsolver++",
                 solver_type="midpoint", lower_order_final=True, euler_at_final=False, use_karras_sigmas=False,
                 use_lu_lambdas=False, final_sigmas_type="sigma_min", lambda_min_clipped=-float("inf"),
                 variance_type=None, timestep_spacing="linspace", steps_offset=0, rescale_betas_zero_snr=False):
        self._register(num_train_timesteps=num_train_timesteps, beta_start=beta_start, beta_end=beta_end,
                       beta_schedule=beta_schedule, trained_betas=trained_betas, solver_order=solver_order,
                       prediction_type=prediction_type, thresholding=thresholding, algorithm_type=algorithm_type,
                       solver_type=solver_type, lower_order_final=lower_order_final, euler_at_final=euler_at_final,
                       use_karras_sigmas=use_karras_sigmas, use_lu_lambdas=use_lu_lambdas,
                       final_sigmas_type=final_sigmas_type, lambda_min_clipped=lambda_min_clipped,
                       variance_type=variance_type, timestep_spacing=timestep_spacing, steps_offset=steps_offset,
                       rescale_betas_zero_snr=rescale_betas_zero_snr)
        if solver_type not in ("midpoint", "heun"):
            raise NotImplementedError(f"DPMSolverMultistepScheduler: solver_type {solver_type!r}")
        if final_sigmas_type not in ("sigma_min", "zero"):
            raise ValueError(f"final_sigmas_type {final_sigmas_type!r}")
        self.betas = _betas(num_train_timesteps, beta_start, beta_end, beta_schedule, trained_betas, rescale_betas_zero_snr)
        self.alphas = 1.0 - self.betas
        self.alphas_cumprod = torch.cumprod(self.alphas, dim=0)
        self.alpha_t = torch.sqrt(self.alphas_cumprod)
        self.sigma_t = torch.sqrt(1 - self.alphas_cumprod)
        self.lambda_t = torch.log(self.alpha_t) - torch.log(self.sigma_t)
        self.sigmas = ((1 - self.alphas_cumprod) / self.alphas_cumprod) ** 0.5
        self.init_noise_sigma = 1.0
        self.num_inference_steps = None
        self.timesteps = torch.from_numpy(_np.linspace(0, num_train_timesteps - 1, num_train_timesteps,
                                                       dtype=_np.float32)[::-1].copy())
        self.model_outputs = [None] * solver_order
        self.lower_order_nums = 0
        self._step_index = None

    @property
    def order(self):
        return 1

    def set_timesteps(self, num_inference_steps=None, device=None):
        c = self.config
        clipped_idx = torch.searchsorted(torch.flip(self.lambda_t, [0]), torch.tensor(c.lambda_min_clipped))
        last_timestep = int(c.num_train_timesteps - clipped_idx)
        n = num_inference_steps
        if c.timestep_spacing == "linspace":
            ts = _np.linspace(0, last_timestep - 1, n + 1).round()[::-1][:-1].copy().astype(_np.int64)
        elif c.timestep_spacing == "leading":
            ratio = last_timestep // (n + 1)
            ts = (_np.arange(0, n + 1) * ratio).round()[::-1][:-1].copy().astype(_np.int64) + c.steps_offset
        elif c.timestep_spacing == "trailing":
            ratio = c.num_train_timesteps / n
            ts = _np.arange(last_timestep, 0, -ratio).round().copy().astype(_np.int64) - 1
        else:
            raise ValueError(f"timestep_spacing {c.timestep_spacing!r}")
        sigmas = (((1 - self.alphas_cumprod) / self.alphas_cumprod) ** 0.5).numpy()
        log_sigmas = _np.log(sigmas)
        if c.use_karras_sigmas:
            sigmas = _np.flip(sigmas).copy()
            sigmas = self._convert_to_karras(in_sigmas=sigmas, num_inference_steps=n)
            ts = _np.array([self._sigma_to_t(s, log_sigmas) for s in sigmas]).round().astype(_np.int64)
        else:
            sigmas = _np.interp(ts, _np.arange(0, len(sigmas)), sigmas)
        if c.final_sigmas_type == "sigma_min":
            sigma_last = float(((1 - self.alphas_cumprod[0]) / self.alphas_cumprod[0]) ** 0.5)
        else:
            sigma_last = 0.0
        sigmas = _np.concatenate([sigmas, [sigma_last]]).astype(_np.float32)
        self.sigmas = torch.from_numpy(sigmas)                      # kept on the CPU, like diffusers
        _, unique = _np.unique(ts, return_index=True)
        ts = ts[_np.sort(unique)]
        self.timesteps = torch.from_numpy(ts).to(dtype=torch.int64)
        if device is not None:
            self.timesteps = self.timesteps.to(device)
        self.num_inference_steps = len(ts)
        self.model_outputs = [None] * c.solver_order
        self.lower_order_nums = 0
        self._step_index = None

    def scale_model_input(self, sample, *args, **kwargs):
        return sample

    @staticmethod
    def _sigma_to_alpha_sigma_t(sigma):
        alpha_t = 1 / ((sigma ** 2 + 1) ** 0.5)
        return alpha_t, sigma * alpha_t

    def _check(self):
        c = self.config
        _check_epsilon("DPMSolverMultistepScheduler", c.prediction_type, c.thresholding)
        if c.algorithm_type != "dpmsolver++":
            raise NotImplementedError(f"DPMSolverMultistepScheduler: algorithm_type {c.algorithm_type!r} is not supported")
        if c.solver_order not in (1, 2):
            raise NotImplementedError(f"DPMSolverMultistepScheduler: solver_order {c.solver_order} is not supported")
        if c.use_lu_lambdas:
            raise NotImplementedError("DPMSolverMultistepScheduler: use_lu_lambdas is not supported")

    def convert_model_output(self, model_output, sample):
        alpha_t, sigma_t = self._sigma_to_alpha_sigma_t(self.sigmas[self.step_index])
        return (sample - sigma_t * model_output) / alpha_t

    def dpm_solver_first_order_update(self, model_output, sample):
        alpha_t, sigma_t = self._sigma_to_alpha_sigma_t(self.sigmas[self.step_index + 1])
        alpha_s, sigma_s = self._sigma_to_alpha_sigma_t(self.sigmas[self.step_index])
        h = (torch.log(alpha_t) - torch.log(sigma_t)) - (torch.log(alpha_s) - torch.log(sigma_s))
        return (sigma_t / sigma_s) * sample - (alpha_t * (torch.exp(-h) - 1.0)) * model_output

    def multistep_dpm_solver_second_order_update(self, model_output_list, sample):
        alpha_t, sigma_t = self._sigma_to_alpha_sigma_t(self.sigmas[self.step_index + 1])
        alpha_s0, sigma_s0 = self._sigma_to_alpha_sigma_t(self.sigmas[self.step_index])
        alpha_s1, sigma_s1 = self._sigma_to_alpha_sigma_t(self.sigmas[self.step_index - 1])
        lambda_t = torch.log(alpha_t) - torch.log(sigma_t)
        lambda_s0 = torch.log(alpha_s0) - torch.log(sigma_s0)
        lambda_s1 = torch.log(alpha_s1) - torch.log(sigma_s1)
        m0, m1 = model_output_list[-1], model_output_list[-2]
        h, h_0 = lambda_t - lambda_s0, lambda_s0 - lambda_s1
        r0 = h_0 / h
        D0, D1 = m0, (1.0 / r0) * (m0 - m1)
        if self.config.solver_type == "midpoint":
            return ((sigma_t / sigma_s0) * sample - (alpha_t * (torch.exp(-h) - 1.0)) * D0
                    - 0.5 * (alpha_t * (torch.exp(-h) - 1.0)) * D1)
        return ((sigma_t / sigma_s0) * sample - (alpha_t * (torch.exp(-h) - 1.0)) * D0
                + (alpha_t * ((torch.exp(-h) - 1.0) / h + 1.0)) * D1)

    def step(self, model_output, timestep, sample, generator=None, return_dict=True):
        self._check()
        c = self.config
        if self.step_index is None:
            self._init_step_index(timestep)
        n = len(self.timesteps)
        lower_order_final = (self.step_index == n - 1) and (
            c.euler_at_final or (c.lower_order_final and n < 15) or c.final_sigmas_type == "zero")
        model_output = self.convert_model_output(model_output, sample=sample)
        for i in range(c.solver_order - 1):
            self.model_outputs[i] = self.model_outputs[i + 1]
        self.model_outputs[-1] = model_output
        # first order also onto sigma 0 and for a zero-length step (Karras sigmas end on sigma_min twice), where the
        # second-order term is unbounded (0/0 for "heun"); diffusers' own step gives inf / NaN there
        degenerate = self.sigmas[self.step_index + 1] == 0 or self.sigmas[self.step_index + 1] == self.sigmas[self.step_index]
        if c.solver_order == 1 or self.lower_order_nums < 1 or lower_order_final or degenerate:
            prev_sample = self.dpm_solver_first_order_update(model_output, sample=sample)
        else:
            prev_sample = self.multistep_dpm_solver_second_order_update(self.model_outputs, sample=sample)
        if self.lower_order_nums < c.solver_order:
            self.lower_order_nums += 1
        self._step_index += 1
        return _output("DPMSolverMultistepSchedulerOutput", return_dict, prev_sample, model_output)


DDPMScheduler.from_config = classmethod(_FromConfig.from_config.__func__)
