"""The denoising hot loop of IDM-VTON on the B200 engine (src/tryon_pipeline.py:1765-1866).

Per step the reference runs the garment UNet (batch Bg), zero-pads its 70 features for the CFG-uncond half, runs the
try-on UNet (batch 2B), applies CFG and the scheduler update. Here one step is a fixed launch sequence over static buffers:
  latents -> [NCHW->NHWC scatter into the 13(+pad)-channel input, x scale_model_input for Euler] -> garment UNet ->
  try-on UNet (garment K/V streamed as a second attention segment, uncond half in closed form) -> fused CFG+update
  (DDPM: b200vton_cfg_ddpm_step; DDIM / Euler / Euler-ancestral / DPM-Solver++: b200vton_cfg_sched_step, fed by the
  per-step rows of step_plan)
captured once in a CUDA graph and replayed per step; step-invariant work (cross-attention K/V of text / IP tokens,
aug_emb, the static input channels) is hoisted to prepare().
"""
import torch

from .engine import CIN_PAD, UNetEngine


class nvtx_range:
    """NVTX range around a host-side stage (visible in nsys / ncu --nvtx; a no-op cost of ~1 us otherwise)."""

    def __init__(self, name):
        self.name = name

    def __enter__(self):
        torch.cuda.nvtx.range_push(self.name)

    def __exit__(self, *a):
        torch.cuda.nvtx.range_pop()


def ddpm_step_coefficients(scheduler, t):
    """(sqrt(1-abar_t), 1/sqrt(abar_t), x0 coeff, x_t coeff, sigma_t) of DDPMScheduler.step at timestep t, computed in
    fp32 torch like diffusers does, from the GENERIC scheduler interface only — `alphas_cumprod`,
    `config.num_train_timesteps`, `num_inference_steps` (and `previous_timestep` when the object has it) — so the
    caller's own `diffusers.DDPMScheduler` works (inference.py passes `DDPMScheduler.from_pretrained(...)`). The fused
    kernel implements epsilon prediction with fixed_small variance and no clipping / thresholding: anything else raises."""
    cfg = getattr(scheduler, "config", None)
    get = (lambda k, d=None: cfg.get(k, d)) if isinstance(cfg, dict) else (lambda k, d=None: getattr(cfg, k, d))
    if get("prediction_type", "epsilon") != "epsilon" or get("variance_type", "fixed_small") != "fixed_small" \
            or get("clip_sample", False) or get("thresholding", False):
        raise NotImplementedError("the fused CFG+DDPM step covers epsilon prediction, fixed_small variance, no "
                                  "clip_sample / thresholding (the IDM-VTON scheduler config)")
    if not hasattr(scheduler, "alphas_cumprod"):
        raise TypeError(f"{type(scheduler).__name__} has no alphas_cumprod: the engine needs a DDPM-family scheduler")
    t = int(t)
    n_train = int(get("num_train_timesteps", len(scheduler.alphas_cumprod)))
    if hasattr(scheduler, "previous_timestep"):
        prev_t = int(scheduler.previous_timestep(t))
    else:
        steps = getattr(scheduler, "num_inference_steps", None) or n_train
        prev_t = t - n_train // steps
    ac = scheduler.alphas_cumprod.to(device="cpu", dtype=torch.float32)
    a_t = ac[t]
    a_prev = ac[prev_t] if prev_t >= 0 else torch.tensor(1.0)
    b_t, b_prev = 1 - a_t, 1 - a_prev
    cur_a = a_t / a_prev
    cur_b = 1 - cur_a
    c0 = (a_prev ** 0.5 * cur_b) / b_t
    c1 = cur_a ** 0.5 * b_prev / b_t
    var = torch.clamp((1 - a_prev) / (1 - a_t) * cur_b, min=1e-20)
    sigma = var ** 0.5 if t > 0 else torch.tensor(0.0)
    inv_sa = torch.tensor(1.0, dtype=torch.float32) / (a_t ** 0.5)
    return float(b_t ** 0.5), float(inv_sa), float(c0), float(c1), float(sigma)


# diffusers scheduler classes by what the engine does with them: the four it runs besides DDPM, and the known ones it
# refuses (with the reason). Any other class name takes the DDPM path (a caller's own DDPM-family object).
_SCHED_FAMILIES = {"DDPMScheduler": "ddpm", "DDIMScheduler": "ddim", "EulerDiscreteScheduler": "euler",
                   "EulerAncestralDiscreteScheduler": "euler_ancestral", "DPMSolverMultistepScheduler": "dpmsolver++"}
_TWO_EVALS = "second order: two UNet evaluations per step (needs two try-on passes and garment K/V at intermediate timesteps)"
_SCHED_REFUSED = {
    "HeunDiscreteScheduler": _TWO_EVALS, "KDPM2DiscreteScheduler": _TWO_EVALS, "KDPM2AncestralDiscreteScheduler": _TWO_EVALS,
    "DPMSolverSDEScheduler": _TWO_EVALS + " and Brownian-tree noise",
    "LMSDiscreteScheduler": "linear multistep over up to 4 stored derivatives with integrated coefficients",
    "PNDMScheduler": "pseudo-numerical multistep with a Runge-Kutta warm-up (several evaluations per timestep)",
    "UniPCMultistepScheduler": "predictor-corrector: the corrector rewrites the previous update with the new model output",
    "DEISMultistepScheduler": "multistep update over up to 3 stored predictions not covered by the fused kernel",
    "DPMSolverSinglestepScheduler": "single-step solver: intermediate UNet evaluations inside each step",
    "EDMDPMSolverMultistepScheduler": "EDM preconditioning of the model input and output",
    "EDMEulerScheduler": "EDM preconditioning of the model input and output",
    "LCMScheduler": "consistency-model boundary conditions", "TCDScheduler": "consistency-model boundary conditions",
    "IPNDMScheduler": "pseudo-numerical multistep over 4 stored derivatives",
    "DDIMInverseScheduler": "inversion (the timesteps run upwards)",
    "CMStochasticIterativeScheduler": "consistency-model sampling",
}


def _cfg_get(scheduler):
    cfg = getattr(scheduler, "config", None)
    return (lambda k, d=None: cfg.get(k, d)) if isinstance(cfg, dict) else (lambda k, d=None: getattr(cfg, k, d))


def scheduler_family(scheduler):
    """'ddpm' | 'ddim' | 'euler' | 'euler_ancestral' | 'dpmsolver++' for the caller's scheduler object, named by
    `config._class_name` when present (what diffusers' from_config records) else by its class name. Unsupported
    classes and configurations raise NotImplementedError naming the scheduler and the reason; host-only, so a caller
    can validate before any GPU work."""
    get = _cfg_get(scheduler)
    name = get("_class_name", None) or type(scheduler).__name__
    if name in _SCHED_REFUSED:
        raise NotImplementedError(f"{name} is not supported by the B200 engine: {_SCHED_REFUSED[name]}")
    fam = _SCHED_FAMILIES.get(name, "ddpm")
    if fam == "ddpm":
        return fam                         # ddpm_step_coefficients checks its own configuration
    if get("prediction_type", "epsilon") != "epsilon":
        raise NotImplementedError(f"{name}: prediction_type {get('prediction_type')!r} is not supported (epsilon only)")
    if get("thresholding", False) or get("clip_sample", False):
        raise NotImplementedError(f"{name}: thresholding / clip_sample are not supported")
    if fam == "dpmsolver++":
        if get("algorithm_type", "dpmsolver++") != "dpmsolver++":
            raise NotImplementedError(f"{name}: algorithm_type {get('algorithm_type')!r} is not supported (SDE variants "
                                      "draw noise inside the solver; only 'dpmsolver++' is fused)")
        if get("solver_order", 2) not in (1, 2):
            raise NotImplementedError(f"{name}: solver_order {get('solver_order')} is not supported (orders 1 and 2)")
        if get("use_lu_lambdas", False):
            raise NotImplementedError(f"{name}: use_lu_lambdas is not supported")
        if get("solver_type", "midpoint") not in ("midpoint", "heun"):
            raise NotImplementedError(f"{name}: solver_type {get('solver_type')!r} is not supported")
        if get("variance_type", None) in ("learned", "learned_range"):
            raise NotImplementedError(f"{name}: variance_type {get('variance_type')!r} is not supported")
    return fam


class StepPlan:
    """What the denoise loop needs from the scheduler, per step i: rows[i] (the fused kernel's coefficients after the
    guidance scale: 5 for DDPM, 7 otherwise, the last being the model-input scale), t[i] (the float timestep fed to the
    time embedding) and draws[i] (whether the reference's scheduler.step draws noise of the latents' shape)."""

    def __init__(self, family, rows, t, draws):
        self.family, self.rows, self.t, self.draws = family, rows, t, draws

    @property
    def scaled_input(self):
        return self.family in ("euler", "euler_ancestral")


def _f32(x):
    return torch.as_tensor(x, dtype=torch.float32, device="cpu")


def step_plan(scheduler, timesteps=None, eta=0.0):
    """The per-step plan of `scheduler` (after its set_timesteps) over `timesteps` (default: all of scheduler.timesteps; a
    suffix of them is allowed, as get_timesteps returns). Reads the object's own tables — timesteps, sigmas,
    alphas_cumprod, config — so spacing variants, Karras sigmas and the final-sigma convention come from it; only the
    step formulas are restated, in fp32 torch on the CPU like diffusers (see csrc/sched.cu for the row layouts). The
    scheduler object is not modified and its step() is never called."""
    fam = scheduler_family(scheduler)
    all_ts = scheduler.timesteps
    timesteps = all_ts if timesteps is None else timesteps
    T, N = len(timesteps), len(all_ts)
    off = N - T
    if T == 0 or off < 0 or [float(t) for t in all_ts[off:]] != [float(t) for t in timesteps]:
        raise ValueError("timesteps must be a suffix of scheduler.timesteps")
    t_vals = [float(t) for t in timesteps]
    if fam == "ddpm":
        rows = [list(ddpm_step_coefficients(scheduler, int(t))) for t in timesteps]
        return StepPlan(fam, rows, t_vals, [int(t) > 0 for t in timesteps])
    get = _cfg_get(scheduler)
    rows = []
    if fam == "ddim":
        ac = _f32(scheduler.alphas_cumprod)
        n_train = int(get("num_train_timesteps", len(ac)))
        n_inf = getattr(scheduler, "num_inference_steps", None) or N
        final = getattr(scheduler, "final_alpha_cumprod", None)
        final = _f32(1.0 if get("set_alpha_to_one", True) else ac[0]) if final is None else _f32(final)
        for t in timesteps:
            t = int(t)
            prev_t = t - n_train // n_inf
            a_t = ac[t]
            a_prev = ac[prev_t] if prev_t >= 0 else final
            b_t, b_prev = 1 - a_t, 1 - a_prev
            std = eta * ((b_prev / b_t) * (1 - a_t / a_prev)) ** 0.5
            cdir = (1 - a_prev - std ** 2) ** 0.5
            rows.append([float(b_t ** 0.5), float(a_t ** 0.5), float(a_prev ** 0.5), float(cdir), float(std), 0.0, 1.0])
        return StepPlan(fam, rows, t_vals, [eta > 0] * T)
    sig = _f32(scheduler.sigmas)
    if fam in ("euler", "euler_ancestral"):
        for i in range(T):
            k = off + i
            s, s_next = sig[k], sig[k + 1]
            in_scale = _f32(1.0) / ((s ** 2 + 1) ** 0.5)
            if fam == "euler":
                sigma_hat = s * (0.0 + 1)
                rows.append([float(sigma_hat), float(s_next - sigma_hat), 0.0, 0.0, 0.0, 0.0, float(in_scale)])
            else:
                up = (s_next ** 2 * (s ** 2 - s_next ** 2) / s ** 2) ** 0.5
                down = (s_next ** 2 - up ** 2) ** 0.5
                rows.append([float(s), float(down - s), float(up), 0.0, 0.0, 0.0, float(in_scale)])
        return StepPlan(fam, rows, t_vals, [True] * T)
    # DPM-Solver++ (multistep): the solver's own order schedule, replayed from a fresh set_timesteps
    order = int(get("solver_order", 2))
    heun = get("solver_type", "midpoint") == "heun"

    def a_s(x):                                         # _sigma_to_alpha_sigma_t
        alpha = 1 / ((x ** 2 + 1) ** 0.5)
        return alpha, x * alpha

    def lam(alpha, s):
        return torch.log(alpha) - torch.log(s)

    for i in range(T):
        k = off + i
        lower_final = k == N - 1 and (get("euler_at_final", False) or (get("lower_order_final", True) and N < 15)
                                      or get("final_sigmas_type", "sigma_min") == "zero")
        alpha_t, sig_t = a_s(sig[k + 1])
        alpha_s0, sig_s0 = a_s(sig[k])
        h = lam(alpha_t, sig_t) - lam(alpha_s0, sig_s0)
        c1 = alpha_t * (torch.exp(-h) - 1.0)
        ratio = sig_t / sig_s0
        c2 = rr = 0.0
        # a step onto sigma 0 (lambda = +inf, exp(-h) = 0) is taken first order: the second-order term is unbounded there;
        # so is a zero-length step (h = 0, Karras sigmas ending on sigma_min twice), where its limit is 0
        if not (order == 1 or i < 1 or lower_final or float(sig[k + 1]) == 0.0 or float(h) == 0.0):
            alpha_s1, sig_s1 = a_s(sig[k - 1])
            h_0 = lam(alpha_s0, sig_s0) - lam(alpha_s1, sig_s1)
            r0 = h_0 / h
            rr = float(1.0 / r0)
            c2 = float(alpha_t * ((torch.exp(-h) - 1.0) / h + 1.0)) if heun else -float(0.5 * c1)
        rows.append([float(sig_s0), float(alpha_s0), float(ratio), float(c1), c2, rr, 1.0])
    return StepPlan(fam, rows, t_vals, [False] * T)


def apply_plan_row(family, row, x, g, noise=None, hist=None):
    """One step of `family` with plan row `row` in the arithmetic of the input tensors (the fp64 restatement the tests
    compare with each scheduler's own step(); the engine runs the same formulas in csrc/sched.cu). Divisors are applied
    as divisions. Returns (prev, x0)."""
    if family == "ddim":
        sb, sa, sap, cdir, std = row[:5]
        x0 = (x - sb * g) / sa
        prev = sap * x0 + cdir * g
        if noise is not None and std != 0.0:
            prev = prev + std * noise
        return prev, x0
    if family in ("euler", "euler_ancestral"):
        sigma, dt = row[0], row[1]
        x0 = x - sigma * g
        prev = x + (x - x0) / sigma * dt
        if family == "euler_ancestral":
            prev = prev + row[2] * noise
        return prev, x0
    if family == "dpmsolver++":
        sig_s, alpha_s, ratio, c1, c2, rr = row[:6]
        x0 = (x - sig_s * g) / alpha_s
        prev = ratio * x - c1 * x0
        if c2 != 0.0:
            prev = prev + c2 * (rr * (x0 - hist))
        return prev, x0
    raise ValueError(family)


def garment_cache_signature(t_values, h, w):
    """What a cached garment's K/V depend on besides the garment: the timesteps the garment UNet saw (as floats, so
    Euler's non-integer timesteps get their own entries, while DDPM's keys equal the integer ones: (999.0,) == (999,))
    and the latent size."""
    return (tuple(float(t) for t in t_values), h, w)


class GarmentKVCache:
    """LRU cache of hoisted garment K/V across requests (SURVEY.md 8f item 4). One entry = the K/V of ONE garment for every
    denoise step and every try-on block ([T, Ng, 2C] fp16 per block: 4.7 GB at 768x1024 / 30 steps), keyed by the caller's
    garment id plus everything the values depend on (timestep list, latent size). A hit replaces the garment's T
    garment-UNet passes (~160 ms per garment on B200) by device-to-device copies (~2 ms)."""

    def __init__(self, max_bytes=40 << 30):
        import collections
        self.max_bytes = int(max_bytes)
        self.entries = collections.OrderedDict()
        self.bytes = 0
        self.hits = self.misses = 0

    def get(self, key):
        e = self.entries.get(key)
        if e is None:
            self.misses += 1
            return None
        self.entries.move_to_end(key)
        self.hits += 1
        return e[0]

    def put(self, key, tensors):
        n = sum(t.numel() * t.element_size() for t in tensors)
        if n > self.max_bytes:
            return
        if key in self.entries:
            self.bytes -= self.entries.pop(key)[1]
        while self.entries and self.bytes + n > self.max_bytes:
            self.bytes -= self.entries.popitem(last=False)[1][1]
        self.entries[key] = (tensors, n)
        self.bytes += n


class TryOnDenoiser:
    def __init__(self, tryon: UNetEngine, garment: UNetEngine, hoist_garment=True, garment_chunk=None, max_kv_bytes=None):
        """max_kv_bytes: budget for the resident garment K/V of the hoisted passes (default: 60% of the free device memory
        when the step tables are set). When all denoise steps do not fit (e.g. 1024x1024, 50 steps, batch 4 = 84 GB),
        the steps are hoisted window by window: K/V of `window` consecutive steps are resident at a time and the next
        window's garment passes run when the loop reaches it — same arithmetic, same graph.
        hoist_garment: the garment UNet depends on the timestep but not on the latents (SURVEY.md App. D.4), so all
        its passes are run BEFORE the loop, batched over `garment_chunk` timesteps at a time (large-M GEMMs, weights
        read once per chunk instead of once per step), and the garment K/V of every try-on block are projected once
        for all steps; the per-step graph then contains the try-on UNet only and walks the K/V by a device-side
        step index. Exactly the same arithmetic per (step, garment) as the step-by-step order."""
        self.tryon = tryon
        self.garment = garment
        self.L = tryon.L
        self.device = tryon.device
        self._graph = None
        self.hoist_garment = hoist_garment
        if garment_chunk is None:
            garment_chunk = int(__import__("os").environ.get("B200VTON_GARMENT_CHUNK", "0")) or None
        self._garment_chunk = garment_chunk      # None: as many timesteps per pass as keep the pass at <= 64 samples
        self.max_kv_bytes = max_kv_bytes
        self.gkv_all = None
        self.window = None
        self.win_start = -1

    # -------------------------------------------------------------------------------------------
    def prepare(self, latents, mask, masked_image_latents, pose_latents, cloth_latents, prompt_embeds,
                add_text_embeds, add_time_ids, image_embeds, text_embeds_cloth, guidance_scale=2.0, do_cfg=True):
        """All tensors on the device. latents [B,4,h,w]; mask [Bt,1,h,w], masked_image_latents / pose_latents
        [Bt,4,h,w], prompt_embeds [Bt,77,X], add_text_embeds [Bt,P], add_time_ids [Bt,6], image_embeds [Bt,16,X]
        with Bt = 2B under CFG ([uncond ; cond] order, src/tryon_pipeline.py:1711-1714); cloth_latents [Bg,4,h,w],
        text_embeds_cloth [Bg,77,X]."""
        torch.cuda.nvtx.range_push("b200vton.prepare(context K/V, aug_emb, static input channels)")
        try:
            self._prepare(latents, mask, masked_image_latents, pose_latents, cloth_latents, prompt_embeds, add_text_embeds,
                          add_time_ids, image_embeds, text_embeds_cloth, guidance_scale, do_cfg)
        finally:
            torch.cuda.nvtx.range_pop()

    def _prepare(self, latents, mask, masked_image_latents, pose_latents, cloth_latents, prompt_embeds, add_text_embeds,
                 add_time_ids, image_embeds, text_embeds_cloth, guidance_scale, do_cfg):
        L = self.L
        f16 = torch.float16
        B, _, h, w = latents.shape
        Bt = 2 * B if do_cfg else B
        Bg = cloth_latents.shape[0]
        dev = self.device
        key = (B, Bt, Bg, h, w, bool(do_cfg), tuple(prompt_embeds.shape), tuple(image_embeds.shape),
               tuple(text_embeds_cloth.shape))
        fresh = key != getattr(self, "_key", None)
        self._key = key
        self.B, self.Bt, self.Bg, self.h, self.w = B, Bt, Bg, h, w
        self.do_cfg = do_cfg
        self.guidance_scale = float(guidance_scale)
        if fresh:
            # (re)allocate every static buffer the step graph points at; same-shaped requests reuse them (and the
            # captured graph) and only overwrite their contents
            self._graph = None
            self.gkv_all = None
            self.latents = torch.empty((B, 4, h, w), dtype=f16, device=dev)
            self.latents_next = torch.empty_like(self.latents)
            self.noise = torch.zeros_like(self.latents)
            self.x_t = torch.zeros((Bt, h, w, CIN_PAD), dtype=f16, device=dev)
            self.x_g = torch.zeros((Bg, h, w, CIN_PAD), dtype=f16, device=dev)
            self.t_dev = torch.zeros(1, dtype=torch.float32, device=dev)
            self.coef = torch.zeros(8, dtype=torch.float32, device=dev)     # DDPM reads the first 6
            self.hist = torch.zeros_like(self.latents)       # DPM-Solver++: the previous step's x0 prediction
            self.step_base = torch.zeros(1, dtype=torch.int32, device=dev)   # step index * Bg (hoisted garment K/V)
            self.ctx_t = self.ctx_g = self.aug = None
            self.eps = None
        self.latents.copy_(latents.to(dev, f16))
        L.nchw_to_nhwc(mask.to(dev, f16).contiguous(), self.x_t, c_off=4)
        L.nchw_to_nhwc(masked_image_latents.to(dev, f16).contiguous(), self.x_t, c_off=5)
        L.nchw_to_nhwc(pose_latents.to(dev, f16).contiguous(), self.x_t, c_off=9)
        L.nchw_to_nhwc(cloth_latents.to(dev, f16).contiguous(), self.x_g, c_off=0)
        self.ctx_t = self.tryon.encode_context(prompt_embeds.to(dev, f16), image_embeds.to(dev, f16), out=self.ctx_t)
        self.ctx_g = self.garment.encode_context(text_embeds_cloth.to(dev, f16), out=self.ctx_g)
        self.aug = self.tryon.aug_embedding(add_text_embeds.to(dev, f16), add_time_ids.to(dev), out=self.aug)

    def set_step_tables(self, scheduler, timesteps, garment_keys=None, cache=None, eta=0.0, plan=None):
        """Uploads the per-step scalars of step_plan(scheduler, timesteps, eta) (or `plan`): t and the fused kernel's
        coefficient row — DDPM {gs, sqrt(1-abar), 1/sqrt(abar), c0, c1, sigma}, other schedulers see csrc/sched.cu —
        then runs the hoisted garment passes. A scheduler family other than the one the step graph was captured for
        drops the graph (recaptured at the next step). garment_keys (one hashable per garment of this batch) + cache
        (GarmentKVCache): garments whose K/V of all steps are cached are copied in instead of recomputed — valid only
        when the caller guarantees that a key identifies (cloth latents, text_embeds_cloth); the timestep list and latent
        size are added to the key here."""
        plan = plan if plan is not None else step_plan(scheduler, timesteps, eta)
        if plan.family != getattr(self, "family", None):
            self._graph = None
        self.family = plan.family
        self.plan = plan
        if plan.family == "dpmsolver++":
            self.hist.zero_()                            # no x0 prediction of an earlier request leaks in
        rows = [[self.guidance_scale, *r] for r in plan.rows]
        self.coef_table = torch.tensor(rows, dtype=torch.float32, device=self.device)
        self.t_table = torch.tensor(plan.t, dtype=torch.float32, device=self.device)
        T = len(rows)
        self.window = T
        if self.hoist_garment:
            budget = self.max_kv_bytes
            if budget is None:
                # memory this process could still use: free on the device + blocks the caching allocator holds but has
                # not handed out + the K/V buffers of the previous request, which are overwritten in place
                free, _ = torch.cuda.mem_get_info(self.device)
                cached = torch.cuda.memory_reserved(self.device) - torch.cuda.memory_allocated(self.device)
                held = sum(g.numel() * 2 for g in self.gkv_all) if self.gkv_all is not None else 0
                budget = int(0.6 * (free + cached + held))
            per_step = self.kv_bytes_per_step()
            if per_step * T > budget:
                w = max(1, budget // per_step)
                self.window = max(self.garment_chunk, w // self.garment_chunk * self.garment_chunk) if w >= self.garment_chunk else w
        self.base_table = (torch.arange(T, dtype=torch.int32, device=self.device) % self.window) * self.Bg
        if self.hoist_garment:
            use_cache = cache is not None and garment_keys is not None and len(garment_keys) == self.Bg and self.window == T
            if use_cache:
                sig = garment_cache_signature(plan.t, self.h, self.w)
                full = [(k, sig) for k in garment_keys]
                hit = [cache.get(k) for k in full]
                if all(e is not None for e in hit):
                    if self.gkv_all is None or self.gkv_all[0].shape[0] != T * self.Bg:
                        # first request of this shape (prepare() dropped the static buffers): allocate them from the cached
                        # entries' geometry instead of re-running the garment passes; the step graph is captured afterwards
                        self.gkv_all = [torch.empty((T * self.Bg, *src.shape[1:]), dtype=src.dtype, device=self.device)
                                        for src in hit[0]]
                        self._graph = None
                    for g, e in enumerate(hit):                         # timestep-major rows: row = t * Bg + g
                        for dst, src in zip(self.gkv_all, e):
                            dst.view(T, self.Bg, *dst.shape[1:])[:, g].copy_(src)
                    self.win_start = 0
                    return
            self.precompute_garment(0)
            if use_cache:
                for g, k in enumerate(full):
                    if k not in cache.entries:
                        cache.put(k, [t.view(T, self.Bg, *t.shape[1:])[:, g].clone() for t in self.gkv_all])

    @property
    def garment_chunk(self):
        """Timesteps batched into one hoisted garment-UNet pass. Measured on B200 at config 2 (2 garments): 8 -> 1096 ms per
        loop, 15 -> 1085, 30 -> 1081 (fewer, larger launches: 936 instead of 3708 eager launches per loop); default = up to
        64 samples per pass."""
        if self._garment_chunk:
            return self._garment_chunk
        return max(1, 64 // max(1, getattr(self, "Bg", 1)))

    def kv_bytes_per_step(self):
        """Bytes of garment K/V one denoise step keeps resident: sum over the try-on blocks of Bg * Ng * 2C fp16."""
        ch = self.tryon.ch
        n, lvl_tokens = (self.h, self.w), {}
        for lvl, c in enumerate(ch):
            lvl_tokens[c] = n[0] * n[1]
            n = ((n[0] - 1) // 2 + 1, (n[1] - 1) // 2 + 1)
        return sum(self.Bg * lvl_tokens[b.c] * 2 * b.c * 2 for b in self.tryon.blocks())

    def precompute_garment(self, win_start=0):
        """The garment-UNet passes of the steps [win_start, win_start + window) of the request (one per timestep), batched,
        then the garment K/V projection of every try-on block for those timesteps: gkv_all[i] = [window*Bg, Ng, 2C] in
        timestep-major order (window = all steps unless the K/V budget forces several windows)."""
        with nvtx_range(f"b200vton.garment_passes[{win_start}:{win_start + self.window}]"):
            self._precompute_garment(win_start)

    def _precompute_garment(self, win_start):
        L = self.L
        T_all, Bg = self.t_table.numel(), self.Bg
        T = min(self.window, T_all - win_start)
        blocks = self.tryon.blocks()
        gkv = self.gkv_all            # buffers of an earlier same-shaped request are overwritten in place
        if gkv is not None and gkv[0].shape[0] != min(self.window, T_all) * Bg:
            gkv = None
            self._graph = None
        self.gkv_all = None
        for c0 in range(0, T, self.garment_chunk):
            n = min(self.garment_chunk, T - c0)
            t_rows = self.t_table[win_start + c0:win_start + c0 + n].repeat_interleave(Bg).contiguous()   # timestep-major rows
            x_big = self.x_g.repeat(n, 1, 1, 1)
            ctx_big = [(kv_t.repeat(n, 1, 1), None) for kv_t, _ in self.ctx_g]
            feats = []
            self.garment.forward(x_big, self.garment.time_embedding(t_rows, n * Bg), ctx_big, collect=feats)
            if gkv is None:
                gkv = [torch.empty((min(self.window, T_all) * Bg, f.shape[1], 2 * f.shape[2]), dtype=torch.float16,
                                   device=self.device) for f in feats]
            for i, (blk, f) in enumerate(zip(blocks, feats)):
                self.tryon.garment_kv(blk, f, out=gkv[i][c0 * Bg:(c0 + n) * Bg])
            del feats, x_big, ctx_big
        self.gkv_all = gkv
        self.win_start = win_start

    # -------------------------------------------------------------------------------------------
    def _launch_step(self):
        """The launch sequence of one denoise step over the static buffers (graph-capturable)."""
        L = self.L
        if self.family in ("euler", "euler_ancestral"):
            L.nchw_to_nhwc_scaled(self.latents, self.x_t, self.coef[7:8], c_off=0)     # + scale_model_input
        else:
            L.nchw_to_nhwc(self.latents, self.x_t, c_off=0)      # CFG duplication + channel concat as offsets
        temb_t = self.tryon.time_embedding(self.t_dev, self.Bt, self.aug)
        n_persons = self.B if self.do_cfg else 0
        if self.gkv_all is not None:
            self.eps = self.tryon.forward(self.x_t, temb_t, self.ctx_t, n_persons=n_persons,
                                          gkv_pre=(self.gkv_all, self.Bg, self.step_base))
        else:
            feats = []
            temb_g = self.garment.time_embedding(self.t_dev, self.Bg)
            self.garment.forward(self.x_g, temb_g, self.ctx_g, collect=feats)
            self.eps = self.tryon.forward(self.x_t, temb_t, self.ctx_t, gfeats=feats, n_persons=n_persons)
        if self.family == "ddpm":
            L.cfg_ddpm_step(self.eps, self.latents, self.noise, self.coef, do_cfg=self.do_cfg, out=self.latents_next)
        else:
            L.cfg_sched_step(self.eps, self.latents, self.noise, self.hist, self.coef, self.family, do_cfg=self.do_cfg,
                             out=self.latents_next)
        self.latents.copy_(self.latents_next)

    # Programmatic dependent launch INSIDE the captured step only (B200VTON_PDL_GRAPH, default below): every kernel node
    # of the graph is one of this library's kernels, which call griddepcontrol.wait before they allocate tensor memory
    # or touch global memory, so the set-up of kernel n+1 overlaps the tail of kernel n (+1.3 % of the loop, round 1).
    # Eager launches — which interleave with cuBLAS / cuDNN / ATen kernels in the pipeline call, where round 1 saw two
    # stalls before the wait-before-alloc fix — keep plain stream order unless B200VTON_PDL=1 asks otherwise.
    # Round 2 on B200: 1126 -> 1116 ms per 30-step loop (profiles/r2_pdl_in_graph.json), 3 of 3 bench runs with the e2e
    # section clean; with PDL on every launch (eager ones included) 4 of 4 clean after the wait-before-alloc fix and
    # `compute-sanitizer --tool synccheck` reports no hazard. Default: ON inside the graph, OFF for eager launches.
    PDL_IN_GRAPH = __import__("os").environ.get("B200VTON_PDL_GRAPH", "1") == "1"

    def capture(self):
        """Capture one step into a CUDA graph (after a warm-up launch on a side stream)."""
        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream())
        keep = self.latents.clone()
        keep_hist = self.hist.clone() if self.family == "dpmsolver++" else None   # the warm-up launch rewrites it
        with torch.cuda.stream(s):
            self._launch_step()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        pdl_before = self.L.get_option("programmatic_launch", 0)
        if self.PDL_IN_GRAPH:
            self.L.set_option("programmatic_launch", 1)
        try:
            with torch.cuda.graph(g):
                self._launch_step()
        finally:
            if self.PDL_IN_GRAPH:
                self.L.set_option("programmatic_launch", pdl_before)
        self.latents.copy_(keep)
        if keep_hist is not None:
            self.hist.copy_(keep_hist)
        self._graph = g

    def step(self, i, noise=None, use_graph=True):
        """Runs denoise step i (tables from set_step_tables). noise: [B,4,h,w] fp16 variance noise or None."""
        if self.hoist_garment and self.gkv_all is not None and (i // self.window) * self.window != self.win_start:
            self.precompute_garment((i // self.window) * self.window)      # next K/V window (budgeted hoisting)
        self.t_dev.copy_(self.t_table[i:i + 1])
        self.coef[:self.coef_table.shape[1]].copy_(self.coef_table[i])
        self.step_base.copy_(self.base_table[i:i + 1])
        if noise is not None:
            self.noise.copy_(noise)
        else:
            self.noise.zero_()
        with nvtx_range("b200vton.denoise_step"):
            if use_graph:
                if self._graph is None:
                    self.capture()
                    self.t_dev.copy_(self.t_table[i:i + 1])
                    self.coef[:self.coef_table.shape[1]].copy_(self.coef_table[i])
                    self.step_base.copy_(self.base_table[i:i + 1])
                self._graph.replay()
            else:
                self._launch_step()
        return self.latents
