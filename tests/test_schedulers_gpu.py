"""The scheduler choice on the B200: the fused CFG + scheduler-update kernel and the scaled latent scatter against each
scheduler's host step() on the same fp16 inputs, the tiny engine's loop per scheduler (graph replay == eager, and against
the oracle loop with the paper-form steps), the pipeline per scheduler (oracle loop on the pipeline's own tensors, graph
recapture when the scheduler changes, the caller's generator state) and 3 hoisted steps at SDXL width."""
import pytest
import torch

pytestmark = pytest.mark.gpu

FAMS = ["ddim", "euler", "euler_ancestral", "dpmsolver++"]


def _sched(fam, steps, **over):
    from idm_vton_b200 import scheduler as S
    cls = {"ddim": S.DDIMScheduler, "euler": S.EulerDiscreteScheduler, "euler_ancestral": S.EulerAncestralDiscreteScheduler,
           "dpmsolver++": S.DPMSolverMultistepScheduler}[fam]
    s = cls.from_config(S.DDPMScheduler().config, **over)
    s.set_timesteps(steps)
    return s


def _err(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return (a - b).abs().max().item() / max(1.0, b.abs().max().item())


def _to(d, device, dtype):
    return {k: (v.to(device=device, dtype=dtype) if torch.is_floating_point(v) else v.to(device)) for k, v in d.items()}


# ------------------------------------------------------------------------------------------------
# kernels
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fam", FAMS)
@pytest.mark.parametrize("do_cfg", [True, False])
def test_cfg_sched_kernel_matches_host_step(fam, do_cfg):
    """Kernel vs the scheduler's own step() on the same fp16 CUDA tensors (CFG combined in fp16 torch first), at the
    first, a middle and the final step: within 1 fp16 ulp per element; the count of non-bit-equal elements is printed."""
    from idm_vton_b200 import lib as L
    from idm_vton_b200.denoise import step_plan
    from idm_vton_b200.engine import CIN_PAD
    dev, f16 = "cuda", torch.float16
    B, h, w, gs, steps = 2, 24, 20, 2.5, 20
    eta = 0.7 if fam == "ddim" else 0.0
    s = _sched(fam, steps, use_karras_sigmas=True) if fam == "dpmsolver++" else _sched(fam, steps)
    plan = step_plan(s, eta=eta)
    g = torch.Generator().manual_seed(3)
    for i in (0, steps // 2, steps - 1):
        scale = 14.0 if fam.startswith("euler") and i == 0 else 1.0
        x = (torch.randn(B, 4, h, w, generator=g) * scale).to(dev, f16)
        eps = torch.zeros(2 * B if do_cfg else B, h, w, CIN_PAD, dtype=f16, device=dev)
        eps[..., :4] = torch.randn(eps.shape[:-1] + (4,), generator=g).to(dev, f16)
        noise = torch.randn(B, 4, h, w, generator=g).to(dev, f16)
        hist = torch.randn(B, 4, h, w, generator=g).to(dev, f16)
        e_nchw = eps[..., :4].permute(0, 3, 1, 2)
        if do_cfg:
            u, c = e_nchw.chunk(2)
            guided = u + gs * (c - u)
        else:
            guided = e_nchw.contiguous()
        # host step at index i (the scheduler's own state set as after i steps)
        t = s.timesteps[i]
        kw = {}
        if fam == "ddim":
            kw = dict(eta=eta, variance_noise=noise)
        elif fam.startswith("euler"):
            s._step_index = i
            real = torch.randn
            torch.randn = lambda *a, **k: noise.clone()            # the step's own draw, replaced by the shared noise
        else:
            s._step_index = i
            s.lower_order_nums = min(i, s.config.solver_order)
            s.model_outputs = [None, hist.clone()]
        try:
            out = s.step(guided.contiguous(), t, x, **kw)
        finally:
            if fam.startswith("euler"):
                torch.randn = real
        ref = out.prev_sample
        coef = torch.tensor([gs, *plan.rows[i]], dtype=torch.float32, device=dev)
        hist_k = hist.clone()
        got = L.cfg_sched_step(eps, x, noise, hist_k, coef, fam, do_cfg=do_cfg)
        torch.cuda.synchronize()
        ulp = (torch.nextafter(ref.abs(), torch.tensor(float("inf"), dtype=f16, device=dev)) - ref.abs()).float()
        diff = (got.float() - ref.float()).abs()
        n_ne = int((got != ref).sum())
        print(f"{fam} cfg={do_cfg} step {i}: {n_ne} of {ref.numel()} elements not bit-equal, max |d|/ulp "
              f"{(diff / ulp).max().item():.2f}")
        assert torch.isfinite(got.float()).all()
        assert bool((diff <= ulp).all())
        if fam == "dpmsolver++":
            x0 = out.pred_original_sample
            assert bool(((hist_k.float() - x0.float()).abs() <= (torch.nextafter(x0.abs(), torch.tensor(float("inf"), dtype=f16, device=dev)) - x0.abs()).float()).all())


def test_scaled_scatter_matches_scale_model_input():
    from idm_vton_b200 import lib as L
    from idm_vton_b200.denoise import step_plan
    from idm_vton_b200.engine import CIN_PAD
    dev, f16 = "cuda", torch.float16
    B, h, w = 2, 16, 24
    s = _sched("euler", 30)
    plan = step_plan(s)
    x = (torch.randn(B, 4, h, w, generator=torch.Generator().manual_seed(1)) * 14).to(dev, f16)
    for i in (0, 15, 29):
        s._step_index = i
        ref = s.scale_model_input(torch.cat([x] * 2), s.timesteps[i])
        dst = torch.zeros(2 * B, h, w, CIN_PAD, dtype=f16, device=dev)
        scale = torch.tensor([plan.rows[i][-1]], dtype=torch.float32, device=dev)
        L.nchw_to_nhwc_scaled(x, dst, scale, c_off=0)
        assert torch.equal(dst[..., :4].permute(0, 3, 1, 2), ref), i
        assert dst[..., 4:].abs().max().item() == 0.0


def test_cfg_sched_rejects_bad_arguments():
    from idm_vton_b200 import lib as L
    l = L.load()
    dummy = torch.zeros(8, dtype=torch.float16, device="cuda")
    rc = l.b200vton_cfg_sched_step(dummy.data_ptr(), 8, 1, 4, 1, 1, dummy.data_ptr(), None, None, dummy.data_ptr(), 3, 1,
                                   dummy.data_ptr(), None)
    assert rc == 1 and b"history" in l.b200vton_last_error()
    rc = l.b200vton_cfg_sched_step(dummy.data_ptr(), 8, 1, 4, 1, 1, dummy.data_ptr(), None, None, dummy.data_ptr(), 7, 1,
                                   dummy.data_ptr(), None)
    assert rc == 1 and b"family" in l.b200vton_last_error()


# ------------------------------------------------------------------------------------------------
# tiny engine loop per scheduler
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tiny():
    from oracle import unet_ref as R
    from idm_vton_b200.engine import UNetEngine
    prev_tf32 = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    cfg_t, cfg_g = R.tiny_config("tryon"), R.tiny_config("garment")
    sd_t = {k: v.half() for k, v in R.make_state_dict(cfg_t, seed=11).items()}
    sd_g = {k: v.half() for k, v in R.make_state_dict(cfg_g, seed=22).items()}
    yield dict(R=R, cfg_t=cfg_t, cfg_g=cfg_g, sd_t=sd_t, sd_g=sd_g, eng_t=UNetEngine(cfg_t, sd_t, "tryon"),
               eng_g=UNetEngine(cfg_g, sd_g, "garment"))
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev_tf32


@pytest.mark.parametrize("fam", FAMS)
def test_tiny_loop_per_scheduler(tiny, fam):
    """3 steps per scheduler: graph replay == eager launches bit for bit; engine-vs-fp32 oracle <= 2 x (fp16 oracle vs
    fp32) + 2e-3, the contract of test_tiny_loop_and_graph."""
    from oracle import loop_ref as LR
    from oracle.schedulers_ref import PaperScheduler, denoise_loop
    from idm_vton_b200.denoise import TryOnDenoiser
    B, h, w, run = 2, 16, 16, 3
    steps = 20 if fam == "dpmsolver++" else 30
    eta = 0.5 if fam == "ddim" else 0.0
    sch = _sched(fam, steps)
    inp = LR.synth_loop_inputs(tiny["cfg_t"], tiny["cfg_g"], B, h, w, seed=3)
    inp["latents"] = inp["latents"] * float(sch.init_noise_sigma)
    inp = {k: (v.half().float() if k != "add_time_ids" else v) for k, v in inp.items()}
    g = torch.Generator().manual_seed(5)
    noises = [torch.randn(B, 4, h, w, generator=g).half().float() for _ in range(run)]
    dev = "cuda"
    den = TryOnDenoiser(tiny["eng_t"], tiny["eng_g"])

    def run_engine(use_graph):
        den.prepare(**{k: v.to(dev) for k, v in inp.items()}, guidance_scale=2.0)
        den.set_step_tables(sch, sch.timesteps, eta=eta)
        for i in range(run):
            den.step(i, noises[i].half().to(dev) if den.plan.draws[i] else None, use_graph=use_graph)
        torch.cuda.synchronize()
        return den.latents.clone()

    lat_eager = run_engine(False)
    lat_graph = run_engine(True)
    assert torch.equal(lat_eager, lat_graph), "graph replay must be bit-identical to eager launches"
    with torch.no_grad():
        ref = denoise_loop(_to(tiny["sd_t"], dev, torch.float32), tiny["cfg_t"], _to(tiny["sd_g"], dev, torch.float32),
                              tiny["cfg_g"], _to(inp, dev, torch.float32), steps, scheduler=PaperScheduler(_sched(fam, steps), eta),
                              noises=[n.to(dev) for n in noises], max_steps=run)
        with torch.autocast("cuda", dtype=torch.float16):
            i16 = _to(inp, dev, torch.float16)
            i16["add_time_ids"] = inp["add_time_ids"].to(dev)
            ref16 = denoise_loop(_to(tiny["sd_t"], dev, torch.float16), tiny["cfg_t"], _to(tiny["sd_g"], dev, torch.float16),
                                    tiny["cfg_g"], i16, steps, scheduler=PaperScheduler(_sched(fam, steps), eta),
                                    noises=[n.half().to(dev) for n in noises], max_steps=run)
    d_eng, d_ref = _err(lat_graph, ref), _err(ref16, ref)
    print(f"{fam} loop {run} steps: engine-32 {d_eng:.2e}, ref16-32 {d_ref:.2e}, engine-ref16 {_err(lat_graph, ref16):.2e}")
    assert d_eng <= 2 * d_ref + 2e-3


# ------------------------------------------------------------------------------------------------
# pipeline
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tiny_pipe():
    from oracle import make_golden_pipeline as MG
    from oracle import unet_ref as R
    from idm_vton_b200 import unet as U
    from idm_vton_b200.pipeline import StableDiffusionXLInpaintPipeline
    from idm_vton_b200.scheduler import DDPMScheduler
    dev, f16 = "cuda", torch.float16
    cfg_t, cfg_g = R.tiny_config("tryon"), R.tiny_config("garment")
    sd_t, sd_g = R.make_state_dict(cfg_t, seed=11), R.make_state_dict(cfg_g, seed=22)
    net_t = U.UNet2DConditionModel(cfg_t, sd_t).to(dev, f16)
    net_g = U.UNet2DConditionModelGarment(cfg_g, sd_g).to(dev, f16)
    vae = MG.make_vae().to(dev, f16)
    enc = MG.make_image_encoder(cfg_t["resampler"]["embedding_dim"]).to(dev, f16)

    def make():
        return StableDiffusionXLInpaintPipeline(vae=vae, text_encoder=None, text_encoder_2=None, tokenizer=None,
                                                tokenizer_2=None, unet=net_t, unet_encoder=net_g, scheduler=DDPMScheduler(),
                                                image_encoder=enc)

    inp = {k: (v.to(dev, f16) if k not in ("image", "mask_image") else v.to(dev)) for k, v in MG.make_call_inputs(cfg_t).items()}
    return dict(MG=MG, make=make, inp=inp, cfg_t=cfg_t, cfg_g=cfg_g, sd_t=sd_t, sd_g=sd_g)


def _call(env, pipe, steps, seed=42, eta=0.0, record=None):
    kw = env["MG"].call_kwargs(env["inp"], torch.Generator().manual_seed(seed))
    kw.update(num_inference_steps=steps, eta=eta)
    gen = kw["generator"]
    if record is not None:
        den = pipe._denoiser
        names = ("latents", "mask", "masked_image_latents", "pose_latents", "cloth_latents", "prompt_embeds",
                 "add_text_embeds", "add_time_ids", "image_embeds", "text_embeds_cloth")
        real_prepare, real_step = den.prepare, den.step

        def prepare(*a, **k):
            record["inputs"] = {n: v.detach().float().clone() for n, v in zip(names, a)}
            return real_prepare(*a, **k)

        def step(i, noise=None, use_graph=True):
            record.setdefault("noises", []).append(None if noise is None else noise.detach().float().clone())
            return real_step(i, noise, use_graph=use_graph)

        den.prepare, den.step = prepare, step
    torch.manual_seed(1234)
    try:
        pipe(**kw, output_type="pt")
    finally:
        if record is not None:
            den.prepare, den.step = real_prepare, real_step
    return pipe._last_latents.float().cpu(), gen.get_state()


@pytest.mark.parametrize("fam", FAMS)
def test_pipeline_call_per_scheduler_tracks_oracle_loop(tiny_pipe, fam):
    from oracle import loop_ref as LR
    from oracle.schedulers_ref import PaperScheduler, denoise_loop
    from idm_vton_b200.denoise import TryOnDenoiser
    env = tiny_pipe
    steps, eta = 4, (0.5 if fam == "ddim" else 0.0)
    pipe = env["make"]()
    pipe.scheduler = _sched(fam, steps).__class__.from_config(pipe.scheduler.config)
    pipe._denoiser = TryOnDenoiser(pipe.unet.engine(), pipe.unet_encoder.engine())
    rec = {}
    lat, _ = _call(env, pipe, steps, eta=eta, record=rec)
    assert len(rec["noises"]) == steps
    assert [n is not None for n in rec["noises"]] == pipe._denoiser.plan.draws
    dev = "cuda"
    sd_t32 = {k: v.half().float().to(dev) for k, v in env["sd_t"].items()}
    sd_g32 = {k: v.half().float().to(dev) for k, v in env["sd_g"].items()}
    with torch.no_grad():
        ref = denoise_loop(sd_t32, env["cfg_t"], sd_g32, env["cfg_g"], rec["inputs"], steps,
                              guidance_scale=env["MG"].GUIDANCE, scheduler=PaperScheduler(_sched(fam, steps), eta),
                              noises=rec["noises"])
    e = _err(lat, ref)
    print(f"pipeline {fam}: engine loop vs oracle loop on the pipeline's tensors {e:.2e}")
    assert e < 4e-3


def test_pipeline_scheduler_switch_recaptures_and_generator_state(tiny_pipe):
    """DDPM, then DPM-Solver++, then DDPM on ONE pipeline == fresh pipelines (the step graph is recaptured when the
    scheduler family changes); the caller's generator ends where the reference's draw sequence leaves it."""
    from idm_vton_b200 import scheduler as S
    env, steps = tiny_pipe, 4
    pipe = env["make"]()
    a, st_ddpm = _call(env, pipe, steps)
    pipe.scheduler = S.DPMSolverMultistepScheduler.from_config(pipe.scheduler.config)
    b, st_dpm = _call(env, pipe, steps)
    pipe.scheduler = S.DDPMScheduler.from_config(pipe.scheduler.config)
    c, _ = _call(env, pipe, steps)
    assert torch.equal(a, c)
    fresh = env["make"]()
    fresh.scheduler = S.DPMSolverMultistepScheduler.from_config(fresh.scheduler.config)
    b2, _ = _call(env, fresh, steps)
    assert torch.equal(b, b2) and not torch.equal(a, b)
    # generator: DPM-Solver++ draws no step noise, DDPM one latents-shaped fp16 draw per step (t > 0), Euler every step
    lat_shape = tuple(a.shape)
    gen = torch.Generator()
    gen.set_state(st_dpm)
    for _ in range(steps):
        torch.randn(lat_shape, generator=gen, dtype=torch.float16)
    assert torch.equal(gen.get_state(), st_ddpm)
    pipe.scheduler = S.EulerDiscreteScheduler.from_config(pipe.scheduler.config)
    _, st_euler = _call(env, pipe, steps)
    assert torch.equal(st_euler, st_ddpm)
    pipe.scheduler = S.DDIMScheduler.from_config(S.DDPMScheduler().config)   # (DDIM's own default clips the sample)
    _, st_ddim0 = _call(env, pipe, steps, eta=0.0)
    assert torch.equal(st_ddim0, st_dpm)
    # unsupported schedulers raise before any GPU work
    heun = type("HeunDiscreteScheduler", (), {})()
    heun.config = {}
    pipe.scheduler = heun
    with pytest.raises(NotImplementedError, match="HeunDiscreteScheduler"):
        _call(env, pipe, steps)


# ------------------------------------------------------------------------------------------------
# full size
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fam", ["euler", "dpmsolver++"])
def test_fullsize_hoisted_loop_per_scheduler(fam):
    """3 hoisted steps at config-2 shapes (128x96 latents, B = 2) at SDXL width: engine-vs-ref32 <= ref16-vs-ref32 + 2.5e-4."""
    from oracle import loop_ref as LR
    from oracle import unet_ref as R
    from oracle.schedulers_ref import PaperScheduler, denoise_loop
    from idm_vton_b200 import unet as U
    from idm_vton_b200.denoise import TryOnDenoiser
    from idm_vton_b200.engine import SDXL_GARMENT, SDXL_TRYON, UNetEngine
    prev_tf32 = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    try:
        dev = "cuda"
        sd_t = U.random_state_dict(SDXL_TRYON, seed=11, device=dev)
        sd_g = U.random_state_dict(SDXL_GARMENT, seed=22, device=dev)
        B, h, w, run = 2, 128, 96, 3
        steps = 20 if fam == "dpmsolver++" else 30
        sch = _sched(fam, steps)
        inp = LR.synth_loop_inputs(SDXL_TRYON, SDXL_GARMENT, B, h, w, seed=3)
        inp["latents"] = inp["latents"] * float(sch.init_noise_sigma)
        inp = {k: (v.half().float() if k != "add_time_ids" else v).to(dev) for k, v in inp.items()}
        den = TryOnDenoiser(UNetEngine(SDXL_TRYON, sd_t, "tryon"), UNetEngine(SDXL_GARMENT, sd_g, "garment"))
        den.prepare(**inp, guidance_scale=2.0)
        den.set_step_tables(sch, sch.timesteps)
        g = torch.Generator().manual_seed(5)
        noises = [torch.randn(B, 4, h, w, generator=g).half().float().to(dev) for _ in range(run)]
        for i in range(run):
            den.step(i, noises[i].half() if den.plan.draws[i] else None, use_graph=True)
        torch.cuda.synchronize()
        lat = den.latents.clone()
        del den
        with torch.no_grad():
            sd_t32 = {k: v.float() for k, v in sd_t.items()}
            sd_g32 = {k: v.float() for k, v in sd_g.items()}
            ref = denoise_loop(sd_t32, SDXL_TRYON, sd_g32, SDXL_GARMENT, inp, steps, scheduler=PaperScheduler(_sched(fam, steps)),
                                  noises=noises, max_steps=run)
            del sd_t32, sd_g32
            with torch.autocast("cuda", dtype=torch.float16):
                i16 = {k: (v.half() if k != "add_time_ids" else v) for k, v in inp.items()}
                ref16 = denoise_loop(sd_t, SDXL_TRYON, sd_g, SDXL_GARMENT, i16, steps,
                                        scheduler=PaperScheduler(_sched(fam, steps)), noises=[n.half() for n in noises],
                                        max_steps=run)
        d_eng32, d_ref32, d_eng16 = _err(lat, ref), _err(ref16, ref), _err(lat, ref16)
        print(f"PARITY fullsize {fam} {run} of {steps} steps B={B} {h}x{w}: eng_vs_32 {d_eng32:.2e} ref16_vs_32 {d_ref32:.2e} "
              f"eng_vs_ref16 {d_eng16:.2e}")
        assert d_eng32 <= d_ref32 + 2.5e-4
    finally:
        torch.cuda.empty_cache()
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev_tf32
