"""Scheduler choice on the host (no GPU): the per-step plan the engine runs (denoise.step_plan) against each scheduler's
own step(), fp64 cross-identities between the schedulers, the oracle's paper-form steps, convergence orders on an exact
probability-flow ODE, noise-draw plans, garment-cache keys and the configurations that are refused."""
import math

import numpy as np
import pytest
import torch

from idm_vton_b200 import scheduler as S
from idm_vton_b200.denoise import apply_plan_row, garment_cache_signature, scheduler_family, step_plan

CLASSES = {"ddim": S.DDIMScheduler, "euler": S.EulerDiscreteScheduler, "euler_ancestral": S.EulerAncestralDiscreteScheduler,
           "dpmsolver++": S.DPMSolverMultistepScheduler}
SHAPE = (2, 4, 3, 5)


def _make(fam, steps, **over):
    """The usual switching idiom: <Class>.from_config(<IDM-VTON DDPM scheduler>.config), then set_timesteps."""
    s = CLASSES[fam].from_config(S.DDPMScheduler().config, **over)
    s.set_timesteps(steps)
    return s


def _run_both(s, plan, fam, seed=0, eta=0.0):
    """Steps the scheduler object with its own step() in fp64 and the plan rows with apply_plan_row; returns the worst
    relative difference over all steps."""
    g = torch.Generator().manual_seed(seed)
    worst, hist = 0.0, None
    for i, t in enumerate(s.timesteps):
        x = torch.randn(SHAPE, generator=g, dtype=torch.float64) * 3
        e = torch.randn(SHAPE, generator=g, dtype=torch.float64)
        kw, noise = {}, None
        if fam == "ddim":
            noise = torch.randn(SHAPE, generator=g, dtype=torch.float64)
            kw = dict(eta=eta, variance_noise=noise)
        elif fam in ("euler", "euler_ancestral"):
            gen = torch.Generator().manual_seed(1000 + i)
            noise = torch.randn(SHAPE, generator=torch.Generator().manual_seed(1000 + i), dtype=torch.float64)
            kw = dict(generator=gen)
        ref = s.step(e, t, x, **kw).prev_sample
        got, x0 = apply_plan_row(fam, plan.rows[i], x, e, noise=noise, hist=hist)
        hist = x0
        worst = max(worst, ((got - ref).abs().max() / max(1.0, ref.abs().max())).item())
    return worst


@pytest.mark.parametrize("fam", list(CLASSES))
@pytest.mark.parametrize("spacing", ["leading", "trailing", "linspace"])
def test_plan_reproduces_step(fam, spacing):
    """Plan == step: for every step count and step index (DPM-Solver++'s first and lower-order final steps included)
    the plan's coefficients applied in fp64 reproduce the class's own step() to 1e-12."""
    for steps in (5, 14, 20, 30, 50):
        s = _make(fam, steps, timestep_spacing=spacing)
        for eta in ((0.0, 0.6, 1.0) if fam == "ddim" else (0.0,)):
            s.set_timesteps(steps)
            plan = step_plan(s, eta=eta)
            assert plan.family == fam and len(plan.rows) == len(s.timesteps)
            err = _run_both(s, plan, fam, seed=steps, eta=eta)
            assert err < 1e-12, (fam, spacing, steps, eta, err)


@pytest.mark.parametrize("over", [dict(solver_order=1), dict(solver_type="heun"), dict(lower_order_final=False),
                                  dict(euler_at_final=True), dict(use_karras_sigmas=True), dict(final_sigmas_type="zero"),
                                  dict(use_karras_sigmas=True, final_sigmas_type="zero", solver_type="heun"),
                                  dict(use_karras_sigmas=True, solver_type="heun", lower_order_final=False)])
def test_plan_reproduces_step_dpm_variants(over):
    for steps in (5, 14, 20, 30):
        s = _make("dpmsolver++", steps, **over)
        plan = step_plan(s)
        assert all(math.isfinite(v) for r in plan.rows for v in r)
        assert _run_both(s, plan, "dpmsolver++", seed=steps) < 1e-12, (over, steps)
        orders = [2 if r[4] != 0.0 else 1 for r in plan.rows]
        assert orders[0] == 1 and (over.get("solver_order") != 1 or set(orders) == {1})


def test_plan_reproduces_step_euler_karras():
    for fam in ("euler",):
        for steps in (5, 20, 30):
            s = _make(fam, steps, use_karras_sigmas=True)
            assert any(float(t) != int(t) for t in s.timesteps)         # non-integer timesteps
            plan = step_plan(s)
            assert plan.t == [float(t) for t in s.timesteps]
            assert _run_both(s, plan, fam, seed=steps) < 1e-12


def _foreign(s):
    """An object with only diffusers' attribute surface: class name, config dict, tables."""
    cls = type(type(s).__name__, (), {})
    o = cls()
    o.config = {k: v for k, v in s.config.items()}
    for k in ("timesteps", "sigmas", "alphas_cumprod", "num_inference_steps", "final_alpha_cumprod"):
        if hasattr(s, k):
            setattr(o, k, getattr(s, k))
    return o


@pytest.mark.parametrize("fam", list(CLASSES))
def test_foreign_object_gives_the_same_plan(fam):
    s = _make(fam, 20)
    a, b = step_plan(s, eta=0.5), step_plan(_foreign(s), eta=0.5)
    assert a.family == b.family == fam and a.rows == b.rows and a.t == b.t and a.draws == b.draws
    # the plan leaves the caller's object unmodified
    before = (s.timesteps.clone(), getattr(s, "_step_index", None), getattr(s, "lower_order_nums", None))
    step_plan(s)
    assert torch.equal(s.timesteps, before[0]) and getattr(s, "_step_index", None) == before[1]
    assert getattr(s, "lower_order_nums", None) == before[2]
    # class name taken from config._class_name (what from_config records)
    o = _foreign(s)
    o.__class__ = type("Wrapper", (), {})
    assert scheduler_family(o) == fam


def test_suffix_of_the_timesteps():
    s = _make("euler", 10)
    full, tail = step_plan(s), step_plan(s, s.timesteps[3:])
    assert tail.rows == full.rows[3:] and tail.t == full.t[3:]
    with pytest.raises(ValueError):
        step_plan(s, s.timesteps[:3])


def test_ddim_eta1_equals_ddpm_step():
    """DDIM with eta = 1 is the DDPM ancestral step (same timesteps, same noise): ties the new code to the pinned DDPM."""
    ddpm = S.DDPMScheduler()
    ddpm.set_timesteps(30)
    ddim = _make("ddim", 30)
    assert ddim.timesteps.tolist() == ddpm.timesteps.tolist()
    g = torch.Generator().manual_seed(0)
    for t in ddpm.timesteps:
        x = torch.randn(SHAPE, generator=g, dtype=torch.float64)
        e = torch.randn(SHAPE, generator=g, dtype=torch.float64)
        a = ddpm.step(e, t, x, generator=torch.Generator().manual_seed(int(t))).prev_sample
        b = ddim.step(e, t, x, eta=1.0, variance_noise=ddpm._last_noise).prev_sample
        assert (a - b).abs().max().item() < 2e-5 * max(1.0, a.abs().max().item()), int(t)


def test_dpm_order1_equals_ddim_eta0():
    """DPM-Solver++ with solver_order 1 is DDIM with eta = 0 (Lu et al. 2022, Sec. 4): same timesteps (trailing spacing),
    DDIM's final alpha = abar_0 matching DPM-Solver's final sigma."""
    for steps in (10, 20, 25, 50):
        dpm = _make("dpmsolver++", steps, solver_order=1, timestep_spacing="trailing")
        ddim = _make("ddim", steps, timestep_spacing="trailing", set_alpha_to_one=False)
        assert dpm.timesteps.tolist() == ddim.timesteps.tolist()
        g = torch.Generator().manual_seed(steps)
        for t in ddim.timesteps:
            x = torch.randn(SHAPE, generator=g, dtype=torch.float64)
            e = torch.randn(SHAPE, generator=g, dtype=torch.float64)
            a = ddim.step(e, t, x, eta=0.0).prev_sample
            b = dpm.step(e, t, x).prev_sample
            assert (a - b).abs().max().item() < 2e-5 * max(1.0, a.abs().max().item())


@pytest.mark.parametrize("fam,over", [("ddim", {}), ("ddim", {"eta": 0.8}), ("euler", {}), ("euler_ancestral", {}),
                                      ("dpmsolver++", {}), ("dpmsolver++", {"solver_type": "heun"}),
                                      ("dpmsolver++", {"final_sigmas_type": "zero"})])
def test_product_steps_agree_with_paper_forms(fam, over):
    from oracle.schedulers_ref import PaperScheduler
    over = dict(over)
    eta = over.pop("eta", 0.0)
    for steps in (7, 20):
        s = _make(fam, steps, **over)
        ref = PaperScheduler(CLASSES[fam].from_config(s.config), eta=eta)
        ref.set_timesteps(steps)
        g = torch.Generator().manual_seed(steps)
        for i, t in enumerate(s.timesteps):
            x = torch.randn(SHAPE, generator=g, dtype=torch.float64)
            e = torch.randn(SHAPE, generator=g, dtype=torch.float64)
            noise = torch.randn(SHAPE, generator=torch.Generator().manual_seed(i), dtype=torch.float64)
            kw = dict(eta=eta, variance_noise=noise) if fam == "ddim" else (
                dict(generator=torch.Generator().manual_seed(i)) if fam.startswith("euler") else {})
            a = s.step(e, t, x, **kw).prev_sample
            b = ref.step(e, t, x, noise=noise)
            assert (a - b).abs().max().item() < 1e-5 * max(1.0, b.abs().max().item()), (fam, steps, i)


def _ode_error(fam, n, s_data=0.5, **over):
    """Endpoint error of the plan's arithmetic (fp64) on data x0 ~ N(0, s^2): the exact eps-prediction is
    eps(x_in, sigma) = sigma sqrt(1+sigma^2) x_in / (s^2 + sigma^2) (x_in = the VP sample = the UNet input), and the
    probability-flow ODE scales the VE sample by sqrt(s^2 + sigma^2), from the run's first sigma to its last."""
    sch = _make(fam, n, timestep_spacing="leading", **over)
    plan = step_plan(sch)
    sigma_of = {"ddim": lambda r: r[0] / r[1], "euler": lambda r: r[0], "dpmsolver++": lambda r: r[0] / r[1]}[fam]
    x = torch.ones(1, dtype=torch.float64)
    x_start, hist = x.clone(), None
    for r in plan.rows:
        sig = sigma_of(r)
        x_in = x * r[-1] if fam == "euler" else x
        eps = sig * math.sqrt(1 + sig ** 2) * x_in / (s_data ** 2 + sig ** 2)
        x, hist = apply_plan_row(fam, r, x, eps, hist=hist)
    sig0 = sigma_of(plan.rows[0])
    if fam == "ddim":
        a_f = 1.0                                             # set_alpha_to_one
        sig_end = math.sqrt((1 - a_f) / a_f)
    else:
        sig_end = float(sch.sigmas[len(plan.rows)])               # where the last step lands
    ratio = math.sqrt(s_data ** 2 + sig_end ** 2) / math.sqrt(s_data ** 2 + sig0 ** 2)
    if fam != "euler":                                         # VP sample = VE sample / sqrt(1 + sigma^2)
        ratio *= math.sqrt(1 + sig0 ** 2) / math.sqrt(1 + sig_end ** 2)
    return abs(float(x) - ratio * float(x_start))


@pytest.mark.parametrize("fam,over,lo", [("ddim", {}, 0.8), ("euler", {}, 0.8), ("dpmsolver++", {"solver_order": 1}, 0.8),
                                         ("dpmsolver++", {"solver_order": 1, "use_karras_sigmas": True}, 0.8),
                                         ("dpmsolver++", {"solver_order": 2, "use_karras_sigmas": True}, 1.7),
                                         ("dpmsolver++", {"solver_order": 2, "use_karras_sigmas": True, "solver_type": "heun"},
                                          1.7)])
def test_convergence_order_on_exact_ode(fam, over, lo):
    """Fitted order of the endpoint error over N = 10, 20, 40, 80 steps: about 1 for DDIM, Euler and DPM-Solver++(1),
    about 2 for DPM-Solver++(2M). The second-order runs use Karras sigmas: on a uniform timestep grid the final step
    onto sigma(t=0) does not shrink in lambda as N grows, which caps any method at first order."""
    ns = [10, 20, 40, 80]
    errs = [_ode_error(fam, n, **over) for n in ns]
    slope = -np.polyfit(np.log(ns), np.log(errs), 1)[0]
    print(f"{fam} {over}: errors {['%.3e' % e for e in errs]} order {slope:.2f}")
    assert slope >= lo, (errs, slope)


def test_noise_draw_plans():
    ddpm = S.DDPMScheduler()
    ddpm.set_timesteps(10)
    assert step_plan(ddpm).draws == [int(t) > 0 for t in ddpm.timesteps]
    ddim = _make("ddim", 10)
    assert step_plan(ddim, eta=0.0).draws == [False] * 10 and step_plan(ddim, eta=0.3).draws == [True] * 10
    assert step_plan(_make("euler", 10)).draws == [True] * 10            # drawn (and unused) every step
    assert step_plan(_make("euler_ancestral", 10)).draws == [True] * 10
    assert step_plan(_make("dpmsolver++", 10)).draws == [False] * 10
    # input scaling only for the Euler families
    assert [step_plan(_make(f, 10)).scaled_input for f in CLASSES] == [False, True, True, False]


def test_garment_cache_keys():
    ddpm = S.DDPMScheduler()
    ddpm.set_timesteps(30)
    plan = step_plan(ddpm)
    today = (tuple(int(t) for t in ddpm.timesteps), 128, 96)              # the keys DDPM requests were cached under
    assert garment_cache_signature(plan.t, 128, 96) == today and hash(garment_cache_signature(plan.t, 128, 96)) == hash(today)
    e = step_plan(_make("euler", 30, timestep_spacing="linspace"))
    sig = garment_cache_signature(e.t, 128, 96)
    assert any(t != int(t) for t in e.t)
    assert sig != garment_cache_signature([int(t) for t in e.t], 128, 96)


@pytest.mark.parametrize("name", ["HeunDiscreteScheduler", "KDPM2DiscreteScheduler", "KDPM2AncestralDiscreteScheduler",
                                  "LMSDiscreteScheduler", "PNDMScheduler", "UniPCMultistepScheduler",
                                  "DEISMultistepScheduler", "DPMSolverSinglestepScheduler", "DPMSolverSDEScheduler"])
def test_unsupported_scheduler_classes_raise(name):
    o = type(name, (), {})()
    o.config = {"prediction_type": "epsilon"}
    with pytest.raises(NotImplementedError, match=name):
        scheduler_family(o)
    with pytest.raises(NotImplementedError, match=name):
        step_plan(o)


@pytest.mark.parametrize("fam,over,what", [
    ("dpmsolver++", {"algorithm_type": "sde-dpmsolver++"}, "algorithm_type"),
    ("dpmsolver++", {"algorithm_type": "sde-dpmsolver"}, "algorithm_type"),
    ("dpmsolver++", {"solver_order": 3}, "solver_order"),
    ("dpmsolver++", {"use_lu_lambdas": True}, "use_lu_lambdas"),
    ("ddim", {"prediction_type": "v_prediction"}, "prediction_type"),
    ("euler", {"prediction_type": "v_prediction"}, "prediction_type"),
    ("euler_ancestral", {"prediction_type": "sample"}, "prediction_type"),
    ("dpmsolver++", {"prediction_type": "v_prediction"}, "prediction_type"),
    ("ddim", {"thresholding": True}, "thresholding"),
    ("dpmsolver++", {"thresholding": True}, "thresholding"),
    ("ddim", {"clip_sample": True}, "clip_sample"),
])
def test_unsupported_configurations_raise(fam, over, what):
    s = CLASSES[fam].from_config(S.DDPMScheduler().config)
    s.set_timesteps(10)
    o = _foreign(s)
    o.config.update(over)
    with pytest.raises(NotImplementedError, match=what):
        step_plan(o)


def test_unknown_class_takes_the_ddpm_path():
    class Foreign:
        def __init__(self):
            self.alphas_cumprod = S.DDPMScheduler().alphas_cumprod
            self.config = dict(num_train_timesteps=1000, prediction_type="epsilon", variance_type="fixed_small",
                               clip_sample=False)
            self.num_inference_steps = 30
            self.timesteps = torch.tensor([967, 934])
    s = S.DDPMScheduler()
    s.set_timesteps(30)
    p = step_plan(Foreign())
    assert p.family == "ddpm" and p.rows[0] == list(s.step_coefficients(967)) and p.t == [967.0, 934.0]


def test_from_config_switching_and_surface():
    base = S.DDPMScheduler()
    for fam, cls in CLASSES.items():
        s = cls.from_config(base.config)
        assert s.config["_class_name"] == cls.__name__ and s.config.beta_schedule == "scaled_linear"
        t = cls.from_config(s.config)                   # round trip through another scheduler's config
        assert dict(t.config) == dict(s.config)
        s.set_timesteps(10)
        x = torch.randn(1, 4, 2, 2)
        y = s.scale_model_input(x, s.timesteps[0])
        if fam.startswith("euler"):
            assert torch.allclose(y, x / (s.sigmas[0] ** 2 + 1) ** 0.5) and float(s.init_noise_sigma) > 1
        else:
            assert y is x and s.init_noise_sigma == 1.0
        assert s.order == 1


def test_diffusers_classes_if_available():
    """The plan against the real diffusers classes' step() (runs only where diffusers is installed)."""
    diffusers = pytest.importorskip("diffusers")
    cfg = dict(num_train_timesteps=1000, beta_start=0.00085, beta_end=0.012, beta_schedule="scaled_linear",
               steps_offset=1, clip_sample=False, set_alpha_to_one=False, timestep_spacing="leading")
    for name in ("DDIMScheduler", "EulerDiscreteScheduler", "EulerAncestralDiscreteScheduler", "DPMSolverMultistepScheduler"):
        s = getattr(diffusers, name).from_config(cfg)
        for steps in (5, 20, 30):
            s.set_timesteps(steps)
            plan = step_plan(s, eta=0.0)
            g = torch.Generator().manual_seed(steps)
            hist = None
            for i, t in enumerate(s.timesteps):
                x = torch.randn(SHAPE, generator=g) * 3
                e = torch.randn(SHAPE, generator=g)
                noise = torch.randn(SHAPE, generator=torch.Generator().manual_seed(i))
                kw = {"generator": torch.Generator().manual_seed(i)} if name.startswith("Euler") else {}
                ref = s.step(e, t, x, **kw).prev_sample
                got, hist = apply_plan_row(plan.family, plan.rows[i], x, e, noise=noise, hist=hist)
                assert (got - ref).abs().max().item() < 1e-4 * max(1.0, ref.abs().max().item()), (name, steps, i)


def test_scheduler_loop_oracle_matches_pinned_ddpm_loop():
    """oracle.schedulers_ref.denoise_loop with the paper-form DDIM at eta = 1 (= the DDPM ancestral step, same timesteps and
    noises) reproduces loop_ref.denoise_loop with DDPMRef, the loop oracle pinned by the reference pipeline: ties the
    scheduler-generic loop (scale_model_input, float timesteps) to the pinned one."""
    from oracle import loop_ref as LR
    from oracle import unet_ref as R
    from oracle.schedulers_ref import PaperScheduler, denoise_loop
    cfg_t, cfg_g = R.tiny_config("tryon"), R.tiny_config("garment")
    sd_t, sd_g = R.make_state_dict(cfg_t, seed=11), R.make_state_dict(cfg_g, seed=22)
    B, h, w, steps, run = 1, 8, 8, 30, 2
    inp = LR.synth_loop_inputs(cfg_t, cfg_g, B, h, w, seed=4)
    g = torch.Generator().manual_seed(6)
    noises = [torch.randn(B, 4, h, w, generator=g) for _ in range(run)]
    with torch.no_grad():
        ref = LR.denoise_loop(sd_t, cfg_t, sd_g, cfg_g, inp, steps, noises=noises, max_steps=run)
        got = denoise_loop(sd_t, cfg_t, sd_g, cfg_g, inp, steps, scheduler=PaperScheduler(_make("ddim", steps), eta=1.0),
                           noises=noises, max_steps=run)
    e = (got - ref).abs().max().item() / max(1.0, ref.abs().max().item())
    assert e < 1e-5, e
