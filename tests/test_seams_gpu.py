"""GPU parity of the drop-in seams (SURVEY.md 8b) against outputs of the REFERENCE's own code (tests/golden/*.pt, made by
oracle/make_golden.py and oracle/make_golden_seams.py with /root/reference imported in place):

  B3  attention-processor protocol : AttnProcessor2_0 / IPAttnProcessor2_0 (ip_adapter/attention_processor.py:189-278,
      1879-2010) called as `processor(attn, hidden_states, encoder_hidden_states, ...)`; `set_attn_processor`
  a12 Resampler                    : `unet.encoder_hid_proj(x)` (ip_adapter/resampler.py, src/tryon_pipeline.py:1726)
  B2  UNet modules                 : `UNet2DConditionModel.forward(..., garment_features=<reference-format, zero-padded>)`
      and the garment UNet's `forward(...) -> ((sample,), features)` (src/tryon_pipeline.py:1787-1808)
Tolerances: the golden tensors are fp32 CPU results of the reference modules; the engine computes in fp16 with fp32
accumulation, so gates are a few fp16 ulp of the output scale (stated per test).
"""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

G = os.path.join(os.path.dirname(__file__), "golden")


def _err(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return (a - b).abs().max().item() / max(1.0, b.abs().max().item())


def _attention_from(weights, C, heads, cross=None, processor=None):
    from idm_vton_b200.attention_processor import Attention
    a = Attention(query_dim=C, cross_attention_dim=cross, heads=heads, processor=processor, device="cuda", dtype=torch.float16)
    sd = {k: v for k, v in weights.items() if not k.startswith("to_k_ip") and not k.startswith("to_v_ip")}
    a.load_state_dict({k: v.cuda().half() for k, v in sd.items()}, strict=False)
    return a


# ------------------------------------------------------------------------------------------------
# B3
# ------------------------------------------------------------------------------------------------
def test_attn_processors_vs_reference_golden():
    from idm_vton_b200.attention_processor import AttnProcessor2_0, IPAttnProcessor2_0
    g = torch.load(os.path.join(G, "attn_processors_ref.pt"))
    C, heads = g["C"], g["heads"]
    cross = g["cross"]["weights"]["to_k.weight"].shape[1]      # (the fixture's "cross" entry is the cross-attention case)
    # self-attention
    s = g["self"]
    a1 = _attention_from(s["weights"], C, heads)
    y = a1(s["x"].cuda())
    e_self = _err(y, s["y"])
    # plain cross-attention (the garment UNet's attn2)
    c = g["cross"]
    a2 = _attention_from(c["weights"], C, heads, cross, AttnProcessor2_0())
    e_cross = _err(a2(c["x"].cuda(), encoder_hidden_states=c["enc"].cuda()), c["y"])
    # decoupled text + IP cross-attention, scale 1.0 (inference) and 0.5
    i = torch.load(os.path.join(G, "attn_processors_ip_ref.pt"))["ip"]
    errs = []
    for scale, key in ((1.0, "y_scale_1"), (0.5, "y_scale_0p5")):
        proc = IPAttnProcessor2_0(hidden_size=C, cross_attention_dim=cross, scale=scale, num_tokens=i["num_tokens"],
                                  device="cuda", dtype=torch.float16)
        proc.load_state_dict({k: i["weights"][k].cuda().half() for k in ("to_k_ip.weight", "to_v_ip.weight")})
        a3 = _attention_from(i["weights"], C, heads, cross, proc)
        assert "processor.to_k_ip.weight" in a3.state_dict()          # ...attn2.processor.to_k_ip.weight (:1904-1905)
        errs.append(_err(a3(i["x"].cuda(), encoder_hidden_states=i["enc"].cuda()), i[key]))
    print(f"B3 vs reference processors: self {e_self:.2e} cross {e_cross:.2e} ip(1.0) {errs[0]:.2e} ip(0.5) {errs[1]:.2e}")
    assert max(e_self, e_cross, *errs) < 2e-3


def test_processor_accepts_foreign_attention_container():
    """The protocol only needs `attn.to_q/.to_k/.to_v/.to_out[0]` with `.weight` and `attn.heads` — e.g. a diffusers
    `Attention` built from nn.Linear layers — not this package's container class."""
    import torch.nn as nn
    from idm_vton_b200.attention_processor import AttnProcessor2_0
    g = torch.load(os.path.join(G, "attn_processors_ref.pt"))
    s, C = g["self"], g["C"]

    class Foreign(nn.Module):
        def __init__(self):
            super().__init__()
            self.heads = g["heads"]
            self.to_q, self.to_k, self.to_v = (nn.Linear(C, C, bias=False) for _ in range(3))
            self.to_out = nn.ModuleList([nn.Linear(C, C), nn.Dropout(0.0)])
            self.spatial_norm = self.group_norm = self.norm_cross = None
            self.residual_connection, self.rescale_output_factor = False, 1.0

    f = Foreign()
    f.load_state_dict({k: v.float() for k, v in s["weights"].items()})
    f = f.cuda().half()
    y = AttnProcessor2_0()(f, s["x"].cuda())
    assert _err(y, s["y"]) < 2e-3
    with pytest.raises(RuntimeError):
        AttnProcessor2_0()(f.float(), s["x"].cuda().float())      # fp32: no PyTorch fallback
    with pytest.raises(NotImplementedError):
        AttnProcessor2_0()(f.half(), s["x"].cuda(), attention_mask=torch.ones(1, device="cuda"))


def test_protocol_path_equals_fused_hacked_self_attention():
    """src/attentionhacked_tryon.py:334-348 through the protocol — attn1(cat([norm_hidden, garment_feature], 1))[:, :N] —
    equals the engine's fused formulation (Q rows = N only, garment K/V streamed as a second segment, no cat)."""
    from idm_vton_b200 import lib as L
    from idm_vton_b200.attention_processor import Attention
    C, heads, B, N = 1280, 20, 2, 768
    gen = torch.Generator(device="cuda").manual_seed(3)
    r = lambda *s, sc=1.0: (torch.randn(*s, generator=gen, device="cuda") * sc).half()  # noqa: E731
    attn = Attention(query_dim=C, heads=heads, device="cuda", dtype=torch.float16)
    for n, p in attn.named_parameters():
        p.data.copy_(r(*p.shape, sc=(C ** -0.5 if p.ndim == 2 else 0.1)))
    n1, gf = r(B, N, C), r(B, N, C)
    y_protocol = attn(torch.cat([n1, gf], dim=1))[:, :N]
    wqkv = torch.cat([attn.to_q.weight, attn.to_k.weight, attn.to_v.weight], 0).contiguous()
    qkv = L.gemm(n1.view(B * N, C), wqkv).view(B, N, 3 * C)
    gkv = L.gemm(gf.view(B * N, C), wqkv[C:]).view(B, N, 2 * C)
    a = L.attention(qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:], gkv[..., :C], gkv[..., C:], kv1_off=0, heads=heads)
    y_fused = L.gemm(a.view(B * N, C), attn.to_out[0].weight, bias=attn.to_out[0].bias).view(B, N, C)
    e = _err(y_fused, y_protocol)
    print(f"hacked self-attention: fused vs protocol {e:.2e}")
    assert e < 1e-3


@pytest.fixture(scope="module")
def tiny_modules():
    from oracle import unet_ref as R
    from idm_vton_b200 import unet as U
    cfg_t, cfg_g = R.tiny_config("tryon"), R.tiny_config("garment")
    sd_t, sd_g = R.make_state_dict(cfg_t, seed=11), R.make_state_dict(cfg_g, seed=22)      # = make_golden.py's weights
    net_t = U.UNet2DConditionModel(cfg_t, sd_t).to("cuda", torch.float16)
    net_g = U.UNet2DConditionModelGarment(cfg_g, sd_g).to("cuda", torch.float16)
    return dict(R=R, cfg_t=cfg_t, cfg_g=cfg_g, sd_t=sd_t, sd_g=sd_g, net_t=net_t, net_g=net_g)


def test_set_attn_processor_installs_ip_weights_and_scale(tiny_modules):
    """New IPAttnProcessor2_0 instances (fresh to_k_ip / to_v_ip, scale 0.5) installed through set_attn_processor must
    change the engine's output exactly like the oracle run with those weights and `hidden + 0.5 * ip_hidden`."""
    from oracle.make_golden import synth_inputs
    from idm_vton_b200.attention_processor import AttnProcessor2_0, IPAttnProcessor2_0
    from idm_vton_b200 import unet as U
    R, cfg_t = tiny_modules["R"], tiny_modules["cfg_t"]
    net = U.UNet2DConditionModel(cfg_t, tiny_modules["sd_t"]).to("cuda", torch.float16)
    sd = {k: v.clone() for k, v in tiny_modules["sd_t"].items()}
    gen = torch.Generator().manual_seed(99)
    procs = {}
    for name, old in net.attn_processors.items():
        if isinstance(old, IPAttnProcessor2_0):
            p = IPAttnProcessor2_0(old.hidden_size, old.cross_attention_dim, scale=0.5, num_tokens=old.num_tokens)
            for n in ("to_k_ip", "to_v_ip"):
                w = (torch.randn(getattr(p, n).weight.shape, generator=gen) * old.cross_attention_dim ** -0.5).half()
                getattr(p, n).weight.data.copy_(w)
                sd[f"{name}.{n}.weight"] = w.float()
            procs[name] = p.to("cuda", torch.float16)
        else:
            procs[name] = AttnProcessor2_0()
    with pytest.raises(ValueError, match="number of processors"):
        net.set_attn_processor({k: procs[k] for k in list(procs)[:3]})
    with pytest.raises(TypeError):
        net.set_attn_processor(AttnProcessor2_0())          # attn2 of the try-on UNet needs the IP processor
    net.set_attn_processor(dict(procs))
    assert set(net.state_dict()) == set(tiny_modules["sd_t"])
    B, h, w = 1, 16, 16
    x = synth_inputs(cfg_t, tiny_modules["cfg_g"], B, h, w, seed=5)
    x = {k: (v.half().float() if torch.is_floating_point(v) else v) for k, v in x.items()}
    dev = "cuda"
    with torch.no_grad():
        sd32 = {k: v.half().float().to(dev) for k, v in sd.items()}
        x32 = {k: v.to(dev) for k, v in x.items()}
        img = R.resampler_forward(sd32, "encoder_hid_proj", cfg_t["resampler"], x32["clip_tokens"]).half().float()
        feats = [torch.randn(2 * B, (h // s) * (w // s), c, generator=torch.Generator().manual_seed(7 + i)).half().float().to(dev)
                 for i, (s, c) in enumerate([(2, 128)] * 2 + [(4, 256)] * 12 + [(2, 128)] * 3)]
        added = {"text_embeds": x32["text_embeds"], "time_ids": x32["time_ids"], "image_embeds": img}
        ref = R.unet_tryon_forward(sd32, dict(cfg_t, ip_scale=0.5), x32["sample"], x32["timestep"], x32["prompt_embeds"],
                                   added, feats)
        ref_scale1 = R.unet_tryon_forward(sd32, cfg_t, x32["sample"], x32["timestep"], x32["prompt_embeds"], added, feats)
    out = net(x32["sample"].half(), x32["timestep"], encoder_hidden_states=x32["prompt_embeds"].half(),
              added_cond_kwargs={k: (v.half() if k != "time_ids" else v) for k, v in added.items()}, return_dict=False,
              garment_features=[f.half() for f in feats])[0]
    e, sep = _err(out, ref), _err(ref_scale1, ref)
    print(f"set_attn_processor: engine vs oracle(new IP weights, scale 0.5) {e:.2e}; scale 1.0 would differ by {sep:.2e}")
    assert e < 3e-3 and sep > 4 * e


# ------------------------------------------------------------------------------------------------
# a12 Resampler
# ------------------------------------------------------------------------------------------------
def test_resampler_tiny_vs_reference_golden(tiny_modules):
    """`unet.encoder_hid_proj(clip_tokens)` vs the reference module's output stored by oracle/make_golden.py."""
    from oracle.make_golden import synth_inputs
    g = torch.load(os.path.join(G, "unet_tiny_ref.pt"))
    x = synth_inputs(tiny_modules["cfg_t"], tiny_modules["cfg_g"], g["B"], g["h"], g["w"])
    y = tiny_modules["net_t"].encoder_hid_proj(x["clip_tokens"].cuda().half())
    e = _err(y, g["image_embeds"])
    print(f"resampler (tiny cfg) vs reference golden: {e:.2e}")
    assert y.shape == g["image_embeds"].shape and e < 3e-3


def test_resampler_sdxl_geometry_vs_reference_golden():
    """The Resampler at the geometry the try-on UNet hard-codes (src/unet_hacked_tryon.py:476-485) vs the output of
    /root/reference/ip_adapter/resampler.py (loaded standalone by oracle/make_golden_seams.py)."""
    from oracle.make_golden_seams import resampler_weights
    from idm_vton_b200 import lib as L
    from idm_vton_b200.unet import resampler_forward
    g = torch.load(os.path.join(G, "resampler_sdxl_ref.pt"))
    sd = resampler_weights(g["cfg"], g["weight_seed"])
    assert abs(sum(v.double().sum().item() for v in sd.values()) - g["w_checksum"]) < 1e-6 * max(1.0, abs(g["w_checksum"]))
    x = torch.randn(2, 257, 1280, generator=torch.Generator().manual_seed(g["input_seed"])).half()
    L.load()
    y = resampler_forward(L, {f"p.{k}": v.cuda().half() for k, v in sd.items()}, "p", g["cfg"], x.cuda())
    e = _err(y, g["y"])
    print(f"resampler (SDXL geometry) vs reference golden: {e:.2e}")
    assert e < 3e-3


# ------------------------------------------------------------------------------------------------
# B2 UNet modules
# ------------------------------------------------------------------------------------------------
def test_unet_modules_forward_vs_reference_golden(tiny_modules):
    """Both nn.Module facades called exactly as src/tryon_pipeline.py:1787-1808 calls them: the garment UNet returns
    ((sample,), features); the features are zero-padded for the CFG-uncond half (:1796) and handed to the try-on UNet in
    the reference's full [2B, Ng, C] format."""
    from oracle.make_golden import synth_inputs
    g = torch.load(os.path.join(G, "unet_tiny_ref.pt"))
    B, h, w = g["B"], g["h"], g["w"]
    x = synth_inputs(tiny_modules["cfg_t"], tiny_modules["cfg_g"], B, h, w)
    net_t, net_g = tiny_modules["net_t"], tiny_modules["net_g"]
    dev, f16 = "cuda", torch.float16
    down, feats = net_g(x["cloth"].to(dev, f16), x["timestep"], x["text_embeds_cloth"].to(dev, f16), return_dict=False)
    assert isinstance(down, tuple) and len(feats) == len(g["garment_feature_norms"])
    e0, e1 = _err(feats[0], g["garment_feature_0"]), _err(feats[-1], g["garment_feature_last"])
    fc = [torch.cat([torch.zeros_like(d), d]) for d in feats]                          # :1796
    img = net_t.encoder_hid_proj(x["clip_tokens"].to(dev, f16))                       # :1726
    added = {"text_embeds": x["text_embeds"].to(dev, f16), "time_ids": x["time_ids"].to(dev), "image_embeds": img}
    out = net_t(x["sample"].to(dev, f16), x["timestep"], encoder_hidden_states=x["prompt_embeds"].to(dev, f16),
                timestep_cond=None, cross_attention_kwargs=None, added_cond_kwargs=added, return_dict=False,
                garment_features=fc)[0]
    ee = _err(out, g["noise_pred"])
    print(f"B2 modules vs reference golden: feat0 {e0:.2e} feat_last {e1:.2e} noise_pred {ee:.2e}")
    assert out.shape == g["noise_pred"].shape
    # golden = fp32 weights / activations; here fp16 weights and fp16 activations through 17 blocks
    assert e0 < 4e-3 and e1 < 8e-3 and ee < 8e-3


# ------------------------------------------------------------------------------------------------
# B1 pipeline: __call__ vs the REFERENCE pipeline's own output (oracle/make_golden_pipeline.py)
# ------------------------------------------------------------------------------------------------
def test_pipeline_call_vs_reference_golden(tiny_modules):
    """`StableDiffusionXLInpaintPipeline.__call__` with the keyword set of inference.py:397-414 at BASELINE config 1
    (256x256 px, 2 steps, B=1) against the REFERENCE pipeline run on CPU fp32 with the same components / seeds
    (oracle/make_golden_pipeline.py). Three checks:
      (i)   every tensor the pipeline hands to the denoising loop — initial latents, mask, masked-image / pose / cloth
            latents, prompt / pooled / time-id conditioning, Resampler output — equals what the reference pipeline handed
            to ITS loop (golden `loop_inputs`) to fp16 / TF32 rounding: pins the RNG draw order
            (src/tryon_pipeline.py:889,964,1646,1654), the 13-channel order (:1777), [uncond ; cond] (:1711-1714,1769),
            mask preprocessing (:934-980, 1588-1602) and the conditioning plumbing (:1018-1075,1700-1726);
      (ii)  the engine's loop on those tensors equals the oracle loop (pinned to the reference loop with max|d| = 0.0) on
            the SAME tensors and step noises, per step: pins timesteps, CFG, DDPM step and the per-step noise draw (:1823);
      (iii) end to end vs the reference's own latents / images: loose gate — this random-weight tiny UNet amplifies the
            fp16 rounding of its conditioning inputs by ~50x (printed), so (i) + (ii) are the tight statements."""
    from oracle import loop_ref as LR
    from oracle import make_golden_pipeline as MG
    from idm_vton_b200.denoise import TryOnDenoiser
    from idm_vton_b200.pipeline import StableDiffusionXLInpaintPipeline
    from idm_vton_b200.scheduler import DDPMScheduler
    g = torch.load(os.path.join(G, "pipeline_call_ref.pt"))
    dev, f16 = "cuda", torch.float16
    cfg_t, cfg_g = tiny_modules["cfg_t"], tiny_modules["cfg_g"]
    inp = {k: (v.to(dev, f16) if k not in ("image", "mask_image") else v.to(dev)) for k, v in MG.make_call_inputs(cfg_t).items()}
    pipe = StableDiffusionXLInpaintPipeline(
        vae=MG.make_vae().to(dev, f16), text_encoder=None, text_encoder_2=None, tokenizer=None, tokenizer_2=None,
        unet=tiny_modules["net_t"], unet_encoder=tiny_modules["net_g"], scheduler=DDPMScheduler(),
        image_encoder=MG.make_image_encoder(cfg_t["resampler"]["embedding_dim"]).to(dev, f16))
    den = TryOnDenoiser(pipe.unet.engine(), pipe.unet_encoder.engine())
    pipe._denoiser = den
    rec = {"noises": [], "latents": []}
    names = ("latents", "mask", "masked_image_latents", "pose_latents", "cloth_latents", "prompt_embeds", "add_text_embeds",
             "add_time_ids", "image_embeds", "text_embeds_cloth")
    real_prepare, real_step = den.prepare, den.step

    def prepare(*a, **kw):
        rec["inputs"] = {n: v.detach().float().cpu().clone() for n, v in zip(names, a)}
        return real_prepare(*a, **kw)

    def step(i, noise=None, use_graph=True):
        rec["noises"].append(None if noise is None else noise.detach().float().clone())
        return real_step(i, noise, use_graph=use_graph)

    den.prepare, den.step = prepare, step

    def on_step_end(p, i, t, kw):
        rec["latents"].append((int(t), kw["latents"].float().cpu().clone()))
        return {}

    # The golden run drew every random tensor in fp32 on the CPU generator. CPU fp16 and fp32 normal draws come from
    # different streams (torch uses a different kernel per dtype), so the fp16 pipeline's draws from the same generator are
    # taken in fp32 and rounded: order, shapes and count of the draws stay the pipeline's own — that is what is pinned.
    gen = torch.Generator().manual_seed(42)
    real_randn = torch.randn

    def randn_fp32_draws(*size, generator=None, dtype=None, **kw):
        if generator is gen and dtype == torch.float16:
            return real_randn(*size, generator=generator, dtype=torch.float32, **kw).to(torch.float16)
        return real_randn(*size, generator=generator, dtype=dtype, **kw)

    torch.manual_seed(1234)
    torch.randn = randn_fp32_draws
    try:
        images = pipe(**MG.call_kwargs(inp, gen), output_type="pt", callback_on_step_end=on_step_end)[0]
    finally:
        torch.randn = real_randn
    assert [t for t, _ in rec["latents"]] == g["timesteps"].tolist() and images.shape == g["images"].shape
    # ---- (i) the loop's inputs
    e_in = {n: _err(rec["inputs"][n], g["loop_inputs"][n]) for n in names}
    print("B1 (i) loop inputs vs reference pipeline: " + ", ".join(f"{n} {e:.1e}" for n, e in e_in.items()))
    for n in ("mask", "prompt_embeds", "add_text_embeds", "add_time_ids", "text_embeds_cloth"):
        assert e_in[n] == 0.0, n                                   # plumbing only: exact
    assert e_in["latents"] < 1e-3                                  # the fp32 draw rounded to fp16
    for n in ("masked_image_latents", "pose_latents", "cloth_latents"):
        assert e_in[n] < 3e-3, n                                   # fp32 VAE with TF32 convolutions, result rounded to fp16
    assert e_in["image_embeds"] < 5e-3                             # fp16 CLIP + the engine's Resampler
    # ---- (ii) the loop itself, on the pipeline's own inputs and noises
    sd_t32 = {k: v.half().float().to(dev) for k, v in tiny_modules["sd_t"].items()}
    sd_g32 = {k: v.half().float().to(dev) for k, v in tiny_modules["sd_g"].items()}
    li = {n: v.to(dev) for n, v in rec["inputs"].items()}
    steps = len(rec["latents"])
    e_loop = []
    with torch.no_grad():
        for n in range(1, steps + 1):
            ref = LR.denoise_loop(sd_t32, cfg_t, sd_g32, cfg_g, li, steps, guidance_scale=MG.GUIDANCE, noises=rec["noises"], max_steps=n)
            e_loop.append(_err(rec["latents"][n - 1][1], ref))
    # ---- (iii) end to end
    e_e2e = [_err(l, r) for (_, l), r in zip(rec["latents"], g["latents_per_step"])]
    d_img = (images.float().cpu() - g["images"].float()).abs()
    amp = max(e_e2e) / max(max(e_in[n] for n in ("masked_image_latents", "pose_latents", "cloth_latents", "image_embeds", "latents")), 1e-9)
    print(f"B1 (ii) engine loop vs oracle loop on the same inputs, per step: {[f'{e:.2e}' for e in e_loop]}; (iii) end to end vs the "
          f"reference's latents: {[f'{e:.2e}' for e in e_e2e]} (= {amp:.0f}x the largest input difference), image max {d_img.max():.3f} "
          f"mean {d_img.mean():.2e}")
    assert max(e_loop) < 4e-3
    assert max(e_e2e) < 5e-2 and d_img.mean().item() < 2e-2


def test_pipeline_rebuilds_denoiser_after_weight_reload(tiny_modules):
    """ADVICE r1: `pipe.unet.load_state_dict(...)` re-packs the engine lazily; the pipeline must not keep stepping a
    denoiser (and CUDA graph) that still points at the old packed weights."""
    from oracle import make_golden_pipeline as MG
    from oracle import unet_ref as R
    from idm_vton_b200 import unet as U
    from idm_vton_b200.pipeline import StableDiffusionXLInpaintPipeline
    from idm_vton_b200.scheduler import DDPMScheduler
    dev, f16 = "cuda", torch.float16
    cfg_t = tiny_modules["cfg_t"]
    net_t = U.UNet2DConditionModel(cfg_t, tiny_modules["sd_t"]).to(dev, f16)
    pipe = StableDiffusionXLInpaintPipeline(
        vae=MG.make_vae().to(dev, f16), text_encoder=None, text_encoder_2=None, tokenizer=None, tokenizer_2=None,
        unet=net_t, unet_encoder=tiny_modules["net_g"], scheduler=DDPMScheduler(),
        image_encoder=MG.make_image_encoder(cfg_t["resampler"]["embedding_dim"]).to(dev, f16))
    inp = {k: (v.to(dev, f16) if k not in ("image", "mask_image") else v.to(dev)) for k, v in MG.make_call_inputs(cfg_t).items()}

    def run():
        torch.manual_seed(1234)
        pipe(**MG.call_kwargs(inp, torch.Generator().manual_seed(42)), output_type="pt")
        return pipe._last_latents.float().cpu()

    a = run()
    den0 = pipe._denoiser
    assert torch.equal(a, run()) and pipe._denoiser is den0            # same weights: same denoiser, same result
    new = {k: v.to(dev, f16) for k, v in R.make_state_dict(cfg_t, seed=77).items()}
    pipe.unet.load_state_dict(new)
    b = run()
    assert pipe._denoiser is not den0 and _err(b, a) > 1e-2            # new weights took effect
    fresh = U.UNet2DConditionModel(cfg_t, R.make_state_dict(cfg_t, seed=77)).to(dev, f16)
    pipe.unet = fresh
    assert torch.equal(run(), b)


def test_serving_front_end_garment_batching_and_kv_cache(tiny_modules):
    """serving.TryOnServer on the engine: persons sharing a garment run as one batch with the garment UNet at batch 1
    (config 3), a garment seen before skips its garment passes (K/V from the LRU cache) and the result is bit-identical to
    the uncached run."""
    from oracle import make_golden_pipeline as MG
    from idm_vton_b200 import lib as L
    from idm_vton_b200.pipeline import StableDiffusionXLInpaintPipeline
    from idm_vton_b200.scheduler import DDPMScheduler
    from idm_vton_b200.serving import TryOnRequest, TryOnServer
    dev, f16 = "cuda", torch.float16
    cfg_t = tiny_modules["cfg_t"]

    def make_pipe():
        return StableDiffusionXLInpaintPipeline(
            vae=MG.make_vae().to(dev, f16), text_encoder=None, text_encoder_2=None, tokenizer=None, tokenizer_2=None,
            unet=tiny_modules["net_t"], unet_encoder=tiny_modules["net_g"], scheduler=DDPMScheduler(),
            image_encoder=MG.make_image_encoder(cfg_t["resampler"]["embedding_dim"]).to(dev, f16))

    def req(gid, seed):
        i = MG.make_call_inputs(cfg_t, B=1, seed=seed)
        gi = MG.make_call_inputs(cfg_t, B=1, seed=1000 + {"A": 1, "B": 2}[gid])      # garment-side tensors depend on the garment only
        return TryOnRequest(garment_id=gid, image=i["image"][0], mask_image=i["mask_image"][0], pose_img=i["pose_img"][0],
                            prompt_embeds=i["prompt_embeds"][0], negative_prompt_embeds=i["negative_prompt_embeds"][0],
                            pooled_prompt_embeds=i["pooled_prompt_embeds"][0],
                            negative_pooled_prompt_embeds=i["negative_pooled_prompt_embeds"][0], cloth=gi["cloth"][0],
                            ip_adapter_image=gi["ip_adapter_image"][0], text_embeds_cloth=gi["text_embeds_cloth"][0])

    kw = dict(height=MG.H, width=MG.W, num_inference_steps=3, guidance_scale=2.0, max_batch=4, seed=7)
    srv = TryOnServer(make_pipe(), **kw)
    t = [srv.submit(req("A", 1)), srv.submit(req("A", 2)), srv.submit(req("B", 3))]
    out1 = srv.run()
    assert srv.stats["batches"] == 2 and srv.stats["garments_encoded"] == 2 and srv.pipe.garment_cache.hits == 0
    # garment A again: its K/V of all steps come from the cache -> fewer launches, bit-identical images
    n0 = L.launch_count()
    t2 = [srv.submit(req("A", 1)), srv.submit(req("A", 2))]
    out2 = srv.run()
    cached_launches = L.launch_count() - n0
    assert srv.pipe.garment_cache.hits == 1 and srv.stats["garments_encoded"] == 2
    assert torch.equal(out2[t2[0]], out1[t[0]]) and torch.equal(out2[t2[1]], out1[t[1]])
    srv_nc = TryOnServer(make_pipe(), garment_cache_bytes=0, **kw)
    n0 = L.launch_count()
    srv_nc.submit(req("A", 1)), srv_nc.submit(req("A", 2))
    out3 = srv_nc.run()
    uncached_launches = L.launch_count() - n0
    assert torch.equal(out3[0], out1[t[0]]) and cached_launches < uncached_launches
    print(f"serving: garment seen before -> {cached_launches} launches instead of {uncached_launches}")
