"""`StableDiffusionXLInpaintPipeline` — drop-in mirror of the reference's try-on pipeline (seam B1, SURVEY.md 8b).

Same constructor components, `encode_prompt` and `__call__` signatures and defaults as src/tryon_pipeline.py:387-401,
511-526,1254-1301 (tests/test_pipeline_signature.py compares them with `ast`), same call-time behaviour
(check_inputs errors, RNG draw order, CFG ordering [uncond ; cond], `(images,)` tuple return, the
`output_type="latent"` quirk), but the denoising loop (:1765-1866) runs on the B200 engine:
both UNets, garment-feature attention, CFG and the DDPM update are libb200vton.so launches replayed from one CUDA
graph per step (denoise.TryOnDenoiser). Pre/post-processing (VAE, CLIP) is host-side PyTorch plumbing.
"""
import inspect
import os
import types
from typing import Any, Callable, Dict, List, Optional, Tuple, Union

import torch

from . import clip as _clip
from .denoise import TryOnDenoiser, scheduler_family, step_plan
from .vae import VaeImageProcessor

PipelineImageInput = Any


def retrieve_latents(encoder_output, generator=None, sample_mode="sample"):
    if hasattr(encoder_output, "latent_dist") and sample_mode == "sample":
        return encoder_output.latent_dist.sample(generator)
    elif hasattr(encoder_output, "latent_dist") and sample_mode == "argmax":
        return encoder_output.latent_dist.mode()
    elif hasattr(encoder_output, "latents"):
        return encoder_output.latents
    raise AttributeError("Could not access latents of provided encoder_output")


def retrieve_timesteps(scheduler, num_inference_steps=None, device=None, timesteps=None, **kwargs):
    if timesteps is not None:
        if "timesteps" not in set(inspect.signature(scheduler.set_timesteps).parameters.keys()):
            raise ValueError(f"The current scheduler class {scheduler.__class__}'s `set_timesteps` does not support "
                             "custom timestep schedules. Please check whether you are using the correct scheduler.")
        scheduler.set_timesteps(timesteps=timesteps, device=device, **kwargs)
        timesteps = scheduler.timesteps
        num_inference_steps = len(timesteps)
    else:
        scheduler.set_timesteps(num_inference_steps, device=device, **kwargs)
        timesteps = scheduler.timesteps
    return timesteps, num_inference_steps


def randn_tensor(shape, generator=None, device=None, dtype=None):
    """diffusers.utils.torch_utils.randn_tensor: a CPU generator draws on the CPU, then the sample is moved."""
    device = torch.device(device) if device is not None else torch.device("cpu")
    rand_device = device
    if generator is not None and generator.device.type != device.type and generator.device.type == "cpu":
        rand_device = torch.device("cpu")
    return torch.randn(shape, generator=generator, device=rand_device, dtype=dtype).to(device)


def _weights_version(module):
    """Changes whenever a parameter of `module` is replaced or written in place (load_state_dict, .to(), optimizer
    steps): keys the caches derived from its weights (fp32 VAE twin, unconditional CLIP tokens)."""
    return tuple((p.data_ptr(), p._version) for p in module.parameters())


class _StageTrace:
    """B200VTON_TRACE=1: device-time per pipeline stage (CUDA events), printed to stderr at the end of __call__."""

    def __init__(self):
        self.ev = [("start", self._rec())]

    @staticmethod
    def _rec():
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def mark(self, name):
        self.ev.append((name, self._rec()))
        torch.cuda.nvtx.mark(f"b200vton.pipeline:{name}")

    def report(self):
        import sys
        torch.cuda.synchronize()
        parts = [f"{n}: {self.ev[i][1].elapsed_time(e):.1f} ms" for i, (n, e) in enumerate(self.ev[1:])]
        print("[b200vton trace] " + " | ".join(parts), file=sys.stderr, flush=True)


class StableDiffusionXLInpaintPipeline:
    _optional_components = ["tokenizer", "tokenizer_2", "text_encoder", "text_encoder_2"]
    _callback_tensor_inputs = ["latents", "prompt_embeds", "negative_prompt_embeds", "add_text_embeds", "add_time_ids",
                               "negative_pooled_prompt_embeds", "add_neg_time_ids", "mask", "masked_image_latents"]

    def __init__(
        self,
        vae,
        text_encoder,
        text_encoder_2,
        tokenizer,
        tokenizer_2,
        unet,
        unet_encoder,
        scheduler,
        image_encoder=None,
        feature_extractor=None,
        requires_aesthetics_score: bool = False,
        force_zeros_for_empty_prompt: bool = True,
    ):
        self.vae, self.text_encoder, self.text_encoder_2 = vae, text_encoder, text_encoder_2
        self.tokenizer, self.tokenizer_2 = tokenizer, tokenizer_2
        self.unet, self.unet_encoder, self.scheduler = unet, unet_encoder, scheduler
        self.image_encoder, self.feature_extractor = image_encoder, feature_extractor
        self.config = types.SimpleNamespace(force_zeros_for_empty_prompt=force_zeros_for_empty_prompt,
                                            requires_aesthetics_score=requires_aesthetics_score)
        self.vae_scale_factor = 2 ** (len(self.vae.config.block_out_channels) - 1)
        self.image_processor = VaeImageProcessor(vae_scale_factor=self.vae_scale_factor)
        self.mask_processor = VaeImageProcessor(vae_scale_factor=self.vae_scale_factor, do_normalize=False,
                                                do_binarize=True, do_convert_grayscale=True)
        self._denoiser = None
        self._interrupt = False
        self._guidance_scale = 7.5
        self.use_cuda_graph = True
        self.garment_cache = None      # serving.TryOnServer installs a denoise.GarmentKVCache here (off by default)

    # ---------------------------------------------------------------------------------------------
    @classmethod
    def from_pretrained(cls, pretrained_model_name_or_path=None, **components):
        """The reference passes every component explicitly (inference.py:316-329); loading from the hub is
        impossible offline, so all components must be given."""
        components.pop("torch_dtype", None)
        need = [p for p in inspect.signature(cls.__init__).parameters if p not in ("self", "image_encoder",
                "feature_extractor", "requires_aesthetics_score", "force_zeros_for_empty_prompt")]
        missing = [n for n in need if n not in components]
        if missing:
            raise ValueError(f"from_pretrained needs explicit components (no hub access): missing {missing}")
        return cls(**components)

    def register_to_config(self, **kw):
        for k, v in kw.items():
            setattr(self.config, k, v)

    def to(self, device=None, dtype=None):
        for name in ("vae", "text_encoder", "text_encoder_2", "unet", "unet_encoder", "image_encoder"):
            m = getattr(self, name)
            if m is not None and hasattr(m, "to"):
                m.to(device) if dtype is None else m.to(device=device, dtype=dtype)
        self._denoiser = None
        self._vae_fp32 = None
        self._uncond_clip_key = None
        return self

    @property
    def _execution_device(self):
        return self.unet.device

    @property
    def device(self):
        return self.unet.device

    def progress_bar(self, iterable=None, total=None):
        from tqdm.auto import tqdm
        cfg = getattr(self, "_progress_bar_config", {"disable": True})
        return tqdm(iterable, **cfg) if iterable is not None else tqdm(total=total, **cfg)

    def set_progress_bar_config(self, **kwargs):
        self._progress_bar_config = kwargs

    def maybe_free_model_hooks(self):
        pass

    def enable_vae_slicing(self):
        self.vae.enable_slicing()

    def disable_vae_slicing(self):
        self.vae.disable_slicing()

    def enable_vae_tiling(self):
        self.vae.enable_tiling()

    def disable_vae_tiling(self):
        self.vae.disable_tiling()

    # ---------------------------------------------------------------------------------------------
    @property
    def guidance_scale(self):
        return self._guidance_scale

    @property
    def guidance_rescale(self):
        return self._guidance_rescale

    @property
    def clip_skip(self):
        return self._clip_skip

    @property
    def do_classifier_free_guidance(self):
        return self._guidance_scale > 1 and self.unet.config.time_cond_proj_dim is None

    @property
    def cross_attention_kwargs(self):
        return self._cross_attention_kwargs

    @property
    def denoising_end(self):
        return self._denoising_end

    @property
    def denoising_start(self):
        return self._denoising_start

    @property
    def num_timesteps(self):
        return self._num_timesteps

    @property
    def interrupt(self):
        return self._interrupt

    # ---------------------------------------------------------------------------------------------
    def encode_image(self, image, device, num_images_per_prompt, output_hidden_states=None):
        """src/tryon_pipeline.py:460-482."""
        dtype = next(self.image_encoder.parameters()).dtype
        if not isinstance(image, torch.Tensor):
            image = self.feature_extractor(image, return_tensors="pt").pixel_values
        image = image.to(device=device, dtype=dtype)
        tower = _clip.tower_for(self.image_encoder)     # the module's weights on the engine's kernels (None: unsupported)
        if output_hidden_states:
            penultimate = (lambda x: tower.vision_hidden(x, -2).to(dtype)) if tower is not None else (
                lambda x: self.image_encoder(x, output_hidden_states=True).hidden_states[-2])
            hs = penultimate(image)
            hs = hs.repeat_interleave(num_images_per_prompt, dim=0)
            # the unconditional branch encodes an all-zero image: the same tensor for every call with this encoder,
            # so it is computed once per (shape, dtype, device) and reused
            key = (tuple(image.shape), image.dtype, str(image.device), id(self.image_encoder), _weights_version(self.image_encoder),
                   tower is not None)
            if getattr(self, "_uncond_clip_key", None) != key:
                self._uncond_clip = penultimate(torch.zeros_like(image))
                self._uncond_clip_key = key
            un = self._uncond_clip.repeat_interleave(num_images_per_prompt, dim=0)
            return hs, un
        emb = (tower.vision_forward(image).image_embeds.to(dtype) if tower is not None
               else self.image_encoder(image).image_embeds).repeat_interleave(num_images_per_prompt, dim=0)
        return emb, torch.zeros_like(emb)

    def prepare_ip_adapter_image_embeds(self, ip_adapter_image, device, num_images_per_prompt):
        """src/tryon_pipeline.py:485-507: penultimate CLIP tokens of the garment image, [zeros-image ; image] for CFG."""
        image_embeds, negative_image_embeds = self.encode_image(ip_adapter_image, device, 1, True)
        if self.do_classifier_free_guidance:
            image_embeds = torch.cat([negative_image_embeds, image_embeds]).to(device)
        return image_embeds

    def encode_prompt(
        self,
        prompt: str,
        prompt_2: Optional[str] = None,
        device: Optional[torch.device] = None,
        num_images_per_prompt: int = 1,
        do_classifier_free_guidance: bool = True,
        negative_prompt: Optional[str] = None,
        negative_prompt_2: Optional[str] = None,
        prompt_embeds: Optional[torch.FloatTensor] = None,
        negative_prompt_embeds: Optional[torch.FloatTensor] = None,
        pooled_prompt_embeds: Optional[torch.FloatTensor] = None,
        negative_pooled_prompt_embeds: Optional[torch.FloatTensor] = None,
        lora_scale: Optional[float] = None,
        clip_skip: Optional[int] = None,
    ):
        """src/tryon_pipeline.py:511-743. fp16 CLIP text encoders on the GPU run on the engine's kernels (clip.ClipTower),
        anything else through the caller's module as in the reference."""
        device = device or self._execution_device
        prompt = [prompt] if isinstance(prompt, str) else prompt
        batch_size = len(prompt) if prompt is not None else prompt_embeds.shape[0]
        tokenizers = [self.tokenizer, self.tokenizer_2] if self.tokenizer is not None else [self.tokenizer_2]
        text_encoders = [self.text_encoder, self.text_encoder_2] if self.text_encoder is not None else [self.text_encoder_2]

        def _encode(texts, max_length=None):
            embeds, pooled = [], None
            for text, tok, enc in zip(texts, tokenizers, text_encoders):
                ids = tok(text, padding="max_length", max_length=max_length or tok.model_max_length, truncation=True,
                          return_tensors="pt").input_ids
                tower = _clip.tower_for(enc)
                if tower is not None:
                    out = tower.text_forward(ids.to(device), output_hidden_states=True)
                    # out[0] of the module: text_embeds with a projection head, else last_hidden_state (:598)
                    pooled = out.text_embeds if out.text_embeds is not None else out.last_hidden_state
                else:
                    out = enc(ids.to(device), output_hidden_states=True)
                    pooled = out[0]
                embeds.append(out.hidden_states[-2] if clip_skip is None else out.hidden_states[-(clip_skip + 2)])
            return torch.concat(embeds, dim=-1), pooled

        if prompt_embeds is None:
            prompt_2 = prompt_2 or prompt
            prompt_2 = [prompt_2] if isinstance(prompt_2, str) else prompt_2
            prompt_embeds, pooled_prompt_embeds = _encode([prompt, prompt_2])
        zero_out = negative_prompt is None and self.config.force_zeros_for_empty_prompt
        if do_classifier_free_guidance and negative_prompt_embeds is None and zero_out:
            negative_prompt_embeds = torch.zeros_like(prompt_embeds)
            negative_pooled_prompt_embeds = torch.zeros_like(pooled_prompt_embeds)
        elif do_classifier_free_guidance and negative_prompt_embeds is None:
            negative_prompt = negative_prompt or ""
            negative_prompt_2 = negative_prompt_2 or negative_prompt
            negative_prompt = batch_size * [negative_prompt] if isinstance(negative_prompt, str) else negative_prompt
            negative_prompt_2 = batch_size * [negative_prompt_2] if isinstance(negative_prompt_2, str) else negative_prompt_2
            if prompt is not None and type(prompt) is not type(negative_prompt):
                raise TypeError(f"`negative_prompt` should be the same type to `prompt`, but got {type(negative_prompt)} !="
                                f" {type(prompt)}.")
            if batch_size != len(negative_prompt):
                raise ValueError(f"`negative_prompt`: {negative_prompt} has batch size {len(negative_prompt)}, but `prompt`:"
                                 f" {prompt} has batch size {batch_size}. Please make sure that passed `negative_prompt` "
                                 "matches the batch size of `prompt`.")
            negative_prompt_embeds, negative_pooled_prompt_embeds = _encode([negative_prompt, negative_prompt_2],
                                                                            max_length=prompt_embeds.shape[1])
        dtype = self.text_encoder_2.dtype if self.text_encoder_2 is not None else self.unet.dtype
        prompt_embeds = prompt_embeds.to(dtype=dtype, device=device)
        bs_embed, seq_len, _ = prompt_embeds.shape
        prompt_embeds = prompt_embeds.repeat(1, num_images_per_prompt, 1).view(bs_embed * num_images_per_prompt, seq_len, -1)
        if do_classifier_free_guidance:
            seq_len = negative_prompt_embeds.shape[1]
            negative_prompt_embeds = negative_prompt_embeds.to(dtype=dtype, device=device)
            negative_prompt_embeds = negative_prompt_embeds.repeat(1, num_images_per_prompt, 1).view(
                batch_size * num_images_per_prompt, seq_len, -1)
        pooled_prompt_embeds = pooled_prompt_embeds.repeat(1, num_images_per_prompt).view(bs_embed * num_images_per_prompt, -1)
        if do_classifier_free_guidance:
            negative_pooled_prompt_embeds = negative_pooled_prompt_embeds.repeat(1, num_images_per_prompt).view(
                bs_embed * num_images_per_prompt, -1)
        return prompt_embeds, negative_prompt_embeds, pooled_prompt_embeds, negative_pooled_prompt_embeds

    def prepare_extra_step_kwargs(self, generator, eta):
        """src/tryon_pipeline.py: the kwargs `scheduler.step` accepts (DDIM takes `eta`, the others ignore it)."""
        step = getattr(self.scheduler, "step", None)
        params = set(inspect.signature(step).parameters.keys()) if step is not None else set()
        extra = {}
        if "eta" in params:
            extra["eta"] = eta
        if "generator" in params:
            extra["generator"] = generator
        return extra

    def check_inputs(self, prompt, prompt_2, image, mask_image, height, width, strength, callback_steps, output_type,
                     negative_prompt=None, negative_prompt_2=None, prompt_embeds=None, negative_prompt_embeds=None,
                     callback_on_step_end_tensor_inputs=None, padding_mask_crop=None):
        """src/tryon_pipeline.py:763-848 — same conditions, same ValueErrors."""
        if strength < 0 or strength > 1:
            raise ValueError(f"The value of strength should in [0.0, 1.0] but is {strength}")
        if height % 8 != 0 or width % 8 != 0:
            raise ValueError(f"`height` and `width` have to be divisible by 8 but are {height} and {width}.")
        if callback_steps is not None and (not isinstance(callback_steps, int) or callback_steps <= 0):
            raise ValueError(f"`callback_steps` has to be a positive integer but is {callback_steps} of type"
                             f" {type(callback_steps)}.")
        if callback_on_step_end_tensor_inputs is not None and not all(
                k in self._callback_tensor_inputs for k in callback_on_step_end_tensor_inputs):
            bad = [k for k in callback_on_step_end_tensor_inputs if k not in self._callback_tensor_inputs]
            raise ValueError(f"`callback_on_step_end_tensor_inputs` has to be in {self._callback_tensor_inputs}, but found {bad}")
        if prompt is not None and prompt_embeds is not None:
            raise ValueError(f"Cannot forward both `prompt`: {prompt} and `prompt_embeds`: {prompt_embeds}. Please make sure to"
                             " only forward one of the two.")
        elif prompt_2 is not None and prompt_embeds is not None:
            raise ValueError(f"Cannot forward both `prompt_2`: {prompt_2} and `prompt_embeds`: {prompt_embeds}. Please make sure to"
                             " only forward one of the two.")
        elif prompt is None and prompt_embeds is None:
            raise ValueError("Provide either `prompt` or `prompt_embeds`. Cannot leave both `prompt` and `prompt_embeds` undefined.")
        elif prompt is not None and (not isinstance(prompt, str) and not isinstance(prompt, list)):
            raise ValueError(f"`prompt` has to be of type `str` or `list` but is {type(prompt)}")
        elif prompt_2 is not None and (not isinstance(prompt_2, str) and not isinstance(prompt_2, list)):
            raise ValueError(f"`prompt_2` has to be of type `str` or `list` but is {type(prompt_2)}")
        if negative_prompt is not None and negative_prompt_embeds is not None:
            raise ValueError(f"Cannot forward both `negative_prompt`: {negative_prompt} and `negative_prompt_embeds`:"
                             f" {negative_prompt_embeds}. Please make sure to only forward one of the two.")
        elif negative_prompt_2 is not None and negative_prompt_embeds is not None:
            raise ValueError(f"Cannot forward both `negative_prompt_2`: {negative_prompt_2} and `negative_prompt_embeds`:"
                             f" {negative_prompt_embeds}. Please make sure to only forward one of the two.")
        if prompt_embeds is not None and negative_prompt_embeds is not None:
            if prompt_embeds.shape != negative_prompt_embeds.shape:
                raise ValueError("`prompt_embeds` and `negative_prompt_embeds` must have the same shape when passed directly, but"
                                 f" got: `prompt_embeds` {prompt_embeds.shape} != `negative_prompt_embeds`"
                                 f" {negative_prompt_embeds.shape}.")
        if padding_mask_crop is not None:
            raise ValueError("padding_mask_crop is not supported by the B200 engine pipeline (not used by inference.py)")

    def _fused_preprocess_ok(self, image, mask_image, height, width):
        """The one-launch pre-processing covers what inference.py passes: CUDA float tensors [B,3,H,W] / [B,1|3,H,W]
        already at the target size (PIL / numpy inputs, resizes and latent-space images take the VaeImageProcessor path)."""
        ok = lambda t, ch: (torch.is_tensor(t) and t.is_cuda and t.dim() == 4 and t.shape[1] in ch  # noqa: E731
                            and t.shape[-2] == height and t.shape[-1] == width and torch.is_floating_point(t))
        return (ok(image, (3,)) and ok(mask_image, (1, 3)) and image.shape[0] == mask_image.shape[0]
                and height % self.vae_scale_factor == 0 and width % self.vae_scale_factor == 0)

    def _postprocess(self, image, output_type):
        """VaeImageProcessor.postprocess (src/tryon_pipeline.py:1885); fp32 CUDA decoder outputs take the one-launch kernel
        (denormalise + clamp, and for "pil" the uint8 NHWC conversion on the device: 4x less D2H)."""
        if (output_type in ("pt", "pil") and torch.is_tensor(image) and image.is_cuda and image.dtype == torch.float32
                and image.dim() == 4 and image.shape[1] == 3):
            from . import lib as L
            pt, u8 = L.postprocess_image(image, want_pt=output_type == "pt", want_u8=output_type == "pil")
            if output_type == "pt":
                return pt
            import PIL.Image
            return [PIL.Image.fromarray(a) for a in u8.cpu().numpy()]
        return self.image_processor.postprocess(image, output_type=output_type)

    def _vae32(self):
        """fp32 twin of the VAE for the reference's force_upcast path (src/tryon_pipeline.py:913-915,1076-1093).
        The reference flips the one VAE between fp16 and fp32 around every use; keeping a persistent fp32 copy is the
        same arithmetic without converting 84M parameters eight times per call."""
        if self.vae.dtype == torch.float32:
            return self.vae
        twin = getattr(self, "_vae_fp32", None)
        ver = _weights_version(self.vae)
        if twin is None or twin[0] is not self.vae or twin[1].device != self.vae.device or twin[2] != ver:
            import copy
            twin = (self.vae, copy.deepcopy(self.vae).to(dtype=torch.float32), ver)
            self._vae_fp32 = twin
        return twin[1]

    def _encode_vae_image(self, image, generator):
        """src/tryon_pipeline.py:911-932."""
        dtype = image.dtype
        vae = self.vae
        if self.vae.config.force_upcast:
            image = image.float()
            vae = self._vae32()
        if isinstance(generator, list):
            image_latents = torch.cat([retrieve_latents(vae.encode(image[i:i + 1]), generator=generator[i])
                                       for i in range(image.shape[0])], dim=0)
        else:
            image_latents = retrieve_latents(vae.encode(image), generator=generator)
        return self.vae.config.scaling_factor * image_latents.to(dtype)

    def prepare_latents(self, batch_size, num_channels_latents, height, width, dtype, device, generator, latents=None,
                        image=None, timestep=None, is_strength_max=True, add_noise=True, return_noise=False,
                        return_image_latents=False):
        """src/tryon_pipeline.py:850-909 (strength < 1 needs scheduler.add_noise: not on the inference.py path)."""
        shape = (batch_size, num_channels_latents, height // self.vae_scale_factor, width // self.vae_scale_factor)
        if isinstance(generator, list) and len(generator) != batch_size:
            raise ValueError(f"You have passed a list of generators of length {len(generator)}, but requested an effective batch"
                             f" size of {batch_size}. Make sure the batch size matches the length of the generators.")
        if (image is None or timestep is None) and not is_strength_max:
            raise ValueError("Since strength < 1. initial latents are to be initialised as a combination of Image + Noise."
                             "However, either the image or the noise timestep has not been provided.")
        if not is_strength_max or not add_noise:
            raise NotImplementedError("strength < 1 / denoising_start are not on the IDM-VTON inference path")
        image_latents = None
        if image.shape[1] == 4:
            image_latents = image.to(device=device, dtype=dtype).repeat(batch_size // image.shape[0], 1, 1, 1)
        elif return_image_latents:
            image_latents = self._encode_vae_image(image.to(device=device, dtype=dtype), generator)
            image_latents = image_latents.repeat(batch_size // image_latents.shape[0], 1, 1, 1)
        if latents is None:
            noise = randn_tensor(shape, generator=generator, device=device, dtype=dtype)
            latents = noise * self.scheduler.init_noise_sigma
        else:
            noise = latents.to(device)
            latents = noise * self.scheduler.init_noise_sigma
        outputs = (latents,)
        if return_noise:
            outputs += (noise,)
        if return_image_latents:
            outputs += (image_latents,)
        return outputs

    def prepare_mask_latents(self, mask, masked_image, batch_size, height, width, dtype, device, generator,
                             do_classifier_free_guidance, _mask_latent=None):
        """src/tryon_pipeline.py:934-980. `_mask_latent`: the nearest-resized mask when the fused pre-processing kernel
        already produced it."""
        if _mask_latent is not None:
            mask = _mask_latent
        else:
            mask = torch.nn.functional.interpolate(mask, size=(height // self.vae_scale_factor, width // self.vae_scale_factor))
        mask = mask.to(device=device, dtype=dtype)
        if mask.shape[0] < batch_size:
            if not batch_size % mask.shape[0] == 0:
                raise ValueError("The passed mask and the required batch size don't match. Masks are supposed to be duplicated to"
                                 f" a total batch size of {batch_size}, but {mask.shape[0]} masks were passed. Make sure the number"
                                 " of masks that you pass is divisible by the total requested batch size.")
            mask = mask.repeat(batch_size // mask.shape[0], 1, 1, 1)
        mask = torch.cat([mask] * 2) if do_classifier_free_guidance else mask
        masked_image_latents = masked_image if (masked_image is not None and masked_image.shape[1] == 4) else None
        if masked_image is not None:
            if masked_image_latents is None:
                masked_image = masked_image.to(device=device, dtype=dtype)
                masked_image_latents = self._encode_vae_image(masked_image, generator=generator)
            if masked_image_latents.shape[0] < batch_size:
                if not batch_size % masked_image_latents.shape[0] == 0:
                    raise ValueError("The passed images and the required batch size don't match. Images are supposed to be duplicated"
                                     f" to a total batch size of {batch_size}, but {masked_image_latents.shape[0]} images were passed."
                                     " Make sure the number of images that you pass is divisible by the total requested batch size.")
                masked_image_latents = masked_image_latents.repeat(batch_size // masked_image_latents.shape[0], 1, 1, 1)
            masked_image_latents = torch.cat([masked_image_latents] * 2) if do_classifier_free_guidance else masked_image_latents
            masked_image_latents = masked_image_latents.to(device=device, dtype=dtype)
        return mask, masked_image_latents

    def get_timesteps(self, num_inference_steps, strength, device, denoising_start=None):
        """src/tryon_pipeline.py:983-1016 (denoising_start unsupported here)."""
        if denoising_start is not None:
            raise NotImplementedError("denoising_start is not on the IDM-VTON inference path")
        init_timestep = min(int(num_inference_steps * strength), num_inference_steps)
        t_start = max(num_inference_steps - init_timestep, 0)
        timesteps = self.scheduler.timesteps[t_start * self.scheduler.order:]
        return timesteps, num_inference_steps - t_start

    def _get_add_time_ids(self, original_size, crops_coords_top_left, target_size, aesthetic_score,
                          negative_aesthetic_score, negative_original_size, negative_crops_coords_top_left,
                          negative_target_size, dtype, text_encoder_projection_dim=None):
        """src/tryon_pipeline.py:1018-1075."""
        if self.config.requires_aesthetics_score:
            add_time_ids = list(original_size + crops_coords_top_left + (aesthetic_score,))
            add_neg_time_ids = list(negative_original_size + negative_crops_coords_top_left + (negative_aesthetic_score,))
        else:
            add_time_ids = list(original_size + crops_coords_top_left + target_size)
            add_neg_time_ids = list(negative_original_size + crops_coords_top_left + negative_target_size)
        passed = self.unet.config.addition_time_embed_dim * len(add_time_ids) + text_encoder_projection_dim
        expected = self.unet.add_embedding.linear_1.in_features
        if expected != passed:
            raise ValueError(f"Model expects an added time embedding vector of length {expected}, but a vector of {passed} was "
                             "created. The model has an incorrect config. Please check `unet.config.time_embedding_type` and "
                             "`text_encoder_2.config.projection_dim`.")
        return torch.tensor([add_time_ids], dtype=dtype), torch.tensor([add_neg_time_ids], dtype=dtype)

    # ---------------------------------------------------------------------------------------------
    @torch.no_grad()
    def __call__(
        self,
        prompt: Union[str, List[str]] = None,
        prompt_2: Optional[Union[str, List[str]]] = None,
        image: PipelineImageInput = None,
        mask_image: PipelineImageInput = None,
        masked_image_latents: torch.FloatTensor = None,
        height: Optional[int] = None,
        width: Optional[int] = None,
        padding_mask_crop: Optional[int] = None,
        strength: float = 0.9999,
        num_inference_steps: int = 50,
        timesteps: List[int] = None,
        denoising_start: Optional[float] = None,
        denoising_end: Optional[float] = None,
        guidance_scale: float = 7.5,
        negative_prompt: Optional[Union[str, List[str]]] = None,
        negative_prompt_2: Optional[Union[str, List[str]]] = None,
        num_images_per_prompt: Optional[int] = 1,
        eta: float = 0.0,
        generator: Optional[Union[torch.Generator, List[torch.Generator]]] = None,
        latents: Optional[torch.FloatTensor] = None,
        prompt_embeds: Optional[torch.FloatTensor] = None,
        negative_prompt_embeds: Optional[torch.FloatTensor] = None,
        pooled_prompt_embeds: Optional[torch.FloatTensor] = None,
        negative_pooled_prompt_embeds: Optional[torch.FloatTensor] = None,
        ip_adapter_image: Optional[PipelineImageInput] = None,
        output_type: Optional[str] = "pil",
        cloth =None,
        pose_img = None,
        text_embeds_cloth=None,
        return_dict: bool = True,
        cross_attention_kwargs: Optional[Dict[str, Any]] = None,
        guidance_rescale: float = 0.0,
        original_size: Tuple[int, int] = None,
        crops_coords_top_left: Tuple[int, int] = (0, 0),
        target_size: Tuple[int, int] = None,
        negative_original_size: Optional[Tuple[int, int]] = None,
        negative_crops_coords_top_left: Tuple[int, int] = (0, 0),
        negative_target_size: Optional[Tuple[int, int]] = None,
        aesthetic_score: float = 6.0,
        negative_aesthetic_score: float = 2.5,
        clip_skip: Optional[int] = None,
        pooled_prompt_embeds_c=None,
        callback_on_step_end: Optional[Callable[[int, int, Dict], None]] = None,
        callback_on_step_end_tensor_inputs: List[str] = ["latents"],
        **kwargs,
    ):
        callback = kwargs.pop("callback", None)
        callback_steps = kwargs.pop("callback_steps", None)
        # extension (serving front-end, SURVEY.md 8f item 4): one hashable id per garment of this call; with
        # `self.garment_cache` set, the hoisted garment K/V of known garments are reused instead of recomputed
        garment_keys = kwargs.pop("garment_keys", None)
        height = height or self.unet.config.sample_size * self.vae_scale_factor
        width = width or self.unet.config.sample_size * self.vae_scale_factor
        self.check_inputs(prompt, prompt_2, image, mask_image, height, width, strength, callback_steps, output_type,
                          negative_prompt, negative_prompt_2, prompt_embeds, negative_prompt_embeds,
                          callback_on_step_end_tensor_inputs, padding_mask_crop)
        self._guidance_scale = guidance_scale
        self._guidance_rescale = guidance_rescale
        self._clip_skip = clip_skip
        self._cross_attention_kwargs = cross_attention_kwargs
        self._denoising_end = denoising_end
        self._denoising_start = denoising_start
        self._interrupt = False
        if guidance_rescale > 0.0 or denoising_end is not None or denoising_start is not None or timesteps is not None:
            raise NotImplementedError("guidance_rescale / denoising_start / denoising_end / custom timesteps are not on the "
                                      "IDM-VTON inference path (inference.py:397-414)")
        if cloth is None or pose_img is None or text_embeds_cloth is None:
            raise ValueError("cloth, pose_img and text_embeds_cloth are required (src/tryon_pipeline.py:1644-1654,1787)")
        scheduler_family(self.scheduler)          # an unsupported scheduler raises here, before any GPU work

        # 2. call parameters
        if prompt is not None and isinstance(prompt, str):
            batch_size = 1
        elif prompt is not None and isinstance(prompt, list):
            batch_size = len(prompt)
        else:
            batch_size = prompt_embeds.shape[0]
        device = self._execution_device

        trace = _StageTrace() if os.environ.get("B200VTON_TRACE") else None
        # 3. prompt
        (prompt_embeds, negative_prompt_embeds, pooled_prompt_embeds, negative_pooled_prompt_embeds) = self.encode_prompt(
            prompt=prompt, prompt_2=prompt_2, device=device, num_images_per_prompt=num_images_per_prompt,
            do_classifier_free_guidance=self.do_classifier_free_guidance, negative_prompt=negative_prompt,
            negative_prompt_2=negative_prompt_2, prompt_embeds=prompt_embeds,
            negative_prompt_embeds=negative_prompt_embeds, pooled_prompt_embeds=pooled_prompt_embeds,
            negative_pooled_prompt_embeds=negative_pooled_prompt_embeds, clip_skip=self.clip_skip)

        # 4. timesteps
        timesteps, num_inference_steps = retrieve_timesteps(self.scheduler, num_inference_steps, device, timesteps)
        timesteps, num_inference_steps = self.get_timesteps(num_inference_steps, strength, device)
        if num_inference_steps < 1:
            raise ValueError(f"After adjusting the num_inference_steps by strength parameter: {strength}, the number of pipeline"
                             f"steps is {num_inference_steps} which is < 1 and not appropriate for this pipeline.")
        # per-step coefficients, timesteps and noise draws of the caller's scheduler (host only; its step() is not called)
        eta = self.prepare_extra_step_kwargs(generator, eta).get("eta", 0.0)
        plan = step_plan(self.scheduler, timesteps, eta)
        latent_timestep = timesteps[:1].repeat(batch_size * num_images_per_prompt)
        is_strength_max = strength == 1.0

        if trace:
            trace.mark("prompt+timesteps")
        # 5. image / mask
        mask_latent = None
        if masked_image_latents is None and self._fused_preprocess_ok(image, mask_image, height, width):
            # GPU tensors at the target size: image normalisation, mask grayscale + binarisation, the masked image and the
            # latent-resolution mask in ONE launch (b200vton_preprocess_inpaint; same arithmetic as the two
            # VaeImageProcessor.preprocess calls below + :1598 + the nearest resize of :940-943)
            from . import lib as L
            init_image, mask, masked_image, mask_latent = L.preprocess_inpaint(
                image.to(torch.float32).contiguous(), mask_image.to(torch.float32).contiguous(), self.vae_scale_factor)
        else:
            init_image = self.image_processor.preprocess(image, height=height, width=width).to(dtype=torch.float32)
            mask = self.mask_processor.preprocess(mask_image, height=height, width=width)
            if masked_image_latents is not None:
                masked_image = masked_image_latents
            elif init_image.shape[1] == 4:
                masked_image = None
            else:
                masked_image = init_image * (mask.to(init_image.device) < 0.5)

        # 6. latents (RNG draw #1)
        num_channels_latents = self.vae.config.latent_channels
        num_channels_unet = self.unet.config.in_channels
        if num_channels_unet != 13:
            raise NotImplementedError("the try-on UNet has 13 input channels (src/tryon_pipeline.py:1776-1777)")
        latents, noise = self.prepare_latents(batch_size * num_images_per_prompt, num_channels_latents, height, width,
                                              prompt_embeds.dtype, device, generator, latents, image=init_image,
                                              timestep=latent_timestep, is_strength_max=is_strength_max, add_noise=True,
                                              return_noise=True, return_image_latents=False)
        # 7. mask latents (RNG draw #2), pose latents (global RNG!), cloth latents (RNG draw #3)
        pose_img = pose_img.to(device=device, dtype=prompt_embeds.dtype)
        cloth_is_latents = cloth.shape[1] == self.vae.config.latent_channels
        if (masked_image is not None and masked_image.shape[1] == 3 and not cloth_is_latents and not isinstance(generator, list)
                and self.vae.config.force_upcast and masked_image.shape[1:] == pose_img.shape[1:] == cloth.shape[1:]):
            # The reference encodes the masked image (:964 via 911-932), the pose image (:1646) and the garment (:1654) in
            # three VAE passes. The encoder is per-sample (convolutions, per-sample GroupNorm, per-sample attention), so ONE
            # pass over the concatenated batch gives the same posteriors; the three draws then happen in the reference's
            # order and from the reference's generators (user generator, GLOBAL generator for the pose, user generator).
            vae = self._vae32()
            nb = (masked_image.shape[0], pose_img.shape[0], cloth.shape[0])
            x = torch.cat([masked_image.to(device=device, dtype=torch.float32), pose_img.float(),
                           cloth.to(device=device, dtype=torch.float32)])
            # (at most 8 images per encoder pass: the fp32 activations of a 1024x768 image are ~0.4 GB per tensor)
            dists = [vae.encode(x[i:i + 8]).latent_dist for i in range(0, x.shape[0], 8)]
            parts = torch.split(torch.cat([torch.cat([d_.mean, d_.logvar], dim=1) for d_ in dists]), nb)
            from .vae import DiagonalGaussianDistribution
            d_m, d_p, d_c = (DiagonalGaussianDistribution(p_) for p_ in parts)
            sf, dt = self.vae.config.scaling_factor, prompt_embeds.dtype
            masked_lat = sf * d_m.sample(generator).to(dt)                     # draw #2
            pose_lat = d_p.sample().to(dt) * sf                                # global RNG, like the reference
            cloth = sf * d_c.sample(generator).to(dt)                          # draw #3
            mask, masked_image_latents = self.prepare_mask_latents(mask, masked_lat, batch_size * num_images_per_prompt,
                                                                   height, width, dt, device, generator,
                                                                   self.do_classifier_free_guidance, _mask_latent=mask_latent)
            pose_img = torch.cat([pose_lat] * 2) if self.do_classifier_free_guidance else pose_lat
        else:
            mask, masked_image_latents = self.prepare_mask_latents(mask, masked_image, batch_size * num_images_per_prompt,
                                                                   height, width, prompt_embeds.dtype, device, generator,
                                                                   self.do_classifier_free_guidance, _mask_latent=mask_latent)
            pose_img = self.vae.encode(pose_img.to(self.vae.dtype)).latent_dist.sample().to(prompt_embeds.dtype)
            pose_img = pose_img * self.vae.config.scaling_factor
            pose_img = torch.cat([pose_img] * 2) if self.do_classifier_free_guidance else pose_img
            if cloth_is_latents:
                # extension: already-encoded (and scaled) garment latents, as image / masked_image_latents may be
                # (:854-856); the serving front-end encodes each garment once. No RNG draw happens for the garment then.
                cloth = cloth.to(device=device, dtype=prompt_embeds.dtype)
            else:
                cloth = self._encode_vae_image(cloth.to(device=device, dtype=prompt_embeds.dtype), generator=generator)

        if trace:
            trace.mark("vae_encode(image, masked, pose, cloth)")
        # 9./10. added conditions
        height, width = latents.shape[-2:]
        height, width = height * self.vae_scale_factor, width * self.vae_scale_factor
        original_size = original_size or (height, width)
        target_size = target_size or (height, width)
        negative_original_size = negative_original_size or original_size
        negative_target_size = negative_target_size or target_size
        add_text_embeds = pooled_prompt_embeds
        if self.text_encoder_2 is None:
            text_encoder_projection_dim = int(pooled_prompt_embeds.shape[-1])
        else:
            text_encoder_projection_dim = self.text_encoder_2.config.projection_dim
        add_time_ids, add_neg_time_ids = self._get_add_time_ids(
            original_size, crops_coords_top_left, target_size, aesthetic_score, negative_aesthetic_score,
            negative_original_size, negative_crops_coords_top_left, negative_target_size, dtype=prompt_embeds.dtype,
            text_encoder_projection_dim=text_encoder_projection_dim)
        add_time_ids = add_time_ids.repeat(batch_size * num_images_per_prompt, 1)
        if self.do_classifier_free_guidance:
            prompt_embeds = torch.cat([negative_prompt_embeds, prompt_embeds], dim=0)
            add_text_embeds = torch.cat([negative_pooled_prompt_embeds, add_text_embeds], dim=0)
            add_neg_time_ids = add_neg_time_ids.repeat(batch_size * num_images_per_prompt, 1)
            add_time_ids = torch.cat([add_neg_time_ids, add_time_ids], dim=0)
        prompt_embeds, add_text_embeds, add_time_ids = prompt_embeds.to(device), add_text_embeds.to(device), add_time_ids.to(device)
        if ip_adapter_image is None:
            raise ValueError("ip_adapter_image is required: the try-on UNet concatenates the IP tokens "
                             "(src/unet_hacked_tryon.py:1234-1242)")
        image_embeds = self.prepare_ip_adapter_image_embeds(ip_adapter_image, device, batch_size * num_images_per_prompt)
        image_embeds = self.unet.encoder_hid_proj(image_embeds).to(prompt_embeds.dtype)      # Resampler, once (:1726)
        n_img, n_req = image_embeds.shape[0], prompt_embeds.shape[0]
        if n_img != n_req:          # extension: ONE garment image for all persons of the batch ([uncond ; cond] each x B)
            if n_req % n_img:
                raise ValueError(f"ip_adapter_image batch {n_img} does not divide the request batch {n_req}")
            halves = image_embeds.chunk(2) if self.do_classifier_free_guidance else (image_embeds,)
            image_embeds = torch.cat([h.repeat_interleave(n_req // n_img, dim=0) for h in halves])

        if trace:
            trace.mark("clip_image_encoder+resampler")
        # 11. denoising loop on the B200 engine
        self._num_timesteps = len(timesteps)
        # unet.engine() re-packs after load_state_dict() / .to() on the module; a denoiser built on older engines (and its
        # captured graph) would silently run stale weights
        eng_t, eng_g = self.unet.engine(), self.unet_encoder.engine()
        if self._denoiser is None or self._denoiser.tryon is not eng_t or self._denoiser.garment is not eng_g:
            self._denoiser = TryOnDenoiser(eng_t, eng_g)
        den = self._denoiser
        den.prepare(latents, mask, masked_image_latents, pose_img, cloth, prompt_embeds, add_text_embeds, add_time_ids,
                    image_embeds, text_embeds_cloth.to(device), guidance_scale=self.guidance_scale,
                    do_cfg=self.do_classifier_free_guidance)
        den.set_step_tables(self.scheduler, timesteps, garment_keys=garment_keys, cache=self.garment_cache, plan=plan)
        if trace:
            trace.mark("denoiser.prepare (context K/V, garment passes)")
        with self.progress_bar(total=num_inference_steps) as progress_bar:
            for i, t in enumerate(timesteps):
                if self.interrupt:
                    continue
                step_noise = None
                if plan.draws[i]:         # the draw the reference's scheduler.step makes (DDPM: t > 0; DDIM: eta > 0;
                    # Euler / Euler-ancestral: every step), same generator, shape, device and dtype
                    step_noise = randn_tensor(latents.shape, generator=generator, device=device, dtype=latents.dtype)
                latents = den.step(i, step_noise, use_graph=self.use_cuda_graph)
                if callback_on_step_end is not None:
                    callback_kwargs = {k: locals()[k] for k in callback_on_step_end_tensor_inputs}
                    callback_outputs = callback_on_step_end(self, i, t, callback_kwargs)
                    new_latents = callback_outputs.pop("latents", latents)
                    if new_latents is not latents:
                        den.latents.copy_(new_latents)
                progress_bar.update()
                if callback is not None and i % (callback_steps or 1) == 0:
                    callback(i, t, latents)
        latents = latents.clone()
        if trace:
            trace.mark("denoise loop")

        if not output_type == "latent":
            needs_upcasting = self.vae.dtype == torch.float16 and self.vae.config.force_upcast
            vae = self._vae32() if needs_upcasting else self.vae
            image = vae.decode(latents.to(vae.dtype) / self.vae.config.scaling_factor, return_dict=False)[0]
        # NB (reference quirk, src/tryon_pipeline.py:1868-1885): with output_type == "latent", `image` is still the
        # caller's input image, and that is what gets returned.
        image = self._postprocess(image, output_type)
        if trace:
            trace.mark("vae_decode+postprocess")
            trace.report()
        self.maybe_free_model_hooks()
        self._last_latents = latents
        return (image,)
