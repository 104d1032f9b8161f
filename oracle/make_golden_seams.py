"""Golden vectors for the seam tests (tests/test_seams_gpu.py), produced by the REFERENCE's own code.

Needs a checkout of the original IDM-VTON repository, whose modules are imported unmodified and in place:
  * ip_adapter/attention_processor.py  AttnProcessor2_0 (:189-278), IPAttnProcessor2_0 (:1879-2010), executed on the
    diffusers-shim `Attention` container (oracle/shim/diffusers/models/attention_processor.py), CPU fp32;
  * ip_adapter/resampler.py            Resampler at the geometry the try-on UNet hard-codes
    (src/unet_hacked_tryon.py:476-485: dim 1280, depth 4, 20 heads x 64, 16 queries, CLIP width 1280 -> 2048).
Writes tests/golden/attn_processors_ref.pt (self- and cross-attention) and tests/golden/attn_processors_ip_ref.pt
(IP-Adapter cross-attention): weights + inputs + outputs, fp16 storage of fp16-representable values so every
implementation sees identical numbers, split in two so that each file stays under 1 MB; and
tests/golden/resampler_sdxl_ref.pt (seeds + output).

Usage:  python oracle/make_golden_seams.py <path of the IDM-VTON checkout>
"""
import importlib.util
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def _load_by_path(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def resampler_weights(r, seed):
    """Seeded Resampler state dict (keys of ip_adapter/resampler.py's module) — shared with the GPU test."""
    from oracle import unet_ref as R
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for k, shp in R._resampler_shapes("x", r).items():
        k = k[2:]
        if k == "latents":
            w = torch.randn(shp, generator=g) / shp[-1] ** 0.5
        elif len(shp) == 1:
            w = (1.0 + 0.1 * torch.randn(shp, generator=g)) if k.endswith("weight") else 0.1 * torch.randn(shp, generator=g)
        else:
            w = (torch.rand(shp, generator=g) * 2 - 1) * (3.0 / shp[1]) ** 0.5
        sd[k] = w.half().float()
    return sd


def main(ref):
    sys.path.insert(0, os.path.join(ROOT, "oracle", "shim"))
    sys.path.insert(0, ROOT)
    from diffusers.models.attention_processor import Attention           # the shim's container
    ap = _load_by_path("ref_attention_processor", os.path.join(ref, "ip_adapter", "attention_processor.py"))
    rs = _load_by_path("ref_resampler", os.path.join(ref, "ip_adapter", "resampler.py"))
    os.makedirs(GOLDEN, exist_ok=True)
    g = torch.Generator().manual_seed(2024)

    def r(*s, scale=1.0):
        return (torch.randn(*s, generator=g) * scale).half().float()

    C, heads, cross, B, T, Tt, Ti = 128, 2, 256, 2, 160, 77, 16
    out = {"C": C, "heads": heads, "cross": cross}
    with torch.no_grad():
        # ---- self-attention (AttnProcessor2_0, encoder_hidden_states=None)
        a1 = Attention(query_dim=C, heads=heads, dim_head=64, bias=False, out_bias=True, processor=ap.AttnProcessor2_0())
        w1 = {"to_q.weight": r(C, C, scale=C ** -0.5), "to_k.weight": r(C, C, scale=C ** -0.5),
              "to_v.weight": r(C, C, scale=C ** -0.5), "to_out.0.weight": r(C, C, scale=C ** -0.5),
              "to_out.0.bias": r(C, scale=0.1)}
        a1.load_state_dict(w1, strict=True)
        x = r(B, T, C)
        xh = x.half()                  # one stored copy, shared by every case
        out["self"] = dict(weights={k: v.half() for k, v in w1.items()}, x=xh, y=a1(x))
        # ---- plain cross-attention (AttnProcessor2_0 with encoder_hidden_states: the garment UNet's attn2)
        a2 = Attention(query_dim=C, cross_attention_dim=cross, heads=heads, dim_head=64, bias=False, out_bias=True,
                       processor=ap.AttnProcessor2_0())
        w2 = {"to_q.weight": r(C, C, scale=C ** -0.5), "to_k.weight": r(C, cross, scale=cross ** -0.5),
              "to_v.weight": r(C, cross, scale=cross ** -0.5), "to_out.0.weight": r(C, C, scale=C ** -0.5),
              "to_out.0.bias": r(C, scale=0.1)}
        a2.load_state_dict(w2, strict=True)
        enc = r(B, Tt, cross)
        w2h = {k: v.half() for k, v in w2.items()}
        out["cross"] = dict(weights=w2h, x=xh, enc=enc.half(), y=a2(x, encoder_hidden_states=enc))
        # ---- IP-Adapter decoupled cross-attention (IPAttnProcessor2_0), scale 1.0 (inference) and 0.5
        enc_ip = r(B, Tt + Ti, cross)
        wip = {"to_k_ip.weight": r(C, cross, scale=cross ** -0.5), "to_v_ip.weight": r(C, cross, scale=cross ** -0.5)}
        ys = {}
        for s in (1.0, 0.5):
            proc = ap.IPAttnProcessor2_0(hidden_size=C, cross_attention_dim=cross, scale=s, num_tokens=Ti)
            proc.load_state_dict(wip, strict=True)
            a3 = Attention(query_dim=C, cross_attention_dim=cross, heads=heads, dim_head=64, bias=False, out_bias=True,
                           processor=proc)
            a3.load_state_dict({**w2, **{f"processor.{k}": v for k, v in wip.items()}}, strict=True)
            ys[s] = a3(x, encoder_hidden_states=enc_ip)
        ip = dict(weights={**w2h, **{k: v.half() for k, v in wip.items()}}, x=xh, enc=enc_ip.half(),
                  y_scale_1=ys[1.0], y_scale_0p5=ys[0.5], num_tokens=Ti)
    note = ("outputs (fp32) of the REFERENCE processors ip_adapter/attention_processor.py AttnProcessor2_0 / "
            "IPAttnProcessor2_0 on the diffusers-shim Attention container, CPU fp32; weights and inputs are "
            "fp16-representable and stored here")
    out["note"] = note + "; the IP-Adapter case is in attn_processors_ip_ref.pt"
    torch.save(out, os.path.join(GOLDEN, "attn_processors_ref.pt"))
    torch.save({"C": C, "heads": heads, "ip": ip, "note": note + "; self / cross cases: attn_processors_ref.pt"},
               os.path.join(GOLDEN, "attn_processors_ip_ref.pt"))
    print("wrote attn_processors_ref.pt", {k: tuple(v["y"].shape) for k, v in out.items() if isinstance(v, dict)},
          "and attn_processors_ip_ref.pt", tuple(ip["y_scale_1"].shape))

    # ---- Resampler at the SDXL / IDM-VTON geometry, reference module loaded standalone
    rcfg = dict(dim=1280, depth=4, dim_head=64, heads=20, num_queries=16, embedding_dim=1280, output_dim=2048, ff_mult=4)
    net = rs.Resampler(**rcfg).eval()
    sd = resampler_weights(rcfg, seed=77)
    net.load_state_dict(sd, strict=True)
    gi = torch.Generator().manual_seed(78)
    x = torch.randn(2, 257, 1280, generator=gi).half().float()
    with torch.no_grad():
        y = net(x)
        from oracle import unet_ref as R
        y_or = R.resampler_forward({f"p.{k}": v for k, v in sd.items()}, "p", rcfg, x)
    print("resampler (SDXL geometry): reference vs oracle max|d| =", (y - y_or).abs().max().item(), "|y|max", y.abs().max().item())
    assert (y - y_or).abs().max().item() < 2e-5 * max(1.0, y.abs().max().item())
    torch.save({"note": "output of the REFERENCE ip_adapter/resampler.py Resampler(dim=1280, depth=4, dim_head=64, heads=20, "
                        "num_queries=16, embedding_dim=1280, output_dim=2048, ff_mult=4), CPU fp32; weights = "
                        "oracle.make_golden_seams.resampler_weights(cfg, seed=77); input = randn(2,257,1280, seed 78) "
                        "rounded to fp16", "cfg": rcfg, "weight_seed": 77, "input_seed": 78, "y": y.half(),
                "w_checksum": float(sum(v.double().sum().item() for v in sd.values()))},
               os.path.join(GOLDEN, "resampler_sdxl_ref.pt"))
    print("wrote resampler_sdxl_ref.pt")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit("usage: python oracle/make_golden_seams.py <path of the IDM-VTON checkout>")
    main(sys.argv[1])
