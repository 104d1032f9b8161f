"""Denoise-loop time per scheduler at BASELINE config 2 (768x1024 px, batch 2, two garments, synthetic inputs, random
SDXL-shaped weights): DDPM / DDIM / Euler at 30 steps and DPM-Solver++ 2M at 20, alternated round by round in one
process. Device events time the whole loop (hoisted garment passes + every step's graph replay, the step noise drawn as
the pipeline draws it) and each step's replay. The graph of each scheduler is captured before the timed rounds (the
family change recaptures it). GPU name, power limit and SM clock are recorded beside the numbers.

Usage: python scripts/scheduler_bench.py [--rounds 3] [--out FILE.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

RUNS = [("DDPMScheduler", 30), ("DDIMScheduler", 30), ("EulerDiscreteScheduler", 30), ("DPMSolverMultistepScheduler", 20)]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, sm, sm_max = [x.strip() for x in q.split(",")]
        return dict(gpu=name, power_limit=power, sm_clock=sm, sm_clock_max=sm_max)
    except Exception as e:                       # informational only
        return dict(gpu=torch.cuda.get_device_name(), query_error=str(e))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import bench
    from idm_vton_b200 import lib as L
    from idm_vton_b200 import scheduler as S
    from idm_vton_b200.denoise import TryOnDenoiser
    from idm_vton_b200.engine import SDXL_GARMENT, SDXL_TRYON
    if not torch.cuda.is_available():
        raise SystemExit("scheduler_bench needs a GPU")
    dev = torch.device("cuda", 0)
    L.load()
    log = lambda m: print(m, file=sys.stderr, flush=True)  # noqa: E731
    unet, unet_enc, _ = bench.build_components(dev, 0, 1, log)
    den = TryOnDenoiser(unet.engine(), unet_enc.engine())
    B, h, w = 2, 128, 96
    req = bench.synth_request(SDXL_TRYON, SDXL_GARMENT, B, h, w, seed=42, device=dev, garments=2)
    den.prepare(**req, guidance_scale=bench.GUIDANCE)
    base = S.DDPMScheduler()
    scheds = {}
    for name, steps in RUNS:
        s = getattr(S, name).from_config(base.config)
        s.set_timesteps(steps)
        scheds[name] = s
    gen = torch.Generator(device=dev).manual_seed(0)

    def loop(name, timed):
        s = scheds[name]
        den.latents.copy_(req["latents"] * float(s.init_noise_sigma))
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * len(s.timesteps) + 2)]
        ev[0].record()
        den.set_step_tables(s, s.timesteps)                          # hoisted garment passes
        if den._graph is None:
            if timed:
                raise RuntimeError("graph recapture inside a timed loop")
            den.capture()
        for i in range(len(s.timesteps)):
            noise = torch.randn(den.latents.shape, generator=gen, device=dev, dtype=torch.float16) if den.plan.draws[i] else None
            ev[2 * i + 1].record()
            den.step(i, noise, use_graph=True)
            ev[2 * i + 2].record()
        ev[-1].record()
        return ev

    def capture_then_loop(name):
        loop(name, timed=False)                 # warm-up round: captures this scheduler's graph
        return loop(name, timed=False)

    for name, _ in RUNS:                        # warm-up of every shape
        capture_then_loop(name)
    torch.cuda.synchronize()
    res = {name: {"loop_ms": [], "replay_ms": []} for name, _ in RUNS}
    for r in range(args.rounds):
        for name, _ in RUNS:                    # alternating: the family change recaptures the graph, outside the timing
            den.set_step_tables(scheds[name], scheds[name].timesteps)
            if den._graph is None:
                den.capture()
            ev = loop(name, timed=True)
            torch.cuda.synchronize()
            res[name]["loop_ms"].append(ev[0].elapsed_time(ev[-1]))
            n = len(scheds[name].timesteps)
            res[name]["replay_ms"].append(statistics.median(ev[2 * i + 1].elapsed_time(ev[2 * i + 2]) for i in range(n)))
            assert torch.isfinite(den.latents.float()).all(), name
    out = dict(info=gpu_info(), config="BASELINE config 2: 768x1024 px, batch 2, 2 garments, random SDXL-shaped weights",
               rounds=args.rounds, method="device events; loop = set_step_tables (hoisted garment passes) + every step's "
               "graph replay incl. the step-noise draw; replay = median over the steps of one loop; schedulers alternated "
               "round by round", results={})
    ddpm_loop = statistics.median(res["DDPMScheduler"]["loop_ms"])
    for name, steps in RUNS:
        lo, rp = res[name]["loop_ms"], res[name]["replay_ms"]
        out["results"][name] = dict(steps=steps, loop_ms_median=statistics.median(lo), loop_ms=lo,
                                    loop_ms_spread=max(lo) - min(lo), replay_ms_median=statistics.median(rp), replay_ms=rp,
                                    loop_vs_ddpm30=statistics.median(lo) / ddpm_loop)
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
