"""DDPM (ancestral, 1000 steps) against DDIM (10 steps) per denoising step, one GPU, synthetic weights.

    python tools/ddpm_bench.py [--datasets bair,kth] [--batch 32] [--repeats 2] [--profile DIR]

For each dataset: after a warm-up round of each sampler, times DDIM and DDPM rounds alternately with CUDA events
(GaussianDiffusion.sample on the conditioning of one clip, CUDA-graphed as shipped) and the UNet prologue on its own.
ms/step = (round - prologue) / steps, so the prologue that both samplers run once per round does not favour the longer
loop.  Also times the time MLP as a graph node (what each DDPM step would pay to evaluate it in the loop) and the
broadcast of the precomputed per-step rows that the DDPM iteration runs instead, and reads the card name and power
limit.  Prints one JSON line.  --profile DIR writes a torch.profiler chrome trace of a few DDIM and DDPM steps to DIR.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import extdm_b200  # noqa: E402,F401
from extdm_b200 import configs, ops  # noqa: E402
from benchlib import event_ms, power_limit  # noqa: E402

DDIM_STEPS, DDPM_STEPS = 10, 1000


def use(diff, steps):
    diff.sampling_timesteps, diff.is_ddim_sampling = steps, steps < diff.num_timesteps


def graph_ms(fn, reps):
    """Device time of one call of fn, from a CUDA graph holding `reps` calls (no launch overhead)."""
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    g.replay()
    return event_ms(g.replay, 5) / reps


def bench(name, B, repeats, profile_dir):
    model, cfg = configs.build_model(name, device="cuda")
    diff = model.diffusion
    tc, hw = model.cond_frame_num, cfg["dataset_params"]["frame_shape"]
    clip = torch.rand((B, 3, tc, hw, hw), generator=torch.Generator().manual_seed(0)).cuda()
    _, x_cond, cond_fea, _ = model.condition(clip)
    r = diff.denoise_fn.runner(B, x_cond.shape[3], x_cond.shape[4], cond_fea.shape[-1])

    def round_of(steps):
        use(diff, steps)
        return lambda: diff.sample(x_cond, cond_fea=cond_fea)

    ddim, ddpm = round_of(DDIM_STEPS), round_of(DDPM_STEPS)
    for steps, fn in ((DDIM_STEPS, ddim), (DDPM_STEPS, ddpm)):           # warm-up: graph capture, clocks
        use(diff, steps)
        fn()
        if steps == DDIM_STEPS:
            fn()
    t = {"ddim": [], "ddpm": []}
    for _ in range(repeats):
        use(diff, DDIM_STEPS)
        t["ddim"].append(event_ms(ddim))
        use(diff, DDPM_STEPS)
        t["ddpm"].append(event_ms(ddpm))
    r.set_conditioning(x_cond.float(), cond_fea.float())
    prologue = graph_ms(r.run_prologue, 10)
    time_mlp = graph_ms(r.time_rec.run, 50)
    _, st = next(v for k, v in r.graphs.items() if k[0] == "ddpm")
    broadcast = graph_ms(lambda: ops.ddpm_broadcast_row(ops.IMMEDIATE, st["ss_rows"], st["step"], r.ss), 50)
    ddim_round, ddpm_round = min(t["ddim"]), min(t["ddpm"])
    ddim_step = (ddim_round - prologue) / DDIM_STEPS
    ddpm_step = (ddpm_round - prologue) / DDPM_STEPS

    if profile_dir:
        from torch.profiler import ProfilerActivity, profile
        os.makedirs(profile_dir, exist_ok=True)
        use(diff, DDPM_STEPS)
        g, st = next(v for k, v in r.graphs.items() if k[0] == "ddpm")
        st["step"].zero_()                          # replay from the first step, as a round does
        r.time.fill_(DDPM_STEPS - 1)
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            use(diff, DDIM_STEPS)
            ddim()
            for _ in range(DDIM_STEPS):
                g.replay()
            torch.cuda.synchronize()
        prof.export_chrome_trace(os.path.join(profile_dir, f"ddpm_vs_ddim_{name}_b{B}.json"))

    use(diff, DDIM_STEPS)
    return {"dataset": name, "batch": B, "ddim_ms_per_step": round(ddim_step, 4),
            "ddpm_ms_per_step": round(ddpm_step, 4), "ddpm_over_ddim": round(ddpm_step / ddim_step, 4),
            "ddpm_round_ms": round(ddpm_round, 2), "ddim_round_ms": round(ddim_round, 3),
            "prologue_ms": round(prologue, 4), "time_mlp_ms": round(time_mlp, 4),
            "time_mlp_share_of_ddpm_step": round(time_mlp / ddpm_step, 5), "ss_broadcast_ms": round(broadcast, 4),
            "ddim_rounds_ms": [round(x, 3) for x in t["ddim"]], "ddpm_rounds_ms": [round(x, 2) for x in t["ddpm"]]}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--datasets", default="bair,kth")
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--profile", default="", help="directory for a torch.profiler trace of a few steps")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("ddpm_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    res = [bench(n, a.batch, a.repeats, a.profile) for n in a.datasets.split(",")]
    print(json.dumps({"gpu": torch.cuda.get_device_name(), "power_limit": power_limit(), "results": res}))


if __name__ == "__main__":
    main()
