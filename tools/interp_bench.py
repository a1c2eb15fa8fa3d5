"""Cost of interpolating between two futures against one sampling round, one GPU, synthetic weights.

    python tools/interp_bench.py [--datasets bair,kth] [--batch 32] [--rounds 10]

For each dataset (its shipped DDIM configuration, S = sampling_timesteps): ms per call of
FlowDiffusion.interpolate_one_video (conditioning, mix, S-step DDIM loop as one CUDA graph, decode; per-video seeds)
at t = T - 1 and t = T / 2, against one sample_one_video round on the same clips, each after two warm-up calls (graph
capture), timed alternately with CUDA events; median (min-max).  x1 is encode_future of the clips, x2 a sample.  Then
the extdm_q_interpolate kernel alone, timed with CUDA events over 200 launches, against its HBM byte bound at 7.7 TB/s:
with injected epsilon it reads x1, x2, eps1, eps2 and writes x_t, 20 bytes per element; with Philox epsilon it reads
x1, x2 and writes x_t, 12 bytes per element.  It is timed at the round's size (which stays in the 126 MB L2 across
launches) and at 16 times that size (beyond L2).  Reads the card name and power limit in the same run; prints one JSON
line.  No interpolation quality is measured: the weights are random.
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import extdm_b200  # noqa: E402,F401
from extdm_b200 import configs, ops  # noqa: E402
from benchlib import HBM_BYTES_PER_S, event_ms, power_limit, spread  # noqa: E402


def kernel_time(diff, B, n, injected):
    """ms per extdm_q_interpolate launch on (B, n) fp32 tensors."""
    g = torch.Generator(device="cuda").manual_seed(0)
    x1, x2 = (torch.randn(B, n, device="cuda", generator=g) for _ in range(2))
    noise = torch.randn(2, B, n, device="cuda", generator=g) if injected else None
    seeds = None if injected else torch.arange(B, dtype=torch.long, device="cuda")
    out = torch.empty_like(x1)
    acp, a1m = diff.sqrt_alphas_cumprod, diff.sqrt_one_minus_alphas_cumprod

    def launch():
        ops.q_interpolate(ops.IMMEDIATE, x1, x2, 500, seeds, noise, acp, a1m, 0.7, 0.3, out)

    for _ in range(20):
        launch()
    return event_ms(launch, 200)


def bench(name, B, rounds):
    model, cfg = configs.build_model(name, device="cuda")
    diff = model.diffusion
    tc, tp, hw = model.cond_frame_num, model.pred_frame_num, cfg["dataset_params"]["frame_shape"]
    clips = torch.rand((B, 3, tc + tp, hw, hw), generator=torch.Generator().manual_seed(0)).cuda()
    past = clips[:, :, :tc].contiguous()
    gen = torch.Generator().manual_seed(1)

    def seeds():
        return torch.randint(0, 2 ** 62, (B,), dtype=torch.long, generator=gen)

    x1 = model.encode_future(clips)
    x2 = diff.sample(*model.condition(past)[1:3], seeds=seeds())
    T = diff.num_timesteps
    runs = [("sample_one_video", lambda: model.sample_one_video(cond_scale=1.0, real_vid=past, seeds=seeds()))]
    for t in (T - 1, T // 2):
        runs.append((f"interpolate_t{t}", lambda t=t: model.interpolate_one_video(past, x1, x2, t=t, lam=0.5,
                                                                                  seeds=seeds())))
    for _, fn in runs:                                                   # warm-up: graph capture, clocks
        fn()
        fn()
    times = {k: [] for k, _ in runs}
    for _ in range(rounds):
        for k, fn in runs:
            times[k].append(event_ms(fn))
    n = x1[0].numel()
    kern = {}
    for label, b in (("round_size", B), ("x16", 16 * B)):
        for mode, injected, per_el in (("injected", True, 20), ("philox", False, 12)):
            bound_ms = b * n * per_el / HBM_BYTES_PER_S * 1e3
            ms = kernel_time(diff, b, n, injected)
            kern[f"{label}_{mode}"] = {"batch": b, "elements": b * n, "bytes_per_element": per_el, "ms": round(ms, 5),
                                       "hbm_bound_ms": round(bound_ms, 5), "bound_over_time": round(bound_ms / ms, 3)}
    base = statistics.median(times["sample_one_video"])
    return {"dataset": name, "batch": B, "rounds": rounds, "sampling_timesteps": int(diff.sampling_timesteps),
            "call_ms": {k: spread(v) for k, v in times.items()},
            "over_sample_one_video": {k: round(statistics.median(v) / base, 4) for k, v in times.items()},
            "mix_kernel": kern}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--datasets", default="bair,kth")
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--rounds", type=int, default=10)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("interp_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    res = [bench(n, a.batch, a.rounds) for n in a.datasets.split(",")]
    print(json.dumps({"gpu": torch.cuda.get_device_name(), "power_limit": power_limit(), "results": res}))


if __name__ == "__main__":
    main()
