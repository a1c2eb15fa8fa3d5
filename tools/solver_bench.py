"""Cost of the DPM-Solver++(2M) sampler against DDIM, one GPU, synthetic weights.

    python tools/solver_bench.py [--datasets bair,kth] [--batch 32] [--rounds 10]

For each dataset: ms per sampling round (one GaussianDiffusion.sample call on the conditioning of one clip, CUDA-graphed
as shipped, with per-video seeds; conditioning excluded, UNet prologue included) of four arms -- DDIM at S = 10,
dpmpp_2m at S = 5 and 10, dpmpp_2m_sde at S = 10 -- after one warm-up round each (graph capture), timed alternately
with CUDA events; median (min-max).  Then the extdm_dpmpp_update kernel alone, timed with CUDA events over 200
launches, against its HBM byte bound: x, eps and D_prev read, x and D_prev written, 20 bytes per element, at
7.7 TB/s.  It is timed at the round's size (whose 20 bytes per element stay in the 126 MB L2 across launches) and at
16 times that size (beyond L2).  Reads the card name and power limit in the same run; prints one JSON line.

The synthetic weights are random, so no sample quality is measured or printed here: whether fewer solver steps match
DDIM's quality needs trained weights.
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

ARMS = [("ddim", None, 10), ("dpmpp_2m", "dpmpp_2m", 5), ("dpmpp_2m", "dpmpp_2m", 10),
        ("dpmpp_2m_sde", "dpmpp_2m_sde", 10)]
BYTES_PER_ELEMENT = 20


def kernel_time(B, n, sde):
    """ms per extdm_dpmpp_update launch on (B, n) fp32 tensors (a middle step: C term present; Philox z when sde)."""
    g = torch.Generator(device="cuda").manual_seed(0)
    x, eps, dp = (torch.randn(B, n, device="cuda", generator=g) for _ in range(3))
    s = torch.ones(B, device="cuda")
    seeds = torch.arange(B, dtype=torch.long, device="cuda") if sde else None
    rec = ops.IMMEDIATE

    def launch():
        ops.dpmpp_update(rec, x, eps, dp, seeds, None, 3, s, 1.0, 0.9, 0.95, 0.03, -0.01, 0.2 if sde else 0.0,
                         False, x, dp)

    for _ in range(20):
        launch()
    return event_ms(launch, 200)


def bench(name, B, rounds):
    model, cfg = configs.build_model(name, device="cuda")
    diff = model.diffusion
    tc, hw = model.cond_frame_num, cfg["dataset_params"]["frame_shape"]
    clip = torch.rand((B, 3, tc, hw, hw), generator=torch.Generator().manual_seed(0)).cuda()
    _, x_cond, cond_fea, _ = model.condition(clip)
    gen = torch.Generator().manual_seed(1)

    def arm(solver, S):
        def run():
            diff.solver, diff.sampling_timesteps, diff.is_ddim_sampling = solver, S, True
            diff.sample(x_cond, cond_fea=cond_fea, seeds=torch.randint(0, 2 ** 62, (B,), dtype=torch.long,
                                                                      generator=gen))
        return run

    runs = [(f"{label}_S{S}", arm(solver, S)) for label, solver, S in ARMS]
    for _, fn in runs:                                                   # warm-up: graph capture, clocks
        fn()
        fn()
    times = {k: [] for k, _ in runs}
    for _ in range(rounds):
        for k, fn in runs:
            times[k].append(event_ms(fn))
    diff.solver = None
    n = 3 * (diff.num_frames - tc) * x_cond.shape[3] * x_cond.shape[4]
    kern = {}
    for label, b in (("round_size", B), ("x16", 16 * B)):
        bound_ms = b * n * BYTES_PER_ELEMENT / HBM_BYTES_PER_S * 1e3
        for mode, sde in (("ode", False), ("sde_philox", True)):
            ms = kernel_time(b, n, sde)
            kern[f"{label}_{mode}"] = {"batch": b, "elements": b * n, "ms": round(ms, 5),
                                       "hbm_bound_ms": round(bound_ms, 5), "bound_over_time": round(bound_ms / ms, 3)}
    ddim = statistics.median(times["ddim_S10"])
    return {"dataset": name, "batch": B, "rounds": rounds,
            "round_ms": {k: spread(v) for k, v in times.items()},
            "over_ddim_S10": {k: round(statistics.median(v) / ddim, 4) for k, v in times.items()},
            "update_kernel": kern}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--datasets", default="bair,kth")
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--rounds", type=int, default=10)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("solver_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    res = [bench(n, a.batch, a.rounds) for n in a.datasets.split(",")]
    print(json.dumps({"gpu": torch.cuda.get_device_name(), "power_limit": power_limit(), "results": res}))


if __name__ == "__main__":
    main()
