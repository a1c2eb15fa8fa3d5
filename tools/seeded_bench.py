"""DDIM with per-video seeds against DDIM with its default torch.randn noise, one GPU, synthetic weights.

    python tools/seeded_bench.py [--datasets bair,kth] [--batch 32] [--rounds 20]

For each dataset: after warm-up rounds of both modes (graph capture, clocks), times `--rounds` rounds of each mode
alternately with CUDA events.  A round is one GaussianDiffusion.sample call (10 DDIM steps, CUDA-graphed as shipped) on
the conditioning of one clip: with default noise it includes the torch.randn draws and the copy into the graph's noise
buffer, with seeds the pinned host-to-device copy of the seeds.  Reports the median, min and max ms per round of each
mode, and the bytes of sampler noise state computed from shapes at 10 and 250 DDIM steps: the default path holds the
drawn noise tensor and the graph's copy of it, the seeded path one int64 per video.  Reads the card name and power limit
in the same run.  Prints one JSON line.
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
from extdm_b200 import configs  # noqa: E402
from benchlib import event_ms, power_limit, spread  # noqa: E402

STEPS = 10


def noise_state_bytes(shape, steps, B):
    """(default, seeded) bytes of sampler noise state: S fp32 noise tensors drawn per call plus the graph's copy of
    them, against the graph's (B,) int64 seed buffer."""
    n = 4
    for d in shape:
        n *= d
    return 2 * steps * n, 8 * B


def bench(name, B, rounds):
    model, cfg = configs.build_model(name, device="cuda")
    diff = model.diffusion
    diff.sampling_timesteps, diff.is_ddim_sampling = STEPS, True
    tc, hw = model.cond_frame_num, cfg["dataset_params"]["frame_shape"]
    clip = torch.rand((B, 3, tc, hw, hw), generator=torch.Generator().manual_seed(0)).cuda()
    _, x_cond, cond_fea, _ = model.condition(clip)
    gen = torch.Generator().manual_seed(1)

    def default():
        diff.sample(x_cond, cond_fea=cond_fea)

    def seeded():
        diff.sample(x_cond, cond_fea=cond_fea, seeds=torch.randint(0, 2 ** 62, (B,), dtype=torch.long, generator=gen))

    for _ in range(3):                                                   # warm-up: graph capture, clocks
        default()
        seeded()
    t = {"default": [], "seeded": []}
    for _ in range(rounds):
        t["default"].append(event_ms(default))
        t["seeded"].append(event_ms(seeded))
    shape = (B, 3, diff.num_frames - x_cond.shape[2], x_cond.shape[3], x_cond.shape[4])
    mem = {}
    for steps in (STEPS, 250):
        d, s = noise_state_bytes(shape, steps, B)
        mem[f"S{steps}"] = {"default_bytes": d, "seeded_bytes": s}
    med_d, med_s = statistics.median(t["default"]), statistics.median(t["seeded"])
    return {"dataset": name, "batch": B, "steps": STEPS, "rounds": rounds,
            "default_ms": spread(t["default"]), "seeded_ms": spread(t["seeded"]),
            "seeded_over_default": round(med_s / med_d, 4), "noise_state": mem,
            "default_rounds_ms": [round(x, 3) for x in t["default"]],
            "seeded_rounds_ms": [round(x, 3) for x in t["seeded"]]}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--datasets", default="bair,kth")
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--rounds", type=int, default=20)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("seeded_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    res = [bench(n, a.batch, a.rounds) for n in a.datasets.split(",")]
    print(json.dumps({"gpu": torch.cuda.get_device_name(), "power_limit": power_limit(), "results": res}))


if __name__ == "__main__":
    main()
