"""Cost of prediction with known future frames against one plain sampling round, one GPU, synthetic weights.

    python tools/keyframe_bench.py [--datasets bair,kth] [--batch 32] [--rounds 10]

For each dataset (its shipped DDIM configuration): ms per call of FlowDiffusion.sample_with_keyframes with one known
frame, the last predicted one (conditioning, encode_future over tc + tp frames, the S-step DDIM loop with S + 1
replacements as one CUDA graph, decode; per-video seeds), against sample_one_video on the same clips, each after two
warm-up calls (graph capture), timed alternately with CUDA events; median (min-max).  Then the extdm_impose_known
kernel alone (DDIM coefficient mode), timed with CUDA events over 200 launches, against its HBM byte bound at 7.7
TB/s.  Per element of a known frame it reads x_known and writes x, 8 bytes, plus 4 for eps when eps is injected;
elements of unknown frames move no data; the mask is one byte per (video, frame).  It is timed with the last frame
known and with every frame known, at the round's size (which stays in the 126 MB L2 across launches) and at 16 times
that size (beyond L2).  Reads the card name and power limit in the same run; prints one JSON line.  No sample quality
is measured: the weights are random.
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


def kernel_bytes(known, per_frame, injected):
    """HBM bytes one extdm_impose_known launch must move: x_known read and x written (and eps read when injected) at
    the known frames, plus the mask."""
    return int(known.sum()) * per_frame * (12 if injected else 8) + known.numel()


def kernel_time(shape, known, injected):
    """ms per extdm_impose_known launch on (B, 3, tp, h, w) fp32 tensors."""
    g = torch.Generator(device="cuda").manual_seed(0)
    x, xk = (torch.randn(shape, device="cuda", generator=g) for _ in range(2))
    noise = torch.randn(1, *shape, device="cuda", generator=g) if injected else None
    seeds = None if injected else torch.arange(shape[0], dtype=torch.long, device="cuda")
    known = known.cuda()

    def launch():
        ops.impose_known(ops.IMMEDIATE, x, xk, known, seeds, noise, 0.7, 0.7, 0, False)

    for _ in range(20):
        launch()
    return event_ms(launch, 200)


def bench(name, B, rounds):
    model, cfg = configs.build_model(name, device="cuda")
    tc, tp, hw = model.cond_frame_num, model.pred_frame_num, cfg["dataset_params"]["frame_shape"]
    clips = torch.rand((B, 3, tc + tp, hw, hw), generator=torch.Generator().manual_seed(0)).cuda()
    past = clips[:, :, :tc].contiguous()
    last = torch.zeros(B, tp, dtype=torch.bool)
    last[:, tp - 1] = True
    gen = torch.Generator().manual_seed(1)

    def seeds():
        return torch.randint(0, 2 ** 62, (B,), dtype=torch.long, generator=gen)

    runs = [("sample_one_video", lambda: model.sample_one_video(cond_scale=1.0, real_vid=past, seeds=seeds())),
            ("sample_with_keyframes", lambda: model.sample_with_keyframes(clips, last, seeds=seeds()))]
    for _, fn in runs:                                                   # warm-up: graph capture, clocks
        fn()
        fn()
    times = {k: [] for k, _ in runs}
    for _ in range(rounds):
        for k, fn in runs:
            times[k].append(event_ms(fn))
    x_shape = tuple(model.encode_future(clips).shape)
    per_frame = 3 * x_shape[3] * x_shape[4]
    kern = {}
    for label, b in (("round_size", B), ("x16", 16 * B)):
        for mask_name in ("last", "all"):
            known = torch.zeros(b, tp, dtype=torch.bool)
            known[:, tp - 1 if mask_name == "last" else slice(None)] = True
            for mode, injected in (("philox", False), ("injected", True)):
                nbytes = kernel_bytes(known, per_frame, injected)
                bound_ms = nbytes / HBM_BYTES_PER_S * 1e3
                ms = kernel_time((b, *x_shape[1:]), known, injected)
                kern[f"{label}_{mask_name}_{mode}"] = {"batch": b, "bytes": nbytes, "ms": round(ms, 5),
                                                       "hbm_bound_ms": round(bound_ms, 5),
                                                       "bound_over_time": round(bound_ms / ms, 3)}
    base = statistics.median(times["sample_one_video"])
    return {"dataset": name, "batch": B, "rounds": rounds, "sampling_timesteps": int(model.diffusion.sampling_timesteps),
            "call_ms": {k: spread(v) for k, v in times.items()},
            "over_sample_one_video": {k: round(statistics.median(v) / base, 4) for k, v in times.items()},
            "impose_kernel": kern}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--datasets", default="bair,kth")
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--rounds", type=int, default=10)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("keyframe_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    res = [bench(n, a.batch, a.rounds) for n in a.datasets.split(",")]
    print(json.dumps({"gpu": torch.cuda.get_device_name(), "power_limit": power_limit(), "results": res}))


if __name__ == "__main__":
    main()
