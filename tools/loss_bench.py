"""Denoising-loss evaluation (FlowDiffusion.denoising_loss) against one DDIM round on the same batch, one GPU, synthetic
weights.

    python tools/loss_bench.py [--datasets bair,kth] [--batch 32] [--rounds 10]

For each dataset, on clips of tc + tp frames (the loss's input) at `--batch` videos, after warm-up calls of every timed
function (graph capture, clocks), `--rounds` alternating rounds, each timed with CUDA events:
  * loss: one FlowDiffusion.denoising_loss call (LFAE conditioning over tc + tp frames, cond_fea, then the captured
    graph of GaussianDiffusion.denoising_loss) with fresh timesteps and seeds -> videos/s;
  * its split: loss_inputs (the LFAE conditioning and cond_fea) and the graph (UNet prologue, forward diffusion, time
    MLP, UNet step, loss) on the same inputs;
  * ddim: one FlowDiffusion.sample_one_video round (conditioning over tc frames, 10 DDIM steps, decode) on the first tc
    frames of the same clips, with seeds, and its GaussianDiffusion.sample alone.
The two new kernels are timed on their own, eagerly, `KERNEL_REPS` launches between one event pair, on the graph's
shapes: q_sample (seeded, as shipped) and denoise_loss; graph_call_minus_kernels_ms is the rest of the graph call
(input copies, UNet prologue, time MLP, UNet step).  Their inputs (a few MB) stay in the 126 MB L2 between
launches; their HBM byte bound (bytes moved once / 7.7 TB/s, the data-sheet bandwidth) is printed beside them.  Reads
the card name and power limit in the same run.  Prints one JSON line.
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

KERNEL_REPS = 200


def bench(name, B, rounds):
    model, cfg = configs.build_model(name, device="cuda")
    diff = model.diffusion
    tc, tp, hw = model.cond_frame_num, model.pred_frame_num, cfg["dataset_params"]["frame_shape"]
    clip = torch.rand((B, 3, tc + tp, hw, hw), generator=torch.Generator().manual_seed(0)).cuda()
    cond = clip[:, :, :tc].contiguous()
    gen = torch.Generator().manual_seed(1)

    def draw():
        return (torch.randint(0, diff.num_timesteps, (B,), generator=gen),
                torch.randint(0, 2 ** 62, (B,), dtype=torch.long, generator=gen))

    inputs = model.loss_inputs(clip)
    arms = {
        "loss": lambda: model.denoising_loss(clip, *draw()),
        "loss_inputs": lambda: model.loss_inputs(clip),
        "loss_graph": lambda: diff.denoising_loss(*inputs, *draw()),
        "ddim_round": lambda: model.sample_one_video(1.0, cond, seeds=draw()[1]),
    }
    _, x_cond, cond_fea, _ = model.condition(cond)
    arms["ddim_sample"] = lambda: diff.sample(x_cond, cond_fea, seeds=draw()[1])
    for _ in range(3):                                                   # warm-up: graph capture, clocks
        for fn in arms.values():
            fn()
    t = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            t[k].append(event_ms(fn))

    # the new kernels alone, on the graph's buffers
    x_start = inputs[0]
    r = diff.denoise_fn.runner(B, x_start.shape[3], x_start.shape[4], inputs[2].shape[-1])
    g, st = next(v for k, v in r.graphs.items() if k[:2] == ("loss", tuple(x_start.shape)))
    R = ops.IMMEDIATE
    q_ms = event_ms(lambda: ops.q_sample(R, st["x_start"], r.time, st["seeds"], None, st["acp"], st["a1m"], r.x,
                                         st["eps"]), KERNEL_REPS)
    l_ms = event_ms(lambda: ops.denoise_loss(R, st["eps"], r.out, st["lpf"], diff.loss_type == "l1"), KERNEL_REPS)
    n = x_start.numel()
    q_bytes = 3 * 4 * n + 2 * 8 * B                                      # x_start in, x_t + eps out; t, seeds
    l_bytes = 2 * 4 * n + 4 * B * tp                                     # eps, pred in; (B, tp) out
    med = {k: statistics.median(v) for k, v in t.items()}
    kern = {"q_sample_us": round(1e3 * q_ms, 2), "q_sample_bytes": q_bytes,
            "q_sample_hbm_bound_us": round(1e6 * q_bytes / HBM_BYTES_PER_S, 2),
            "denoise_loss_us": round(1e3 * l_ms, 2), "denoise_loss_bytes": l_bytes,
            "denoise_loss_hbm_bound_us": round(1e6 * l_bytes / HBM_BYTES_PER_S, 2)}
    return {"dataset": name, "batch": B, "frames": tc + tp, "rounds": rounds,
            "loss_videos_per_s": round(B / (med["loss"] / 1e3), 1),
            "ms": {k: spread(v) for k, v in t.items()},
            "graph_call_minus_kernels_ms": round(med["loss_graph"] - (q_ms + l_ms), 3),
            "kernels": kern,
            "ddim_round_over_loss": round(med["ddim_round"] / med["loss"], 3),
            "ddim_sample_over_loss_graph": round(med["ddim_sample"] / med["loss_graph"], 3)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--datasets", default="bair,kth")
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--rounds", type=int, default=10)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("loss_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    res = [bench(n, a.batch, a.rounds) for n in a.datasets.split(",")]
    print(json.dumps({"gpu": torch.cuda.get_device_name(), "power_limit": power_limit(), "results": res}))


if __name__ == "__main__":
    main()
