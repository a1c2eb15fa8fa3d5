"""Stage-1 reconstruction throughput: FlowAE.reconstruct on the CUDA graph against the torch modules, one GPU,
synthetic weights from configs.build_model.

    python tools/recon_bench.py [--datasets kth,bair,cityscapes] [--batch 32] [--rounds 5]

For each dataset: batch --batch of the full evaluation clip (cond + predicted frames: KTH 10 + 40 = 50, BAIR 2 + 28 = 30,
Cityscapes-128 2 + 28 = 30), source frame 0.  Three arms: the native graph, the torch modules at PyTorch defaults
(cuDNN TF32 on) and the torch modules with TF32 off.  After one warm-up call of each arm (graph capture, cuDNN
algorithm choice), --rounds rounds time one call of each arm in turn with CUDA events around a synchronised call.
A call is the whole FlowAE.reconstruct: input staging, the stage, the output copies.  Reports reconstructed frames/s
(B*T / call time) as median and min-max over rounds; the flow difference of the native arm and of the cuDNN-TF32 arm
against the fp32 arm (max-abs, and the share of flow values off by more than 1e-2), and the native frames' PSNR against
the fp32 arm; the card name and its power limit.  Prints one JSON line.
"""
import argparse
import gc
import json
import math
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402
import extdm_b200  # noqa: E402,F401
from extdm_b200 import configs  # noqa: E402
from extdm_b200.flow_autoenc import FlowAE  # noqa: E402
from benchlib import event_ms, power_limit, spread  # noqa: E402


def bench(name, batch, rounds):
    model, cfg = configs.build_model(name, device="cuda")
    ae = FlowAE.from_flow_diffusion(model)
    T = model.cond_frame_num + cfg["dataset_params"]["valid_params"]["pred_frames"]
    hw = cfg["dataset_params"]["frame_shape"]
    g = torch.Generator().manual_seed(31)
    coarse = torch.rand((batch, 3, T // 4, 8, 8), generator=g)
    vid = F.interpolate(coarse, size=(T, hw, hw), mode="trilinear", align_corners=True).clamp(0, 1).cuda()

    def native():
        return ae.reconstruct(vid, 0)

    def torch_arm(tf32):
        def run():
            old = torch.backends.cudnn.allow_tf32
            torch.backends.cudnn.allow_tf32 = tf32
            try:
                return ae.reconstruct_torch(vid, 0)
            finally:
                torch.backends.cudnn.allow_tf32 = old
        return run

    arms = {"native_graph": native, "torch_default": torch_arm(torch.backends.cudnn.allow_tf32),
            "torch_fp32": torch_arm(False)}
    outs = {k: fn() for k, fn in arms.items()}                            # warm-up
    flow_err = {}
    for k in ("native_graph", "torch_default"):
        d = (outs[k]["optical_flow"] - outs["torch_fp32"]["optical_flow"]).abs()
        flow_err[f"{k}_vs_fp32_flow_max_abs"] = d.max().item()
        flow_err[f"{k}_vs_fp32_flow_share_over_1e-2"] = (d > 1e-2).float().mean().item()
    mse = ((outs["native_graph"]["prediction"] - outs["torch_fp32"]["prediction"]) ** 2).mean().item()
    del outs
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            times[k].append(event_ms(fn))
    frames = batch * T
    res = {"dataset": name, "batch": batch, "frames_per_video": T, "hw": hw}
    for k, ts in times.items():
        res[f"{k}_frames_per_s"] = spread([frames / (t / 1e3) for t in ts], digits=1)
        res[f"{k}_ms"] = [round(t, 2) for t in ts]
    med = {k: statistics.median(ts) for k, ts in times.items()}
    res["speedup_vs_torch_default"] = round(med["torch_default"] / med["native_graph"], 2)
    res["speedup_vs_torch_fp32"] = round(med["torch_fp32"] / med["native_graph"], 2)
    res.update(flow_err)
    res["native_vs_fp32_prediction_psnr_db"] = round(99.0 if mse == 0 else -10 * math.log10(mse), 2)
    del ae, model, vid
    gc.collect()
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--datasets", default="kth,bair,cityscapes")
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("recon_bench.py measures on a CUDA device; none is available")
    results = [bench(n, args.batch, args.rounds) for n in args.datasets.split(",")]
    print(json.dumps({"gpu": torch.cuda.get_device_name(), "power_limit": power_limit(),
                      "cudnn_allow_tf32_default": torch.backends.cudnn.allow_tf32, "results": results}))


if __name__ == "__main__":
    main()
