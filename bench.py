#!/usr/bin/env python
"""bench.py -- predicted frames/s of the ExtDM sampling hot path (BASELINE.json metric) on N B200s.

  python bench.py [--gpus N] [--steps K] [--warmup W]           # this repo's CUDA path
  python bench.py [...] --dump-outputs DIR                      # + the last timed step's predicted frames, as .npy
  python bench.py --impl reference [...]                        # the UNMODIFIED reference on the host CPU cores

Headline workload = the configuration BASELINE.json's metric names: BAIR 64x64, 2 -> 28 autoregressive rollout
(3 rounds of conditioning + 10 DDIM steps + 12-frame decode), 32 synthetic clips per GPU (at N = 8 this is BASELINE
config 3, batch 256 over 8 GPUs).  A "step" is one full rollout of one batch.  Videos shard over ranks (weak scaling, no
data-path collective); the predicted frames are all-gathered over NCCL at the end of a step.  Rank 0 prints ONE JSON
line.  Besides the base contract's keys the line carries

  per_config            the other BASELINE configurations on the same GPUs (SMMNIST b32 and the config-1 batch-1 case,
                        KTH, UCF batch sweep, Cityscapes 128x128 / 64x64), device-timed rollouts
  cpu_baseline          the unmodified reference (oracle/_ref, kind "reference") on the host cores: BAIR, 1 video,
                        the full 3-round rollout, really timed (N = 1 only)
  gpu_eager_reference   the same unmodified reference in PyTorch eager on the same B200 (the "kernel to beat", SURVEY.md
                        8d): BAIR, the bench batch, TF32 default (cudnn on, matmul off) and TF32 off, plus a live
                        full-batch parity figure of this repo's path against it (same weights, same injected noise)
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HEADLINE = "bair"
BATCH = 32
try:
    METRIC = json.load(open(os.path.join(ROOT, "BASELINE.json")))["metric"]
except Exception:
    METRIC = "predicted frames/sec (DDIM, SMMNIST/BAIR 64²) at 1/2/4/8 B200; roofline %"

DESCR = {
    "bair": "BAIR 64x64 ch3, 2->28 autoregressive rollout (3 rounds x 10 DDIM steps, eta=1, dynamic threshold; "
            "VideoFlowDiffusion_multi_w_ref + traj_u12 UNet3D)",
    "smmnist": "SMMNIST 64x64 ch1->3, 10->10 rollout (2 rounds; VideoFlowDiffusion_multi1248 + base UNet3D)",
    "kth": "KTH 64x64 ch1->3, 10->40 rollout (2 rounds; multi_w_ref + traj_ada UNet3D)",
    "ucf": "UCF-101 64x64 ch3, 4->12 rollout (2 rounds; multi_w_ref + traj_ada UNet3D, 64 regions)",
    "cityscapes": "Cityscapes 128x128 ch3 (shipped yaml: scale factor 0.25, perspective bg), 2->28 rollout (6 rounds; "
                  "multi_w_ref + traj_ada UNet3D)",
    "cityscapes64": "Cityscapes 64x64 ch3 (BASELINE.json wording; scale factor 0.5), 2->28 rollout (6 rounds)",
}
GRAY = ("smmnist", "kth")


# ------------------------------------------------------------------------------------------------ helpers
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.thread.join(timeout=2)
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx[0] if mx else None,
                "reasons": reasons, "samples": len(sm)}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p.get("bf16_tflops_sustained"),
                "hbm_gbs": p["hbm_gbs"], "source": "measured"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback"}


def make_clip(name, B, tc, hw, seed):
    """Synthetic conditioning clips in [0, 1] on the host; gray datasets replicate one channel to three
    (data/video_dataset.py:26-33)."""
    import torch
    g = torch.Generator(device="cpu").manual_seed(seed)
    c = 1 if name in GRAY else 3
    return torch.rand(B, c, tc, hw, hw, generator=g).expand(B, 3, tc, hw, hw).contiguous()


DUMP_BYTES = 64_000_000


def dump_frames(path, frames, seed=0):
    """--dump-outputs: the predicted frames (B, 3, T, H, W) of the last timed step as <path>/pred_frames.npy, float32.
    Above DUMP_BYTES only a fixed, seeded subset of the videos is written, in index order; a single video over
    DUMP_BYTES is cut to its first frames (one frame of 3 x H x W floats is assumed to fit)."""
    import numpy as np
    import torch
    per_video = frames[0].numel() * 4
    if frames.shape[0] * per_video > DUMP_BYTES:
        keep = max(1, DUMP_BYTES // per_video)
        idx = torch.randperm(frames.shape[0], generator=torch.Generator().manual_seed(seed))[:keep].sort().values
        frames = frames[idx.to(frames.device)]
    if frames.numel() * 4 > DUMP_BYTES:
        frames = frames[:, :, :DUMP_BYTES // (frames[0, :, 0].numel() * 4)]
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "pred_frames.npy"), frames.float().cpu().numpy())


# ------------------------------------------------------------------------------------------------ reference legs
def build_reference(name, device, seed=1234):
    """The UNMODIFIED reference FlowDiffusion for a dataset (oracle/_ref staged by oracle/make_ref.py, import shims of
    oracle/ref_shims.py), with the same deterministic synthetic weights as configs.build_model(name, seed)."""
    import importlib
    import torch
    import yaml
    import extdm_b200  # noqa: F401
    from extdm_b200 import configs
    from extdm_b200.weights import synth_state_dict
    from oracle import ref_shims
    if not ref_shims.available():
        raise FileNotFoundError(f"{ref_shims.REF_ROOT}: run oracle/make_ref.py in the build container")
    ref_shims.install()
    ref_shims.cuda_identity(device == "cpu")
    _, dm_arch, unet_arch = configs.dataset(name)
    ds = {"cityscapes64": "cityscapes"}.get(name, name)
    cfg = yaml.safe_load(open(os.path.join(ref_shims.REF_ROOT, "config", "DM", ds + ".yaml")))
    cfg["flow_params"]["model_params"]["generator_params"]["pixelwise_flow_predictor_params"][
        "estimate_occlusion_map"] = True                   # scripts/DM/valid.py:81 with --estimate_occlusion_map
    kw = dict(config=cfg, pretrained_pth="", is_train=False)
    if dm_arch != "VideoFlowDiffusion_multi1248":
        kw["Unet3D_architecture"] = unet_arch
    devnull = open(os.devnull, "w")
    stdout, sys.stdout = sys.stdout, devnull               # the wrappers print their config
    try:
        fd = importlib.import_module("model.BaseDM_adaptor." + dm_arch).FlowDiffusion(**kw).eval()
    finally:
        sys.stdout = stdout
    for i, part in enumerate(("generator", "region_predictor", "bg_predictor", "diffusion")):
        m = getattr(fd, part)
        base = m.state_dict()
        m.load_state_dict(synth_state_dict({k: tuple(v.shape) for k, v in base.items()}, seed + i, base=base))
    fd = fd.to(device)                                     # scripts/DM/valid.py:113 model.cuda()
    return fd, cfg


def reference_rollout(fd, clip_host, total_pred, device):
    """The autoregressive loop of scripts/DM/valid.py:167-172, host tensors in and out (`.cuda()` / `.cpu()` per round)."""
    import torch
    tc, tp = fd.cond_frame_num, fd.pred_frame_num
    preds, cond = [], clip_host
    with torch.no_grad():
        for _ in range(math.ceil(total_pred / tp)):
            out = fd.sample_one_video(cond_scale=1.0, real_vid=cond.to(device))["sample_out_vid"].clone().detach().cpu()
            preds.append(out[:, :, -tp:])
            cond = out[:, :, -tc:]
    return torch.cat(preds, dim=2)[:, :, :total_pred]


class _Quiet:
    """tqdm progress bars of the reference's sampling loop go to stderr: silence them for the timed legs."""

    def __enter__(self):
        self.fd = os.dup(2)
        self.null = os.open(os.devnull, os.O_WRONLY)
        os.dup2(self.null, 2)

    def __exit__(self, *a):
        os.dup2(self.fd, 2)
        os.close(self.null)
        os.close(self.fd)


def cpu_reference(name=HEADLINE, videos=1, repeats=1, threads=None):
    """The unmodified reference on the host cores: `videos` clips of `name`, the FULL rollout (every round: conditioning,
    10 DDIM steps, decode), really timed.  Warm-up = one rollout with sampling_timesteps = 1 (creates every oneDNN
    primitive; the attribute is the reference's own knob, Diffusion.py:212).  -> (cpu_baseline dict, seconds per rollout)"""
    import torch
    from extdm_b200 import configs
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    fd, cfg = build_reference(name, "cpu")
    total = configs.dataset(name)[0]["dataset_params"]["valid_params"]["pred_frames"]
    tc, hw = fd.cond_frame_num, cfg["dataset_params"]["frame_shape"]
    clip = make_clip(name, videos, tc, hw, 1000)
    steps = fd.diffusion.sampling_timesteps
    with _Quiet():
        fd.diffusion.sampling_timesteps = 1
        reference_rollout(fd, clip, total, "cpu")
        fd.diffusion.sampling_timesteps = steps
        times = []
        for _ in range(repeats):
            t0 = time.perf_counter()
            out = reference_rollout(fd, clip, total, "cpu")
            times.append(time.perf_counter() - t0)
    assert out.shape[2] == total
    sec = sum(times) / len(times)
    rounds = math.ceil(total / fd.pred_frame_num)
    return {"value": videos * total / sec, "unit": "frames/s", "cores": threads, "kind": "reference",
            "sample": f"{DESCR[name]}: {videos} of the step's videos, the whole {rounds}-round rollout "
                      f"(conditioning + {steps} DDIM steps + decode per round) really timed: {sec:.1f} s per rollout, "
                      f"{repeats} timed after a 1-DDIM-step warm-up rollout; unmodified reference from oracle/_ref, fp32, "
                      f"torch {torch.__version__}", "seconds_per_rollout": sec, "timed_rollouts": repeats}, sec


def cpu_port_fallback(threads=None, repeats=1):
    """Only when oracle/_ref was not staged: the oracle port (kind 'port'), one BAIR round at batch 1, timed `repeats`
    times."""
    import torch
    from oracle import extdm_oracle as O
    from extdm_b200.manifest import UnetConfig, unet_manifest
    from extdm_b200.weights import synth_state_dict
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    tc, tp = 2, 10
    sd = {"denoise_fn." + k: v for k, v in synth_state_dict(unet_manifest(UnetConfig("u12", tc, tp)), seed=1).items()}
    g = torch.Generator().manual_seed(0)
    x_cond = torch.randn(1, 3, tc, 32, 32, generator=g)
    fea = torch.randn(1, 256, tc + tp, 16, 16, generator=g)
    nz = [torch.randn(1, 3, tp, 32, 32, generator=g) for _ in range(10)]
    with torch.no_grad():
        O.ddim_sample(O.SD(sd), O.unet_config("u12", tc, tp), x_cond, fea, nz[0], nz[1:2] + [None], sampling=1)
        times = []
        for _ in range(repeats):
            t0 = time.perf_counter()
            O.ddim_sample(O.SD(sd), O.unet_config("u12", tc, tp), x_cond, fea, nz[0], nz[1:] + [None], sampling=10)
            times.append(time.perf_counter() - t0)
        sec = sum(times) / len(times)
    return {"value": tp / sec, "unit": "frames/s", "cores": threads, "kind": "port",
            "sample": f"oracle/_ref not staged: oracle port, BAIR u12 batch 1, ONE round's 10-step DDIM loop timed "
                      f"{repeats}x ({sec:.1f} s each; conditioning and decode excluded)"}, sec


def run_reference_arm(args):
    """`--impl reference`: the reference's own CPU implementation of the path on the host cores, on the headline
    configuration (bounded sample: one video per step, the whole rollout) and on BASELINE config 1 (SMMNIST 10->10,
    batch 1).  `--steps` timed repeats are really executed (one rollout on the host cores takes minutes)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle import ref_shims
    n = args.steps
    if ref_shims.available():
        cb, sec = cpu_reference(HEADLINE, videos=1, repeats=n)
        try:
            c1, s1 = cpu_reference("smmnist", videos=1, repeats=1)
            per_config = {"smmnist_b1": {"workload": "BASELINE config 1: " + DESCR["smmnist"] + ", batch 1",
                                         "value": c1["value"], "unit": "frames/s", "seconds_per_rollout": s1}}
        except Exception as e:
            per_config = {"smmnist_b1": {"error": str(e)}}
    else:
        cb, sec = cpu_port_fallback(repeats=n)
        per_config = {}
    line = {"metric": METRIC, "value": cb["value"], "unit": "frames/s", "n_gpus": args.gpus, "steps": n,
            "steps_requested": args.steps, "warmup": 1, "ms_per_step": 1e3 * sec, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": DESCR[HEADLINE] + "; bounded sample: 1 video per step on the host CPU cores "
                                                     "(see cpu_baseline.sample)"},
            "cpu_baseline": cb, "per_config": per_config,
            "e2e": {"value": cb["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def gpu_eager_reference(model, name, B, total_pred, dev):
    """SURVEY.md 8d "kernel to beat": the unmodified reference in PyTorch eager on this GPU (cuDNN / cuBLAS / ATen), the
    bench batch, the whole rollout with the reference driver's per-round host hops; PyTorch's default precision flags
    (cudnn.allow_tf32 = True, matmul TF32 off -- scripts/DM/valid.py never changes them) and true fp32.  Then one round
    with injected noise through both implementations (same weights, same clips): parity at the full bench batch."""
    import torch
    fd, cfg = build_reference(name, dev)
    tc, tp, hw = fd.cond_frame_num, fd.pred_frame_num, cfg["dataset_params"]["frame_shape"]
    clip = make_clip(name, B, tc, hw, 1000)
    out = {"workload": DESCR[name] + f", batch {B}, PyTorch {torch.__version__} eager on the same GPU"}
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    try:
        with _Quiet():
            for key, conv_tf32 in (("tf32_default", True), ("fp32", False)):
                torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = conv_tf32, False
                reference_rollout(fd, clip, total_pred, dev)            # warm-up (cuDNN heuristics, allocator)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                reference_rollout(fd, clip, total_pred, dev)
                torch.cuda.synchronize()
                sec = time.perf_counter() - t0
                out[key] = {"value": B * total_pred / sec, "unit": "frames/s", "ms_per_step": 1e3 * sec}
            # ---- parity at full batch: one round, injected noise; the reference's PCA runs on cuSOLVER here, this repo's
            # in its closed form with the same sign convention.  Smooth, natural-video-like clips (the recipe of the test
            # fixtures): the white-noise clips of the throughput runs make frame PSNR a measure of the noise, not the path.
            import torch.nn.functional as F
            gc = torch.Generator(device="cpu").manual_seed(1000)
            coarse = torch.rand((B, 1 if name in GRAY else 3, 4, 8, 8), generator=gc)
            clip = F.interpolate(coarse, size=(tc, hw, hw), mode="trilinear", align_corners=True).clamp(0, 1)
            clip = clip.expand(B, 3, tc, hw, hw).contiguous()
            steps = fd.diffusion.sampling_timesteps
            g = torch.Generator(device="cpu").manual_seed(77)
            noise = torch.randn(steps, B, 3, tp, 32, 32, generator=g).to(dev)
            queue = [noise[i] for i in range(steps)]
            real_randn, real_randn_like = torch.randn, torch.randn_like
            torch.randn = lambda *a, **k: queue.pop(0)
            torch.randn_like = lambda *a, **k: queue.pop(0)
            torch.backends.cudnn.allow_tf32 = False
            try:
                with torch.no_grad():
                    want = fd.sample_one_video(cond_scale=1.0, real_vid=clip.to(dev))
            finally:
                torch.randn, torch.randn_like = real_randn, real_randn_like
        got = model.sample_one_video(cond_scale=1.0, real_vid=clip.to(dev), noise=noise)
        rel = lambda a, b: ((a.float() - b.float()).norm() / b.float().norm()).item()
        mse = ((got["sample_out_vid"] - want["sample_out_vid"]) ** 2).mean().item()
        out["parity_full_batch"] = {
            "what": f"one sample_one_video round, batch {B}, {steps} DDIM steps, injected noise, smooth synthetic clips: "
                    "this repo's path vs the reference on the same GPU in fp32",
            "cond_flow_max_abs": (got["real_vid_grid"] - want["real_vid_grid"]).abs().max().item(),
            "pred_flow_rel_l2": rel(got["sample_vid_grid"][:, :, tc:], want["sample_vid_grid"][:, :, tc:]),
            "frames_psnr_db": 99.0 if mse == 0 else 10 * math.log10(1.0 / mse)}
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
        del fd
        torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------ GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dataset", default=HEADLINE, choices=sorted(DESCR))
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-per-config", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true")
    ap.add_argument("--profile-kernels", action="store_true", help="also print the per-kernel time table")
    ap.add_argument("--ncu-range", action="store_true",
                    help="for `ncu --profile-from-start off`: after the warm-up, bracket ONE step with "
                         "cudaProfilerStart/Stop and exit without printing a bench line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the predicted frames of the last timed step to DIR/pred_frames.npy (float32; above "
                         "64 MB a fixed, seeded subset of the videos), to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist
    import extdm_b200  # noqa: F401
    from extdm_b200 import configs, lib, sharding

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib.load()                                                # fails loudly when the CUDA library is missing

    def time_rollouts(fn, n):
        """n calls of fn bracketed by barrier + synchronize, CUDA events, max over ranks -> ms per call."""
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms / n

    name, B = args.dataset, args.batch
    model, cfg = configs.build_model(name, seed=1234, device=dev)
    tc, tp = model.cond_frame_num, model.pred_frame_num
    hw = cfg["dataset_params"]["frame_shape"]
    total_pred = cfg["dataset_params"]["valid_params"]["pred_frames"]
    clip_host = make_clip(name, B, tc, hw, 1000 + rank)
    clip_dev = clip_host.to(dev)
    # end-to-end buffers: the step's input in pinned host memory, its result in pinned host memory; two of each so the
    # copies of neighbouring steps overlap the rollout (copy stream)
    pin_in = clip_host.pin_memory()
    pin_out = [torch.empty(B, 3, total_pred, hw, hw).pin_memory() for _ in range(2)]
    dev_in = [torch.empty_like(clip_dev) for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    h2d_done = [torch.cuda.Event() for _ in range(2)]
    keep = [None, None]
    last = {}                                                  # what the latest step_dev returned (--dump-outputs)

    def step_dev(i):
        pred = configs.rollout(model, clip_dev, total_pred)
        if world > 1:
            pred = sharding.gather_predictions(pred.contiguous(), world * B)
        last["pred"] = pred
        return pred

    def issue_h2d(i):
        with torch.cuda.stream(copy_stream):
            dev_in[i % 2].copy_(pin_in, non_blocking=True)
            h2d_done[i % 2].record(copy_stream)

    def step_e2e(i):
        """The end-to-end call with HOST buffers: H2D of this step's clips from pinned memory, the rollout (rounds stay
        on the device, SURVEY.md 8f-2), the gather, D2H of the predicted frames into pinned memory.  The copies run on
        a second stream: step i+1's input goes up and step i's frames come down while the neighbouring rollout runs."""
        main_stream = torch.cuda.current_stream()
        if i == 0:
            issue_h2d(0)
        main_stream.wait_event(h2d_done[i % 2])
        issue_h2d(i + 1)                                       # next step's input (same synthetic clips), overlapped
        pred = configs.rollout(model, dev_in[i % 2], total_pred)
        if world > 1:
            sharding.gather_predictions(pred.contiguous(), world * B)
        done = torch.cuda.Event()
        done.record(main_stream)
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(done)
            pin_out[i % 2].copy_(pred, non_blocking=True)
        keep[i % 2] = pred                                     # alive until its copy has run

    def timed_e2e(n):
        def body(i):
            step_e2e(i)
            if i == n - 1:
                torch.cuda.current_stream().wait_stream(copy_stream)       # every copy inside the timed region
        return time_rollouts(body, n)

    for i in range(max(args.warmup, 3)):
        step_dev(i)
    if args.ncu_range:
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        step_dev(0)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        sys.stderr.write("ncu range done (no bench value is reported from a profiled run)\n")
        return
    timed_e2e(1)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    # the timed steps draw their DDIM noise from the default generator: seeded here, the same arguments give the same
    # outputs run after run, whatever ran before
    torch.manual_seed(1234)
    ms_dev = time_rollouts(step_dev, args.steps)
    ms_e2e = timed_e2e(args.steps)
    clock_info = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_frames(args.dump_outputs, last["pred"])

    # ---- kernel accounting: the per-kernel roofline, measured live with CUDA events (eager replay of the launch lists)
    runner = next(iter(model.unet._runners.values()))
    dec = next(r_ for k_, r_ in model.generator._runners.items() if k_[0] != "enc")
    n_rounds = math.ceil(total_pred / tp)
    n_ddim = model.diffusion.sampling_timesteps
    cond_recs = [r_ for cr in model._cond_runners.values() for r_ in cr.recorders()]
    cond_recs += [r_.rec for k_, r_ in model.generator._runners.items() if k_[0] == "enc"]
    # launches of this library per step (the DDIM loop is replayed from a CUDA graph, so they are counted from the
    # launch lists: prologue + 10 x (step list + threshold + update) + decode + conditioning, per round)
    launches_per_step = n_rounds * (len(runner.prologue) + n_ddim * (len(runner.step) + 2) + len(dec.rec)
                                    + sum(len(r_) for r_ in cond_recs))
    peaks = load_peaks()
    table, shapes = {}, {}
    for rec_, mult in [(runner.prologue, 1), (runner.step, n_ddim), (dec.rec, 1)] + [(r_, 1) for r_ in cond_recs]:
        rec_.run()
        torch.cuda.synchronize()
        for kname, meta, ms in rec_.run_timed():
            if meta.get("tf32"):
                kname += "[tf32]"                         # the conditioning convolutions: fp32 operands, kind::tf32
            t = table.setdefault(kname, {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "n": 0})
            t["ms"] += ms * mult
            t["flops"] += meta.get("flops", 0.0) * mult
            t["bytes"] += meta.get("bytes", 0.0) * mult
            t["n"] += mult
            if kname == "extdm_conv_gemm":                 # the dominant GEMM SHAPE: all launches of one shape in a round
                sk = (meta["rows"], meta["n"], meta["k"], meta["taps"])
                e = shapes.setdefault(sk, [meta, 0.0, 0])
                e[1] += ms * mult
                e[2] += mult
    gemm = table["extdm_conv_gemm"]
    top_meta, top_ms_total, top_n = max(shapes.values(), key=lambda e: e[1])
    top = ("extdm_conv_gemm", top_meta, top_ms_total / top_n, top_n)         # (name, meta, mean ms per launch, launches per round)
    # The composite init_conv (DESIGN.md section 5) EXECUTES a 13x13 convolution of the flow (K = 832) + four 21-tap ring
    # corrections where the reference's algorithm -- and this path until round 2 -- runs a 7x7 convolution over 256 channels
    # (K = 12544): `achieved` counts executed FLOPs only, `achieved_at_reference_k` counts that operation at the
    # reference's K so that the figure stays comparable with earlier rounds.
    ref_extra = 0.0
    for m_ in runner.step.meta:
        if m_.get("taps") == 13 and m_.get("k") == 832:
            ref_extra += n_ddim * (2.0 * m_["rows"] * m_["n"] * 12544 - m_["flops"])
        elif m_.get("taps") == 21:
            ref_extra -= n_ddim * m_["flops"]
    total_kernel_ms = sum(t["ms"] for t in table.values())
    peak_tf, peak_bw = peaks["bf16_tflops"], peaks["hbm_gbs"]
    traffic = None                                    # dram bytes per launch of the top GEMM shape, from the ncu capture
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    top_key = f"rows={top[1]['rows']} n={top[1]['n']} k={top[1]['k']} taps={top[1]['taps']}"
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get(top_key)
    # The dominant kernel of a round is the tcgen05 implicit-GEMM (conv_gemm_kernel / conv_halo_kernel templates,
    # one C-ABI entry point): `achieved` is algorithmic FLOPs of ALL its launches in a round over their summed
    # CUDA-event durations; `top_launch` is its single most expensive shape; `other_kernels` are the rest.
    others = {}
    for kname, t in table.items():
        if kname == "extdm_conv_gemm":
            continue
        share = t["ms"] / total_kernel_ms
        if kname == "extdm_conv_gemm[tf32]":
            tf = t["flops"] / (t["ms"] * 1e-3) / 1e12
            others[kname] = {"bound": "tensor", "achieved": tf, "peak": peak_tf / 2, "unit": "TFLOP/s",
                             "frac": tf / (peak_tf / 2), "peak_source": "half the measured bf16 peak (tf32 rate)",
                             "share_of_kernel_time": share}
        elif t["flops"] > 0 and t["bytes"] == 0:
            tf = t["flops"] / (t["ms"] * 1e-3) / 1e12
            others[kname] = {"bound": "tensor", "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s",
                             "frac": tf / peak_tf, "share_of_kernel_time": share}
        elif t["bytes"] > 0:
            gbs = t["bytes"] / (t["ms"] * 1e-3) / 1e9
            others[kname] = {"bound": "hbm", "achieved": gbs, "peak": peak_bw, "unit": "GB/s", "frac": gbs / peak_bw,
                             "share_of_kernel_time": share}
            if t["flops"] > 0:                             # fused attention layers: also their executed tensor work
                others[kname]["tensor_tflops"] = t["flops"] / (t["ms"] * 1e-3) / 1e12
        elif share >= 0.005:
            others[kname] = {"share_of_kernel_time": share, "ms_per_round": t["ms"], "launches": t["n"]}
    roofline = {
        "bound": "tensor", "kernel": "extdm_conv_gemm (tcgen05 implicit GEMM: conv_gemm_kernel / conv_halo_kernel), all "
                                     f"{gemm['n']} launches of one round",
        "achieved": gemm["flops"] / (gemm["ms"] * 1e-3) / 1e12, "peak": peak_tf, "unit": "TFLOP/s",
        "frac": gemm["flops"] / (gemm["ms"] * 1e-3) / 1e12 / peak_tf, "peak_source": peaks["source"] + " burst",
        "achieved_at_reference_k": (gemm["flops"] + ref_extra) / (gemm["ms"] * 1e-3) / 1e12,
        "frac_at_reference_k": (gemm["flops"] + ref_extra) / (gemm["ms"] * 1e-3) / 1e12 / peak_tf,
        "note": "achieved / frac count EXECUTED FLOPs; *_at_reference_k counts the composite init_conv (13x13 convolution "
                "of the flow + ring correction) at the K = 12544 of the 7x7 convolution it replaces",
        "share_of_kernel_time": gemm["ms"] / total_kernel_ms,
        "traffic": traffic,
        "top_launch": {"shape": top_key, "achieved": top[1]["flops"] / (top[2] * 1e-3) / 1e12,
                       "frac": top[1]["flops"] / (top[2] * 1e-3) / 1e12 / peak_tf,
                       "algorithmic_bytes": top[1]["bytes"], "ms": top[2], "launches_per_round": top[3]},
        "other_kernels": others,
    }
    if args.profile_kernels and rank == 0:
        for kname, t in sorted(table.items(), key=lambda kv: -kv[1]["ms"]):
            sys.stderr.write(f"{kname:28s} {t['ms']:9.3f} ms/round  {t['n']:5d} launches  "
                             f"{t['flops'] / max(t['ms'], 1e-9) / 1e9:8.1f} TFLOP/s\n")
    executed_tflop_per_step = sum(t["flops"] for t in table.values()) * n_rounds / 1e12

    frames = world * B * total_pred
    line = {
        "metric": METRIC, "value": frames / (ms_dev * 1e-3), "unit": "frames/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_dev, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"{DESCR[name]}, batch {B} per GPU, random-init LFAE + DM",
                   "cache": "working set per step (GBs of activations) exceeds the 126 MB L2; no explicit flush",
                   "parallelism": f"dp{world} (videos sharded, one all_gather of predicted frames per step)"},
        "e2e": {"value": frames / (ms_e2e * 1e-3), "unit": "frames/s",
                "h2d_bytes_per_step": pin_in.numel() * 4, "d2h_bytes_per_step": pin_out[0].numel() * 4,
                "ms_per_step": ms_e2e, "copies": "pinned host buffers, H2D / D2H on a second stream overlapped with the "
                                                 "neighbouring step's rollout; all inside the timed region"},
        "gpu_launches": launches_per_step * args.steps,
        "gpu_launches_per_step": launches_per_step,
        "executed_tflop_per_step": executed_tflop_per_step,
        "end_to_end_tflops": executed_tflop_per_step / (ms_dev * 1e-3),
        "roofline": roofline,
        "clocks": clock_info,
        "kernel_time_ms_per_round": {k: round(v["ms"], 3) for k, v in table.items()},
    }

    # ---- the other BASELINE configurations on the same GPUs (device-timed, on-device rollout)
    if not args.no_per_config:
        del model, runner, dec, cond_recs, table
        torch.cuda.empty_cache()
        per = {}

        def measure(cname, b, label=None, mdl=None):
            m_, c_ = mdl if mdl is not None else configs.build_model(cname, seed=1234, device=dev)
            hw_ = c_["dataset_params"]["frame_shape"]
            tot = c_["dataset_params"]["valid_params"]["pred_frames"]
            clip = make_clip(cname, b, m_.cond_frame_num, hw_, 1000 + rank).to(dev)
            # warm up until the SM clock has ramped: building a model leaves the GPU idle for seconds, and the first
            # ~0.5 s of work after that runs below the boost clock (measured: SMMNIST 170 vs 149.5 ms per rollout)
            t_warm, n_warm = time.perf_counter(), 0
            while n_warm < 2 or time.perf_counter() - t_warm < 1.0:
                configs.rollout(m_, clip, tot)
                torch.cuda.synchronize()
                n_warm += 1
            ms = time_rollouts(lambda i: configs.rollout(m_, clip, tot), 2)
            per[label or cname] = {"workload": f"{DESCR[cname]}, batch {b} per GPU", "value": world * b * tot / (ms * 1e-3),
                                   "unit": "frames/s", "ms_per_step": ms, "batch_per_gpu": b}
            return m_, c_

        for cname in ("smmnist", "kth", "cityscapes", "cityscapes64"):
            try:
                mdl = measure(cname, B)
                if cname == "smmnist":                       # BASELINE config 1's shape on the GPU: batch 1 (latency)
                    measure(cname, 1, "smmnist_b1", mdl)
                del mdl
            except Exception as e:                           # reported-only extras never fail the bench
                per[cname] = {"error": repr(e)}
            torch.cuda.empty_cache()
        try:                                                 # the headline configuration at larger per-GPU batches
            mdl = configs.build_model(name, seed=1234, device=dev)
            for b in (64, 128):
                measure(name, b, f"{name}_b{b}", mdl)
                mdl[0].unet._runners.clear()
                mdl[0].generator._runners.clear()
                mdl[0]._cond_runners.clear()
                torch.cuda.empty_cache()
            del mdl
        except Exception as e:
            per[f"{name}_batch_sweep"] = {"error": repr(e)}
        torch.cuda.empty_cache()
        try:                                                 # BASELINE config 5: UCF-101 large-batch sweep
            mdl = configs.build_model("ucf", seed=1234, device=dev)
            for b in (8, 16, 32, 64, 128):
                measure("ucf", b, f"ucf_b{b}", mdl)
                mdl[0].unet._runners.clear()
                mdl[0].generator._runners.clear()
                mdl[0]._cond_runners.clear()
                torch.cuda.empty_cache()
            del mdl
        except Exception as e:
            per["ucf"] = {"error": repr(e)}
        torch.cuda.empty_cache()
        line["per_config"] = per
        model = None

    if rank == 0 and world == 1:
        from oracle import ref_shims
        if not args.no_gpu_reference and ref_shims.available():
            try:
                if model is None:
                    model, _ = configs.build_model(name, seed=1234, device=dev)
                line["gpu_eager_reference"] = gpu_eager_reference(model, name, B, total_pred, dev)
                line["gpu_eager_reference"]["speedup_device_timed"] = \
                    line["value"] / line["gpu_eager_reference"]["tf32_default"]["value"]
            except Exception as e:
                line["gpu_eager_reference"] = {"error": repr(e)}
        if not args.no_cpu_baseline:
            try:
                line["cpu_baseline"] = cpu_reference(name)[0] if ref_shims.available() else cpu_port_fallback()[0]
            except Exception as e:                           # the baseline is reported-only: never fail the bench on it
                line["cpu_baseline"] = {"value": None, "unit": "frames/s", "cores": os.cpu_count(), "kind": "reference",
                                        "sample": f"failed: {e!r}"}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
