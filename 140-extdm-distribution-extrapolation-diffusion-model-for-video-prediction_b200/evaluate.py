"""The caller side of the hot path (SURVEY.md section 8f-2 / 8f-4): the evaluation loop of scripts/DM/valid.py:150-197
(repeat-n sampling + autoregressive rollout), its checkpoint / result wire formats (:111-112, :281-286) and the PSNR /
SSIM of metrics/calculate_psnr.py:6-15 and metrics/calculate_ssim.py:6-42 as batched torch ops that run on the GPU.

    model = extdm_b200.flow_diffusion_class(dm_arch)(config=cfg, pretrained_pth=ae_ckpt, is_train=False, ...)
    evaluate.load_dm_checkpoint(model, dm_ckpt)
    origin, result = evaluate.sample_videos(model, real_vids, total_pred, num_sample_video=n)
    evaluate.save_results(log_dir, origin, result)
    evaluate.psnr_videos(origin[:, 0], result[:, 0]);  evaluate.ssim_videos(...)

Stage 1 (LFAE reconstruction, the upper bound of every DM prediction) uses the same layout and metrics:

    ae = extdm_b200.FlowAE(cfg, pretrained_pth=ae_ckpt)        # or FlowAE.from_flow_diffusion(model)
    origin, result = evaluate.reconstruct_videos(ae, real_vids)

The diffusion model's own training objective on held-out clips of tc + tp frames (checkpoint selection, loss against
timestep):

    out = evaluate.denoising_loss_videos(model, real_vids, timesteps=[100, 500, 900], seed=0)

Interpolation between two futures of the same past (e.g. the encoded ground truth and a sample), decoded to RGB:

    x1 = model.encode_future(real_vids);  x2 = model.diffusion.sample(...)    # (B, 3, tp, h, w) latents
    origin, result = evaluate.interpolate_videos(model, real_vids, x1, x2, lams=[0.0, 0.25, 0.5, 0.75, 1.0], seed=0)

Goal-conditioned prediction: the last predicted frame (e.g. the goal of a BAIR push) is known, taken from the ground
truth, and imposed in its rollout round:

    origin, result = evaluate.sample_videos(model, real_vids, total_pred, keyframes=[total_pred - 1], seed=0)
"""
import os

import torch
import torch.nn.functional as F


def load_dm_checkpoint(model, ckpt):
    """`model.diffusion.load_state_dict(ckpt['diffusion'])` (scripts/DM/valid.py:111-112).  `ckpt` is a path or the
    loaded dict {'example', 'epoch', 'diffusion', 'optimizer'} (scripts/DM/train.py:404-412).  Keys under
    `*.rotary_emb.*` are derivable constants whose exact set depends on the rotary-embedding-torch version that wrote
    the checkpoint (SURVEY.md App. E11): unknown ones are dropped, missing ones keep their constructed values."""
    if isinstance(ckpt, (str, os.PathLike)):
        ckpt = torch.load(ckpt, map_location="cpu")
    sd = ckpt["diffusion"] if "diffusion" in ckpt else ckpt
    own = model.diffusion.state_dict()
    filtered = {k: v for k, v in sd.items() if k in own or ".rotary_emb." not in k}
    missing = [k for k in own if k not in filtered and ".rotary_emb." not in k]
    unexpected = [k for k in filtered if k not in own]
    if missing or unexpected:
        raise RuntimeError(f"diffusion checkpoint mismatch: missing {missing[:5]} unexpected {unexpected[:5]}")
    model.diffusion.load_state_dict(filtered, strict=False)
    return {k: ckpt[k] for k in ("example", "epoch") if k in ckpt}


@torch.no_grad()
def sample_videos(model, real_vids, total_pred, num_sample_video=1, on_device=True, seed=None, video_offset=0,
                  keyframes=None):
    """valid.py:156-197 for one batch: real_vids (B, C, T, H, W) in [0,1] with T >= cond frames (+ total_pred ground
    truth frames if available) -> (origin, result), both (B, n, T', C, H, W) on the CPU, result = cond frames followed
    by total_pred predicted frames.  on_device=False reproduces the reference's per-round .cpu()/.cuda() hops.

    seed: optional int.  Then repeat k of video b is sampled with the per-video base seed
    sharding.video_seeds(seed, (video_offset + b) * num_sample_video + k), a function of its *global* index only:
    a sharded evaluation passes video_offset = lo of sharding.shard_range and samples every video with the same noise
    as a single-GPU run.  Default: the sampler's own noise (torch's default generator).

    keyframes: optional list of predicted-frame indices in [0, total_pred), known for every video, or a (B, total_pred)
    bool mask.  Those frames are taken from the ground truth real_vids[:, :, tc + j] (so T >= tc + total_pred) and
    imposed in their rollout round (configs.rollout); the decoded known frames are their LFAE reconstructions."""
    from .configs import rollout
    from .sharding import video_seeds
    tc = model.cond_frame_num
    dev = next(model.parameters()).device
    B = real_vids.shape[0]
    rep = real_vids.repeat_interleave(num_sample_video, dim=0)                     # 'b c t h w -> (b n) c t h w'
    cond = rep[:, :, :tc].to(dev).float().contiguous()
    seeds = None
    if seed is not None:                                                            # row b*n + k of rep = (b, k)
        seeds = video_seeds(seed, torch.arange(B * num_sample_video) + video_offset * num_sample_video)
    kf = None
    if keyframes is not None:
        if real_vids.shape[2] < tc + total_pred:
            raise ValueError(f"sample_videos: keyframes need {tc + total_pred} ground-truth frames, got "
                             f"{real_vids.shape[2]}")
        if torch.is_tensor(keyframes):
            if keyframes.dtype != torch.bool or tuple(keyframes.shape) != (B, total_pred):
                raise ValueError(f"sample_videos: a keyframe mask must be a ({B}, {total_pred}) bool tensor")
            mask = keyframes.cpu()
        else:
            idx = list(keyframes)
            if any(isinstance(j, bool) or not isinstance(j, int) or not 0 <= j < total_pred for j in idx):
                raise ValueError(f"sample_videos: keyframes must be ints in [0, {total_pred}), got {keyframes!r}")
            mask = torch.zeros(B, total_pred, dtype=torch.bool)
            mask[:, idx] = True
        kf = (rep[:, :, tc:tc + total_pred].to(dev).float(), mask.repeat_interleave(num_sample_video, dim=0))
    if on_device:
        pred = rollout(model, cond, total_pred, seeds=seeds, keyframes=kf)
    else:
        pin_in = torch.empty(cond.shape).pin_memory()
        pin_out = torch.empty(cond.shape[0], cond.shape[1], tc + model.pred_frame_num, *cond.shape[3:]).pin_memory()
        pred = rollout(model, cond.cpu(), total_pred, host_buffers=(pin_in, pin_out), seeds=seeds, keyframes=kf)
    res = torch.cat([rep[:, :, :tc].cpu().float(), pred.cpu()], dim=2)

    def shape(t):                                                                   # '(b n) c t h w -> b n t c h w'
        return t.reshape(B, num_sample_video, *t.shape[1:]).permute(0, 1, 3, 2, 4, 5).contiguous()
    return shape(rep.cpu().float()), shape(res)


@torch.no_grad()
def reconstruct_videos(ae, real_vids, source_frame=0):
    """Stage-1 counterpart of sample_videos: real_vids (B, C, T, H, W) in [0,1] -> (origin, result), both (B, 1, T, C,
    H, W) on the CPU, result = FlowAE.reconstruct(real_vids, source_frame)['prediction'], every frame reconstructed
    from frame `source_frame` of its video.  psnr_videos / ssim_videos / summarize / save_results apply unchanged."""
    dev = ae.generator.final.weight.device
    pred = ae.reconstruct(real_vids.to(dev).float(), source_frame)["prediction"]

    def shape(t):                                                                   # 'b c t h w -> b 1 t c h w'
        return t.cpu().float().permute(0, 2, 1, 3, 4).unsqueeze(1).contiguous()
    return shape(real_vids), shape(pred)


@torch.no_grad()
def denoising_loss_videos(model, real_vids, timesteps=None, seed=None, video_offset=0):
    """FlowDiffusion.denoising_loss over real_vids (B, C, tc + tp, H, W) in [0, 1] (any device) -> dict of CPU tensors
    {'loss', 'loss_per_frame', 'timesteps'}.

    timesteps: None (drawn), an int (every video at that timestep), a (B,) int64 tensor, or a list of K ints: a loss
    curve, one graph replay per timestep on the same conditioning, and then 'loss' is (B, K), 'loss_per_frame'
    (B, K, tp) and 'timesteps' (B, K); otherwise (B,), (B, tp) and (B,).

    seed: optional int.  Then video b, whose *global* index is g = video_offset + b, draws its epsilon with the seed
    sharding.video_seeds(seed, g, 0), and, when timesteps is None, is evaluated at the timestep
    sharding.video_seeds(seed, g, 1) % num_timesteps.  Both depend on (seed, g) only, so a sharded evaluation that
    passes video_offset = lo of sharding.shard_range evaluates every video exactly as a single-GPU run does.  Within a
    loss curve the epsilon still differs per timestep (the Philox counter holds t).  Without seed, the timesteps and
    the seeds come from torch's default generator (GaussianDiffusion.denoising_loss)."""
    from .sharding import video_seeds
    B = real_vids.shape[0]
    n_t = model.diffusion.num_timesteps
    ids = torch.arange(B) + video_offset
    seeds = video_seeds(seed, ids, 0) if seed is not None else None
    curve = isinstance(timesteps, (list, tuple))
    if timesteps is None:
        ts = [video_seeds(seed, ids, 1) % n_t if seed is not None else None]
    elif curve or not torch.is_tensor(timesteps):
        ks = list(timesteps) if curve else [timesteps]
        if not ks or any(isinstance(k, bool) or not isinstance(k, int) or not 0 <= k < n_t for k in ks):
            raise ValueError(f"denoising_loss_videos: timesteps must be ints in [0, {n_t}), got {timesteps!r}")
        ts = [torch.full((B,), k, dtype=torch.long) for k in ks]
    else:
        ts = [timesteps]
    dev = next(model.parameters()).device
    inputs = model.loss_inputs(real_vids.to(dev).float())
    outs = [model.diffusion.denoising_loss(*inputs, timesteps=t, seeds=seeds) for t in ts]
    if not curve:
        return {k: v.cpu() for k, v in outs[0].items()}
    return {k: torch.stack([o[k] for o in outs], dim=1).cpu() for k in outs[0]}


@torch.no_grad()
def interpolate_videos(model, real_vids, x1, x2, lams, t=None, seed=None, video_offset=0):
    """FlowDiffusion.interpolate_one_video over real_vids (B, C, >= tc, H, W) in [0, 1] and the futures x1, x2 (B, 3,
    tp, h, w) (any device) -> (origin, result) in the layout of sample_videos, both (B, K, T', C, H, W) on the CPU:
    result[:, k] = the cond frames followed by the tp frames decoded from the interpolation at lams[k] (lams: a list
    of K floats, or one float for K = 1), origin[:, k] = real_vids.  psnr_videos / ssim_videos / summarize /
    save_results apply unchanged.  t: as GaussianDiffusion.interpolate.

    seed: optional int.  Then video b, whose *global* index is g = video_offset + b, is interpolated with the seed
    sharding.video_seeds(seed, g, 2), so a sharded evaluation that passes video_offset = lo of sharding.shard_range
    equals a single-GPU run.  Default: seeds from torch's default generator."""
    from .sharding import video_seeds
    B, tc = real_vids.shape[0], model.cond_frame_num
    lams = list(lams) if isinstance(lams, (list, tuple)) else [lams]
    seeds = video_seeds(seed, torch.arange(B) + video_offset, 2) if seed is not None else None
    dev = next(model.parameters()).device
    out = model.interpolate_one_video(real_vids.to(dev).float(), x1.to(dev), x2.to(dev), t=t, lam=lams, seeds=seeds)
    pred = out["sample_out_vid"][:, :, :, tc:].cpu()                               # (K, B, 3, tp, H, W)
    cond = real_vids[:, :, :tc].cpu().float()
    res = torch.cat([cond.expand(len(lams), *cond.shape), pred], dim=3)
    origin = real_vids.cpu().float().permute(0, 2, 1, 3, 4).unsqueeze(1)          # 'b c t h w -> b 1 t c h w'
    return origin.expand(B, len(lams), *origin.shape[2:]).contiguous(), res.permute(1, 0, 3, 2, 4, 5).contiguous()


def save_results(log_dir, origin_videos, result_videos, best_videos=None):
    """The .pt dumps of valid.py:281-286: origin.pt = origin[:, 0], result_{k}.pt = result[:, k] (b t c h w)."""
    os.makedirs(log_dir, exist_ok=True)
    torch.save(origin_videos[:, 0].clone(), os.path.join(log_dir, "origin.pt"))
    if best_videos is not None:
        torch.save(best_videos.clone(), os.path.join(log_dir, "result_best.pt"))
    for k in range(result_videos.shape[1]):
        torch.save(result_videos[:, k].clone(), os.path.join(log_dir, f"result_{k}.pt"))


def psnr_videos(videos1, videos2):
    """img_psnr per frame (calculate_psnr.py:6-15): videos (B, T, C, H, W) in [0,1] -> (B, T) tensor; mse < 1e-10 -> 100."""
    assert videos1.shape == videos2.shape
    mse = ((videos1.double() - videos2.double()) ** 2).mean(dim=(2, 3, 4))
    val = 20.0 * torch.log10(1.0 / torch.sqrt(mse.clamp_min(1e-300)))
    return torch.where(mse < 1e-10, torch.full_like(val, 100.0), val)


def _gaussian_window(device):
    # cv2.getGaussianKernel(11, 1.5): exp(-(i-5)^2 / (2 sigma^2)) normalised to sum 1
    x = torch.arange(11, dtype=torch.float64, device=device) - 5.0
    g = torch.exp(-(x * x) / (2.0 * 1.5 * 1.5))
    g = g / g.sum()
    return torch.outer(g, g)


def ssim_videos(videos1, videos2):
    """calculate_ssim_function per frame (calculate_ssim.py:6-42): 11x11 Gaussian (sigma 1.5) window, 'valid' region,
    float64, mean over channels -> (B, T) tensor."""
    assert videos1.shape == videos2.shape
    B, T, C, H, W = videos1.shape
    a = videos1.double().reshape(B * T * C, 1, H, W)
    b = videos2.double().reshape(B * T * C, 1, H, W)
    win = _gaussian_window(a.device)[None, None]
    C1, C2 = 0.01 ** 2, 0.03 ** 2
    mu1, mu2 = F.conv2d(a, win), F.conv2d(b, win)
    s11 = F.conv2d(a * a, win) - mu1 * mu1
    s22 = F.conv2d(b * b, win) - mu2 * mu2
    s12 = F.conv2d(a * b, win) - mu1 * mu2
    m = ((2 * mu1 * mu2 + C1) * (2 * s12 + C2)) / ((mu1 * mu1 + mu2 * mu2 + C1) * (s11 + s22 + C2))
    return m.mean(dim=(1, 2, 3)).reshape(B, T, C).mean(dim=2)


def summarize(per_frame):
    """{'avg[t]': mean over videos, 'std[t]': population std} like calculate_psnr / calculate_ssim, plus the overall mean."""
    out = {f"avg[{t}]": per_frame[:, t].mean().item() for t in range(per_frame.shape[1])}
    out.update({f"std[{t}]": per_frame[:, t].std(unbiased=False).item() for t in range(per_frame.shape[1])})
    out["mean"] = per_frame.mean().item()
    return out
