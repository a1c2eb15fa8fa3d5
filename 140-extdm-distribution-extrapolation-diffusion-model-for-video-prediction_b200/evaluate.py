"""The caller side of the hot path (SURVEY.md section 8f-2 / 8f-4): the evaluation loop of scripts/DM/valid.py:150-197
(repeat-n sampling + autoregressive rollout), its checkpoint / result wire formats (:111-112, :281-286) and the PSNR /
SSIM of metrics/calculate_psnr.py:6-15 and metrics/calculate_ssim.py:6-42 as batched torch ops that run on the GPU.

    model = extdm_b200.flow_diffusion_class(dm_arch)(config=cfg, pretrained_pth=ae_ckpt, is_train=False, ...)
    evaluate.load_dm_checkpoint(model, dm_ckpt)
    origin, result = evaluate.sample_videos(model, real_vids, total_pred, num_sample_video=n)
    evaluate.save_results(log_dir, origin, result)
    evaluate.psnr_videos(origin[:, 0], result[:, 0]);  evaluate.ssim_videos(...)
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
def sample_videos(model, real_vids, total_pred, num_sample_video=1, on_device=True, seed=None, video_offset=0):
    """valid.py:156-197 for one batch: real_vids (B, C, T, H, W) in [0,1] with T >= cond frames (+ total_pred ground
    truth frames if available) -> (origin, result), both (B, n, T', C, H, W) on the CPU, result = cond frames followed
    by total_pred predicted frames.  on_device=False reproduces the reference's per-round .cpu()/.cuda() hops.

    seed: optional int.  Then repeat k of video b is sampled with the per-video base seed
    sharding.video_seeds(seed, (video_offset + b) * num_sample_video + k), a function of its *global* index only:
    a sharded evaluation passes video_offset = lo of sharding.shard_range and samples every video with the same noise
    as a single-GPU run.  Default: the sampler's own noise (torch's default generator)."""
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
    if on_device:
        pred = rollout(model, cond, total_pred, seeds=seeds)
    else:
        pin_in = torch.empty(cond.shape).pin_memory()
        pin_out = torch.empty(cond.shape[0], cond.shape[1], tc + model.pred_frame_num, *cond.shape[3:]).pin_memory()
        pred = rollout(model, cond.cpu(), total_pred, host_buffers=(pin_in, pin_out), seeds=seeds)
    res = torch.cat([rep[:, :, :tc].cpu().float(), pred.cpu()], dim=2)

    def shape(t):                                                                   # '(b n) c t h w -> b n t c h w'
        return t.reshape(B, num_sample_video, *t.shape[1:]).permute(0, 1, 3, 2, 4, 5).contiguous()
    return shape(rep.cpu().float()), shape(res)


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
