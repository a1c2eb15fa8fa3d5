"""The reference's dataset configurations (config/DM/{kth,smmnist,bair,ucf,cityscapes}.yaml) reduced to the
fields `FlowDiffusion` reads, so benchmarks and tests do not need /root/reference at run time.  A user's
own `yaml.safe_load(...)` dict is accepted unchanged by `FlowDiffusion`."""
import copy


def _config(frame_shape, tc, tp, total_pred, num_regions=10, scale_factor=0.5, bg_type="affine", split="test"):
    return {
        "dataset_params": {
            "frame_shape": frame_shape,
            "train_params": {"type": "train", "cond_frames": tc, "pred_frames": tp},
            "valid_params": {"total_videos": 256, "type": split, "cond_frames": tc, "pred_frames": total_pred},
        },
        "flow_params": {"model_params": {
            "num_regions": num_regions, "num_channels": 3, "estimate_affine": True, "revert_axis_swap": True,
            "bg_predictor_params": {"block_expansion": 32, "max_features": 1024, "num_blocks": 5, "bg_type": bg_type},
            "region_predictor_params": {"temperature": 0.1, "block_expansion": 32, "max_features": 1024,
                                        "scale_factor": scale_factor, "num_blocks": 5, "pca_based": True, "pad": 0,
                                        "fast_svd": False},
            "generator_params": {
                "block_expansion": 64, "max_features": 512, "num_down_blocks": 2, "num_bottleneck_blocks": 6,
                "skips": True,
                "pixelwise_flow_predictor_params": {"block_expansion": 64, "max_features": 1024, "num_blocks": 5,
                                                    "scale_factor": scale_factor, "use_deformed_source": True,
                                                    "use_covar_heatmap": True, "estimate_occlusion_map": True}},
        }},
        "diffusion_params": {"model_params": {"null_cond_prob": 0.0, "use_residual_flow": False,
                                              "only_use_flow": False, "sampling_timesteps": 10, "loss_type": "l2",
                                              "ada_layers": "auto"}},
    }


# name -> (config, DM wrapper, Unet3D architecture)   -- SURVEY.md App. A
_DATASETS = {
    "kth": (_config(64, 10, 20, 40, split="valid"), "VideoFlowDiffusion_multi_w_ref",
            "DenoiseNet_STWAtt_w_w_ref_adaptor_cross_multi_traj_ada"),
    "smmnist": (_config(64, 10, 5, 10), "VideoFlowDiffusion_multi1248",
                "DenoiseNet_STWAtt_w_wo_ref_adaptor_cross_multi"),
    "bair": (_config(64, 2, 10, 28), "VideoFlowDiffusion_multi_w_ref",
             "DenoiseNet_STWAtt_w_w_ref_adaptor_cross_multi_traj_u12"),
    # ucf.yaml's valid_params say 16 predicted frames; BASELINE.json names the 4 -> 12 rollout (2 rounds either way)
    "ucf": (_config(64, 4, 8, 12, num_regions=64), "VideoFlowDiffusion_multi_w_ref",
            "DenoiseNet_STWAtt_w_w_ref_adaptor_cross_multi_traj_ada"),
    "cityscapes": (_config(128, 2, 5, 28, num_regions=20, scale_factor=0.25, bg_type="perspective"),
                   "VideoFlowDiffusion_multi_w_ref", "DenoiseNet_STWAtt_w_w_ref_adaptor_cross_multi_traj_ada"),
    # BASELINE.json words Cityscapes as 64x64: the shipped scale_factor 0.25 cannot run at 64 (the 5-block hourglass
    # would reach 16 -> 0, SURVEY.md section 8d config 4), so the 64x64 variant uses scale_factor 0.5 like BAIR
    "cityscapes64": (_config(64, 2, 5, 28, num_regions=20, scale_factor=0.5, bg_type="perspective"),
                     "VideoFlowDiffusion_multi_w_ref", "DenoiseNet_STWAtt_w_w_ref_adaptor_cross_multi_traj_ada"),
    # the pairing the reference's valid_DM_cityscapes.sh:8-9 names
    "cityscapes_u22": (_config(128, 2, 5, 28, num_regions=20, scale_factor=0.25, bg_type="perspective"),
                       "VideoFlowDiffusion_multi_w_ref_u22",
                       "DenoiseNet_STWAtt_w_w_ref_adaptor_cross_multi_traj_ada_u22"),
}


def dataset(name):
    cfg, wrapper, unet = _DATASETS[name]
    return copy.deepcopy(cfg), wrapper, unet


def build_model(name, seed=1234, device="cuda"):
    """FlowDiffusion for a named dataset with deterministic synthetic weights (no checkpoints offline)."""
    from .flow_diffusion import flow_diffusion_class
    from .weights import synth_state_dict
    cfg, wrapper, unet = dataset(name)
    model = flow_diffusion_class(wrapper)(config=cfg, pretrained_pth="", is_train=False,
                                          Unet3D_architecture=unet).eval()
    for i, part in enumerate(("generator", "region_predictor", "bg_predictor", "diffusion")):
        m = getattr(model, part)
        base = m.state_dict()
        m.load_state_dict(synth_state_dict({k: tuple(v.shape) for k, v in base.items()}, seed + i, base=base))
    return model.to(device), cfg


def rollout(model, clip, total_pred, host_buffers=None, noise_fn=None, seeds=None, keyframes=None):
    """Autoregressive rollout of scripts/DM/valid.py:167-172 -> (B, 3, total_pred, H, W).
    host_buffers=None keeps every round on the device (SURVEY.md section 8f-2).  With
    host_buffers=(pinned_in, pinned_out) each round copies its conditioning clip host->device and its
    sample_out_vid device->host exactly like the reference driver (`.cuda()` / `.cpu()` per round).
    seeds: optional per-video base seeds ((B,) int64 tensor or list); round r samples video b with the seed
    sharding.video_seeds(seeds[b], 0, r), so every round draws fresh noise and a video's rollout depends on its own
    base seed only.
    keyframes: optional (frames (B, 3, total_pred, H, W) in [0, 1], mask (B, total_pred) bool): predicted frame j of
    video b is known to be frames[b, :, j] where mask[b, j].  Round r imposes the known frames of its window
    [r*tp, (r+1)*tp) with FlowDiffusion.sample_with_keyframes, encoded against that round's source frame (a predicted
    frame after round 0); a round without a known frame calls sample_one_video as without keyframes.  Keyframes take
    seeds or the default noise, not noise_fn."""
    import math
    import torch
    from .sharding import video_seeds
    if seeds is not None and noise_fn is not None:
        raise ValueError("rollout: pass noise_fn or seeds, not both")
    if seeds is not None and len(seeds) != clip.shape[0]:
        raise ValueError(f"rollout: {len(seeds)} seeds for {clip.shape[0]} videos")
    tc, tp = model.cond_frame_num, model.pred_frame_num
    n_rounds = math.ceil(total_pred / tp)
    if keyframes is not None:
        if noise_fn is not None:
            raise ValueError("rollout: keyframes take seeds or the default noise, not noise_fn")
        kf_frames, kf_mask = keyframes
        B, _, _, H, W = clip.shape
        if not torch.is_tensor(kf_frames) or tuple(kf_frames.shape) != (B, 3, total_pred, H, W):
            raise ValueError(f"rollout: keyframe frames must be a ({B}, 3, {total_pred}, {H}, {W}) tensor")
        if not torch.is_tensor(kf_mask) or kf_mask.dtype != torch.bool or tuple(kf_mask.shape) != (B, total_pred):
            raise ValueError(f"rollout: the keyframe mask must be a ({B}, {total_pred}) bool tensor")
        pad = n_rounds * tp - total_pred                         # the last round's window may reach past total_pred
        kf_mask = torch.cat([kf_mask.cpu(), torch.zeros(B, pad, dtype=torch.bool)], dim=1)
        kf_frames = torch.cat([kf_frames, kf_frames.new_zeros(B, 3, pad, H, W)], dim=2)
    preds = []
    cond = clip
    for r in range(n_rounds):
        if host_buffers is not None:
            pin_in, pin_out = host_buffers
            pin_in.copy_(cond)                                   # host -> pinned staging (host memcpy)
            dev_in = pin_in.to("cuda", non_blocking=True)
        else:
            dev_in = cond
        round_seeds = None if seeds is None else video_seeds(seeds, 0, r)
        window = slice(r * tp, (r + 1) * tp)
        if keyframes is not None and bool(kf_mask[:, window].any()):
            real_vid = torch.cat([dev_in, kf_frames[:, :, window].to(dev_in.device, dev_in.dtype)], dim=2)
            out = model.sample_with_keyframes(real_vid, kf_mask[:, window].contiguous(),
                                              seeds=round_seeds)["sample_out_vid"]
        else:
            out = model.sample_one_video(cond_scale=1.0, real_vid=dev_in,
                                         noise=None if noise_fn is None else noise_fn(),
                                         seeds=round_seeds)["sample_out_vid"]
        if host_buffers is not None:
            pin_out.copy_(out, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            out = pin_out.clone()
        preds.append(out[:, :, -tp:])
        cond = out[:, :, -tc:].contiguous()
    return torch.cat(preds, dim=2)[:, :, :total_pred]
