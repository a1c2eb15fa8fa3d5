"""FlowDiffusion: the reference's pipeline wrapper (model/BaseDM_adaptor/VideoFlowDiffusion_multi_w_ref.py,
VideoFlowDiffusion_multi1248.py, VideoFlowDiffusion_multi.py) with the same constructor, attributes and
`sample_one_video(cond_scale, real_vid) -> dict`.

  (A) conditioning  : torch (RegionPredictor / BGMotionPredictor / Generator.forward), batched over the tc frames
  (B) denoise       : GaussianDiffusion.sample  -> CUDA-graphed UNet3D + DDIM kernels
                      (interpolate_one_video: GaussianDiffusion.interpolate between two given futures)
                      (sample_with_keyframes: GaussianDiffusion.sample_with_known, some future frames given)
  (C) decode        : Generator.decode_video    -> CUDA warp / blend / conv kernels
"""
import torch
import torch.nn.functional as F
from torch import nn

from .diffusion import GaussianDiffusion
from .lfae import BGMotionPredictor, CondRunner, Generator, RegionPredictor
from .unet import Unet3D

_DEFAULT_UNET = {
    "w_ref": "DenoiseNet_STWAtt_w_w_ref_adaptor_cross_multi_traj_ada",
    "multi1248": "DenoiseNet_STWAtt_w_wo_ref_adaptor_cross_multi",
    "multi": "DenoiseNet_STWAtt_w_wo_ref_adaptor_cross_multi",
}


class FlowDiffusion(nn.Module):
    WRAPPER = "w_ref"            # "w_ref" | "multi1248" | "multi"
    native_conditioning = True   # class-level switch: False runs the conditioning stage as torch modules (tests A/B)

    def __init__(self, config="", pretrained_pth="", is_train=True, ddim_sampling_eta=1.0, timesteps=1000,
                 dim_mults=None, learn_null_cond=False, use_deconv=True, padding_mode="zeros", withFea=True,
                 Unet3D_architecture=None):
        super().__init__()
        kind = self.WRAPPER
        if dim_mults is None:
            dim_mults = (1, 2, 4, 8) if kind == "multi1248" else (1, 2, 4, 4)
        if Unet3D_architecture is None or kind == "multi1248":      # multi1248 imports the base UNet unconditionally
            Unet3D_architecture = _DEFAULT_UNET[kind]
        flow_params = config["flow_params"]["model_params"]
        diffusion_params = config["diffusion_params"]["model_params"]
        dataset_params = config["dataset_params"]
        self.estimate_occlusion_map = \
            flow_params["generator_params"]["pixelwise_flow_predictor_params"]["estimate_occlusion_map"]
        self.use_residual_flow = diffusion_params["use_residual_flow"]
        self.only_use_flow = diffusion_params["only_use_flow"]
        self.withFea = withFea
        dev = "cuda" if torch.cuda.is_available() else "cpu"
        ckpt = torch.load(pretrained_pth, map_location=dev) if pretrained_pth != "" else None

        self.generator = Generator(num_regions=flow_params["num_regions"], num_channels=flow_params["num_channels"],
                                   revert_axis_swap=flow_params["revert_axis_swap"],
                                   **flow_params["generator_params"]).to(dev)
        self.region_predictor = RegionPredictor(num_regions=flow_params["num_regions"],
                                                num_channels=flow_params["num_channels"],
                                                estimate_affine=flow_params["estimate_affine"],
                                                **flow_params["region_predictor_params"]).to(dev)
        self.bg_predictor = BGMotionPredictor(num_channels=flow_params["num_channels"],
                                              **flow_params["bg_predictor_params"]).to(dev)
        if ckpt is not None:
            # VideoFlowDiffusion_multi_w_ref.py:51 (and _u22) load the generator with strict=False; multi1248 / multi
            # (VideoFlowDiffusion_multi1248.py:50) load it strictly
            self.generator.load_state_dict(ckpt["generator"], strict=kind != "w_ref")
            self.region_predictor.load_state_dict(ckpt["region_predictor"])
            self.bg_predictor.load_state_dict(ckpt["bg_predictor"])
        for m in (self.generator, self.region_predictor, self.bg_predictor):
            m.eval()
            for p in m.parameters():
                p.requires_grad = False

        tc = dataset_params["train_params"]["cond_frames"]
        tp = dataset_params["train_params"]["pred_frames"]
        from .manifest import UNET_ARCHITECTURES
        if Unet3D_architecture not in UNET_ARCHITECTURES:
            # the reference silently constructs NotImplementedError() and then dies with a NameError
            # (VideoFlowDiffusion_multi_w_ref.py:71-80); fail with a message instead
            raise NotImplementedError(f"unknown Unet3D architecture {Unet3D_architecture!r}")
        # base and ada_u22 feed the 3-channel flow volume to init_conv directly (VideoFlowDiffusion_multi1248.py:72,
        # VideoFlowDiffusion_multi_w_ref_u22.py:199-201); the others go through init_noise_conv (3 -> 256) first
        base = UNET_ARCHITECTURES[Unet3D_architecture] in ("base", "u22")
        self.unet = Unet3D(dim=64, channels=3 + 256 if base else 256 + 256, out_grid_dim=2, out_conf_dim=1,
                           dim_mults=dim_mults, use_bert_text_cond=False, learn_null_cond=learn_null_cond,
                           use_final_activation=False, use_deconv=use_deconv, padding_mode=padding_mode,
                           cond_num=tc, pred_num=tp, architecture=Unet3D_architecture).to(dev)
        self.diffusion = GaussianDiffusion(
            self.unet, image_size=dataset_params["frame_shape"] // 2, num_frames=tc + tp,
            sampling_timesteps=diffusion_params["sampling_timesteps"], timesteps=timesteps,
            loss_type=diffusion_params["loss_type"], use_dynamic_thres=True,
            null_cond_prob=diffusion_params["null_cond_prob"], ddim_sampling_eta=ddim_sampling_eta,
            solver=diffusion_params.get("solver")).to(dev)
        self.cond_frame_num, self.pred_frame_num, self.frame_num = tc, tp, tc + tp
        self._cond_runners = {}
        for m in (self.generator, self.region_predictor, self.bg_predictor):
            m.register_load_state_dict_post_hook(lambda mod, k: self._cond_runners.clear())
        self.is_train = is_train
        if is_train:
            raise NotImplementedError("training (FlowDiffusion.forward / p_losses) is outside the sampling hot path")

    # ------------------------------------------------------------------ (A) conditioning, torch
    @torch.no_grad()
    def condition(self, real_vid, with_decode=False):
        """real_vid (B,3,tc,H,W) in [0,1] -> dict with x_cond, cond_fea and the 'real_*' entries of the reference
        result dict (VideoFlowDiffusion_multi_w_ref.py:231-278 / VideoFlowDiffusion_multi1248.py:221-264).
        The tc per-frame passes of the reference are batched into one pass over B*tc images."""
        B, _, tc, H, W = real_vid.shape
        assert tc == self.cond_frame_num
        tp = self.pred_frame_num
        ref = real_vid[:, :, tc - 1]
        frames = real_vid.permute(0, 2, 1, 3, 4).reshape(B * tc, 3, H, W).contiguous(memory_format=torch.channels_last)
        pfp = self.generator.pixelwise_flow_predictor
        if real_vid.is_cuda and self.native_conditioning and not with_decode and \
                CondRunner.supported(self.region_predictor, self.bg_predictor, pfp):
            # (A) on the CUDA kernels: tf32 tcgen05 convolutions + fp32 element-wise kernels (lfae.CondRunner)
            key = (real_vid.device, B, tc, H, W)
            if key not in self._cond_runners:
                self._cond_runners[key] = CondRunner(self.region_predictor, self.bg_predictor, pfp, real_vid.device,
                                                     B, tc, H, W)
            grid, conf = self._cond_runners[key].run(real_vid.float())
            ret = {"real_vid_grid": grid.clone()}
            if self.estimate_occlusion_map:
                ret["real_vid_conf"] = conf.clone()
            elif self.WRAPPER != "w_ref":
                raise KeyError("occlusion_map")
        else:
            ret = self._condition_torch(real_vid, ref, frames, with_decode)
        fea = self._cond_fea(frames, B, ret["real_vid_grid"].shape[-2:])
        x_cond = flow_to_x_start(ret["real_vid_grid"], ret.get("real_vid_conf"), False)
        return ret, x_cond, fea, ref

    def _cond_fea(self, frames, B, flow_hw):
        """cond_fea of condition() from its (B*tc, 3, H, W) frames: the bottleneck features of frames 0..tc-2, then the
        reference frame's repeated."""
        tc, tp = self.cond_frame_num, self.pred_frame_num
        H, W = frames.shape[-2:]
        enc_frames = self.generator.forward_bottle(frames).reshape(B, tc, 256, H // 4, W // 4)
        ref_fea = enc_frames[:, tc - 1]
        n_rep = (1 + tp) if self.WRAPPER == "w_ref" else tp
        fea = torch.cat([enc_frames[:, :tc - 1], ref_fea[:, None].expand(B, n_rep, *ref_fea.shape[1:])], dim=1)
        fea = fea.transpose(1, 2).contiguous()                                       # (B, 256, T', h, w)
        if self.WRAPPER != "w_ref" and not fea.is_cuda:
            # VideoFlowDiffusion_multi1248.py:243-245 resizes cond_fea to the flow resolution before the UNet.  On the
            # CUDA path the UNet prologue does that resize itself (extdm_bilinear_resize_cl, align_corners=False like
            # F.interpolate), so the features stay at H/4 here; this branch serves the CPU parity fixtures only.
            n, c, t, h, w = fea.shape
            fea = F.interpolate(fea.transpose(1, 2).reshape(n * t, c, h, w), size=flow_hw, mode="bilinear")
            fea = fea.reshape(n, t, c, *flow_hw).transpose(1, 2).contiguous()
        return fea

    def _condition_torch(self, real_vid, ref, frames, with_decode):
        """The same stage as ordinary torch modules (cuDNN on a GPU): CPU parity fixtures, unsupported predictor
        hyper-parameters, and the A/B partner of the native path in the tests."""
        B, _, tc, H, W = real_vid.shape
        ref_rep = ref.repeat_interleave(tc, dim=0)
        src_params = self.region_predictor(ref)
        src_rep = {k: v.repeat_interleave(tc, dim=0) for k, v in src_params.items()}
        drv_params = self.region_predictor(frames)
        bg = self.bg_predictor(ref_rep, frames)
        # Generator.forward = flow predictor + the same warp/blend decode as forward_with_flow (generator.py:105-144 vs
        # :152-206): only the flow predictor runs here; the decoded conditioning frames ('real_out_vid',
        # 'real_warped_vid') are the first tc frames of the decode in sample_one_video, which the reference
        # computes a second time from identical inputs (VideoFlowDiffusion_multi_w_ref.py:295-306).
        gen = self.generator.pixelwise_flow_predictor(source_image=ref_rep, driving_region_params=drv_params,
                                                      source_region_params=src_rep, bg_params=bg)
        per_frame = lambda t: t.reshape(B, tc, *t.shape[1:]).transpose(1, 2)       # (B*tc, C, ..) -> (B, C, tc, ..)
        ret = {"real_vid_grid": per_frame(gen["optical_flow"].permute(0, 3, 1, 2)).contiguous()}
        if self.estimate_occlusion_map:
            ret["real_vid_conf"] = per_frame(gen["occlusion_map"]).contiguous()
        elif self.WRAPPER != "w_ref":
            raise KeyError("occlusion_map")         # VideoFlowDiffusion_multi1248.py:236 without estimate_occlusion_map
        if with_decode:
            # the reference's own torch decode of the conditioning frames (used by the CPU parity test only)
            full = self.generator(ref_rep, source_region_params=src_rep, driving_region_params=drv_params, bg_params=bg)
            ret["real_out_vid"] = per_frame(full["prediction"]).contiguous()
            ret["real_warped_vid"] = per_frame(full["deformed"]).contiguous()
        return ret

    # ------------------------------------------------------------------ full round
    @torch.no_grad()
    def sample_one_video(self, cond_scale, real_vid, noise=None, seeds=None):
        """seeds: optional (B,) int64 tensor or list, one sampler seed per video (GaussianDiffusion.sample)."""
        ret, x_cond, cond_fea, ref = self.condition(real_vid)
        pred = self.diffusion.sample(x_cond, cond_fea=cond_fea, batch_size=1, cond_scale=cond_scale, noise=noise,
                                     seeds=seeds)
        ret.update(self._decode_sample(ret, ref, pred))
        return ret

    def _decode_sample(self, ret, ref, pred):
        """sample_one_video's post-processing and decode of a sampled x (B, 3, tp, h, w) after condition()'s ret and
        ref: the 'sample_*' entries of the result and the decoded conditioning frames."""
        tc = self.cond_frame_num
        grid, conf = x_start_to_flow(pred, self.use_residual_flow, self.estimate_occlusion_map)
        sample_vid_grid = torch.cat([ret["real_vid_grid"][:, :, :tc], grid], dim=2)
        sample_vid_conf = None
        if self.estimate_occlusion_map:
            sample_vid_conf = torch.cat([ret["real_vid_conf"][:, :, :tc], conf], dim=2)
        out, warped = self.generator.decode_video(ref, sample_vid_grid, sample_vid_conf)
        res = {"sample_vid_grid": sample_vid_grid}
        if sample_vid_conf is not None:
            res["sample_vid_conf"] = sample_vid_conf
        res["sample_out_vid"] = out
        res["sample_warped_vid"] = warped
        res["real_out_vid"] = out[:, :, :tc]
        res["real_warped_vid"] = warped[:, :, :tc]
        return res

    # ------------------------------------------------------------------ interpolation between two futures
    @torch.no_grad()
    def encode_future(self, real_vid):
        """The latent of the tp future frames of real_vid (B, 3, tc + tp, H, W) in [0, 1]: loss_inputs(real_vid)'s
        x_start (B, 3, tp, h, w), in the space of what sample() returns.  Decoding it as sample_one_video decodes a
        sample gives the LFAE reconstruction of those frames from source frame tc - 1."""
        return self.loss_inputs(real_vid)[0]

    @torch.no_grad()
    def interpolate_one_video(self, real_vid, x1, x2, t=None, lam=0.5, seeds=None, noise=None):
        """Condition on the first tc frames of real_vid (B, 3, >= tc, H, W) in [0, 1], interpolate between the futures
        x1 and x2 (B, 3, tp, h, w; e.g. encode_future of a clip, or a sample) with GaussianDiffusion.interpolate (t,
        lam, seeds, noise as there), then post-process and decode as sample_one_video.  Returns sample_one_video's
        dict; when lam is a list of K values its 'sample_*' entries carry a leading K axis (the decoded conditioning
        frames 'real_out_vid' / 'real_warped_vid' do not depend on lam).  Argument errors raise ValueError before
        anything runs."""
        tc = self.cond_frame_num
        if not torch.is_tensor(real_vid) or real_vid.dim() != 5 or real_vid.shape[1] != 3 or real_vid.shape[2] < tc:
            raise ValueError(f"interpolate_one_video: real_vid must be a (B, 3, >= {tc}, H, W) tensor")
        self.diffusion.interp_args(x1, x2, tc, t, lam, seeds, noise, who="interpolate_one_video")
        st = int(round(1 / self.region_predictor.scale_factor))
        B, _, _, H, W = real_vid.shape
        if tuple(x1.shape) != (B, 3, self.pred_frame_num, H // st, W // st):
            raise ValueError(f"interpolate_one_video: x1 {tuple(x1.shape)} does not fit real_vid "
                             f"{tuple(real_vid.shape)}: expected {(B, 3, self.pred_frame_num, H // st, W // st)}")
        ret, x_cond, cond_fea, ref = self.condition(real_vid[:, :, :tc].contiguous())
        pred = self.diffusion.interpolate(x1, x2, x_cond, cond_fea, t=t, lam=lam, seeds=seeds, noise=noise)
        if not isinstance(lam, (list, tuple)):
            ret.update(self._decode_sample(ret, ref, pred))
            return ret
        parts = [self._decode_sample(ret, ref, p) for p in pred]
        for k in parts[0]:
            ret[k] = parts[0][k] if k.startswith("real_") else torch.stack([d[k] for d in parts])
        return ret

    # ------------------------------------------------------------------ prediction with known future frames
    @torch.no_grad()
    def sample_with_keyframes(self, real_vid, known, seeds=None, noise=None):
        """sample_one_video with some future frames known: real_vid (B, 3, tc + tp, H, W) in [0, 1], known (B, tp) bool,
        one flag per (video, predicted frame); future frames at unknown positions may hold anything.  x_cond, cond_fea
        and the conditioning entries are condition(real_vid[:, :, :tc]), as sample_one_video computes them; the known
        frames enter as encode_future(real_vid), the LFAE flow of each future frame from source frame tc - 1, imposed
        with GaussianDiffusion.sample_with_known (seeds, noise as there).  Returns sample_one_video's dict, decoded the
        same way.  The latent of a known frame is its encoding bit for bit, so its decoded RGB is the LFAE
        reconstruction of the keyframe, not the keyframe itself.  Argument errors raise ValueError before anything
        runs."""
        tc, tp = self.cond_frame_num, self.pred_frame_num
        if not torch.is_tensor(real_vid) or real_vid.dim() != 5 or real_vid.shape[1] != 3 or \
                real_vid.shape[2] != tc + tp:
            raise ValueError(f"sample_with_keyframes: real_vid must be a (B, 3, {tc + tp} = tc + tp, H, W) tensor")
        B, _, _, H, W = real_vid.shape
        st = int(round(1 / self.region_predictor.scale_factor))
        self.diffusion.known_args((B, 3, tp, H // st, W // st), known, tc, seeds, noise, who="sample_with_keyframes")
        ret, x_cond, cond_fea, ref = self.condition(real_vid[:, :, :tc].contiguous())
        x_known = self.encode_future(real_vid)
        pred = self.diffusion.sample_with_known(x_cond, cond_fea, x_known, known, seeds=seeds, noise=noise)
        ret.update(self._decode_sample(ret, ref, pred))
        return ret

    # ------------------------------------------------------------------ denoising loss (forward-only training objective)
    def _loss_video_shape(self, real_vid):
        """(B, h, w) of a denoising-loss input: real_vid (B, 3, tc + tp, H, W); (h, w) is the flow resolution."""
        if not torch.is_tensor(real_vid) or real_vid.dim() != 5:
            raise ValueError("denoising_loss: real_vid must be a (B, 3, tc + tp, H, W) tensor")
        B, C, T, H, W = real_vid.shape
        if C != 3 or T != self.frame_num or B < 1:
            raise ValueError(f"denoising_loss: real_vid {tuple(real_vid.shape)}: expected (B >= 1, 3, "
                             f"{self.frame_num} = tc + tp, H, W)")
        st = int(round(1 / self.region_predictor.scale_factor))
        return B, H // st, W // st

    @torch.no_grad()
    def loss_inputs(self, real_vid):
        """(x_start, x_cond, cond_fea) of denoising_loss for real_vid (B, 3, tc + tp, H, W) in [0, 1] (DESIGN.md
        section 1): one CondRunner over all tc + tp frames of each video with the source at slot tc - 1.  Its first tc
        flows give x_cond, cond_fea is condition()'s, and x_start is flow_to_x_start of frames tc .. tc + tp - 1, the
        inverse of sample_one_video's post-processing: decoding x_start gives the LFAE reconstruction of those frames."""
        B, _, _ = self._loss_video_shape(real_vid)
        if not real_vid.is_cuda:
            raise RuntimeError("denoising_loss runs on CUDA only (hand-written sm_100a kernels, no CPU fallback)")
        rp, bgp, pfp = self.region_predictor, self.bg_predictor, self.generator.pixelwise_flow_predictor
        if not CondRunner.supported(rp, bgp, pfp):
            raise NotImplementedError("denoising_loss: the conditioning kernels do not cover these predictor "
                                      "hyper-parameters (lfae.CondRunner.supported)")
        if not self.estimate_occlusion_map and self.WRAPPER != "w_ref":
            raise KeyError("occlusion_map")                            # as condition()
        tc, T = self.cond_frame_num, self.frame_num
        _, _, _, H, W = real_vid.shape
        key = (real_vid.device, B, T, H, W, tc - 1)
        if key not in self._cond_runners:
            self._cond_runners[key] = CondRunner(rp, bgp, pfp, real_vid.device, B, T, H, W, src_slot=tc - 1)
        grid, conf = self._cond_runners[key].run(real_vid.float())
        frames = real_vid[:, :, :tc].permute(0, 2, 1, 3, 4).reshape(B * tc, 3, H, W) \
            .contiguous(memory_format=torch.channels_last)
        fea = self._cond_fea(frames, B, grid.shape[-2:])
        if not self.estimate_occlusion_map:
            conf = None
        x_cond = flow_to_x_start(grid[:, :, :tc], None if conf is None else conf[:, :, :tc], False)
        x_start = flow_to_x_start(grid[:, :, tc:], None if conf is None else conf[:, :, tc:], self.use_residual_flow)
        return x_start, x_cond, fea

    @torch.no_grad()
    def denoising_loss(self, real_vid, timesteps=None, seeds=None, noise=None):
        """The diffusion model's training objective evaluated forward-only on real_vid (B, 3, tc + tp, H, W) in [0, 1]:
        GaussianDiffusion.denoising_loss on loss_inputs(real_vid).  timesteps, seeds, noise: as there (noise has the
        shape of x_start, (B, 3, tp, h, w)).  Returns {'loss': (B,), 'loss_per_frame': (B, tp), 'timesteps': (B,)}.
        Argument errors raise ValueError before anything runs; CPU tensors then raise RuntimeError."""
        B, h, w = self._loss_video_shape(real_vid)
        self.diffusion.loss_args(B, (B, 3, self.pred_frame_num, h, w), timesteps, seeds, noise)
        x_start, x_cond, cond_fea = self.loss_inputs(real_vid)
        return self.diffusion.denoising_loss(x_start, x_cond, cond_fea, timesteps=timesteps, seeds=seeds, noise=noise)

    def forward(self, real_vid):
        raise NotImplementedError("training forward is outside the sampling hot path (SURVEY.md section 2, row 3a)")

    @staticmethod
    def get_grid(b, nf, H, W, normalize=True):
        if normalize:
            hr, wr = torch.linspace(-1, 1, H), torch.linspace(-1, 1, W)
        else:
            hr, wr = torch.arange(0, H), torch.arange(0, W)
        grid = torch.stack(torch.meshgrid(hr, wr, indexing="xy"), -1).repeat(b, 1, 1, 1).flip(3).float()
        return grid.permute(0, 3, 1, 2).unsqueeze(dim=2).repeat(1, 1, nf, 1, 1)


def x_start_to_flow(x, use_residual_flow, with_conf):
    """sample_one_video's post-processing of a sampled x (B, 3, tp, h, w): (grid (B, 2, tp, h, w), conf (B, 1, tp, h, w)
    or None).  grid = x[:, :2] (+ the identity grid with use_residual_flow); conf = (x[:, 2:3] + 1) * 0.5."""
    grid = x[:, :2]
    if use_residual_flow:
        grid = grid + FlowDiffusion.get_grid(grid.shape[0], 1, grid.shape[3], grid.shape[4]).to(grid.device)
    return grid, ((x[:, 2:3] + 1) * 0.5 if with_conf else None)


def flow_to_x_start(grid, conf, use_residual_flow):
    """The inverse of x_start_to_flow: (grid - the identity grid with use_residual_flow | conf * 2 - 1, or zeros
    without an occlusion map) -> (B, 3, T, h, w).  With use_residual_flow=False this is condition()'s x_cond."""
    if use_residual_flow:
        grid = grid - FlowDiffusion.get_grid(grid.shape[0], 1, grid.shape[3], grid.shape[4]).to(grid.device)
    third = conf * 2 - 1 if conf is not None else torch.zeros_like(grid)[:, 0:1]
    return torch.cat((grid, third), dim=1)


class FlowDiffusionMulti1248(FlowDiffusion):
    WRAPPER = "multi1248"


class FlowDiffusionU22(FlowDiffusion):
    """VideoFlowDiffusion_multi_w_ref_u22.py:142-236,415-510: the w_ref pipeline around the ada_u22 UNet.  The
    reference spreads LFAE and DM over `device_ids` (model parallel, one video batch at a time); here the whole
    round runs on one GPU and videos shard across ranks (sharding.py), so `device_ids` is accepted and ignored."""

    def __init__(self, config="", pretrained_pth="", is_train=True, ddim_sampling_eta=1.0, timesteps=1000,
                 dim_mults=(1, 2, 4, 4), learn_null_cond=False, use_deconv=True, padding_mode="zeros", withFea=True,
                 Unet3D_architecture="DenoiseNet_STWAtt_w_w_ref_adaptor_cross_multi_traj_ada_u22", device_ids=None):
        super().__init__(config, pretrained_pth, is_train, ddim_sampling_eta, timesteps, dim_mults, learn_null_cond,
                         use_deconv, padding_mode, withFea, Unet3D_architecture)


class FlowDiffusionMulti(FlowDiffusion):
    WRAPPER = "multi"


WRAPPERS = {
    "VideoFlowDiffusion_multi_w_ref": FlowDiffusion,
    "VideoFlowDiffusion_multi1248": FlowDiffusionMulti1248,
    "VideoFlowDiffusion_multi": FlowDiffusionMulti,
    "VideoFlowDiffusion_multi_w_ref_u22": FlowDiffusionU22,
}


def flow_diffusion_class(dm_arch):
    """`--DM_arch` string (scripts/DM/valid.py:83-92) -> class."""
    if dm_arch not in WRAPPERS:
        raise NotImplementedError(f"unknown DM architecture {dm_arch!r}")
    return WRAPPERS[dm_arch]
