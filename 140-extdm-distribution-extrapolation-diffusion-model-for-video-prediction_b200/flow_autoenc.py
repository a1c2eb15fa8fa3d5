"""FlowAE: stage-1 inference of the latent flow autoencoder (LFAE), the reference's `FlowAE` inference shell
(model/LFAE/flow_autoenc.py) and its AE validation (scripts/AE/valid.py).  Every frame of a video is reconstructed
from one source frame of the same video plus that frame's region motion:

    src_params = region_predictor(source)        drv_params = region_predictor(frame_t)
    bg         = bg_predictor(source, frame_t)
    out        = generator(source, source_region_params=src_params, driving_region_params=drv_params, bg_params=bg)

A predicted frame of the diffusion model is the LFAE decode of a sampled flow, so the reconstruction of the true frame
bounds what sampling can reach.

On a CUDA device the whole video batch runs as one CUDA graph (lfae.ReconRunner): the conditioning kernels with the
source at any slot, then the decoder of Generator.decode_video.  CPU tensors, and predictor hyper-parameters the
kernels do not cover (lfae.CondRunner.supported), run the torch modules.
"""
import operator
import weakref
from collections import OrderedDict

import torch
from torch import nn

from .lfae import BGMotionPredictor, CondRunner, Generator, ReconRunner, RegionPredictor

_PARTS = ("generator", "region_predictor", "bg_predictor")


class FlowAE(nn.Module):
    native = True      # class-level switch: False runs the torch modules on CUDA too (tests A/B, tools/recon_bench.py)
    # CUDA runners kept per FlowAE, least recently used evicted first.  Each (device, B, T, H, W, source_frame) has its own
    # runner: fp32 buffers for all B*T frames plus a graph (several GB at B = 32, T = 50), so a sweep over source frames
    # must not keep one per frame.  The decoder's buffers are the Generator's, one set per shape.
    max_runners = 2

    def __init__(self, config, pretrained_pth=""):
        """config: the dataset configuration dict (configs.dataset or a user's yaml.safe_load); the modules are built
        from config["flow_params"]["model_params"] as FlowDiffusion builds them.  pretrained_pth: an LFAE checkpoint
        whose 'generator', 'region_predictor' and 'bg_predictor' entries are loaded strictly."""
        super().__init__()
        flow_params = config["flow_params"]["model_params"]
        dev = "cuda" if torch.cuda.is_available() else "cpu"
        self.generator = Generator(num_regions=flow_params["num_regions"], num_channels=flow_params["num_channels"],
                                   revert_axis_swap=flow_params["revert_axis_swap"],
                                   **flow_params["generator_params"]).to(dev)
        self.region_predictor = RegionPredictor(num_regions=flow_params["num_regions"],
                                                num_channels=flow_params["num_channels"],
                                                estimate_affine=flow_params["estimate_affine"],
                                                **flow_params["region_predictor_params"]).to(dev)
        self.bg_predictor = BGMotionPredictor(num_channels=flow_params["num_channels"],
                                              **flow_params["bg_predictor_params"]).to(dev)
        if pretrained_pth != "":
            ckpt = torch.load(pretrained_pth, map_location=dev)
            absent = [p for p in _PARTS if p not in ckpt]
            if absent:
                raise KeyError(f"LFAE checkpoint {pretrained_pth}: no {absent} entries")
            for part in _PARTS:
                getattr(self, part).load_state_dict(ckpt[part], strict=True)
        self._setup()

    @classmethod
    def from_flow_diffusion(cls, model):
        """A FlowAE on the LFAE modules of a FlowDiffusion model: the modules are shared, not copied."""
        ae = cls.__new__(cls)
        nn.Module.__init__(ae)
        for part in _PARTS:
            setattr(ae, part, getattr(model, part))
        ae._setup()
        return ae

    def _setup(self):
        if self.generator.pixelwise_flow_predictor is None:
            raise ValueError("FlowAE: the generator has no pixelwise_flow_predictor (generator_params)")
        for m in (self.generator, self.region_predictor, self.bg_predictor):
            m.eval()
            for p in m.parameters():
                p.requires_grad = False
        self.estimate_occlusion_map = self.generator.pixelwise_flow_predictor.occlusion is not None
        self._runners = OrderedDict()
        # new weights invalidate the runners' packed copies.  The hooks hold only a weak reference, so modules shared
        # with a FlowDiffusion do not keep this FlowAE (and its graphs) alive, and they are removed when it goes.
        ref = weakref.ref(self)

        def clear_runners(module, incompatible_keys):
            ae = ref()
            if ae is not None:
                ae._runners.clear()

        handles = [m.register_load_state_dict_post_hook(clear_runners)
                   for m in (self.generator, self.region_predictor, self.bg_predictor)]
        weakref.finalize(self, _remove_hooks, handles)

    def _check(self, real_vid, source_frame):
        if not torch.is_tensor(real_vid) or real_vid.dim() != 5:
            raise ValueError(f"FlowAE: real_vid must be a (B, C, T, H, W) tensor, got "
                             f"{tuple(real_vid.shape) if torch.is_tensor(real_vid) else type(real_vid).__name__}")
        B, C, T, H, W = real_vid.shape
        if C != self.generator.num_channels or B < 1 or T < 1:
            raise ValueError(f"FlowAE: real_vid {tuple(real_vid.shape)}: expected (B >= 1, "
                             f"{self.generator.num_channels}, T >= 1, H, W)")
        try:
            index = None if isinstance(source_frame, bool) else operator.index(source_frame)
        except TypeError:
            index = None
        if index is None or not 0 <= index < T:
            raise ValueError(f"FlowAE: source_frame {source_frame!r} is not a frame index in [0, {T})")
        dev = self.generator.final.weight.device
        if real_vid.device != dev:
            raise ValueError(f"FlowAE: real_vid on {real_vid.device}, modules on {dev}")
        return index

    @torch.no_grad()
    def reconstruct(self, real_vid, source_frame=0):
        """real_vid (B, 3, T, H, W) in [0, 1] -> {'prediction', 'deformed': (B, 3, T, H, W), 'optical_flow':
        (B, 2, T, h, w), 'occlusion_map': (B, 1, T, h, w) when the generator estimates one}: frame t of video b
        reconstructed from frame `source_frame` of video b (any integer type).  The tensors are the caller's: later
        calls do not overwrite them."""
        source_frame = self._check(real_vid, source_frame)
        pfp = self.generator.pixelwise_flow_predictor
        if not (real_vid.is_cuda and self.native and CondRunner.supported(self.region_predictor, self.bg_predictor, pfp)):
            return self.reconstruct_torch(real_vid, source_frame)
        B, _, T, H, W = real_vid.shape
        key = (real_vid.device, B, T, H, W, source_frame)
        if key in self._runners:
            self._runners.move_to_end(key)
        else:
            while len(self._runners) >= max(self.max_runners, 1):
                self._runners.popitem(last=False)
            self._runners[key] = ReconRunner(self.generator, self.region_predictor, self.bg_predictor, real_vid.device,
                                             B, T, H, W, source_frame)
        out = self._runners[key].run(real_vid.float())
        # copies, never views: the runner's buffers are rewritten by the next call of the same shape
        return {k: v.clone(memory_format=torch.contiguous_format) for k, v in out.items()}

    @torch.no_grad()
    def reconstruct_torch(self, real_vid, source_frame=0):
        """The same reconstruction with the torch modules, batched over the B*T frames: the CPU path and the parity
        partner of the CUDA graph."""
        source_frame = self._check(real_vid, source_frame)
        B, _, T, H, W = real_vid.shape
        real_vid = real_vid.float()
        source = real_vid[:, :, source_frame]
        frames = real_vid.permute(0, 2, 1, 3, 4).reshape(B * T, -1, H, W)
        src_rep = source.repeat_interleave(T, dim=0)
        src_params = {k: v.repeat_interleave(T, dim=0) for k, v in self.region_predictor(source).items()}
        drv_params = self.region_predictor(frames)
        bg = self.bg_predictor(src_rep, frames)
        gen = self.generator(src_rep, source_region_params=src_params, driving_region_params=drv_params, bg_params=bg)
        per_video = lambda t: t.reshape(B, T, *t.shape[1:]).transpose(1, 2).contiguous()    # (B*T, C, ..) -> (B, C, T, ..)
        out = {"prediction": per_video(gen["prediction"]), "deformed": per_video(gen["deformed"]),
               "optical_flow": per_video(gen["optical_flow"].permute(0, 3, 1, 2))}
        if "occlusion_map" in gen:
            out["occlusion_map"] = per_video(gen["occlusion_map"])
        return out

    def forward(self, real_vid, source_frame=0):
        return self.reconstruct(real_vid, source_frame)


def _remove_hooks(handles):
    for h in handles:
        h.remove()
