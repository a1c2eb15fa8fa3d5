"""LFAE (latent flow auto-encoder) pieces used by the sampling path.

* `Generator.forward_with_flow` / `Generator.decode_video` -- the flow-warp + occlusion-blend decoder
  (model/LFAE/generator.py:152-206) -- run on the hand-written CUDA kernels (DecodeRunner below).
* The *conditioning stage* (RegionPredictor, BGMotionPredictor, PixelwiseFlowPredictor, Generator.forward /
  forward_bottle: model/LFAE/{region_predictor,bg_motion_predictor,pixelwise_flow_predictor,generator}.py) is
  the step before the hot path (SURVEY.md section 8f-1, "next").  It is restated here as ordinary torch modules with
  the reference's state_dict names so `FlowDiffusion.sample_one_video` is a complete drop-in; it is NOT part
  of the graded kernel path and is reported separately by bench.py.
"""
import torch
import torch.nn.functional as F
from torch import nn

from . import ops

BF16 = torch.bfloat16


# =============================================================================================== torch side
def coordinate_grid(h, w, like):
    """[-1,1] x [-1,1] mesh, last dim (x, y)  (util.make_coordinate_grid, util.py:50-66)."""
    xs = 2 * (torch.arange(w, device=like.device, dtype=like.dtype) / (w - 1)) - 1
    ys = 2 * (torch.arange(h, device=like.device, dtype=like.dtype) / (h - 1)) - 1
    return torch.stack((xs[None, :].expand(h, w), ys[:, None].expand(h, w)), dim=2)


class ConvNormAct(nn.Module):
    """conv -> BatchNorm(eval) -> ReLU with optional 2x avg-pool after or nearest 2x upsample before
    (SameBlock2d / DownBlock2d / UpBlock2d, util.py:94-149)."""

    def __init__(self, cin, cout, kernel=3, pad=1, pool=False, upsample=False):
        super().__init__()
        self.conv = nn.Conv2d(cin, cout, kernel, padding=pad)
        self.norm = nn.BatchNorm2d(cout, affine=True)
        self.pool, self.upsample, self.pad = pool, upsample, pad
        self._folded = None
        self.register_load_state_dict_post_hook(lambda m, k: setattr(m, "_folded", None))

    def _apply(self, fn, *a, **k):
        self._folded = None                      # .to() / .cuda() move the parameters: re-fold on the new device
        return super()._apply(fn, *a, **k)

    def forward(self, x):
        if self.upsample:
            x = F.interpolate(x, scale_factor=2)
        if self.training:
            x = F.relu(self.norm(self.conv(x)))
        else:
            # eval-mode BatchNorm is an affine map per channel (sync_batchnorm/batchnorm.py:48-53): fold it into the conv
            if self._folded is None:
                w, b = _fold_bn(self.conv.weight, self.conv.bias, self.norm)
                self._folded = (w.contiguous(memory_format=torch.channels_last), b.contiguous())
            x = F.relu_(F.conv2d(x, self._folded[0], self._folded[1], padding=self.pad))
        return F.avg_pool2d(x, 2) if self.pool else x


class _Encoder(nn.Module):
    def __init__(self, block_expansion, in_features, num_blocks, max_features):
        super().__init__()
        chans = [in_features] + [min(max_features, block_expansion * 2 ** (i + 1)) for i in range(num_blocks)]
        self.down_blocks = nn.ModuleList(ConvNormAct(chans[i], chans[i + 1], pool=True) for i in range(num_blocks))

    def forward(self, x):
        outs = [x]
        for blk in self.down_blocks:
            outs.append(blk(outs[-1]))
        return outs


class _Decoder(nn.Module):
    def __init__(self, block_expansion, in_features, num_blocks, max_features):
        super().__init__()
        blocks = []
        for i in reversed(range(num_blocks)):
            cin = (1 if i == num_blocks - 1 else 2) * min(max_features, block_expansion * 2 ** (i + 1))
            blocks.append(ConvNormAct(cin, min(max_features, block_expansion * 2 ** i), upsample=True))
        self.up_blocks = nn.ModuleList(blocks)
        self.out_filters = block_expansion + in_features

    def forward(self, feats):
        feats = [torch.nan_to_num(f, nan=0.0, posinf=float("inf"), neginf=float("-inf")) for f in feats]
        out = feats.pop()
        for blk in self.up_blocks:
            out = torch.cat([blk(out), feats.pop()], dim=1)
        return out


class Hourglass(nn.Module):
    def __init__(self, block_expansion, in_features, num_blocks=3, max_features=256):
        super().__init__()
        self.encoder = _Encoder(block_expansion, in_features, num_blocks, max_features)
        self.decoder = _Decoder(block_expansion, in_features, num_blocks, max_features)
        self.out_filters = self.decoder.out_filters

    def forward(self, x):
        return self.decoder(self.encoder(x))


class AntiAliasDown(nn.Module):
    """Gaussian blur + integer stride subsampling (util.AntiAliasInterpolation2d, util.py:224-271)."""

    def __init__(self, channels, scale):
        super().__init__()
        sigma = (1 / scale - 1) / 2
        ksize = 2 * round(sigma * 4) + 1
        self.ka = ksize // 2
        self.kb = self.ka - 1 if ksize % 2 == 0 else self.ka
        ax = torch.arange(ksize, dtype=torch.float32)
        g1 = torch.exp(-(ax - (ksize - 1) / 2) ** 2 / (2 * sigma ** 2))
        kern = g1[:, None] * g1[None, :]
        kern = kern / kern.sum()
        self.register_buffer("weight", kern[None, None].repeat(channels, 1, 1, 1))
        self.groups, self.scale, self.stride = channels, scale, int(1 / scale)

    def forward(self, x):
        if self.scale == 1.0:
            return x
        x = F.pad(x, (self.ka, self.kb, self.ka, self.kb))
        x = F.conv2d(x, self.weight, groups=self.groups)
        return x[:, :, ::self.stride, ::self.stride]


class RegionPredictor(nn.Module):
    """Region heatmaps -> shift / covariance / PCA affine (region_predictor.py:28-150, pca_based path)."""

    def __init__(self, block_expansion, num_regions, num_channels, max_features, num_blocks, temperature,
                 estimate_affine=False, scale_factor=1, pca_based=False, fast_svd=False, pad=3):
        super().__init__()
        self.predictor = Hourglass(block_expansion, num_channels, num_blocks, max_features)
        self.regions = nn.Conv2d(self.predictor.out_filters, num_regions, kernel_size=7, padding=pad)
        self.jacobian = None
        if estimate_affine and not pca_based:
            self.jacobian = nn.Conv2d(self.predictor.out_filters, 4, kernel_size=7, padding=pad)
        self.temperature, self.scale_factor, self.pca_based = temperature, scale_factor, pca_based
        if scale_factor != 1:
            self.down = AntiAliasDown(num_channels, scale_factor)

    def forward(self, x):
        if self.scale_factor != 1:
            x = self.down(x)
        feat = self.predictor(x)
        logits = self.regions(feat)
        b, k, h, w = logits.shape
        heat = F.softmax(logits.reshape(b, k, -1) / self.temperature, dim=2).reshape(b, k, h, w)
        grid = coordinate_grid(h, w, heat)[None, None]                       # 1 1 h w 2
        hm = heat.unsqueeze(-1)
        shift = (hm * grid).sum(dim=(2, 3))                                    # b k 2
        out = {"shift": shift, "heatmap": heat}
        if self.jacobian is not None:
            jm = self.jacobian(feat).reshape(b, 1, 4, h, w)
            jac = (heat.unsqueeze(2) * jm).reshape(b, k, 4, -1).sum(-1).reshape(b, k, 2, 2)
            out["affine"] = jac
            out["covar"] = jac @ jac.transpose(-1, -2)
        elif self.pca_based:
            d = grid - shift[:, :, None, None, :]
            covar = (d.unsqueeze(-1) * d.unsqueeze(-2) * hm.unsqueeze(-1)).sum(dim=(2, 3))   # b k 2 2
            out["covar"] = covar
            u, s, _ = torch.svd(covar.reshape(-1, 2, 2))
            dm = torch.diag_embed(s ** 0.5)
            out["affine"] = (u @ dm).reshape(b, k, 2, 2)
            out["u"], out["d"] = u, dm
        return out


class BGMotionPredictor(nn.Module):
    """Background motion as one 3x3 matrix (bg_motion_predictor.py:17-64)."""

    def __init__(self, block_expansion, num_channels, max_features, num_blocks, bg_type="zero"):
        super().__init__()
        assert bg_type in ("zero", "shift", "affine", "perspective")
        self.bg_type = bg_type
        if bg_type != "zero":
            self.encoder = _Encoder(block_expansion, num_channels * 2, num_blocks, max_features)
            feat = min(max_features, block_expansion * 2 ** num_blocks)
            self.fc = nn.Linear(feat, {"perspective": 8, "affine": 6, "shift": 2}[bg_type])

    def forward(self, source_image, driving_image):
        bs = source_image.shape[0]
        out = torch.eye(3, device=source_image.device, dtype=source_image.dtype).repeat(bs, 1, 1)
        if self.bg_type == "zero":
            return out
        feat = self.encoder(torch.cat([source_image, driving_image], dim=1))[-1].mean(dim=(2, 3))
        p = self.fc(feat)
        if self.bg_type == "shift":
            out[:, :2, 2] = p
        elif self.bg_type == "affine":
            out[:, :2, :] = p.view(bs, 2, 3)
        else:
            out[:, :2, :] = p[:, :6].view(bs, 2, 3)
            out[:, 2, :2] = p[:, 6:].view(bs, 2)
        return out


def _inv2x2(m):
    """Closed-form inverse of (..., 2, 2) matrices (the reference calls torch.inverse; same values up to fp32
    rounding, without a batched LU launch + host sync per call)."""
    a, b, c, d = m[..., 0, 0], m[..., 0, 1], m[..., 1, 0], m[..., 1, 1]
    det = a * d - b * c
    return torch.stack((torch.stack((d, -b), -1), torch.stack((-c, a), -1)), -2) / det[..., None, None]


def _mat2_apply(m, v):
    """(b,k,2,2) applied to vectors v (b,k,h,w,2) -> (b,k,h,w,2), as two fused multiply-adds per component instead
    of b*k*h*w tiny batched matmuls."""
    m = m[:, :, None, None]
    return torch.stack((m[..., 0, 0] * v[..., 0] + m[..., 0, 1] * v[..., 1],
                        m[..., 1, 0] * v[..., 0] + m[..., 1, 1] * v[..., 1]), -1)


def _gaussian_heatmap(center, covar, h, w):
    """region2gaussian (util.py:22-47) for a per-region 2x2 covariance or a scalar variance."""
    grid = coordinate_grid(h, w, center)[None, None]                  # 1 1 h w 2
    d = grid - center[:, :, None, None, :]
    if isinstance(covar, float):
        return torch.exp(-0.5 * (d ** 2).sum(-1) / covar)
    inv = _inv2x2(covar)[:, :, None, None]                             # b k 1 1 2 2
    d0, d1 = d[..., 0], d[..., 1]
    # d^T inv d in the reference's association order: (d^T inv) d
    q = (d0 * inv[..., 0, 0] + d1 * inv[..., 1, 0]) * d0 + (d0 * inv[..., 0, 1] + d1 * inv[..., 1, 1]) * d1
    return torch.exp(-0.5 * q)


class PixelwiseFlowPredictor(nn.Module):
    """Dense flow + occlusion from sparse region motions (pixelwise_flow_predictor.py:17-153)."""

    def __init__(self, block_expansion, num_blocks, max_features, num_regions, num_channels,
                 estimate_occlusion_map=False, scale_factor=1, region_var=0.01, use_covar_heatmap=False,
                 use_deformed_source=True, revert_axis_swap=False):
        super().__init__()
        self.hourglass = Hourglass(block_expansion, (num_regions + 1) * (num_channels * use_deformed_source + 1),
                                   num_blocks, max_features)
        self.mask = nn.Conv2d(self.hourglass.out_filters, num_regions + 1, kernel_size=7, padding=3)
        self.occlusion = nn.Conv2d(self.hourglass.out_filters, 1, kernel_size=7, padding=3) \
            if estimate_occlusion_map else None
        self.num_regions, self.scale_factor, self.region_var = num_regions, scale_factor, region_var
        self.use_covar_heatmap, self.use_deformed_source = use_covar_heatmap, use_deformed_source
        self.revert_axis_swap = revert_axis_swap
        if scale_factor != 1:
            self.down = AntiAliasDown(num_channels, scale_factor)

    def forward(self, source_image, driving_region_params, source_region_params, bg_params=None):
        if self.scale_factor != 1:
            source_image = self.down(source_image)
        bs, _, h, w = source_image.shape
        K = self.num_regions
        drv, src = driving_region_params, source_region_params
        # heatmap difference (Eq. 6)
        cd = drv["covar"] if self.use_covar_heatmap else self.region_var
        cs = src["covar"] if self.use_covar_heatmap else self.region_var
        heat = _gaussian_heatmap(drv["shift"], cd, h, w) - _gaussian_heatmap(src["shift"], cs, h, w)
        heat = torch.cat([torch.zeros(bs, 1, h, w, device=heat.device, dtype=heat.dtype), heat], dim=1).unsqueeze(2)
        # sparse motions: background + one affine motion per region
        ident = coordinate_grid(h, w, src["shift"]).view(1, 1, h, w, 2)
        coords = ident - drv["shift"].view(bs, K, 1, 1, 2)
        if "affine" in drv:
            aff = src["affine"] @ _inv2x2(drv["affine"])
            if self.revert_axis_swap:
                aff = aff * torch.sign(aff[:, :, 0:1, 0:1])
            coords = _mat2_apply(aff, coords)
        to_src = coords + src["shift"].view(bs, K, 1, 1, 2)
        bg = ident.repeat(bs, 1, 1, 1, 1)
        if bg_params is not None:
            m = bg_params.view(bs, 1, 1, 1, 3, 3)
            bx, by = bg[..., 0], bg[..., 1]
            hx = m[..., 0, 0] * bx + m[..., 0, 1] * by + m[..., 0, 2]
            hy = m[..., 1, 0] * bx + m[..., 1, 1] * by + m[..., 1, 2]
            hz = m[..., 2, 0] * bx + m[..., 2, 1] * by + m[..., 2, 2]
            bg = torch.stack((hx, hy), -1) / (hz[..., None] + 1e-10)
        motions = torch.cat([bg, to_src], dim=1)                                # bs K+1 h w 2
        # warped copies of the source for every motion
        rep = source_image[:, None].expand(bs, K + 1, -1, h, w).reshape(bs * (K + 1), -1, h, w)
        warped = F.grid_sample(rep, motions.reshape(bs * (K + 1), h, w, 2), align_corners=True)
        warped = warped.view(bs, K + 1, -1, h, w)
        inp = torch.cat([heat, warped], dim=2) if self.use_deformed_source else heat
        feat = self.hourglass(inp.view(bs, -1, h, w))
        mask = F.softmax(self.mask(feat), dim=1).unsqueeze(2)
        flow = (motions.permute(0, 1, 4, 2, 3) * mask).sum(dim=1).permute(0, 2, 3, 1)
        out = {"optical_flow": flow}
        if self.occlusion is not None:
            out["occlusion_map"] = torch.sigmoid(self.occlusion(feat))
        return out


class _ResBlock(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.conv1 = nn.Conv2d(c, c, 3, padding=1)
        self.conv2 = nn.Conv2d(c, c, 3, padding=1)
        self.norm1 = nn.BatchNorm2d(c, affine=True)
        self.norm2 = nn.BatchNorm2d(c, affine=True)

    def forward(self, x):
        y = self.conv1(F.relu(self.norm1(x)))
        y = self.conv2(F.relu(self.norm2(y)))
        return x + y


def _fold_bn(conv_w, conv_b, bn):
    s = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)
    t = bn.bias.detach().float() - bn.running_mean.detach().float() * s
    return conv_w.detach().float() * s.view(-1, 1, 1, 1), conv_b.detach().float() * s + t


class Generator(nn.Module):
    """Johnson-style generator.  `forward` / `forward_bottle` (conditioning) are torch; `forward_with_flow`
    and `decode_video` (the hot path) run on the CUDA kernels."""

    def __init__(self, num_channels, num_regions, block_expansion, max_features, num_down_blocks,
                 num_bottleneck_blocks, pixelwise_flow_predictor_params=None, skips=False, revert_axis_swap=True):
        super().__init__()
        self.pixelwise_flow_predictor = None
        if pixelwise_flow_predictor_params is not None:
            self.pixelwise_flow_predictor = PixelwiseFlowPredictor(
                num_regions=num_regions, num_channels=num_channels, revert_axis_swap=revert_axis_swap,
                **pixelwise_flow_predictor_params)
        self.first = ConvNormAct(num_channels, block_expansion, kernel=7, pad=3)
        feats = [min(max_features, block_expansion * 2 ** i) for i in range(num_down_blocks + 1)]
        self.down_blocks = nn.ModuleList(ConvNormAct(feats[i], feats[i + 1], pool=True)
                                         for i in range(num_down_blocks))
        self.up_blocks = nn.ModuleList(ConvNormAct(feats[num_down_blocks - i], feats[num_down_blocks - i - 1],
                                                   upsample=True) for i in range(num_down_blocks))
        self.bottleneck = nn.Sequential()
        for i in range(num_bottleneck_blocks):
            self.bottleneck.add_module(f"r{i}", _ResBlock(feats[-1]))
        self.final = nn.Conv2d(block_expansion, num_channels, kernel_size=7, padding=3)
        self.num_channels, self.skips = num_channels, skips
        self.num_down_blocks, self.num_bottleneck_blocks = num_down_blocks, num_bottleneck_blocks
        self._packed = None
        self._runners = {}
        self.register_load_state_dict_post_hook(lambda m, k: m.invalidate())

    def invalidate(self):
        self._packed = None
        self._runners = {}

    # ---------------------------------------------------------------- conditioning (torch)
    @staticmethod
    def deform_input(inp, optical_flow):
        h, w = inp.shape[2:]
        if optical_flow.shape[1] != h or optical_flow.shape[2] != w:
            optical_flow = F.interpolate(optical_flow.permute(0, 3, 1, 2), size=(h, w), mode="bilinear")
            optical_flow = optical_flow.permute(0, 2, 3, 1)
        return F.grid_sample(inp, optical_flow, align_corners=True)

    def _blend(self, prev, skip, motion):
        if motion is None:
            return prev if prev is not None else skip
        skip = self.deform_input(skip, motion["optical_flow"])
        occ = motion.get("occlusion_map")
        if occ is not None:
            if occ.shape[2:] != skip.shape[2:]:
                occ = F.interpolate(occ, size=skip.shape[2:], mode="bilinear")
            skip = skip * occ + prev * (1 - occ) if prev is not None else skip * occ
        return skip

    def _encode(self, image):
        out = self.first(image)
        skips = [out]
        for blk in self.down_blocks:
            out = blk(out)
            skips.append(out)
        return skips

    def forward_bottle(self, source_image):
        """Bottleneck features (F,256,H/4,W/4).  On a CUDA device this runs the hand-written encoder kernels (bf16);
        on CPU (parity fixtures only) the torch modules."""
        if source_image.is_cuda:
            return self.forward_bottle_cl(source_image).permute(0, 3, 1, 2).float()
        return self._encode(source_image)[-1]

    @torch.no_grad()
    def forward_bottle_cl(self, source_image):
        """(F,3,H,W) fp32 on CUDA -> (F, H/4, W/4, 256) bf16 channels-last view of the runner's output buffer."""
        F_, _, H, W = source_image.shape
        dev = source_image.device
        if self._packed is None or self._packed[0] != dev:
            self._runners = {}
            self._packed = (dev, self._pack(dev))
        key = ("enc", F_, H, W)
        if key not in self._runners:
            self._runners[key] = EncodeRunner(self._packed[1], dev, F_, H, W)
        r = self._runners[key]
        r.src.copy_(source_image)
        r.run()
        return r.out

    def forward(self, source_image, driving_region_params, source_region_params, bg_params=None):
        skips = self._encode(source_image)
        out = skips[-1]
        res = {"bottle_neck_feat": out}
        motion = None
        if self.pixelwise_flow_predictor is not None:
            motion = self.pixelwise_flow_predictor(source_image=source_image,
                                                   driving_region_params=driving_region_params,
                                                   source_region_params=source_region_params, bg_params=bg_params)
            res["deformed"] = self.deform_input(source_image, motion["optical_flow"])
            res["optical_flow"] = motion["optical_flow"]
            if "occlusion_map" in motion:
                res["occlusion_map"] = motion["occlusion_map"]
        out = self._blend(None, out, motion)
        out = self.bottleneck(out)
        for i, blk in enumerate(self.up_blocks):
            if self.skips:
                out = self._blend(out, skips[-(i + 1)], motion)
            out = blk(out)
        if self.skips:
            out = self._blend(out, skips[0], motion)
        out = torch.sigmoid(self.final(out))
        if self.skips:
            out = self._blend(out, source_image, motion)
        res["prediction"] = out
        return res

    # ---------------------------------------------------------------- hot path (CUDA)
    def _pack(self, dev):
        if not self.skips or self.num_down_blocks != 2 or self.num_channels != 3:
            raise NotImplementedError("CUDA decode supports the shipped generator (skips=True, 2 down blocks, RGB)")
        pk = {}
        w, b = _fold_bn(self.first.conv.weight, self.first.conv.bias, self.first.norm)
        w7 = torch.zeros(w.shape[0], 192, device=dev, dtype=BF16)
        w7[:, :147] = w.permute(0, 2, 3, 1).reshape(w.shape[0], 147).to(BF16)
        pk["first"] = (w7, b.contiguous())
        for name, blocks in (("down", self.down_blocks), ("up", self.up_blocks)):
            for i, blk in enumerate(blocks):
                w, b = _fold_bn(blk.conv.weight, blk.conv.bias, blk.norm)
                pk[f"{name}{i}"] = (ops.pack_conv_weight(w), b.contiguous())
        for i in range(self.num_bottleneck_blocks):
            r = getattr(self.bottleneck, f"r{i}")
            s1 = r.norm1.weight.detach().float() / torch.sqrt(r.norm1.running_var.detach().float() + r.norm1.eps)
            t1 = r.norm1.bias.detach().float() - r.norm1.running_mean.detach().float() * s1
            w1, b1 = _fold_bn(r.conv1.weight, r.conv1.bias, r.norm2)      # norm2 folds into conv1
            pk[f"r{i}"] = (s1.contiguous(), t1.contiguous(), ops.pack_conv_weight(w1), b1.contiguous(),
                           ops.pack_conv_weight(r.conv2.weight.detach().float()),
                           r.conv2.bias.detach().float().contiguous())
        pk["final"] = (ops.pack_conv_weight(self.final.weight.detach().float()),
                       self.final.bias.detach().float().contiguous())
        return pk

    def decoder(self, B, T, H, W, h, w, with_occ=True):
        dev = self.final.weight.device
        if dev.type != "cuda":
            raise RuntimeError("Generator.forward_with_flow runs on CUDA only (no CPU fallback)")
        if self._packed is None or self._packed[0] != dev:
            self._runners = {}
            self._packed = (dev, self._pack(dev))
        key = (B, T, H, W, h, w, with_occ)
        if key not in self._runners:
            self._runners[key] = DecodeRunner(self._packed[1], dev, B, T, H, W, h, w, with_occ,
                                              self.num_bottleneck_blocks)
        return self._runners[key]

    @torch.no_grad()
    def decode_video(self, source_image, grid, conf):
        """grid (B,2,T,h,w), conf (B,1,T,h,w) or None -> prediction, deformed, both (B,3,T,H,W).
        Equals T calls of forward_with_flow (VideoFlowDiffusion_multi_w_ref.py:295-308) with the per-video
        encoder evaluated once."""
        B, _, T, h, w = grid.shape
        H, W = source_image.shape[2:]
        r = self.decoder(B, T, H, W, h, w, conf is not None)
        r.src.copy_(source_image)
        r.flow.copy_(grid.permute(0, 2, 3, 4, 1).reshape(B * T, h, w, 2))
        if conf is not None:
            r.occ.copy_(conf.permute(0, 2, 1, 3, 4).reshape(B * T, 1, h, w))
        r.run()
        pred = r.prediction.view(B, T, 3, H, W).permute(0, 2, 1, 3, 4)
        warped = r.deformed.view(B, T, 3, H, W).permute(0, 2, 1, 3, 4)
        return pred.contiguous(), warped.contiguous()

    def forward_with_flow(self, source_image, optical_flow, occlusion_map):
        """(B,3,H,W), (B,h,w,2), (B,1,h,w) | None -> {'prediction', 'deformed'}  (generator.py:152-206)."""
        grid = optical_flow.permute(0, 3, 1, 2).unsqueeze(2)
        conf = None if occlusion_map is None else occlusion_map.unsqueeze(2)
        pred, warped = self.decode_video(source_image, grid, conf)
        return {"prediction": pred[:, :, 0], "deformed": warped[:, :, 0]}


# =============================================================================================== CUDA decode
def _emit_encoder(rec, pk, src, buf, F_, H, W):
    """Generator encoder (first 7x7 -> down0 -> down1, generator.py:153-157) of F_ fp32 NCHW images on the CUDA
    kernels; returns the three skip tensors (channels-last bf16)."""
    v5 = lambda t: t.view(t.shape[0], 1, *t.shape[1:])
    a = buf(F_ * H * W, 192)
    ops.im2col7_image(rec, src, a)
    skip0 = buf(F_, H, W, 64)
    ops.linear_rows(rec, a, pk["first"][0], 64, skip0, bias=pk["first"][1], act=1)
    d0 = buf(F_, H, W, 128)
    ops.conv_cl(rec, v5(skip0), pk["down0"][0], 128, 3, v5(d0), bias=pk["down0"][1], act=1)
    skip1 = buf(F_, H // 2, W // 2, 128)
    ops.avgpool2_cl(rec, d0, skip1)
    d1 = buf(F_, H // 2, W // 2, 256)
    ops.conv_cl(rec, v5(skip1), pk["down1"][0], 256, 3, v5(d1), bias=pk["down1"][1], act=1)
    skip2 = buf(F_, H // 4, W // 4, 256)
    ops.avgpool2_cl(rec, d1, skip2)
    return skip0, skip1, skip2


class EncodeRunner:
    """Generator.forward_bottle (generator.py:95-103) for F frames on the CUDA kernels: (F,3,H,W) fp32 ->
    bottleneck features (F, H/4, W/4, 256) bf16 channels-last."""

    def __init__(self, pk, dev, F_, H, W):
        self.rec = ops.Recorder(record=True)
        self.src = torch.zeros(F_, 3, H, W, device=dev, dtype=torch.float32)
        buf = lambda *s, dtype=BF16: torch.empty(*s, device=dev, dtype=dtype)
        self.out = _emit_encoder(self.rec, pk, self.src, buf, F_, H, W)[2]

    def run(self):
        self.rec.run()


class DecodeRunner:
    """Static buffers + launch list of the batched flow-warp / occlusion-blend decode of F = B*T frames."""

    def __init__(self, pk, dev, B, T, H, W, h, w, with_occ, n_bottleneck):
        self.rec = ops.Recorder(record=True)
        rec = self.rec
        Fn = B * T
        f32 = dict(device=dev, dtype=torch.float32)
        self.src = torch.zeros(B, 3, H, W, **f32)
        self.flow = torch.zeros(Fn, h, w, 2, **f32)
        self.occ = torch.zeros(Fn, 1, h, w, **f32) if with_occ else None
        self.prediction = torch.zeros(Fn, 3, H, W, **f32)
        self.deformed = torch.zeros(Fn, 3, H, W, **f32)
        if not with_occ:
            # generator.py:81-90 with occlusion_map=None: prediction == deformed source, decoder output unused
            ops.warp_image(rec, self.src, None, self.flow, None, self.prediction, self.deformed)
            return
        buf = lambda *s, dtype=BF16: torch.empty(*s, device=dev, dtype=dtype)
        v5 = lambda t: t.view(t.shape[0], 1, *t.shape[1:])
        # ---- encoder, once per video
        skip0, skip1, skip2 = _emit_encoder(rec, pk, self.src, buf, B, H, W)
        # ---- per-frame decode
        Hb, Wb = H // 4, W // 4
        out = buf(Fn, Hb, Wb, 256)
        ops.warp_blend_cl(rec, skip2, None, self.flow, self.occ, out)
        act, hid = buf(Fn, Hb, Wb, 256), buf(Fn, Hb, Wb, 256)
        for i in range(n_bottleneck):
            s1, t1, w1, b1, w2, b2 = pk[f"r{i}"]
            ops.bn_relu_cl(rec, out, s1, t1, act)
            ops.conv_cl(rec, v5(act), w1, 256, 3, v5(hid), bias=b1, act=1)
            nxt = buf(Fn, Hb, Wb, 256)
            ops.conv_cl(rec, v5(hid), w2, 256, 3, v5(nxt), bias=b2, res=v5(out))
            out = nxt
        u0 = buf(Fn, 2 * Hb, 2 * Wb, 256)
        ops.warp_blend_cl(rec, skip2, out, self.flow, self.occ, u0, up2=True)
        o0 = buf(Fn, 2 * Hb, 2 * Wb, 128)
        ops.conv_cl(rec, v5(u0), pk["up0"][0], 128, 3, v5(o0), bias=pk["up0"][1], act=1)
        u1 = buf(Fn, H, W, 128)
        ops.warp_blend_cl(rec, skip1, o0, self.flow, self.occ, u1, up2=True)
        o1 = buf(Fn, H, W, 64)
        ops.conv_cl(rec, v5(u1), pk["up1"][0], 64, 3, v5(o1), bias=pk["up1"][1], act=1)
        fin = buf(Fn, H, W, 64)
        ops.warp_blend_cl(rec, skip0, o1, self.flow, self.occ, fin)
        self.dec = buf(Fn, H, W, 4, dtype=torch.float32)
        ops.conv_cl(rec, v5(fin), pk["final"][0], 3, 7, v5(self.dec), bias=pk["final"][1], act=3, out_fp32=True)
        ops.warp_image(rec, self.src, self.dec, self.flow, self.occ, self.prediction, self.deformed)

    def run(self):
        self.rec.run()


# =============================================================================================== CUDA conditioning
_BG_TYPES = {"shift": 1, "affine": 2, "perspective": 3}


def _pad32(c):
    return (c + 31) // 32 * 32


class CondRunner:
    """The conditioning stage of FlowDiffusion.sample_one_video (VideoFlowDiffusion_multi_w_ref.py:231-262) for F = B*tc
    frames on the CUDA kernels: RegionPredictor -> BGMotionPredictor -> PixelwiseFlowPredictor.  The same stage serves
    stage-1 reconstruction (ReconRunner) with tc = T frames per video and the source at slot `src_slot` of each video.

    Convolutions run on the tcgen05 implicit GEMM in its tf32 mode (fp32 tensors, fp32 accumulate: the precision of the
    reference's cuDNN path), everything else on the fp32 kernels of csrc/lfae_cond.cu, including the PCA of the region
    covariances (region_predictor.py:130-136): `pca = "gesvdj"` evaluates the 2x2 SVD in closed form with the
    singular-vector signs of cuSOLVER's batched Jacobi -- what torch.svd, hence the reference, returns on a GPU -- so
    the whole stage is one launch list replayed from a CUDA graph.  `pca = "torch"` calls torch.svd between the two
    halves instead (the fixture tests route it through LAPACK, whose signs differ: DESIGN.md section 1).

    The reference evaluates the region predictor twice on each video's last conditioning frame (once as `ref_img`,
    once as driving frame tc-1, same weights, same input); here the source parameters are read from frame tc-1, or in
    general from the driving batch's copy of the source frame, slot `src_slot` (default tc - 1) of each video."""

    pca = "gesvdj"           # class-level switch, see above
    use_cuda_graph = True

    @staticmethod
    def supported(rp, bgp, pfp):
        return (rp.pca_based and rp.jacobian is None and rp.scale_factor == pfp.scale_factor
                and rp.scale_factor in (1, 0.5, 0.25) and pfp.use_deformed_source
                and rp.regions.kernel_size == (7, 7) and rp.regions.padding[0] <= 3)

    def __init__(self, rp, bgp, pfp, dev, B, tc, H, W, src_slot=None):
        self.src_slot = tc - 1 if src_slot is None else src_slot
        if not 0 <= self.src_slot < tc:
            raise ValueError(f"CondRunner: src_slot {self.src_slot} outside [0, {tc})")
        self.recA, self.recB = ops.Recorder(record=True), ops.Recorder(record=True)
        self.recP = ops.Recorder(record=True)                  # the closed-form PCA between the two halves
        self._graph = None
        f32 = dict(device=dev, dtype=torch.float32)
        buf = lambda *s: torch.empty(*s, **f32)
        Fn = B * tc
        self.frames = torch.zeros(Fn, 3, H, W, **f32)          # frame f = video f // tc, time f % tc
        self.ref = torch.zeros(B, 3, H, W, **f32)
        K = pfp.num_regions
        st = int(round(1 / rp.scale_factor))
        h, w = H // st, W // st
        kern = rp.down.weight[0, 0].to(**f32).contiguous() if rp.scale_factor != 1 else None
        # ---- region predictor
        xd = buf(Fn, h, w, 32)
        ops.image_to_cl(self.recA, self.frames, 1, xd, kern=kern, stride=st)
        feat, xin = self._hourglass(self.recA, rp.predictor, xd, 3, buf)
        be = feat.shape[-1]
        wr = ops.pack_conv_weight_f32(rp.regions.weight.detach().to(**f32), splits=[(0, be, be), (be, be + 3, 32)])
        logits = buf(Fn, h, w, 16 * ((K + 15) // 16))
        ops.conv_cl_tf32(self.recA, feat, wr, K, 7, logits, x2=xin, bias=rp.regions.bias.detach().to(**f32).contiguous(),
                         round_out=False)
        self.shift, self.covar = torch.zeros(Fn, K, 2, **f32), torch.zeros(Fn, K, 2, 2, **f32)
        self.affine = torch.zeros(Fn, K, 2, 2, **f32)
        ops.region_moments(self.recA, logits, K, 3 - rp.regions.padding[0], float(rp.temperature), self.shift, self.covar)
        ops.pca_affine(self.recP, self.covar, self.affine)
        # ---- background predictor (full resolution, [reference | frame] channels)
        rec = self.recB
        self.bg = None
        if bgp.bg_type != "zero":
            xb = buf(Fn, H, W, 32)
            ops.image_to_cl(rec, self.ref, tc, xb, b=self.frames, b_div=1)
            cur, ci, hh, ww = xb, 6, H, W
            for blk in bgp.encoder.down_blocks:
                cur = self._down(rec, blk, cur, ci, hh, ww, buf)
                ci, hh, ww = cur.shape[-1], hh // 2, ww // 2
            self.bg = torch.zeros(Fn, 3, 3, **f32)
            ops.bg_head(rec, cur, bgp.fc.weight.detach().to(**f32).contiguous(),
                        bgp.fc.bias.detach().to(**f32).contiguous(), _BG_TYPES[bgp.bg_type], self.bg)
        # ---- pixel-wise flow predictor
        cin = 4 * (K + 1)
        cpad = _pad32(cin)
        inp, self.motion = buf(Fn, h, w, cpad), buf(Fn, K + 1, h, w, 2)
        if self.src_slot == tc - 1:                             # the conditioning stage's own entry
            ops.sparse_motion(rec, xd, self.shift, self.covar, self.affine, self.bg, tc, pfp.revert_axis_swap,
                              pfp.use_covar_heatmap, float(pfp.region_var), inp, self.motion)
        else:
            ops.sparse_motion_src(rec, xd, self.shift, self.covar, self.affine, self.bg, tc, self.src_slot,
                                  pfp.revert_axis_swap, pfp.use_covar_heatmap, float(pfp.region_var), inp, self.motion)
        feat, xin = self._hourglass(rec, pfp.hourglass, inp, cin, buf)
        be = feat.shape[-1]
        heads = [pfp.mask] + ([pfp.occlusion] if pfp.occlusion is not None else [])
        wh = torch.cat([m.weight.detach().to(**f32) for m in heads], 0)
        bh = torch.cat([m.bias.detach().to(**f32) for m in heads], 0).contiguous()
        whp = ops.pack_conv_weight_f32(wh, splits=[(0, be, be), (be, be + cin, cpad)])
        head = buf(Fn, h, w, 16 * ((wh.shape[0] + 15) // 16))
        ops.conv_cl_tf32(rec, feat, whp, wh.shape[0], 7, head, x2=xin, bias=bh, round_out=False)
        self.grid = torch.zeros(B, 2, tc, h, w, **f32)
        self.conf = torch.zeros(B, 1, tc, h, w, **f32) if pfp.occlusion is not None else None
        ops.flow_compose(rec, head, self.motion, K, tc, self.grid, self.conf)

    @staticmethod
    def _folded(blk, dev):
        w, b = _fold_bn(blk.conv.weight, blk.conv.bias, blk.norm)
        return w.to(dev), b.to(dev).contiguous()

    def _down(self, rec, blk, x, cin_real, hh, ww, buf):
        """DownBlock2d: conv3x3 + BN(eval, folded) + ReLU + AvgPool2 (util.py:118-131)."""
        w, b = self._folded(blk, x.device)
        wp = ops.pack_conv_weight_f32(w, splits=[(0, cin_real, x.shape[-1])])
        y = buf(x.shape[0], hh, ww, w.shape[0])
        ops.conv_cl_tf32(rec, x, wp, w.shape[0], 3, y, bias=b, act=1)
        p = buf(x.shape[0], hh // 2, ww // 2, w.shape[0])
        ops.avgpool2_f32_cl(rec, y, p)
        return p

    def _hourglass(self, rec, hg, x, cin_real, buf):
        """Hourglass.forward (util.py:152-221) on x (F, h, w, pad32(cin)).  Returns the two channel groups of its
        output [last up-block (block_expansion) | x] un-concatenated: the consumer's convolution reads both."""
        Fn, hh, ww, _ = x.shape
        feats, cur, ci = [x], x, cin_real
        for blk in hg.encoder.down_blocks:
            cur = self._down(rec, blk, cur, ci, hh, ww, buf)
            feats.append(cur)
            ci, hh, ww = cur.shape[-1], hh // 2, ww // 2
        out, skip = feats.pop(), None
        for blk in hg.decoder.up_blocks:
            w, b = self._folded(blk, x.device)
            ua = buf(Fn, 2 * hh, 2 * ww, out.shape[-1])
            ops.upsample2_f32_cl(rec, out, ua)
            ub = None
            if skip is not None:
                ub = buf(Fn, 2 * hh, 2 * ww, skip.shape[-1])
                ops.upsample2_f32_cl(rec, skip, ub)
            hh, ww = 2 * hh, 2 * ww
            y = buf(Fn, hh, ww, w.shape[0])
            ops.conv_cl_tf32(rec, ua, ops.pack_conv_weight_f32(w), w.shape[0], 3, y, x2=ub, bias=b, act=1)
            out, skip = y, feats.pop()
        return out, skip

    def recorders(self):
        """The stage's launch lists, in execution order (bench.py / tools/kernel_table.py account for them)."""
        return [self.recA, self.recP, self.recB] if self.pca == "gesvdj" else [self.recA, self.recB]

    def stage(self, real_vid):
        """Copy real_vid (B, 3, tc, H, W) fp32 on the device into the static input buffers."""
        B, _, tc, H, W = real_vid.shape
        self.frames.view(B, tc, 3, H, W).copy_(real_vid.permute(0, 2, 1, 3, 4))
        self.ref.copy_(real_vid[:, :, self.src_slot])

    def launch(self):
        """Issue the stage on the current stream, without the graph."""
        if self.pca != "gesvdj":
            self.recA.run()
            u, s, _ = torch.svd(self.covar.view(-1, 2, 2))                 # region_predictor.py:130-136
            self.affine.view(-1, 2, 2).copy_(u @ torch.diag_embed(s ** 0.5))
            self.recB.run()
            return
        for rec in (self.recA, self.recP, self.recB):
            rec.run()

    def run(self, real_vid):
        """real_vid (B, 3, tc, H, W) fp32 on the device -> (grid (B,2,tc,h,w), conf (B,1,tc,h,w) | None)."""
        self.stage(real_vid)
        if self.pca != "gesvdj" or not self.use_cuda_graph or torch.cuda.is_current_stream_capturing():
            self.launch()
            return self.grid, self.conf
        if self._graph is None:                                # static buffers: the launch lists replay as one graph
            self._graph = _capture(self.launch)
        self._graph.replay()
        return self.grid, self.conf


def _capture(launch):
    """One CUDA graph of `launch` (a function that issues kernels on the current stream), after one eager warm-up run
    (lazy per-kernel attribute set-up)."""
    launch()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        launch()
    return g


class ReconRunner:
    """Stage-1 reconstruction (the LFAE forward of model/LFAE/generator.py:105-144, FlowAE.reconstruct) of B videos of T
    frames on the CUDA kernels: CondRunner with tc = T and the source at slot src_slot of each video, then the
    DecodeRunner of Generator.decode_video (encoder once per video, fused warp + blend, bf16 decoder).  Static buffers;
    with the closed-form PCA the whole thing replays as one CUDA graph with no host sync and no library call inside.
    `use_cuda_graph = False` (or CondRunner.pca = "torch") issues the same launch lists eagerly."""

    use_cuda_graph = True

    def __init__(self, gen, rp, bgp, dev, B, T, H, W, src_slot):
        pfp = gen.pixelwise_flow_predictor
        self.cond = CondRunner(rp, bgp, pfp, dev, B, T, H, W, src_slot=src_slot)
        h, w = self.cond.grid.shape[-2:]
        self.dec = gen.decoder(B, T, H, W, h, w, pfp.occlusion is not None)
        self.src_slot = src_slot
        self._graph = None

    def launch(self):
        c, d = self.cond, self.dec
        c.launch()
        # (B, 2, T, h, w) -> the decoder's (B*T, h, w, 2); the occlusion map has the same memory order in both
        d.flow.view(c.grid.shape[0], c.grid.shape[2], *d.flow.shape[1:]).copy_(c.grid.permute(0, 2, 3, 4, 1))
        if d.occ is not None:
            d.occ.view(c.conf.shape).copy_(c.conf)
        d.run()

    def run(self, real_vid):
        """real_vid (B, 3, T, H, W) fp32 on the device -> dict of (B, C, T, ...) tensors (views of the static buffers
        but optical_flow / occlusion_map, which are the CondRunner's)."""
        B, _, T, H, W = real_vid.shape
        self.cond.stage(real_vid)
        self.dec.src.copy_(real_vid[:, :, self.src_slot])
        if self.cond.pca != "gesvdj" or not self.use_cuda_graph or torch.cuda.is_current_stream_capturing():
            self.launch()
        else:
            if self._graph is None:
                self._graph = _capture(self.launch)
            self._graph.replay()
        per_video = lambda t: t.view(B, T, *t.shape[1:]).transpose(1, 2)
        out = {"prediction": per_video(self.dec.prediction), "deformed": per_video(self.dec.deformed),
               "optical_flow": self.cond.grid}
        if self.cond.conf is not None:
            out["occlusion_map"] = self.cond.conf
        return out
