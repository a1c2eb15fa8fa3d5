"""Unet3D: the ExtDM denoiser on hand-written sm_100a kernels.

Public surface mirrors the reference (model/BaseDM_adaptor/DenoiseNet_STWAtt_*.py): same constructor
arguments, same `forward(x, time, cond_frames, cond_fea, ...)`, same state_dict keys.  Internally the
forward is a *launch list* of C-ABI kernels (ops.Recorder) over channels-last bf16 buffers, split into
  * a prologue that only depends on the conditioning (cond_frames, cond_fea) -- cond_adaptor,
    cond_temporal_attn, the bilinear resize, the cond_fea half of init_conv and the conditioning frames of
    init_noise_conv / init_conv (SURVEY.md fact 7: exact up to fp re-association), run once per round, and
  * a step list run once per DDIM iteration; on the predicted frames init_conv(init_noise_conv(x)) is evaluated as one
    13x13 convolution of the flow plus a ring correction (UnetRunner._composite_init: exact, 4x fewer FLOPs).
No torch op touches activations; torch supplies memory, weights and the state_dict plumbing.
"""
import math

import torch
from torch import nn

from . import composite, ops
from .manifest import UNET_ARCHITECTURES, UnetConfig, is_int_key, unet_manifest
from .paramtree import ParamTree
from .weights import synth_state_dict

BF16 = torch.bfloat16


def _rope_tables(n, dh, device):
    """rotary-embedding-torch 0.8.3 angles (interleaved pairs): (n, dh/2) cos / sin, fp32."""
    freqs = 1.0 / (10000.0 ** (torch.arange(0, dh, 2, dtype=torch.float32)[: dh // 2] / dh))
    ang = torch.arange(n, dtype=torch.float32)[:, None] * freqs[None, :]
    return ang.cos().contiguous().to(device), ang.sin().contiguous().to(device)


def _t5_rel_bias(emb, T, num_buckets=32, max_distance=32):
    """RelativePositionBias (...cross_multi.py:43-80) folded to (heads, 2T-1), index (j - i) + T - 1."""
    rel = torch.arange(-(T - 1), T)            # j - i
    n = -rel
    nb = num_buckets // 2
    ret = (n < 0).long() * nb
    n = n.abs()
    max_exact = nb // 2
    large = max_exact + (torch.log(n.float().clamp(min=1) / max_exact) / math.log(max_distance / max_exact)
                         * (nb - max_exact)).long()
    large = torch.minimum(large, torch.full_like(large, nb - 1))
    bucket = ret + torch.where(n < max_exact, n, large)
    return emb.detach().float().cpu()[bucket].t().contiguous()     # (heads, 2T-1)


class PackedUnet:
    """Kernel-layout weights (bf16 K-major GEMM operands, fp32 vectors), built once per state_dict."""

    def __init__(self, sd, cfg, device):
        self.cfg = cfg
        self.dev = device
        self.f32, self.w = {}, {}
        for k in sd:
            if is_int_key(k) or k.endswith("rotary_emb.freqs"):
                continue
            t = sd[k].detach().to(device=device, dtype=torch.float32)
            if k in ("init_conv.weight", "init_noise_conv.weight") or k.startswith(("time_mlp.", "time_rel_pos_bias.")) \
                    or ".mlp.1." in k or k.endswith("relative_position_bias_table"):
                self.f32[k] = t.contiguous()
            elif k in ("final_conv.1.weight", "occlusion_map.1.weight"):
                self.f32[k] = t.reshape(t.shape[0], -1).contiguous()
            elif k.endswith((".bias", ".gamma", "norm.weight")):
                self.f32[k] = t.reshape(-1).contiguous()
            elif k.startswith("downs.") and k.endswith(f".{cfg.resample_slot}.weight"):
                self.w[k] = ops.pack_downsample_weight(t)
            elif k.startswith("ups.") and k.endswith(f".{cfg.resample_slot}.weight"):
                self.w[k] = ops.pack_upsample_weight_merged(t)
            elif t.dim() == 5 and t.shape[2] == 3:
                self.w[k] = ops.pack_conv3d_weight(t)
            elif t.dim() == 5:
                self.w[k] = ops.pack_conv_weight(t)
            else:
                self.w[k] = ops.pack_linear_weight(t)
        # 7x7 convs on the 3-channel flow volume run as im2col GEMMs with K = 147 -> 192
        def pack7(w3):                                    # (N, 3, 1, 7, 7) -> (N, 192) bf16
            n = w3.shape[0]
            out = torch.zeros(n, 192, device=device, dtype=BF16)
            out[:, :147] = w3[:, :, 0].permute(0, 2, 3, 1).reshape(n, 147).to(BF16)
            return out
        ic = self.f32["init_conv.weight"]
        if cfg.variant in ("base", "u22"):
            self.w["init_flow"] = pack7(ic[:, :3])
            self.w["init_fea"] = ops.pack_conv_weight(ic[:, 3:])
        elif cfg.variant == "u12":
            # TrajWarp makes the cond_fea half of init_conv depend on x_t: nothing to hoist, one conv over 512 channels
            self.w["init_noise"] = pack7(self.f32["init_noise_conv.weight"])
            self.w["init_full"] = ops.pack_conv_weight(ic)
            self.w["init_fea"] = ops.pack_conv_weight(ic[:, 256:])
            self._pack_composite_init(ic[:, :256, 0])
            # the cond_fea half acts on a x2 bilinearly up-sampled tensor: 5x5 polyphase kernels on the low-resolution
            # tensor + 1-D border corrections (composite.compose_upsampled, UnetRunner._polyphase_fea)
            c2 = composite.compose_upsampled(ic[:, 256:, 0])
            co = ic.shape[0]
            self.w["init_poly"] = [c2["poly"][i].reshape(co, 25 * 256).to(BF16).contiguous() for i in range(4)]
            for side in ("top", "bottom", "left", "right"):
                self.w["init_fea_" + side] = c2[side].reshape(3 * co, 7 * 256).to(BF16).contiguous()
        else:
            self.w["init_noise"] = pack7(self.f32["init_noise_conv.weight"])
            self.w["init_x"] = ops.pack_conv_weight(ic[:, :256])
            self.w["init_fea"] = ops.pack_conv_weight(ic[:, 256:])
            self._pack_composite_init(ic[:, :256, 0])
        # all ResnetBlock time-MLPs stacked: one GEMV kernel produces every (scale, shift)
        rows, biases, self.ss_off = [], [], {}
        off = 0
        for k in sorted(sd):
            if k.endswith(".mlp.1.weight"):
                p = k[: -len(".mlp.1.weight")]
                self.ss_off[p] = off
                rows.append(self.f32[k])
                biases.append(self.f32[p + ".mlp.1.bias"])
                off += rows[-1].shape[0]
        self.wss = torch.cat(rows, 0).contiguous()
        self.bss = torch.cat(biases, 0).contiguous()
        self.n_ss = off
        self.rel_bias = _t5_rel_bias(sd["time_rel_pos_bias.relative_attention_bias.weight"], cfg.T).to(device)
        self.rope_t = _rope_tables(32, cfg.dim_head, device)
        wd, wh, ww = cfg.window
        self.rope_w = _rope_tables(wd * wh * ww, cfg.dim_head, device)


    def _pack_composite_init(self, w2):
        """Weight blocks of the composite init_conv (composite.compose: the 13x13 kernel w2 * w1 over the flow, the four
        ring sides as GEMM phases, the corner table), cast to the kernels' dtypes / layouts -- UnetRunner._composite_init."""
        c = composite.compose(self.f32["init_noise_conv.weight"][:, :, 0], self.f32["init_noise_conv.bias"], w2)
        co = w2.shape[0]
        self.w["init_comp"] = c["comp"].reshape(co, 13 * 64).to(BF16).contiguous()
        self.f32["init_comp.bias"] = c["comp_bias"].float().contiguous()
        for side in ("top", "bottom", "left", "right"):            # phases stacked along the rows: (3 * Cout, taps * 64)
            self.w["init_ring_" + side] = c[side].reshape(3 * co, -1).to(BF16).contiguous()
        self.f32["init_ring_corners"] = c["corners"].float().contiguous()


class UnetRunner:
    """Launch lists + static buffers for one (config, batch, resolution)."""

    fuse_stw = True          # class-level switch (tests compare the fused and the un-fused STW paths)
    # ResnetBlock's last GroupNorm applied inside the following attention kernel (extdm_stw_fused_pre).  Parity green but
    # no faster on B200 (800 vs 716 + 98 us per level-0 pair: the attention kernel is compute bound and the extra
    # element-wise work lands on its critical path), so it is off by default.
    fuse_gn_stw = False
    # dim_head 32 (u12 / base / ada_u22): the fused temporal layer runs on the tcgen05 kernel of csrc/attn_ws32.cu
    # (16-token packing for T <= 16: eight pixel sequences per M = 128 tile).  The earlier mma.sync edition
    # (EXTDM_ATTN32_LEGACY=1) padded T = 12 ... 15 to 32 tokens and lost to the un-fused path.
    fuse_temporal_dh32 = True
    # init_conv(init_noise_conv(x)) on the predicted frames as one composite 13x13 convolution of the 3-channel flow plus a
    # ring correction (_composite_init) instead of a 7x7 convolution over 256 channels (K = 12544) per DDIM step
    composite_init = True
    # u12: the cond_fea half of init_conv (7x7 over the x2 up-sampled TrajWarp features) as 5x5 polyphase convolutions of the
    # low-resolution features + 1-D border corrections (_polyphase_fea); needs composite_init
    polyphase_fea = True

    def __init__(self, packed, B, H=32, W=32, fea_hw=16):
        cfg = packed.cfg
        self.pk, self.cfg, self.B, self.H, self.W = packed, cfg, B, H, W
        dev = packed.dev
        self.dev = dev
        T, tc, tp, tm = cfg.T, cfg.tc, cfg.tp, cfg.tm
        f32 = dict(device=dev, dtype=torch.float32)
        self.x = torch.zeros(B, 3, tp, H, W, **f32)
        self.cond_frames = torch.zeros(B, 3, tc, H, W, **f32)
        self.cond_fea = torch.zeros(B, 256, T, fea_hw, fea_hw, **f32)
        self.time = torch.zeros(B, dtype=torch.long, device=dev)
        self.out = torch.zeros(B, 3, tp, H, W, **f32)
        self.gn_ws = torch.zeros(B * max(32, ops.gn_parts_per_sample(T, H, W, 64)) * cfg.groups * 2, **f32)
        self.ss = torch.zeros(B, packed.n_ss, **f32)
        self.prologue = ops.Recorder(record=True)
        self.step = ops.Recorder(record=True)
        # time embedding + the 20 per-block (scale, shift) MLPs: depends on the timestep and the weights only, so the
        # sampler evaluates it once per schedule (ss_for_times) instead of once per DDIM step and round
        self.time_rec = ops.Recorder(record=True)
        self._ss_tables = {}
        self._ss_rows = {}
        self.taps = {}                      # name -> buffer, for layer-by-layer parity tests
        self.graphs = {}                    # key -> (CUDA graph, state) over these buffers (GaussianDiffusion._graph)
        self._build()

    # ------------------------------------------------------------------ helpers
    def buf(self, *shape, dtype=BF16):
        return torch.empty(*shape, device=self.dev, dtype=dtype)

    def _temporal(self, rec, x, p):
        cfg, pk = self.cfg, self.pk
        B, T, H, W, C = x.shape
        if self.fuse_stw and ops.temporal_fused_supported(C, cfg.heads, cfg.dim_head, T) and \
                (cfg.dim_head == 16 or self.fuse_temporal_dh32):
            y = self.buf(B, T, H, W, C)
            ops.temporal_fused(rec, x, y, pk.f32[p + ".fn.norm.gamma"], pk.f32[p + ".fn.fn.fn.norm.weight"],
                               pk.f32[p + ".fn.fn.fn.norm.bias"], pk.w[p + ".fn.fn.fn.attn.to_qkv.weight"],
                               pk.w[p + ".fn.fn.fn.attn.to_out.weight"], pk.rel_bias, pk.rope_t[0], pk.rope_t[1],
                               cfg.heads, cfg.dim_head)
            return y
        u, xz = self.buf(B, T, H, W, C), self.buf(B, T, H, W, C)
        ops.temporal_prenorm(rec, x, pk.f32[p + ".fn.norm.gamma"], pk.f32[p + ".fn.fn.fn.norm.weight"],
                             pk.f32[p + ".fn.fn.fn.norm.bias"], u, xz)
        qkv = self.buf(B, T, H, W, 3 * cfg.hidden)
        ops.linear_rows(rec, u, pk.w[p + ".fn.fn.fn.attn.to_qkv.weight"], 3 * cfg.hidden, qkv)
        o = self.buf(B, T, H, W, cfg.hidden)
        ops.temporal_attention(rec, qkv, o, pk.rel_bias, pk.rope_t[0], pk.rope_t[1], cfg.heads, cfg.dim_head)
        y = self.buf(B, T, H, W, C)
        ops.linear_rows(rec, o, pk.w[p + ".fn.fn.fn.attn.to_out.weight"], C, y, res=xz)
        return y

    def _window_shift(self, T, H, W, shifted):
        """get_window_size (...cross_multi.py:393-406): a dim no larger than its window is not shifted."""
        cfg = self.cfg
        window, shift = list(cfg.window), list(cfg.shift if shifted else (0, 0, 0))
        for i, size in enumerate((T, H, W)):
            if size <= window[i]:
                if size != window[i]:
                    raise NotImplementedError(f"window {cfg.window} larger than the volume {(T, H, W)}")
                shift[i] = 0
        return window, shift

    def _res_stw(self, rec, x, pres, pstw, cout, shifted, x2=None):
        """ResnetBlock followed by its STW attention layer.  Where the 16-warp fused attention kernel applies, the
        block's last GroupNorm + SiLU + residual are applied by that kernel on load (no stand-alone apply pass)."""
        cfg, pk = self.cfg, self.pk
        B, T, H, W, _ = x.shape
        window, shift = self._window_shift(T, H, W, shifted)
        if self.fuse_stw and self.fuse_gn_stw and cfg.groups == 8 and \
                ops.stw_fused_pre_supported(cout, cfg.heads, cfg.dim_head, window):
            h2, r, gnp, npart = self._resblock(rec, x, pres, cout, x2=x2, defer_norm2="shared")
            ad = self.buf(B, 2, cout, dtype=torch.float32)
            ops.groupnorm_affine(rec, gnp, npart, pk.f32[pres + ".block2.norm.weight"],
                                 pk.f32[pres + ".block2.norm.bias"], ad, T * H * W, cout)
            y = self.buf(B, T, H, W, cout)
            ops.stw_fused_pre(rec, h2, r, ad, y, pk.f32[pstw + ".fn.norm.gamma"], pk.w[pstw + ".fn.fn.attn.qkv.weight"],
                              pk.w[pstw + ".fn.fn.attn.proj.weight"], pk.f32[pstw + ".fn.fn.attn.proj.bias"],
                              pk.f32[pstw + ".fn.fn.attn.relative_position_bias_table"], pk.rope_w[0], pk.rope_w[1],
                              cfg.heads, cfg.dim_head, window, shift)
            self.taps[pstw] = y
            return y
        x = self._resblock(rec, x, pres, cout, x2=x2)
        self.taps[pres] = x
        x = self._stw(rec, x, pstw, shifted)
        self.taps[pstw] = x
        return x

    def _stw(self, rec, x, p, shifted):
        cfg, pk = self.cfg, self.pk
        B, T, H, W, C = x.shape
        window, shift = self._window_shift(T, H, W, shifted)
        if self.fuse_stw and ops.stw_fused_supported(C, cfg.heads, cfg.dim_head, window):
            y = self.buf(B, T, H, W, C)
            ops.stw_fused(rec, x, y, pk.f32[p + ".fn.norm.gamma"], pk.w[p + ".fn.fn.attn.qkv.weight"],
                          pk.w[p + ".fn.fn.attn.proj.weight"], pk.f32[p + ".fn.fn.attn.proj.bias"],
                          pk.f32[p + ".fn.fn.attn.relative_position_bias_table"], pk.rope_w[0], pk.rope_w[1],
                          cfg.heads, cfg.dim_head, window, shift)
            return y
        z = self.buf(B, T, H, W, C)
        ops.chan_layernorm(rec, x, pk.f32[p + ".fn.norm.gamma"], z)
        qkv = self.buf(B, T, H, W, 3 * cfg.hidden)
        ops.linear_rows(rec, z, pk.w[p + ".fn.fn.attn.qkv.weight"], 3 * cfg.hidden, qkv)
        o = self.buf(B, T, H, W, cfg.hidden)
        ops.window_attention(rec, qkv, o, pk.f32[p + ".fn.fn.attn.relative_position_bias_table"], pk.rope_w[0],
                             pk.rope_w[1], cfg.heads, cfg.dim_head, window, shift)
        y = self.buf(B, T, H, W, C)
        ops.linear_rows(rec, o, pk.w[p + ".fn.fn.attn.proj.weight"], C, y, bias=pk.f32[p + ".fn.fn.attn.proj.bias"],
                        res=x)
        return y

    def _resblock(self, rec, x, p, cout, x2=None, time=True, defer_norm2=False):
        """defer_norm2: stop after block2's convolution and return (h2, residual, gn partial workspace, n_part) --
        the caller fuses the last GroupNorm + SiLU + residual into its own kernel."""
        cfg, pk = self.cfg, self.pk
        B, T, H, W, _ = x.shape
        h1 = self.buf(B, T, H, W, cout)
        # GroupNorm statistics come out of the convolution's epilogue (per-tile partial sums), not a second pass
        fused = cfg.groups == 8 and cout in (64, 128, 256, 512)
        npart = ops.gn_parts_per_sample(T, H, W, cout) if fused else None
        gnp = self.gn_ws if fused else None
        ops.conv_cl(rec, x, pk.w[p + ".block1.proj.weight"], cout, 3, h1, x2=x2, bias=pk.f32[p + ".block1.proj.bias"],
                    gn_partials=gnp)
        ops.groupnorm_silu(rec, h1, self.gn_ws, pk.f32[p + ".block1.norm.weight"], pk.f32[p + ".block1.norm.bias"], h1,
                           groups=cfg.groups, scale_shift=self.ss if time else None,
                           ss_off=pk.ss_off[p] if time else 0, n_part=npart)
        h2 = self.buf(B, T, H, W, cout)
        if defer_norm2:
            if not fused:
                raise NotImplementedError("deferred GroupNorm needs the fused-statistics convolution")
            if defer_norm2 != "shared":                   # own workspace: it must survive until the consumer runs
                gnp = torch.zeros_like(self.gn_ws)
        ops.conv_cl(rec, h1, pk.w[p + ".block2.proj.weight"], cout, 3, h2, bias=pk.f32[p + ".block2.proj.bias"],
                    gn_partials=gnp)
        if (p + ".res_conv.weight") in pk.w:
            r = self.buf(B, T, H, W, cout)
            ops.conv_cl(rec, x, pk.w[p + ".res_conv.weight"], cout, 1, r, x2=x2, bias=pk.f32[p + ".res_conv.bias"])
        else:
            r = x
        if defer_norm2:
            return h2, r, gnp, npart
        # in place: h2 has no other reader, and a line rewritten while it is still dirty in L2 is written back once
        ops.groupnorm_silu(rec, h2, self.gn_ws, pk.f32[p + ".block2.norm.weight"], pk.f32[p + ".block2.norm.bias"], h2,
                           groups=cfg.groups, res=r, n_part=npart)
        return h2

    def _adaptor(self, rec, x, p):
        """MotionAdaptor, in place on frames [tm, T) of x (..._traj_ada.py:659-718)."""
        cfg, pk = self.cfg, self.pk
        B, T, H, W, C = x.shape
        tm, tp, L, nf = cfg.tm, cfg.tp, cfg.L, cfg.n_extra
        hw = H * W
        Te = tm * 2 ** L
        E = self.buf(B, Te, H, W, C)
        ln = self.buf(B, tm, H, W, C)
        ops.chan_layernorm(rec, x, pk.f32[p + ".adaptors.predictor.fn.norm.gamma"], ln, t_range=(0, tm))
        ops.conv_cl(rec, ln, pk.w[p + ".adaptors.predictor.fn.fn.weight"], C, 1, E,
                    bias=pk.f32[p + ".adaptors.predictor.fn.fn.bias"], res=x)
        ws = ops.adaptor_workspace(B, C, self.dev)
        for i in range(L):
            n_i = tm * 2 ** i
            nh = self.buf(B, n_i, H, W, C)
            ms = self.buf(2, B, C, dtype=torch.float32)
            ops.adaptor_normalize(rec, E, n_i, nh, ms, ws)
            # ada_u22's extrapolators are 3x3x3 (zero padding along T as well): 27 taps, the frame offsets are
            # coordinate offsets of the same TMA loads and out-of-range frames read as zeros
            ops.conv_cl(rec, nh, pk.w[p + f".adaptors.extrapolators.{i}.fn.weight"], C, 3, E, out_t_offset=n_i,
                        res=nh, col_scale=ms[1], col_shift=ms[0],
                        taps=ops.conv3d_taps(3) if cfg.extrap_kt == 3 else None)
        m1 = self.buf(B, tp, H, W, C)
        if hw >= 128:
            box, cnt = (128, 1, 1, 1), (hw, 1, 1, B)
        else:
            box, cnt = (hw, 1, 1, 128 // hw), (hw, 1, 1, B)
        ops.gemm(rec, a0=E, c0=C, dims=(hw, 1, Te, B), strides0=(C, hw * C, hw * C, Te * hw * C), box=box,
                 start=(0, 0, 0, 0), count=cnt, taps=[(0, 0, tm + t) for t in range(nf)],
                 w=pk.w[p + ".Tmodulator.weight"], n=tp * C, out=m1, out_stride=(C, 0, 0, tp * hw * C),
                 col_group=C, col_group_stride=hw * C, bias=pk.f32[p + ".Tmodulator.bias"])
        ln2 = self.buf(B, tp, H, W, 2 * C)
        ops.chan_layernorm(rec, m1, pk.f32[p + ".fuser.norm.gamma"], ln2, x2=x, t2_range=(tm, T))
        ops.conv_cl(rec, ln2, pk.w[p + ".fuser.fn.weight"], C, 1, x, bias=pk.f32[p + ".fuser.fn.bias"],
                    out_t_offset=tm, res=x, res_t_offset=tm)
        return x

    def _downsample(self, rec, x, p):
        pk = self.pk
        B, T, H, W, C = x.shape
        Ho, Wo = H // 2, W // 2
        z = self.buf(B, T, Ho + 1, Wo + 1, 4 * C)
        ops.space_to_depth(rec, x, z)
        y = self.buf(B, T, Ho, Wo, C)
        bw, bh, bt = ops.std_box(Ho, Wo)
        ops.gemm(rec, a0=z, c0=4 * C, dims=(Wo + 1, Ho + 1, T, B),
                 strides0=(4 * C, (Wo + 1) * 4 * C, (Ho + 1) * (Wo + 1) * 4 * C, T * (Ho + 1) * (Wo + 1) * 4 * C),
                 box=(bw, bh, bt, 1), start=(0, 0, 0, 0), count=(Wo, Ho, T, B),
                 taps=[(0, 0, 0), (1, 0, 0), (0, 1, 0), (1, 1, 0)], w=pk.w[p + ".weight"], n=C, out=y,
                 out_stride=(C, Wo * C, Ho * Wo * C, T * Ho * Wo * C), bias=pk.f32[p + ".bias"])
        return y

    def _upsample(self, rec, x, p):
        pk = self.pk
        B, T, H, W, C = x.shape
        y = self.buf(B, T, 2 * H, 2 * W, C)
        ops.upsample_cl(rec, x, pk.w[p + ".weight"], C, y, bias=pk.f32[p + ".bias"])     # four phases, one launch
        return y

    def _stage_u22(self, rec, x, p, cout, has_adaptor, x2=None):
        """..._traj_ada_u22.py:1268-1279: block1, block2, STW (shifted), STW, adaptor, temporal attention."""
        x = self._resblock(rec, x, p + ".0", cout, x2=x2)
        self.taps[p + ".0"] = x
        x = self._resblock(rec, x, p + ".2", cout)
        self.taps[p + ".2"] = x
        x = self._stw(rec, x, p + ".1", True)
        self.taps[p + ".1"] = x
        x = self._stw(rec, x, p + ".3", False)
        self.taps[p + ".3"] = x
        if has_adaptor:
            x = self._adaptor(rec, x, p + ".4")
            self.taps[p + ".4"] = x
        x = self._temporal(rec, x, p + ".5")
        self.taps[p + ".5"] = x
        return x

    def _stage(self, rec, x, p, cout, has_adaptor, x2=None):
        if self.cfg.variant == "u22":
            return self._stage_u22(rec, x, p, cout, has_adaptor, x2=x2)
        x = self._res_stw(rec, x, p + ".0", p + ".1", cout, True, x2=x2)
        x = self._res_stw(rec, x, p + ".2", p + ".3", cout, False)
        if has_adaptor:
            x = self._adaptor(rec, x, p + ".4")
            self.taps[p + ".4"] = x
        return x

    # ------------------------------------------------------------------ launch lists
    def _build(self):
        cfg, pk, B, H, W = self.cfg, self.pk, self.B, self.H, self.W
        T, tc, tp, tm = cfg.T, cfg.tc, cfg.tp, cfg.tm
        hw = H * W
        pro, st = self.prologue, self.step
        d = cfg.dim

        # ---- conditioning features -> flow resolution, channels-last (prologue)
        fh = self.cond_fea.shape[-1]
        cf = self.buf(B, T, fh, fh, 256)
        ops.ncthw_to_cl(pro, self.cond_fea, cf)
        if cfg.variant == "u12":
            return self._build_u12_front(cf)
        if cfg.variant in ("ada", "u22"):
            cf = self._adaptor(pro, cf, "cond_adaptor")
            cf = self._temporal(pro, cf, "cond_temporal_attn")
        if fh != H:
            cfu = self.buf(B, T, H, W, 256)
            ops.bilinear_resize_cl(pro, cf, cfu)
        else:
            cfu = cf
        self.taps["cond_up"] = cfu
        h0 = self.buf(B, T, H, W, d, dtype=torch.float32)           # cond_fea half of init_conv (+ bias), fp32
        ops.conv_cl(pro, cfu, pk.w["init_fea"], d, 7, h0, bias=pk.f32["init_conv.bias"], out_fp32=True)

        x0 = self.buf(B, T, H, W, d)
        a_c = self.buf(B * tm * hw, 192)
        a_p = self.buf(B * tp * hw, 192)
        if cfg.variant in ("base", "u22"):
            # init_conv on [flow(3) | cond_fea(256)] channels = im2col GEMM on the flow part + hoisted h0
            ops.im2col7_flow(pro, self.cond_frames, self.x, a_c, 0, tm)
            self._im2col_gemm(pro, a_c, pk.w["init_flow"], d, x0, 0, tm, res=h0)
            ops.im2col7_flow(st, self.cond_frames, self.x, a_p, tc, tp)
            self._im2col_gemm(st, a_p, pk.w["init_flow"], d, x0, tm, tp, res=h0)
        else:
            xn = self.buf(B, T, H, W, 256)
            nb = pk.f32["init_noise_conv.bias"]
            ops.im2col7_flow(pro, self.cond_frames, self.x, a_c, 0, tc)
            self._im2col_gemm(pro, a_c, pk.w["init_noise"], 256, xn, 0, tc, bias=nb)
            ops.conv_cl(pro, xn, pk.w["init_x"], d, 7, x0, t_range=(0, tc), res=h0, res_fp32=True)
            if self.composite_init and H == 32 and W == 32:
                self._composite_init(st, x0, res=h0, res_fp32=True, bias=pk.f32["init_comp.bias"])
            else:
                ops.im2col7_flow(st, self.cond_frames, self.x, a_p, tc, tp)
                self._im2col_gemm(st, a_p, pk.w["init_noise"], 256, xn, tc, tp, bias=nb)
                ops.conv_cl(st, xn, pk.w["init_x"], d, 7, x0, t_range=(tc, T), res=h0, res_fp32=True)
                self.taps["init_noise_conv"] = xn
        self.taps["init_conv"] = x0

        self._build_body(x0)

    def _build_u12_front(self, cf):
        """BAIR variant (..._traj_u12.py:1017-1042): init_noise_conv -> TrajWarp (cross attention of the future
        frames' pooled features over the conditioning frames' cond_fea) -> bilinear resize -> init_conv over
        [x | cond_fea].  Hoisted to the prologue: K / V projections, and everything on the tc conditioning frames."""
        cfg, pk, B, H, W = self.cfg, self.pk, self.B, self.H, self.W
        T, tc, tp = cfg.T, cfg.tc, cfg.tp
        hw = H * W
        pro, st = self.prologue, self.step
        d = cfg.dim
        fh = cf.shape[2]
        if H != 2 * fh or W != 2 * fh:
            raise NotImplementedError("TrajWarp needs cond_fea at half the flow resolution (MaxPool (1,2,2))")
        ca = "init_traj.cross_att."
        kk, vv = self.buf(B, tc, fh, fh, 256), self.buf(B, tc, fh, fh, 256)
        ops.conv_cl(pro, cf, pk.w[ca + "linear_k.weight"], 256, 1, kk, bias=pk.f32[ca + "linear_k.bias"], act=1,
                    t_range=(0, tc))
        ops.conv_cl(pro, cf, pk.w[ca + "linear_v.weight"], 256, 1, vv, bias=pk.f32[ca + "linear_v.bias"], act=1,
                    t_range=(0, tc))
        cfu = self.buf(B, T, H, W, 256)
        ops.bilinear_resize_frames_cl(pro, cf, cfu, (0, tc), 0)
        xn = self.buf(B, T, H, W, 256)
        x0 = self.buf(B, T, H, W, d)
        a_c, a_p = self.buf(B * tc * hw, 192), self.buf(B * tp * hw, 192)
        nb = pk.f32["init_noise_conv.bias"]
        ops.im2col7_flow(pro, self.cond_frames, self.x, a_c, 0, tc)
        self._im2col_gemm(pro, a_c, pk.w["init_noise"], 256, xn, 0, tc, bias=nb)
        ops.conv_cl(pro, xn, pk.w["init_full"], d, 7, x0, x2=cfu, t_range=(0, tc), bias=pk.f32["init_conv.bias"])
        # ---- per DDIM step
        ops.im2col7_flow(st, self.cond_frames, self.x, a_p, tc, tp)
        self._im2col_gemm(st, a_p, pk.w["init_noise"], 256, xn, tc, tp, bias=nb)
        self.taps["init_noise_conv"] = xn
        xp = self.buf(B, tp, fh, fh, 256)
        ops.maxpool2_frames_cl(st, xn, xp, (tc, T))
        qq = self.buf(B, tp, fh, fh, 256)
        ops.linear_rows(st, xp, pk.w[ca + "linear_q.weight"], 256, qq, bias=pk.f32[ca + "linear_q.bias"], act=1)
        ao = self.buf(B, tp * fh * fh, 256)
        ops.cross_attention(st, qq.view(B, -1, 256), kk.view(B, -1, 256), vv.view(B, -1, 256), ao, 8)
        yo = self.buf(B, tp, fh, fh, 256)
        ops.linear_rows(st, ao, pk.w[ca + "linear_o.weight"], 256, yo, bias=pk.f32[ca + "linear_o.bias"], act=1)
        if self.composite_init and self.polyphase_fea and H == 32 and W == 32:
            fpad = torch.zeros(B, tp, fh + 4, fh + 4, 256, device=self.dev, dtype=BF16)
            ops.conv_cl(st, cf, pk.w["init_traj.fuser.weight"], 256, 1, fpad, x2=yo, x2_t_offset=tc, t_range=(tc, T),
                        out_t_offset=-tc, bias=pk.f32["init_traj.fuser.bias"], out_pixel_offset=(2, 2))
            self._polyphase_fea(st, fpad, x0)
            self._composite_init(st, x0, res=x0, res_fp32=False, bias=pk.f32["init_comp.bias"])
            self.taps["init_conv"] = x0
            self._build_body(x0)
            return
        fpn = self.buf(B, tp, fh, fh, 256)
        ops.conv_cl(st, cf, pk.w["init_traj.fuser.weight"], 256, 1, fpn, x2=yo, x2_t_offset=tc, t_range=(tc, T),
                    out_t_offset=-tc, bias=pk.f32["init_traj.fuser.bias"])
        ops.bilinear_resize_frames_cl(st, fpn, cfu, (0, tp), tc)
        self.taps["cond_up"] = cfu
        if self.composite_init and H == 32 and W == 32:
            # the cond_fea half stays a 7x7 convolution (it depends on x_t through TrajWarp); the x half is composed
            ops.conv_cl(st, cfu, pk.w["init_fea"], d, 7, x0, t_range=(tc, T), bias=pk.f32["init_conv.bias"])
            self._composite_init(st, x0, res=x0, res_fp32=False, bias=pk.f32["init_comp.bias"])
        else:
            ops.conv_cl(st, xn, pk.w["init_full"], d, 7, x0, x2=cfu, t_range=(tc, T), bias=pk.f32["init_conv.bias"])
        self.taps["init_conv"] = x0
        self._build_body(x0)

    def _build_body(self, x0):
        cfg, pk, B, H, W = self.cfg, self.pk, self.B, self.H, self.W
        T, tc, tp, tm = cfg.T, cfg.tc, cfg.tp, cfg.tm
        st = self.step
        d = cfg.dim
        x = self._temporal(st, x0, "init_temporal_attn")
        self.taps["init_temporal_attn"] = x
        ops.time_mlp(self.time_rec, self.time, pk.f32["time_mlp.1.weight"], pk.f32["time_mlp.1.bias"],
                     pk.f32["time_mlp.3.weight"], pk.f32["time_mlp.3.bias"], pk.wss, pk.bss, self.ss, d)

        levels = cfg.levels
        nres = len(levels)
        skips = []
        u22, rs = cfg.variant == "u22", cfg.resample_slot
        for i, co in enumerate(levels):
            p = f"downs.{i}"
            x = self._stage(st, x, p, co, i > 1 or u22)
            skips.append(x)
            if i < nres - 1:
                x = self._downsample(st, x, f"{p}.{rs}")
                self.taps[f"{p}.{rs}"] = x
        mid = levels[-1]
        x = self._resblock(st, x, "mid_block1", mid)
        x = self._stw(st, x, "mid_attn1", True)
        if u22:                                            # ..._traj_ada_u22.py:1283-1287
            x = self._stw(st, x, "mid_attn2", False)
            x = self._adaptor(st, x, "mid_adaptor")
            x = self._resblock(st, x, "mid_block2", mid)
        else:
            x = self._resblock(st, x, "mid_block2", mid)
            x = self._stw(st, x, "mid_attn2", False)
            x = self._adaptor(st, x, "mid_adaptor")
        self.taps["mid"] = x
        dims = [d] + levels
        in_out = list(zip(dims[:-1], dims[1:]))
        for i, (ci, co) in enumerate(reversed(in_out)):
            p = f"ups.{i}"
            x = self._stage(st, x, p, ci, i > 1, x2=skips.pop())
            if i < nres - 1:
                x = self._upsample(st, x, f"{p}.{rs}")
                self.taps[f"{p}.{rs}"] = x
        if cfg.groups == 8 and d in (64, 128, 256):
            # the heads' last GroupNorm + SiLU + residual run inside the projection kernel, on the tp frames only
            h2f, rf, pf, npart = self._resblock(st, x, "final_conv.0", d, x2=x0, time=False, defer_norm2=True)
            h2o, ro, po, _ = self._resblock(st, x, "occlusion_map.0", d, x2=x0, time=False, defer_norm2=True)
            ops.head_project_gn(st, h2f, rf, pf, pk.f32["final_conv.0.block2.norm.weight"],
                                pk.f32["final_conv.0.block2.norm.bias"], h2o, ro, po,
                                pk.f32["occlusion_map.0.block2.norm.weight"],
                                pk.f32["occlusion_map.0.block2.norm.bias"], npart, pk.f32["final_conv.1.weight"],
                                pk.f32["final_conv.1.bias"], pk.f32["occlusion_map.1.weight"],
                                pk.f32["occlusion_map.1.bias"], self.out, tm)
            return
        hf = self._resblock(st, x, "final_conv.0", d, x2=x0, time=False)
        ho = self._resblock(st, x, "occlusion_map.0", d, x2=x0, time=False)
        ops.head_project(st, hf, ho, pk.f32["final_conv.1.weight"], pk.f32["final_conv.1.bias"],
                         pk.f32["occlusion_map.1.weight"], pk.f32["occlusion_map.1.bias"], self.out, tm)

    def _polyphase_fea(self, rec, fpad, x0):
        """frames [tc, T) of x0 = init_conv's cond_fea half over up2(f) + bias, computed on the low-resolution f (interior
        of fpad (B, tp, h + 4, w + 4, 256), ..._traj_u12.py:1039-1042): per output parity a 5x5 convolution of the
        replicate-padded f (25 instead of 49 taps per output pixel), then the zero padding of the 7x7 window at the image
        border: outside the image the replicate-extended up-sampled tensor repeats its border rows / columns, so each side
        is a 3-phase GEMM of 7 taps over one row / column (composite.compose_upsampled)."""
        cfg, pk, B, H, W = self.cfg, self.pk, self.B, self.H, self.W
        T, tc, tp = cfg.T, cfg.tc, cfg.tp
        d, hw = cfg.dim, H * W
        hp, h = fpad.shape[2], fpad.shape[2] - 4
        top, bottom = self.buf(B, tp, W + 6, 256), self.buf(B, tp, W + 6, 256)
        left, right = self.buf(B, tp, H, 256), self.buf(B, tp, H, 256)
        ops.upsample2_border(rec, fpad, top, bottom, left, right)
        base = tc * hw * d
        for py in range(2):
            for px in range(2):
                ops.gemm(rec, a0=fpad, c0=256, dims=(hp, hp, tp, B), strides0=(256, hp * 256, hp * hp * 256, tp * hp * hp * 256),
                         box=(16, 8, 1, 1), start=(2, 2, 0, 0), count=(h, h, tp, B), taps=ops.conv_taps(5),
                         w=pk.w["init_poly"][py * 2 + px], n=d, out=x0, out_stride=(2 * d, 2 * W * d, hw * d, T * hw * d),
                         out_base=base - 4 * d - 4 * W * d + (py * W + px) * d, bias=pk.f32["init_conv.bias"])
        ostr = (d, W * d, hw * d, T * hw * d)
        for side, a, y0 in (("top", top, 0), ("bottom", bottom, H - 3)):
            taps = [(kx + 3, 0, 0) for kx in range(-3, 4)]
            ops.gemm(rec, a0=a, c0=256, dims=(W + 6, 1, tp, B), strides0=(256, (W + 6) * 256, (W + 6) * 256, tp * (W + 6) * 256),
                     box=(32, 1, 4, 1), start=(0, 0, 0, 0), count=(W, 1, tp, B), taps=taps, w=pk.w["init_fea_" + side], n=d,
                     out=x0, out_stride=ostr, out_base=base + y0 * W * d, res=x0, res_base=base + y0 * W * d, res_stride=ostr,
                     phases=[(taps, pr * W * d) for pr in range(3)])
        for side, a, x_0 in (("left", left, 0), ("right", right, W - 3)):
            taps = [(0, ky, 0) for ky in range(-3, 4)]
            ops.gemm(rec, a0=a, c0=256, dims=(1, H, tp, B), strides0=(256, 256, H * 256, tp * H * 256), box=(1, 32, 4, 1),
                     start=(0, 0, 0, 0), count=(1, H, tp, B), taps=taps, w=pk.w["init_fea_" + side], n=d, out=x0,
                     out_stride=ostr, out_base=base + x_0 * d, res=x0, res_base=base + x_0 * d, res_stride=ostr,
                     phases=[(taps, pr * d) for pr in range(3)])

    def _composite_init(self, rec, x0, res, res_fp32, bias):
        """frames [tc, T) of x0 (B, T, H, W, d) (+)= init_conv_x(init_noise_conv(x)), exactly, without the 256-channel
        intermediate:  xn = b1 + w1 * pad3(x) is zero padded before init_conv's 7x7 window, so
            w2 * pad3(xn)  =  w2 * xn_ext  -  w2 * ring,
        with xn_ext = b1 + w1 * pad6(x) the intermediate evaluated on the image extended by 3 pixels and `ring` its values
        outside the image.  The first term is ONE 13x13 convolution of the 3-channel flow (w12 = w2 * w1, K = 13 * 64 after
        an x-direction im2col, plus the constant w2 . b1); the second only touches output pixels within 3 of the border
        and only the kernel rows / columns that reach outside.  The ring values are linear in x (init_noise_conv is
        folded into the correction weights), and summed over ALL ring positions of a side the correction of an output row
        / column is position independent: one 3-phase GEMM per side over the same x-im2col tensor (rows above / below:
        K = 192; columns left / right: K = 832), then the four 3x3 corner blocks, which two sides both contain, are
        added back by a small kernel (36 pixels per frame)."""
        cfg, pk, B, H, W = self.cfg, self.pk, self.B, self.H, self.W
        T, tc, tp = cfg.T, cfg.tc, cfg.tp
        d = cfg.dim
        hw = H * W
        xc = torch.zeros(B, T, H, W, 64, device=self.dev, dtype=BF16)
        ops.im2col13x_flow(rec, self.x, xc, tc)
        rbase = tc * hw * d
        ops.conv_cl(rec, xc, pk.w["init_comp"], d, 0, x0, t_range=(tc, T), taps=[(0, dy, 0) for dy in range(-6, 7)],
                    bias=bias, res=res, res_fp32=res_fp32)
        # ---- ring correction: im2col rows (147 patch values + a constant 1) of the four strips; init_noise_conv is folded
        # into the correction weights, so the intermediate's ring values are never materialised
        ostr = (d, W * d, hw * d, T * hw * d)
        xstr = (64, W * 64, hw * 64, T * hw * 64)
        # rows above / below: three phases (output rows) over the image's first / last three rows
        for side, y0 in (("top", 0), ("bottom", H - 3)):
            taps = [(0, 0, 0), (0, 1, 0), (0, 2, 0)]
            ops.gemm(rec, a0=xc, c0=64, dims=(W, H, T, B), strides0=xstr, box=(32, 1, 4, 1), start=(0, y0, tc, 0),
                     count=(W, 1, tp, B), taps=taps, w=pk.w["init_ring_" + side], n=d, out=x0, out_stride=ostr, res=x0,
                     res_stride=ostr, phases=[(taps, pr * W * d) for pr in range(3)])
        # columns left / right: three phases (output columns), the 13 row offsets as taps, read at the output column
        for side, x_0 in (("left", 0), ("right", W - 3)):
            ops.gemm(rec, a0=xc, c0=64, dims=(W, H, T, B), strides0=xstr, box=(1, 32, 4, 1), start=(x_0, 0, tc, 0),
                     count=(1, H, tp, B), taps=[(0, dy, 0) for dy in range(-6, 7)], w=pk.w["init_ring_" + side], n=d,
                     out=x0, out_stride=ostr, res=x0, res_stride=ostr,
                     phases=[([(pr, dy, 0) for dy in range(-6, 7)], pr * d) for pr in range(3)])
        # the corner blocks of the ring were subtracted twice
        ops.init_corner_fix(rec, self.x, pk.f32["init_ring_corners"], x0, tc)

    def _im2col_gemm(self, rec, a, w, n, out, t0, nt, bias=None, res=None):
        """rows of `a` are (b, t, p) for t in [0, nt); write to frames [t0, t0+nt) of out (B, T, H, W, n')."""
        B, T, H, W, ld = out.shape
        hw = H * W
        ops.gemm(rec, a0=a, c0=192, dims=(hw, 1, nt, B), strides0=(192, hw * 192, hw * 192, nt * hw * 192),
                 box=(128, 1, 1, 1), start=(0, 0, 0, 0), count=(hw, 1, nt, B), taps=[(0, 0, 0)], w=w, n=n, out=out,
                 out_stride=(ld, 0, hw * ld, T * hw * ld), out_base=t0 * hw * ld, bias=bias, res=res,
                 res_fp32=res is not None, res_base=t0 * hw * ld if res is not None else 0)

    # ------------------------------------------------------------------ execution
    def set_conditioning(self, cond_frames, cond_fea):
        self.cond_frames.copy_(cond_frames)
        self.cond_fea.copy_(cond_fea)

    def run_prologue(self):
        self.prologue.run()

    def run_step(self, ss=None):
        """One Unet3D forward on the static buffers.  ss: pre-computed (scale, shift) rows for this timestep
        (ss_for_times); None evaluates the time MLPs from self.time."""
        if ss is None:
            self.time_rec.run()
        else:
            self.ss.copy_(ss)
        self.step.run()

    def ss_for_times(self, times):
        """(len(times), B, n_ss): the ResnetBlocks' time-conditioned (scale, shift) for each sampling timestep
        (...cross_multi.py:812-817, :185-188), cached per schedule."""
        key = tuple(int(t) for t in times)
        if key not in self._ss_tables:
            rows = []
            for t in key:
                self.time.fill_(t)
                self.time_rec.run()
                rows.append(self.ss.clone())
            self._ss_tables[key] = torch.stack(rows)
        return self._ss_tables[key]

    def ss_rows_for_times(self, times):
        """(len(times), n_ss): as ss_for_times, one row per timestep instead of B identical ones (each sample's rows
        are computed independently, so row 0 is every sample's row), cached per schedule.  The ancestral sampler
        broadcasts row `step` into self.ss on the device (ops.ddpm_broadcast_row)."""
        key = tuple(int(t) for t in times)
        if key not in self._ss_rows:
            rows = torch.empty(len(key), self.pk.n_ss, device=self.dev)
            for i, t in enumerate(key):
                self.time.fill_(t)
                self.time_rec.run()
                rows[i].copy_(self.ss[0])
            self._ss_rows[key] = rows
        return self._ss_rows[key]


class Unet3D(ParamTree):
    """Drop-in for the reference Unet3D (same ctor / forward / state_dict), CUDA-only execution."""

    def __init__(self, dim, cond_dim=None, out_grid_dim=2, out_conf_dim=1, window_size=None, dim_mults=(1, 2, 4),
                 channels=3, cond_channels=3, attn_heads=8, attn_dim_head=None, use_bert_text_cond=False,
                 init_dim=None, init_kernel_size=7, resnet_groups=8, use_final_activation=False,
                 learn_null_cond=False, use_deconv=True, padding_mode="zeros", cond_num=0, pred_num=0, l=None,
                 framesize=32, architecture="DenoiseNet_STWAtt_w_w_ref_adaptor_cross_multi_traj_ada"):
        super().__init__()
        if cond_dim is not None or use_bert_text_cond:
            raise NotImplementedError("text conditioning is dead code on the sampling path (has_cond=False)")
        if not use_deconv or use_final_activation or init_kernel_size != 7 or out_grid_dim != 2 or out_conf_dim != 1:
            raise NotImplementedError("only the shipped Unet3D hyper-parameters are supported")
        variant = UNET_ARCHITECTURES.get(architecture, architecture)
        self.cfg = UnetConfig(variant, cond_num, pred_num, dim=dim, dim_mults=dim_mults, channels=channels,
                              heads=attn_heads, groups=resnet_groups)
        self.tc, self.tp = cond_num, pred_num
        self.has_cond = False
        man = unet_manifest(self.cfg)
        self.build_tree(man, synth_state_dict(man, seed=0))
        self._fill_constants()
        self._packed = None
        self._runners = {}
        self.register_load_state_dict_post_hook(lambda m, k: m.invalidate())

    def invalidate(self):
        self._packed = None
        self._runners = {}

    def _fill_constants(self):
        """Architecture constants that the reference keeps in its state_dict (rotary freqs, Swin index table)."""
        cfg = self.cfg
        rot = min(32, cfg.dim_head)
        freqs = 1.0 / (10000.0 ** (torch.arange(0, rot, 2)[: rot // 2].float() / rot))
        wd, wh, ww = cfg.window
        coords = torch.stack(torch.meshgrid(torch.arange(wd), torch.arange(wh), torch.arange(ww), indexing="ij"))
        cf = coords.flatten(1)
        rel = (cf[:, :, None] - cf[:, None, :]).permute(1, 2, 0).contiguous()
        rel[:, :, 0] += wd - 1
        rel[:, :, 1] += wh - 1
        rel[:, :, 2] += ww - 1
        rel[:, :, 0] *= (2 * wh - 1) * (2 * ww - 1)
        rel[:, :, 1] *= 2 * ww - 1
        index = rel.sum(-1)
        for k, v in self.flat_state_dict().items():
            if k.endswith("rotary_emb.freqs"):
                v.copy_(freqs)
            elif k.endswith("relative_position_index"):
                v.copy_(index)

    def runner(self, B, H, W, fea_hw):
        dev = next(self.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError("Unet3D runs on CUDA only (hand-written sm_100a kernels, no CPU fallback)")
        if self._packed is None or self._packed.dev != dev:
            self.invalidate()
            self._packed = PackedUnet(self.flat_state_dict(), self.cfg, dev)
        key = (B, H, W, fea_hw)
        if key not in self._runners:
            self._runners[key] = UnetRunner(self._packed, B, H, W, fea_hw)
        return self._runners[key]

    @torch.no_grad()
    def forward(self, x, time, cond_frames, cond_fea=None, cond=None, null_cond_prob=0.0, none_cond_mask=None):
        cfg = self.cfg
        tc, tp = cond_frames.shape[2], x.shape[2]
        assert tc == self.tc
        assert tp == self.tp
        assert cond_fea.shape[2] == cfg.T
        r = self.runner(x.shape[0], x.shape[3], x.shape[4], cond_fea.shape[-1])
        r.set_conditioning(cond_frames.float(), cond_fea.float())
        r.x.copy_(x)
        r.time.copy_(time)
        r.run_prologue()
        r.run_step()
        return r.out.clone()

    def forward_with_cond_scale(self, *args, cond_scale=2.0, **kwargs):
        return self.forward(*args, **kwargs)          # has_cond is False: cond_scale is inert (…cross_multi.py:898-904)
