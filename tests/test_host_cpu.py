"""CPU: host logic of the product -- state_dict manifests, schedules, the C ABI surface, sharding."""
import ctypes
import os
import re
import subprocess
import sys

import pytest
import torch

import extdm_b200  # noqa: F401
from extdm_b200 import lib
from extdm_b200.manifest import UnetConfig, adaptor_layers, unet_manifest
from rollout_common import load as load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


@pytest.mark.parametrize("name,variant,tc,tp,dm", [("unet_ada_c2p5", "ada", 2, 5, (1, 2, 4, 4)),
                                                   ("unet_u12_c2p3", "u12", 2, 3, (1, 2, 4, 4)),
                                                   ("unet_base_c3p2", "base", 3, 2, (1, 2, 4, 8)),
                                                   ("unet_u22_c2p5", "u22", 2, 5, (1, 2, 4, 4)),
                                                   ("unet_ada_c10p20", "ada", 10, 20, (1, 2, 4, 4)),
                                                   ("unet_u12_c2p10", "u12", 2, 10, (1, 2, 4, 4)),
                                                   ("unet_base_c10p5", "base", 10, 5, (1, 2, 4, 8))])
def test_unet_manifest_matches_reference(name, variant, tc, tp, dm):
    fx = torch.load(os.path.join(GOLD, name + ".pt"))
    ref = {k: tuple(v) for k, v in fx["manifest"].items()}
    assert unet_manifest(UnetConfig(variant, tc, tp, dim_mults=dm)) == ref


def test_adaptor_layers():
    # SURVEY App. B.7: KTH L=2/30 frames, BAIR L=3/14, SMMNIST L=1/9, UCF L=2/12, City L=2/6
    assert adaptor_layers(10, 20) == (2, 30)
    assert adaptor_layers(2, 10) == (3, 14)
    assert adaptor_layers(9, 5) == (1, 9)
    assert adaptor_layers(4, 8) == (2, 12)
    assert adaptor_layers(2, 5) == (2, 6)


def test_wrapper_state_dicts_match_reference():
    from extdm_b200.flow_diffusion import FlowDiffusion
    fx = load_golden("pipeline_kth_c2p5")
    fd = FlowDiffusion(config=fx["cfg"], pretrained_pth="", is_train=False,
                       Unet3D_architecture="DenoiseNet_STWAtt_w_w_ref_adaptor_cross_multi_traj_ada")
    for part in ("generator", "region_predictor", "bg_predictor", "diffusion"):
        mine = {k: tuple(v.shape) for k, v in getattr(fd, part).state_dict().items()}
        assert mine == {k: tuple(v) for k, v in fx["manifests"][part].items()}, part
    assert fd.cond_frame_num == 2 and fd.pred_frame_num == 5


def test_conditioning_stage_matches_reference_on_cpu():
    from extdm_b200.flow_diffusion import FlowDiffusion
    from extdm_b200.weights import synth_state_dict
    fx = load_golden("pipeline_kth_c2p5")
    # the constructor puts the LFAE modules on cuda:0 when there is one (as the reference does): keep them on the CPU
    fd = FlowDiffusion(config=fx["cfg"], pretrained_pth="", is_train=False,
                       Unet3D_architecture="DenoiseNet_STWAtt_w_w_ref_adaptor_cross_multi_traj_ada").eval().cpu()
    for part, seed in fx["weight_seeds"].items():
        m = getattr(fd, part)
        m.load_state_dict(synth_state_dict(fx["manifests"][part], seed, base=m.state_dict()), strict=True)
    real_vid = torch.rand((1, 1, 2, 64, 64), generator=torch.Generator().manual_seed(500)).expand(1, 3, 2, 64, 64)
    ret, x_cond, fea, _ = fd.condition(real_vid.contiguous(), with_decode=True)
    for k in ("real_vid_grid", "real_vid_conf", "real_out_vid", "real_warped_vid"):
        assert (ret[k] - fx["out"][k]).abs().max().item() < 2e-4, k
    assert x_cond.shape == (1, 3, 2, 32, 32) and fea.shape == (1, 256, 7, 16, 16)


def test_hot_path_refuses_cpu():
    """No CPU / PyTorch fallback: the UNet and the decoder raise when they are not on a CUDA device."""
    from extdm_b200.unet import Unet3D
    u = Unet3D(dim=64, channels=512, dim_mults=(1, 2, 4, 4), cond_num=2, pred_num=5)
    with pytest.raises(RuntimeError):
        u(torch.zeros(1, 3, 5, 32, 32), torch.zeros(1, dtype=torch.long), cond_frames=torch.zeros(1, 3, 2, 32, 32),
          cond_fea=torch.zeros(1, 256, 7, 16, 16))


def test_ddim_schedule_matches_oracle():
    from oracle import extdm_oracle as O
    from extdm_b200.diffusion import GaussianDiffusion
    d = GaussianDiffusion(torch.nn.Identity(), image_size=32, num_frames=30, sampling_timesteps=10, timesteps=1000)
    sched = d.ddim_schedule()
    assert [s[0] for s in sched] == [909, 818, 727, 636, 545, 454, 363, 272, 181, 90]
    assert [(a, b) for a, b, *_ in sched] == O.ddim_time_pairs()
    tab = O.cosine_schedule_tables()
    for k in ("alphas_cumprod_prev", "sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod"):
        assert torch.equal(getattr(d, k), tab[k])
    assert sched[-1][5] == 0.0 and sched[-1][6] == 0.0 and sched[-1][4] == 1.0      # last step: img = x_start


def test_c_abi_exports_every_declared_symbol():
    """The shared library loads without a GPU and exports every function include/extdm_b200.h declares."""
    hdr = open(os.path.join(ROOT, "include", "extdm_b200.h")).read()
    declared = set(re.findall(r"\b(extdm_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 25
    cdll = ctypes.CDLL(lib.LIB_PATH)
    for name in declared:
        assert hasattr(cdll, name), f"{name} declared in the header but not exported"
    assert declared == set(lib.PROTOTYPES), declared ^ set(lib.PROTOTYPES)
    assert lib.load().extdm_abi_version() == 5
    assert ctypes.sizeof(lib.ExtdmGemm) == lib.load().extdm_sizeof_gemm()


def test_pack_weights_layouts():
    from extdm_b200 import ops
    w = torch.arange(2 * 3 * 9, dtype=torch.float32).reshape(2, 3, 1, 3, 3)
    p = ops.pack_conv_weight(w).float()
    assert p.shape == (2, 27) and p[1, (1 * 3 + 2) * 3 + 1] == w[1, 1, 0, 1, 2]
    wd = torch.randn(4, 2, 1, 4, 4)
    pd = ops.pack_downsample_weight(wd).float()
    a, b, py, px, ci = 1, 0, 1, 1, 1
    assert torch.allclose(pd[3, (a * 2 + b) * 8 + (py * 2 + px) * 2 + ci], wd[3, ci, 0, 2 * a + py, 2 * b + px].bfloat16().float())
    assert ops.std_box(32, 32) == (32, 4, 1) and ops.std_box(4, 4) == (4, 4, 8) and ops.std_box(64, 64) == (64, 2, 1)


def test_two_rank_sharding_gloo(tmp_path):
    """world_size-2 gloo run of the host-side sharding logic: each rank takes its slice of the videos and the
    predicted frames are all-gathered in rank order (bench.py's N>1 path, without a GPU)."""
    script = tmp_path / "shard.py"
    script.write_text(
        "import os, sys, torch, torch.distributed as dist\n"
        f"sys.path.insert(0, {ROOT!r})\n"
        "import extdm_b200\n"
        "from extdm_b200.sharding import shard_range, gather_predictions\n"
        "dist.init_process_group('gloo')\n"
        "r, w = dist.get_rank(), dist.get_world_size()\n"
        "lo, hi = shard_range(10, r, w)\n"
        "vids = torch.arange(10.).view(10, 1, 1, 1, 1).expand(10, 3, 4, 2, 2)\n"
        "out = gather_predictions(vids[lo:hi].contiguous() * 2, 10)\n"
        "assert torch.equal(out, vids * 2), out.flatten()[:12]\n"
        "assert shard_range(10, 0, 4) == (0, 3) and shard_range(10, 3, 4) == (8, 10)\n"
        "dist.destroy_process_group()\n")
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29581")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29581", str(script)],
                       capture_output=True, text=True, env=env, timeout=240)
    assert r.returncode == 0, r.stdout + r.stderr


def test_metrics_match_reference():
    """evaluate.psnr_videos / ssim_videos against the reference's metrics/calculate_{psnr,ssim}.py (golden fixture)."""
    from extdm_b200 import evaluate
    fx = torch.load(os.path.join(GOLD, "metrics_ref.pt"))
    g = torch.Generator().manual_seed(fx["seed"])
    v1 = torch.rand(3, 4, 3, 32, 32, generator=g)
    v2 = (v1 + 0.05 * torch.randn(3, 4, 3, 32, 32, generator=g)).clamp(0, 1)
    v2[0, 0] = v1[0, 0]
    p, s = evaluate.summarize(evaluate.psnr_videos(v1, v2)), evaluate.summarize(evaluate.ssim_videos(v1, v2))
    for t in range(4):
        assert abs(p[f"avg[{t}]"] - fx["psnr"][f"avg[{t}]"]) < 1e-6
        assert abs(p[f"std[{t}]"] - fx["psnr_std"][f"std[{t}]"]) < 1e-6
        assert abs(s[f"avg[{t}]"] - fx["ssim"][f"avg[{t}]"]) < 1e-9
        assert abs(s[f"std[{t}]"] - fx["ssim_std"][f"std[{t}]"]) < 1e-9


def test_result_wire_format(tmp_path):
    """origin.pt / result_{k}.pt dumps (scripts/DM/valid.py:281-286) and the tolerant diffusion-checkpoint loader."""
    from extdm_b200 import evaluate
    origin, result = torch.rand(2, 3, 6, 3, 8, 8), torch.rand(2, 3, 6, 3, 8, 8)
    evaluate.save_results(str(tmp_path), origin, result)
    assert torch.equal(torch.load(tmp_path / "origin.pt"), origin[:, 0])
    assert torch.equal(torch.load(tmp_path / "result_2.pt"), result[:, 2])
    from extdm_b200.flow_diffusion import FlowDiffusion
    fx = load_golden("pipeline_kth_c2p5")
    fd = FlowDiffusion(config=fx["cfg"], pretrained_pth="", is_train=False,
                       Unet3D_architecture="DenoiseNet_STWAtt_w_w_ref_adaptor_cross_multi_traj_ada").eval()
    sd = {k: v.clone() + 1 for k, v in fd.diffusion.state_dict().items() if v.dtype.is_floating_point}
    sd.update({k: v for k, v in fd.diffusion.state_dict().items() if not v.dtype.is_floating_point})
    sd["denoise_fn.init_temporal_attn.fn.fn.fn.attn.rotary_emb.some_new_buffer"] = torch.zeros(3)   # App. E11
    info = evaluate.load_dm_checkpoint(fd, {"diffusion": sd, "example": 7, "epoch": 1})
    assert info == {"example": 7, "epoch": 1}
    k = "denoise_fn.init_conv.bias"
    assert torch.equal(fd.diffusion.state_dict()[k], sd[k])
    del sd[k]
    with pytest.raises(RuntimeError):
        evaluate.load_dm_checkpoint(fd, {"diffusion": sd})


def test_pack_weights_conv3d_and_tf32():
    """Host-side packing for the 27-tap extrapolator convolution (ada_u22) and for the tf32 GEMM mode: the packed
    matrices reproduce F.conv3d / F.conv2d when contracted against explicitly gathered taps."""
    import torch.nn.functional as F
    from extdm_b200 import ops
    g = torch.Generator().manual_seed(5)
    # ---- 3x3x3: K index ((kt*3 + ky)*3 + kx)*Cin + ci, taps in the same order
    w = torch.randn(4, 3, 3, 3, 3, generator=g)
    x = torch.randn(1, 3, 5, 6, 7, generator=g)
    ref = F.conv3d(x, w, padding=1)
    wp = ops.pack_conv3d_weight(w).float()                           # bf16-rounded
    taps = ops.conv3d_taps(3)
    assert len(taps) == 27 and taps[0] == (-1, -1, -1) and taps[13] == (0, 0, 0) and taps[-1] == (1, 1, 1)
    xp = F.pad(x, (1, 1, 1, 1, 1, 1))
    cols = torch.cat([xp[0, :, 1 + dt:6 + dt, 1 + dy:7 + dy, 1 + dx:8 + dx] for dx, dy, dt in taps], dim=0)  # (27*3,T,H,W)
    got = torch.einsum("ok,kthw->othw", wp, cols)
    assert (got - ref[0]).abs().max() <= 2e-2 * ref.abs().max()
    # ---- tf32 packing: channel groups zero-padded to multiples of 32, values rounded to the nearest tf32
    w2 = torch.randn(5, 35, 3, 3, generator=g)
    p2 = ops.pack_conv_weight_f32(w2, splits=[(0, 32, 32), (32, 35, 32)])
    assert p2.shape == (5, 9 * 64)
    v = p2.view(5, 3, 3, 64)
    assert torch.count_nonzero(v[..., 35:]) == 0
    assert (v[..., :32] - w2[:, :32].permute(0, 2, 3, 1)).abs().max() <= 2.0 ** -11 * w2.abs().max()
    assert (v[..., 32:35] - w2[:, 32:].permute(0, 2, 3, 1)).abs().max() <= 2.0 ** -11 * w2.abs().max()
    assert (p2.view(torch.int32) & 0x1FFF).abs().max() == 0          # low 13 mantissa bits cleared = exact tf32 values


def test_wrapper_registry():
    """`--DM_arch` / `--Unet3D_arch` strings of the reference's scripts map to classes / variants (valid.py:83-99)."""
    from extdm_b200 import flow_diffusion_class
    from extdm_b200.flow_diffusion import FlowDiffusion, FlowDiffusionU22
    from extdm_b200.manifest import UNET_ARCHITECTURES, UnetConfig
    assert flow_diffusion_class("VideoFlowDiffusion_multi_w_ref") is FlowDiffusion
    assert flow_diffusion_class("VideoFlowDiffusion_multi_w_ref_u22") is FlowDiffusionU22
    with pytest.raises(NotImplementedError):
        flow_diffusion_class("VideoFlowDiffusion_nope")
    assert UNET_ARCHITECTURES["DenoiseNet_STWAtt_w_w_ref_adaptor_cross_multi_traj_ada_u22"] == "u22"
    c = UnetConfig("u22", 2, 5)
    assert (c.window, c.dim_head, c.channels, c.resample_slot, c.extrap_kt) == ((4, 4, 4), 32, 259, 6, 3)


def test_composite_init_conv_algebra():
    """extdm_b200/composite.py: init_conv(init_noise_conv(x)) = 13x13 convolution of x - ring correction (four position-
    independent sides + corner add-back), emulated with torch in float64 exactly as the runner's GEMMs and corner kernel
    read the blocks, against the two-stage zero-padded convolution (..._traj_ada.py:916,1032-1042).  Exact algebra: 1e-10."""
    import torch.nn.functional as F
    from extdm_b200 import composite
    g = torch.Generator().manual_seed(5)
    M, co, H, W = 12, 5, 11, 9
    w1 = torch.randn(M, 3, 7, 7, generator=g, dtype=torch.float64)
    b1 = torch.randn(M, generator=g, dtype=torch.float64)
    w2 = torch.randn(co, M, 7, 7, generator=g, dtype=torch.float64)
    x = torch.randn(1, 3, H, W, generator=g, dtype=torch.float64)
    want = F.conv2d(F.conv2d(x, w1, b1, padding=3), w2, None, padding=3)[0].permute(1, 2, 0)       # (H, W, co)
    c = composite.compose(w1, b1, w2)
    # x-direction im2col with the constant channel, zero rows / columns outside the image
    xc = torch.zeros(H, W, 64, dtype=torch.float64)
    for dx in range(-6, 7):
        for ch in range(3):
            lo, hi = max(0, -dx), min(W, W - dx)
            xc[:, lo:hi, (dx + 6) * 3 + ch] = x[0, ch, :, lo + dx:hi + dx]
    xc[:, :, 39] = 1.0
    row = lambda y, xx: xc[y, xx] if 0 <= y < H and 0 <= xx < W else torch.zeros(64, dtype=torch.float64)
    got = torch.zeros(H, W, co, dtype=torch.float64)
    for y in range(H):
        for xx in range(W):
            got[y, xx] = c["comp_bias"] + sum(c["comp"][:, dy + 6] @ row(y + dy, xx) for dy in range(-6, 7))
    for pr in range(3):
        for xx in range(W):
            got[pr, xx] += sum(c["top"][pr][:, sr] @ row(sr, xx) for sr in range(3))
            got[H - 3 + pr, xx] += sum(c["bottom"][pr][:, sr] @ row(H - 3 + sr, xx) for sr in range(3))
        for y in range(H):
            got[y, pr] += sum(c["left"][pr][:, dy + 6] @ row(y + dy, pr) for dy in range(-6, 7))
            got[y, W - 3 + pr] += sum(c["right"][pr][:, dy + 6] @ row(y + dy, W - 3 + pr) for dy in range(-6, 7))
    for cn, (y0, x0) in enumerate(((0, 0), (0, W - 3), (H - 3, 0), (H - 3, W - 3))):
        patch = torch.cat([x[0, :, y0:y0 + 3, x0:x0 + 3].permute(1, 2, 0).reshape(27), torch.ones(1, dtype=torch.float64)])
        for py in range(3):
            for px in range(3):
                got[y0 + py, x0 + px] += patch @ c["corners"][cn, py * 3 + px]
    err = (got - want).abs().max().item()
    assert err <= 1e-10 * want.abs().max().item(), err


def test_composite_upsampled_conv_algebra():
    """extdm_b200/composite.py::compose_upsampled: 7x7 zero-padded convolution of a x2 bilinearly up-sampled tensor as 5x5
    polyphase convolutions of the replicate-padded low-resolution tensor minus four 1-D border corrections, emulated in
    float64 as the runner's GEMMs read the blocks, against F.interpolate + F.conv2d (..._traj_u12.py:1039-1042)."""
    import torch.nn.functional as F
    from extdm_b200 import composite
    g = torch.Generator().manual_seed(9)
    M, co, h, w = 6, 4, 5, 7
    H, W = 2 * h, 2 * w
    w2 = torch.randn(co, M, 7, 7, generator=g, dtype=torch.float64)
    f = torch.randn(1, M, h, w, generator=g, dtype=torch.float64)
    up = F.interpolate(f, scale_factor=2, mode="bilinear", align_corners=False)
    want = F.conv2d(up, w2, None, padding=3)[0].permute(1, 2, 0)                       # (H, W, co)
    c = composite.compose_upsampled(w2)
    fpad = F.pad(f, (2, 2, 2, 2), mode="replicate")[0].permute(1, 2, 0)                # (h + 4, w + 4, M)
    u = up[0].permute(1, 2, 0)                                                         # (H, W, M)
    got = torch.zeros(H, W, co, dtype=torch.float64)
    for i in range(h):
        for j in range(w):
            for py in range(2):
                for px in range(2):
                    blk = c["poly"][py * 2 + px]
                    got[2 * i + py, 2 * j + px] = sum(blk[:, a, b] @ fpad[i + a, j + b] for a in range(5) for b in range(5))
    clampx = lambda xx: min(max(xx, 0), W - 1)
    zero = torch.zeros(M, dtype=torch.float64)
    col = lambda t, y: t[y] if 0 <= y < H else zero
    for p in range(3):
        for xx in range(W):
            got[p, xx] += sum(c["top"][p][:, kx + 3] @ u[0, clampx(xx + kx)] for kx in range(-3, 4))
            got[H - 3 + p, xx] += sum(c["bottom"][p][:, kx + 3] @ u[H - 1, clampx(xx + kx)] for kx in range(-3, 4))
        for y in range(H):
            got[y, p] += sum(c["left"][p][:, ky + 3] @ col(u[:, 0], y + ky) for ky in range(-3, 4))
            got[y, W - 3 + p] += sum(c["right"][p][:, ky + 3] @ col(u[:, W - 1], y + ky) for ky in range(-3, 4))
    err = (got - want).abs().max().item()
    assert err <= 1e-10 * want.abs().max().item(), err
