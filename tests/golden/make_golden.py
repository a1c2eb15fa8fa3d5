"""Generate golden fixtures by running the UNMODIFIED reference (/root/reference) on CPU.

Run in the build container only:   python tests/golden/make_golden.py
Writes tests/golden/<case>.pt = {cfg, manifest (key -> shape of the reference state_dict), seeds,
outputs}.  Inputs and weights are NOT stored: they are regenerated from seeds by `inputs_for()` below
and `weights.synth_state_dict` (both deterministic on the CPU generator), so fixtures stay small.  The pipeline and
rollout fixtures go through tests/rollout_common.py::save: xz-compressed as <case>.pt.xz above 1 MB, and a rollout in
a compact form that rollout_common.load() expands exactly; save() refuses a file over 1 MB.
"""
import importlib
import os
import sys

import torch
import yaml

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

from oracle import ref_shims  # noqa: E402
from rollout_common import save  # noqa: E402

ref_shims.install()
import extdm_b200  # noqa: E402
from extdm_b200.weights import synth_state_dict  # noqa: E402

UNET_MODULES = {
    "ada": "DenoiseNet_STWAtt_w_w_ref_adaptor_cross_multi_traj_ada",
    "u12": "DenoiseNet_STWAtt_w_w_ref_adaptor_cross_multi_traj_u12",
    "base": "DenoiseNet_STWAtt_w_wo_ref_adaptor_cross_multi",
    "u22": "DenoiseNet_STWAtt_w_w_ref_adaptor_cross_multi_traj_ada_u22",
}

UNET_CASES = {
    # name: (variant, tc, tp, dim_mults, B)
    "unet_ada_c2p5": ("ada", 2, 5, (1, 2, 4, 4), 1),
    "unet_u12_c2p3": ("u12", 2, 3, (1, 2, 4, 4), 1),
    "unet_base_c3p2": ("base", 3, 2, (1, 2, 4, 8), 1),
    "unet_u22_c2p5": ("u22", 2, 5, (1, 2, 4, 4), 1),
    # the shipped (tc, tp) of the benchmark configurations (SURVEY.md section 8d): KTH, BAIR, SMMNIST
    "unet_ada_c10p20": ("ada", 10, 20, (1, 2, 4, 4), 1),
    "unet_u12_c2p10": ("u12", 2, 10, (1, 2, 4, 4), 1),
    "unet_base_c10p5": ("base", 10, 5, (1, 2, 4, 8), 1),
}


def rnd(shape, seed, scale=1.0):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed)) * scale


def unet_inputs(variant, tc, tp, B, seed):
    tm = tc - 1 if variant == "base" else tc
    fea_hw = 32 if variant == "base" else 16
    return dict(
        x=rnd((B, 3, tp, 32, 32), seed + 1),
        cond_frames=rnd((B, 3, tc, 32, 32), seed + 2, 0.5),
        cond_fea=rnd((B, 256, tm + tp, fea_hw, fea_hw), seed + 3, 0.5).abs(),
        time=torch.full((B,), 545, dtype=torch.long),
    )


def build_ref_unet(variant, tc, tp, dim_mults):
    mod = importlib.import_module("model.BaseDM_adaptor." + UNET_MODULES[variant])
    # ada_u22 feeds the 3-channel flow volume straight into init_conv (its forward never calls init_noise_conv,
    # ..._traj_ada_u22.py:1176-1242), so it takes 3 + 256 input channels like the base variant
    channels = 3 + 256 if variant in ("base", "u22") else 512
    return mod.Unet3D(dim=64, channels=channels, out_grid_dim=2, out_conf_dim=1, dim_mults=dim_mults,
                      use_bert_text_cond=False, learn_null_cond=False, use_final_activation=False,
                      use_deconv=True, padding_mode="zeros", cond_num=tc, pred_num=tp).eval()


def manifest_of(module_or_sd):
    sd = module_or_sd if isinstance(module_or_sd, dict) else module_or_sd.state_dict()
    return {k: tuple(v.shape) for k, v in sd.items()}


def gen_unet(name):
    variant, tc, tp, dim_mults, B = UNET_CASES[name]
    net = build_ref_unet(variant, tc, tp, dim_mults)
    base = net.state_dict()
    man = manifest_of(base)
    sd = synth_state_dict(man, seed=11, base=base)
    net.load_state_dict(sd, strict=True)
    inp = unet_inputs(variant, tc, tp, B, seed=100)
    with torch.no_grad():
        out = net(inp["x"], inp["time"], cond_frames=inp["cond_frames"], cond_fea=inp["cond_fea"])
    torch.save(dict(kind="unet", variant=variant, tc=tc, tp=tp, dim_mults=dim_mults, B=B, weight_seed=11,
                    input_seed=100, manifest=man, out=out.clone(),
                    input_checksum=float(sum(v.double().sum() for v in inp.values()))),
               os.path.join(HERE, name + ".pt"))
    print(name, tuple(out.shape), float(out.abs().mean()))


def gen_ddim():
    """GaussianDiffusion.ddim_sample on the mini 'ada' UNet, 3 sampling steps, injected noise."""
    variant, tc, tp, dim_mults, B = "ada", 2, 5, (1, 2, 4, 4), 2
    net = build_ref_unet(variant, tc, tp, dim_mults)
    base = net.state_dict()
    man = manifest_of(base)
    net.load_state_dict(synth_state_dict(man, seed=11, base=base), strict=True)
    dmod = importlib.import_module("model.BaseDM_adaptor.Diffusion")
    diff = dmod.GaussianDiffusion(net, image_size=32, num_frames=tc + tp, sampling_timesteps=3,
                                  timesteps=1000, loss_type="l2", use_dynamic_thres=True,
                                  null_cond_prob=0.0, ddim_sampling_eta=1.0).eval()
    inp = unet_inputs(variant, tc, tp, B, seed=200)
    noises = [rnd((B, 3, tp, 32, 32), 300 + i) for i in range(4)]   # [init, step0, step1, (unused last)]
    queue = list(noises)
    real_randn, real_randn_like = torch.randn, torch.randn_like
    torch.randn = lambda *a, **k: queue.pop(0)
    torch.randn_like = lambda *a, **k: queue.pop(0)
    try:
        with torch.no_grad():
            out = diff.sample(inp["cond_frames"], cond_fea=inp["cond_fea"], batch_size=B, cond_scale=1.0)
    finally:
        torch.randn, torch.randn_like = real_randn, real_randn_like
    tables = {k: v.clone() for k, v in diff.state_dict().items() if not k.startswith("denoise_fn.")}
    torch.save(dict(kind="ddim", variant=variant, tc=tc, tp=tp, dim_mults=dim_mults, B=B, weight_seed=11,
                    input_seed=200, noise_seed=300, sampling=3, manifest=man, out=out.clone(),
                    tables={k: tables[k] for k in ("alphas_cumprod_prev", "sqrt_recip_alphas_cumprod",
                                                   "sqrt_recipm1_alphas_cumprod")}),
               os.path.join(HERE, "ddim_ada_c2p5.pt"))
    print("ddim", tuple(out.shape), float(out.abs().mean()))


def kth_config():
    return yaml.safe_load(open(os.path.join(ref_shims.REF_ROOT, "config/DM/kth.yaml")))


def gen_generator():
    cfg = kth_config()
    fp = cfg["flow_params"]["model_params"]
    gmod = importlib.import_module("model.LFAE.generator")
    gen = gmod.Generator(num_regions=fp["num_regions"], num_channels=fp["num_channels"],
                         revert_axis_swap=fp["revert_axis_swap"], **fp["generator_params"]).eval()
    base = gen.state_dict()
    man = manifest_of(base)
    gen.load_state_dict(synth_state_dict(man, seed=21, base=base), strict=True)
    B = 2
    src = torch.rand((B, 3, 64, 64), generator=torch.Generator().manual_seed(400))
    ident = torch.stack(torch.meshgrid(torch.linspace(-1, 1, 32), torch.linspace(-1, 1, 32), indexing="xy"), -1)
    flow = ident[None] + rnd((B, 32, 32, 2), 401, 0.15)          # some samples fall out of bounds
    occ = torch.rand((B, 1, 32, 32), generator=torch.Generator().manual_seed(402))
    with torch.no_grad():
        a = gen.forward_with_flow(src, flow, occ)
        b = gen.forward_with_flow(src, flow, None)
    torch.save(dict(kind="generator", B=B, weight_seed=21, manifest=man,
                    prediction=a["prediction"].clone(), deformed=a["deformed"].clone(),
                    prediction_noocc=b["prediction"].clone()),
               os.path.join(HERE, "generator_fwf.pt"))
    print("generator", float(a["prediction"].mean()), float(b["prediction"].mean()))


def gen_pipeline():
    """Whole FlowDiffusion.sample_one_video on a shrunk KTH config (tc=2, tp=5, 2 DDIM steps)."""
    cfg = kth_config()
    cfg["dataset_params"]["train_params"]["cond_frames"] = 2
    cfg["dataset_params"]["train_params"]["pred_frames"] = 5
    cfg["diffusion_params"]["model_params"]["sampling_timesteps"] = 2
    wmod = importlib.import_module("model.BaseDM_adaptor.VideoFlowDiffusion_multi_w_ref")
    fd = wmod.FlowDiffusion(config=cfg, pretrained_pth="", is_train=False,
                            Unet3D_architecture=UNET_MODULES["ada"]).eval()
    mans, seeds = {}, dict(generator=21, region_predictor=22, bg_predictor=23, diffusion=11)
    for part, seed in seeds.items():
        m = getattr(fd, part)
        base = m.state_dict()
        mans[part] = manifest_of(base)
        m.load_state_dict(synth_state_dict(mans[part], seed=seed, base=base), strict=True)
    B = 1
    real_vid = torch.rand((B, 1, 2, 64, 64), generator=torch.Generator().manual_seed(500)).expand(B, 3, 2, 64, 64)
    noises = [rnd((B, 3, 5, 32, 32), 600 + i) for i in range(3)]
    queue = list(noises)
    real_randn, real_randn_like = torch.randn, torch.randn_like
    torch.randn = lambda *a, **k: queue.pop(0)
    torch.randn_like = lambda *a, **k: queue.pop(0)
    try:
        with torch.no_grad():
            ret = fd.sample_one_video(cond_scale=1.0, real_vid=real_vid.contiguous())
    finally:
        torch.randn, torch.randn_like = real_randn, real_randn_like
    save(dict(kind="pipeline", cfg=cfg, B=B, weight_seeds=seeds, manifests=mans, input_seed=500,
              noise_seed=600, out={k: v.clone() for k, v in ret.items()}), "pipeline_kth_c2p5")
    print("pipeline", {k: tuple(v.shape) for k, v in ret.items()})


def gen_pipeline_full():
    """FlowDiffusion.sample_one_video at the benchmark configuration itself: shipped KTH config (tc=10, tp=20, 10 DDIM
    steps, eta=1, dynamic threshold), one video.  Stored: latent flow / occlusion in fp32, decoded frames in fp16."""
    cfg = kth_config()
    wmod = importlib.import_module("model.BaseDM_adaptor.VideoFlowDiffusion_multi_w_ref")
    fd = wmod.FlowDiffusion(config=cfg, pretrained_pth="", is_train=False,
                            Unet3D_architecture=UNET_MODULES["ada"]).eval()
    mans, seeds = {}, dict(generator=21, region_predictor=22, bg_predictor=23, diffusion=11)
    for part, seed in seeds.items():
        m = getattr(fd, part)
        base = m.state_dict()
        mans[part] = manifest_of(base)
        m.load_state_dict(synth_state_dict(mans[part], seed=seed, base=base), strict=True)
    B, tc, tp, steps = 1, 10, 20, 10
    # a smooth gray clip (low-resolution noise, tri-linearly up-sampled): natural-video-like content; on white noise a
    # 0.1-pixel flow difference already dominates the frame PSNR
    coarse = torch.rand((B, 1, 4, 8, 8), generator=torch.Generator().manual_seed(700))
    real_vid = torch.nn.functional.interpolate(coarse, size=(tc, 64, 64), mode="trilinear", align_corners=True)
    real_vid = real_vid.clamp(0, 1).expand(B, 3, tc, 64, 64)
    queue = [rnd((B, 3, tp, 32, 32), 800 + i) for i in range(steps + 1)]
    real_randn, real_randn_like = torch.randn, torch.randn_like
    torch.randn = lambda *a, **k: queue.pop(0)
    torch.randn_like = lambda *a, **k: queue.pop(0)
    try:
        with torch.no_grad():
            ret = fd.sample_one_video(cond_scale=1.0, real_vid=real_vid.contiguous())
    finally:
        torch.randn, torch.randn_like = real_randn, real_randn_like
    out = {"sample_vid_grid": ret["sample_vid_grid"].clone(), "sample_vid_conf": ret["sample_vid_conf"].clone(),
           "sample_out_vid": ret["sample_out_vid"].half()}
    save(dict(kind="pipeline_full", B=B, tc=tc, tp=tp, steps=steps, weight_seeds=seeds, input_seed=700,
              noise_seed=800, noises_left=len(queue), out=out), "pipeline_kth_full")
    print("pipeline_full", {k: tuple(v.shape) for k, v in out.items()}, "unused noises", len(queue))


# ---------------------------------------------------------------------------------------------------------------------
# End-to-end fixtures for every BASELINE.json configuration (SURVEY.md section 8d): the UNMODIFIED reference wrapper run
# through the autoregressive loop of scripts/DM/valid.py:167-172 at the shipped (tc, tp), 10 DDIM steps, eta = 1,
# dynamic thresholding, injected noise, LAPACK SVD (this container has no GPU), estimate_occlusion_map = True.
PIPELINE_CASES = {
    # name: (config yaml, --DM_arch wrapper, UNet variant, rounds, DDIM steps)
    "rollout_smmnist": ("smmnist", "VideoFlowDiffusion_multi1248", "base", 2, 10),          # the full 10 -> 10 rollout
    "rollout_bair": ("bair", "VideoFlowDiffusion_multi_w_ref", "u12", 3, 10),               # the full 2 -> 28 rollout
    "rollout_ucf": ("ucf", "VideoFlowDiffusion_multi_w_ref", "ada", 2, 10),                 # the full 4 -> 12 rollout
    # 128x128, sf 0.25, perspective; one round: two rounds of 128x128 frames do not fit in 1 MB
    "rollout_cityscapes": ("cityscapes", "VideoFlowDiffusion_multi_w_ref", "ada", 1, 10),
    "rollout_cityscapes_u22": ("cityscapes", "VideoFlowDiffusion_multi_w_ref_u22", "u22", 1, 10),
}
PIPELINE_SEEDS = dict(generator=21, region_predictor=22, bg_predictor=23, diffusion=11)


def smooth_clip(B, tc, hw, seed, gray):
    """A smooth clip in [0, 1] (coarse noise, tri-linearly up-sampled): natural-video-like content.  On white noise a
    0.1-pixel flow difference already dominates the frame PSNR.  gray: one channel replicated to three
    (data/video_dataset.py:26-33 does that to the KTH / SMMNIST clips)."""
    c = 1 if gray else 3
    coarse = torch.rand((B, c, 4, 8, 8), generator=torch.Generator().manual_seed(seed))
    vid = torch.nn.functional.interpolate(coarse, size=(tc, hw, hw), mode="trilinear", align_corners=True).clamp(0, 1)
    return vid.expand(B, 3, tc, hw, hw).contiguous()


def round_noise(B, tp, steps, seed, rnd_i):
    """The `steps` Gaussian tensors one sample_one_video round consumes: the initial latent, then one per DDIM
    iteration but the last (Diffusion.py:218,251)."""
    return [rnd((B, 3, tp, 32, 32), seed + 100 * rnd_i + i) for i in range(steps)]


def build_ref_pipeline(dataset, dm_arch, variant, steps=None):
    cfg = yaml.safe_load(open(os.path.join(ref_shims.REF_ROOT, f"config/DM/{dataset}.yaml")))
    cfg["flow_params"]["model_params"]["generator_params"]["pixelwise_flow_predictor_params"][
        "estimate_occlusion_map"] = True                       # scripts/DM/valid.py:81 with --estimate_occlusion_map
    if steps is not None:
        cfg["diffusion_params"]["model_params"]["sampling_timesteps"] = steps
    wmod = importlib.import_module("model.BaseDM_adaptor." + dm_arch)
    kw = dict(config=cfg, pretrained_pth="", is_train=False)
    if dm_arch.endswith("_u22"):
        kw["device_ids"] = ["cpu", "cpu", "cpu"]
    elif dm_arch != "VideoFlowDiffusion_multi1248":
        kw["Unet3D_architecture"] = UNET_MODULES[variant]
    fd = wmod.FlowDiffusion(**kw).eval()
    mans = {}
    for part, seed in PIPELINE_SEEDS.items():
        m = getattr(fd, part)
        base = m.state_dict()
        mans[part] = manifest_of(base)
        m.load_state_dict(synth_state_dict(mans[part], seed=seed, base=base), strict=True)
    return fd, cfg, mans


def gen_rollout(name):
    dataset, dm_arch, variant, rounds, steps = PIPELINE_CASES[name]
    fd, cfg, mans = build_ref_pipeline(dataset, dm_arch, variant, steps)
    tc, tp = fd.cond_frame_num, fd.pred_frame_num
    hw = cfg["dataset_params"]["frame_shape"]
    B, in_seed, nz_seed = 1, 900, 1000
    cond = smooth_clip(B, tc, hw, in_seed, gray=dataset in ("smmnist", "kth"))
    out_rounds = []
    real_randn, real_randn_like = torch.randn, torch.randn_like
    for r in range(rounds):
        queue = round_noise(B, tp, steps, nz_seed, r)
        torch.randn = lambda *a, **k: queue.pop(0)
        torch.randn_like = lambda *a, **k: queue.pop(0)
        try:
            with torch.no_grad():
                ret = fd.sample_one_video(cond_scale=1.0, real_vid=cond.clone())
        finally:
            torch.randn, torch.randn_like = real_randn, real_randn_like
        assert not queue, f"{len(queue)} noise tensors left"
        out_rounds.append({"cond_in": cond.clone(), "real_vid_grid": ret["real_vid_grid"].clone(),
                           "real_vid_conf": ret["real_vid_conf"].clone(),
                           "sample_vid_grid": ret["sample_vid_grid"].clone(),
                           "sample_vid_conf": ret["sample_vid_conf"].clone(),
                           "sample_out_vid": ret["sample_out_vid"].half()})
        cond = ret["sample_out_vid"][:, :, -tc:].clone()             # scripts/DM/valid.py:171
        print(name, "round", r, "flow abs-mean", float(ret["sample_vid_grid"].abs().mean()), flush=True)
    save(dict(kind="rollout", dataset=dataset, dm_arch=dm_arch, variant=variant, rounds=rounds, steps=steps,
              cfg=cfg, B=B, tc=tc, tp=tp, hw=hw, weight_seeds=PIPELINE_SEEDS, input_seed=in_seed, noise_seed=nz_seed,
              manifests={k: v for k, v in mans.items() if k != "diffusion"}, out=out_rounds), name)


if __name__ == "__main__":
    torch.manual_seed(0)
    torch.set_num_threads(8)
    which = sys.argv[1:] or ["unet", "ddim", "generator", "pipeline"]
    if "unet" in which:
        for n in UNET_CASES:
            gen_unet(n)
    for n in which:
        if n in UNET_CASES:
            gen_unet(n)
    if "ddim" in which:
        gen_ddim()
    if "generator" in which:
        gen_generator()
    if "pipeline" in which:
        gen_pipeline()
    if "pipeline_full" in which:
        gen_pipeline_full()
    if "rollout" in which:
        which = which + list(PIPELINE_CASES)
    for n in which:
        if n in PIPELINE_CASES:
            gen_rollout(n)


def gen_metrics():
    """PSNR / SSIM of the reference's metrics/ package on seeded random videos -> tests/golden/metrics_ref.pt
    (checked by tests/test_host_cpu.py::test_metrics_match_reference)."""
    from metrics.calculate_psnr import calculate_psnr
    from metrics.calculate_ssim import calculate_ssim
    g = torch.Generator().manual_seed(77)
    v1 = torch.rand(3, 4, 3, 32, 32, generator=g)
    v2 = (v1 + 0.05 * torch.randn(3, 4, 3, 32, 32, generator=g)).clamp(0, 1)
    v2[0, 0] = v1[0, 0]
    p, s = calculate_psnr(v1, v2), calculate_ssim(v1, v2)
    plain = lambda d: {k: float(v) for k, v in d.items()}
    torch.save({"seed": 77, "psnr": plain(p["psnr"]), "psnr_std": plain(p["psnr_std"]), "ssim": plain(s["ssim"]),
                "ssim_std": plain(s["ssim_std"])}, os.path.join(HERE, "metrics_ref.pt"))
