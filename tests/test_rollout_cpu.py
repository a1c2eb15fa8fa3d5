"""CPU: the end-to-end fixtures of every BASELINE.json configuration (tests/golden/rollout_*, produced by the
unmodified reference wrappers through the autoregressive loop of scripts/DM/valid.py:167-172) against

  * this repo's configuration table (configs.py) -- the fields FlowDiffusion reads equal the reference yaml's,
  * the torch restatement of the LFAE conditioning modules (lfae.py) on every config: 10 / 20 / 64 regions,
    scale factor 0.5 / 0.25, affine / perspective background (bg_motion_predictor.py:47-64), both rounds,
  * the oracle: one whole DDIM round + decode of the metric's own configurations (BAIR u12, SMMNIST base).
"""
import pytest
import torch

import extdm_b200  # noqa: F401
from extdm_b200 import configs
from extdm_b200.weights import synth_state_dict
from oracle import extdm_oracle as O

from rollout_common import ROLLOUTS, build_model, load, rel_l2, round_noise, smooth_clip

_CONFIG_NAME = {"rollout_smmnist": "smmnist", "rollout_bair": "bair", "rollout_ucf": "ucf",
                "rollout_cityscapes": "cityscapes", "rollout_cityscapes_u22": "cityscapes_u22"}


def _subset(mine, ref, path=""):
    """Every key of `mine` exists in the reference yaml with the same value."""
    for k, v in mine.items():
        if path + k == "dataset_params.valid_params.pred_frames":
            continue            # rollout length: BASELINE.json's wording (UCF 4 -> 12; ucf.yaml itself says 16)
        assert k in ref, f"{path}{k} missing in the reference yaml"
        if isinstance(v, dict):
            _subset(v, ref[k], f"{path}{k}.")
        else:
            assert v == ref[k], f"{path}{k}: {v!r} != {ref[k]!r}"


@pytest.mark.parametrize("name", ROLLOUTS)
def test_config_table_matches_reference_yaml(name):
    fx = load(name)
    cfg, wrapper, unet = configs.dataset(_CONFIG_NAME[name])
    assert wrapper == fx["dm_arch"]
    assert extdm_b200.manifest.UNET_ARCHITECTURES[unet] == fx["variant"]
    _subset(cfg, fx["cfg"])
    assert fx["tc"] == cfg["dataset_params"]["train_params"]["cond_frames"]
    assert fx["tp"] == cfg["dataset_params"]["train_params"]["pred_frames"]
    rounds_full = -(-cfg["dataset_params"]["valid_params"]["pred_frames"] // fx["tp"])
    assert fx["rounds"] <= rounds_full


@pytest.mark.parametrize("name", ROLLOUTS)
def test_conditioning_matches_reference_on_cpu(name):
    """FlowDiffusion.condition (torch restatement of RegionPredictor / BGMotionPredictor / PixelwiseFlowPredictor /
    Generator.forward) vs the reference's real_vid_grid / real_vid_conf, every round of the fixture."""
    torch.set_num_threads(8)
    fx = load(name)
    fd = build_model(fx, "cpu")
    first = smooth_clip(fx["B"], fx["tc"], fx["hw"], fx["input_seed"], gray=fx["dataset"] in ("smmnist", "kth"))
    assert torch.equal(first, fx["out"][0]["cond_in"]), "input clip is not reproducible from its seed"
    for r, want in enumerate(fx["out"]):
        ret, x_cond, fea, _ = fd.condition(want["cond_in"])
        for k in ("real_vid_grid", "real_vid_conf"):
            err = (ret[k] - want[k]).abs().max().item()
            assert err < 2e-4, (name, r, k, err)
        tc, tp = fx["tc"], fx["tp"]
        assert x_cond.shape == (fx["B"], 3, tc, 32, 32)
        T = tc - 1 + tp if fx["variant"] == "base" else tc + tp
        fh = 32 if fx["variant"] == "base" else fx["hw"] // 4
        assert fea.shape == (fx["B"], 256, T, fh, fh)


@pytest.mark.parametrize("name", ["rollout_bair", "rollout_smmnist"])
def test_oracle_round_matches_reference(name):
    """The oracle's DDIM loop (10 steps, eta = 1, dynamic threshold, injected noise) and decode on round 0 of the
    metric's own configurations, from the reference's conditioning outputs: latent flow / occlusion <= 1e-4 abs after
    10 steps of fp32 re-association, decoded frames to fp16 storage precision."""
    torch.set_num_threads(8)
    fx = load(name)
    fd = build_model(fx, "cpu")
    want = fx["out"][0]
    tc, tp = fx["tc"], fx["tp"]
    ret, x_cond, fea, ref_img = fd.condition(want["cond_in"])
    base = fd.diffusion.state_dict()
    sd = synth_state_dict({k: tuple(v.shape) for k, v in base.items()}, fx["weight_seeds"]["diffusion"], base=base)
    cfg = O.unet_config(fx["variant"], tc, tp, dim_mults=(1, 2, 4, 8) if fx["variant"] == "base" else (1, 2, 4, 4))
    nz = round_noise(fx, 0)
    with torch.no_grad():
        pred = O.ddim_sample(O.SD(sd), cfg, x_cond, fea, nz[0], list(nz[1:]) + [None], sampling=fx["steps"])
    grid = torch.cat([want["real_vid_grid"], pred[:, :2]], dim=2)
    conf = torch.cat([want["real_vid_conf"], (pred[:, 2:3] + 1) * 0.5], dim=2)
    e_g = (grid - want["sample_vid_grid"]).abs().max().item()
    e_c = (conf - want["sample_vid_conf"]).abs().max().item()
    print(name, "oracle round: flow max-abs", e_g, "occlusion max-abs", e_c)
    assert e_g < 1e-4 and e_c < 1e-4, (e_g, e_c)
    gbase = fd.generator.state_dict()
    gsd = synth_state_dict(fx["manifests"]["generator"], fx["weight_seeds"]["generator"], base=gbase)
    with torch.no_grad():
        out, _ = O.decode_video(O.SD(gsd), ref_img, want["sample_vid_grid"][:, :, :3], want["sample_vid_conf"][:, :, :3])
    assert (out - want["sample_out_vid"][:, :, :3].float()).abs().max().item() < 2e-3
