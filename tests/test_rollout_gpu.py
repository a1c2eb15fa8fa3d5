"""End-to-end parity (-m gpu) of every BASELINE.json configuration against the UNMODIFIED reference wrappers run through
the autoregressive loop of scripts/DM/valid.py:167-172 (tests/golden/rollout_*; generator:
tests/golden/make_golden.py::gen_rollout): SMMNIST via VideoFlowDiffusion_multi1248 (10 -> 10, the full rollout), BAIR
via multi_w_ref + traj_u12 (2 -> 28, the full rollout), UCF (64 regions), Cityscapes 128x128 (perspective background,
scale factor 0.25) and the shipped multi_w_ref_u22 + traj_ada_u22 pairing.  Shipped (tc, tp), 10 DDIM steps, eta = 1,
dynamic thresholding, injected noise.

Gates (bf16 UNet, tf32 conditioning; calibration SURVEY.md section 8c):
  teacher-forced round (each round starts from the reference's own conditioning clip):
      conditioning flow / occlusion  <= 5e-3 abs      latent flow rel-L2 <= 2e-2      frames PSNR >= 35 dB
  free-running rollout (round r+1 is conditioned on this path's own round-r frames, as in valid.py):
      latent flow rel-L2 <= 4e-2 in the last round, predicted frames PSNR >= 30 dB over the whole rollout -- the drift
      budget: a round's frame error (~45 dB) re-enters the conditioning stage of the next round.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu

from rollout_common import ROLLOUTS, build_model, load, psnr, rel_l2, round_noise  # noqa: E402


def _lapack_svd(request):
    """torch.svd's singular-vector signs differ between LAPACK (the CPU run that wrote the fixtures) and cuSOLVER and
    the reference's PCA affine inherits them (region_predictor.py:139-146): use LAPACK's on the device as well."""
    from extdm_b200.lfae import CondRunner
    real_svd, real_pca = torch.svd, CondRunner.pca
    torch.svd = lambda a, *args, **kw: tuple(t.to(a.device) for t in real_svd(a.cpu(), *args, **kw))
    CondRunner.pca = "torch"              # the product's default is the closed form with cuSOLVER's signs
    request.addfinalizer(lambda: (setattr(torch, "svd", real_svd), setattr(CondRunner, "pca", real_pca)))


@pytest.mark.parametrize("name", ROLLOUTS)
def test_round_matches_reference(name, request):
    fx = load(name)
    fd = build_model(fx, "cuda")
    _lapack_svd(request)
    tc = fx["tc"]
    for r, want in enumerate(fx["out"]):
        ret = fd.sample_one_video(cond_scale=1.0, real_vid=want["cond_in"].cuda(), noise=round_noise(fx, r).cuda())
        for k in ("real_vid_grid", "real_vid_conf"):
            err = (ret[k].cpu() - want[k]).abs().max().item()
            assert err <= 5e-3, (name, r, k, err)
        g = rel_l2(ret["sample_vid_grid"][:, :, tc:].cpu(), want["sample_vid_grid"][:, :, tc:])
        c = (ret["sample_vid_conf"].cpu() - want["sample_vid_conf"]).abs().mean().item()
        p = psnr(ret["sample_out_vid"].cpu(), want["sample_out_vid"].float())
        p_pred = psnr(ret["sample_out_vid"][:, :, tc:].cpu(), want["sample_out_vid"][:, :, tc:].float())
        print(f"{name} round {r} (teacher-forced): predicted flow rel-L2 {g:.3e}, occlusion mean-abs {c:.3e}, "
              f"frames PSNR {p:.1f} dB (predicted only {p_pred:.1f} dB)")
        assert tuple(ret["sample_out_vid"].shape) == tuple(want["sample_out_vid"].shape)
        assert g <= 2e-2, (name, r, g)
        assert p >= 35.0 and p_pred >= 35.0, (name, r, p, p_pred)


@pytest.mark.parametrize("name", [n for n in ROLLOUTS if n != "rollout_cityscapes_u22"])
def test_free_running_rollout_matches_reference(name, request):
    """configs.rollout (on-device autoregression, SURVEY.md 8f-2) against the reference's rollout: bf16 drift across
    rounds, stated."""
    from extdm_b200 import configs
    fx = load(name)
    fd = build_model(fx, "cuda")
    _lapack_svd(request)
    tc, tp, rounds = fx["tc"], fx["tp"], fx["rounds"]
    it = iter(range(rounds))
    seen = []

    def noise_fn():
        return round_noise(fx, next(it)).cuda()

    real = fd.sample_one_video

    def spy(*a, **k):
        out = real(*a, **k)
        seen.append(out["sample_vid_grid"][:, :, tc:].cpu())
        return out

    fd.sample_one_video = spy
    pred = configs.rollout(fd, fx["out"][0]["cond_in"].cuda(), rounds * tp, noise_fn=noise_fn).cpu()
    want = torch.cat([o["sample_out_vid"][:, :, tc:].float() for o in fx["out"]], dim=2)
    assert pred.shape == want.shape
    drift = [rel_l2(seen[r], fx["out"][r]["sample_vid_grid"][:, :, tc:]) for r in range(rounds)]
    per_round = [psnr(pred[:, :, r * tp:(r + 1) * tp], want[:, :, r * tp:(r + 1) * tp]) for r in range(rounds)]
    print(f"{name} free-running: predicted flow rel-L2 per round {[f'{d:.3e}' for d in drift]}, "
          f"frames PSNR per round {[f'{p:.1f}' for p in per_round]} dB")
    assert drift[-1] <= 4e-2, drift
    assert psnr(pred, want) >= 30.0, per_round
