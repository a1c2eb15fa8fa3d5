"""DDPM (ancestral) sampler: GaussianDiffusion.p_sample_loop and its kernels (csrc/sampler.cu extdm_ddpm_*), against a
literal restatement of Diffusion.py:136-189 kept in this file (ddpm_step / ddpm_sample below, built on the oracle's
schedule, dynamic threshold and UNet).

CPU: the schedule table, the refusal to run without CUDA, the restated step.  GPU (-m gpu): the kernels bit-exact
against the same torch fp32 ops, the Philox noise, the loop end to end against the restatement (rel-L2 <= 2e-2, the DDIM
gate of DESIGN.md section 3) and one full-size BAIR round.
"""
import os

import numpy as np
import pytest
import torch

import extdm_b200  # noqa: F401
from extdm_b200.diffusion import GaussianDiffusion
from oracle import extdm_oracle as O

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
POSTERIOR = ("sqrt_recip_alphas_cumprod", "sqrt_recipm1_alphas_cumprod", "posterior_mean_coef1",
             "posterior_mean_coef2")


def rnd(shape, seed, scale=1.0):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed)) * scale


def rel_l2(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm()).item()


def bits(t):
    return t.contiguous().view(torch.int32)


# ------------------------------------------------------------------------------------------------ reference restatement
def schedule_tables(timesteps):
    """oracle.cosine_schedule_tables plus the posterior q(x_{t-1} | x_t, x_0) buffers, Diffusion.py:39-49,76-115 (fp64,
    then cast to fp32 as register_buffer does)."""
    x = torch.linspace(0, timesteps, timesteps + 1, dtype=torch.float64)
    ac = torch.cos(((x / timesteps) + 0.008) / (1 + 0.008) * torch.pi * 0.5) ** 2
    ac = ac / ac[0]
    betas = torch.clip(1 - (ac[1:] / ac[:-1]), 0, 0.9999)
    alphas = 1.0 - betas
    alphas_cumprod = torch.cumprod(alphas, dim=0)
    prev = torch.nn.functional.pad(alphas_cumprod[:-1], (1, 0), value=1.0)
    posterior_variance = betas * (1.0 - prev) / (1.0 - alphas_cumprod)
    tab = O.cosine_schedule_tables(timesteps)
    tab.update(posterior_log_variance_clipped=torch.log(posterior_variance.clamp(min=1e-20)).float(),
               posterior_mean_coef1=(betas * torch.sqrt(prev) / (1.0 - alphas_cumprod)).float(),
               posterior_mean_coef2=((1.0 - prev) * torch.sqrt(alphas) / (1.0 - alphas_cumprod)).float())
    return tab


def ddpm_step(tab, img, pred_noise, t, noise):
    """One iteration body of p_sample_loop after the denoiser call, Diffusion.py:136-177 (clip_denoised=True with
    dynamic thresholding); t is the integer timestep, shared by the batch."""
    b = img.shape[0]
    tt = torch.full((b,), t, dtype=torch.long)

    def extract(name):
        return tab[name][tt].reshape(b, *((1,) * (img.ndim - 1)))

    x_start = extract("sqrt_recip_alphas_cumprod") * img - extract("sqrt_recipm1_alphas_cumprod") * pred_noise
    x_start, s = O.dynamic_threshold(x_start)
    mean = extract("posterior_mean_coef1") * x_start + extract("posterior_mean_coef2") * img
    nonzero_mask = (1 - (tt == 0).float()).reshape(b, *((1,) * (img.ndim - 1)))
    log_var = extract("posterior_log_variance_clipped")
    return mean + nonzero_mask * (0.5 * log_var).exp() * noise, x_start, s


def ddpm_sample(sd, cfg, x_cond, cond_fea, init_noise, step_noises, total, trace=None):
    """p_sample_loop with *injected* noise and the keyword fix of SURVEY App. E10 (cond_fea and t passed by keyword):
    init_noise replaces x_T, step_noises[i] the randn_like of iteration i (drawn at t = 0 too)."""
    tab = schedule_tables(total)
    img = init_noise
    unet = sd.sub("denoise_fn")
    for i, t in enumerate(reversed(range(total))):
        tcond = torch.full((img.shape[0],), t, dtype=torch.long)
        pred_noise = O.unet_forward(unet, cfg, img, tcond, x_cond, cond_fea)
        img, x_start, s = ddpm_step(tab, img, pred_noise, t, step_noises[i])
        if trace is not None:
            trace.append(dict(pred_noise=pred_noise, x_start=x_start, s=s.flatten(), img=img))
    return img


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("T", [1000, 20])
def test_ddpm_schedule_matches_reference(T):
    d = GaussianDiffusion(torch.nn.Identity(), image_size=32, num_frames=7, sampling_timesteps=T, timesteps=T)
    assert not d.is_ddim_sampling
    times, rows = d.ddpm_schedule()
    tab = schedule_tables(T)
    for k, v in tab.items():
        assert torch.equal(getattr(d, k), v), k
    assert times.dtype == torch.long and times.tolist() == list(range(T - 1, -1, -1))
    assert rows.dtype == torch.float32 and rows.shape == (T, 5)
    for j, k in enumerate(POSTERIOR):
        assert torch.equal(rows[:, j], tab[k][times]), k
    nonzero = (times != 0).float()
    assert torch.equal(rows[:, 4], nonzero * (0.5 * tab["posterior_log_variance_clipped"][times]).exp())
    assert rows[-1, 4] == 0.0 and rows[-1, 2] == 1.0 and rows[-1, 3] == 0.0        # last step: img = thresholded x0
    assert (rows[:-1, 4] > 0).all()


def test_ddpm_sample_refuses_cpu():
    from extdm_b200.unet import Unet3D
    u = Unet3D(dim=64, channels=512, dim_mults=(1, 2, 4, 4), cond_num=2, pred_num=5)
    d = GaussianDiffusion(u, image_size=32, num_frames=7, sampling_timesteps=20, timesteps=20)
    with pytest.raises(RuntimeError) as e:
        d.sample(torch.zeros(1, 3, 2, 32, 32), cond_fea=torch.zeros(1, 256, 7, 16, 16))
    assert not isinstance(e.value, NotImplementedError)
    d = GaussianDiffusion(u, image_size=32, num_frames=7, sampling_timesteps=None, timesteps=20)
    with pytest.raises(RuntimeError) as e:
        d.sample(torch.zeros(1, 3, 2, 32, 32), cond_fea=torch.zeros(1, 256, 7, 16, 16))
    assert not isinstance(e.value, NotImplementedError)


@pytest.mark.parametrize("t", [19, 7, 1, 0])
def test_reference_ddpm_step(t):
    tab = schedule_tables(20)
    img, pred, z = rnd((2, 3, 5, 8, 8), 1), rnd((2, 3, 5, 8, 8), 2), rnd((2, 3, 5, 8, 8), 3)
    shrink = 0.3 / tab["sqrt_recip_alphas_cumprod"][t]                     # a sample whose quantile clamps to 1
    img[1] *= shrink
    pred[1] *= shrink
    out, x0, s = ddpm_step(tab, img, pred, t, z)
    ref_x0 = tab["sqrt_recip_alphas_cumprod"][t] * img - tab["sqrt_recipm1_alphas_cumprod"][t] * pred
    ref_s = torch.quantile(ref_x0.flatten(1).abs(), 0.9, dim=-1).clamp(min=1.0).view(2, 1, 1, 1, 1)
    assert ref_s[1] == 1.0
    ref_x0 = ref_x0.clamp(-ref_s, ref_s) / ref_s
    mean = tab["posterior_mean_coef1"][t] * ref_x0 + tab["posterior_mean_coef2"][t] * img
    sig = (1.0 - float(t == 0)) * (0.5 * tab["posterior_log_variance_clipped"][t]).exp()
    assert torch.equal(s, ref_s) and torch.equal(x0, ref_x0)
    assert torch.equal(out, mean + sig * z)
    if t == 0:
        assert torch.equal(out, ref_x0) and out.abs().max() <= 1.0
    else:
        assert not torch.equal(out, mean)


# ------------------------------------------------------------------------------------------------ GPU: kernels
DEV = "cuda"


def _rec():
    from extdm_b200 import ops
    return ops, ops.IMMEDIATE


@pytest.mark.gpu
@pytest.mark.parametrize("n", [15360, 61440, 3072])
def test_ddpm_step_bit_exact(n):
    """Threshold + update from a device row against the same torch fp32 ops on the device, at t > 0 and t = 0 (sig = 0,
    where the add of 0 * z still decides signed zeros: compared bit for bit)."""
    ops, R = _rec()
    B = 3
    gen = torch.Generator(device=DEV).manual_seed(5)
    img, pred = torch.randn(B, n, device=DEV, generator=gen), torch.randn(B, n, device=DEV, generator=gen)
    img[1] *= 0.2                                   # one sample whose quantile is < 1 (clamped to 1)
    pred[1] *= 0.2
    noise = torch.randn(2, B, n, device=DEV, generator=gen)
    d = GaussianDiffusion(torch.nn.Identity(), image_size=32, num_frames=7, sampling_timesteps=1000, timesteps=1000)
    times, rows = d.ddpm_schedule(DEV)
    rows = rows[[1000 - 1 - 545, 999]].contiguous()                      # t = 545, t = 0
    for step in (0, 1):
        a, b2, c1, c2, sig = rows[step]
        xs = a * img - b2 * pred
        s_ref = torch.quantile(xs.abs(), 0.9, dim=-1).clamp_(min=1.0)
        assert s_ref[1] == 1.0 and s_ref[0] > 1.0
        xs_c = xs.clamp(-s_ref[:, None], s_ref[:, None]) / s_ref[:, None]
        ref = (c1 * xs_c + c2 * img) + sig * noise[step]
        st = torch.full((1,), step, dtype=torch.int32, device=DEV)
        s = torch.zeros(B, device=DEV)
        ops.ddpm_threshold(R, img, pred, rows, st, 0.9, s)
        assert torch.equal(s, s_ref), (s, s_ref)
        out, xso = torch.zeros_like(img), torch.zeros_like(img)
        ops.ddpm_update(R, img, pred, rows, st, None, noise, s, out, xso)
        assert torch.equal(bits(xso), bits(xs_c))
        assert torch.equal(bits(out), bits(ref))
        if step == 1:
            assert torch.equal(out, xs_c) and out.abs().max() <= 1.0


def _draws(seeds, n, step=None):
    """The x_T draw (step None) or the loop noise of `step` for each seed: (len(seeds), n)."""
    ops, R = _rec()
    sd = torch.tensor(seeds, dtype=torch.long, device=DEV)
    out = torch.empty(len(seeds), n, device=DEV)
    if step is None:
        ops.ddpm_fill_normal(R, sd, out)
        return out
    rows = torch.tensor([[0.0, 0.0, 0.0, 0.0, 1.0]] * (step + 1), device=DEV)   # img_out = 0 + 1 * z
    zero = torch.zeros(len(seeds), n, device=DEV)
    ops.ddpm_update(R, zero, zero, rows, torch.full((1,), step, dtype=torch.int32, device=DEV), sd, None,
                    torch.ones(len(seeds), device=DEV), out)
    return out


def _philox_normals(seed, n, step, stream):
    """numpy restatement of the documented generator (include/extdm_b200.h) in fp64."""
    m32 = np.uint64(0xFFFFFFFF)
    u = np.uint64(seed & 0xFFFFFFFFFFFFFFFF)
    k0, k1 = u & m32, u >> np.uint64(32)
    c = [np.arange(n // 4, dtype=np.uint64), np.full(n // 4, step, np.uint64), np.full(n // 4, stream, np.uint64),
         np.zeros(n // 4, np.uint64)]
    for r in range(10):
        if r:
            k0, k1 = (k0 + np.uint64(0x9E3779B9)) & m32, (k1 + np.uint64(0xBB67AE85)) & m32
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        c = [((p1 >> np.uint64(32)) ^ c[1] ^ k0) & m32, p1 & m32, ((p0 >> np.uint64(32)) ^ c[3] ^ k1) & m32, p0 & m32]
    out = np.empty((n // 4, 4))
    for j, (a, b) in enumerate(((c[0], c[1]), (c[2], c[3]))):
        u1 = ((a >> np.uint64(9)).astype(np.float64) + 0.5) * 2.0 ** -23
        u2 = (b >> np.uint64(8)).astype(np.float64) * 2.0 ** -24
        r = np.sqrt(-2.0 * np.log(u1))
        out[:, 2 * j], out[:, 2 * j + 1] = r * np.cos(2 * np.pi * u2), r * np.sin(2 * np.pi * u2)
    return out.reshape(-1)


@pytest.mark.gpu
def test_philox_noise_matches_documented_generator():
    """Philox4x32-10 keyed by (seed, element / 4, step, stream) + Box-Muller, as include/extdm_b200.h documents it."""
    n = 4096
    for seed in (0, 12345, -7, 2 ** 62 + 3):
        for step, stream in ((None, 1), (0, 0), (731, 0)):
            got = _draws([seed], n, step)[0].double().cpu().numpy()
            ref = _philox_normals(seed, n, 0 if step is None else step, stream)
            assert np.abs(got - ref).max() <= 2e-5 * max(1.0, np.abs(ref).max())


@pytest.mark.gpu
def test_philox_noise_batch_independent_and_deterministic():
    n, k = 3 * 10 * 32 * 32, 987654321
    for step in (None, 0, 999):
        alone = _draws([k], n, step)
        batch = _draws([11, k, 22], n, step)
        assert torch.equal(batch[1], alone[0])
        assert torch.equal(_draws([11, k, 22], n, step), batch)
        assert not torch.equal(batch[0], batch[1])


@pytest.mark.gpu
def test_philox_noise_statistics():
    from scipy import stats
    n = 1 << 22                                               # 4 M draws per video
    z = _draws([1, 2], n, None).double()
    for v in (z[0], _draws([1], n, 5)[0].double()):
        mean, std = v.mean().item(), v.std().item()
        assert abs(mean) < 3e-3 and abs(std - 1.0) < 3e-3, (mean, std)
        p = stats.kstest(v.cpu().numpy(), "norm").pvalue
        assert p > 1e-3, p

    def corr(a, b):
        a, b = a - a.mean(), b - b.mean()
        return ((a * b).mean() / (a.std() * b.std())).item()

    s0, s1 = _draws([1], n, 5)[0].double(), _draws([1], n, 6)[0].double()
    assert abs(corr(s0, s1)) < 3e-3                         # consecutive steps, same video
    assert abs(corr(z[0], z[1])) < 3e-3                     # consecutive seeds, same step
    assert abs(corr(z[0], _draws([1], n, 0)[0].double())) < 3e-3     # x_T against the first loop step


# ------------------------------------------------------------------------------------------------ GPU: the loop
@pytest.mark.gpu
def test_time_rows_broadcast_equals_time_mlp():
    """The loop broadcasts one precomputed time-MLP row per step into every sample's (scale, shift): bit-identical to
    evaluating the time MLP for the whole batch at that timestep."""
    ops, R = _rec()
    fx = torch.load(os.path.join(GOLD, "ddim_ada_c2p5.pt"))
    u, _ = _build_unet(fx)
    r = u.runner(3, 32, 32, 16)
    times = [999, 545, 1, 0]
    table = r.ss_rows_for_times(times)
    assert table.shape == (len(times), r.ss.shape[1])
    out = torch.empty_like(r.ss)
    for i, t in enumerate(times):
        r.time.fill_(t)
        r.time_rec.run()
        ops.ddpm_broadcast_row(R, table, torch.full((1,), i, dtype=torch.int32, device=DEV), out)
        assert torch.equal(bits(out), bits(r.ss)), t


def _build_unet(fx):
    from extdm_b200.unet import Unet3D
    from extdm_b200.weights import synth_state_dict
    u = Unet3D(dim=64, channels=512, dim_mults=fx["dim_mults"], cond_num=fx["tc"], pred_num=fx["tp"],
               architecture=fx["variant"]).cuda()
    sd = synth_state_dict(fx["manifest"], fx["weight_seed"])
    assert not u.load_state_dict(sd, strict=False).unexpected_keys
    return u, sd


@pytest.mark.gpu
def test_ddpm_sample_matches_reference():
    """20-step ancestral loop on the ddim_ada_c2p5 weights / inputs, injected noise (21 slices), against
    ddpm_sample above; graphed == eager == a second graphed run, bit for bit."""
    torch.set_num_threads(8)
    T = 20
    fx = torch.load(os.path.join(GOLD, "ddim_ada_c2p5.pt"))
    u, sd = _build_unet(fx)
    B, tc, tp = fx["B"], fx["tc"], fx["tp"]
    diff = GaussianDiffusion(u, image_size=32, num_frames=tc + tp, sampling_timesteps=T, timesteps=T,
                             loss_type="l2", null_cond_prob=0.0).cuda()
    tm = tc
    cond_frames = rnd((B, 3, tc, 32, 32), fx["input_seed"] + 2, 0.5)
    cond_fea = rnd((B, 256, tm + tp, 16, 16), fx["input_seed"] + 3, 0.5).abs()
    noise = torch.stack([rnd((B, 3, tp, 32, 32), fx["noise_seed"] + i) for i in range(T + 1)])
    trace = []
    eager = diff.p_sample_loop(cond_frames.cuda(), (B, 3, tp, 32, 32), cond_fea.cuda(), noise=noise.cuda(),
                               trace=trace).cpu()
    ref_trace = []
    with torch.no_grad():
        ref = ddpm_sample(O.SD({"denoise_fn." + k: v for k, v in sd.items()}), O.unet_config("ada", tc, tp),
                            cond_frames, cond_fea, noise[0], list(noise[1:]), total=T, trace=ref_trace)
    assert len(trace) == len(ref_trace) == T
    per_step = [rel_l2(a["pred_noise"].cpu(), b["pred_noise"]) for a, b in zip(trace, ref_trace)]
    growth = [rel_l2(a["img"].cpu(), b["img"]) for a, b in zip(trace, ref_trace)]
    r = rel_l2(eager, ref)
    print("ddpm rel-L2", r, "per-step pred_noise", max(per_step), "img by step", growth)
    assert max(per_step) <= 2e-2, per_step
    assert r <= 2e-2, (r, growth)
    assert torch.equal(trace[-1]["img"].cpu(), eager)
    assert eager.abs().max() <= 1.0                          # t = 0: the output is the thresholded x0
    diff.use_cuda_graph = True
    g1 = diff.sample(cond_frames.cuda(), cond_fea=cond_fea.cuda(), noise=noise.cuda()).cpu()
    g2 = diff.sample(cond_frames.cuda(), cond_fea=cond_fea.cuda(), noise=noise.cuda()).cpu()
    assert torch.equal(g1, eager), "graphed and eager loops differ"
    assert torch.equal(g1, g2), "graph replay is not deterministic"
    diff.use_cuda_graph = False
    assert torch.equal(diff.sample(cond_frames.cuda(), cond_fea=cond_fea.cuda(), noise=noise.cuda()).cpu(), eager)


@pytest.mark.gpu
def test_ddpm_full_size_bair_round():
    """FlowDiffusion on the BAIR configuration with sampling_timesteps 1000, batch 2: one round of 1000 replays with no
    host synchronisation and no launch inside the loop, reproducible under torch.manual_seed."""
    from extdm_b200 import configs, lib
    from extdm_b200.flow_diffusion import flow_diffusion_class
    from extdm_b200.weights import synth_state_dict
    cfg, wrapper, arch = configs.dataset("bair")
    cfg["diffusion_params"]["model_params"]["sampling_timesteps"] = 1000
    model = flow_diffusion_class(wrapper)(config=cfg, pretrained_pth="", is_train=False, Unet3D_architecture=arch).eval()
    for i, part in enumerate(("generator", "region_predictor", "bg_predictor", "diffusion")):
        m = getattr(model, part)
        base = m.state_dict()
        m.load_state_dict(synth_state_dict({k: tuple(v.shape) for k, v in base.items()}, 1234 + i, base=base))
    model = model.cuda()
    diff = model.diffusion
    assert not diff.is_ddim_sampling and diff.num_timesteps == 1000
    tc, tp = model.cond_frame_num, model.pred_frame_num
    real_vid = torch.rand((2, 3, tc, 64, 64), generator=torch.Generator().manual_seed(9)).cuda()

    torch.manual_seed(0)
    a = model.sample_one_video(cond_scale=1.0, real_vid=real_vid)
    torch.manual_seed(0)
    b = model.sample_one_video(cond_scale=1.0, real_vid=real_vid)
    for k in a:
        assert torch.equal(a[k], b[k]), k
        assert torch.isfinite(a[k]).all(), k
    flow = a["sample_vid_grid"][:, :, tc:]
    assert flow.abs().max() <= 1.0
    torch.manual_seed(1)
    c = model.sample_one_video(cond_scale=1.0, real_vid=real_vid)
    assert not torch.equal(c["sample_vid_grid"], a["sample_vid_grid"])

    # the round issues the prologue and the x_T fill, then only graph replays; nothing in it waits for the device
    _, x_cond, cond_fea, _ = model.condition(real_vid)
    r = diff.denoise_fn.runner(2, x_cond.shape[3], x_cond.shape[4], cond_fea.shape[-1])
    torch.cuda.synchronize()
    n0 = lib.launches()
    torch.cuda.set_sync_debug_mode("error")
    try:
        pred = diff.sample(x_cond, cond_fea=cond_fea)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert lib.launches() - n0 == len(r.prologue) + 1
    torch.cuda.synchronize()
    assert pred.abs().max() <= 1.0

    diff.sampling_timesteps, diff.is_ddim_sampling = 10, True            # the DDIM path on the same model
    torch.manual_seed(0)
    d = model.sample_one_video(cond_scale=1.0, real_vid=real_vid)
    assert set(d) == set(a) and all(d[k].shape == a[k].shape for k in a)
