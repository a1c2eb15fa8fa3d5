"""Denoising-loss evaluation: the forward-only training objective of p_losses (GaussianDiffusion.denoising_loss,
FlowDiffusion.denoising_loss, evaluate.denoising_loss_videos) and its kernels (csrc/sampler.cu extdm_q_sample,
extdm_denoise_loss).

CPU: argument errors before the CUDA-only refusal, the x_start helper against sample_one_video's post-processing, the
evaluation's seed / timestep policy under sharding.  GPU (-m gpu): forward diffusion bit-exact against the torch fp32
expression and its epsilon against the numpy Philox restatement of tests/test_ddpm.py; the loss reduction against
float64; the whole evaluation on the ddim_ada_c2p5 mini UNet against the oracle; every dataset configuration end to end;
samplers unaffected; batch independence and sharding.
"""
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import extdm_b200  # noqa: F401
from extdm_b200 import configs, evaluate
from extdm_b200.diffusion import GaussianDiffusion
from extdm_b200.flow_diffusion import flow_to_x_start, x_start_to_flow
from extdm_b200.sharding import shard_range, video_seeds
from test_ddpm import _philox_normals

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DEV = "cuda"
# Loss gate for batch dependence.  The UNet's GEMM tile widths follow the batch, so pred differs by a rel-L2 of up to
# 2e-2 (the gate of test_full_batch_is_sample_independent).  With L = |eps - pred|^2 / n and pred -> pred + d,
# |L' - L| / L <= 2 |d| / |eps - pred| + O(d^2), and |eps - pred| >= |pred| for an eps independent of pred, so the loss
# moves by at most about 2 * 2e-2.
LOSS_BATCH_GATE = 4e-2


def bits(t):
    return t.contiguous().view(torch.int32)


def n_graphs(r, kind):
    """The number of CUDA graphs of one kind (the first field of the key) on the UNet runner r."""
    return sum(k[0] == kind for k in r.graphs)


def _rnd(shape, seed, scale=1.0):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed)) * scale


def _clips(B, T, hw, seed):
    """Smooth grey clips (B, 3, T, hw, hw) in [0, 1], as the batch-independence gates were calibrated on."""
    coarse = torch.rand((B, 1, 4, 8, 8), generator=torch.Generator().manual_seed(seed))
    clip = F.interpolate(coarse, size=(T, hw, hw), mode="trilinear", align_corners=True).clamp(0, 1)
    return clip.expand(B, 3, T, hw, hw).contiguous()


# ------------------------------------------------------------------------------------------------ CPU
@pytest.fixture(scope="module")
def kth_cpu():
    model, cfg = configs.build_model("kth", device="cpu")
    return model, cfg


def test_flow_diffusion_loss_argument_errors(kth_cpu):
    model, cfg = kth_cpu
    tc, tp, hw = model.cond_frame_num, model.pred_frame_num, cfg["dataset_params"]["frame_shape"]
    vid = torch.zeros(2, 3, tc + tp, hw, hw)
    h = hw // 2                                                        # scale_factor 0.5
    bad = {
        "tc frames only": dict(real_vid=torch.zeros(2, 3, tc, hw, hw)),
        "one frame too many": dict(real_vid=torch.zeros(2, 3, tc + tp + 1, hw, hw)),
        "4-D": dict(real_vid=torch.zeros(3, tc + tp, hw, hw)),
        "t negative": dict(timesteps=[-1, 0]), "t = T": dict(timesteps=[0, 1000]),
        "t float": dict(timesteps=torch.tensor([1.0, 2.0])), "t int32": dict(timesteps=torch.tensor([1, 2]).int()),
        "t length": dict(timesteps=[1, 2, 3]), "t floats in a list": dict(timesteps=[1.5, 2.0]),
        "noise and seeds": dict(noise=torch.zeros(2, 3, tp, h, h), seeds=[1, 2]),
        "noise shape": dict(noise=torch.zeros(2, 3, tp, h + 1, h)), "seeds length": dict(seeds=[1]),
    }
    for what, kw in bad.items():
        kw = dict(kw)
        with pytest.raises(ValueError):
            model.denoising_loss(kw.pop("real_vid", vid), **kw)
        print("rejected:", what)
    model.diffusion.loss_type = "huber"
    try:
        with pytest.raises(ValueError):
            model.denoising_loss(vid, timesteps=[0, 1])
    finally:
        model.diffusion.loss_type = "l2"
    for kw in (dict(), dict(timesteps=[0, 999], seeds=[1, 2]), dict(noise=torch.zeros(2, 3, tp, h, h))):
        with pytest.raises(RuntimeError) as e:                            # valid arguments reach the CUDA-only refusal
            model.denoising_loss(vid, **kw)
        assert not isinstance(e.value, (ValueError, NotImplementedError))
    with pytest.raises(NotImplementedError):
        model(vid)                                                          # training forward still raises


def test_gaussian_loss_argument_errors():
    from extdm_b200.unet import Unet3D
    u = Unet3D(dim=64, channels=512, dim_mults=(1, 2, 4, 4), cond_num=2, pred_num=5)
    d = GaussianDiffusion(u, image_size=32, num_frames=7, sampling_timesteps=10, timesteps=20, loss_type="l1")
    xs, xc, fea = torch.zeros(2, 3, 5, 32, 32), torch.zeros(2, 3, 2, 32, 32), torch.zeros(2, 256, 7, 16, 16)
    for args in ((torch.zeros(2, 3, 4, 32, 32), xc, fea), (xs, torch.zeros(1, 3, 2, 32, 32), fea),
                 (xs, xc, torch.zeros(3, 256, 7, 16, 16)), (torch.zeros(2, 2, 5, 32, 32), xc, fea)):
        with pytest.raises(ValueError):
            d.denoising_loss(*args)
    with pytest.raises(ValueError):
        d.denoising_loss(xs, xc, fea, timesteps=[0, 20])                    # this schedule has 20 timesteps
    with pytest.raises(RuntimeError) as e:
        d.denoising_loss(xs, xc, fea, timesteps=[0, 19])
    assert not isinstance(e.value, ValueError)


@pytest.mark.parametrize("residual", [False, True])
@pytest.mark.parametrize("occlusion", [True, False])
def test_x_start_inverts_post_processing(residual, occlusion):
    """flow_to_x_start followed by sample_one_video's post-processing (x_start_to_flow) returns (grid, conf).  Square
    frames: FlowDiffusion.get_grid, the identity grid of the residual flow, is square (as every configuration)."""
    B, tp, h, w = 2, 5, 16, 16
    grid = torch.rand(B, 2, tp, h, w, generator=torch.Generator().manual_seed(1)) * 2 - 1
    conf = torch.rand(B, 1, tp, h, w, generator=torch.Generator().manual_seed(2)) if occlusion else None
    x = flow_to_x_start(grid, conf, residual)
    assert x.shape == (B, 3, tp, h, w)
    g2, c2 = x_start_to_flow(x, residual, occlusion)
    assert (g2 - grid).abs().max() <= 1e-6
    if occlusion:
        assert torch.equal(x[:, 2:], conf * 2 - 1) and (c2 - conf).abs().max() <= 1e-7
    else:
        assert c2 is None and not x[:, 2].any()
    if not residual:
        assert torch.equal(x[:, :2], grid) and torch.equal(g2, grid)
    else:
        from extdm_b200.flow_diffusion import FlowDiffusion
        ident = FlowDiffusion.get_grid(B, 1, h, w)
        assert torch.equal(x[:, :2], grid - ident)


class _LossRecorder(torch.nn.Module):
    """Stands in for FlowDiffusion on the CPU: records the timesteps and seeds of every denoising_loss call."""
    cond_frame_num, pred_frame_num = 2, 3

    class _Diffusion:
        num_timesteps = 1000

        def __init__(self):
            self.calls = []

        def denoising_loss(self, x_start, x_cond, cond_fea, timesteps=None, seeds=None, noise=None):
            self.calls.append((timesteps, seeds))
            B = x_start.shape[0]
            t = timesteps if timesteps is not None else torch.zeros(B, dtype=torch.long)
            lpf = (t.float()[:, None] + torch.arange(3.0)) * (seeds.float()[:, None] if seeds is not None else 1)
            return {"loss": lpf.mean(1), "loss_per_frame": lpf, "timesteps": t}

    def __init__(self):
        super().__init__()
        self.w = torch.nn.Parameter(torch.zeros(1))
        self.diffusion = self._Diffusion()

    def loss_inputs(self, real_vid):
        B = real_vid.shape[0]
        return torch.zeros(B, 3, 3, 4, 4), torch.zeros(B, 3, 2, 4, 4), torch.zeros(B, 256, 5, 2, 2)


def test_loss_evaluation_seeds_follow_global_video_index():
    """denoising_loss_videos(seed, video_offset): video b uses video_seeds(seed, g, 0) as its seed and, without given
    timesteps, video_seeds(seed, g, 1) % num_timesteps as its timestep, g = video_offset + b; one call or shards."""
    m, base, n = _LossRecorder(), 17, 7
    vids = torch.zeros(n, 3, 5, 8, 8)
    whole = evaluate.denoising_loss_videos(m, vids, seed=base)
    (t, s), = m.diffusion.calls
    assert torch.equal(s, video_seeds(base, range(n), 0))
    assert torch.equal(t, video_seeds(base, range(n), 1) % 1000)
    assert whole["loss"].shape == (n,) and whole["loss_per_frame"].shape == (n, 3)
    assert not torch.equal(t, s % 1000)                                     # distinct rounds
    for world in (2, 3):
        parts = []
        for rank in range(world):
            lo, hi = shard_range(n, rank, world)
            parts.append(evaluate.denoising_loss_videos(m, vids[lo:hi], seed=base, video_offset=lo))
        for k in whole:
            assert torch.equal(torch.cat([p[k] for p in parts]), whole[k]), (world, k)
    m.diffusion.calls = []
    curve = evaluate.denoising_loss_videos(m, vids, timesteps=[10, 500, 999], seed=base, video_offset=4)
    assert [c[0].tolist() for c in m.diffusion.calls] == [[k] * n for k in (10, 500, 999)]
    assert all(torch.equal(c[1], video_seeds(base, range(4, 4 + n), 0)) for c in m.diffusion.calls)
    assert curve["loss"].shape == (n, 3) and curve["loss_per_frame"].shape == (n, 3, 3)
    assert curve["timesteps"][:, 1].tolist() == [500] * n
    m.diffusion.calls = []
    evaluate.denoising_loss_videos(m, vids, timesteps=3)
    assert m.diffusion.calls[0][0].tolist() == [3] * n and m.diffusion.calls[0][1] is None
    m.diffusion.calls = []
    evaluate.denoising_loss_videos(m, vids)
    assert m.diffusion.calls == [(None, None)]
    for bad in (1000, -1, [5, 1000], [], 2.0, [True]):
        with pytest.raises(ValueError):
            evaluate.denoising_loss_videos(m, vids, timesteps=bad)


# ------------------------------------------------------------------------------------------------ GPU: kernels
def _ops():
    from extdm_b200 import ops
    return ops, ops.IMMEDIATE


def _tables():
    d = GaussianDiffusion(torch.nn.Identity(), image_size=32, num_frames=7, sampling_timesteps=10, timesteps=1000)
    return d.sqrt_alphas_cumprod.to(DEV), d.sqrt_one_minus_alphas_cumprod.to(DEV)


def _q_sample(x_start, t, seeds=None, noise=None):
    ops, R = _ops()
    acp, a1m = _tables()
    x_t, eps = torch.empty_like(x_start), torch.empty_like(x_start)
    ops.q_sample(R, x_start, torch.as_tensor(t, dtype=torch.long).to(DEV),
                 None if seeds is None else torch.as_tensor(seeds, dtype=torch.long).to(DEV), noise, acp, a1m, x_t, eps)
    return x_t, eps


@pytest.mark.gpu
def test_q_sample_bit_exact_with_injected_noise():
    acp, a1m = _tables()
    gen = torch.Generator(device=DEV).manual_seed(3)
    t = torch.tensor([0, 1, 500, 999], device=DEV)
    x0 = torch.randn(4, 3, 5, 32, 32, device=DEV, generator=gen) * 0.7
    noise = torch.randn(4, 3, 5, 32, 32, device=DEV, generator=gen)
    ref = acp[t].view(4, 1, 1, 1, 1) * x0 + a1m[t].view(4, 1, 1, 1, 1) * noise        # Diffusion.py q_sample
    x_t, eps = _q_sample(x0, t, noise=noise)
    assert torch.equal(bits(x_t), bits(ref)) and torch.equal(eps, noise)
    ops, R = _ops()
    with pytest.raises(ValueError):
        ops.q_sample(R, x0, t, torch.zeros(4, dtype=torch.long, device=DEV), noise, acp, a1m, x_t, eps)
    with pytest.raises(ValueError):
        ops.q_sample(R, x0, t[:3].contiguous(), None, noise, acp, a1m, x_t, eps)
    with pytest.raises(ValueError):
        ops.q_sample(R, x0, t.int(), None, noise, acp, a1m, x_t, eps)


@pytest.mark.gpu
def test_q_sample_noise_matches_documented_generator():
    """The drawn eps is Philox4x32-10 keyed by (seed, element / 4, t, stream 2) + Box-Muller (include/extdm_b200.h)."""
    n = 3 * 4 * 16 * 16
    seeds, t = [0, 12345, -7, 2 ** 62 + 3], [0, 731, 999, 5]
    _, eps = _q_sample(torch.zeros(4, n, device=DEV), t, seeds=seeds)
    for b in range(4):
        ref = _philox_normals(seeds[b], n, t[b], 2)
        got = eps[b].double().cpu().numpy()
        assert np.abs(got - ref).max() <= 2e-5 * max(1.0, np.abs(ref).max()), b
    other = _philox_normals(seeds[1], n, t[1], 0)                           # stream 2 is not the sampler's stream 0
    assert np.abs(eps[1].double().cpu().numpy() - other).max() > 1.0


@pytest.mark.gpu
def test_q_sample_seeds_batch_independent():
    gen = torch.Generator(device=DEV).manual_seed(4)
    x0 = torch.randn(5, 3, 5, 32, 32, device=DEV, generator=gen)
    seeds, t = [7, 12345, 7, -3, 7], [10, 500, 10, 999, 11]
    x_t, eps = _q_sample(x0, t, seeds=seeds)
    assert torch.equal(eps[0], eps[2]) and not torch.equal(eps[0], eps[1])     # repeated (seed, t): same draw
    assert not torch.equal(eps[0], eps[4])                                    # same seed, other t: another draw
    perm = [3, 0, 4, 2, 1]
    x_p, e_p = _q_sample(x0[perm].contiguous(), [t[i] for i in perm], seeds=[seeds[i] for i in perm])
    assert torch.equal(bits(x_p), bits(x_t[perm])) and torch.equal(bits(e_p), bits(eps[perm]))
    x_1, e_1 = _q_sample(x0[1:2].contiguous(), t[1:2], seeds=seeds[1:2])
    assert torch.equal(bits(x_1), bits(x_t[1:2])) and torch.equal(bits(e_1), bits(eps[1:2]))
    again = _q_sample(x0, t, seeds=seeds)
    assert torch.equal(bits(again[0]), bits(x_t)) and torch.equal(bits(again[1]), bits(eps))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(3, 3, 5, 32, 32), (2, 3, 7, 16, 24), (1, 3, 1, 8, 8)])
@pytest.mark.parametrize("l1", [False, True])
def test_denoise_loss_matches_float64(shape, l1):
    ops, R = _ops()
    gen = torch.Generator(device=DEV).manual_seed(shape[2])
    eps, pred = torch.randn(shape, device=DEV, generator=gen), torch.randn(shape, device=DEV, generator=gen) * 0.8
    B, _, tp = shape[:3]
    out = torch.empty(B, tp, device=DEV)
    ops.denoise_loss(R, eps, pred, out, l1)
    d = eps.double() - pred.double()
    ref = (d.abs() if l1 else d * d).mean(dim=(1, 3, 4))
    rel = ((out.double() - ref).abs() / ref).max().item()
    print(f"denoise_loss {shape} l1={l1}: max rel err vs float64 {rel:.2e}")
    assert rel <= 1e-6
    again = torch.empty_like(out)
    ops.denoise_loss(R, eps, pred, again, l1)
    assert torch.equal(bits(again), bits(out))
    one = torch.empty(1, tp, device=DEV)
    ops.denoise_loss(R, eps[-1:].contiguous(), pred[-1:].contiguous(), one, l1)
    assert torch.equal(bits(one), bits(out[-1:]))
    with pytest.raises(ValueError):
        ops.denoise_loss(R, eps, pred, torch.empty(B, tp + 1, device=DEV), l1)


# ------------------------------------------------------------------------------------------------ GPU: mini UNet
def _mini():
    from extdm_b200.unet import Unet3D
    from extdm_b200.weights import synth_state_dict
    fx = torch.load(os.path.join(GOLD, "ddim_ada_c2p5.pt"))
    u = Unet3D(dim=64, channels=512, dim_mults=fx["dim_mults"], cond_num=fx["tc"], pred_num=fx["tp"],
               architecture=fx["variant"]).cuda()
    sd = synth_state_dict(fx["manifest"], fx["weight_seed"])
    assert not u.load_state_dict(sd, strict=False).unexpected_keys
    B, tc, tp = fx["B"], fx["tc"], fx["tp"]
    diff = GaussianDiffusion(u, image_size=32, num_frames=tc + tp, sampling_timesteps=fx["sampling"], timesteps=1000,
                             loss_type="l2", null_cond_prob=0.0).cuda()
    x_cond = _rnd((B, 3, tc, 32, 32), fx["input_seed"] + 2, 0.5).cuda()
    fea = _rnd((B, 256, tc + tp, 16, 16), fx["input_seed"] + 3, 0.5).abs().cuda()
    x_start = _rnd((B, 3, tp, 32, 32), fx["input_seed"] + 4, 0.5).clamp(-1, 1).cuda()
    return u, sd, fx, diff, x_start, x_cond, fea


@pytest.mark.gpu
def test_denoising_loss_mini_unet_graph_cache():
    from oracle import extdm_oracle as O
    torch.set_num_threads(8)
    u, sd, fx, diff, x_start, x_cond, fea = _mini()
    B, tc, tp = fx["B"], fx["tc"], fx["tp"]
    r = u.runner(B, 32, 32, fea.shape[-1])
    t, seeds = torch.tensor([17, 731]), torch.tensor([5, 1000008])
    diff.use_cuda_graph = False
    eager = diff.denoising_loss(x_start, x_cond, fea, timesteps=t, seeds=seeds)
    x_t, pred = r.x.clone(), r.out.clone()
    assert torch.equal(eager["timesteps"].cpu(), t)
    # x_t: the torch expression on the kernel's eps
    _, eps = _q_sample(x_start, t, seeds=seeds)
    acp, a1m = _tables()
    ref_xt = acp[t.cuda()].view(B, 1, 1, 1, 1) * x_start + a1m[t.cuda()].view(B, 1, 1, 1, 1) * eps
    assert torch.equal(bits(x_t), bits(ref_xt))
    # pred: Unet3D.forward with one timestep per video
    assert torch.equal(bits(u(x_t, t.cuda(), cond_frames=x_cond, cond_fea=fea)), bits(pred))
    d = eps.double() - pred.double()
    assert ((eager["loss_per_frame"].double() - (d * d).mean(dim=(1, 3, 4))).abs()
            / (d * d).mean(dim=(1, 3, 4))).max() <= 1e-6
    assert torch.allclose(eager["loss"], eager["loss_per_frame"].mean(1))
    # against the oracle's fp32 UNet (the UNet's rel-L2 gate, 2e-2)
    with torch.no_grad():
        pred_ref = O.unet_forward(O.SD({"denoise_fn." + k: v for k, v in sd.items()}).sub("denoise_fn"),
                                  O.unet_config("ada", tc, tp), x_t.cpu(), t, x_cond.cpu(), fea.cpu())
    loss_ref = ((eps.cpu().double() - pred_ref.double()) ** 2).mean(dim=(1, 2, 3, 4))
    rel = ((eager["loss"].cpu().double() - loss_ref).abs() / loss_ref)
    print("loss vs oracle fp32 UNet, relative per video:", rel.tolist(), "loss", eager["loss"].tolist())
    assert rel.max() <= 2e-2
    # graph == eager, one capture for every t and seed vector
    diff.use_cuda_graph = True
    g1 = diff.denoising_loss(x_start, x_cond, fea, timesteps=t, seeds=seeds)
    assert torch.equal(bits(g1["loss_per_frame"]), bits(eager["loss_per_frame"]))
    assert n_graphs(r, "loss") == 1
    for t2, s2 in ((torch.tensor([999, 0]), torch.tensor([-3, 2 ** 62 + 1])), ([1, 1], [9, 9])):
        g2 = diff.denoising_loss(x_start, x_cond, fea, timesteps=t2, seeds=s2)
        diff.use_cuda_graph = False
        e2 = diff.denoising_loss(x_start, x_cond, fea, timesteps=t2, seeds=s2)
        diff.use_cuda_graph = True
        assert torch.equal(bits(g2["loss_per_frame"]), bits(e2["loss_per_frame"]))
        assert not torch.equal(g2["loss"], g1["loss"])
    assert n_graphs(r, "loss") == 1
    dev_t = diff.denoising_loss(x_start, x_cond, fea, timesteps=t.cuda(), seeds=seeds.cuda())
    assert torch.equal(bits(dev_t["loss_per_frame"]), bits(eager["loss_per_frame"]))
    # injected noise: its own graph, equal to the seeded evaluation fed the same eps
    inj = diff.denoising_loss(x_start, x_cond, fea, timesteps=t, noise=eps)
    assert torch.equal(bits(inj["loss_per_frame"]), bits(eager["loss_per_frame"])) and n_graphs(r, "loss") == 2
    # drawn t and seeds: torch.randint from the default generator, t first
    torch.manual_seed(3)
    drawn = diff.denoising_loss(x_start, x_cond, fea)
    torch.manual_seed(3)
    t3 = torch.randint(0, 1000, (B,))
    s3 = torch.randint(0, 2 ** 62, (B,), dtype=torch.long)
    assert torch.equal(drawn["timesteps"].cpu(), t3)
    given = diff.denoising_loss(x_start, x_cond, fea, timesteps=t3, seeds=s3)
    assert torch.equal(bits(given["loss_per_frame"]), bits(drawn["loss_per_frame"]))
    # l1: its own graph, graph == eager, against float64
    diff.loss_type = "l1"
    g_l1 = diff.denoising_loss(x_start, x_cond, fea, timesteps=t, seeds=seeds)
    diff.use_cuda_graph = False
    e_l1 = diff.denoising_loss(x_start, x_cond, fea, timesteps=t, seeds=seeds)
    assert torch.equal(bits(g_l1["loss_per_frame"]), bits(e_l1["loss_per_frame"]))
    ref_l1 = d.abs().mean(dim=(1, 3, 4))
    assert ((e_l1["loss_per_frame"].double() - ref_l1).abs() / ref_l1).max() <= 1e-6


@pytest.mark.gpu
def test_sampling_unaffected_by_loss_evaluation():
    """A seeded DDIM sample and a DDPM round on the runner the loss evaluation shares (r.x, r.time, r.ss): bit-identical
    before and after it."""
    u, sd, fx, diff, x_start, x_cond, fea = _mini()
    B, tc, tp = fx["B"], fx["tc"], fx["tp"]
    ddpm = GaussianDiffusion(u, image_size=32, num_frames=tc + tp, sampling_timesteps=None, timesteps=20,
                             loss_type="l2").cuda()
    shape = (B, 3, tp, 32, 32)
    seeds = [11, 22]

    def samples():
        return diff.sample(x_cond, fea, seeds=seeds), ddpm.p_sample_loop(x_cond, shape, fea, seeds=seeds)

    before = samples()
    for graphed in (True, False):
        diff.use_cuda_graph = graphed
        diff.denoising_loss(x_start, x_cond, fea, timesteps=[3, 900], seeds=[1, 2])
    diff.use_cuda_graph = True
    after = samples()
    for a, b in zip(before, after):
        assert torch.equal(bits(a), bits(b))


# ------------------------------------------------------------------------------------------------ GPU: FlowDiffusion
def _capture_inputs(model):
    """Wraps model.diffusion.denoising_loss to record its (x_start, x_cond, cond_fea)."""
    seen = []
    real = model.diffusion.denoising_loss

    def recording(x_start, x_cond, cond_fea, **kw):
        seen.append((x_start.clone(), x_cond.clone(), cond_fea.clone()))
        return real(x_start, x_cond, cond_fea, **kw)

    model.diffusion.denoising_loss = recording
    return seen


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["kth", "smmnist", "bair", "ucf", "cityscapes", "cityscapes_u22"])
def test_flow_diffusion_denoising_loss(name):
    from extdm_b200.flow_autoenc import FlowAE
    model, cfg = configs.build_model(name, device="cuda")
    tc, tp, hw = model.cond_frame_num, model.pred_frame_num, cfg["dataset_params"]["frame_shape"]
    vid = _clips(2, tc + tp, hw, 5).cuda()
    seen = _capture_inputs(model)
    try:
        out = model.denoising_loss(vid, seeds=[3, 4])
    finally:
        del model.diffusion.denoising_loss
    assert out["loss"].shape == (2,) and out["loss_per_frame"].shape == (2, tp)
    assert torch.isfinite(out["loss_per_frame"]).all() and (out["loss"] > 0).all()
    assert ((0 <= out["timesteps"]) & (out["timesteps"] < 1000)).all()
    (x_start, x_cond, fea), = seen
    _, ref_cond, ref_fea, _ = model.condition(vid[:, :, :tc].contiguous())
    assert torch.equal(fea, ref_fea)
    # the cond-frame flows come from a CondRunner over tc + tp frames instead of tc: bit for bit where the kernels'
    # tiling does not depend on the frame count, else within the tf32 floor of test_native_conditioning_matches_torch_fp32
    diff = (x_cond - ref_cond).abs().max().item()
    print(f"{name}: x_cond vs condition() max-abs {diff:.3e} ({'bit-identical' if diff == 0 else 'differs'}); "
          f"loss {out['loss'].tolist()}")
    assert diff <= 2e-3
    rec = FlowAE.from_flow_diffusion(model).reconstruct(vid, tc - 1)
    flow_ref = flow_to_x_start(rec["optical_flow"][:, :, tc:], rec["occlusion_map"][:, :, tc:],
                               model.use_residual_flow)
    assert torch.equal(bits(x_start), bits(flow_ref))


@pytest.mark.gpu
def test_loss_batch_independence_and_sharding():
    """Video k alone against a batch of 3 and a 2-way sharded evaluate.denoising_loss_videos against one call: the
    timesteps equal, x_t bit-identical on the same x_start, the loss within LOSS_BATCH_GATE."""
    model, cfg = configs.build_model("kth", device="cuda")
    tc, tp, hw = model.cond_frame_num, model.pred_frame_num, cfg["dataset_params"]["frame_shape"]
    vids = _clips(3, tc + tp, hw, 21)
    diff = model.diffusion
    # x_t on the same x_start, alone and in the batch
    x_start, x_cond, fea = model.loss_inputs(vids.cuda())
    t, seeds = torch.tensor([100, 500, 900]), torch.tensor([101, 4242, 77])
    diff.denoising_loss(x_start, x_cond, fea, timesteps=t, seeds=seeds)
    r3 = diff.denoise_fn.runner(3, x_start.shape[3], x_start.shape[4], fea.shape[-1])
    xt3 = r3.x.clone()
    diff.denoising_loss(x_start[1:2], x_cond[1:2], fea[1:2], timesteps=t[1:2], seeds=seeds[1:2])
    r1 = diff.denoise_fn.runner(1, x_start.shape[3], x_start.shape[4], fea.shape[-1])
    assert torch.equal(bits(r1.x), bits(xt3[1:2]))
    # the whole evaluation, alone / batch / shards
    whole = evaluate.denoising_loss_videos(model, vids, seed=9)
    alone = evaluate.denoising_loss_videos(model, vids[1:2], seed=9, video_offset=1)
    parts = [evaluate.denoising_loss_videos(model, vids[lo:hi], seed=9, video_offset=lo)
             for lo, hi in (shard_range(3, r, 2) for r in range(2))]
    sharded = {k: torch.cat([p[k] for p in parts]) for k in whole}
    assert torch.equal(alone["timesteps"], whole["timesteps"][1:2])
    assert torch.equal(sharded["timesteps"], whole["timesteps"])
    d_alone = ((alone["loss"] - whole["loss"][1:2]).abs() / whole["loss"][1:2]).max().item()
    d_shard = ((sharded["loss"] - whole["loss"]).abs() / whole["loss"]).max().item()
    print(f"loss alone vs batch of 3: rel {d_alone:.3e}; 2-way sharded vs one call: rel {d_shard:.3e}")
    assert d_alone <= LOSS_BATCH_GATE and d_shard <= LOSS_BATCH_GATE
    again = evaluate.denoising_loss_videos(model, vids, seed=9)
    assert torch.equal(again["loss_per_frame"], whole["loss_per_frame"])
    curve = evaluate.denoising_loss_videos(model, vids, timesteps=[50, 500, 950], seed=9)
    assert curve["loss"].shape == (3, 3) and torch.isfinite(curve["loss"]).all()
    assert curve["timesteps"].tolist() == [[50, 500, 950]] * 3
    assert not math.isclose(curve["loss"][0, 0].item(), curve["loss"][0, 2].item())
