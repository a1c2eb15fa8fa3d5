"""Interpolation between two futures: GaussianDiffusion.interpolate (Diffusion.py:261-274 with the keyword fix of SURVEY
App. E10, DESIGN.md section 1), its mix kernel (csrc/sampler.cu extdm_q_interpolate), FlowDiffusion.encode_future /
interpolate_one_video and evaluate.interpolate_videos.

CPU: the DDIM-mode grid against an independent restatement of torch.linspace, argument errors before the CUDA-only
refusal, the refusal of a selected solver, the exported symbol.  GPU (-m gpu): the mix bit-exact against torch fp32
with injected and with Philox epsilon; lam = 0 / 1 and t = 0; both loops on the mini UNet against restatements on the
oracle (rel-L2 <= 2e-2, the gate of DESIGN.md section 3); graph == eager; seeds and batch independence; the lambda
sweep; sharded evaluation; the pipeline's result dict and the encoded future against the LFAE reconstruction.
"""
import ctypes
import math
import os
import re

import numpy as np
import pytest
import torch

import extdm_b200  # noqa: F401
from extdm_b200 import lib
from extdm_b200.diffusion import GaussianDiffusion

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
DEV = "cuda"


def _cpu_unet():
    from extdm_b200.unet import Unet3D
    return Unet3D(dim=64, channels=512, dim_mults=(1, 2, 4, 4), cond_num=2, pred_num=5)


def _linspace_int(t, S):
    """torch.linspace(0, t, S + 1).int() restated: fp32 step t / S; the first half start + i*step, the second half
    end - (S - i)*step with one rounding (a fused multiply-add), each truncated toward zero."""
    step = np.float32(np.float32(t) / np.float32(S))
    half = (S + 1) // 2
    out = []
    for i in range(S + 1):
        if i < half:
            v = np.float32(np.float64(i) * np.float64(step))
        else:
            v = np.float32(np.float64(t) - np.float64(S - i) * np.float64(step))
        out.append(int(v))
    return out


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("S", [1, 3, 5, 10, 14, 25])
def test_interp_grid_matches_restatement(S):
    d = GaussianDiffusion(torch.nn.Identity(), image_size=32, num_frames=7, sampling_timesteps=S, timesteps=1000)
    for t in range(0, 1000):
        ref = list(reversed(_linspace_int(t, S)))
        if t < S:                                     # repeated timesteps: rejected
            assert any(a <= b for a, b in zip(ref, ref[1:]))
            with pytest.raises(ValueError):
                d.interp_times(t)
            continue
        got = d.interp_times(t)
        assert got == ref, (t, got, ref)
        assert got[0] == t and got[-1] == 0 and all(a > b for a, b in zip(got, got[1:]))
    rows = d._ddim_rows(d.interp_times(999))
    assert [(a, b) for a, b, *_ in rows] == list(zip(d.interp_times(999)[:-1], d.interp_times(999)[1:]))
    assert rows[-1][5] == 0.0 and rows[-1][6] == 0.0 and rows[-1][4] == 1.0      # last step: img = x_start


@pytest.mark.parametrize("S", [20, 5])
def test_interp_argument_errors(S):
    u = _cpu_unet()
    d = GaussianDiffusion(u, image_size=32, num_frames=7, sampling_timesteps=S, timesteps=20)
    ancestral = S == 20
    x_cond, fea = torch.zeros(2, 3, 2, 32, 32), torch.zeros(2, 256, 7, 16, 16)
    shape = (2, 3, 5, 32, 32)
    x1, x2 = torch.zeros(shape), torch.ones(shape)
    t = 11
    n_loop = t if ancestral else S - 1
    noise = torch.zeros(2 + n_loop, *shape)
    bad = {"noise and seeds": dict(noise=noise, seeds=[1, 2]),
           "noise shape": dict(noise=torch.zeros(3 + n_loop, *shape)),
           "noise per step": dict(noise=torch.zeros(shape)), "noise dtype": dict(noise=noise.double()),
           "seed length": dict(seeds=[1, 2, 3]), "seed dtype": dict(seeds=torch.tensor([1, 2], dtype=torch.int32)),
           "float seeds": dict(seeds=[1.5, 2.5]),
           "x1 vs x2": dict(x2=torch.zeros(2, 3, 5, 32, 16)), "x1 frames": dict(x1=torch.zeros(2, 3, 4, 32, 32),
                                                                               x2=torch.zeros(2, 3, 4, 32, 32)),
           "x1 dtype": dict(x1=x1.double()), "x1 rank": dict(x1=x1[0], x2=x2[0]),
           "x_cond batch": dict(x_cond=x_cond[:1]), "cond_fea batch": dict(cond_fea=fea[:1]),
           "t high": dict(t=20), "t negative": dict(t=-1), "t float": dict(t=3.0), "t bool": dict(t=True),
           "lam nan": dict(lam=float("nan")), "lam inf": dict(lam=[0.0, float("inf")]), "lam empty": dict(lam=[]),
           "lam str": dict(lam="0.5")}
    if not ancestral:
        bad["grid"] = dict(t=S - 1)                   # linspace(0, S-1, S+1).int() repeats a timestep
    for what, kw in bad.items():
        args = dict(x1=x1, x2=x2, x_cond=x_cond, cond_fea=fea, t=t) | kw
        with pytest.raises(ValueError):
            d.interpolate(**args)
        print("rejected:", what)
    valid = [dict(seeds=[1, 2]), dict(noise=noise), {}, dict(lam=[0.0, 0.5, 1.0]), dict(t=None, seeds=[1, 2])]
    if ancestral:
        valid.append(dict(t=0, noise=torch.zeros(2, *shape)))
    for kw in valid:                                  # valid calls reach the CUDA-only refusal
        with pytest.raises(RuntimeError) as e:
            d.interpolate(**(dict(x1=x1, x2=x2, x_cond=x_cond, cond_fea=fea, t=t) | kw))
        assert not isinstance(e.value, (ValueError, NotImplementedError))


def test_interp_rejects_solver():
    d = GaussianDiffusion(_cpu_unet(), image_size=32, num_frames=7, sampling_timesteps=5, timesteps=20,
                          solver="dpmpp_2m")
    x = torch.zeros(2, 3, 5, 32, 32)
    for solver in ("dpmpp_2m", "dpmpp_2m_sde"):
        d.solver = solver
        with pytest.raises(ValueError):
            d.interpolate(x, x, torch.zeros(2, 3, 2, 32, 32), torch.zeros(2, 256, 7, 16, 16), t=10, seeds=[1, 2])


def test_symbol_is_exported():
    hdr = open(os.path.join(ROOT, "include", "extdm_b200.h")).read()
    assert re.search(r"\bextdm_q_interpolate\s*\(", hdr)
    assert "extdm_q_interpolate" in lib.PROTOTYPES
    assert hasattr(ctypes.CDLL(lib.LIB_PATH), "extdm_q_interpolate")
    assert lib.load().extdm_abi_version() == 5
    from extdm_b200 import evaluate
    from extdm_b200.flow_diffusion import FlowDiffusion
    assert callable(evaluate.interpolate_videos)
    assert callable(FlowDiffusion.encode_future) and callable(FlowDiffusion.interpolate_one_video)


# ------------------------------------------------------------------------------------------------ GPU helpers
def bits(t):
    return t.contiguous().view(torch.int32)


def rel_l2(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm()).item()


def _rnd(shape, seed, scale=1.0):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed)) * scale


def _torch_mix(d, x1, x2, t, lam, e1, e2):
    """The reference expression, torch fp32 ops on x1's device."""
    a, b = d.sqrt_alphas_cumprod[t].to(x1.device), d.sqrt_one_minus_alphas_cumprod[t].to(x1.device)
    return (1 - lam) * (a * x1 + b * e1) + lam * (a * x2 + b * e2)


def _philox_normals(seed, n, step, stream):
    """numpy restatement of the documented generator (include/extdm_b200.h) in fp64, as tests/test_ddpm.py has it."""
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


def _interp_eps(seeds, shape, t, T=1000):
    """(eps1, eps2) the kernel draws for these seeds at t, read back exactly: with tables a = 0, b = 1 and c1 = 1,
    c2 = 0 (or 0, 1) the mix is eps1 (or eps2) itself."""
    from extdm_b200 import ops
    sd = torch.as_tensor(seeds, dtype=torch.long).to(DEV)
    zero = torch.zeros(shape, device=DEV)
    a, b = torch.zeros(T, device=DEV), torch.ones(T, device=DEV)
    out = []
    for c1, c2 in ((1.0, 0.0), (0.0, 1.0)):
        e = torch.empty(shape, device=DEV)
        ops.q_interpolate(ops.IMMEDIATE, zero, zero, t, sd, None, a, b, c1, c2, e)
        out.append(e)
    return out


# ------------------------------------------------------------------------------------------------ GPU: kernel
@pytest.mark.gpu
@pytest.mark.parametrize("n", [3072, 15360, 61440])
def test_q_interpolate_bit_exact(n):
    """The mix against the torch fp32 expression, with injected eps and with the Philox eps of streams 4 and 5 (read
    back through the kernel, checked against the numpy generator, then fed to the torch expression)."""
    from extdm_b200 import ops
    d = GaussianDiffusion(torch.nn.Identity(), image_size=32, num_frames=7, sampling_timesteps=10,
                          timesteps=1000).to(DEV)
    B = 3
    gen = torch.Generator(device=DEV).manual_seed(n)
    x1, x2 = torch.randn(B, n, device=DEV, generator=gen), torch.randn(B, n, device=DEV, generator=gen) * 0.5
    noise = torch.randn(2, B, n, device=DEV, generator=gen)
    acp, a1m = d.sqrt_alphas_cumprod, d.sqrt_one_minus_alphas_cumprod
    seeds = [5, 2 ** 40 + 1, -9]
    for t in (999, 500, 1, 0):
        for lam in (0.5, 0.3, 0.0, 1.0, 1.7, -0.25):
            ref = _torch_mix(d, x1, x2, t, lam, noise[0], noise[1])
            out = torch.empty_like(x1)
            ops.q_interpolate(ops.IMMEDIATE, x1, x2, t, None, noise, acp, a1m, 1.0 - lam, lam, out)
            assert torch.equal(bits(out), bits(ref)), (t, lam)
        e1, e2 = _interp_eps(seeds, (B, n), t)
        for b, s in enumerate(seeds):
            for e, stream in ((e1, 4), (e2, 5)):
                want = _philox_normals(s, n, t, stream)
                got = e[b].double().cpu().numpy()
                assert np.abs(got - want).max() <= 2e-5 * max(1.0, np.abs(want).max()), (t, s, stream)
        assert not torch.equal(e1, e2)
        out = torch.empty_like(x1)
        ops.q_interpolate(ops.IMMEDIATE, x1, x2, t, torch.tensor(seeds, device=DEV), None, acp, a1m, 0.7, 0.3, out)
        assert torch.equal(bits(out), bits(_torch_mix(d, x1, x2, t, 0.3, e1, e2))), t


# ------------------------------------------------------------------------------------------------ GPU: the loops
def _mini(S, T):
    from extdm_b200.unet import Unet3D
    from extdm_b200.weights import synth_state_dict
    fx = torch.load(os.path.join(GOLD, "ddim_ada_c2p5.pt"))
    u = Unet3D(dim=64, channels=512, dim_mults=fx["dim_mults"], cond_num=fx["tc"], pred_num=fx["tp"],
               architecture=fx["variant"]).cuda()
    sd = synth_state_dict(fx["manifest"], fx["weight_seed"])
    assert not u.load_state_dict(sd, strict=False).unexpected_keys
    d = GaussianDiffusion(u, image_size=32, num_frames=fx["tc"] + fx["tp"], sampling_timesteps=S, timesteps=T,
                          loss_type="l2", null_cond_prob=0.0).cuda()
    return d, sd, fx


def _inputs(fx, B=None):
    B = B or fx["B"]
    x = _rnd((B, 3, fx["tc"], 32, 32), fx["input_seed"] + 2, 0.5)
    fea = _rnd((B, 256, fx["tc"] + fx["tp"], 16, 16), fx["input_seed"] + 3, 0.5).abs()
    shape = (B, 3, fx["tp"], 32, 32)
    x1 = _rnd(shape, fx["input_seed"] + 4, 0.5).clamp(-1, 1)
    x2 = _rnd(shape, fx["input_seed"] + 5, 0.5).clamp(-1, 1)
    return x.cuda(), fea.cuda(), x1.cuda(), x2.cuda()


def _oracle(sd, fx):
    from oracle import extdm_oracle as O
    return O, O.SD({"denoise_fn." + k: v for k, v in sd.items()}).sub("denoise_fn"), O.unet_config("ada", fx["tc"],
                                                                                                  fx["tp"])


def _check_graph_eager(d, args, kw, eager):
    d.use_cuda_graph = True
    g1 = d.interpolate(*args, **kw)
    g2 = d.interpolate(*args, **kw)
    d.use_cuda_graph = False
    assert torch.equal(g1, eager), "graphed and eager loops differ"
    assert torch.equal(g1, g2), "graph replay is not deterministic"


@pytest.mark.gpu
def test_interp_ancestral_matches_reference():
    """T = 20, t = 13, injected noise: p_sample at i = 12 .. 0 on the oracle's UNet and the restated schedule of
    tests/test_ddpm.py; graph == eager == a second replay; t = 0 is the mix."""
    from test_ddpm import ddpm_step, schedule_tables
    torch.set_num_threads(8)
    T, t, lam = 20, 13, 0.3
    d, sd, fx = _mini(T, T)
    x, fea, x1, x2 = _inputs(fx)
    shape = x1.shape
    noise = torch.stack([_rnd(shape, fx["noise_seed"] + i) for i in range(2 + t)])
    d.use_cuda_graph = False
    eager = d.interpolate(x1, x2, x, fea, t=t, lam=lam, noise=noise.cuda()).cpu()
    O, unet, cfg = _oracle(sd, fx)
    tab = schedule_tables(T)
    img = _torch_mix(d, x1.cpu(), x2.cpu(), t, lam, noise[0], noise[1])
    with torch.no_grad():
        for j, i in enumerate(reversed(range(t))):            # the reference quirk: mixed at t, denoised from t - 1
            pred = O.unet_forward(unet, cfg, img, torch.full((shape[0],), i, dtype=torch.long), x.cpu(), fea.cpu())
            img, _, _ = ddpm_step(tab, img, pred, i, noise[2 + j])
    r = rel_l2(eager, img)
    print("ancestral interpolate rel-L2", r)
    assert r <= 2e-2, r
    assert eager.abs().max() <= 1.0
    _check_graph_eager(d, (x1, x2, x, fea), dict(t=t, lam=lam, noise=noise.cuda()), eager.cuda())
    for graph in (True, False):
        d.use_cuda_graph = graph
        zero = d.interpolate(x1, x2, x, fea, t=0, lam=lam, noise=noise[:2].cuda())
        assert torch.equal(bits(zero), bits(_torch_mix(d, x1, x2, 0, lam, noise[0].cuda(), noise[1].cuda())))
    d.use_cuda_graph = True


@pytest.mark.gpu
def test_interp_ancestral_shares_p_sample_loop_graph_and_noise():
    """Seeded ancestral interpolation replays p_sample_loop's captured iteration from row T - t, and its loop noise at
    timestep tau is p_sample_loop's with the same seed: feeding the same draws as injected noise gives the same output.
    p_sample_loop is unchanged around it."""
    T, t = 20, 9
    d, _, fx = _mini(T, T)
    x, fea, x1, x2 = _inputs(fx)
    shape, B = x1.shape, x1.shape[0]
    seeds = torch.tensor([17, 2 ** 50 + 5][:B])
    before = d.p_sample_loop(x, shape, fea, seeds=seeds)
    r = d.denoise_fn.runner(B, 32, 32, fea.shape[-1])
    n_graphs = sum(k[0] == "ddpm" for k in r.graphs)
    got = d.interpolate(x1, x2, x, fea, t=t, lam=0.6, seeds=seeds)
    assert sum(k[0] == "ddpm" for k in r.graphs) == n_graphs      # the same captured iteration
    from test_ddpm import _draws
    n = math.prod(shape[1:])
    e1, e2 = _interp_eps(seeds, shape, t, T)
    loop = [_draws(seeds.tolist(), n, T - t + j).view(shape) for j in range(t)]   # row of timestep t - 1 - j
    noise = torch.stack([e1, e2] + loop)
    assert torch.equal(d.interpolate(x1, x2, x, fea, t=t, lam=0.6, noise=noise), got)
    assert torch.equal(d.p_sample_loop(x, shape, fea, seeds=seeds), before)


@pytest.mark.gpu
def test_interp_ddim_matches_reference():
    """S = 5, t = 600, injected noise: DDIM steps over interp_times(600) on the oracle's UNet and ddim_step; graph ==
    eager == a second replay; the lambda sweep equals single calls; lam = 0 / 1 ignore x2 / x1."""
    torch.set_num_threads(8)
    S, t = 5, 600
    d, sd, fx = _mini(S, 1000)
    x, fea, x1, x2 = _inputs(fx)
    shape = x1.shape
    noise = torch.stack([_rnd(shape, fx["noise_seed"] + i) for i in range(2 + S - 1)])
    d.use_cuda_graph = False
    eager = d.interpolate(x1, x2, x, fea, t=t, lam=0.5, noise=noise.cuda()).cpu()
    O, unet, cfg = _oracle(sd, fx)
    tab = O.cosine_schedule_tables(1000)
    img = _torch_mix(d, x1.cpu(), x2.cpu(), t, 0.5, noise[0], noise[1])
    grid = list(reversed(_linspace_int(t, S)))
    with torch.no_grad():
        for i, (time, time_next) in enumerate(zip(grid[:-1], grid[1:])):
            pred = O.unet_forward(unet, cfg, img, torch.full((shape[0],), time, dtype=torch.long), x.cpu(), fea.cpu())
            img, _, _ = O.ddim_step(tab, img, pred, time, time_next, noise[2 + i] if time_next > 0 else None,
                                    d.ddim_sampling_eta)
    r = rel_l2(eager, img)
    print("DDIM interpolate rel-L2", r)
    assert r <= 2e-2, r
    assert eager.abs().max() <= 1.0
    _check_graph_eager(d, (x1, x2, x, fea), dict(t=t, lam=0.5, noise=noise.cuda()), eager.cuda())
    d.use_cuda_graph = True
    lams = [0.0, 0.25, 1.0]
    sweep = d.interpolate(x1, x2, x, fea, t=t, lam=lams, noise=noise.cuda())
    assert sweep.shape == (3, *shape)
    for k, v in enumerate(lams):
        assert torch.equal(sweep[k], d.interpolate(x1, x2, x, fea, t=t, lam=v, noise=noise.cuda())), v
    other = _rnd(shape, 77, 0.5).cuda()
    assert torch.equal(bits(d.interpolate(x1, other, x, fea, t=t, lam=0.0, noise=noise.cuda())), bits(sweep[0]))
    assert torch.equal(bits(d.interpolate(other, x2, x, fea, t=t, lam=1.0, noise=noise.cuda())), bits(sweep[2]))
    assert not torch.equal(sweep[0], sweep[2])


@pytest.mark.gpu
@pytest.mark.parametrize("S", [5, 20])
def test_interp_seeds_graph_cache(S):
    """Seeds: graph == eager, one capture for two seed vectors, a sweep equals single calls, video b alone against the
    batch of 3 within the batch-independence gate, default seeds from torch's generator."""
    T = 1000 if S < 20 else 20
    t = 700 if S < 20 else 15
    d, _, fx = _mini(S, T)
    x, fea, x1, x2 = _inputs(fx, 3)
    seeds = torch.tensor([31, 2 ** 40 + 3, 7])
    d.use_cuda_graph = False
    eager = d.interpolate(x1, x2, x, fea, t=t, lam=0.4, seeds=seeds)
    d.use_cuda_graph = True
    assert torch.equal(d.interpolate(x1, x2, x, fea, t=t, lam=0.4, seeds=seeds), eager)
    r = d.denoise_fn.runner(3, 32, 32, fea.shape[-1])
    kind = "interp" if S < 20 else "ddpm"
    n_graphs = sum(k[0] == kind for k in r.graphs)
    again = d.interpolate(x1, x2, x, fea, t=t, lam=0.4, seeds=(seeds + 1).cuda())
    assert sum(k[0] == kind for k in r.graphs) == n_graphs and not torch.equal(again, eager)
    sweep = d.interpolate(x1, x2, x, fea, t=t, lam=[0.4, 0.9], seeds=seeds)
    assert torch.equal(sweep[0], eager)
    assert torch.equal(sweep[1], d.interpolate(x1, x2, x, fea, t=t, lam=0.9, seeds=seeds))
    k = 1
    alone = d.interpolate(x1[k:k + 1], x2[k:k + 1], x[k:k + 1], fea[k:k + 1], t=t, lam=0.4, seeds=seeds[k:k + 1])
    dd = rel_l2(alone[0], eager[k])
    print(f"S={S}: video alone vs in a batch of 3: rel-L2 {dd:.3e}")
    assert dd <= 2e-2, dd
    torch.manual_seed(4)
    drawn = torch.randint(0, 2 ** 62, (3,), dtype=torch.long)
    torch.manual_seed(4)
    assert torch.equal(d.interpolate(x1, x2, x, fea, t=t, lam=0.4),
                       d.interpolate(x1, x2, x, fea, t=t, lam=0.4, seeds=drawn))


# ------------------------------------------------------------------------------------------------ GPU: the pipeline
def _clips(B, T, hw, seed):
    """Smooth grey clips (B, 3, T, hw, hw) in [0, 1]."""
    import torch.nn.functional as F
    coarse = torch.rand((B, 1, 4, 8, 8), generator=torch.Generator().manual_seed(seed))
    clip = F.interpolate(coarse, size=(T, hw, hw), mode="trilinear", align_corners=True).clamp(0, 1)
    return clip.expand(B, 3, T, hw, hw).contiguous()


def _psnr(a, b):
    mse = ((a.float() - b.float()) ** 2).mean().item()
    return 99.0 if mse == 0 else 10 * math.log10(1.0 / mse)


@pytest.mark.gpu
def test_pipeline_interpolation():
    """FlowDiffusion on KTH (DDIM, synthetic weights): decoding encode_future matches the FlowAE reconstruction from
    source tc - 1; interpolate_one_video returns sample_one_video's keys and shapes (with a leading K axis for a sweep);
    a 2-way sharded evaluate.interpolate_videos against one call."""
    from extdm_b200 import configs, evaluate
    from extdm_b200.flow_autoenc import FlowAE
    from extdm_b200.flow_diffusion import x_start_to_flow
    from extdm_b200.sharding import shard_range
    model, cfg = configs.build_model("kth", device="cuda")
    tc, tp, hw = model.cond_frame_num, model.pred_frame_num, cfg["dataset_params"]["frame_shape"]
    vids = _clips(3, tc + tp, hw, 21).cuda()

    x1 = model.encode_future(vids)
    grid, conf = x_start_to_flow(x1, model.use_residual_flow, model.estimate_occlusion_map)
    dec, _ = model.generator.decode_video(vids[:, :, tc - 1], grid, conf)
    rec = FlowAE.from_flow_diffusion(model).reconstruct(vids, tc - 1)["prediction"][:, :, tc:]
    p = _psnr(dec, rec)
    print(f"decode(encode_future) vs FlowAE reconstruction: PSNR {p:.1f} dB")
    assert p >= 35.0, p

    x2 = model.diffusion.sample(*model.condition(vids[:, :, :tc].contiguous())[1:3], seeds=[1, 2, 3])
    ref = model.sample_one_video(cond_scale=1.0, real_vid=vids[:, :, :tc].contiguous(), seeds=[1, 2, 3])
    one = model.interpolate_one_video(vids, x1, x2, lam=0.5, seeds=[4, 5, 6])
    assert set(one) == set(ref) and all(one[k].shape == ref[k].shape for k in ref)
    assert all(torch.isfinite(v).all() for v in one.values())
    sweep = model.interpolate_one_video(vids, x1, x2, lam=[0.0, 0.5], seeds=[4, 5, 6])
    assert set(sweep) == set(ref)
    for k in ref:
        want = ref[k].shape if not k.startswith("sample_") else (2, *ref[k].shape)
        assert sweep[k].shape == want, k
    assert torch.equal(sweep["sample_out_vid"][1], one["sample_out_vid"])

    lams = [0.0, 0.5, 1.0]
    origin, whole = evaluate.interpolate_videos(model, vids, x1, x2, lams, t=500, seed=11)
    assert origin.shape == whole.shape == (3, 3, tc + tp, 3, hw, hw)
    parts = []
    for rank in range(2):
        lo, hi = shard_range(3, rank, 2)
        parts.append(evaluate.interpolate_videos(model, vids[lo:hi], x1[lo:hi], x2[lo:hi], lams, t=500, seed=11,
                                                 video_offset=lo)[1])
    p = _psnr(torch.cat(parts), whole)
    print(f"sharded interpolate_videos vs one call: frames PSNR {p:.1f} dB")
    assert p >= 35.0, p
    assert evaluate.psnr_videos(origin[:, 0], whole[:, 0]).shape == (3, tc + tp)
