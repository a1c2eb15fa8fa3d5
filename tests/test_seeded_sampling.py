"""Per-video seeded noise: sharding.video_seeds, the seeds argument of the samplers and of the layers above them, and
the seeded DDIM update kernel (csrc/sampler.cu extdm_ddim_update_seeded).

CPU: the seed derivation pinned to literal values and to a plain-integer restatement, its range, collisions and shard
invariance; argument errors of the samplers.  GPU (-m gpu): the kernel bit-exact against extdm_ddim_update fed the
same Philox draws; whole DDIM samples with seeds against the same noise materialised; batch independence; sharded
evaluation against one call; DDPM with given seeds against the seeds it draws itself.
"""
import math
import os

import pytest
import torch

import extdm_b200  # noqa: F401
from extdm_b200.diffusion import GaussianDiffusion
from extdm_b200.sharding import shard_range, video_seeds

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
M64 = (1 << 64) - 1


def _mix(x):
    """splitmix64 step in plain Python integers, as the video_seeds docstring defines it."""
    z = (x + 0x9E3779B97F4A7C15) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def _seed(base, vid, rnd):
    return _mix(_mix(_mix(base & M64) ^ (vid & M64)) ^ (rnd & M64)) >> 2


# ------------------------------------------------------------------------------------------------ CPU
def test_video_seeds_pinned():
    assert video_seeds(0, [0, 1, 2], 0).tolist() == [639684247392563108, 1241144531990192108, 3853996520026480137]
    assert video_seeds(1234, [0, 1, 2], 1).tolist() == [3258528608928783821, 3916341209392686688,
                                                         2082537131308896733]
    assert video_seeds([5, 6], [0, 0], 3).tolist() == [580684757513770505, 3216330469352456121]
    for base, vid, rnd in ((0, 0, 0), (-1, 7, 0), (2 ** 63 - 1, 10 ** 12, 5), (42, 3, 2 ** 40)):
        assert video_seeds(base, [vid], rnd).tolist() == [_seed(base, vid, rnd)]
    per_video = video_seeds(torch.tensor([9, -9, 9]), torch.tensor([4, 4, 5]), 1)
    assert per_video.tolist() == [_seed(9, 4, 1), _seed(-9, 4, 1), _seed(9, 5, 1)]
    assert video_seeds(torch.tensor([9, -9]), 0, 2).tolist() == [_seed(9, 0, 2), _seed(-9, 0, 2)]   # as rollout
    with pytest.raises(ValueError):
        video_seeds([1, 2], [0, 1, 2])


def test_video_seeds_range_and_collisions():
    ids = torch.arange(50_000)
    s = torch.cat([video_seeds(2024, ids, 0), video_seeds(2024, ids, 1)])          # 10^5 (id, round) pairs
    assert s.dtype == torch.int64 and s.shape == (100_000,)
    assert int(s.min()) >= 0 and int(s.max()) < 2 ** 62
    assert torch.unique(s).numel() == s.numel()


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_video_seeds_shard_invariant(world):
    n, base = 29, 77
    whole = video_seeds(base, range(n), 1)
    parts = [video_seeds(base, range(*shard_range(n, r, world)), 1) for r in range(world)]
    assert torch.equal(torch.cat(parts), whole)


class _RecordingModel(torch.nn.Module):
    """Stands in for FlowDiffusion on the CPU: records the seeds of every sample_one_video call."""
    cond_frame_num, pred_frame_num = 2, 3

    def __init__(self):
        super().__init__()
        self.w = torch.nn.Parameter(torch.zeros(1))
        self.calls = []

    def sample_one_video(self, cond_scale, real_vid, noise=None, seeds=None):
        self.calls.append(None if seeds is None else seeds.clone())
        B, _, _, H, W = real_vid.shape
        return {"sample_out_vid": torch.zeros(B, 3, self.cond_frame_num + self.pred_frame_num, H, W)}


def test_evaluation_seeds_follow_global_video_index():
    """sample_videos(seed, video_offset) -> rollout -> sample_one_video: repeat k of video b samples round r with
    video_seeds(video_seeds(seed, (video_offset + b) * n + k), 0, r), on one call or on shards."""
    from extdm_b200 import configs, evaluate
    vids, n, base = torch.zeros(5, 3, 4, 8, 8), 2, 31
    m = _RecordingModel()
    evaluate.sample_videos(m, vids, total_pred=6, num_sample_video=n, seed=base)          # 2 rounds
    assert len(m.calls) == 2
    for r, got in enumerate(m.calls):
        per_video = [_seed(base, i, 0) for i in range(5 * n)]
        assert got.tolist() == [_seed(p, 0, r) for p in per_video]
    whole = list(m.calls)
    for world in (2, 3):
        m.calls = []
        for rank in range(world):
            lo, hi = shard_range(5, rank, world)
            evaluate.sample_videos(m, vids[lo:hi], total_pred=6, num_sample_video=n, seed=base, video_offset=lo)
        for r in range(2):
            assert torch.equal(torch.cat(m.calls[r::2]), whole[r]), (world, r)
    assert not (whole[0] == whole[1]).any()
    m.calls = []
    evaluate.sample_videos(m, vids, total_pred=6, num_sample_video=n)
    assert m.calls == [None, None]
    with pytest.raises(ValueError):
        configs.rollout(m, vids[:, :, :2], 3, seeds=[1, 2])
    with pytest.raises(ValueError):
        configs.rollout(m, vids[:, :, :2], 3, seeds=list(range(5)), noise_fn=lambda: None)


def _cpu_diffusion(sampling_timesteps):
    from extdm_b200.unet import Unet3D
    u = Unet3D(dim=64, channels=512, dim_mults=(1, 2, 4, 4), cond_num=2, pred_num=5)
    return GaussianDiffusion(u, image_size=32, num_frames=7, sampling_timesteps=sampling_timesteps, timesteps=20)


@pytest.mark.parametrize("sampling", [10, None])
def test_seed_argument_errors(sampling):
    d = _cpu_diffusion(sampling)
    x, fea = torch.zeros(2, 3, 2, 32, 32), torch.zeros(2, 256, 7, 16, 16)
    noise = torch.zeros(21, 2, 3, 5, 32, 32)
    bad = {"noise and seeds": dict(noise=noise, seeds=[1, 2]), "length": dict(seeds=[1, 2, 3]),
           "tensor length": dict(seeds=torch.tensor([1])), "dtype": dict(seeds=torch.tensor([1.0, 2.0])),
           "int32": dict(seeds=torch.tensor([1, 2], dtype=torch.int32)), "floats": dict(seeds=[1.5, 2.5]),
           "2-D": dict(seeds=torch.tensor([[1, 2]]))}
    for what, kw in bad.items():
        with pytest.raises(ValueError):
            d.sample(x, cond_fea=fea, **kw)
        print("rejected:", what)
    with pytest.raises(RuntimeError) as e:                                   # valid seeds reach the CUDA-only refusal
        d.sample(x, cond_fea=fea, seeds=[1, 2])
    assert not isinstance(e.value, (ValueError, NotImplementedError))


# ------------------------------------------------------------------------------------------------ GPU helpers
DEV = "cuda"


def _ops():
    from extdm_b200 import ops
    return ops, ops.IMMEDIATE


def _draws(seeds, n, step=None):
    """x_T (step None) or the loop noise of `step` for each seed, (len(seeds), n), from the DDPM kernels."""
    ops, R = _ops()
    sd = torch.as_tensor(seeds, dtype=torch.long).to(DEV)
    out = torch.empty(len(sd), n, device=DEV)
    if step is None:
        ops.ddpm_fill_normal(R, sd, out)
        return out
    rows = torch.tensor([[0.0, 0.0, 0.0, 0.0, 1.0]] * (step + 1), device=DEV)   # img_out = 0 + 1 * z
    zero = torch.zeros(len(sd), n, device=DEV)
    ops.ddpm_update(R, zero, zero, rows, torch.full((1,), step, dtype=torch.int32, device=DEV), sd, None,
                    torch.ones(len(sd), device=DEV), out)
    return out


def _noise_for(seeds, shape, steps):
    """The (steps, *shape) noise tensor ddim_sample(noise=...) needs to reproduce ddim_sample(seeds=seeds)."""
    n = math.prod(shape[1:])
    out = [_draws(seeds, n).view(shape)]
    out += [_draws(seeds, n, i).view(shape) for i in range(steps - 1)]
    return torch.stack(out)


def bits(t):
    return t.contiguous().view(torch.int32)


def rel_l2(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm()).item()


def psnr(a, b):
    mse = ((a.float() - b.float()) ** 2).mean().item()
    return 99.0 if mse == 0 else 10 * math.log10(1.0 / mse)


# ------------------------------------------------------------------------------------------------ GPU: kernel
@pytest.mark.gpu
@pytest.mark.parametrize("tp", [5, 10, 20])
@pytest.mark.parametrize("eta", [1.0, 0.0])
def test_seeded_update_bit_exact(tp, eta):
    """extdm_ddim_update_seeded == extdm_ddim_update fed the materialised Philox draws, img_out and x_start_out,
    several steps, repeated and permuted seeds; at eta = 0 sigma * z is a signed zero in both."""
    ops, R = _ops()
    d = GaussianDiffusion(torch.nn.Identity(), image_size=32, num_frames=2 + tp, sampling_timesteps=10,
                          timesteps=1000, ddim_sampling_eta=eta)
    sched = d.ddim_schedule()
    seeds = torch.tensor([7, 12345, 7, -3, 2 ** 62 + 1], dtype=torch.long, device=DEV)
    B, n = seeds.numel(), 3 * tp * 32 * 32
    gen = torch.Generator(device=DEV).manual_seed(tp)
    img, pred = torch.randn(B, n, device=DEV, generator=gen), torch.randn(B, n, device=DEV, generator=gen)
    img[1] *= 0.2                                                      # a sample whose threshold clamps to 1
    pred[1] *= 0.2
    for step in (0, 3, 8):
        _, _, c_recip, c_recipm1, san, c, sigma = sched[step]
        assert (sigma == 0.0) == (eta == 0.0)
        s = torch.zeros(B, device=DEV)
        ops.ddim_threshold(R, img, pred, c_recip, c_recipm1, 0.9, s)
        z = _draws(seeds, n, step)
        ref, ref_xs = torch.empty_like(img), torch.empty_like(img)
        ops.ddim_update(R, img, pred, z, s, c_recip, c_recipm1, san, c, sigma, ref, ref_xs)
        out, xs = torch.empty_like(img), torch.empty_like(img)
        ops.ddim_update_seeded(R, img, pred, seeds, step, s, c_recip, c_recipm1, san, c, sigma, out, xs)
        assert torch.equal(bits(out), bits(ref)) and torch.equal(bits(xs), bits(ref_xs)), step
        assert torch.equal(z[0], z[2]) and not torch.equal(z[0], z[1])     # repeated seed, same draw
        perm = torch.tensor([3, 0, 4, 2, 1], device=DEV)
        out_p = torch.empty_like(img)
        ops.ddim_update_seeded(R, img[perm].contiguous(), pred[perm].contiguous(), seeds[perm].contiguous(), step,
                               s[perm].contiguous(), c_recip, c_recipm1, san, c, sigma, out_p)
        assert torch.equal(bits(out_p), bits(out[perm]))
    with pytest.raises(ValueError):
        ops.ddim_update_seeded(R, img, pred, seeds[:2].contiguous(), 0, s, 1.0, 1.0, 1.0, 1.0, 1.0, out)
    with pytest.raises(ValueError):
        ops.ddim_update_seeded(R, img, pred, seeds.int(), 0, s, 1.0, 1.0, 1.0, 1.0, 1.0, out)


# ------------------------------------------------------------------------------------------------ GPU: DDIM sample
def _mini_unet():
    from extdm_b200.unet import Unet3D
    from extdm_b200.weights import synth_state_dict
    fx = torch.load(os.path.join(GOLD, "ddim_ada_c2p5.pt"))
    u = Unet3D(dim=64, channels=512, dim_mults=fx["dim_mults"], cond_num=fx["tc"], pred_num=fx["tp"],
               architecture=fx["variant"]).cuda()
    assert not u.load_state_dict(synth_state_dict(fx["manifest"], fx["weight_seed"]), strict=False).unexpected_keys
    return u, fx


def _rnd(shape, seed, scale=1.0):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed)) * scale


@pytest.mark.gpu
def test_ddim_sample_seeds_equal_materialised_noise_graph_cache():
    u, fx = _mini_unet()
    B, tc, tp, S = fx["B"], fx["tc"], fx["tp"], fx["sampling"]
    diff = GaussianDiffusion(u, image_size=32, num_frames=tc + tp, sampling_timesteps=S, timesteps=1000,
                             loss_type="l2", null_cond_prob=0.0).cuda()
    x = _rnd((B, 3, tc, 32, 32), fx["input_seed"] + 2, 0.5).cuda()
    fea = _rnd((B, 256, tc + tp, 16, 16), fx["input_seed"] + 3, 0.5).abs().cuda()
    shape = (B, 3, tp, 32, 32)
    seeds = torch.arange(B, dtype=torch.long) * 1000003 + 5
    noise = _noise_for(seeds, shape, S)
    diff.use_cuda_graph = False
    ref = diff.ddim_sample(x, shape, fea, noise=noise)
    eager = diff.ddim_sample(x, shape, fea, seeds=seeds)
    assert torch.equal(eager, ref), "eager: seeds differ from the materialised noise"
    trace = []
    diff.ddim_sample(x, shape, fea, seeds=seeds.tolist(), trace=trace)
    assert torch.equal(trace[0]["img_in"], noise[0])
    diff.use_cuda_graph = True
    graphed = diff.ddim_sample(x, shape, fea, seeds=seeds)
    assert torch.equal(graphed, ref), "graphed: seeds differ from the materialised noise"
    r = u.runner(B, 32, 32, fea.shape[-1])
    ddim_keys = lambda: [k for k in r.graphs if k[0] == "ddim"]                 # noqa: E731
    n_graphs = len(ddim_keys())
    assert any(("seeded", True) in k for k in ddim_keys())
    seeds2 = seeds + 99
    again = diff.ddim_sample(x, shape, fea, seeds=seeds2.cuda())              # device seeds, the same graph
    assert len(ddim_keys()) == n_graphs
    diff.use_cuda_graph = False
    fresh = diff.ddim_sample(x, shape, fea, seeds=seeds2)
    assert torch.equal(again, fresh) and not torch.equal(again, graphed)


@pytest.mark.gpu
def test_seeded_sample_is_batch_independent():
    """Video k sampled alone, in [a, k, b] and in [b, a, k]: x_T bit-identical, flow and frames within the gate of
    test_full_batch_is_sample_independent (the GEMM tile widths follow the batch)."""
    import torch.nn.functional as F
    from extdm_b200 import configs
    model, _ = configs.build_model("kth", device="cuda")
    tc, tp = model.cond_frame_num, model.pred_frame_num
    coarse = torch.rand((3, 1, 4, 8, 8), generator=torch.Generator().manual_seed(21))
    clip = F.interpolate(coarse, size=(tc, 64, 64), mode="trilinear", align_corners=True).clamp(0, 1)
    clip = clip.expand(3, 3, tc, 64, 64).contiguous().cuda()
    seeds = torch.tensor([101, 4242, 77], dtype=torch.long)                       # [a, k, b]
    runs = {"alone": [1], "batch": [0, 1, 2], "permuted": [2, 0, 1]}
    got = {}
    for name, idx in runs.items():
        c, s = clip[idx].contiguous(), seeds[idx].contiguous()
        _, x_cond, cond_fea, _ = model.condition(c)
        trace = []
        shape = (len(idx), 3, tp, x_cond.shape[3], x_cond.shape[4])
        model.diffusion.ddim_sample(x_cond, shape, cond_fea, seeds=s, trace=trace)
        ret = model.sample_one_video(1.0, c, seeds=s)
        k = idx.index(1)
        got[name] = (trace[0]["img_in"][k], ret["sample_vid_grid"][k:k + 1], ret["sample_out_vid"][k:k + 1])
    for name in ("batch", "permuted"):
        assert torch.equal(got[name][0], got["alone"][0]), name
        d_flow = rel_l2(got[name][1].cpu(), got["alone"][1].cpu())
        p_img = psnr(got[name][2].cpu(), got["alone"][2].cpu())
        print(f"seed k in {name} vs alone: flow rel-L2 {d_flow:.3e}, frames PSNR {p_img:.1f} dB")
        assert d_flow <= 2e-2 and p_img >= 35.0, (name, d_flow, p_img)


@pytest.mark.gpu
def test_sharded_evaluation_matches_one_call():
    """evaluate.sample_videos on 4 videos x 2 repeats in one call against two shards (video_offset 0 and 2)."""
    import torch.nn.functional as F
    from extdm_b200 import configs, evaluate
    model, _ = configs.build_model("ucf", device="cuda")              # tc 4, tp 8 -> 12 predicted = 2 rounds
    coarse = torch.rand((4, 1, 4, 8, 8), generator=torch.Generator().manual_seed(3))
    vids = F.interpolate(coarse, size=(16, 64, 64), mode="trilinear", align_corners=True).clamp(0, 1)
    vids = vids.expand(4, 3, 16, 64, 64).contiguous()                 # smooth clips, as the gate's calibration
    calls = []
    real = model.diffusion.sample

    def recording(x_cond, cond_fea, seeds=None, **kw):
        calls.append((seeds.clone(), (x_cond.shape[0], 3, model.pred_frame_num, *x_cond.shape[3:])))
        return real(x_cond, cond_fea, seeds=seeds, **kw)

    model.diffusion.sample = recording
    try:
        _, whole = evaluate.sample_videos(model, vids, total_pred=12, num_sample_video=2, seed=11)
        whole_calls, calls[:] = list(calls), []
        lo, hi = shard_range(4, 0, 2)
        _, part0 = evaluate.sample_videos(model, vids[lo:hi], total_pred=12, num_sample_video=2, seed=11,
                                          video_offset=lo)
        lo, hi = shard_range(4, 1, 2)
        _, part1 = evaluate.sample_videos(model, vids[lo:hi], total_pred=12, num_sample_video=2, seed=11,
                                          video_offset=lo)
        shard_calls = list(calls)
        _, again = evaluate.sample_videos(model, vids, total_pred=12, num_sample_video=2, seed=11)
    finally:
        del model.diffusion.sample
    assert len(whole_calls) == 2 and len(shard_calls) == 4                  # 2 rounds per call

    def x_T(seeds, shape):
        return _draws(seeds, math.prod(shape[1:])).view(-1, *shape[1:])

    for rnd in (0, 1):
        a = x_T(*whole_calls[rnd])
        b = torch.cat([x_T(*shard_calls[rnd]), x_T(*shard_calls[2 + rnd])])
        assert torch.equal(bits(a), bits(b)), rnd                      # per (video, repeat), rows b * 2 + k
    assert not (whole_calls[0][0] == whole_calls[1][0]).any()
    assert not torch.equal(x_T(*whole_calls[0]), x_T(*whole_calls[1]))    # rounds 1 and 2 draw different noise
    sharded = torch.cat([part0, part1])
    p1 = psnr(sharded[:, :, 4:12], whole[:, :, 4:12])                  # round 1's predicted frames
    p = psnr(sharded, whole)
    print(f"sharded vs one call: frames PSNR {p:.1f} dB (round 1 {p1:.1f} dB)")
    assert p1 >= 35.0 and p >= 35.0, (p1, p)
    assert torch.equal(again, whole), "a second identical call differs"


# ------------------------------------------------------------------------------------------------ GPU: DDPM
@pytest.mark.gpu
def test_ddpm_given_seeds_equal_drawn_seeds():
    u, fx = _mini_unet()
    B, tc, tp, T = fx["B"], fx["tc"], fx["tp"], 20
    diff = GaussianDiffusion(u, image_size=32, num_frames=tc + tp, sampling_timesteps=T, timesteps=T,
                             loss_type="l2", null_cond_prob=0.0).cuda()
    x = _rnd((B, 3, tc, 32, 32), fx["input_seed"] + 2, 0.5).cuda()
    fea = _rnd((B, 256, tc + tp, 16, 16), fx["input_seed"] + 3, 0.5).abs().cuda()
    shape = (B, 3, tp, 32, 32)
    torch.manual_seed(8)
    seeds = torch.randint(0, 2 ** 62, (B,), dtype=torch.long)                  # the call p_sample_loop makes
    for graphed in (False, True):
        diff.use_cuda_graph = graphed
        torch.manual_seed(8)
        drawn = diff.p_sample_loop(x, shape, fea)
        given = diff.p_sample_loop(x, shape, fea, seeds=seeds)
        assert torch.equal(given, drawn), graphed
        assert not torch.equal(diff.p_sample_loop(x, shape, fea, seeds=seeds + 1), drawn)
