"""DPM-Solver++(2M) sampler: GaussianDiffusion.solver_schedule / dpm_solver_sample and its update kernel
(csrc/sampler.cu extdm_dpmpp_update).

CPU: the coefficient table against an independent float64 restatement, the DDIM eta = 0 identity of the first-order
step, the order of accuracy on Gaussian data (exact probability-flow solution known in closed form), argument errors.
GPU (-m gpu): the kernel bit-exact against torch fp32 ops and against the documented Philox generator; the order of
accuracy through the kernels; the mini UNet loop against a restatement on the oracle UNet; seeds, graph reuse and the
absence of host synchronisation; a full-size BAIR model through FlowDiffusion, rollout and a sharded evaluation; the
default sampler unchanged.
"""
import math
import os

import numpy as np
import pytest
import torch

import extdm_b200  # noqa: F401
from extdm_b200.diffusion import SOLVERS, GaussianDiffusion

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SIGMA_D = 0.1           # std of the Gaussian data of the order-of-accuracy tests


def _diffusion(S, solver="dpmpp_2m", T=1000, denoise_fn=None):
    return GaussianDiffusion(denoise_fn or torch.nn.Identity(), image_size=32, num_frames=7, sampling_timesteps=S,
                             timesteps=T, solver=solver)


def _tables(d):
    return d.sqrt_alphas_cumprod.double().numpy(), d.sqrt_one_minus_alphas_cumprod.double().numpy()


def _restated(d, solver):
    """The coefficients from alpha, sigma alone (no lambda, no expm1): e^{-h} = alpha_i sigma_{i+1} / (sigma_i
    alpha_{i+1}), h = log of its inverse."""
    al, sg = _tables(d)
    times = [row[0] for row in d.ddim_schedule()]
    out, h_prev = [], None
    for i, t in enumerate(times[:-1]):
        t1 = times[i + 1]
        e = al[t] * sg[t1] / (sg[t] * al[t1])                          # e^{-h}
        h = -math.log(e)
        if solver == "dpmpp_2m":
            A, G, N = sg[t1] / sg[t], al[t1] * (1.0 - e), 0.0
        else:
            A, G, N = sg[t1] ** 2 * al[t] / (sg[t] ** 2 * al[t1]), al[t1] * (1.0 - e * e), sg[t1] * math.sqrt(1.0 - e * e)
        B, C = (G, 0.0) if h_prev is None else (G * (1.0 + h / (2.0 * h_prev)), -G * h / (2.0 * h_prev))
        out.append((A, B, C, N))
        h_prev = h
    return times, out


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("S", [1, 2, 5, 10])
@pytest.mark.parametrize("solver", SOLVERS)
def test_solver_schedule_matches_restatement(solver, S):
    d = _diffusion(S, solver)
    sched = d.solver_schedule()
    times, ref = _restated(d, solver)
    assert len(sched) == S and [row[0] for row in sched] == times          # the grid of ddim_schedule
    assert all(a > b for a, b in zip(times, times[1:])) and times[-1] > 0
    for i, (t, c_recip, c_recipm1, A, B, C, N, final) in enumerate(sched):
        assert c_recip == d.sqrt_recip_alphas_cumprod[t].item() and c_recipm1 == d.sqrt_recipm1_alphas_cumprod[t].item()
        assert final == (i == S - 1)
        for v in (A, B, C, N):
            assert np.float32(v) == v                                        # rounded to fp32
        if final:
            continue
        np.testing.assert_allclose([A, B, C, N], ref[i], rtol=2e-7, atol=0.0, err_msg=f"step {i}")
        assert (C == 0.0) == (i == 0)
        assert (N == 0.0) == (solver == "dpmpp_2m")
        assert 0.0 < A < 1.0 and B > 0.0


def test_solver_first_order_step_is_ddim_eta0():
    """With D = the unclipped x0 of x = alpha x0 + sigma eps, the first (order-1) ODE step gives alpha' x0 + sigma' eps."""
    d = _diffusion(10)
    al, sg = _tables(d)
    t, _, _, A, B, C, N, _ = d.solver_schedule()[0]
    t1 = d.solver_schedule()[1][0]
    g = np.random.default_rng(1)
    x0, eps = g.standard_normal(1000) * 0.3, g.standard_normal(1000)
    x = al[t] * x0 + sg[t] * eps
    out = A * x + B * x0
    ref = al[t1] * x0 + sg[t1] * eps
    assert C == 0.0 and N == 0.0
    assert np.linalg.norm(out - ref) <= 1e-6 * np.linalg.norm(ref)


def _gaussian_error(d, t_stop, first_order=False, n=4096):
    """Relative error of the solver's state on reaching t_stop against the exact probability-flow solution, for data
    N(0, SIGMA_D^2 I): D(x, t) = E[x0 | x_t] = alpha SIGMA_D^2 x / v(t), v = alpha^2 SIGMA_D^2 + sigma^2, and the exact flow
    scales x by sqrt(v(t') / v(t)).  The threshold stays inactive (asserted: s = 1).  first_order: C folded into B (the
    order-1 step B = G, C = 0)."""
    al, sg = _tables(d)
    sched = d.solver_schedule()
    v = lambda t: al[t] ** 2 * SIGMA_D ** 2 + sg[t] ** 2                   # noqa: E731
    x = np.random.default_rng(0).standard_normal(n) * math.sqrt(v(sched[0][0]))
    x_T, d_prev = x.copy(), None
    for t, c_recip, c_recipm1, A, B, C, N, final in sched:
        if t == t_stop:
            break
        eps = sg[t] * x / v(t)                                                # the optimal epsilon prediction
        s = max(1.0, float(np.quantile(np.abs(c_recip * x - c_recipm1 * eps), 0.9)))
        assert s == 1.0
        D = al[t] * SIGMA_D ** 2 * x / v(t)
        if first_order:
            B, C = B + C, 0.0
        x = A * x + B * D + (C * d_prev if d_prev is not None else 0.0)
        d_prev = D
    assert t == t_stop
    exact = x_T * math.sqrt(v(t_stop) / v(sched[0][0]))
    return np.linalg.norm(x - exact) / np.linalg.norm(exact)


# S + 1 = 10, 20, 40, 80: the grids nest and all contain t = 100.  The error is measured there rather than at t_{S-1}:
# the last steps of the DDIM grid (t_{S-2} = 2 t_{S-1} while t >> 0.008 T) keep a lambda-step of about log 2 whatever S,
# so an error taken at t_{S-1} does not shrink with S for any solver.
ORDER_STEPS, T_STOP = (9, 19, 39, 79), 100


def observed_orders(errs):
    return [math.log2(a / b) for a, b in zip(errs, errs[1:])]


@pytest.mark.parametrize("first_order", [False, True])
def test_solver_order_of_accuracy(first_order):
    errs = [_gaussian_error(_diffusion(S), T_STOP, first_order) for S in ORDER_STEPS]
    orders = observed_orders(errs)
    print("errors", errs, "observed orders", orders)
    if first_order:
        assert 0.8 <= orders[-1] <= 1.2, orders
    else:
        assert orders[-1] >= 1.8, orders
        assert all(a < b for a, b in zip(errs[1:], errs))


def _cpu_unet():
    from extdm_b200.unet import Unet3D
    return Unet3D(dim=64, channels=512, dim_mults=(1, 2, 4, 4), cond_num=2, pred_num=5)


def test_solver_argument_errors():
    with pytest.raises(ValueError):
        _diffusion(5, "dpmpp_3m")
    d = _diffusion(5, denoise_fn=_cpu_unet(), T=20)
    with pytest.raises(ValueError):
        d.solver = "ddim"
    assert d.solver == "dpmpp_2m"
    x, fea = torch.zeros(2, 3, 2, 32, 32), torch.zeros(2, 256, 7, 16, 16)
    shape = (2, 3, 5, 32, 32)
    for S in (20, 25, 0):                                         # grids that are not strictly decreasing
        d.sampling_timesteps = S
        with pytest.raises(ValueError):
            d.solver_schedule()
        with pytest.raises(ValueError):
            d.sample(x, cond_fea=fea, seeds=[1, 2])
    d.sampling_timesteps = 5
    noise = torch.zeros(5, *shape)
    bad = {"noise and seeds": dict(noise=noise, seeds=[1, 2]), "noise shape": dict(noise=torch.zeros(6, *shape)),
           "noise per step": dict(noise=torch.zeros(shape)), "noise dtype": dict(noise=noise.long()),
           "seed length": dict(seeds=[1, 2, 3]), "seed dtype": dict(seeds=torch.tensor([1, 2], dtype=torch.int32)),
           "float seeds": dict(seeds=[1.5, 2.5])}
    for solver in SOLVERS:
        d.solver = solver
        for what, kw in bad.items():
            with pytest.raises(ValueError):
                d.sample(x, cond_fea=fea, **kw)
            print("rejected:", solver, what)
        for kw in (dict(seeds=[1, 2]), dict(noise=noise), {}):           # valid calls reach the CUDA-only refusal
            with pytest.raises(RuntimeError) as e:
                d.sample(x, cond_fea=fea, **kw)
            assert not isinstance(e.value, (ValueError, NotImplementedError))
    d.solver = None
    with pytest.raises(ValueError):
        d.solver_schedule()


# ------------------------------------------------------------------------------------------------ GPU helpers
DEV = "cuda"


def _ops():
    from extdm_b200 import ops
    return ops, ops.IMMEDIATE


def bits(t):
    return t.contiguous().view(torch.int32)


def rel_l2(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm()).item()


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


def _solver_z(seeds, n, step):
    """The device's stream-3 draw of each seed at `step`: the update with A = B = 0, no C term, N = 1 returns z."""
    ops, R = _ops()
    sd = torch.as_tensor(seeds, dtype=torch.long).to(DEV)
    zero = torch.zeros(len(sd), n, device=DEV)
    out, dd = torch.empty_like(zero), torch.empty_like(zero)
    ops.dpmpp_update(R, zero, zero, None, sd, None, step, torch.ones(len(sd), device=DEV), 0.0, 0.0, 0.0, 0.0, 0.0,
                     1.0, False, out, dd)
    return out


# ------------------------------------------------------------------------------------------------ GPU: kernel
@pytest.mark.gpu
@pytest.mark.parametrize("n", [3072, 15360, 61440])
def test_dpmpp_update_bit_exact(n):
    """Threshold + update against the same torch fp32 ops (each product rounded, sums left to right) at the first,
    a middle and the final step; ODE, SDE with injected z, SDE with Philox z (= the numpy generator, fed through the
    injected path bit for bit); d_out in place over d_prev and img_out over img."""
    ops, R = _ops()
    B = 3
    gen = torch.Generator(device=DEV).manual_seed(n)
    img0, pred0 = torch.randn(B, n, device=DEV, generator=gen), torch.randn(B, n, device=DEV, generator=gen)
    x0_1 = 0.3 * torch.randn(n, device=DEV, generator=gen)
    d_prev = torch.randn(B, n, device=DEV, generator=gen).clamp(-1, 1)
    z_inj = torch.randn(B, n, device=DEV, generator=gen)
    seeds = torch.tensor([5, 2 ** 61 + 7, -11], dtype=torch.long, device=DEV)
    for solver in SOLVERS:
        d = _diffusion(10, solver)
        sched = d.solver_schedule()
        for i in (0, 4, 9):
            t, c_recip, c_recipm1, A, Bc, Cc, N, final = sched[i]
            # sample 1 is x = alpha x0 + sigma eps with pred = eps: its x0 prediction is ~x0 (std 0.3) at every t, so its
            # threshold clamps to 1 whatever c_recip is; samples 0 and 2 are unit noise, whose thresholds exceed 1
            img, pred = img0.clone(), pred0.clone()
            img[1] = d.sqrt_alphas_cumprod[t].item() * x0_1 + d.sqrt_one_minus_alphas_cumprod[t].item() * pred0[1]
            s = torch.zeros(B, device=DEV)
            ops.ddim_threshold(R, img, pred, c_recip, c_recipm1, 0.9, s)
            xs = c_recip * img - c_recipm1 * pred
            s_ref = torch.quantile(xs.abs(), 0.9, dim=-1).clamp_(min=1.0)
            assert torch.equal(s, s_ref) and s_ref[1] == 1.0 and s_ref[0] > 1.0
            D = xs.clamp(-s_ref[:, None], s_ref[:, None]) / s_ref[:, None]
            modes = [("ode", None, None)] if solver == "dpmpp_2m" else [("inj", None, z_inj), ("philox", seeds, None)]
            for mode, sd, nz in modes:
                ref = A * img + Bc * D
                if i:
                    ref = ref + Cc * d_prev
                if mode != "ode" and not final:
                    z = nz if nz is not None else _solver_z(seeds, n, i)
                    if nz is None:                                       # the device draw is the documented one
                        for b in range(B):
                            want = _philox_normals(int(seeds[b]), n, i, 3)
                            got = z[b].double().cpu().numpy()
                            assert np.abs(got - want).max() <= 2e-5 * max(1.0, np.abs(want).max())
                    ref = ref + N * z
                if final:
                    ref = D
                x_io, d_io = img.clone(), d_prev.clone()
                ops.dpmpp_update(R, x_io, pred, d_io if i else None, sd, nz, i, s, c_recip, c_recipm1, A, Bc, Cc, N,
                                 final, x_io, d_io)
                assert torch.equal(bits(d_io), bits(D)), (solver, i, mode)
                assert torch.equal(bits(x_io), bits(ref)), (solver, i, mode)
                if final:
                    assert x_io.abs().max() <= 1.0
    with pytest.raises(ValueError):
        ops.dpmpp_update(R, img, pred, None, seeds, z_inj, 1, s, 1.0, 1.0, 1.0, 1.0, 0.0, 1.0, False, img, d_prev)
    with pytest.raises(ValueError):
        ops.dpmpp_update(R, img, pred, None, seeds.int(), None, 1, s, 1.0, 1.0, 1.0, 1.0, 0.0, 1.0, False, img, d_prev)


@pytest.mark.gpu
def test_solver_order_on_device():
    """_gaussian_error's experiment through ddim_threshold + dpmpp_update in fp32, epsilon computed by torch between
    the launches."""
    ops, R = _ops()
    n = 4 * 4096
    errs = {False: [], True: []}
    for first_order in (False, True):
        for S in ORDER_STEPS:
            d = _diffusion(S)
            al, sg = d.sqrt_alphas_cumprod.to(DEV), d.sqrt_one_minus_alphas_cumprod.to(DEV)
            v = lambda t: al[t] ** 2 * SIGMA_D ** 2 + sg[t] ** 2              # noqa: E731
            sched = d.solver_schedule()
            g = torch.Generator(device=DEV).manual_seed(0)
            x = torch.randn(1, n, device=DEV, generator=g) * v(sched[0][0]).sqrt()
            x_T, dd, s = x.clone(), torch.zeros_like(x), torch.zeros(1, device=DEV)
            for i, (t, c_recip, c_recipm1, A, Bc, Cc, N, final) in enumerate(sched):
                if t == T_STOP:
                    break
                eps = (sg[t] * x / v(t)).contiguous()
                ops.ddim_threshold(R, x, eps, c_recip, c_recipm1, 0.9, s)
                assert s.item() == 1.0
                if first_order:
                    Bc, Cc = Bc + Cc, 0.0
                ops.dpmpp_update(R, x, eps, dd if i else None, None, None, i, s, c_recip, c_recipm1, A, Bc, Cc, N,
                                 False, x, dd)
            assert t == T_STOP
            exact = x_T.double() * (v(T_STOP).double() / v(sched[0][0]).double()).sqrt()
            errs[first_order].append(((x.double() - exact).norm() / exact.norm()).item())
    print("device errors", errs)
    orders = observed_orders(errs[False])
    assert orders[-1] >= 1.8, orders
    orders = observed_orders(errs[True])
    assert 0.8 <= orders[-1] <= 1.2, orders


# ------------------------------------------------------------------------------------------------ GPU: the loop
def _mini():
    from extdm_b200.unet import Unet3D
    from extdm_b200.weights import synth_state_dict
    fx = torch.load(os.path.join(GOLD, "ddim_ada_c2p5.pt"))
    u = Unet3D(dim=64, channels=512, dim_mults=fx["dim_mults"], cond_num=fx["tc"], pred_num=fx["tp"],
               architecture=fx["variant"]).cuda()
    sd = synth_state_dict(fx["manifest"], fx["weight_seed"])
    assert not u.load_state_dict(sd, strict=False).unexpected_keys
    return u, sd, fx


def _rnd(shape, seed, scale=1.0):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed)) * scale


def _inputs(fx, B=None):
    B = B or fx["B"]
    x = _rnd((B, 3, fx["tc"], 32, 32), fx["input_seed"] + 2, 0.5)
    fea = _rnd((B, 256, fx["tc"] + fx["tp"], 16, 16), fx["input_seed"] + 3, 0.5).abs()
    return x, fea, (B, 3, fx["tp"], 32, 32)


def _oracle_solver(sd, fx, sched, x_cond, cond_fea, noise, sde):
    """The solver loop restated on the oracle's fp32 UNet, torch ops on the CPU."""
    from oracle import extdm_oracle as O
    unet, cfg = O.SD({"denoise_fn." + k: v for k, v in sd.items()}).sub("denoise_fn"), O.unet_config("ada", fx["tc"],
                                                                                                   fx["tp"])
    img, d_prev, trace = noise[0], None, []
    for i, (t, c_recip, c_recipm1, A, B, C, N, final) in enumerate(sched):
        pred = O.unet_forward(unet, cfg, img, torch.full((img.shape[0],), t, dtype=torch.long), x_cond, cond_fea)
        D, _ = O.dynamic_threshold(c_recip * img - c_recipm1 * pred)
        if final:
            img = D
        else:
            img = A * img + B * D + (C * d_prev if d_prev is not None else 0.0) + (N * noise[1 + i] if sde else 0.0)
        d_prev = D
        trace.append(dict(pred_noise=pred, img=img))
    return img, trace


@pytest.mark.gpu
@pytest.mark.parametrize("solver", SOLVERS)
def test_solver_mini_unet_matches_oracle(solver):
    """S = 5 on the ddim_ada_c2p5 weights and inputs, injected noise, against _oracle_solver; graph == eager == a
    second graphed run, bit for bit."""
    torch.set_num_threads(8)
    u, sd, fx = _mini()
    S = 5
    diff = GaussianDiffusion(u, image_size=32, num_frames=fx["tc"] + fx["tp"], sampling_timesteps=S, timesteps=1000,
                             loss_type="l2", null_cond_prob=0.0, solver=solver).cuda()
    x, fea, shape = _inputs(fx)
    noise = torch.stack([_rnd(shape, fx["noise_seed"] + i) for i in range(S)])
    trace = []
    eager = diff.dpm_solver_sample(x.cuda(), shape, fea.cuda(), noise=noise.cuda(), trace=trace).cpu()
    with torch.no_grad():
        ref, ref_trace = _oracle_solver(sd, fx, diff.solver_schedule(), x, fea, noise, solver == "dpmpp_2m_sde")
    assert len(trace) == len(ref_trace) == S
    per_step = [rel_l2(a["pred_noise"].cpu(), b["pred_noise"]) for a, b in zip(trace, ref_trace)]
    by_step = [rel_l2(a["img"].cpu(), b["img"]) for a, b in zip(trace, ref_trace)]
    r = rel_l2(eager, ref)
    print(solver, "rel-L2", r, "per-step pred_noise", per_step, "img by step", by_step)
    assert max(per_step) <= 2e-2 and max(by_step) <= 2e-2 and r <= 2e-2, (per_step, by_step, r)
    assert torch.equal(trace[-1]["img"].cpu(), eager) and torch.equal(trace[-1]["x_start"].cpu(), eager)
    assert eager.abs().max() <= 1.0
    diff.use_cuda_graph = True
    g1 = diff.sample(x.cuda(), cond_fea=fea.cuda(), noise=noise.cuda()).cpu()
    g2 = diff.sample(x.cuda(), cond_fea=fea.cuda(), noise=noise.cuda()).cpu()
    assert torch.equal(g1, eager), "graphed and eager loops differ"
    assert torch.equal(g1, g2), "graph replay is not deterministic"
    diff.use_cuda_graph = False
    assert torch.equal(diff.sample(x.cuda(), cond_fea=fea.cuda(), noise=noise.cuda()).cpu(), eager)


@pytest.mark.gpu
@pytest.mark.parametrize("solver", SOLVERS)
def test_solver_seeds_graph_cache(solver):
    """Seeds against the injected noise they stand for, batch independence (video b alone vs in a batch of 4), one
    graph for two seed vectors, default seeds from torch's generator."""
    u, _, fx = _mini()
    S = 5
    diff = GaussianDiffusion(u, image_size=32, num_frames=fx["tc"] + fx["tp"], sampling_timesteps=S, timesteps=1000,
                             loss_type="l2", null_cond_prob=0.0, solver=solver).cuda()
    x, fea, shape = _inputs(fx, 4)
    x, fea = x.cuda(), fea.cuda()
    seeds = torch.tensor([31, 2 ** 40 + 3, 7, 99], dtype=torch.long)
    n = math.prod(shape[1:])
    from extdm_b200 import ops
    x_T = torch.empty(4, n, device=DEV)
    ops.ddpm_fill_normal(ops.IMMEDIATE, seeds.cuda(), x_T)
    noise = [x_T.view(shape)] + [_solver_z(seeds, n, i).view(shape) for i in range(S - 1)]
    noise = torch.stack(noise)
    diff.use_cuda_graph = False
    ref = diff.dpm_solver_sample(x, shape, fea, noise=noise)
    assert torch.equal(diff.dpm_solver_sample(x, shape, fea, seeds=seeds), ref)
    diff.use_cuda_graph = True
    graphed = diff.dpm_solver_sample(x, shape, fea, seeds=seeds)
    assert torch.equal(graphed, ref)
    r = u.runner(4, 32, 32, fea.shape[-1])
    n_graphs = sum(k[0] == "solver" for k in r.graphs)
    again = diff.dpm_solver_sample(x, shape, fea, seeds=(seeds + 1).cuda())
    assert sum(k[0] == "solver" for k in r.graphs) == n_graphs and not torch.equal(again, graphed)
    diff.use_cuda_graph = False
    assert torch.equal(diff.dpm_solver_sample(x, shape, fea, seeds=seeds + 1), again)
    k = 2
    trace = []
    alone = diff.dpm_solver_sample(x[k:k + 1].contiguous(), (1, *shape[1:]), fea[k:k + 1].contiguous(),
                                   seeds=seeds[k:k + 1], trace=trace)
    assert torch.equal(trace[0]["img_in"][0], x_T[k].view(shape[1:]))
    d = rel_l2(alone[0], ref[k])
    print(solver, "video alone vs in a batch of 4: rel-L2", d)
    assert d <= 2e-2, d
    torch.manual_seed(4)
    drawn = torch.randint(0, 2 ** 62, (4,), dtype=torch.long)
    torch.manual_seed(4)
    assert torch.equal(diff.sample(x, cond_fea=fea), diff.sample(x, cond_fea=fea, seeds=drawn))


def _bair(solver="dpmpp_2m", S=5):
    from extdm_b200 import configs
    from extdm_b200.flow_diffusion import flow_diffusion_class
    from extdm_b200.weights import synth_state_dict
    cfg, wrapper, arch = configs.dataset("bair")
    mp = cfg["diffusion_params"]["model_params"]
    mp["sampling_timesteps"] = S
    if solver is not None:
        mp["solver"] = solver
    model = flow_diffusion_class(wrapper)(config=cfg, pretrained_pth="", is_train=False, Unet3D_architecture=arch).eval()
    for i, part in enumerate(("generator", "region_predictor", "bg_predictor", "diffusion")):
        m = getattr(model, part)
        base = m.state_dict()
        m.load_state_dict(synth_state_dict({k: tuple(v.shape) for k, v in base.items()}, 1234 + i, base=base))
    return model.cuda()


@pytest.mark.gpu
def test_solver_full_size_bair():
    """FlowDiffusion with diffusion_params.model_params.solver = dpmpp_2m, S = 5: sample_one_video reproducible under
    torch.manual_seed, a seeded call is one graph replay with no host synchronisation, a 2-round rollout with seeds,
    a sharded evaluation against one call."""
    import torch.nn.functional as F
    from extdm_b200 import configs, evaluate, lib
    from extdm_b200.sharding import shard_range
    model = _bair()
    diff = model.diffusion
    assert diff.solver == "dpmpp_2m" and diff.sampling_timesteps == 5
    tc = model.cond_frame_num
    real_vid = torch.rand((2, 3, tc, 64, 64), generator=torch.Generator().manual_seed(9)).cuda()
    torch.manual_seed(0)
    a = model.sample_one_video(cond_scale=1.0, real_vid=real_vid)
    torch.manual_seed(0)
    b = model.sample_one_video(cond_scale=1.0, real_vid=real_vid)
    for k in a:
        assert torch.equal(a[k], b[k]), k
        assert torch.isfinite(a[k]).all(), k
    assert a["sample_vid_grid"][:, :, tc:].abs().max() <= 1.0

    _, x_cond, cond_fea, _ = model.condition(real_vid)
    r = diff.denoise_fn.runner(2, x_cond.shape[3], x_cond.shape[4], cond_fea.shape[-1])
    seeds = torch.tensor([3, 4], dtype=torch.long)
    diff.sample(x_cond, cond_fea=cond_fea, seeds=seeds)                       # capture
    replays = []
    real_replay = torch.cuda.CUDAGraph.replay
    torch.cuda.CUDAGraph.replay = lambda g: (replays.append(g), real_replay(g))[1]
    torch.cuda.synchronize()
    n0 = lib.launches()
    torch.cuda.set_sync_debug_mode("error")
    try:
        pred = diff.sample(x_cond, cond_fea=cond_fea, seeds=seeds + 1)
    finally:
        torch.cuda.set_sync_debug_mode("default")
        torch.cuda.CUDAGraph.replay = real_replay
    # prologue, x_T fill and the S steps are all inside the one replay: no launch is issued around it
    assert lib.launches() - n0 == 0 and len(replays) == 1
    torch.cuda.synchronize()
    assert pred.abs().max() <= 1.0

    clip = torch.rand((2, 3, tc, 64, 64), generator=torch.Generator().manual_seed(5)).cuda()
    out1 = configs.rollout(model, clip, 20, seeds=[11, 12])                    # tp = 10: two rounds
    out2 = configs.rollout(model, clip, 20, seeds=[11, 12])
    assert out1.shape == (2, 3, 20, 64, 64) and torch.equal(out1, out2) and torch.isfinite(out1).all()

    coarse = torch.rand((4, 1, 4, 8, 8), generator=torch.Generator().manual_seed(3))
    vids = F.interpolate(coarse, size=(tc + 20, 64, 64), mode="trilinear", align_corners=True).clamp(0, 1)
    vids = vids.expand(4, 3, tc + 20, 64, 64).contiguous()
    _, whole = evaluate.sample_videos(model, vids, total_pred=20, num_sample_video=2, seed=11)
    parts = []
    for rank in range(2):
        lo, hi = shard_range(4, rank, 2)
        parts.append(evaluate.sample_videos(model, vids[lo:hi], total_pred=20, num_sample_video=2, seed=11,
                                            video_offset=lo)[1])
    sharded = torch.cat(parts)
    mse = ((sharded.float() - whole.float()) ** 2).mean().item()
    p = 99.0 if mse == 0 else 10 * math.log10(1.0 / mse)
    print(f"sharded vs one call: frames PSNR {p:.1f} dB")
    assert p >= 35.0, p


@pytest.mark.gpu
def test_default_sampler_untouched_no_solver_graph():
    """solver=None: DDIM output bit-identical to a model constructed without the argument."""
    u, _, fx = _mini()
    x, fea, shape = _inputs(fx)
    kw = dict(image_size=32, num_frames=fx["tc"] + fx["tp"], sampling_timesteps=fx["sampling"], timesteps=1000,
              loss_type="l2", null_cond_prob=0.0)
    seeds = torch.tensor([1, 2, 3, 4][:fx["B"]], dtype=torch.long)
    with_arg = GaussianDiffusion(u, solver=None, **kw).cuda()
    without = GaussianDiffusion(u, **kw).cuda()
    assert with_arg.solver is None and without.solver is None
    a = with_arg.sample(x.cuda(), cond_fea=fea.cuda(), seeds=seeds)
    b = without.sample(x.cuda(), cond_fea=fea.cuda(), seeds=seeds)
    assert torch.equal(a, b)
    r = u.runner(fx["B"], 32, 32, fea.shape[-1])
    assert not any(k[0] == "solver" for k in r.graphs)
