"""Stage-1 reconstruction (FlowAE.reconstruct, evaluate.reconstruct_videos) and the source-slot sparse-motion kernel
(csrc/lfae_cond.cu extdm_sparse_motion_src).

CPU: the batched torch path against a literal per-frame loop of the LFAE calls, argument and checkpoint errors, the
evaluation layout, the exported symbol.  GPU (-m gpu): the kernel against torch, the CUDA graph against torch fp32 and
against the DM conditioning stage, graph replay against the eager launch lists, batch independence.
"""
import ctypes
import gc
import math

import pytest
import torch
import torch.nn.functional as F

import extdm_b200  # noqa: F401
from extdm_b200 import configs, evaluate, lib
from extdm_b200.flow_autoenc import FlowAE
from extdm_b200.weights import synth_state_dict

PARTS = ("generator", "region_predictor", "bg_predictor")


def make_ae(name, device):
    """FlowAE of a named dataset configuration with the synthetic LFAE weights configs.build_model gives it."""
    cfg = configs.dataset(name)[0]
    ae = FlowAE(cfg)
    for i, part in enumerate(PARTS):
        m = getattr(ae, part)
        base = m.state_dict()
        m.load_state_dict(synth_state_dict({k: tuple(v.shape) for k, v in base.items()}, 1234 + i, base=base))
    return ae.to(device), cfg


def smooth_clip(B, T, hw, seed):
    """Natural-video-like clip: trilinear up-sampling of coarse colour noise, in [0, 1]."""
    coarse = torch.rand((B, 3, max(T // 2, 2), 8, 8), generator=torch.Generator().manual_seed(seed))
    return F.interpolate(coarse, size=(T, hw, hw), mode="trilinear", align_corners=True).clamp(0, 1).contiguous()


def rel_l2(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm()).item()


def psnr(a, b):
    mse = ((a.float() - b.float()) ** 2).mean().item()
    return 99.0 if mse == 0 else 10 * math.log10(1.0 / mse)


# ================================================================================================ CPU
@pytest.fixture(scope="module")
def ae_cpu():
    return make_ae("smmnist", "cpu")[0]


@pytest.mark.parametrize("source_frame", [0, 2])
def test_batched_torch_path_equals_per_frame_loop(ae_cpu, source_frame):
    """The batched torch path of reconstruct is the reference's per-frame LFAE call (generator.py:105-144) repeated
    over frames with the source repeated: region_predictor(source), region_predictor(frame), bg_predictor(source,
    frame), generator(source, ...)."""
    B, T = 2, 4
    vid = smooth_clip(B, T, 64, seed=3)
    got = ae_cpu.reconstruct(vid, source_frame=source_frame)
    assert set(got) == {"prediction", "deformed", "optical_flow", "occlusion_map"}
    want = {k: torch.zeros_like(v) for k, v in got.items()}
    with torch.no_grad():
        for b in range(B):
            src = vid[b:b + 1, :, source_frame]
            for t in range(T):
                frame = vid[b:b + 1, :, t]
                src_params = ae_cpu.region_predictor(src)
                drv_params = ae_cpu.region_predictor(frame)
                bg = ae_cpu.bg_predictor(src, frame)
                out = ae_cpu.generator(src, source_region_params=src_params, driving_region_params=drv_params,
                                       bg_params=bg)
                want["prediction"][b, :, t] = out["prediction"][0]
                want["deformed"][b, :, t] = out["deformed"][0]
                want["optical_flow"][b, :, t] = out["optical_flow"][0].permute(2, 0, 1)
                want["occlusion_map"][b, :, t] = out["occlusion_map"][0]
    assert got["prediction"].shape == (B, 3, T, 64, 64) and got["optical_flow"].shape == (B, 2, T, 32, 32)
    assert got["occlusion_map"].shape == (B, 1, T, 32, 32)
    for k in want:
        err = (got[k] - want[k]).abs().max().item()
        assert err <= 1e-5, (k, err)


def test_argument_errors(ae_cpu):
    vid = torch.rand(1, 3, 3, 64, 64)
    for bad in (3, -1, 1.0, True, None):
        with pytest.raises(ValueError):
            ae_cpu.reconstruct(vid, source_frame=bad)
    with pytest.raises(ValueError):
        ae_cpu.reconstruct(torch.rand(1, 1, 3, 64, 64))                  # wrong channel count
    with pytest.raises(ValueError):
        ae_cpu.reconstruct(torch.rand(3, 3, 64, 64))                     # no time axis
    with pytest.raises(ValueError):
        evaluate.reconstruct_videos(ae_cpu, vid, source_frame=5)


def test_source_frame_takes_any_integer_type(ae_cpu):
    import numpy as np
    vid = smooth_clip(1, 3, 64, seed=5)
    want = ae_cpu.reconstruct(vid, source_frame=2)
    for idx in (np.int64(2), torch.tensor(2)):
        got = ae_cpu.reconstruct(vid, source_frame=idx)
        assert all(torch.equal(got[k], want[k]) for k in want)
    for bad in (torch.tensor(2.0), np.float32(2), np.bool_(True)):
        with pytest.raises(ValueError):
            ae_cpu.reconstruct(vid, source_frame=bad)


def test_dropped_flowae_leaves_shared_modules_loadable():
    """A FlowAE on a FlowDiffusion's modules hooks their load_state_dict; once it is gone the model still loads
    weights, and its hooks are gone with it."""
    model, _ = configs.build_model("smmnist", device="cpu")
    n_hooks = {p: len(getattr(model, p)._load_state_dict_post_hooks) for p in PARTS}
    for _ in range(3):
        ae = FlowAE.from_flow_diffusion(model)
        ae._runners["stale"] = object()
        model.generator.load_state_dict(model.generator.state_dict())
        assert not ae._runners                                        # new weights drop the runners
        assert ae.generator is model.generator                        # shared, not copied
    del ae
    gc.collect()
    assert {p: len(getattr(model, p)._load_state_dict_post_hooks) for p in PARTS} == n_hooks
    model.load_state_dict(model.state_dict())
    model.generator.load_state_dict(model.generator.state_dict())


def test_checkpoint_is_loaded_strictly(tmp_path):
    cfg = configs.dataset("smmnist")[0]
    ae, _ = make_ae("smmnist", "cpu")
    ckpt = {p: {k: v.clone() for k, v in getattr(ae, p).state_dict().items()} for p in PARTS}
    ckpt["optimizer"] = {}                                               # other entries of the checkpoint are ignored
    path = tmp_path / "ae.pth"
    torch.save(ckpt, path)
    loaded = FlowAE(cfg, pretrained_pth=str(path))
    for p in PARTS:
        for k, v in getattr(loaded, p).state_dict().items():
            assert torch.equal(v.cpu(), ckpt[p][k]), (p, k)
        assert not getattr(loaded, p).training
        assert not any(q.requires_grad for q in getattr(loaded, p).parameters())
    missing = {p: dict(v) for p, v in ckpt.items()}
    missing["generator"].pop(next(iter(missing["generator"])))
    extra = {p: dict(v) for p, v in ckpt.items()}
    extra["region_predictor"]["unexpected.weight"] = torch.zeros(1)
    no_part = {p: v for p, v in ckpt.items() if p != "bg_predictor"}
    for name, bad, exc in (("missing", missing, RuntimeError), ("extra", extra, RuntimeError),
                           ("no_part", no_part, KeyError)):
        torch.save(bad, tmp_path / f"{name}.pth")
        with pytest.raises(exc):
            FlowAE(cfg, pretrained_pth=str(tmp_path / f"{name}.pth"))


def test_reconstruct_videos_layout_feeds_the_metrics(ae_cpu, tmp_path):
    """reconstruct_videos returns sample_videos' (B, n=1, T, C, H, W) CPU layout; psnr / ssim / summarize /
    save_results take it unchanged.  One frame per video: the frame is reconstructed from itself."""
    vids = smooth_clip(2, 1, 64, seed=9)
    origin, result = evaluate.reconstruct_videos(ae_cpu, vids)
    assert origin.shape == result.shape == (2, 1, 1, 3, 64, 64)
    assert origin.device.type == result.device.type == "cpu"
    assert torch.equal(origin[:, 0], vids.permute(0, 2, 1, 3, 4))
    assert torch.equal(result[:, 0], ae_cpu.reconstruct(vids)["prediction"].permute(0, 2, 1, 3, 4))
    p, s = evaluate.psnr_videos(origin[:, 0], result[:, 0]), evaluate.ssim_videos(origin[:, 0], result[:, 0])
    assert p.shape == s.shape == (2, 1) and torch.isfinite(p).all() and torch.isfinite(s).all()
    assert "mean" in evaluate.summarize(p)
    evaluate.save_results(str(tmp_path), origin, result)
    assert torch.equal(torch.load(tmp_path / "result_0.pt"), result[:, 0])
    assert torch.equal(torch.load(tmp_path / "origin.pt"), origin[:, 0])


def test_symbol_is_exported():
    assert "extdm_sparse_motion_src" in lib.PROTOTYPES
    assert hasattr(ctypes.CDLL(lib.LIB_PATH), "extdm_sparse_motion_src")
    assert lib.load().extdm_abi_version() == 5
    assert extdm_b200.FlowAE is FlowAE


# ================================================================================================ GPU
def _sparse_motion_inputs(Fn, K, h, w, seed):
    g = torch.Generator().manual_seed(seed)
    img = torch.rand(Fn, 3, h, w, generator=g)
    shift = torch.rand(Fn, K, 2, generator=g) - 0.5
    m = torch.randn(Fn, K, 2, 2, generator=g) * 0.2 + torch.eye(2) * 0.5
    covar = m @ m.transpose(-1, -2) * 0.05 + torch.eye(2) * 0.01
    affine = torch.randn(Fn, K, 2, 2, generator=g) * 0.2 + torch.eye(2)
    bg = torch.eye(3).repeat(Fn, 1, 1)
    bg[:, :2] += torch.randn(Fn, 2, 3, generator=g) * 0.05
    return img, shift, covar, affine, bg


@pytest.mark.gpu
@pytest.mark.parametrize("use_covar,with_bg", [(True, True), (False, False)])
def test_sparse_motion_src_matches_torch(use_covar, with_bg):
    """extdm_sparse_motion_src: slot group-1 is extdm_sparse_motion bit for bit; slots 0 and a middle one match the
    torch PixelwiseFlowPredictor fed the source of frame f from frame f // group * group + src_slot."""
    from extdm_b200 import lfae, ops
    B, group, K, h, w = 2, 4, 10, 16, 16
    Fn = B * group
    img, shift, covar, affine, bg = _sparse_motion_inputs(Fn, K, h, w, seed=6)
    xd = torch.zeros(Fn, h, w, 32, device="cuda")
    xd[..., :3] = img.permute(0, 2, 3, 1).cuda()
    dev = [t.cuda() for t in (shift, covar, affine)] + [bg.cuda() if with_bg else None]
    cpad = 64

    def run(slot):
        inp, motion = torch.empty(Fn, h, w, cpad, device="cuda"), torch.empty(Fn, K + 1, h, w, 2, device="cuda")
        if slot is None:
            ops.sparse_motion(ops.IMMEDIATE, xd, *dev, group, True, use_covar, 0.01, inp, motion)
        else:
            ops.sparse_motion_src(ops.IMMEDIATE, xd, *dev, group, slot, True, use_covar, 0.01, inp, motion)
        torch.cuda.synchronize()
        return inp, motion

    old, new = run(None), run(group - 1)
    assert torch.equal(old[0], new[0]) and torch.equal(old[1], new[1])
    pfp = lfae.PixelwiseFlowPredictor(block_expansion=8, num_blocks=2, max_features=16, num_regions=K, num_channels=3,
                                      estimate_occlusion_map=True, scale_factor=1, use_covar_heatmap=use_covar,
                                      revert_axis_swap=True)
    captured = {}
    pfp.hourglass.register_forward_pre_hook(lambda mod, args: captured.__setitem__("inp", args[0]))
    drv = {"shift": shift, "covar": covar, "affine": affine}
    for slot in (0, 1):
        src_of = torch.arange(Fn) // group * group + slot
        with torch.no_grad():
            pfp(source_image=img[src_of], driving_region_params=drv,
                source_region_params={k: v[src_of] for k, v in drv.items()}, bg_params=bg if with_bg else None)
        inp, _ = run(slot)
        assert torch.count_nonzero(inp[..., 4 * (K + 1):]) == 0
        err = (inp[..., :4 * (K + 1)].cpu() - captured["inp"].permute(0, 2, 3, 1)).abs().max().item()
        assert err <= 2e-3, (slot, err)                                  # tf32-rounded storage of O(1) values
    with pytest.raises(lib.ExtdmError):
        run(group)


@pytest.mark.gpu
@pytest.mark.parametrize("name,B", [("kth", 2), ("ucf", 1), ("bair", 2), ("cityscapes", 1)])
def test_reconstruction_matches_torch_fp32(name, B):
    """The CUDA graph against the torch modules in true fp32 (TF32 off): flow and occlusion as close to fp32 as cuDNN's
    own TF32 path within a factor of two (the gate of test_native_conditioning_matches_torch_fp32), frames >= 35 dB."""
    ae, cfg = make_ae(name, "cuda")
    hw = cfg["dataset_params"]["frame_shape"]
    vid = smooth_clip(B, 6, hw, seed=11).cuda()
    old = torch.backends.cudnn.allow_tf32
    try:
        ae.native = False
        torch.backends.cudnn.allow_tf32 = False
        exact = ae.reconstruct(vid, 0)
        torch.backends.cudnn.allow_tf32 = True
        cudnn_tf32 = ae.reconstruct(vid, 0)
    finally:
        torch.backends.cudnn.allow_tf32 = old
        ae.native = True
    native = ae.reconstruct(vid, 0)
    assert ae._runners, "the CUDA path did not run"
    assert set(native) == set(exact) == {"prediction", "deformed", "optical_flow", "occlusion_map"}
    for k in native:
        assert native[k].shape == exact[k].shape, k
    for key in ("optical_flow", "occlusion_map"):
        e_nat = (native[key] - exact[key]).abs().max().item()
        e_lib = (cudnn_tf32[key] - exact[key]).abs().max().item()
        print(name, key, "native vs fp32", e_nat, "| cuDNN tf32 vs fp32", e_lib)
        assert e_nat <= max(2 * e_lib, 2e-3), (key, e_nat, e_lib)
    for key in ("prediction", "deformed"):
        p = psnr(native[key], exact[key])
        print(name, key, "PSNR vs fp32", p)
        assert p >= 35.0, (key, p)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["kth", "cityscapes"])
def test_reconstruction_flow_equals_dm_conditioning(name):
    """With T = tc and the source at tc - 1, the flow and occlusion of the reconstruction are the DM conditioning
    stage's, bit for bit."""
    model, cfg = configs.build_model(name, device="cuda")
    tc = model.cond_frame_num
    clip = smooth_clip(2, tc, cfg["dataset_params"]["frame_shape"], seed=13).cuda()
    cond = model.condition(clip)[0]
    rec = FlowAE.from_flow_diffusion(model).reconstruct(clip, source_frame=tc - 1)
    assert torch.equal(rec["optical_flow"], cond["real_vid_grid"])
    assert torch.equal(rec["occlusion_map"], cond["real_vid_conf"])


@pytest.mark.gpu
def test_graph_replay_is_bit_identical_to_eager():
    """Replays equal the eager launch lists and each other, across calls, inputs and two source frames in one process."""
    from extdm_b200.lfae import ReconRunner
    ae, cfg = make_ae("kth", "cuda")
    vids = [smooth_clip(2, 6, 64, seed=s).cuda() for s in (15, 16)]
    slots = (0, 3)
    graph = [[ae.reconstruct(v, s) for s in slots] for v in vids]
    again = [[ae.reconstruct(v, s) for s in slots] for v in vids]
    assert len(ae._runners) == 2
    ae.reconstruct(vids[0], 5)                                           # a third source frame evicts the oldest runner
    assert len(ae._runners) == ae.max_runners == 2
    assert [k[-1] for k in ae._runners] == [3, 5]
    ReconRunner.use_cuda_graph = False
    try:
        ae._runners.clear()
        eager = [[ae.reconstruct(v, s) for s in slots] for v in vids]
        assert all(r._graph is None for r in ae._runners.values())
    finally:
        ReconRunner.use_cuda_graph = True
    for i in range(len(vids)):
        for j in range(len(slots)):
            for k in graph[i][j]:
                assert torch.equal(graph[i][j][k], again[i][j][k]), (i, j, k)
                assert torch.equal(graph[i][j][k], eager[i][j][k]), (i, j, k)
    assert not torch.equal(graph[0][0]["optical_flow"], graph[0][1]["optical_flow"])
    assert not torch.equal(graph[0][0]["prediction"], graph[1][0]["prediction"])


@pytest.mark.gpu
def test_results_are_not_overwritten_by_the_next_call():
    """The returned tensors are the caller's, also for T = 1, where the decoder's (B*T, ...) buffers and the
    (B, C, T, ...) result have the same memory layout."""
    ae, _ = make_ae("kth", "cuda")
    for T in (1, 3):
        v1, v2 = smooth_clip(2, T, 64, seed=19).cuda(), smooth_clip(2, T, 64, seed=20).cuda()
        a = ae.reconstruct(v1)
        kept = {k: t.clone() for k, t in a.items()}
        b = ae.reconstruct(v2)
        for k in a:
            assert torch.equal(a[k], kept[k]), (T, k)
            assert a[k].data_ptr() != b[k].data_ptr(), (T, k)
        assert not torch.equal(a["prediction"], b["prediction"])


@pytest.mark.gpu
def test_reconstruction_is_batch_independent():
    """Video b reconstructed alone matches video b inside a batch of 8 up to rounding (GEMM tile widths follow the
    batch)."""
    ae, _ = make_ae("kth", "cuda")
    vids = smooth_clip(8, 10, 64, seed=17).cuda()
    full = ae.reconstruct(vids, source_frame=2)
    for b in (0, 5):
        one = ae.reconstruct(vids[b:b + 1].contiguous(), source_frame=2)
        d_flow = rel_l2(full["optical_flow"][b:b + 1], one["optical_flow"])
        p = psnr(full["prediction"][b:b + 1], one["prediction"])
        print(f"video {b}: batch-8 vs alone flow rel-L2 {d_flow:.3e}, frames PSNR {p:.1f} dB")
        assert d_flow <= 2e-2 and p >= 35.0, (b, d_flow, p)
