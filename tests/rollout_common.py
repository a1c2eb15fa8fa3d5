"""Shared helpers of the end-to-end rollout parity tests (tests/golden/rollout_*, written by
tests/golden/make_golden.py::gen_rollout from the UNMODIFIED reference)."""
import hashlib
import io
import lzma
import math
import os

import torch
import torch.nn.functional as F

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
MAX_FILE_BYTES = 1_000_000              # per stored fixture file: save() refuses anything larger

ROLLOUTS = ["rollout_smmnist", "rollout_bair", "rollout_ucf", "rollout_cityscapes", "rollout_cityscapes_u22"]

UNET_ARCH = {
    "ada": "DenoiseNet_STWAtt_w_w_ref_adaptor_cross_multi_traj_ada",
    "u12": "DenoiseNet_STWAtt_w_w_ref_adaptor_cross_multi_traj_u12",
    "base": "DenoiseNet_STWAtt_w_wo_ref_adaptor_cross_multi",
    "u22": "DenoiseNet_STWAtt_w_w_ref_adaptor_cross_multi_traj_ada_u22",
}


def rnd(shape, seed, scale=1.0):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed)) * scale


def load(name):
    """tests/golden/<name>.pt, or <name>.pt.xz written by save(); a rollout fixture comes back whole (_expand)."""
    path = os.path.join(GOLD, name + ".pt")
    if os.path.exists(path):
        fx = torch.load(path)
    else:
        with lzma.open(path + ".xz") as f:
            fx = torch.load(io.BytesIO(f.read()))
    return _expand(fx) if fx.get("kind") == "rollout" else fx


def save(fx, name):
    """Write a fixture for load(): <name>.pt, or xz-compressed <name>.pt.xz when that is over MAX_FILE_BYTES; a
    rollout fixture in its compact form (_compact).  Raises when even the compressed file is over the limit."""
    path = os.path.join(GOLD, name + ".pt")
    buf = io.BytesIO()
    torch.save(_compact(fx) if fx["kind"] == "rollout" else fx, buf)
    data, out = buf.getvalue(), path
    if len(data) > MAX_FILE_BYTES:
        data, out = lzma.compress(data, preset=9 | lzma.PRESET_EXTREME), path + ".xz"
    if len(data) > MAX_FILE_BYTES:
        raise ValueError(f"{name}: {len(data)} bytes after compression, over {MAX_FILE_BYTES}: store fewer rounds")
    for stale in (path, path + ".xz"):
        if os.path.exists(stale):
            os.remove(stale)
    with open(out, "wb") as f:
        f.write(data)


def _planes(t):
    """A tensor as its byte planes (every element's first byte, then every second byte, ...): floats compress far
    better so."""
    return {"shape": tuple(t.shape), "dtype": str(t.dtype).removeprefix("torch."),
            "planes": t.contiguous().view(torch.uint8).reshape(-1, t.element_size()).T.contiguous()}


def _unplanes(d):
    return d["planes"].T.contiguous().view(getattr(torch, d["dtype"])).reshape(d["shape"])


def _compact(fx):
    """A rollout fixture without what _expand() rebuilds exactly: the seeded first clip (its SHA-256 is kept), each
    round's real_vid_grid / real_vid_conf (= the first frames of sample_vid_grid / sample_vid_conf) and the last tc
    frames of every round's sample_out_vid but the last one's (= the next round's clip, in fp16)."""
    tc, rounds = fx["tc"], []
    for r, o in enumerate(fx["out"]):
        k = o["real_vid_grid"].shape[2]
        assert torch.equal(o["sample_vid_grid"][:, :, :k], o["real_vid_grid"])
        assert torch.equal(o["sample_vid_conf"][:, :, :k], o["real_vid_conf"])
        o = {key: v for key, v in o.items() if key not in ("real_vid_grid", "real_vid_conf")}
        if r + 1 < len(fx["out"]):
            assert torch.equal(o["sample_out_vid"][:, :, -tc:], fx["out"][r + 1]["cond_in"].half())
            o["sample_out_vid"] = o["sample_out_vid"][:, :, :-tc]
        if r == 0:
            o.pop("cond_in")
        rounds.append({key: _planes(v) for key, v in o.items()})
    sha = hashlib.sha256(fx["out"][0]["cond_in"].numpy().tobytes()).hexdigest()
    return dict(fx, out=rounds, real_vid_frames=fx["out"][0]["real_vid_grid"].shape[2], cond_in_sha256=sha)


def _expand(fx):
    fx = dict(fx)
    k, sha = fx.pop("real_vid_frames"), fx.pop("cond_in_sha256")
    out = [{key: _unplanes(v) for key, v in o.items()} for o in fx["out"]]
    out[0]["cond_in"] = smooth_clip(fx["B"], fx["tc"], fx["hw"], fx["input_seed"],
                                    gray=fx["dataset"] in ("smmnist", "kth"))
    if hashlib.sha256(out[0]["cond_in"].numpy().tobytes()).hexdigest() != sha:
        raise ValueError("the first clip of the fixture is not reproducible from its seed")
    for r, o in enumerate(out):
        if r + 1 < len(out):
            o["sample_out_vid"] = torch.cat([o["sample_out_vid"], out[r + 1]["cond_in"].half()], dim=2)
        o["real_vid_grid"] = o["sample_vid_grid"][:, :, :k].clone()
        o["real_vid_conf"] = o["sample_vid_conf"][:, :, :k].clone()
    fx["out"] = out
    return fx


def smooth_clip(B, tc, hw, seed, gray):
    """= tests/golden/make_golden.py::smooth_clip (seeded on the CPU generator)."""
    c = 1 if gray else 3
    coarse = torch.rand((B, c, 4, 8, 8), generator=torch.Generator().manual_seed(seed))
    vid = F.interpolate(coarse, size=(tc, hw, hw), mode="trilinear", align_corners=True).clamp(0, 1)
    return vid.expand(B, 3, tc, hw, hw).contiguous()


def round_noise(fx, r):
    """(steps, B, 3, tp, 32, 32): the Gaussian tensors round r of the fixture consumed, in draw order."""
    return torch.stack([rnd((fx["B"], 3, fx["tp"], 32, 32), fx["noise_seed"] + 100 * r + i)
                        for i in range(fx["steps"])])


def build_model(fx, device):
    """This repo's FlowDiffusion for the fixture's (config, wrapper, UNet) with the fixture's synthetic weights."""
    import extdm_b200  # noqa: F401
    from extdm_b200.flow_diffusion import flow_diffusion_class
    from extdm_b200.weights import synth_state_dict
    fd = flow_diffusion_class(fx["dm_arch"])(config=fx["cfg"], pretrained_pth="", is_train=False,
                                             Unet3D_architecture=UNET_ARCH[fx["variant"]]).eval()
    for part, seed in fx["weight_seeds"].items():
        m = getattr(fd, part)
        base = m.state_dict()
        man = fx["manifests"].get(part) or {k: tuple(v.shape) for k, v in base.items()}
        m.load_state_dict(synth_state_dict(man, seed, base=base), strict=True)
    return fd.to(device)


def rel_l2(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm()).item()


def psnr(a, b):
    mse = ((a.float() - b.float()) ** 2).mean().item()
    return 99.0 if mse == 0 else 10 * math.log10(1.0 / mse)
