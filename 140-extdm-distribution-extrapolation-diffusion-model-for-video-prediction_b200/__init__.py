"""ExtDM sampling hot path, B200-native: UNet3D DDIM loop + LFAE flow-warp decode on hand-written sm_100a
kernels behind the reference's Python class surface (see DESIGN.md / INTEGRATION.md)."""
from .manifest import UNET_ARCHITECTURES, UnetConfig  # noqa: F401


def __getattr__(name):
    # torch-dependent classes are imported lazily so that `import extdm_b200` stays cheap
    if name in ("FlowDiffusion", "flow_diffusion_class", "WRAPPERS"):
        from . import flow_diffusion
        return getattr(flow_diffusion, name)
    if name == "GaussianDiffusion":
        from .diffusion import GaussianDiffusion
        return GaussianDiffusion
    if name == "Unet3D":
        from .unet import Unet3D
        return Unet3D
    if name == "FlowAE":
        from .flow_autoenc import FlowAE
        return FlowAE
    if name in ("Generator", "RegionPredictor", "BGMotionPredictor"):
        from . import lfae
        return getattr(lfae, name)
    raise AttributeError(name)
