"""savsr_b200: B200-native (sm_100a) forward hot path of SAVSR behind the reference's arch interface.

Public API:  ``savsr_b200.SAVSR`` (drop-in nn.Module), ``savsr_b200.build_network`` (registry builder),
``savsr_b200.VideoUpscaler`` (frame-in / frame-out 8-bit video of any length, BGR or YUV 4:2:0),
``savsr_b200.colour`` (YUV 4:2:0 <-> BGR on the device, as cv2.cvtColor converts),
``savsr_b200.overlay.install`` (serve the class to an unmodified reference checkout).
Importing the package does not need a GPU; running the model does, and fails loudly without
``savsr_b200/lib/libsavsr_sm100.so`` (built by ``python -m savsr_b200.build``).
"""
from .registry import ARCH_REGISTRY, build_network  # noqa: F401
from .archs.savsr_arch import SAVSR, get_HW  # noqa: F401
from .videostream import VideoUpscaler  # noqa: F401
from . import colour  # noqa: F401

__all__ = ["SAVSR", "ARCH_REGISTRY", "build_network", "get_HW", "VideoUpscaler", "colour"]
