"""Drop-in ``SAVSR`` arch backed by libsavsr_sm100 (B200 / sm_100a).

Boundary contract (reference: lbasicsr/archs/savsr_arch.py:574-742, SURVEY.md section 8b):
  * class name ``SAVSR``, registered in ``ARCH_REGISTRY`` (the reference's registry when ``lbasicsr`` is
    importable -- see ``savsr_b200.overlay`` -- otherwise a local registry of the same shape);
  * identical constructor keyword arguments;
  * ``set_scale(scale)`` then ``forward(x)`` with ``x`` float32 ``[b, 7, 3, h, w]`` in [0, 1], returning a
    fresh float32 ``[b, 3, H, W]`` tensor (not clamped), ``H, W = round(h * s_h), round(w * s_w)``;
  * identical parameter / buffer names, shapes and order, so ``load_state_dict(strict=True)`` round-trips
    with reference checkpoints (``{'params': state_dict}``).

The sub-modules below are *parameter containers* that reproduce the reference's state_dict layout; they
never run.  ``forward`` hands the parameters to ``savsr_b200.engine.Plan`` which launches the CUDA
kernels through the C ABI.  There is no CPU / eager fallback: CPU tensors raise.
"""
from __future__ import annotations

import math
import os
from collections import OrderedDict
from typing import Dict, Optional, Tuple, Union

import torch
import torch.nn as nn

from savsr_b200 import colour, engine

if __name__ == "lbasicsr.archs.savsr_arch":
    # served by savsr_b200.overlay in place of the reference's own file: register in the reference's registry
    # (lbasicsr/utils/registry.py:11-47; lbasicsr/archs/__init__.py:13-16 imports this module by that name)
    from lbasicsr.utils.registry import ARCH_REGISTRY  # type: ignore
else:
    # standalone use.  Never touch the reference's registry from here: importing lbasicsr would register the reference's
    # own SAVSR first and this class's registration would then trip the registry's uniqueness assertion.
    from savsr_b200.registry import ARCH_REGISTRY


def _no_forward(self, *a, **k):
    raise RuntimeError(f"{type(self).__name__} is a parameter container of savsr_b200.SAVSR; call the top-level module")


class _Holder(nn.Module):
    forward = _no_forward


def _conv(ci: int, co: int, k: int, bias: bool = True) -> nn.Conv2d:
    return nn.Conv2d(ci, co, k, 1, k // 2, bias=bias)


class ScaleAttention(_Holder):
    """Parameters of savsr_arch.py:16-60 (kernel_size 3, kernel_num 8)."""

    def __init__(self, in_planes: int, out_planes: int, kernel_num: int = 8, reduction: float = 0.0625, min_channel: int = 16):
        super().__init__()
        a = max(int(in_planes * reduction), min_channel)
        self.fc = _conv(in_planes, a, 1, bias=False)
        self.bn = nn.BatchNorm2d(a)
        self.channel_fc = _conv(a, in_planes, 1)
        self.filter_fc = _conv(a, out_planes, 1)
        self.spatial_fc = _conv(a, 9, 1)
        self.kernel_fc = _conv(a, kernel_num, 1)
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
                if m.bias is not None:
                    nn.init.constant_(m.bias, 0)


class OSConv2d(_Holder):
    """Parameters of the omni-dimensional scale-attention conv (savsr_arch.py:99-134)."""

    def __init__(self, in_planes: int, out_planes: int, kernel_num: int = 8):
        super().__init__()
        self.weight = nn.Parameter(torch.randn(kernel_num, out_planes, in_planes, 3, 3))
        self.attention = ScaleAttention(in_planes, out_planes, kernel_num)
        self.scale_routing = nn.Sequential(nn.Linear(in_planes + 2, in_planes * 2), nn.ReLU(True),
                                           nn.Linear(in_planes * 2, in_planes), nn.ReLU(True))
        with torch.no_grad():
            for i in range(kernel_num):
                nn.init.kaiming_normal_(self.weight[i], mode="fan_out", nonlinearity="relu")


class OSAdapt(_Holder):
    def __init__(self, channels: int, ratio: int = 4):
        super().__init__()
        c = channels // ratio
        self.mask = nn.Sequential(
            _conv(channels, c, 3), nn.BatchNorm2d(c), nn.ReLU(True), nn.AvgPool2d(2),
            _conv(c, c, 3), nn.BatchNorm2d(c), nn.ReLU(True),
            _conv(c, c, 3), nn.BatchNorm2d(c), nn.ReLU(True),
            nn.Upsample(scale_factor=2, mode="bilinear", align_corners=False),
            _conv(c, 1, 3), nn.BatchNorm2d(1), nn.Sigmoid())
        self.adapt = OSConv2d(channels, channels)


class STAUpsample(_Holder):
    def __init__(self, channels: int, num_experts: int = 4, st_ksize: int = 5):
        super().__init__()
        wc = torch.empty(num_experts, channels // 8, channels, 1, 1)
        we = torch.empty(num_experts, channels, channels // 8, 1, 1)
        for i in range(num_experts):
            nn.init.kaiming_uniform_(wc[i], a=math.sqrt(5))
            nn.init.kaiming_uniform_(we[i], a=math.sqrt(5))
        self.weight_compress = nn.Parameter(wc)
        self.weight_expand = nn.Parameter(we)
        self.kernel_conv = nn.Sequential(_conv(channels, channels * st_ksize ** 2, 1), nn.LeakyReLU(0.1, True))
        self.body = nn.Sequential(_conv(4, 64, 1), nn.ReLU(True), _conv(64, 64, 1), nn.ReLU(True))
        self.routing = nn.Sequential(_conv(64, num_experts, 1), nn.Sigmoid())
        self.offset = _conv(64, 2, 1)
        self.st_offset = _conv(64, 2, 1)
        self.fusion = _conv(2 * channels, channels, 1)


class ResidualBlock(_Holder):
    def __init__(self, num_feat: int = 64, num_frame: int = 3, use_osconv: bool = False):
        super().__init__()
        self.conv0 = nn.Sequential(*[_conv(num_feat, num_feat, 3) for _ in range(num_frame)])
        if use_osconv:
            self.osconv = OSConv2d(num_feat * num_frame, num_feat)
        else:
            self.conv1 = _conv(num_feat * num_frame, num_feat, 1)
        self.conv2 = nn.Sequential(*[_conv(num_feat * 2, num_feat, 3) for _ in range(num_frame)])


class WindowUnit_l1(_Holder):
    def __init__(self, num_in_ch: int = 3, num_feat: int = 64, win_size: int = 3, num_block: int = 4):
        super().__init__()
        self.conv_c = _conv(num_in_ch, num_feat, 3)
        self.conv_sup = _conv(num_in_ch * (win_size - 1), num_feat, 3)
        self.blocks = nn.Sequential(*[ResidualBlock(num_feat, 3, use_osconv=i >= 1) for i in range(num_block)])
        self.merge = _conv(3 * num_feat, num_feat, 3)


class WindowUnit_l2(_Holder):
    def __init__(self, num_feat: int = 64, win_size: int = 5, slid_win: int = 3, num_block: int = 2):
        super().__init__()
        self.conv_h = nn.Sequential(*[_conv(num_feat * 2, num_feat, 3) for _ in range(win_size)])
        self.blocks = nn.Sequential(*[ResidualBlock(num_feat, slid_win, use_osconv=True) for _ in range(num_block)])
        self.merge = _conv(slid_win * num_feat, num_feat * 2, 3)


class ChannelAttention(_Holder):
    def __init__(self, num_feat: int, squeeze_factor: int = 16):
        super().__init__()
        self.attention = nn.Sequential(nn.AdaptiveAvgPool2d(1), nn.Conv2d(num_feat, num_feat // squeeze_factor, 1),
                                       nn.ReLU(True), nn.Conv2d(num_feat // squeeze_factor, num_feat, 1), nn.Sigmoid())


class RCAB(_Holder):
    def __init__(self, num_feat: int, squeeze_factor: int = 16):
        super().__init__()
        self.rcab = nn.Sequential(_conv(num_feat, num_feat, 3), nn.ReLU(True), _conv(num_feat, num_feat, 3),
                                  ChannelAttention(num_feat, squeeze_factor))


class ResidualGroup(_Holder):
    def __init__(self, num_feat: int, num_block: int, squeeze_factor: int = 16):
        super().__init__()
        self.residual_group = nn.Sequential(*[RCAB(num_feat, squeeze_factor) for _ in range(num_block)])
        self.conv = _conv(num_feat, num_feat, 3)


@ARCH_REGISTRY.register()
class SAVSR(nn.Module):
    """B200-native SAVSR forward.  Same constructor as the reference (savsr_arch.py:576-589)."""

    def __init__(self, num_in_ch=3, num_feat=64, num_frame=7, slid_win=3, fusion_win=5, interval=0, w1_num_block=4,
                 w2_num_block=2, n_resgroups=4, n_resblocks=8, downsample_scale=2, center_frame_idx=None):
        super().__init__()
        if interval != 0:
            raise NotImplementedError("savsr_b200 implements the shipped configuration interval=0 only")
        if (num_in_ch, num_feat, num_frame, slid_win, fusion_win, w1_num_block, w2_num_block, n_resgroups, n_resblocks) != \
                (3, 64, 7, 3, 5, 4, 2, 4, 8):
            raise NotImplementedError(
                "savsr_b200 kernels are specialised for the shipped SAVSR YAML (num_feat=64, num_frame=7, slid_win=3, "
                "fusion_win=5, w1_num_block=4, w2_num_block=2, n_resgroups=4, n_resblocks=8)")
        self.scale: Union[tuple, float, int] = (4, 4)
        self.center_frame_idx = num_frame // 2 if center_frame_idx is None else center_frame_idx
        if self.center_frame_idx != num_frame // 2:
            raise NotImplementedError("center_frame_idx must be the middle frame")
        self.num_frame, self.iter_win, self.slid_win, self.interval = num_frame, num_frame, slid_win, interval
        self.num_feat, self.downsample_scale = num_feat, downsample_scale

        self.f2p_win = WindowUnit_l1(num_in_ch, num_feat, slid_win, w1_num_block)
        self.p2f_win = WindowUnit_l1(num_in_ch, num_feat, slid_win, w1_num_block)
        self.h_win = nn.Sequential(*[WindowUnit_l2(num_feat, (self.iter_win - slid_win + 1) - 2 * i, fusion_win, w2_num_block)
                                     for i in range((self.iter_win - fusion_win + 1) // 2)])
        self.h_win_act = nn.LeakyReLU(0.2, True)
        self.h_win_conv_h = _conv(num_feat * 2, num_feat, 3)
        self.RG = nn.ModuleList([ResidualGroup(num_feat, n_resblocks) for _ in range(n_resgroups)])
        self.K = 1
        self.adapt = nn.ModuleList([OSAdapt(num_feat) for _ in range(n_resgroups // self.K)])
        self.gamma = nn.Parameter(torch.ones(1))
        self.conv_last = _conv(num_feat, num_feat, 3)
        self.upsample = STAUpsample(num_feat)
        self.tail = _conv(num_feat, num_in_ch, 3)

        self._plans: "OrderedDict[tuple, engine.Plan]" = OrderedDict()
        self._stores: Dict[tuple, engine.WeightStore] = {}     # packed weights / folded BN shared by all plans of one weights version
        self._wlist = None                                     # cached list of parameters + buffers (version check per forward)
        self._wepoch = 0                                       # bumped by _apply (.to/.cuda/.half) and load_state_dict
        self._wkey = None
        self.plan_cache_bytes = int(float(os.environ.get("SAVSR_PLAN_CACHE_GB", "48")) * 2 ** 30)
        self.conv_impl = os.environ.get("SAVSR_CONV_IMPL", "halo")   # "halo": one TMA halo tile per source (default, fastest); "tap": one box per tap
        self.use_graph = os.environ.get("SAVSR_GRAPH", "1") != "0"
        # 16-bit operand format: "bf16" (throughput path, wide range) or "fp16" (same speed, 10-bit mantissa: meets the
        # <= 1e-3 max-abs bound against the fp32 reference; needs activations below 65504)
        self.precision = os.environ.get("SAVSR_PRECISION", "bf16")
        self.native_training = os.environ.get("SAVSR_NATIVE_TRAIN", "1") != "0"     # train-mode forward on the native launch list (trainplan.py)
        self.debug_taps: Tuple[str, ...] = ()
        self.last_plan_build_ms = 0.0
        self.register_load_state_dict_post_hook(lambda module, incompatible: module._invalidate_weights())

    # ---- reference API ---------------------------------------------------------------------------
    def set_scale(self, scale: Union[tuple, float, int]):
        self.scale = scale

    def forward(self, x: torch.Tensor, scale=None) -> torch.Tensor:
        """savsr_arch.py:692-742.  Returns a fresh [b, 3, H, W] fp32 tensor (the caller may delete it and call
        empty_cache(), as video_base_model.py:72-74 does every frame: the plan's arenas are not affected)."""
        if scale is not None:
            self.scale = scale
        if self.training:
            # optimisation path (sr_model.py:101-128 calls net_g(lq) in train mode).  Default: the native launch list of
            # savsr_b200/trainplan.py behind ONE autograd node (forward + backward of every trunk op on libsavsr_sm100; the caller's loss,
            # optimizer, EMA and DistributedDataParallel work on the module's parameters as usual).  Fallback (odd sizes, more than
            # trainplan.MAX_NATIVE_BATCH = 32 samples per GPU, no_grad, native_training = False): savsr_b200/train.py, the ATen tape with the 3x3 convolutions on the tcgen05 kernels.
            from savsr_b200 import trainplan as _tp
            if self.native_training and torch.is_grad_enabled() and self.precision == "bf16" and _tp.ModuleTraining.supports(x):
                st = self.__dict__.get("_train_state")
                if st is None or not st.flat.intact():
                    st = _tp.ModuleTraining(self)
                    self.__dict__["_train_state"] = st
                return st.forward(x, self.scale)
            from savsr_b200 import train as _train
            return _train.forward(self, x, self.scale)
        if x.dim() == 5 and x.shape[0] == 0 and x.is_cuda:        # an empty batch of windows (a rank with no frames of the clip): nothing to launch
            H, W = engine.get_hw(x.shape[3], x.shape[4], self.scale)
            return x.new_empty((0, 3, H, W))
        return self._run_plan(self.plan_for(x), x)

    def forward_bgr_u8(self, x: torch.Tensor, scale=None) -> torch.Tensor:
        """Upscale decoded 8-bit video: x uint8 [b, 7, h, w, 3] BGR windows (the layout cv2.imread and video decoders produce) ->
        a fresh uint8 [b, H, W, 3] BGR tensor.  Bit for bit the image tensor2img makes of forward(x') (postproc.tensor2img_psnr),
        where x' = the windows as fp32 RGB planes, u / 255 correctly rounded, as the reference's img.astype(np.float32) / 255.
        Inference only (training takes fp32 windows through forward); same plan cache, precision, conv_impl and CUDA graphs as
        forward, with its own plan per shape."""
        if self.training:
            raise RuntimeError("forward_bgr_u8 is inference only: call eval() first (training takes fp32 windows through forward)")
        if scale is not None:
            self.scale = scale
        b, h, w = self._window_shape(x, "bgr_u8")
        if b == 0:                  # an empty batch of windows (a rank with no frames of the clip): nothing to launch
            return x.new_empty((0, *engine.get_hw(h, w, self.scale), 3))
        return self._run_plan(self.plan_for(x, io="bgr_u8"), x)

    def forward_bgr_u8_indexed(self, pool: torch.Tensor, windows, scale=None) -> torch.Tensor:
        """forward_bgr_u8(pool[windows]), bit for bit, without gathering the windows: pool is a uint8 CUDA tensor [N, h, w, 3] whose
        rows are BGR frames (a clip, or a ring of decoded frames), windows a host sequence or CPU integer tensor [b, 7] of row
        indices (any order, repeats allowed).  Each forward reads its frames in place through a device table of frame addresses,
        so every frame is read once per window instead of being copied 7 times.  Returns a fresh uint8 [b, H, W, 3] BGR tensor.
        The pool is read on the device's current stream: it must stay valid, in stream order, until the forward has run."""
        if scale is not None:
            self.scale = scale
        return self._forward_bgr_u8_indexed(pool, windows, self.scale, dtype=torch.uint8)

    def forward_bgr48(self, x: torch.Tensor, scale=None) -> torch.Tensor:
        """Upscale deep video: x uint16 [b, 7, h, w, 3] BGR windows (bgr48, full scale 65535: 16-bit PNG / TIFF frames as
        cv2.IMREAD_UNCHANGED loads them, or decoded 10-bit video) on CUDA -> a fresh uint16 [b, H, W, 3] BGR tensor.  Bit for bit
        round(clamp(forward(x') , 0, 1) * 65535) in fp32 with round half to even, where x' = the windows as fp32 RGB planes, v / 65535
        correctly rounded.  On 257 * x8 it computes what forward_bgr_u8 computes on x8, before the output's quantisation.  The windows
        are read in place through a frame table (the plan of forward_bgr48_indexed), so x must stay valid, in stream order, until the
        forward has run.  Inference only; same plan cache, precision and CUDA graphs as forward."""
        if self.training:
            raise RuntimeError("forward_bgr48 is inference only: call eval() first (training takes fp32 windows through forward)")
        if scale is not None:
            self.scale = scale
        if x.dtype != torch.uint16:
            raise TypeError(f"forward_bgr48 takes uint16 windows, got {x.dtype}")
        if x.dim() != 5 or x.shape[1] != self.num_frame or x.shape[4] != 3:
            raise ValueError(f"expected uint16 BGR windows [b, {self.num_frame}, h, w, 3], got {tuple(x.shape)}")
        b, t, h, w, _ = x.shape
        windows = torch.arange(b * t).reshape(b, t)
        return self._forward_bgr_u8_indexed(x.reshape(b * t, h, w, 3), windows, self.scale, dtype=torch.uint16)

    def forward_bgr48_indexed(self, pool: torch.Tensor, windows, scale=None) -> torch.Tensor:
        """forward_bgr48(pool[windows]), bit for bit, without gathering the windows: pool is a contiguous uint16 CUDA tensor [N, h, w, 3]
        of bgr48 frames, windows as for forward_bgr_u8_indexed.  Returns a fresh uint16 [b, H, W, 3] BGR tensor; the pool is read on
        the device's current stream and must stay valid, in stream order, until the forward has run."""
        if scale is not None:
            self.scale = scale
        return self._forward_bgr_u8_indexed(pool, windows, self.scale, dtype=torch.uint16)

    def _forward_bgr_u8_indexed(self, pool: torch.Tensor, windows, scale, out_format: Optional[str] = None,
                                dtype: Optional[torch.dtype] = None, out_colorspace: str = "bt601",
                                out_color_range: str = "tv") -> torch.Tensor:
        """forward_bgr_u8_indexed (uint8 pool) or forward_bgr48_indexed (uint16 pool) at `scale`, leaving self.scale as it is
        (savsr_b200.VideoUpscaler keeps its own scale).  The I/O mode follows the pool's dtype; `dtype`, when given, is the one the
        public caller takes.  With a YUV out_format of the pool's depth (4:2:0 or 4:2:2, savsr_b200.colour) the HR frames come back as
        [b, *colour.yuv_shape(H, W, out_format)], converted from the plan's output staging buffer instead
        of copied, with the matrix out_colorspace and the range out_color_range; None is packed BGR."""
        name = {torch.uint16: "forward_bgr48_indexed"}.get(dtype if dtype is not None else pool.dtype, "forward_bgr_u8_indexed")
        if self.training:
            raise RuntimeError(f"{name} is inference only: call eval() first (training takes fp32 windows through forward)")
        want = (dtype,) if dtype is not None else tuple(engine.FRAME_MODES.values())
        if pool.dtype not in want:
            raise TypeError(f"{name} takes a {' or '.join(str(d).replace('torch.', '') for d in want)} frame pool, got {pool.dtype}")
        io = "bgr48_frames" if pool.dtype == torch.uint16 else "bgr_u8_frames"
        tn = str(pool.dtype).replace("torch.", "")
        if pool.dim() != 4 or pool.shape[3] != 3:
            raise ValueError(f"expected a {tn} BGR frame pool [N, h, w, 3], got {tuple(pool.shape)}")
        if not pool.is_contiguous():
            raise ValueError("the frame pool must be contiguous (each row one [h, w, 3] frame)")
        idx = torch.as_tensor(windows)
        if idx.numel() == 0 and not idx.is_cuda:
            idx = idx.reshape(0, self.num_frame).long()
        if idx.is_cuda or idx.is_floating_point() or idx.is_complex() or idx.dtype == torch.bool:
            raise TypeError(f"windows must be a host sequence or CPU integer tensor of row indices, got {idx.dtype} on {idx.device}")
        if idx.dim() != 2 or idx.shape[1] != self.num_frame:
            raise ValueError(f"expected windows [b, {self.num_frame}] of row indices, got shape {tuple(idx.shape)}")
        n, h, w, _ = pool.shape
        b = idx.shape[0]
        self._check_device(pool)
        bgr = "bgr48le" if io == "bgr48_frames" else "bgr24"
        out_format = bgr if out_format is None else colour.check_format(out_format, "out_format")
        if colour.bgr_format(out_format) != bgr:
            raise ValueError(f"out_format {out_format!r} has another depth than the {tn} frame pool")
        out_colorspace = colour.check_colorspace(out_colorspace, "out_colorspace")
        out_color_range = colour.check_color_range(out_color_range, "out_color_range")
        if out_format == bgr and (out_colorspace, out_color_range) != ("bt601", "tv"):
            raise ValueError(f"out_colorspace / out_color_range ({out_colorspace!r}, {out_color_range!r}) need a YUV out_format: "
                             f"{out_format} output is not converted")
        if b == 0:
            H, W = engine.get_hw(h, w, scale)
            return pool.new_empty((0, H, W, 3) if out_format == bgr else (0, *colour.yuv_shape(H, W, out_format)))
        idx = idx.to(torch.int64)
        lo, hi = int(idx.min()), int(idx.max())
        if lo < 0 or hi >= n:
            raise IndexError(f"window row index {lo if lo < 0 else hi} out of range for a pool of {n} frames")
        ptrs = (idx.reshape(-1) * (h * w * 3 * pool.element_size()) + pool.data_ptr()).tolist()
        return self._run_plan(self._plan(b, h, w, pool.device, io, scale), frames=ptrs, out_format=out_format,
                              out_colorspace=out_colorspace, out_color_range=out_color_range)

    def _forward_ring_scenes(self, ring: torch.Tensor, cut: torch.Tensor, first: int, count: int, received: int, finished: bool, scale,
                             out_format: Optional[str] = None, out_colorspace: str = "bt601", out_color_range: str = "tv") -> torch.Tensor:
        """The forward of savsr_b200.VideoUpscaler with scene detection: the windows of frames first .. first + count - 1 of a stream
        whose frame t sits in slot t % R of `ring` (uint8 or uint16 [R, h, w, 3]), each folded into its shot as the device cut flags
        `cut` (uint8 [R], savsr_b200.scenes.Detector) mark it.  The frame table is written on the device (Plan.forward_scene_frames_into),
        so no flag is read back.  Output, formats and colour as _forward_bgr_u8_indexed at `scale`."""
        if self.training:
            raise RuntimeError("_forward_ring_scenes is inference only: call eval() first")
        if ring.dtype not in engine.FRAME_MODES.values() or ring.dim() != 4 or ring.shape[3] != 3 or not ring.is_contiguous():
            raise ValueError(f"expected a contiguous uint8 or uint16 BGR ring [R, h, w, 3], got {ring.dtype} {tuple(ring.shape)}")
        self._check_device(ring)
        io = "bgr48_frames" if ring.dtype == torch.uint16 else "bgr_u8_frames"
        out_format = ("bgr48le" if io == "bgr48_frames" else "bgr24") if out_format is None else colour.check_format(out_format, "out_format")
        out_colorspace = colour.check_colorspace(out_colorspace, "out_colorspace")
        out_color_range = colour.check_color_range(out_color_range, "out_color_range")
        return self._run_plan(self._plan(int(count), ring.shape[1], ring.shape[2], ring.device, io, scale), out_format=out_format,
                              out_colorspace=out_colorspace, out_color_range=out_color_range,
                              scene=(ring, cut, int(first), int(received), bool(finished)))

    def _run_plan(self, plan: engine.Plan, x: Optional[torch.Tensor] = None, frames: Optional[list] = None,
                  out_format: str = "bgr24", out_colorspace: str = "bt601", out_color_range: str = "tv",
                  scene: Optional[tuple] = None) -> torch.Tensor:
        with torch.cuda.device(plan.device):
            if out_format in ("bgr24", "bgr48le"):
                out = torch.empty_like(plan.out)
            else:
                out = plan.out.new_empty((plan.B, *colour.yuv_shape(plan.H, plan.W, out_format)))
            cs = {} if (out_colorspace, out_color_range) == ("bt601", "tv") else \
                {"out_colorspace": out_colorspace, "out_color_range": out_color_range}
            if scene is not None:
                plan.forward_scene_frames_into(*scene, out, graph=self.use_graph, out_format=out_format, **cs)
            elif frames is None:
                plan.forward_into(x, out, graph=self.use_graph)
            else:
                plan.forward_frames_into(frames, out, graph=self.use_graph, out_format=out_format, **cs)
            if self.precision == "fp16" and not plan.__dict__.get("_range_checked"):
                # fp16 operands meet the <= 1e-3 bound but saturate at 65504: look at every trunk activation of this plan's FIRST forward
                # (one pass over the arena, once per plan) and refuse to continue silently when the headroom is below 4x
                plan._range_checked = True
                peak = plan.activation_absmax()
                self.fp16_peak_activation = max(getattr(self, "fp16_peak_activation", 0.0), peak)
                if not peak < 65504.0 / 4:
                    raise FloatingPointError(
                        f"precision='fp16': the largest trunk activation of this input is {peak:.4g} (fp16 saturates at 65504); "
                        "use precision='bf16' (same speed, fp32 range) for these weights")
        return out

    # ---- plan management ---------------------------------------------------------------------------
    def _invalidate_weights(self) -> None:
        self._wlist = None
        self._wepoch += 1

    def _apply(self, fn, *a, **k):          # .to() / .cuda() / .half() ...: parameters get new storage
        r = super()._apply(fn, *a, **k)
        if hasattr(self, "_wepoch"):
            self._invalidate_weights()
        return r

    def __setattr__(self, name, value):     # a replaced parameter / sub-module invalidates the cached tensor list
        if isinstance(value, (torch.Tensor, nn.Module)) and "_wepoch" in self.__dict__:
            self._invalidate_weights()
        super().__setattr__(name, value)

    def _weights_version(self) -> tuple:
        """Cheap per-forward check: the sum of the tensors' in-place version counters (optimizer steps, copy_, load_state_dict)
        plus an epoch bumped whenever storage may have been replaced.  The (data_ptr, version) tuple hash of the ~800
        tensors is recomputed only when that changes."""
        if self._wlist is None:
            self._wlist = list(self.parameters()) + list(self.buffers())
            self._wkey = None
        ver = self._wepoch
        for t in self._wlist:
            ver += t._version
        if self._wkey is None or self._wkey[0] != ver:
            self._wkey = (ver, hash(tuple((t.data_ptr(), t._version) for t in self._wlist)))
        return self._wkey

    def _store_for(self, device: torch.device, wkey: tuple) -> "engine.WeightStore":
        key = (device.index, self.precision)
        st = self._stores.get(key)
        if st is None or st.version != wkey:
            st = engine.WeightStore(wkey)
            self._stores[key] = st
        return st

    def _window_shape(self, x: torch.Tensor, io: str) -> Tuple[int, int, int]:
        """(b, h, w) of a batch of windows in the layout of `io`, after checking that it can run on this module's device."""
        if io == "bgr_u8":
            if x.dtype != torch.uint8:
                raise TypeError(f"forward_bgr_u8 takes uint8 windows, got {x.dtype}")
            if x.dim() != 5 or x.shape[1] != self.num_frame or x.shape[4] != 3:
                raise ValueError(f"expected uint8 BGR windows [b, {self.num_frame}, h, w, 3], got {tuple(x.shape)}")
            b, _, h, w, _ = x.shape
        else:
            if x.dim() != 5 or x.shape[1] != self.num_frame or x.shape[2] != 3:
                raise ValueError(f"expected input [b, {self.num_frame}, 3, h, w], got {tuple(x.shape)}")
            b, _, _, h, w = x.shape
        self._check_device(x)
        return b, h, w

    def _check_device(self, x: torch.Tensor) -> None:
        if not x.is_cuda:
            raise RuntimeError("savsr_b200.SAVSR runs on CUDA (sm_100a) only; there is no CPU fallback")
        p0 = self.gamma
        if p0.device != x.device:
            raise RuntimeError(f"module parameters on {p0.device}, input on {x.device}")

    def plan_for(self, x: torch.Tensor, io: str = "f32") -> engine.Plan:
        """The cached plan for windows like `x`: io="f32" takes [b, 7, 3, h, w] (forward), io="bgr_u8" uint8 [b, 7, h, w, 3]
        (forward_bgr_u8).  Plans of every I/O mode (also "bgr_u8_frames" and "bgr48_frames", the *_indexed forwards) share one
        WeightStore."""
        b, h, w = self._window_shape(x, io)
        return self._plan(b, h, w, x.device, io, self.scale)

    def _plan(self, b: int, h: int, w: int, device: torch.device, io: str, scale) -> engine.Plan:
        if self.training:
            raise RuntimeError("plans are the inference path; in train mode forward() runs savsr_b200.train.forward")
        s = engine.normalize_scale(scale)
        wkey = self._weights_version()
        key = (b, h, w, float(s[0]), float(s[1]), self.conv_impl, self.precision, tuple(self.debug_taps), device.index, io) + wkey
        plan = self._plans.get(key)
        if plan is not None:
            self._plans.move_to_end(key)
            return plan
        import time
        t0 = time.perf_counter()
        params = {k: v for k, v in self.state_dict(keep_vars=True).items()}
        plan = engine.Plan(params, b, h, w, s, device, conv_impl=self.conv_impl, num_frame=self.num_frame,
                           taps=self.debug_taps, precision=self.precision, store=self._store_for(device, wkey), io=io)
        self.last_plan_build_ms = 1e3 * (time.perf_counter() - t0)
        self._plans[key] = plan
        # bound the device memory held by cached plans (arenas + graphs): evict least recently used down to the byte budget
        total = sum(p.nbytes for p in self._plans.values())
        while total > self.plan_cache_bytes and len(self._plans) > 1:
            _, old = self._plans.popitem(last=False)
            total -= old.nbytes
            old.release()
        return plan

    def release_plans(self) -> None:
        for p in self._plans.values():
            p.release()
        self._plans.clear()
        self._stores.clear()


def get_HW(h, w, scale):
    """savsr_arch.py:745-751."""
    return engine.get_hw(h, w, scale)
