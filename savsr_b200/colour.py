"""YUV 4:2:0 <-> packed BGR on the device: 8-bit byte-identical to OpenCV's ``cv2.cvtColor``, and 10-bit YUV <-> 16-bit BGR.

Video decoders hand out YUV 4:2:0 (NVDEC: NV12 surfaces in device memory; ``ffmpeg -f rawvideo -pix_fmt yuv420p``: planar I420) and
encoders take it back, while ``SAVSR.forward_bgr_u8`` and ``VideoUpscaler`` work on packed BGR [h, w, 3].  The formats carry ffmpeg's
``pix_fmt`` names:

* ``"bgr24"``: uint8 [h, w, 3], the layout ``cv2.imread`` produces;
* ``"yuv420p"``: one uint8 [3h/2, w] array per frame: the Y plane, then the U plane (h/2 x w/2), then the V plane, packed;
* ``"nv12"``: one uint8 [3h/2, w] array per frame: the Y plane, then h/2 rows of interleaved U, V bytes (U first).  It may have a
  row pitch (``stride(0) >= w``, ``stride(1) == 1``; the UV rows start at row h of the same pitch), as a decoder surface does when it
  is exposed as a tensor view.  yuv420p frames must have contiguous rows.

Deep video (HEVC Main10, 10-bit AV1, 16-bit PNG / TIFF sequences) has formats of its own, all uint16:

* ``"bgr48le"``: uint16 [h, w, 3] BGR, full scale 65535 (``cv2.imread(path, cv2.IMREAD_UNCHANGED)`` of a 16-bit image);
* ``"yuv420p10le"``: one uint16 [3h/2, w] array per frame laid out as yuv420p, the 10-bit value in bits 0-9 (ffmpeg's rawvideo);
* ``"p010"``: one uint16 [3h/2, w] array per frame laid out as nv12, the value in bits 6-15 (NVDEC's 10-bit surfaces); it may have a
  row pitch like nv12.

Several frames are [n, 3h/2, w].  By default the conversion is BT.601, limited range, in OpenCV's 20-bit fixed point: decoding gives
each pixel the chroma sample of its 2x2 block (``COLOR_YUV2BGR_I420`` / ``COLOR_YUV2BGR_NV12``), encoding takes U and V from the
top-left pixel of each 2x2 block (``COLOR_BGR2YUV_I420``).  Sizes must be even, as cv2 requires.  The 10-bit formats use the same
matrix and chroma handling, rescaled (one 10-bit step is a quarter of an 8-bit step, one 8-bit BGR step is 257 sixteen-bit steps), in
a fixed-point form within 0.53 of an output step of the real-valued map; decoding saturates to [0, 65535].

Other colour matrices and ranges, named as ffmpeg's ``-colorspace`` and ``-color_range`` options (``COLORSPACES``, ``COLOR_RANGES``):
``colorspace`` "bt601" (aliases "bt470bg", "smpte170m"), "bt709" or "bt2020nc" ("bt2020"), ``color_range`` "tv" ("limited", "mpeg")
or "pc" ("full", "jpeg").  Every pair but the default ("bt601", "tv") converts with the Y'CbCr <-> R'G'B' map of ITU-T H.273 (the
same chroma handling), in integer forms within 0.55 of an output step of the real-valued map at both depths: tv has its black level
at 16 (64 in 10 bits) and spans of 219 and 224 steps, pc uses every code value.  Decoding saturates to the BGR range and does not clamp
Y at the black level; encoding saturates to [0, 2^n - 1].  Only code values are converted: no transfer function (PQ / HLG, tone
mapping) is applied, and BT.2020 is the non-constant-luminance matrix.  The default pair keeps OpenCV's constants exactly.

Each call is one launch on the current stream of the tensors' device (savsr_yuv420_to_bgr / savsr_bgr_to_yuv420,
savsr_yuv420_10_to_bgr48 / savsr_bgr48_to_yuv420_10 of libsavsr_sm100, and their _cs forms for the other pairs); there is no CPU path.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import _capi as K, engine

FORMATS = ("bgr24", "yuv420p", "nv12", "bgr48le", "yuv420p10le", "p010")
YUV_FORMATS = ("yuv420p", "nv12", "yuv420p10le", "p010")
DEEP_FORMATS = ("bgr48le", "yuv420p10le", "p010")
PITCHED_FORMATS = ("nv12", "p010")          # may have a row pitch; their U, V samples are interleaved
COLORSPACES = {"bt601": 0, "bt709": 1, "bt2020nc": 2}      # enum savsr_colorspace
COLOR_RANGES = {"tv": 0, "pc": 1}                          # enum savsr_color_range
_COLORSPACE_ALIASES = {"bt470bg": "bt601", "smpte170m": "bt601", "bt2020": "bt2020nc"}
_COLOR_RANGE_ALIASES = {"limited": "tv", "mpeg": "tv", "full": "pc", "jpeg": "pc"}


def dtype_of(fmt: str) -> torch.dtype:
    """The sample type of `fmt`: uint16 for the deep formats, uint8 otherwise."""
    return torch.uint16 if fmt in DEEP_FORMATS else torch.uint8


def bgr_format(fmt: str) -> str:
    """The packed BGR format of the same depth: what the forward reads and writes for `fmt`."""
    return "bgr48le" if fmt in DEEP_FORMATS else "bgr24"


def check_format(fmt: str, what: str = "format") -> str:
    if fmt not in FORMATS:
        raise ValueError(f"unknown {what} {fmt!r}: expected one of {', '.join(FORMATS)}")
    return fmt


def check_colorspace(name: str, what: str = "colorspace") -> str:
    """The canonical name of colour matrix `name` (ffmpeg's -colorspace names and aliases)."""
    cs = _COLORSPACE_ALIASES.get(name, name)
    if cs not in COLORSPACES:
        names = [*COLORSPACES, *_COLORSPACE_ALIASES]
        raise ValueError(f"unknown {what} {name!r}: expected one of {', '.join(names)}")
    return cs


def check_color_range(name: str, what: str = "color_range") -> str:
    """The canonical name of colour range `name`: "tv" (limited) or "pc" (full), ffmpeg's -color_range names and aliases."""
    r = _COLOR_RANGE_ALIASES.get(name, name)
    if r not in COLOR_RANGES:
        names = [*COLOR_RANGES, *_COLOR_RANGE_ALIASES]
        raise ValueError(f"unknown {what} {name!r}: expected one of {', '.join(names)}")
    return r


def _cs_args(colorspace: str, color_range: str) -> tuple:
    """() for the default pair ("bt601", "tv"), which the plain entry points convert; else the enumerator values for the _cs ones."""
    cs, r = check_colorspace(colorspace), check_color_range(color_range)
    return () if (cs, r) == ("bt601", "tv") else (COLORSPACES[cs], COLOR_RANGES[r])


def yuv_shape(h: int, w: int) -> Tuple[int, int]:
    """The [rows, w] array one YUV 4:2:0 frame of h x w occupies."""
    return 3 * h // 2, w


def yuv_frames(x: torch.Tensor, fmt: str, h: Optional[int] = None, w: Optional[int] = None) -> torch.Tensor:
    """Check that x holds `fmt` frames (uint8, uint16 for the 10-bit formats; [3h/2, w] or [n, 3h/2, w]; h x w from the shape when not
    given) with a layout the kernels read, and return it as [n, 3h/2, w].  Wherever x lives: the device is the caller's concern."""
    if fmt not in YUV_FORMATS:
        raise ValueError(f"{fmt!r} is not a YUV 4:2:0 format ({', '.join(YUV_FORMATS)})")
    dt = dtype_of(fmt)
    tn = str(dt).replace("torch.", "")
    if x.dtype != dt:
        raise TypeError(f"{fmt} frames are {tn}, got {x.dtype}")
    if h is None:
        rows, w = (x.shape[-2], x.shape[-1]) if x.dim() in (2, 3) else (0, 0)
        if rows % 3 or rows == 0:
            raise ValueError(f"expected {tn} {fmt} frames [3h/2, w] or [n, 3h/2, w], got {tuple(x.shape)}")
        h = 2 * rows // 3
    if h % 2 or w % 2:
        raise ValueError(f"{fmt} needs an even frame size, got {h}x{w}")
    if x.dim() == 2:
        x = x.unsqueeze(0)
    if x.dim() != 3 or tuple(x.shape[1:]) != yuv_shape(h, w):
        rows = yuv_shape(h, w)[0]
        raise ValueError(f"expected {tn} {fmt} frames [{rows}, {w}] or [n, {rows}, {w}], got {tuple(x.shape)}")
    if x.stride(2) != 1:
        raise ValueError(f"{fmt} frames need a unit column stride, got {x.stride(2)}")
    if fmt not in PITCHED_FORMATS and x.stride(1) != w:
        raise ValueError(f"{fmt} frames must have contiguous rows: row stride {x.stride(1)} != width {w} "
                         f"(only {' and '.join(PITCHED_FORMATS)} take a row pitch)")
    if x.stride(1) < w:
        raise ValueError(f"{fmt} row stride {x.stride(1)} is below the width {w}")
    return x


def _planes(x: torch.Tensor, fmt: str, h: int, w: int) -> tuple:
    """(y, y_pitch, u, v, c_pitch, c_step, frame_stride) of frames x [n, 3h/2, w] (checked by yuv_frames): addresses in bytes, pitches
    and the frame stride in elements (bytes for the 8-bit formats, uint16 samples for the 10-bit ones)."""
    p, pitch, e = x.data_ptr(), x.stride(1), x.element_size()
    if fmt not in PITCHED_FORMATS:
        u = p + h * w * e
        return p, w, u, u + (h // 2) * (w // 2) * e, w // 2, 1, x.stride(0)
    u = p + h * pitch * e
    return p, pitch, u, u + e, pitch, 2, x.stride(0)


def _on_cuda(*xs: torch.Tensor) -> torch.device:
    dev = xs[0].device
    for x in xs:
        if not x.is_cuda:
            raise RuntimeError("savsr_b200.colour runs on CUDA (sm_100a) only; there is no CPU fallback")
        if x.device != dev:
            raise ValueError(f"tensors on {dev} and {x.device}")
    return dev


def _bgr(x: torch.Tensor, what: str, dt: torch.dtype = torch.uint8) -> torch.Tensor:
    tn = str(dt).replace("torch.", "")
    if x.dtype != dt:
        raise TypeError(f"{what} takes {tn} BGR frames, got {x.dtype}")
    if x.dim() == 3:
        x = x.unsqueeze(0)
    if x.dim() != 4 or x.shape[3] != 3:
        raise ValueError(f"{what}: expected {tn} BGR frames [h, w, 3] or [n, h, w, 3], got {tuple(x.shape)}")
    if not x.is_contiguous():
        raise ValueError(f"{what}: BGR frames must be contiguous")
    return x


def yuv420_to_bgr(frames: torch.Tensor, fmt: str, out: Optional[torch.Tensor] = None, colorspace: str = "bt601",
                  color_range: str = "tv") -> torch.Tensor:
    """`fmt` frames ([3h/2, w] or [n, 3h/2, w], CUDA) -> BGR [h, w, 3] or [n, h, w, 3] of the same depth.  "yuv420p" and "nv12" (uint8)
    decode to uint8 BGR as cv2.cvtColor(frame, COLOR_YUV2BGR_I420 or COLOR_YUV2BGR_NV12) of each frame; "yuv420p10le" and "p010" (uint16)
    to uint16 bgr48 with the same matrix.  Another `colorspace` / `color_range` than ("bt601", "tv") decodes with that pair's H.273
    map.  Writes `out` (contiguous, that shape and dtype) when given, else a fresh tensor.  One launch on the current stream; the
    frames must stay valid, in stream order, until it has run."""
    cs = _cs_args(colorspace, color_range)
    x = yuv_frames(frames, fmt)
    n, h, w = x.shape[0], 2 * x.shape[1] // 3, x.shape[2]
    shape = (n, h, w, 3) if frames.dim() == 3 else (h, w, 3)
    dt = dtype_of(fmt)
    if out is None:
        _on_cuda(x)
        out = torch.empty(shape, dtype=dt, device=x.device)
    elif tuple(out.shape) != shape or out.dtype != dt or not out.is_contiguous():
        raise ValueError(f"out must be a contiguous {str(dt).replace('torch.', '')} tensor of shape {shape}, got {out.dtype} {tuple(out.shape)}")
    dev = _on_cuda(x, out)
    if n == 0:
        return out
    ctx = engine.context(dev.index)
    y, yp, u, v, cp, c_step, fs = _planes(x, fmt, h, w)
    st = torch.cuda.current_stream(dev).cuda_stream
    with torch.cuda.device(dev):
        if fmt in DEEP_FORMATS:
            args = (ctx.handle, y, yp, u, v, cp, c_step, fs, int(fmt == "p010"), n, h, w, out.data_ptr(), *cs, st)
            K.check((ctx.lib.savsr_yuv420_10_to_bgr48_cs if cs else ctx.lib.savsr_yuv420_10_to_bgr48)(*args))
        else:
            args = (ctx.handle, y, yp, u, v, cp, c_step, fs, n, h, w, out.data_ptr(), *cs, st)
            K.check((ctx.lib.savsr_yuv420_to_bgr_cs if cs else ctx.lib.savsr_yuv420_to_bgr)(*args))
    return out


def bgr_to_yuv420(bgr: torch.Tensor, fmt: str, out: Optional[torch.Tensor] = None, colorspace: str = "bt601",
                  color_range: str = "tv") -> torch.Tensor:
    """BGR [H, W, 3] or [n, H, W, 3] (contiguous, CUDA, H and W even) -> `fmt` frames [3H/2, W] or [n, 3H/2, W].  uint8 BGR to "yuv420p"
    or "nv12" as cv2.cvtColor(frame, COLOR_BGR2YUV_I420) of each frame, with U and V interleaved for "nv12"; uint16 bgr48 to
    "yuv420p10le" or "p010" with the same matrix.  Another `colorspace` / `color_range` than ("bt601", "tv") encodes with that pair's
    H.273 map.  Writes `out` when given (any layout yuv_frames accepts, e.g. a pitched NV12 or P010 surface), else a fresh contiguous
    tensor.  One launch on the current stream."""
    cs = _cs_args(colorspace, color_range)
    if fmt not in YUV_FORMATS:
        raise ValueError(f"{fmt!r} is not a YUV 4:2:0 format ({', '.join(YUV_FORMATS)})")
    dt = dtype_of(fmt)
    x = _bgr(bgr, f"bgr_to_yuv420 to {fmt}", dt)
    n, H, W = x.shape[:3]
    shape = (n, *yuv_shape(H, W)) if bgr.dim() == 4 else yuv_shape(H, W)
    if H % 2 or W % 2:
        raise ValueError(f"{fmt} needs an even frame size, got {H}x{W}")
    if out is None:
        _on_cuda(x)
        out = torch.empty(shape, dtype=dt, device=x.device)
    elif tuple(out.shape) != shape:
        raise ValueError(f"out must have shape {shape}, got {tuple(out.shape)}")
    o = yuv_frames(out, fmt, H, W)
    if n > 1 and o.stride(0) < o.shape[1] * o.stride(1):
        raise ValueError(f"the frames of out overlap: frame stride {o.stride(0)}")
    dev = _on_cuda(x, o)
    if n == 0:
        return out
    ctx = engine.context(dev.index)
    y, yp, u, v, cp, c_step, fs = _planes(o, fmt, H, W)
    st = torch.cuda.current_stream(dev).cuda_stream
    with torch.cuda.device(dev):
        if fmt in DEEP_FORMATS:
            args = (ctx.handle, x.data_ptr(), n, H, W, y, yp, u, v, cp, c_step, fs, int(fmt == "p010"), *cs, st)
            K.check((ctx.lib.savsr_bgr48_to_yuv420_10_cs if cs else ctx.lib.savsr_bgr48_to_yuv420_10)(*args))
        else:
            args = (ctx.handle, x.data_ptr(), n, H, W, y, yp, u, v, cp, c_step, fs, *cs, st)
            K.check((ctx.lib.savsr_bgr_to_yuv420_cs if cs else ctx.lib.savsr_bgr_to_yuv420)(*args))
    return out


def widen(bgr: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """uint8 BGR [h, w, 3] or [n, h, w, 3] (contiguous, CUDA) -> `out`, uint16 of the same shape (contiguous, CUDA): each value times
    257, so that out / 65535 is bgr / 255 exactly.  An 8-bit source enters a 16-bit pipeline this way.  One launch on the current stream."""
    x = _bgr(bgr, "widen")
    if out.dtype != torch.uint16 or tuple(out.shape) != tuple(bgr.shape) or not out.is_contiguous():
        raise ValueError(f"out must be a contiguous uint16 tensor of shape {tuple(bgr.shape)}, got {out.dtype} {tuple(out.shape)}")
    dev = _on_cuda(x, out)
    n, h, w = x.shape[:3]
    if n == 0:
        return out
    ctx = engine.context(dev.index)
    with torch.cuda.device(dev):
        K.check(ctx.lib.savsr_widen_u8_to_u16(ctx.handle, x.data_ptr(), n, h, w, out.data_ptr(), torch.cuda.current_stream(dev).cuda_stream))
    return out
