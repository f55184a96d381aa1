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

YUV 4:2:2 (mezzanine and mastering formats such as ProRes 422, broadcast SDI, capture cards) halves the chroma horizontally only.  Its
width must be even; any height works:

* ``"yuv422p"``: one uint8 [2h, w] array per frame: the Y plane, then the U plane (h x w/2), then the V plane, packed, contiguous rows;
* ``"nv16"``: one uint8 [2h, w] array per frame: the Y plane, then h rows of interleaved U, V bytes (U first); may have a row pitch;
* ``"yuyv422"`` / ``"uyvy422"``: one uint8 [h, 2w] array per frame, rows of Y0 U0 Y1 V0 ... / U0 Y0 V0 Y1 ...; may have a row pitch;
* ``"yuv422p10le"``: uint16 [2h, w] laid out as yuv422p, the value in bits 0-9;
* ``"p210"``: uint16 [2h, w] laid out as nv16, the value in bits 6-15 (read as v >> 6); may have a row pitch.

Decoding gives both pixels of each horizontal pair the pair's (U, V): the 4:2:0 decode's rule, byte for byte
``COLOR_YUV2BGR_YUYV`` / ``_UYVY`` at the default pair.  Encoding computes Y as the 4:2:0 encode does and takes U and V from the left
pixel of each pair, the co-sited chroma position of H.264, HEVC and ProRes 4:2:2, so a 4:2:0 encode is the 4:2:2 encode with its odd
chroma rows dropped.  That is deliberately not cv2's ``COLOR_BGR2YUV_YUYV``, which averages the pair's chroma and rounds Y otherwise.
Every colour pair uses the same per-pixel map as for 4:2:0.

Each call is one launch on the current stream of the tensors' device (savsr_yuv420_to_bgr / savsr_bgr_to_yuv420,
savsr_yuv420_10_to_bgr48 / savsr_bgr48_to_yuv420_10 of libsavsr_sm100, and their _cs forms for the other pairs; the four
savsr_yuv422_* / savsr_bgr*_to_yuv422* _cs calls for 4:2:2); there is no CPU path.  yuv_to_bgr and bgr_to_yuv pick the conversion of
a format's subsampling.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from . import _capi as K, engine

FORMATS = ("bgr24", "yuv420p", "nv12", "bgr48le", "yuv420p10le", "p010", "yuv422p", "nv16", "yuyv422", "uyvy422", "yuv422p10le", "p210")
YUV420_FORMATS = ("yuv420p", "nv12", "yuv420p10le", "p010")
YUV422_FORMATS = ("yuv422p", "nv16", "yuyv422", "uyvy422", "yuv422p10le", "p210")
YUV_FORMATS = YUV420_FORMATS + YUV422_FORMATS
DEEP_FORMATS = ("bgr48le", "yuv420p10le", "p010", "yuv422p10le", "p210")
PITCHED_FORMATS = ("nv12", "p010", "nv16", "p210", "yuyv422", "uyvy422")   # may have a row pitch; their U, V samples are interleaved
PACKED_FORMATS = ("yuyv422", "uyvy422")     # [h, 2w]: Y, U and V in one plane of 4-byte macropixels
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


def _cs_values(colorspace: str, color_range: str) -> tuple:
    """The enumerator values (enum savsr_colorspace, enum savsr_color_range) of a colour pair."""
    return COLORSPACES[check_colorspace(colorspace)], COLOR_RANGES[check_color_range(color_range)]


def yuv_shape(h: int, w: int, fmt: str = "yuv420p") -> Tuple[int, int]:
    """The [rows, cols] array one `fmt` frame of h x w occupies: [3h/2, w] for 4:2:0, [2h, w] for planar and semi-planar 4:2:2,
    [h, 2w] for packed 4:2:2."""
    if fmt in PACKED_FORMATS:
        return h, 2 * w
    if fmt in YUV422_FORMATS:
        return 2 * h, w
    return 3 * h // 2, w


def frame_size(x: torch.Tensor, fmt: str) -> Tuple[int, int]:
    """(h, w) of the `fmt` frames x [n, rows, cols] (checked by yuv_frames)."""
    rows, cols = x.shape[-2], x.shape[-1]
    if fmt in PACKED_FORMATS:
        return rows, cols // 2
    return (rows // 2 if fmt in YUV422_FORMATS else 2 * rows // 3), cols


def _uneven(fmt: str, h: int, w: int) -> str:
    """What of an h x w frame must be even for `fmt` and is not: "size" (4:2:0: height and width), "width" (4:2:2), or "" when
    the size suits `fmt` (and for packed BGR, which takes any size)."""
    if fmt in YUV420_FORMATS and (h % 2 or w % 2):
        return "size"
    if fmt in YUV422_FORMATS and w % 2:
        return "width"
    return ""


def _check_even(fmt: str, h: int, w: int) -> None:
    need = _uneven(fmt, h, w)
    if need:
        raise ValueError(f"{fmt} needs an even {'frame size' if need == 'size' else 'width'}, got {h}x{w}")


def yuv_frames(x: torch.Tensor, fmt: str, h: Optional[int] = None, w: Optional[int] = None) -> torch.Tensor:
    """Check that x holds `fmt` frames (uint8, uint16 for the 10-bit formats; one [rows, cols] array per frame as yuv_shape gives it,
    [n, rows, cols] for several; h x w from the shape when not given) with a layout the kernels read, and return it as [n, rows, cols].
    4:2:0 needs an even frame size, 4:2:2 an even width.  Wherever x lives: the device is the caller's concern."""
    if fmt not in YUV_FORMATS:
        raise ValueError(f"{fmt!r} is not a YUV format ({', '.join(YUV_FORMATS)})")
    dt = dtype_of(fmt)
    tn = str(dt).replace("torch.", "")
    if x.dtype != dt:
        raise TypeError(f"{fmt} frames are {tn}, got {x.dtype}")
    four22 = fmt in YUV422_FORMATS
    if h is None:
        rows, cols = (x.shape[-2], x.shape[-1]) if x.dim() in (2, 3) else (0, 0)
        if fmt in PACKED_FORMATS:
            bad, form = cols % 2 or cols == 0 or rows == 0, "[h, 2w] or [n, h, 2w]"
        elif four22:
            bad, form = rows % 2 or rows == 0, "[2h, w] or [n, 2h, w]"
        else:
            bad, form = rows % 3 or rows == 0, "[3h/2, w] or [n, 3h/2, w]"
        if bad:
            raise ValueError(f"expected {tn} {fmt} frames {form}, got {tuple(x.shape)}")
        h, w = frame_size(x, fmt)
    _check_even(fmt, h, w)
    if x.dim() == 2:
        x = x.unsqueeze(0)
    rows, cols = yuv_shape(h, w, fmt)
    if x.dim() != 3 or tuple(x.shape[1:]) != (rows, cols):
        raise ValueError(f"expected {tn} {fmt} frames [{rows}, {cols}] or [n, {rows}, {cols}], got {tuple(x.shape)}")
    if x.stride(2) != 1:
        raise ValueError(f"{fmt} frames need a unit column stride, got {x.stride(2)}")
    if fmt not in PITCHED_FORMATS and x.stride(1) != cols:
        raise ValueError(f"{fmt} frames must have contiguous rows: row stride {x.stride(1)} != width {w} "
                         f"(only {', '.join(PITCHED_FORMATS)} take a row pitch)")
    if x.stride(1) < cols:
        raise ValueError(f"{fmt} row stride {x.stride(1)} is below the " + (f"width {w}" if cols == w else f"row of {cols} samples"))
    return x


def _planes(x: torch.Tensor, fmt: str, h: int, w: int) -> tuple:
    """(y, y_pitch, y_step, u, v, c_pitch, c_step, frame_stride) of `fmt` frames x (checked by yuv_frames), as the kernels take them:
    addresses in bytes, pitches and the frame stride in elements (bytes for the 8-bit formats, uint16 samples for the 10-bit ones)."""
    p, pitch, e = x.data_ptr(), x.stride(1), x.element_size()
    if fmt == "yuyv422":
        return p, pitch, 2, p + 1, p + 3, pitch, 4, x.stride(0)
    if fmt == "uyvy422":
        return p + 1, pitch, 2, p, p + 2, pitch, 4, x.stride(0)
    if fmt in PITCHED_FORMATS:                 # nv12, p010, nv16, p210: the U, V rows follow the h Y rows at the same pitch
        u = p + h * pitch * e
        return p, pitch, 1, u, u + e, pitch, 2, x.stride(0)
    c_rows = h if fmt in YUV422_FORMATS else h // 2
    u = p + h * w * e
    return p, w, 1, u, u + c_rows * (w // 2) * e, w // 2, 1, x.stride(0)


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
    return _decode(frames, fmt, out, colorspace, color_range, YUV420_FORMATS)


def yuv422_to_bgr(frames: torch.Tensor, fmt: str, out: Optional[torch.Tensor] = None, colorspace: str = "bt601",
                  color_range: str = "tv") -> torch.Tensor:
    """yuv420_to_bgr for the 4:2:2 formats: both pixels of each horizontal pair take the pair's (U, V).  For "yuyv422" / "uyvy422" at the
    default pair this is cv2.cvtColor(frame, COLOR_YUV2BGR_YUYV / _UYVY) of each frame."""
    return _decode(frames, fmt, out, colorspace, color_range, YUV422_FORMATS)


def bgr_to_yuv420(bgr: torch.Tensor, fmt: str, out: Optional[torch.Tensor] = None, colorspace: str = "bt601",
                  color_range: str = "tv") -> torch.Tensor:
    """BGR [H, W, 3] or [n, H, W, 3] (contiguous, CUDA, H and W even) -> `fmt` frames [3H/2, W] or [n, 3H/2, W].  uint8 BGR to "yuv420p"
    or "nv12" as cv2.cvtColor(frame, COLOR_BGR2YUV_I420) of each frame, with U and V interleaved for "nv12"; uint16 bgr48 to
    "yuv420p10le" or "p010" with the same matrix.  Another `colorspace` / `color_range` than ("bt601", "tv") encodes with that pair's
    H.273 map.  Writes `out` when given (any layout yuv_frames accepts, e.g. a pitched NV12 or P010 surface), else a fresh contiguous
    tensor.  One launch on the current stream."""
    return _encode(bgr, fmt, out, colorspace, color_range, YUV420_FORMATS)


def bgr_to_yuv422(bgr: torch.Tensor, fmt: str, out: Optional[torch.Tensor] = None, colorspace: str = "bt601",
                  color_range: str = "tv") -> torch.Tensor:
    """bgr_to_yuv420 for the 4:2:2 formats (W even, any H): Y as the 4:2:0 encode computes it, U and V from the left pixel of each
    horizontal pair (co-sited, as H.264, HEVC and ProRes 4:2:2 site them), so the 4:2:0 encode is this one with its odd chroma rows
    dropped.  Not cv2's COLOR_BGR2YUV_YUYV, which averages the pair's chroma and rounds Y otherwise."""
    return _encode(bgr, fmt, out, colorspace, color_range, YUV422_FORMATS)


def yuv_to_bgr(frames: torch.Tensor, fmt: str, **kw) -> torch.Tensor:
    """yuv420_to_bgr or yuv422_to_bgr, as `fmt` subsamples; the keyword arguments are passed on as given."""
    return (yuv422_to_bgr if fmt in YUV422_FORMATS else yuv420_to_bgr)(frames, fmt, **kw)


def bgr_to_yuv(bgr: torch.Tensor, fmt: str, **kw) -> torch.Tensor:
    """bgr_to_yuv420 or bgr_to_yuv422, as `fmt` subsamples; the keyword arguments are passed on as given."""
    return (bgr_to_yuv422 if fmt in YUV422_FORMATS else bgr_to_yuv420)(bgr, fmt, **kw)


def _family(fmt: str, family: tuple) -> None:
    if fmt not in family:
        raise ValueError(f"{fmt!r} is not a YUV {'4:2:2' if family is YUV422_FORMATS else '4:2:0'} format ({', '.join(family)})")


def _decode(frames, fmt, out, colorspace, color_range, family) -> torch.Tensor:
    pair = _cs_values(colorspace, color_range)
    _family(fmt, family)
    x = yuv_frames(frames, fmt)
    n, (h, w) = x.shape[0], frame_size(x, fmt)
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
    _convert(dev, True, fmt, pair, _planes(x, fmt, h, w), out.data_ptr(), n, h, w)
    return out


def _encode(bgr, fmt, out, colorspace, color_range, family) -> torch.Tensor:
    pair = _cs_values(colorspace, color_range)
    _family(fmt, family)
    four22 = family is YUV422_FORMATS
    dt = dtype_of(fmt)
    x = _bgr(bgr, f"bgr_to_yuv{'422' if four22 else '420'} to {fmt}", dt)
    n, H, W = x.shape[:3]
    shape = (n, *yuv_shape(H, W, fmt)) if bgr.dim() == 4 else yuv_shape(H, W, fmt)
    _check_even(fmt, H, W)
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
    _convert(dev, False, fmt, pair, _planes(o, fmt, H, W), x.data_ptr(), n, H, W)
    return out


# The C entry point of each (decode, 4:2:2, deep).  4:2:0 has a plain form for the default colour pair and a _cs form for any pair;
# 4:2:2 has only the _cs form.
_C_CALLS = {
    (True, False, False): "savsr_yuv420_to_bgr", (True, False, True): "savsr_yuv420_10_to_bgr48",
    (True, True, False): "savsr_yuv422_to_bgr_cs", (True, True, True): "savsr_yuv422_10_to_bgr48_cs",
    (False, False, False): "savsr_bgr_to_yuv420", (False, False, True): "savsr_bgr48_to_yuv420_10",
    (False, True, False): "savsr_bgr_to_yuv422_cs", (False, True, True): "savsr_bgr48_to_yuv422_10_cs",
}


def _convert(dev: torch.device, decode: bool, fmt: str, pair: tuple, planes: tuple, bgr: int, n: int, h: int, w: int) -> None:
    """One conversion between `fmt` frames with `planes` (as _planes gives them) and BGR at address `bgr`, on the current stream."""
    four22, deep = fmt in YUV422_FORMATS, fmt in DEEP_FORMATS
    name, cs = _C_CALLS[decode, four22, deep], pair
    if not four22:
        planes = planes[:2] + planes[3:]        # the 4:2:0 entry points take no y_step
        if pair == (0, 0):
            cs = ()                             # the plain form converts the default pair
        else:
            name += "_cs"
    msb = (int(fmt in ("p010", "p210")),) if deep else ()
    args = (*planes, *msb, n, h, w, bgr) if decode else (bgr, n, h, w, *planes, *msb)
    ctx = engine.context(dev.index)
    with torch.cuda.device(dev):
        K.check(getattr(ctx.lib, name)(ctx.handle, *args, *cs, torch.cuda.current_stream(dev).cuda_stream))


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
