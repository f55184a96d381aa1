"""YUV 4:2:2 video in and out: yuv422p, nv16, yuyv422, uyvy422 (8-bit) and yuv422p10le, p210 (10-bit) through savsr_b200.colour
(savsr_yuv422_to_bgr_cs and the three other 4:2:2 entry points) and VideoUpscaler(in_format, out_format).

The conversions are restated here in integer torch (dec422, enc422) over the pixel maps the 4:2:0 tests pin: cv2's BT.601 limited-range
map (8-bit, tests/test_video_yuv.py), its 10-bit form (tests/test_video_deep.py) and the H.273 maps of the other pairs
(tests/test_video_colorspace.py).  Decoding gives both pixels of a horizontal pair the pair's (U, V); encoding takes U and V from the
pair's left pixel.  The restatement is pinned to cv2's COLOR_YUV2BGR_YUYV / _UYVY and to the 4:2:0 restatements; the kernels must equal
it exactly.

CPU: the restatement, layouts accepted and refused, C-call arguments against the recording fake library, and VideoUpscaler's host
logic with a CPU stand-in net.  GPU: all exact with torch.equal.
"""
import random
from types import SimpleNamespace

import cv2
import numpy as np
import pytest
import torch

from fake_lib import CpuPlan, mocked_engine
from oracle.state_dict_fixture import make_state_dict
from savsr_b200 import colour, engine, sharding
from savsr_b200.videostream import VideoUpscaler
from test_video_colorspace import NEW_PAIRS, dec as dec_h273, enc as enc_h273, dec_frames as dec420_h273, enc_frames as enc420_h273
from test_video_deep import ENC8, KUB, KUG, KVG, KVR, KY, _i64, _u16, dec10, dec_frames10, enc10, enc_frames10, frames10
from test_video_yuv import cv_dec, cv_enc

DEFAULT = ("bt601", "tv")
PAIRS = [DEFAULT, *NEW_PAIRS]
F8 = ("yuv422p", "nv16", "yuyv422", "uyvy422")
F10 = ("yuv422p10le", "p210")
PACKED = ("yuyv422", "uyvy422")


# ------------------------------------------------------------------------------------------------ the restatement (torch int64, any device)

def dec_px(Y, U, V, pair, bits):
    """(Y, U, V) -> [B, G, R] with the pixel map of `pair`."""
    if pair != DEFAULT:
        return dec_h273(Y, U, V, *pair, bits)
    if bits == 10:
        return dec10(Y, U, V)
    y, u, v, half = (Y - 16).clamp(min=0) * KY, U - 128, V - 128, 1 << 19      # common.cuh's cv2 form
    return [((y + half + t) >> 20).clamp(0, 255) for t in (KUB * u, KVG * v + KUG * u, KVR * v)]


def enc_px(R, G, B, pair, bits):
    """(R, G, B) -> [Y, U, V] with the pixel map of `pair`."""
    if pair != DEFAULT:
        return enc_h273(R, G, B, *pair, bits)
    if bits == 10:
        return [enc10(R, G, B, ch) for ch in "YUV"]
    return [(a * R + b * G + c * B + (off << 20) + (1 << 19)) >> 20 for a, b, c, off in (ENC8[ch] for ch in "YUV")]


def frames422(Y, U, V, fmt, pitch=None):
    """[n, *yuv_shape(h, w, fmt)] frames of `fmt` from integer planes Y [n, h, w], U, V [n, h, w/2]; a view with row `pitch` (in
    elements) of a wider buffer when given."""
    n, h, w = Y.shape
    if fmt in PACKED:
        mp = [Y[..., 0::2], U, Y[..., 1::2], V] if fmt == "yuyv422" else [U, Y[..., 0::2], V, Y[..., 1::2]]
        x = torch.stack(mp, -1).reshape(n, h, 2 * w)
    elif fmt in ("yuv422p", "yuv422p10le"):
        x = torch.cat([Y.reshape(n, -1), U.reshape(n, -1), V.reshape(n, -1)], 1).reshape(n, 2 * h, w)
    else:
        x = torch.cat([Y, torch.stack([U, V], -1).reshape(n, h, w)], 1)
    if fmt == "p210":
        x = x << 6
    cols = x.shape[2]
    if pitch is not None and pitch != cols:
        buf = torch.zeros(n, x.shape[1], pitch, dtype=x.dtype, device=x.device)
        buf[:, :, :cols] = x
        x = buf
    x = _u16(x) if fmt in F10 else x.to(torch.uint8)
    return x[:, :, :cols]


def planes422(x, fmt):
    """Frames [n, rows, cols] -> integer planes (Y [n, h, w], U, V [n, h, w/2]) as int64."""
    v = _i64(x) if x.dtype == torch.uint16 else x.to(torch.int64)
    n, rows, cols = v.shape
    if fmt in PACKED:
        mp = v.reshape(n, rows, cols // 4, 4)
        iy, iu, iv = ((0, 2), 1, 3) if fmt == "yuyv422" else ((1, 3), 0, 2)
        return torch.stack([mp[..., iy[0]], mp[..., iy[1]]], -1).reshape(n, rows, cols // 2), mp[..., iu], mp[..., iv]
    h, w = rows // 2, cols
    if fmt in ("yuv422p", "yuv422p10le"):
        flat = v.reshape(n, -1) & 0x3FF if fmt == "yuv422p10le" else v.reshape(n, -1)
        q = h * w // 2
        return flat[:, :h * w].reshape(n, h, w), flat[:, h * w:h * w + q].reshape(n, h, w // 2), flat[:, h * w + q:].reshape(n, h, w // 2)
    v = v >> 6 if fmt == "p210" else v
    uv = v[:, h:].reshape(n, h, w // 2, 2)
    return v[:, :h], uv[..., 0], uv[..., 1]


def dec422(x, fmt, pair=DEFAULT):
    """The restatement of colour.yuv422_to_bgr: frames [n, rows, cols] -> BGR [n, h, w, 3] of the format's depth."""
    Y, U, V = planes422(x, fmt)
    bits = 10 if fmt in F10 else 8
    bgr = torch.stack(dec_px(Y, U.repeat_interleave(2, -1), V.repeat_interleave(2, -1), pair, bits), -1)
    return _u16(bgr) if bits == 10 else bgr.to(torch.uint8)


def enc422(bgr, fmt, pair=DEFAULT, pitch=None):
    """The restatement of colour.bgr_to_yuv422: BGR [n, H, W, 3] -> frames; U and V from the left pixel of each pair."""
    b = _i64(bgr) if bgr.dtype == torch.uint16 else bgr.to(torch.int64)
    B, G, R = b[..., 0], b[..., 1], b[..., 2]
    bits = 10 if fmt in F10 else 8
    Y = enc_px(R, G, B, pair, bits)[0]
    _, U, V = enc_px(R[..., ::2], G[..., ::2], B[..., ::2], pair, bits)
    return frames422(Y, U, V, fmt, pitch)


def frames420(Y, U, V, fmt):
    """4:2:0 frames of `fmt` from integer planes Y [n, h, w], U, V [n, h/2, w/2]."""
    n, h, w = Y.shape
    if fmt in ("yuv420p10le", "p010"):
        return frames10(Y, U, V, fmt)
    if fmt == "yuv420p":
        return torch.cat([Y.reshape(n, -1), U.reshape(n, -1), V.reshape(n, -1)], 1).reshape(n, 3 * h // 2, w).to(torch.uint8)
    return torch.cat([Y, torch.stack([U, V], -1).reshape(n, h // 2, w)], 1).to(torch.uint8)


def dec420(x, fmt, pair=DEFAULT):
    """The 4:2:0 references: cv2 (8-bit, default pair), dec_frames10 (10-bit, default pair), the H.273 restatement (other pairs)."""
    if pair != DEFAULT:
        return dec420_h273(x, fmt, *pair)
    if fmt in colour.DEEP_FORMATS:
        return dec_frames10(x, fmt)
    return torch.stack([torch.from_numpy(cv_dec(f.cpu().numpy(), fmt)) for f in x]).to(x.device)


def enc420(bgr, fmt, pair=DEFAULT):
    if pair != DEFAULT:
        return enc420_h273(bgr, fmt, *pair)
    if fmt in colour.DEEP_FORMATS:
        return enc_frames10(bgr, fmt)
    return torch.stack([torch.from_numpy(cv_enc(f.cpu().numpy(), fmt)) for f in bgr]).to(bgr.device)


def _planes_random(n, h, w, bits, seed, device="cpu"):
    g = torch.Generator().manual_seed(seed)
    top = 1 << bits
    Y = torch.randint(0, top, (n, h, w), generator=g)
    U, V = (torch.randint(0, top, (n, h, w // 2), generator=g) for _ in range(2))
    return Y.to(device), U.to(device), V.to(device)


def _bgr_random(n, h, w, deep, seed, device="cpu"):
    g = torch.Generator().manual_seed(seed)
    if deep:
        return _u16(torch.randint(0, 65536, (n, h, w, 3), generator=g)).to(device)
    return torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, generator=g).to(device)


def _as_int(y):
    return _i64(y) if y.dtype == torch.uint16 else y.to(torch.int64)


# ------------------------------------------------------------------------------------------------ CPU: the restatement

def _every_8bit_triple(device="cpu"):
    """Planes of one 4096 x 4096 frame holding all 2^24 (Y, U, V): pair m carries (U, V) = divmod(m // 128, 256) and Y = 2 (m % 128)
    + 0, 1."""
    N = 4096
    m = torch.arange(N * N // 2, device=device)
    U, V = ((m // 128) // 256).reshape(1, N, N // 2), ((m // 128) % 256).reshape(1, N, N // 2)
    y2 = 2 * (m % 128)
    Y = torch.stack([y2, y2 + 1], -1).reshape(1, N, N)
    return Y, U, V


@pytest.mark.parametrize("fmt,code", [("yuyv422", cv2.COLOR_YUV2BGR_YUYV), ("uyvy422", cv2.COLOR_YUV2BGR_UYVY)])
def test_default_decode_is_cv2_on_every_triple(fmt, code):
    Y, U, V = _every_8bit_triple()
    x = frames422(Y, U, V, fmt)
    want = cv2.cvtColor(np.ascontiguousarray(x[0].numpy()).reshape(4096, 4096, 2), code)
    assert np.array_equal(dec422(x, fmt)[0].numpy(), want)


@pytest.mark.parametrize("fmt", F8 + F10)
def test_layouts_round_trip(fmt):
    Y, U, V = _planes_random(2, 5, 12, 10 if fmt in F10 else 8, seed=1)
    for pitch in (None, 40):
        x = frames422(Y, U, V, fmt, pitch)
        assert tuple(x.shape) == (2, *colour.yuv_shape(5, 12, fmt)) and x.dtype == colour.dtype_of(fmt)
        assert all(torch.equal(a, b) for a, b in zip(planes422(x, fmt), (Y, U, V)))
        assert colour.frame_size(x, fmt) == (5, 12)


@pytest.mark.parametrize("pair", PAIRS)
@pytest.mark.parametrize("bits", [8, 10])
def test_relations_to_420(pair, bits):
    """Decode with doubled chroma rows is the 4:2:0 decode; the encode's Y is the 4:2:0 encode's Y and its even chroma rows the 4:2:0
    encode's chroma."""
    f422, f420 = ("yuv422p", "yuv420p") if bits == 8 else ("yuv422p10le", "yuv420p10le")
    n, h, w = 2, 18, 24
    Y, U, V = _planes_random(n, h, w, bits, seed=bits)
    U, V = U[:, ::2].repeat_interleave(2, 1), V[:, ::2].repeat_interleave(2, 1)
    got = dec422(frames422(Y, U, V, f422), f422, pair)
    assert torch.equal(_as_int(got), _as_int(dec420(frames420(Y, U[:, ::2], V[:, ::2], f420), f420, pair)))
    bgr = _bgr_random(n, h, w, bits == 10, seed=bits + 1)
    Y4, U4, V4 = planes422(enc422(bgr, f422, pair), f422)
    e420 = enc420(bgr, f420, pair)
    x = _as_int(e420) & (0x3FF if bits == 10 else 0xFF)
    flat = x.reshape(n, -1)
    q = h * w // 4
    assert torch.equal(Y4, flat[:, :h * w].reshape(n, h, w))
    assert torch.equal(U4[:, ::2], flat[:, h * w:h * w + q].reshape(n, h // 2, w // 2))
    assert torch.equal(V4[:, ::2], flat[:, h * w + q:].reshape(n, h // 2, w // 2))


# ------------------------------------------------------------------------------------------------ CPU: layouts and refusals

class _ClaimsCuda(torch.Tensor):
    """A CPU tensor that reports is_cuda, so the host logic runs without a device (nothing is launched)."""
    is_cuda = property(lambda self: True)


def _c(t):
    return t.as_subclass(_ClaimsCuda)


def test_layouts_accepted_and_refused():
    assert colour.yuv_shape(5, 8) == colour.yuv_shape(5, 8, "nv12") == (7, 8)
    assert colour.yuv_shape(5, 8, "yuv422p") == colour.yuv_shape(5, 8, "p210") == (10, 8)
    assert colour.yuv_shape(5, 8, "yuyv422") == colour.yuv_shape(5, 8, "uyvy422") == (5, 16)
    for fmt in F8 + F10:
        dt = colour.dtype_of(fmt)
        assert dt == (torch.uint16 if fmt in F10 else torch.uint8) and (fmt in colour.DEEP_FORMATS) == (fmt in F10)
        rows, cols = colour.yuv_shape(5, 8, fmt)
        x = colour.yuv_frames(torch.zeros(rows, cols, dtype=dt), fmt)                  # odd height
        assert tuple(x.shape) == (1, rows, cols)
        with pytest.raises(ValueError, match="even width"):
            colour.yuv_frames(torch.zeros(*colour.yuv_shape(4, 7, fmt), dtype=dt), fmt, 4, 7)
        with pytest.raises(TypeError, match=str(dt).replace("torch.", "")):
            colour.yuv_frames(torch.zeros(rows, cols, dtype=torch.uint16 if dt == torch.uint8 else torch.uint8), fmt)
        with pytest.raises(ValueError, match=r"expected"):
            colour.yuv_frames(torch.zeros(rows + 1, cols, dtype=dt), fmt, 5, 8)
        with pytest.raises(ValueError, match="column stride"):
            colour.yuv_frames(torch.zeros(rows, 2 * cols, dtype=dt)[:, ::2], fmt)
        pitched = torch.zeros(rows, cols + 8, dtype=dt)[:, :cols]
        if fmt in ("yuv422p", "yuv422p10le"):
            with pytest.raises(ValueError, match="contiguous rows"):
                colour.yuv_frames(pitched, fmt)
        else:
            assert colour.yuv_frames(pitched, fmt).stride(1) == cols + 8
    with pytest.raises(ValueError, match=r"\[h, 2w\]"):
        colour.yuv_frames(torch.zeros(5, 15, dtype=torch.uint8), "yuyv422")
    with pytest.raises(ValueError, match=r"\[2h, w\]"):
        colour.yuv_frames(torch.zeros(5, 8, dtype=torch.uint8), "nv16")
    with pytest.raises(ValueError, match="not a YUV 4:2:0 format"):
        colour.yuv420_to_bgr(_c(torch.zeros(10, 8, dtype=torch.uint8)), "nv16")
    with pytest.raises(ValueError, match="not a YUV 4:2:2 format"):
        colour.yuv422_to_bgr(_c(torch.zeros(9, 8, dtype=torch.uint8)), "nv12")
    with pytest.raises(ValueError, match="not a YUV 4:2:2 format"):
        colour.bgr_to_yuv422(_c(torch.zeros(6, 8, 3, dtype=torch.uint8)), "bgr24")
    with pytest.raises(ValueError, match="even width"):
        colour.bgr_to_yuv422(_c(torch.zeros(6, 7, 3, dtype=torch.uint8)), "yuyv422")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        colour.yuv422_to_bgr(torch.zeros(10, 8, dtype=torch.uint8), "nv16")
    for bad in ("rgb24", "NV12", "yuv444p", "", "i420", "yuv"):
        assert bad not in colour.FORMATS
        with pytest.raises(ValueError, match="unknown in_format"):
            VideoUpscaler(StandIn(), (6, 8), (2, 2), in_format=bad)
        with pytest.raises(ValueError, match="unknown out_format"):
            VideoUpscaler(StandIn(), (6, 8), (2, 2), out_format=bad)


def test_upscaler_size_rules():
    net = StandIn()
    for fmt in F8 + F10:
        out = fmt if fmt in F10 else "bgr24"
        with pytest.raises(ValueError, match="even LR width"):
            VideoUpscaler(net, (6, 9), (2, 2), in_format=fmt, out_format=out if fmt in F10 else "bgr24")
        VideoUpscaler(net, (7, 8), (2, 2), in_format=fmt, out_format=out)                          # odd LR height
        up = VideoUpscaler(net, (144, 180), (2.7, 2.7), in_format="bgr48le" if fmt in F10 else "bgr24", out_format=fmt)
        assert engine.get_hw(144, 180, up.scale) == (389, 486)                                     # 4:2:0 refuses this HR size
        H, W = engine.get_hw(6, 7, (2, 3))
        assert W % 2
        with pytest.raises(ValueError, match=f"even HR width: 6x7 at scale .* gives W = {W}"):
            VideoUpscaler(net, (6, 7), (2, 3), in_format="bgr48le" if fmt in F10 else "bgr24", out_format=fmt)
    for a in F10:
        for b in ("bgr24", "nv12", *F8):
            with pytest.raises(ValueError, match=f"deep input {a} with 8-bit output {b}"):       # before any size check
                VideoUpscaler(net, (7, 9), (2.7, 2.7), in_format=a, out_format=b)


# ------------------------------------------------------------------------------------------------ CPU: C-call arguments

def test_420_formats_make_the_same_calls():
    n, h, w = 3, 6, 8
    with mocked_engine() as lib:
        for fmt in ("yuv420p", "nv12", "yuv420p10le", "p010"):
            dt = colour.dtype_of(fmt)
            x, b = _c(torch.zeros(n, 9, w, dtype=dt)), _c(torch.zeros(n, h, w, 3, dtype=dt))
            for kw in ({}, {"colorspace": "bt709", "color_range": "pc"}):
                lib.calls.clear()
                colour.yuv420_to_bgr(x, fmt, out=b, **kw)
                colour.bgr_to_yuv420(b, fmt, out=x, **kw)
                want = list(lib.calls)
                lib.calls.clear()
                colour.yuv_to_bgr(x, fmt, out=b, **kw)
                colour.bgr_to_yuv(b, fmt, out=x, **kw)
                assert lib.calls == want and [c[0].startswith("savsr_yuv420") for c in want] == [True, False]


def test_422_c_call_arguments():
    n, h, w = 3, 5, 8
    with mocked_engine() as lib:
        def one(call):
            lib.calls.clear()
            call()
            (name, a), = lib.calls
            return name, a[1:]
        for fmt in F8 + F10:
            deep = fmt in F10
            dt, e = colour.dtype_of(fmt), 2 if deep else 1
            rows, cols = colour.yuv_shape(h, w, fmt)
            pitched = fmt not in ("yuv422p", "yuv422p10le")
            surf = _c(torch.zeros(n, rows, 64, dtype=dt)) if pitched else None
            x = surf[:, :, 16:16 + cols] if pitched else _c(torch.zeros(n, rows, cols, dtype=dt))
            p = x.data_ptr()
            assert p == (surf.data_ptr() + 16 * e if pitched else p)
            pitch, fs = (64, rows * 64) if pitched else (cols, rows * cols)
            planes = {"yuv422p": (p, w, 1, p + h * w, p + h * w + h * w // 2, w // 2, 1, fs),
                      "yuv422p10le": (p, w, 1, p + 2 * h * w, p + 2 * (h * w + h * w // 2), w // 2, 1, fs),
                      "nv16": (p, pitch, 1, p + h * pitch, p + h * pitch + 1, pitch, 2, fs),
                      "p210": (p, pitch, 1, p + 2 * h * pitch, p + 2 * h * pitch + 2, pitch, 2, fs),
                      "yuyv422": (p, pitch, 2, p + 1, p + 3, pitch, 4, fs),
                      "uyvy422": (p + 1, pitch, 2, p, p + 2, pitch, 4, fs)}[fmt]
            msb = (int(fmt == "p210"),) if deep else ()
            bgr = _c(torch.zeros(n, h, w, 3, dtype=dt))
            dname, ename = ("savsr_yuv422_10_to_bgr48_cs", "savsr_bgr48_to_yuv422_10_cs") if deep else \
                ("savsr_yuv422_to_bgr_cs", "savsr_bgr_to_yuv422_cs")
            for kw, pair in (({}, (0, 0)), ({"colorspace": "bt709", "color_range": "full"}, (1, 1)),
                             ({"colorspace": "bt2020", "color_range": "tv"}, (2, 0))):
                assert one(lambda: colour.yuv_to_bgr(x, fmt, out=bgr, **kw)) == (dname, (*planes, *msb, n, h, w, bgr.data_ptr(), *pair, 0))
                assert one(lambda: colour.bgr_to_yuv(bgr, fmt, out=x, **kw)) == (ename, (bgr.data_ptr(), n, h, w, *planes, *msb, *pair, 0))
            k = 8 + len(msb)
            assert one(lambda: colour.yuv422_to_bgr(x[0], fmt, out=bgr[0]))[1][k:k + 3] == (1, h, w)    # one frame
            lib.calls.clear()
            colour.yuv422_to_bgr(x[:0], fmt, out=bgr[:0])
            with pytest.raises(ValueError, match="unknown colorspace"):
                colour.bgr_to_yuv422(bgr, fmt, out=x, colorspace="bt2020c")
            assert lib.calls == []                                 # nothing to launch, or refused before any launch


class CpuPlanFrames(CpuPlan):
    io = "bgr_u8_frames"


def test_422_output_replaces_the_output_copy(monkeypatch):
    with mocked_engine() as lib:
        plan = CpuPlanFrames(make_state_dict(0), 2, 8, 10, (2, 2), store=engine.WeightStore())
        plan.out = plan.out.as_subclass(_ClaimsCuda)
        H, W = plan.H, plan.W
        out = _c(torch.empty(2, H, 2 * W, dtype=torch.uint8))
        lib.calls.clear()
        plan.forward_frames_into([0x1000] * 14, out, graph=False, out_format="uyvy422")
        names = [c[0] for c in lib.calls]
        assert names[-1] == "savsr_bgr_to_yuv422_cs" and sum(nm.startswith("savsr_satu_hr") for nm in names) == 1
        assert lib.calls[-1][1][1:5] == (plan.out.data_ptr(), 2, H, W) and lib.calls[-1][1][5:8] == (out.data_ptr() + 1, 2 * W, 2)
    import savsr_b200
    from savsr_b200.archs import savsr_arch
    net = savsr_b200.SAVSR().eval()
    net.load_state_dict(make_state_dict(0), strict=True)
    seen = []

    class Plan(CpuPlanFrames):
        def forward_frames_into(self, ptrs, out, graph=True, out_format=None, **kw):
            seen.append((tuple(out.shape), out_format))

    with mocked_engine():
        monkeypatch.setattr(savsr_arch, "engine", SimpleNamespace(**{**vars(engine), "Plan": lambda p, b, h, w, s, d, io="f32", **kw:
                                                                       Plan(p, b, h, w, s, **kw)}))
        pool = _c(torch.zeros(9, 8, 10, 3, dtype=torch.uint8))
        assert tuple(net._forward_bgr_u8_indexed(pool, [[0] * 7] * 2, (2, 2), "nv16").shape) == (2, 32, 20)
        assert tuple(net._forward_bgr_u8_indexed(pool, [], (2, 2), "yuyv422").shape) == (0, 16, 40)
        pool = _c(torch.zeros(1, 144, 180, 3, dtype=torch.uint8))                                   # H = 389
        assert tuple(net._forward_bgr_u8_indexed(pool, [], (2.7, 2.7), "yuv422p").shape) == (0, 2 * 389, 486)
        assert seen == [((2, 32, 20), "nv16")]


# ------------------------------------------------------------------------------------------------ CPU: VideoUpscaler

def cpu_dec(frames, fmt, out=None, colorspace="bt601", color_range="tv"):
    x = colour.yuv_frames(torch.as_tensor(frames), fmt)
    pair = (colour.check_colorspace(colorspace), colour.check_color_range(color_range))
    y = dec422(x, fmt, pair) if fmt in colour.YUV422_FORMATS else dec420(x, fmt, pair)
    y = y if torch.as_tensor(frames).dim() == 3 else y[0]
    return y if out is None else out.copy_(y)


def cpu_enc(bgr, fmt, out=None, colorspace="bt601", color_range="tv"):
    x = torch.as_tensor(bgr)
    pair = (colour.check_colorspace(colorspace), colour.check_color_range(color_range))
    y = (enc422 if fmt in colour.YUV422_FORMATS else enc420)(x if x.dim() == 4 else x[None], fmt, pair)
    y = y if x.dim() == 4 else y[0]
    return y if out is None else out.copy_(y)


@pytest.fixture
def cpu_colour(monkeypatch):
    for name, fn in (("yuv420_to_bgr", cpu_dec), ("yuv422_to_bgr", cpu_dec), ("bgr_to_yuv420", cpu_enc), ("bgr_to_yuv422", cpu_enc)):
        monkeypatch.setattr(colour, name, fn)
    monkeypatch.setattr(colour, "widen", lambda bgr, out: out.copy_(_u16(bgr.to(torch.int32) * 257)))


def _up(c):
    return c.repeat_interleave(2, 1).repeat_interleave(2, 2)


def _net(x, full):
    """Stand-in forward on int64 BGR windows [n,7,h,w,3] -> [n,2h,2w,3], a function of every frame of the window."""
    return (_up(x[:, 3]) + _up(x.sum(1)) * 7) % (full + 1)


class StandIn:
    """CPU stand-in for a SAVSR in eval mode, with the output conversion of SAVSR._forward_bgr_u8_indexed."""
    training = False

    def __init__(self):
        self.gamma = torch.zeros(1)

    def _forward_bgr_u8_indexed(self, pool, windows, scale, out_format=None, out_colorspace="bt601", out_color_range="tv"):
        deep = pool.dtype == torch.uint16
        hr = _net(_as_int(pool[torch.as_tensor(windows)]), 65535 if deep else 255)     # read at call time
        hr = _u16(hr) if deep else hr.to(torch.uint8)
        return hr if out_format is None else colour.bgr_to_yuv(hr, out_format, colorspace=out_colorspace, color_range=out_color_range)


def _clip(T, fmt, h, w, seed, pitch=None):
    if fmt in colour.YUV422_FORMATS:
        return frames422(*_planes_random(T, h, w, 10 if fmt in F10 else 8, seed), fmt, pitch)
    g = torch.Generator().manual_seed(seed)
    Y = torch.randint(0, 256, (T, h, w), generator=g)
    U, V = (torch.randint(0, 256, (T, h // 2, w // 2), generator=g) for _ in range(2))
    return frames420(Y, U, V, fmt)


# (in_format, pitch, in pair, out_format, out pair, marked cuts)
STREAMS = [("yuv422p", None, ("bt709", "pc"), "yuv422p", ("bt2020nc", "tv"), ()),
           ("nv16", 24, DEFAULT, "nv16", DEFAULT, ()),
           ("yuyv422", None, DEFAULT, "yuv422p", DEFAULT, (3, 11)),
           ("uyvy422", 40, DEFAULT, "nv12", DEFAULT, ()),
           ("yuv422p10le", None, DEFAULT, "yuv422p10le", DEFAULT, ()),
           ("p210", 24, DEFAULT, "p210", DEFAULT, ()),
           ("nv12", None, DEFAULT, "yuv422p10le", DEFAULT, ())]


@pytest.mark.parametrize("in_fmt,pitch,in_pair,out_fmt,out_pair,marks", STREAMS)
@pytest.mark.parametrize("T", [4, 5, 13, 34, 35])
def test_stream_equals_the_composition(cpu_colour, T, in_fmt, pitch, in_pair, out_fmt, out_pair, marks):
    batch = (26, 8)
    h, w = (5, 8) if in_fmt in colour.YUV422_FORMATS else (6, 8)          # 4:2:2 takes an odd height
    clip = _clip(T, in_fmt, h, w, seed=T, pitch=pitch)
    if pitch is not None:
        assert clip.stride(1) == pitch
    cuts = [c for c in marks if c < T] or None
    deep = out_fmt in colour.DEEP_FORMATS
    bgr = _as_int(cpu_dec(clip, in_fmt, colorspace=in_pair[0], color_range=in_pair[1]))
    if deep and in_fmt not in colour.DEEP_FORMATS:
        bgr = bgr * 257
    hr = sharding.infer_clip(lambda x: _net(x, 65535 if deep else 255), bgr, batch=batch, cuts=cuts)
    want = _as_int(cpu_enc(_u16(hr) if deep else hr.to(torch.uint8), out_fmt, colorspace=out_pair[0], color_range=out_pair[1]))
    rng = random.Random(T)
    kw = dict(in_colorspace=in_pair[0], in_color_range=in_pair[1], out_colorspace=out_pair[0], out_color_range=out_pair[1])
    for chunks in ([1] * T, [rng.choice([1, 2, 3, 5, 9, 17, 40]) for _ in range(T)]):
        up = VideoUpscaler(StandIn(), (h, w), (2, 2), batch=batch, in_format=in_fmt, out_format=out_fmt, **kw)
        outs, k = [], 0
        for c in chunks:
            if k >= T:
                break
            part = clip[k:k + c]
            new = [t for t in range(k, k + part.shape[0]) if cuts and t in cuts]
            for a, b in zip([k, *new], [*new, k + part.shape[0]]):       # a marked cut starts a push
                if b > a:
                    outs += up.push(clip[a:b], new_scene=a in (cuts or ()))
            k += part.shape[0]
        outs += up.finish()
        assert up.scene_cuts() == (cuts or [])
        assert [s for s, _ in outs] == [i for i, _ in sharding.batch_schedule(T, batch)]
        got = torch.cat([y for _, y in outs])
        assert tuple(got.shape[1:]) == colour.yuv_shape(2 * h, 2 * w, out_fmt)
        assert torch.equal(_as_int(got), want), (chunks,)


# ------------------------------------------------------------------------------------------------ GPU

DEV = torch.device("cuda", 0)


@pytest.mark.gpu
@pytest.mark.parametrize("pair", PAIRS)
def test_decode_every_8bit_triple_on_the_device(pair):
    """All 2^24 (Y, U, V) through each 8-bit layout (nv16, YUYV and UYVY pitched), against the restatement, and for the default pair
    against cv2 on the host copy."""
    Y, U, V = _every_8bit_triple(DEV)
    want = torch.stack(dec_px(Y, U.repeat_interleave(2, -1), V.repeat_interleave(2, -1), pair, 8), -1).to(torch.uint8)
    for fmt, pitch in (("yuv422p", None), ("nv16", 4096 + 64), ("yuyv422", 8192 + 64), ("uyvy422", 8192 + 32)):
        x = frames422(Y, U, V, fmt, pitch)
        got = colour.yuv422_to_bgr(x, fmt, colorspace=pair[0], color_range=pair[1])
        assert torch.equal(got, want), (pair, fmt)
        if pair == DEFAULT and fmt in PACKED:
            code = cv2.COLOR_YUV2BGR_YUYV if fmt == "yuyv422" else cv2.COLOR_YUV2BGR_UYVY
            ref = cv2.cvtColor(np.ascontiguousarray(x[0].cpu().numpy()).reshape(4096, 4096, 2), code)
            assert np.array_equal(got[0].cpu().numpy(), ref), fmt
        del x, got


@pytest.mark.gpu
def test_decode_every_10bit_triple_on_pitched_p210():
    """All 2^30 (Y, U, V) in 16 frames of 8192 x 8192: pair b of chunk c carries (U, V) = divmod(c 2^16 + b // 512, 1024) and
    Y = 2 (b % 512) + 0, 1; P210 with a row pitch."""
    N = 8192
    b = torch.arange(N * N // 2, device=DEV)
    y2 = 2 * (b % 512)
    Y = torch.stack([y2, y2 + 1], -1).reshape(1, N, N)
    for chunk in range(16):
        uv = chunk * 65536 + b // 512
        U, V = (uv // 1024).reshape(1, N, N // 2), (uv % 1024).reshape(1, N, N // 2)
        got = _i64(colour.yuv422_to_bgr(frames422(Y, U, V, "p210", N + 256), "p210"))
        want = dec10(Y, U.repeat_interleave(2, -1), V.repeat_interleave(2, -1))
        for k in range(3):
            assert torch.equal(got[..., k], want[k]), (chunk, k)
        del got, want


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,pair", [("yuv422p10le", DEFAULT)] + [(f, p) for p in NEW_PAIRS for f in F10])
def test_decode_every_uv_pair_10bit(fmt, pair):
    """Every 10-bit (U, V) with a sweep of Y (black and white levels, the ends of the code range, and random values)."""
    b = torch.arange(1 << 20, device=DEV)
    U, V = (b // 1024).reshape(1, 1024, 1024), (b % 1024).reshape(1, 1024, 1024)
    g = torch.Generator().manual_seed(5)
    for y0, y1 in [(0, 1), (63, 64), (65, 512), (940, 941), (1022, 1023), tuple(torch.randint(0, 1024, (2,), generator=g).tolist())]:
        Y = torch.tensor([y0, y1], device=DEV).repeat(1024 * 1024).reshape(1, 1024, 2048)
        x = frames422(Y, U, V, fmt, 2048 + 64 if fmt == "p210" else None)
        got = colour.yuv422_to_bgr(x, fmt, colorspace=pair[0], color_range=pair[1])
        assert torch.equal(_i64(got), _i64(dec422(x, fmt, pair))), (fmt, pair, y0, y1)


ENC_SIZES = [(2, 2), (144, 180), (1080, 1920), (1081, 1920), (37, 182), (270, 1918)]


@pytest.mark.gpu
@pytest.mark.parametrize("h,w", ENC_SIZES)
@pytest.mark.parametrize("pair", [DEFAULT, ("bt709", "tv"), ("bt2020nc", "pc")])
def test_encode_and_decode_sizes(h, w, pair):
    """Encode into contiguous and pitched outputs of 3 frames (tails at widths 182 and 1918, an odd height), and decode the result."""
    n = 3
    kw = dict(colorspace=pair[0], color_range=pair[1])
    for fmt in F8 + F10:
        deep = fmt in F10
        bgr = _bgr_random(n, h, w, deep, seed=h + w, device=DEV)
        want = enc422(bgr, fmt, pair)
        got = colour.bgr_to_yuv422(bgr, fmt, **kw)
        assert got.is_contiguous() and torch.equal(_as_int(got), _as_int(want)), (fmt, h, w)
        if fmt not in ("yuv422p", "yuv422p10le"):
            rows, cols = colour.yuv_shape(h, w, fmt)
            surf = torch.full((n, rows, cols + 96), 7, dtype=torch.int32, device=DEV)
            surf = _u16(surf) if deep else surf.to(torch.uint8)
            colour.bgr_to_yuv422(bgr, fmt, out=surf[:, :, :cols], **kw)
            assert torch.equal(_as_int(surf[:, :, :cols]), _as_int(want)), (fmt, h, w)
            assert int((_as_int(surf[:, :, cols:]) != 7).sum()) == 0                        # nothing written past the row
            assert torch.equal(_as_int(colour.yuv422_to_bgr(surf[:, :, :cols], fmt, **kw)), _as_int(dec422(want, fmt, pair)))
        assert torch.equal(_as_int(colour.yuv422_to_bgr(got, fmt, **kw)), _as_int(dec422(got, fmt, pair))), (fmt, h, w)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", F8)
def test_unaligned_8bit_frames(fmt):
    """Frames and BGR buffers that start on odd addresses: every load and store takes its narrowest form."""
    n, h, w = 2, 33, 184
    x = frames422(*_planes_random(n, h, w, 8, seed=3, device=DEV), fmt)
    buf = torch.zeros(x.numel() + 1, dtype=torch.uint8, device=DEV)
    xo = buf[1:].view(x.shape)
    xo.copy_(x)
    obuf = torch.zeros(n * h * w * 3 + 3, dtype=torch.uint8, device=DEV)
    oo = obuf[3:].view(n, h, w, 3)
    colour.yuv422_to_bgr(xo, fmt, out=oo)
    assert torch.equal(oo, dec422(x, fmt))
    colour.bgr_to_yuv422(oo, fmt, out=xo)
    assert torch.equal(xo, enc422(oo, fmt))


@pytest.mark.gpu
@pytest.mark.parametrize("pair", PAIRS)
def test_relations_to_420_on_the_device(pair):
    n, h, w = 2, 144, 182
    kw = dict(colorspace=pair[0], color_range=pair[1])
    for bits, pairs in ((8, (("yuv422p", "yuv420p"), ("nv16", "nv12"), ("yuyv422", "nv12"))), (10, (("yuv422p10le", "yuv420p10le"),
                                                                                                       ("p210", "p010")))):
        Y, U, V = _planes_random(n, h, w, bits, seed=bits, device=DEV)
        U, V = U[:, ::2].repeat_interleave(2, 1), V[:, ::2].repeat_interleave(2, 1)
        bgr = _bgr_random(n, h, w, bits == 10, seed=7, device=DEV)
        for f422, f420 in pairs:
            d422 = colour.yuv422_to_bgr(frames422(Y, U, V, f422), f422, **kw)
            d420 = colour.yuv420_to_bgr(frames420(Y, U[:, ::2], V[:, ::2], f420), f420, **kw)
            assert torch.equal(_as_int(d422), _as_int(d420)), (pair, f422)
            Y4, U4, V4 = planes422(colour.bgr_to_yuv422(bgr, f422, **kw), f422)
            e420 = colour.bgr_to_yuv420(bgr, f420, **kw)
            assert torch.equal(_as_int(frames420(Y4, U4[:, ::2], V4[:, ::2], f420)), _as_int(e420)), (pair, f422)


@pytest.mark.gpu
def test_c_refusals_leave_the_output_untouched():
    ctx = engine.context(0)
    lib, st = ctx.lib, torch.cuda.current_stream().cuda_stream
    n, h, w, pitch = 2, 5, 16, 64
    x8 = torch.zeros(n, h, pitch, dtype=torch.uint8, device=DEV)             # YUYV rows of 32 bytes in a 64-byte pitch
    b8 = torch.zeros(n, h, w, 3, dtype=torch.uint8, device=DEV)
    p = x8.data_ptr()
    dec8 = [p, pitch, 2, p + 1, p + 3, pitch, 4, h * pitch, n, h, w, b8.data_ptr(), 0, 0, st]
    enc8 = [b8.data_ptr(), n, h, w, p, pitch, 2, p + 1, p + 3, pitch, 4, h * pitch, 0, 0, st]
    x16 = _u16(torch.zeros(n, 2 * h, pitch, device=DEV))                     # P210 in a 64-element pitch
    b16 = _u16(torch.zeros(n, h, w, 3, device=DEV))
    q = x16.data_ptr()
    dec16 = [q, pitch, 1, q + 2 * h * pitch, q + 2 * h * pitch + 2, pitch, 2, 2 * h * pitch, 1, n, h, w, b16.data_ptr(), 0, 0, st]
    enc16 = [b16.data_ptr(), n, h, w, q, pitch, 1, q + 2 * h * pitch, q + 2 * h * pitch + 2, pitch, 2, 2 * h * pitch, 1, 0, 0, st]
    b8.fill_(1)
    assert lib.savsr_bgr_to_yuv422_cs(ctx.handle, *enc8) == 0 and lib.savsr_yuv422_to_bgr_cs(ctx.handle, *dec8) == 0
    torch.cuda.synchronize()
    assert int(x8[:, :, 2 * w:].count_nonzero()) == 0 and int(x8[:, :, :2 * w].count_nonzero()) > 0
    cases = [
        ("savsr_yuv422_to_bgr_cs", dec8, 0, [(10, w - 1, b"even width"), (0, None, b"null"), (11, None, b"null"), (2, 1, b"(1, 4)"),
                                             (6, 2, b"(2, 2)"), (2, 3, b"y_step"), (1, 2 * w - 1, b"y_pitch"), (5, 2 * w - 2, b"c_pitch"),
                                             (3, p + 2, b"packed"), (5, pitch + 1, b"packed"), (7, -1, b"frame_stride"),
                                             (12, 3, b"unknown colorspace 3"), (13, 2, b"unknown color range 2")]),
        ("savsr_bgr_to_yuv422_cs", enc8, 4, [(3, w + 1, b"even width"), (0, None, b"null"), (4, None, b"null"), (6, 1, b"(1, 4)"),
                                             (5, 2 * w - 1, b"y_pitch"), (8, p + 2, b"packed"), (11, -5, b"frame_stride"),
                                             (12, -1, b"unknown colorspace -1")]),
        ("savsr_yuv422_10_to_bgr48_cs", dec16, 0, [(11, 3, b"even width"), (12, None, b"null"), (2, 2, b"(2, 2)"), (6, 4, b"(1, 4)"),
                                                  (1, w - 1, b"y_pitch"), (5, w - 1, b"c_pitch"), (4, q + 2 * h * pitch + 4, b"v = u + 1"),
                                                  (8, 2, b"msb"), (14, 2, b"unknown color range 2")]),
        ("savsr_bgr48_to_yuv422_10_cs", enc16, 4, [(3, 7, b"even width"), (8, None, b"null"), (6, 2, b"(2, 2)"), (10, 3, b"(1, 3)"),
                                                  (12, -1, b"msb"), (13, 5, b"unknown colorspace 5")]),
    ]
    for name, args, out_i, bads in cases:
        fn = getattr(lib, name)
        for i, v, msg in bads:
            bad = list(args)
            bad[i] = v
            assert fn(ctx.handle, *bad) != 0, (name, i, v)
            err = lib.savsr_last_error()
            assert msg in err and name.encode() in err, (name, i, v, err)
    x8.zero_(), b8.zero_(), x16.view(torch.int16).zero_(), b16.view(torch.int16).zero_()
    torch.cuda.synchronize()
    for name, args, out_i, bads in cases:
        for i, v, msg in bads:
            bad = list(args)
            bad[i] = v
            getattr(lib, name)(ctx.handle, *bad)
    torch.cuda.synchronize()
    assert all(int(t.view(torch.uint8).count_nonzero()) == 0 for t in (x8, b8, x16, b16))       # refused before any launch


def _gpu_net(precision):
    import savsr_b200
    net = savsr_b200.SAVSR().to(DEV).eval()
    net.load_state_dict(make_state_dict(0), strict=True)
    net.precision = precision
    return net


def _composition(net, src, in_fmt, out_fmt, batch, pair_in=DEFAULT, pair_out=DEFAULT):
    bgr = colour.yuv_to_bgr(src, in_fmt, colorspace=pair_in[0], color_range=pair_in[1])
    if out_fmt in colour.DEEP_FORMATS:
        if bgr.dtype == torch.uint8:
            bgr = colour.widen(bgr, _u16(torch.zeros(bgr.shape, device=DEV)))
        deep = lambda x: net.forward_bgr48(x.view(torch.uint16)).view(torch.int16)  # noqa: E731
        hr = sharding.infer_clip(deep, bgr.view(torch.int16), batch=batch).view(torch.uint16)
    else:
        hr = sharding.infer_clip(net.forward_bgr_u8, bgr, batch=batch)
    return colour.bgr_to_yuv(hr, out_fmt, colorspace=pair_out[0], color_range=pair_out[1])


GPU_STREAMS = [("yuv422p", "yuv422p"), ("nv16", "nv16"), ("yuyv422", "yuv422p"), ("uyvy422", "nv12"), ("yuv422p10le", "yuv422p10le"),
               ("p210", "p210"), ("nv12", "yuv422p10le"), ("uyvy422", "nv16")]


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "fp16"])
@pytest.mark.parametrize("scale", [(4, 4), (1.5, 4)])
def test_video_upscaler_422_streams(precision, scale):
    import savsr_b200
    net = _gpu_net(precision)
    h, w, T, batch = 144, 180, 13, (8, 4)
    net.set_scale(scale)
    with torch.no_grad():
        for in_fmt, out_fmt in GPU_STREAMS:
            host = _clip(T, in_fmt, h, w, seed=len(in_fmt))
            pitch = {"nv16": 256, "p210": 256, "uyvy422": 512}.get(in_fmt)
            dev = host.to(DEV)
            if pitch:                                              # decoder surfaces with a row pitch
                dev = torch.empty(T, host.shape[1], pitch, dtype=host.dtype, device=DEV)[:, :, :host.shape[2]].copy_(dev)
            want = _as_int(_composition(net, host.to(DEV), in_fmt, out_fmt, batch))
            up = savsr_b200.VideoUpscaler(net, (h, w), scale, batch=batch, in_format=in_fmt, out_format=out_fmt)
            for feed in (list(host), list(dev)):                   # host frames and device frames
                up.reset()
                outs = []
                for f in feed:
                    outs += up.push(f)
                outs += up.finish()
                got = torch.cat([y for _, y in outs])
                assert got.is_cuda and tuple(got.shape[1:]) == colour.yuv_shape(*engine.get_hw(h, w, up.scale), out_fmt)
                assert torch.equal(_as_int(got), want), (precision, scale, in_fmt, out_fmt)


@pytest.mark.gpu
def test_video_upscaler_odd_hr_height_and_detection():
    """(144, 180) at 2.7 gives H = 389, which 4:2:0 refuses and 4:2:2 takes; and a stream with scene detection on, colour pairs on both
    sides, equals the composition with the cuts it reports."""
    import savsr_b200
    net = _gpu_net("bf16")
    with torch.no_grad():
        src = _clip(9, "nv16", 144, 180, seed=2).to(DEV)
        up = savsr_b200.VideoUpscaler(net, (144, 180), (2.7, 2.7), batch=4, in_format="nv16", out_format="yuyv422")
        outs = up.push(src) + up.finish()
        net.set_scale((2.7, 2.7))
        got = torch.cat([y for _, y in outs])
        assert tuple(got.shape) == (9, 389, 2 * 486)
        assert torch.equal(got, _composition(net, src, "nv16", "yuyv422", 4))
        # two still shots, cut at frame 6, which the detector finds
        a, b = _clip(1, "p210", 64, 96, seed=3), _clip(1, "p210", 64, 96, seed=4)
        clip = torch.cat([a.expand(6, -1, -1), b.expand(8, -1, -1)]).to(DEV)
        kw = dict(in_colorspace="bt709", out_colorspace="bt2020nc", out_color_range="pc")
        up = savsr_b200.VideoUpscaler(net, (64, 96), (4, 4), batch=(8, 4), in_format="p210", out_format="yuv422p10le", scene_threshold=10,
                                      **kw)
        outs = []
        for k in range(0, clip.shape[0], 3):
            outs += up.push(clip[k:k + 3])
        outs += up.finish()
        cuts = up.scene_cuts()
        assert cuts == [6]
        net.set_scale((4, 4))
        bgr = colour.yuv_to_bgr(clip, "p210", colorspace="bt709")
        deep = lambda x: net.forward_bgr48(x.view(torch.uint16)).view(torch.int16)  # noqa: E731
        hr = sharding.infer_clip(deep, bgr.view(torch.int16), batch=(8, 4), cuts=cuts).view(torch.uint16)
        want = colour.bgr_to_yuv(hr, "yuv422p10le", colorspace="bt2020nc", color_range="pc")
        assert torch.equal(_i64(torch.cat([y for _, y in outs])), _i64(want))
