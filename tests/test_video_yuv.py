"""YUV 4:2:0 video in and out: savsr_b200.colour (savsr_yuv420_to_bgr / savsr_bgr_to_yuv420) and VideoUpscaler(in_format, out_format).

The reference is OpenCV: dec = cv2.cvtColor(f, COLOR_YUV2BGR_I420 or COLOR_YUV2BGR_NV12) per frame, enc = cv2.cvtColor(hr,
COLOR_BGR2YUV_I420) with U and V interleaved for nv12, and a stream must give enc(infer_clip(net.forward_bgr_u8, dec(frames), batch)).

CPU: the driver's host logic with cv2 in place of the two conversions and a CPU stand-in for the forward, for every format pair; the
layouts accepted and refused; the C-call arguments against the recording fake library.
GPU, all exact against cv2: both kernels on every (Y, U, V) and every BGR triple, random frames of several sizes and layouts, the C entry
points, and VideoUpscaler with a SAVSR for all nine format pairs.
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

FORMATS = ("bgr24", "yuv420p", "nv12")
PAIRS = [(a, b) for a in FORMATS for b in FORMATS]


# ------------------------------------------------------------------------------------------------ cv2 reference

def cv_dec(frame: np.ndarray, fmt: str) -> np.ndarray:
    code = cv2.COLOR_YUV2BGR_I420 if fmt == "yuv420p" else cv2.COLOR_YUV2BGR_NV12
    return cv2.cvtColor(np.ascontiguousarray(frame), code)


def cv_enc(bgr: np.ndarray, fmt: str) -> np.ndarray:
    i420 = cv2.cvtColor(np.ascontiguousarray(bgr), cv2.COLOR_BGR2YUV_I420)
    if fmt == "yuv420p":
        return i420
    H, W = bgr.shape[:2]
    u, v = i420.reshape(-1)[H * W:].reshape(2, H // 2, W // 2)         # the U plane, then the V plane (not whole rows when H % 4)
    return np.concatenate([i420[:H], np.stack([u, v], -1).reshape(H // 2, W)], 0)


def dec_all(frames, fmt):
    """[n, 3h/2, w] -> [n, h, w, 3] through cv2 (bgr24: unchanged)."""
    x = torch.as_tensor(frames).cpu()
    return x if fmt == "bgr24" else torch.stack([torch.from_numpy(cv_dec(f.numpy(), fmt)) for f in x])


def enc_all(bgr, fmt):
    x = torch.as_tensor(bgr).cpu()
    return x if fmt == "bgr24" else torch.stack([torch.from_numpy(cv_enc(f.numpy(), fmt)) for f in x])


def yuv_from_planes(Y, U, V, fmt, pitch=None):
    """Frames [n, 3h/2, w] (nv12 with row `pitch` when given: a view of a wider buffer) from planes Y [n,h,w], U, V [n,h/2,w/2]."""
    n, h, w = Y.shape
    if fmt == "yuv420p":
        return torch.cat([Y.reshape(n, -1), U.reshape(n, -1), V.reshape(n, -1)], 1).reshape(n, 3 * h // 2, w)
    x = torch.cat([Y, torch.stack([U, V], -1).reshape(n, h // 2, w)], 1)
    if pitch is None or pitch == w:
        return x
    buf = torch.zeros(n, 3 * h // 2, pitch, dtype=torch.uint8, device=x.device)
    buf[:, :, :w] = x
    return buf[:, :, :w]


def random_yuv(n, h, w, fmt, seed, pitch=None, device="cpu"):
    g = torch.Generator().manual_seed(seed)
    Y = torch.randint(0, 256, (n, h, w), dtype=torch.uint8, generator=g)
    U, V = (torch.randint(0, 256, (n, h // 2, w // 2), dtype=torch.uint8, generator=g) for _ in range(2))
    return yuv_from_planes(Y.to(device), U.to(device), V.to(device), fmt, pitch)


# ------------------------------------------------------------------------------------------------ CPU

def _cv_yuv420_to_bgr(frames, fmt, out=None):
    x = colour.yuv_frames(torch.as_tensor(frames), fmt)
    y = dec_all(x, fmt)
    y = y if torch.as_tensor(frames).dim() == 3 else y[0]
    if out is None:
        return y
    out.copy_(y)
    return out


def _cv_bgr_to_yuv420(bgr, fmt, out=None):
    x = torch.as_tensor(bgr)
    y = enc_all(x if x.dim() == 4 else x[None], fmt)
    y = y if x.dim() == 4 else y[0]
    if out is None:
        return y
    out.copy_(y)
    return out


@pytest.fixture
def cv_colour(monkeypatch):
    monkeypatch.setattr(colour, "yuv420_to_bgr", _cv_yuv420_to_bgr)
    monkeypatch.setattr(colour, "bgr_to_yuv420", _cv_bgr_to_yuv420)


def _u8_net(x):
    """Stand-in for forward_bgr_u8: uint8 [n,7,h,w,3] -> uint8 [n,2h,2w,3], a function of every frame of the window."""
    c = x[:, 3].repeat_interleave(2, 1).repeat_interleave(2, 2)
    return (c.int() + x.int().sum(1).repeat_interleave(2, 1).repeat_interleave(2, 2) * 7).to(torch.uint8)


class StandIn:
    """CPU stand-in for a SAVSR in eval mode, with the YUV output conversion of SAVSR._forward_bgr_u8_indexed."""
    training = False

    def __init__(self):
        self.gamma = torch.zeros(1)
        self.formats = []

    def _forward_bgr_u8_indexed(self, pool, windows, scale, out_format="bgr24"):
        self.formats.append(out_format)
        hr = _u8_net(pool[torch.as_tensor(windows)])      # read at call time: a slot rewritten too early shows here
        return hr if out_format == "bgr24" else colour.bgr_to_yuv420(hr, out_format)


def _clip(T, fmt, h=6, w=8, seed=0):
    if fmt == "bgr24":
        return torch.randint(0, 256, (T, h, w, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(seed))
    return random_yuv(T, h, w, fmt, seed)


def _chunkings(T, rng):
    yield [1] * T
    sizes = []
    while sum(sizes) < T:
        sizes.append(min(rng.choice([1, 2, 3, 5, 9, 17, 40]), T - sum(sizes)))
    yield sizes


def _stream(up, frames, chunks):
    outs, k = [], 0
    for n in chunks:
        outs += up.push(frames[k:k + n])
        k += n
    assert k == frames.shape[0]
    return outs + up.finish()


@pytest.mark.parametrize("in_fmt,out_fmt", PAIRS)
@pytest.mark.parametrize("T", [4, 5, 13, 34, 35])
def test_stream_equals_cv2_composition(cv_colour, T, in_fmt, out_fmt):
    batch = (26, 8)
    clip = _clip(T, in_fmt, seed=T)
    want = enc_all(sharding.infer_clip(_u8_net, dec_all(clip, in_fmt), batch=batch), out_fmt)
    rng = random.Random(T)
    feeds = [clip]
    if in_fmt == "nv12":
        feeds.append(yuv_from_planes(clip[:, :6], *_nv12_chroma(clip), "nv12", pitch=24))      # a pitched view of the same frames
        assert feeds[-1].stride(1) == 24 and torch.equal(feeds[-1], clip)
    for frames in feeds:
        for chunks in _chunkings(T, rng):
            net = StandIn()
            up = VideoUpscaler(net, (6, 8), (2, 2), batch=batch, in_format=in_fmt, out_format=out_fmt)
            outs = _stream(up, frames, chunks)
            assert [s for s, _ in outs] == [i for i, _ in sharding.batch_schedule(T, batch)]
            assert torch.equal(torch.cat([y for _, y in outs]), want)
            assert set(net.formats) == {out_fmt}
            assert tuple(up.ring.shape) == (32, 6, 8, 3)                 # the ring stays BGR


def _nv12_chroma(x):
    n, rows, w = x.shape
    uv = x[:, 2 * rows // 3:].reshape(n, rows // 3, w // 2, 2)
    return uv[..., 0], uv[..., 1]


def test_numpy_and_pitched_frames_are_accepted(cv_colour):
    clip = _clip(9, "nv12", seed=3)
    want = enc_all(sharding.infer_clip(_u8_net, dec_all(clip, "nv12"), batch=4), "yuv420p")
    surf = np.zeros((9, 9, 32), np.uint8)                   # decoder surfaces with a 32-byte pitch, as numpy views
    surf[:, :, :8] = clip.numpy()
    up = VideoUpscaler(StandIn(), (6, 8), (2, 2), batch=4, in_format="nv12", out_format="yuv420p")
    outs = []
    for k in range(9):
        outs += up.push(surf[k, :, :8])
    outs += up.finish()
    assert torch.equal(torch.cat([y for _, y in outs]), want)


def test_refusals(cv_colour):
    net = StandIn()
    for bad in ("rgb24", "NV12", "yuv444p", ""):
        with pytest.raises(ValueError, match="unknown in_format"):
            VideoUpscaler(net, (6, 8), (2, 2), in_format=bad)
        with pytest.raises(ValueError, match="unknown out_format"):
            VideoUpscaler(net, (6, 8), (2, 2), out_format=bad)
    for fmt in ("yuv420p", "nv12"):
        with pytest.raises(ValueError, match="even LR size"):
            VideoUpscaler(net, (7, 8), (2, 2), in_format=fmt)
        with pytest.raises(ValueError, match="even LR size"):
            VideoUpscaler(net, (6, 9), (2, 2), in_format=fmt)
        with pytest.raises(ValueError, match=r"scale \(2\.7, 2\.7\) gives H = 389, W = 486"):
            VideoUpscaler(net, (144, 180), (2.7, 2.7), out_format=fmt)
        VideoUpscaler(net, (144, 180), (2.7, 2.7), in_format=fmt)           # bgr24 output takes any scale
        VideoUpscaler(net, (7, 9), (2, 2), out_format=fmt)                  # odd LR, even HR
        up = VideoUpscaler(net, (6, 8), (2, 2), in_format=fmt)
        with pytest.raises(TypeError, match="uint8"):
            up.push(torch.zeros(9, 8))
        with pytest.raises(ValueError, match=r"\[9, 8\]"):
            up.push(torch.zeros(6, 8, 3, dtype=torch.uint8))                 # a BGR frame
        with pytest.raises(ValueError, match=r"\[9, 8\]"):
            up.push(torch.zeros(12, 8, dtype=torch.uint8))
        with pytest.raises(ValueError, match=r"\[9, 8\]"):
            up.push(torch.zeros(2, 9, 10, dtype=torch.uint8))
        with pytest.raises(ValueError, match="column stride"):
            up.push(torch.zeros(9, 16, dtype=torch.uint8)[:, ::2])
        with pytest.raises(ValueError, match="row stride 6"):              # below the width
            up.push(torch.zeros(80, dtype=torch.uint8).as_strided((9, 8), (6, 1)))
        assert up.received == 0
    up = VideoUpscaler(net, (6, 8), (2, 2), in_format="yuv420p")
    with pytest.raises(ValueError, match="contiguous rows"):
        up.push(torch.zeros(9, 16, dtype=torch.uint8)[:, :8])
    up = VideoUpscaler(net, (6, 8), (2, 2), in_format="nv12")
    up.push(torch.zeros(9, 16, dtype=torch.uint8)[:, :8])                    # the same view is a pitched NV12 frame
    assert up.received == 1


class _ClaimsCuda(torch.Tensor):
    """A CPU tensor that reports is_cuda, so the host logic runs without a device (nothing is launched)."""
    is_cuda = property(lambda self: True)


def test_c_call_arguments():
    n, h, w = 3, 6, 8
    c = lambda t: t.as_subclass(_ClaimsCuda)  # noqa: E731
    with mocked_engine() as lib:
        x = c(torch.zeros(n, 9, w, dtype=torch.uint8))
        y = colour.yuv420_to_bgr(x, "yuv420p", out=c(torch.zeros(n, h, w, 3, dtype=torch.uint8)))
        (name, a), = lib.calls
        p = x.data_ptr()
        assert name == "savsr_yuv420_to_bgr"
        assert a[1:11] == (p, w, p + h * w, p + h * w + (h // 2) * (w // 2), w // 2, 1, 9 * w, n, h, w)
        assert a[11] == y.data_ptr() and tuple(y.shape) == (n, h, w, 3)

        lib.calls.clear()
        surf = torch.zeros(n, 9, 64, dtype=torch.uint8).as_subclass(_ClaimsCuda)
        x = surf[:, :, 16:16 + w]                              # pitched NV12 surfaces, starting 16 bytes into each row
        out = torch.zeros(n, h, w, 3, dtype=torch.uint8).as_subclass(_ClaimsCuda)
        assert colour.yuv420_to_bgr(x, "nv12", out=out) is out
        (name, a), = lib.calls
        p = surf.data_ptr() + 16
        assert a[1:11] == (p, 64, p + h * 64, p + h * 64 + 1, 64, 2, 9 * 64, n, h, w) and a[11] == out.data_ptr()

        lib.calls.clear()
        bgr = torch.zeros(n, h, w, 3, dtype=torch.uint8).as_subclass(_ClaimsCuda)
        yo = colour.bgr_to_yuv420(bgr, "yuv420p", out=c(torch.zeros(n, 9, w, dtype=torch.uint8)))
        (name, a), = lib.calls
        q = yo.data_ptr()
        assert name == "savsr_bgr_to_yuv420"
        assert a[1:12] == (bgr.data_ptr(), n, h, w, q, w, q + h * w, q + h * w + (h // 2) * (w // 2), w // 2, 1, 9 * w)

        lib.calls.clear()
        assert colour.bgr_to_yuv420(bgr, "nv12", out=x) is x   # into the pitched surfaces
        (name, a), = lib.calls
        assert a[1:12] == (bgr.data_ptr(), n, h, w, p, 64, p + h * 64, p + h * 64 + 1, 64, 2, 9 * 64)

        lib.calls.clear()
        colour.yuv420_to_bgr(c(torch.zeros(9, w, dtype=torch.uint8)), "nv12", out=c(torch.zeros(h, w, 3, dtype=torch.uint8)))
        colour.bgr_to_yuv420(bgr[0], "nv12", out=c(torch.zeros(9, w, dtype=torch.uint8)))
        assert [lib.calls[0][1][8], lib.calls[1][1][2]] == [1, 1]          # one frame each
        lib.calls.clear()
        colour.yuv420_to_bgr(c(torch.zeros(0, 9, w, dtype=torch.uint8)), "nv12", out=c(torch.zeros(0, h, w, 3, dtype=torch.uint8)))
        assert lib.calls == []                                 # nothing to launch


def test_colour_refusals():
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        colour.yuv420_to_bgr(torch.zeros(9, 8, dtype=torch.uint8), "nv12")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        colour.bgr_to_yuv420(torch.zeros(6, 8, 3, dtype=torch.uint8), "yuv420p")
    c = lambda t: t.as_subclass(_ClaimsCuda)  # noqa: E731
    with pytest.raises(ValueError, match="YUV 4:2:0"):
        colour.yuv420_to_bgr(c(torch.zeros(9, 8, dtype=torch.uint8)), "bgr24")
    with pytest.raises(ValueError, match="YUV 4:2:0"):
        colour.bgr_to_yuv420(c(torch.zeros(6, 8, 3, dtype=torch.uint8)), "i420")
    with pytest.raises(ValueError, match=r"\[3h/2, w\]"):
        colour.yuv420_to_bgr(c(torch.zeros(8, 8, dtype=torch.uint8)), "nv12")
    with pytest.raises(ValueError, match="even frame size"):
        colour.yuv420_to_bgr(c(torch.zeros(9, 7, dtype=torch.uint8)), "nv12")
    with pytest.raises(ValueError, match="even frame size"):
        colour.bgr_to_yuv420(c(torch.zeros(7, 8, 3, dtype=torch.uint8)), "nv12")
    with pytest.raises(ValueError, match="contiguous"):
        colour.bgr_to_yuv420(c(torch.zeros(8, 6, 3, dtype=torch.uint8).transpose(0, 1)), "nv12")
    with pytest.raises(ValueError, match="overlap"):
        colour.bgr_to_yuv420(c(torch.zeros(2, 6, 8, 3, dtype=torch.uint8)), "nv12", out=c(torch.zeros(9, 8, dtype=torch.uint8)).expand(2, 9, 8))
    with pytest.raises(ValueError, match="out must"):
        colour.yuv420_to_bgr(c(torch.zeros(9, 8, dtype=torch.uint8)), "nv12", out=c(torch.zeros(6, 8, 4, dtype=torch.uint8)))


class CpuPlanFrames(CpuPlan):
    io = "bgr_u8_frames"


def test_yuv_output_replaces_the_output_copy():
    """Plan.forward_frames_into with a YUV out_format: the conversion reads the output staging buffer where the copy was."""
    with mocked_engine() as lib:
        plan = CpuPlanFrames(make_state_dict(0), 2, 8, 10, (2, 2), store=engine.WeightStore())
        plan.out = plan.out.as_subclass(_ClaimsCuda)
        H, W = plan.H, plan.W
        out = torch.empty(2, 3 * H // 2, W, dtype=torch.uint8).as_subclass(_ClaimsCuda)
        lib.calls.clear()
        plan.forward_frames_into([0x1000] * 14, out, graph=False, out_format="nv12")
        names = [c[0] for c in lib.calls]
        assert names[0] == "savsr_write_frame_table" and names[-1] == "savsr_bgr_to_yuv420"
        assert names.count("savsr_bgr_to_yuv420") == 1 and "savsr_satu_hr_u8_table" in names
        a = lib.calls[-1][1]
        assert a[1:5] == (plan.out.data_ptr(), 2, H, W) and a[5] == out.data_ptr() and a[10] == 2
        lib.calls.clear()
        with pytest.raises(ValueError, match="unknown out_format"):
            plan.forward_frames_into([0x1000] * 14, out, graph=False, out_format="yuv")
        assert lib.calls == []                                 # refused before any launch


def test_yuv_output_of_the_module(monkeypatch):
    """SAVSR._forward_bgr_u8_indexed(..., out_format): a fresh [b, 3H/2, W] tensor handed to the plan, the empty batch shaped alike."""
    import savsr_b200
    from savsr_b200.archs import savsr_arch
    net = savsr_b200.SAVSR().eval()
    net.load_state_dict(make_state_dict(0), strict=True)
    seen = []

    class Plan(CpuPlanFrames):
        def forward_frames_into(self, ptrs, out, graph=True, out_format="bgr24"):
            seen.append((tuple(out.shape), out_format, len(ptrs)))

    with mocked_engine():
        monkeypatch.setattr(savsr_arch, "engine", SimpleNamespace(**{**vars(engine), "Plan": lambda p, b, h, w, s, d, io="f32", **kw: Plan(p, b, h, w, s, **kw)}))
        pool = torch.zeros(9, 8, 10, 3, dtype=torch.uint8).as_subclass(_ClaimsCuda)
        y = net._forward_bgr_u8_indexed(pool, [[0, 1, 2, 3, 4, 5, 6]] * 2, (2, 2), "yuv420p")
        assert seen == [((2, 24, 20), "yuv420p", 14)] and tuple(y.shape) == (2, 24, 20)
        assert tuple(net._forward_bgr_u8_indexed(pool, [], (2, 2), "nv12").shape) == (0, 24, 20)


# ------------------------------------------------------------------------------------------------ GPU

DEV = torch.device("cuda", 0)


def _np(x):
    return x.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["yuv420p", "nv12"])
def test_decode_every_yuv_triple(fmt):
    """One 4096 x 4096 frame holds all 2^24 (Y, U, V): chroma block b carries (U, V) = divmod(b // 64, 256) and Y = 4 (b % 64) + 0..3."""
    N = 4096
    b = torch.arange(N // 2 * N // 2, device=DEV)
    uv = b // 64
    U, V = (uv // 256).to(torch.uint8).reshape(N // 2, N // 2), (uv % 256).to(torch.uint8).reshape(N // 2, N // 2)
    y4 = (4 * (b % 64)).reshape(N // 2, N // 2)
    Y = torch.stack([torch.stack([y4, y4 + 1], -1), torch.stack([y4 + 2, y4 + 3], -1)], 1).reshape(N, N).to(torch.uint8)
    x = yuv_from_planes(Y[None], U[None], V[None], fmt)
    got = colour.yuv420_to_bgr(x[0], fmt)
    assert np.array_equal(_np(got), cv_dec(_np(x[0]), fmt))


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["yuv420p", "nv12"])
def test_encode_every_bgr_triple(fmt):
    """All 2^24 BGR triples in one 4096 x 4096 frame, rolled by (0|1, 0|1) pixels in three more frames so that every triple also sits
    on the top-left pixel of a 2x2 block, where U and V are taken."""
    N = 4096
    p = torch.arange(N * N, device=DEV, dtype=torch.int32)
    base = torch.stack([p >> 16, (p >> 8) & 255, p & 255], -1).to(torch.uint8).reshape(N, N, 3)
    bgr = torch.stack([base.roll((dy, dx), (0, 1)) for dy in (0, 1) for dx in (0, 1)])
    got = _np(colour.bgr_to_yuv420(bgr, fmt))
    cpu = _np(bgr)
    for k in range(4):
        assert np.array_equal(got[k], cv_enc(cpu[k], fmt)), k


SIZES = [(2, 2), (144, 180), (180, 318), (270, 480), (1080, 1920)]


@pytest.mark.gpu
@pytest.mark.parametrize("h,w", SIZES)
@pytest.mark.parametrize("fmt", ["yuv420p", "nv12"])
def test_random_frames(h, w, fmt):
    n = 3
    x = random_yuv(n, h, w, fmt, seed=h + w, device=DEV)
    got = colour.yuv420_to_bgr(x, fmt)
    assert np.array_equal(_np(got), dec_all(x, fmt).numpy())
    bgr = torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(w)).to(DEV)
    enc = colour.bgr_to_yuv420(bgr, fmt)
    assert enc.is_contiguous() and tuple(enc.shape) == (n, 3 * h // 2, w)
    assert np.array_equal(_np(enc), enc_all(bgr, fmt).numpy())
    # frames and rows that start on odd addresses: every load and store falls back to byte accesses
    buf = torch.zeros(n * x[0].numel() + 1, dtype=torch.uint8, device=DEV)
    xo = buf[1:].view(n, 3 * h // 2, w)
    xo.copy_(x)
    obuf = torch.zeros(got.numel() + 3, dtype=torch.uint8, device=DEV)
    oo = obuf[3:].view(got.shape)
    colour.yuv420_to_bgr(xo, fmt, out=oo)
    assert torch.equal(oo, got)
    colour.bgr_to_yuv420(got, fmt, out=xo)
    assert torch.equal(xo, colour.bgr_to_yuv420(got, fmt))


@pytest.mark.gpu
@pytest.mark.parametrize("h,w,pitch", [(144, 180, 512), (270, 480, 512), (180, 318, 333), (1080, 1920, 2048)])
def test_pitched_nv12(h, w, pitch):
    n = 2
    x = random_yuv(n, h, w, "nv12", seed=pitch, pitch=pitch, device=DEV)
    assert x.stride(1) == pitch and x.stride(0) == pitch * 3 * h // 2
    got = colour.yuv420_to_bgr(x, "nv12")
    assert np.array_equal(_np(got), dec_all(x, "nv12").numpy())
    surf = torch.full((n, 3 * h // 2, pitch), 7, dtype=torch.uint8, device=DEV)
    colour.bgr_to_yuv420(got, "nv12", out=surf[:, :, :w])
    assert np.array_equal(_np(surf[:, :, :w]), enc_all(got, "nv12").numpy())
    assert int((surf[:, :, w:] != 7).sum()) == 0                                 # nothing written past the width


@pytest.mark.gpu
def test_c_entry_points():
    h, w, pitch, n = 36, 44, 64, 2
    x = random_yuv(n, h, w, "nv12", seed=1, pitch=pitch, device=DEV)
    ctx = engine.context(0)
    lib, st = ctx.lib, torch.cuda.current_stream().cuda_stream
    out = torch.zeros(n, h, w, 3, dtype=torch.uint8, device=DEV)
    p = x.data_ptr()
    args = [p, pitch, p + h * pitch, p + h * pitch + 1, pitch, 2, x.stride(0), n, h, w, out.data_ptr(), st]
    assert lib.savsr_yuv420_to_bgr(ctx.handle, *args) == 0
    torch.cuda.synchronize()
    assert np.array_equal(_np(out), dec_all(x, "nv12").numpy())
    yuv = torch.zeros(n, 3 * h // 2, w, dtype=torch.uint8, device=DEV)
    q = yuv.data_ptr()
    eargs = [out.data_ptr(), n, h, w, q, w, q + h * w, q + h * w + h * w // 4, w // 2, 1, yuv.stride(0), st]
    assert lib.savsr_bgr_to_yuv420(ctx.handle, *eargs) == 0
    torch.cuda.synchronize()
    assert np.array_equal(_np(yuv), enc_all(out, "yuv420p").numpy())
    # refusals, before any launch
    out.zero_()
    yuv.zero_()
    for i, v, msg in [(8, h - 1, b"even"), (9, w - 2 + 1, b"even"), (0, None, b"null"), (2, None, b"null"), (10, None, b"null"),
                      (1, w - 2, b"y_pitch"), (4, w - 2, b"c_pitch"), (5, 3, b"c_step"), (5, 0, b"c_step"), (6, -1, b"frame_stride")]:
        bad = list(args)
        bad[i] = v
        assert lib.savsr_yuv420_to_bgr(ctx.handle, *bad) != 0, (i, v)
        assert msg in lib.savsr_last_error(), (i, v, lib.savsr_last_error())
    for i, v, msg in [(2, h + 1, b"even"), (0, None, b"null"), (7, None, b"null"), (5, w - 1, b"y_pitch"), (8, w // 2 - 1, b"c_pitch"),
                      (9, 4, b"c_step")]:
        bad = list(eargs)
        bad[i] = v
        assert lib.savsr_bgr_to_yuv420(ctx.handle, *bad) != 0, (i, v)
        assert msg in lib.savsr_last_error(), (i, v, lib.savsr_last_error())
    torch.cuda.synchronize()
    assert int(out.count_nonzero()) == 0 and int(yuv.count_nonzero()) == 0


def _gpu_net(precision):
    import savsr_b200
    net = savsr_b200.SAVSR().to(DEV).eval()
    net.load_state_dict(make_state_dict(0), strict=True)
    net.precision = precision
    return net


def _feed(clip, fmt, how):
    """The clip's frames one by one as the caller would hand them: pageable host, pinned host, or device (nv12 with a 256-byte pitch)."""
    if how == "pageable":
        return list(clip)
    if how == "pinned":
        return list(clip.pin_memory())
    if fmt == "nv12":
        return list(yuv_from_planes(clip[:, :clip.shape[1] * 2 // 3].to(DEV), *(c.to(DEV) for c in _nv12_chroma(clip)), "nv12", pitch=256))
    return list(clip.to(DEV))


@pytest.mark.gpu
@pytest.mark.parametrize("scale,precision", [((4, 4), "bf16"), ((4, 4), "fp16"), ((1.5, 4), "bf16"), ((1.5, 4), "fp16")])
def test_video_upscaler_all_format_pairs(scale, precision):
    import savsr_b200
    net = _gpu_net(precision)
    h, w, T, batch = 144, 180, 14, (8, 4)
    bgr_clip = torch.randint(0, 256, (T, h, w, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(5))
    g = torch.Generator().manual_seed(6)
    Y = torch.randint(16, 236, (T, h, w), dtype=torch.uint8, generator=g)
    U, V = (torch.randint(16, 241, (T, h // 2, w // 2), dtype=torch.uint8, generator=g) for _ in range(2))
    clips = {"bgr24": bgr_clip, "yuv420p": yuv_from_planes(Y, U, V, "yuv420p"), "nv12": yuv_from_planes(Y, U, V, "nv12")}
    with torch.no_grad():
        hr = {}
        for src in ("bgr24", "yuv420p"):                     # yuv420p and nv12 hold the same planes: one decoded clip
            hr[src] = sharding.infer_clip(lambda x: _forward_bgr_u8(net, x, scale), dec_all(clips[src], src).to(DEV), batch=batch)
        hr["nv12"] = hr["yuv420p"]
        for in_fmt, out_fmt in PAIRS:
            want = enc_all(hr[in_fmt], out_fmt)
            up = savsr_b200.VideoUpscaler(net, (h, w), scale, batch=batch, in_format=in_fmt, out_format=out_fmt)
            for how in ("pageable", "pinned", "device"):
                up.reset()
                outs = []
                for f in _feed(clips[in_fmt], in_fmt, how):
                    outs += up.push(f)
                outs += up.finish()
                got = torch.cat([y for _, y in outs])
                assert got.is_cuda and got.is_contiguous()
                assert [s for s, _ in outs] == [i for i, _ in sharding.batch_schedule(T, batch)]
                assert torch.equal(got.cpu(), want), (in_fmt, out_fmt, how)


def _forward_bgr_u8(net, x, scale):
    net.set_scale(scale)
    return net.forward_bgr_u8(x)


@pytest.mark.gpu
def test_odd_hr_size_is_refused_for_yuv_output():
    import savsr_b200
    net = _gpu_net("bf16")
    for fmt in ("yuv420p", "nv12"):
        with pytest.raises(ValueError, match=r"scale \(2\.7, 2\.7\) gives H = 389, W = 486"):
            savsr_b200.VideoUpscaler(net, (144, 180), (2.7, 2.7), in_format=fmt, out_format=fmt)
    up = savsr_b200.VideoUpscaler(net, (144, 180), (2.7, 2.7), in_format="nv12")
    x = random_yuv(5, 144, 180, "nv12", seed=2, device=DEV)
    with torch.no_grad():
        outs = up.push(x) + up.finish()
        net.set_scale((2.7, 2.7))
        want = sharding.infer_clip(net.forward_bgr_u8, colour.yuv420_to_bgr(x, "nv12"), batch=1)
    assert torch.equal(torch.cat([y for _, y in outs]), want)
