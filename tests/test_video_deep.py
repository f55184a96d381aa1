"""Deep video: 16-bit BGR windows through the forward (SAVSR.forward_bgr48[_indexed], engine.Plan(io="bgr48_frames"),
savsr_forward_u16_frames), 10-bit YUV 4:2:0 <-> bgr48 on the device (savsr_b200.colour), and VideoUpscaler with the deep formats.

The contract: forward_bgr48(x) == round(clamp(forward(x'), 0, 1) * 65535) in fp32 with round half to even, x' the windows as fp32 RGB
planes, v / 65535 correctly rounded.  The colour maps are restated here in integer numpy / torch (dec10, enc10) and checked against the
real-valued map and against cv2 on 8-bit data; the kernels must equal the restatement exactly.

CPU: the conversions u16_to_unit uses, the restatement, the launch lists and C-call arguments against the recording fake library, and
VideoUpscaler's host logic with a CPU stand-in for the forward.  GPU: all exact with torch.equal.
"""
import random
from fractions import Fraction
from types import SimpleNamespace

import cv2
import numpy as np
import pytest
import torch

from fake_lib import CpuPlan, mocked_engine
from oracle.state_dict_fixture import make_state_dict
from savsr_b200 import colour, engine, sharding
from savsr_b200.videostream import VideoUpscaler

# common.cuh: the 8-bit matrix, and its 10-bit / 16-bit forms
KY, KVR, KVG, KUG, KUB = 1220542, 1673527, -852492, -409993, 2116026
ENC = {"Y": (8389, 16451, 3199, 64), "U": (-4831, -9498, 14329, 512), "V": (14329, -12012, -2317, 512)}      # (R, G, B, offset)
ENC8 = {"Y": (269484, 528482, 102760, 16), "U": (-155188, -305135, 460324, 128), "V": (460324, -385875, -74448, 128)}
DEEP_OUT = ("bgr48le", "yuv420p10le", "p010")
IN_FORMATS = ("bgr24", "yuv420p", "nv12", "bgr48le", "yuv420p10le", "p010")
PAIRS = [(a, b) for a in IN_FORMATS for b in DEEP_OUT]


def dec10(Y, U, V):
    """10-bit (Y, U, V) -> 16-bit (B, G, R): common.cuh's int64 form.  Works on int64 numpy arrays and torch tensors alike."""
    y = Y - 64
    y = y * (y > 0) * (257 * KY)
    u, v, half = U - 512, V - 512, 1 << 21
    out = []
    for c in (y + half + 257 * KUB * u, y + half + 257 * KVG * v + 257 * KUG * u, y + half + 257 * KVR * v):
        c = c >> 22
        c = c * (c > 0)
        out.append(c - (c - 65535) * (c > 65535))
    return out


def enc10(R, G, B, ch):
    cr, cg, cb, off = ENC[ch]
    return (cr * R + cg * G + cb * B + (off << 21) + (1 << 20)) >> 21


def dec10_real(Y, U, V):
    y = np.maximum(Y - 64, 0).astype(np.float64) * KY
    u, v = (U - 512).astype(np.float64), (V - 512).astype(np.float64)
    return [np.clip(257 / 4 * (y + k) / 2 ** 20, 0, 65535) for k in (KUB * u, KVG * v + KUG * u, KVR * v)]


def enc10_real(R, G, B, ch):
    cr, cg, cb, off = ENC8[ch]
    return 4 * off + 4 * (cr * R.astype(np.float64) + cg * G + cb * B) / (257 * 2 ** 20)


# ------------------------------------------------------------------------------------------------ frames (torch, any device)

def _u16(x):
    """Integer tensor with values in [0, 65535] -> uint16 (through int16, whose conversions every backend has)."""
    x = x.to(torch.int32)
    return (x - 65536 * (x >= 32768)).to(torch.int16).view(torch.uint16)


def _i64(x):
    """uint16 tensor -> int64 values."""
    return x.view(torch.int16).to(torch.int64) & 0xFFFF


def frames10(Y, U, V, fmt, pitch=None):
    """[n, 3h/2, w] uint16 frames of `fmt` from 10-bit planes Y [n,h,w], U, V [n,h/2,w/2]; p010 with row `pitch` when given."""
    n, h, w = Y.shape
    if fmt == "yuv420p10le":
        return _u16(torch.cat([Y.reshape(n, -1), U.reshape(n, -1), V.reshape(n, -1)], 1).reshape(n, 3 * h // 2, w))
    x = torch.cat([Y, torch.stack([U, V], -1).reshape(n, h // 2, w)], 1) << 6
    if pitch is None or pitch == w:
        return _u16(x)
    buf = torch.zeros(n, 3 * h // 2, pitch, dtype=torch.int32, device=x.device)
    buf[:, :, :w] = x
    return _u16(buf)[:, :, :w]


def planes10(x, fmt):
    """uint16 frames [n, 3h/2, w] -> 10-bit planes (Y, U, V) as int64."""
    x = _i64(x)
    n, rows, w = x.shape
    h = 2 * rows // 3
    if fmt == "yuv420p10le":
        flat = x.reshape(n, -1) & 0x3FF
        return flat[:, :h * w].reshape(n, h, w), flat[:, h * w:h * w * 5 // 4].reshape(n, h // 2, w // 2), \
            flat[:, h * w * 5 // 4:].reshape(n, h // 2, w // 2)
    x = x >> 6
    uv = x[:, h:].reshape(n, h // 2, w // 2, 2)
    return x[:, :h], uv[..., 0], uv[..., 1]


def dec_frames10(x, fmt):
    """The restatement of yuv420_to_bgr for 10-bit frames: uint16 [n, 3h/2, w] -> uint16 BGR [n, h, w, 3]."""
    Y, U, V = planes10(x, fmt)
    up = lambda c: c.repeat_interleave(2, 1).repeat_interleave(2, 2)  # noqa: E731
    return _u16(torch.stack(dec10(Y, up(U), up(V)), -1))


def enc_frames10(bgr, fmt):
    b = _i64(bgr)
    B, G, R = b[..., 0], b[..., 1], b[..., 2]
    Y = enc10(R, G, B, "Y")
    tl = lambda c: c[:, ::2, ::2]  # noqa: E731
    U, V = enc10(tl(R), tl(G), tl(B), "U"), enc10(tl(R), tl(G), tl(B), "V")
    return frames10(Y, U, V, fmt)


def cv_dec8(frame, fmt):
    return cv2.cvtColor(np.ascontiguousarray(frame), cv2.COLOR_YUV2BGR_I420 if fmt == "yuv420p" else cv2.COLOR_YUV2BGR_NV12)


def dec_any(frames, fmt):
    """dec of the composition: BGR frames of the source, 8-bit sources widened x 257 (uint16 [n, h, w, 3], on the CPU)."""
    x = torch.as_tensor(frames).cpu()
    if fmt == "bgr24":
        return _u16(x.to(torch.int32) * 257)
    if fmt in ("yuv420p", "nv12"):
        return _u16(torch.stack([torch.from_numpy(cv_dec8(f.numpy(), fmt)) for f in x]).to(torch.int32) * 257)
    return x if fmt == "bgr48le" else dec_frames10(x, fmt)


def enc_any(bgr, fmt):
    return bgr if fmt == "bgr48le" else enc_frames10(bgr, fmt)


# ------------------------------------------------------------------------------------------------ CPU: the conversions

def _rn32(q: Fraction) -> np.float32:
    """q correctly rounded to float32 (round half to even), exactly."""
    f = np.float32(float(q))
    cands = [np.nextafter(f, np.float32(-np.inf)), f, np.nextafter(f, np.float32(np.inf))]
    return min(cands, key=lambda c: (abs(Fraction(float(c)) - q), int(c.view(np.uint32)) & 1))


def _u16_to_unit(u: int) -> np.float32:
    """common.cuh's u16_to_unit, every step rounded once: q = u * RN(1/65535), then q + RN(fma(-q, 65535, u)) * RN(1/65535)."""
    r = np.float32(1) / np.float32(65535)
    q = np.float32(np.float32(u) * r)
    rem = _rn32(Fraction(u) - Fraction(float(q)) * 65535)
    return _rn32(Fraction(float(rem)) * Fraction(float(r)) + Fraction(float(q)))


def test_u16_to_unit_is_the_correctly_rounded_quotient():
    got = np.array([_u16_to_unit(u) for u in range(65536)], np.float32)
    want = np.arange(65536, dtype=np.float32) / np.float32(65535)          # IEEE float32 division: correctly rounded
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    for u in (1, 3, 255, 257, 32768, 65534):
        assert want[u] == _rn32(Fraction(u, 65535))
    assert int((np.arange(65536, dtype=np.float32) * (np.float32(1) / np.float32(65535)) != want).sum()) > 0   # the correction is needed
    u8 = np.arange(256, dtype=np.float32) / np.float32(255)               # u8_to_unit (tests/test_video_u8_io.py)
    assert np.array_equal(got[257 * np.arange(256)].view(np.uint32), u8.view(np.uint32))


def test_decode_restatement_is_within_0_55_of_the_real_map():
    grid = np.unique(np.r_[np.arange(0, 1024, 8), [1, 63, 64, 65, 511, 512, 513, 959, 960, 1022, 1023]])
    U, V = np.meshgrid(grid, grid, indexing="ij")
    U, V = U.reshape(1, -1).astype(np.int64), V.reshape(1, -1).astype(np.int64)
    Y = np.arange(1024, dtype=np.int64).reshape(-1, 1)
    got, real = dec10(Y, U, V), dec10_real(Y, U, V)
    for g, r in zip(got, real):
        assert g.min() >= 0 and g.max() <= 65535
        assert float(np.abs(g - r).max()) <= 0.55
    assert int(got[2].max()) == 65535 and int(got[0].min()) == 0             # both ends saturate


def test_encode_restatement_is_within_0_55_of_the_real_map():
    rng = np.random.default_rng(0)
    ends = np.array([0, 1, 256, 32767, 32768, 65279, 65534, 65535])
    e = np.stack(np.meshgrid(ends, ends, ends, indexing="ij"), -1).reshape(-1, 3)
    bgr = np.concatenate([e, rng.integers(0, 65536, (1 << 20, 3))]).astype(np.int64)
    B, G, R = bgr[:, 0], bgr[:, 1], bgr[:, 2]
    for ch, (lo, hi) in {"Y": (64, 940), "U": (64, 960), "V": (64, 960)}.items():
        got = enc10(R, G, B, ch)
        assert float(np.abs(got - enc10_real(R, G, B, ch)).max()) <= 0.55
        assert got.min() >= lo and got.max() <= hi
        cr, cg, cb, off = ENC[ch]                # the int32 bound the kernel relies on
        assert 0 < (min(cr, 0) + min(cg, 0) + min(cb, 0)) * 65535 + (off << 21) and \
            (max(cr, 0) + max(cg, 0) + max(cb, 0)) * 65535 + (off << 21) + (1 << 20) < 2 ** 31


def _every_yuv8_frame():
    """One 4096 x 4096 I420 frame holding all 2^24 (Y, U, V) (as tests/test_video_yuv.py builds it), and its planes."""
    N = 4096
    b = np.arange(N // 2 * N // 2)
    U, V = ((b // 64) // 256).reshape(N // 2, N // 2), ((b // 64) % 256).reshape(N // 2, N // 2)
    y4 = (4 * (b % 64)).reshape(N // 2, N // 2)
    Y = np.stack([np.stack([y4, y4 + 1], -1), np.stack([y4 + 2, y4 + 3], -1)], 1).reshape(N, N)
    i420 = np.concatenate([Y.reshape(-1), U.reshape(-1), V.reshape(-1)]).astype(np.uint8).reshape(3 * N // 2, N)
    return i420, Y, U, V


def test_decode_agrees_with_cv2_on_every_8bit_triple():
    i420, Y, U, V = _every_yuv8_frame()
    bgr8 = cv2.cvtColor(i420, cv2.COLOR_YUV2BGR_I420).astype(np.int64)
    up = lambda c: c.repeat(2, 0).repeat(2, 1).astype(np.int64)  # noqa: E731
    for k, c in enumerate(dec10(Y.astype(np.int64) << 2, up(U) << 2, up(V) << 2)):
        assert int(np.abs(c - 257 * bgr8[..., k]).max()) <= 130, k


def test_encode_agrees_with_cv2_on_every_8bit_triple():
    N = 4096
    p = np.arange(N * N)
    base = np.stack([p >> 16, (p >> 8) & 255, p & 255], -1).astype(np.uint8).reshape(N, N, 3)
    for dy, dx in ((0, 0), (0, 1), (1, 0), (1, 1)):            # every triple on the top-left pixel of a 2x2 block once
        bgr8 = np.roll(base, (dy, dx), (0, 1))
        i420 = cv2.cvtColor(bgr8, cv2.COLOR_BGR2YUV_I420).reshape(-1).astype(np.int64)
        b16 = 257 * bgr8.astype(np.int64)
        B, G, R = b16[..., 0], b16[..., 1], b16[..., 2]
        if (dy, dx) == (0, 0):
            assert int(np.abs(enc10(R, G, B, "Y") - 4 * i420[:N * N].reshape(N, N)).max()) <= 3
        tl = lambda c: c[::2, ::2]  # noqa: E731
        q = N * N // 4
        for ch, plane in (("U", i420[N * N:N * N + q]), ("V", i420[N * N + q:])):
            assert int(np.abs(enc10(tl(R), tl(G), tl(B), ch) - 4 * plane.reshape(N // 2, N // 2)).max()) <= 3, (ch, dy, dx)


# ------------------------------------------------------------------------------------------------ CPU: the plan and the module

class CpuPlanFrames(CpuPlan):
    io = "bgr_u8_frames"


class CpuPlanDeep(CpuPlan):
    io = "bgr48_frames"


class _ClaimsCuda(torch.Tensor):
    """A CPU tensor that reports is_cuda, so the host logic runs without a device (nothing is launched)."""
    is_cuda = property(lambda self: True)


def _record(cls, sd, store, b=2, h=13, w=15, scale=(1.5, 4)):
    with mocked_engine() as lib:
        plan = cls(sd, b, h, w, scale, store=store)
        for op in plan.ops:
            assert op(0) == 0
        return plan, list(lib.calls)


@pytest.fixture(scope="module")
def sd():
    return make_state_dict(0)


def test_deep_plan_swaps_only_the_first_and_last_launch(sd):
    store = engine.WeightStore()
    _record(CpuPlanFrames, sd, store)
    n_keys = len(store.cache)
    p8, c8 = _record(CpuPlanFrames, sd, store)
    pd, cd = _record(CpuPlanDeep, sd, store)
    assert len(store.cache) == n_keys                  # the deep plan's derived weights all came from the shared store
    n8, nd = [c[0] for c in c8], [c[0] for c in cd]
    assert len(n8) == len(nd) and p8.n_launches == pd.n_launches
    assert [(a, b) for a, b in zip(n8, nd) if a != b] == [("savsr_pack_frames_u8_table", "savsr_pack_frames_u16_table"),
                                                         ("savsr_satu_hr_u8_table", "savsr_satu_hr_u16_table")]
    for a, b in zip(c8, cd):
        assert [v for v in a[1] if isinstance(v, (float, str))] == [v for v in b[1] if isinstance(v, (float, str))]
    run = cd[-len(pd.ops):]
    table = pd.frame_table.data_ptr()
    assert run[0][0] == "savsr_pack_frames_u16_table" and run[0][1][2] == table and run[0][1][3:7] == (7, 13, 15, 1)
    assert run[-1][0] == "savsr_satu_hr_u16_table" and run[-1][1][14] == table and run[-1][1][17] == pd.out.data_ptr()
    assert pd.x_in is None and pd.frame_table.dtype == torch.int64 and tuple(pd.frame_table.shape) == (14,)
    assert pd.out.dtype == torch.uint16 and tuple(pd.out.shape) == (2, *engine.get_hw(13, 15, (1.5, 4)), 3)
    with pytest.raises(ValueError, match="forward_frames_into"):
        pd.forward_into(torch.zeros(2, 7, 13, 15, 3, dtype=torch.uint16), torch.empty_like(pd.out))


def test_deep_output_formats_of_the_plan(sd):
    with mocked_engine() as lib:
        plan = CpuPlanDeep(sd, 2, 8, 10, (2, 2), store=engine.WeightStore())
        plan.out = plan.out.as_subclass(_ClaimsCuda)
        H, W = plan.H, plan.W
        out = torch.empty(2, 3 * H // 2, W + 8, dtype=torch.uint16).as_subclass(_ClaimsCuda)[:, :, :W]      # a pitched P010 surface
        lib.calls.clear()
        plan.forward_frames_into([0x1000] * 14, out, graph=False, out_format="p010")
        names = [c[0] for c in lib.calls]
        assert names[0] == "savsr_write_frame_table" and names[-1] == "savsr_bgr48_to_yuv420_10" and "savsr_satu_hr_u16_table" in names
        a = lib.calls[-1][1]
        p = out.data_ptr()
        assert a[1:5] == (plan.out.data_ptr(), 2, H, W)
        assert a[5:14] == (p, W + 8, p + 2 * H * (W + 8), p + 2 * H * (W + 8) + 2, W + 8, 2, out.stride(0), 1, 0)
        lib.calls.clear()
        for bad in ("nv12", "bgr24"):
            with pytest.raises(ValueError, match="another depth"):
                plan.forward_frames_into([0x1000] * 14, out, graph=False, out_format=bad)
        assert lib.calls == []


def _cpu_net():
    import savsr_b200
    net = savsr_b200.SAVSR().eval()
    net.load_state_dict(make_state_dict(0), strict=True)
    net.set_scale((2, 2))
    return net


def test_forward_bgr48_and_indexed_host_logic(monkeypatch):
    net = _cpu_net()
    seen = []

    class Plan(CpuPlanDeep):
        def forward_frames_into(self, ptrs, out, graph=True, out_format=None):
            seen.append((tuple(out.shape), out.dtype, out_format, list(ptrs)))

    from savsr_b200.archs import savsr_arch
    built = []

    def make(p, b, h, w, s, d, io="f32", **kw):
        built.append(io)
        return Plan(p, b, h, w, s, **kw)

    with mocked_engine():
        monkeypatch.setattr(savsr_arch, "engine", SimpleNamespace(**{**vars(engine), "Plan": make}))
        x = torch.zeros(2, 7, 8, 10, 3, dtype=torch.uint16).as_subclass(_ClaimsCuda)
        y = net.forward_bgr48(x)
        f = 8 * 10 * 3 * 2
        assert built == ["bgr48_frames"] and y.dtype == torch.uint16 and tuple(y.shape) == (2, 16, 20, 3)
        assert seen[-1][2] == "bgr48le" and seen[-1][3] == [x.data_ptr() + k * f for k in range(14)]
        pool = torch.zeros(9, 8, 10, 3, dtype=torch.uint16).as_subclass(_ClaimsCuda)
        y = net.forward_bgr48_indexed(pool, [[0, 1, 2, 3, 4, 5, 8]])
        assert tuple(y.shape) == (1, 16, 20, 3) and seen[-1][3] == [pool.data_ptr() + k * f for k in (0, 1, 2, 3, 4, 5, 8)]
        y = net._forward_bgr_u8_indexed(pool, [[0] * 7] * 2, (2, 2), "yuv420p10le")      # the mode follows the pool's dtype
        assert tuple(y.shape) == (2, 24, 20) and y.dtype == torch.uint16 and seen[-1][2] == "yuv420p10le"
        assert tuple(net._forward_bgr_u8_indexed(pool, [], (2, 2), "p010").shape) == (0, 24, 20)
        assert tuple(net.forward_bgr48(x[:0]).shape) == (0, 16, 20, 3) and net.forward_bgr48(x[:0]).dtype == torch.uint16
        assert sorted({k[9] for k in net._plans}) == ["bgr48_frames"]
        with pytest.raises(ValueError, match="another depth"):
            net._forward_bgr_u8_indexed(pool, [[0] * 7], (2, 2), "nv12")
        # the refusals of the 8-bit calls
        with pytest.raises(TypeError, match="uint16"):
            net.forward_bgr48(x.view(torch.int16))
        with pytest.raises(TypeError, match="uint16"):
            net.forward_bgr48_indexed(pool.view(torch.int16), [[0] * 7])
        with pytest.raises(TypeError, match="uint8"):
            net.forward_bgr_u8_indexed(pool, [[0] * 7])                 # the 8-bit call does not take deep frames
        with pytest.raises(ValueError, match=r"\[b, 7, h, w, 3\]"):
            net.forward_bgr48(torch.zeros(2, 7, 3, 8, 10, dtype=torch.uint16).as_subclass(_ClaimsCuda))
        with pytest.raises(ValueError, match=r"\[N, h, w, 3\]"):
            net.forward_bgr48_indexed(pool[0], [[0] * 7])
        with pytest.raises(ValueError, match="contiguous"):
            net.forward_bgr48_indexed(torch.zeros(9, 10, 8, 3, dtype=torch.uint16).transpose(1, 2).as_subclass(_ClaimsCuda), [[0] * 7])
        with pytest.raises(IndexError, match="9 frames"):
            net.forward_bgr48_indexed(pool, [[0, 1, 2, 3, 4, 5, 9]])
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            net.forward_bgr48(torch.zeros(1, 7, 8, 10, 3, dtype=torch.uint16))
        net.train()
        for call in (lambda: net.forward_bgr48(x), lambda: net.forward_bgr48_indexed(pool, [[0] * 7])):
            with pytest.raises(RuntimeError, match="inference only"):
                call()


def test_c_call_arguments():
    n, h, w = 3, 6, 8
    c = lambda t: t.as_subclass(_ClaimsCuda)  # noqa: E731
    with mocked_engine() as lib:
        x = c(torch.zeros(n, 9, w, dtype=torch.uint16))
        y = colour.yuv420_to_bgr(x, "yuv420p10le", out=c(torch.zeros(n, h, w, 3, dtype=torch.uint16)))
        (name, a), = lib.calls
        p = x.data_ptr()
        assert name == "savsr_yuv420_10_to_bgr48" and y.dtype == torch.uint16 and tuple(y.shape) == (n, h, w, 3)
        assert a[1:13] == (p, w, p + 2 * h * w, p + 2 * (h * w + h * w // 4), w // 2, 1, 9 * w, 0, n, h, w, y.data_ptr())
        lib.calls.clear()
        surf = c(torch.zeros(n, 9, 64, dtype=torch.uint16))
        x = surf[:, :, 16:16 + w]                          # pitched P010 surfaces, 16 samples into each row
        out = c(torch.zeros(n, h, w, 3, dtype=torch.uint16))
        assert colour.yuv420_to_bgr(x, "p010", out=out) is out
        (name, a), = lib.calls
        p = surf.data_ptr() + 32
        assert a[1:13] == (p, 64, p + 2 * h * 64, p + 2 * h * 64 + 2, 64, 2, 9 * 64, 1, n, h, w, out.data_ptr())
        lib.calls.clear()
        assert colour.bgr_to_yuv420(out, "p010", out=x) is x
        (name, a), = lib.calls
        assert name == "savsr_bgr48_to_yuv420_10"
        assert a[1:13] == (out.data_ptr(), n, h, w, p, 64, p + 2 * h * 64, p + 2 * h * 64 + 2, 64, 2, 9 * 64, 1)
        lib.calls.clear()
        src, dst = c(torch.zeros(n, h, w, 3, dtype=torch.uint8)), c(torch.zeros(n, h, w, 3, dtype=torch.uint16))
        assert colour.widen(src, dst) is dst
        assert lib.calls == [("savsr_widen_u8_to_u16", ("ctx", src.data_ptr(), n, h, w, dst.data_ptr(), 0))]
        lib.calls.clear()
        colour.yuv420_to_bgr(c(torch.zeros(0, 9, w, dtype=torch.uint16)), "p010", out=c(torch.zeros(0, h, w, 3, dtype=torch.uint16)))
        colour.widen(c(torch.zeros(0, h, w, 3, dtype=torch.uint8)), c(torch.zeros(0, h, w, 3, dtype=torch.uint16)))
        assert lib.calls == []
        # dtype, shape and layout refusals
        with pytest.raises(TypeError, match="uint16"):
            colour.yuv420_to_bgr(c(torch.zeros(9, w, dtype=torch.uint8)), "p010")
        with pytest.raises(TypeError, match="uint8"):
            colour.yuv420_to_bgr(c(torch.zeros(9, w, dtype=torch.uint16)), "nv12")
        with pytest.raises(TypeError, match="uint16"):
            colour.bgr_to_yuv420(src, "yuv420p10le")
        with pytest.raises(TypeError, match="uint8"):
            colour.bgr_to_yuv420(dst, "nv12")
        with pytest.raises(ValueError, match="contiguous rows"):
            colour.yuv420_to_bgr(surf[:, :, :w], "yuv420p10le")            # only p010 takes a pitch
        with pytest.raises(ValueError, match="even frame size"):
            colour.yuv420_to_bgr(c(torch.zeros(9, 7, dtype=torch.uint16)), "p010")
        with pytest.raises(ValueError, match=r"\[3h/2, w\]"):
            colour.yuv420_to_bgr(c(torch.zeros(8, 8, dtype=torch.uint16)), "yuv420p10le")
        with pytest.raises(ValueError, match="out must"):
            colour.yuv420_to_bgr(c(torch.zeros(9, w, dtype=torch.uint16)), "p010", out=c(torch.zeros(h, w, 3, dtype=torch.uint8)))
        with pytest.raises(ValueError, match="out must"):
            colour.widen(src, c(torch.zeros(n, h, w, 3, dtype=torch.uint8)))
        assert lib.calls == []


# ------------------------------------------------------------------------------------------------ CPU: VideoUpscaler

def _cpu_yuv420_to_bgr(frames, fmt, out=None):
    x = colour.yuv_frames(torch.as_tensor(frames), fmt)
    y = dec_frames10(x, fmt) if fmt in colour.DEEP_FORMATS else torch.stack([torch.from_numpy(cv_dec8(f.numpy(), fmt)) for f in x])
    y = y if torch.as_tensor(frames).dim() == 3 else y[0]
    return y if out is None else out.copy_(y)


def _cpu_bgr_to_yuv420(bgr, fmt, out=None):
    assert fmt in colour.DEEP_FORMATS
    x = torch.as_tensor(bgr)
    y = enc_frames10(x if x.dim() == 4 else x[None], fmt)
    y = y if x.dim() == 4 else y[0]
    return y if out is None else out.copy_(y)


@pytest.fixture
def cpu_colour(monkeypatch):
    widened = []

    def widen(bgr, out):
        assert bgr.dtype == torch.uint8 and out.dtype == torch.uint16
        widened.append(tuple(bgr.shape))
        return out.copy_(_u16(bgr.to(torch.int32) * 257))
    monkeypatch.setattr(colour, "yuv420_to_bgr", _cpu_yuv420_to_bgr)
    monkeypatch.setattr(colour, "bgr_to_yuv420", _cpu_bgr_to_yuv420)
    monkeypatch.setattr(colour, "widen", widen)
    return widened


def _net16(x):
    """Stand-in for forward_bgr48 on int64 values [n,7,h,w,3] -> [n,2h,2w,3], a function of every frame of the window."""
    up = lambda c: c.repeat_interleave(2, 1).repeat_interleave(2, 2)  # noqa: E731
    return (up(x[:, 3]) + up(x.sum(1)) * 7) % 65536


class StandIn:
    """CPU stand-in for a SAVSR in eval mode, with the output conversion of SAVSR._forward_bgr_u8_indexed."""
    training = False

    def __init__(self):
        self.gamma = torch.zeros(1)
        self.calls = []

    def _forward_bgr_u8_indexed(self, pool, windows, scale, out_format=None):
        self.calls.append((pool.dtype, out_format))
        hr = _u16(_net16(_i64(pool[torch.as_tensor(windows)])))    # read at call time: a slot rewritten too early shows here
        return hr if out_format is None else colour.bgr_to_yuv420(hr, out_format)


def _clip(T, fmt, h=6, w=8, seed=0, pitch=None):
    g = torch.Generator().manual_seed(seed)
    if fmt == "bgr24":
        return torch.randint(0, 256, (T, h, w, 3), dtype=torch.uint8, generator=g)
    if fmt == "bgr48le":
        return _u16(torch.randint(0, 65536, (T, h, w, 3), generator=g))
    if fmt in ("yuv420p", "nv12"):
        Y = torch.randint(0, 256, (T, h, w), dtype=torch.uint8, generator=g)
        U, V = (torch.randint(0, 256, (T, h // 2, w // 2), dtype=torch.uint8, generator=g) for _ in range(2))
        if fmt == "yuv420p":
            return torch.cat([Y.reshape(T, -1), U.reshape(T, -1), V.reshape(T, -1)], 1).reshape(T, 3 * h // 2, w)
        return torch.cat([Y, torch.stack([U, V], -1).reshape(T, h // 2, w)], 1)
    Y = torch.randint(0, 1024, (T, h, w), generator=g)
    U, V = (torch.randint(0, 1024, (T, h // 2, w // 2), generator=g) for _ in range(2))
    return frames10(Y, U, V, fmt, pitch)


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
    return outs + up.finish()


def _cat(outs):
    return torch.cat([_i64(y) for _, y in outs])


def _composition(clip, in_fmt, out_fmt, batch):
    hr = sharding.infer_clip(lambda x: _net16(x), _i64(dec_any(clip, in_fmt)), batch=batch)
    return _i64(enc_any(_u16(hr), out_fmt))


@pytest.mark.parametrize("in_fmt,out_fmt", PAIRS)
@pytest.mark.parametrize("T", [4, 5, 13, 34, 35])
def test_stream_equals_the_composition(cpu_colour, T, in_fmt, out_fmt):
    batch = (26, 8)
    clip = _clip(T, in_fmt, seed=T)
    want = _composition(clip, in_fmt, out_fmt, batch)
    rng = random.Random(T)
    feeds = [clip]
    if in_fmt == "p010":
        feeds.append(_clip(T, "p010", seed=T, pitch=24))             # a pitched view of the same frames
        assert feeds[-1].stride(1) == 24 and torch.equal(_i64(feeds[-1]), _i64(clip))
    for frames in feeds:
        for chunks in _chunkings(T, rng):
            net = StandIn()
            up = VideoUpscaler(net, (6, 8), (2, 2), batch=batch, in_format=in_fmt, out_format=out_fmt)
            outs = _stream(up, frames, chunks)
            assert [s for s, _ in outs] == [i for i, _ in sharding.batch_schedule(T, batch)]
            assert torch.equal(_cat(outs), want)
            assert up.ring.dtype == torch.uint16 and tuple(up.ring.shape) == (32, 6, 8, 3)
            assert {c[0] for c in net.calls} == {torch.uint16}
            assert {c[1] for c in net.calls} == {None if out_fmt == "bgr48le" else out_fmt}
            assert cpu_colour == ([] if in_fmt in colour.DEEP_FORMATS else [(6, 8, 3)] * T)       # one widening per 8-bit frame
            cpu_colour.clear()


def test_ring_dtype_of_every_pair(cpu_colour):
    for a in IN_FORMATS:
        for b in IN_FORMATS:
            if a in colour.DEEP_FORMATS and b not in colour.DEEP_FORMATS:
                with pytest.raises(ValueError, match=f"deep input {a} with 8-bit output {b}"):
                    VideoUpscaler(StandIn(), (6, 8), (2, 2), in_format=a, out_format=b)
                continue
            up = VideoUpscaler(StandIn(), (6, 8), (2, 2), in_format=a, out_format=b)
            assert up.ring.dtype == (torch.uint16 if b in colour.DEEP_FORMATS else torch.uint8), (a, b)


def test_numpy_and_pitched_p010_frames(cpu_colour):
    clip = _clip(9, "p010", seed=3)
    want = _composition(clip, "p010", "yuv420p10le", 4)
    surf = np.zeros((9, 9, 32), np.uint16)                  # decoder surfaces with a 64-byte pitch, as numpy views
    surf[:, :, :8] = _i64(clip).numpy()
    up = VideoUpscaler(StandIn(), (6, 8), (2, 2), batch=4, in_format="p010", out_format="yuv420p10le")
    outs = []
    for k in range(9):
        outs += up.push(surf[k, :, :8])
    outs += up.finish()
    assert torch.equal(_cat(outs), want)
    up = VideoUpscaler(StandIn(), (6, 8), (2, 2), batch=4, in_format="bgr48le", out_format="p010")
    b = np.asarray(_i64(_clip(5, "bgr48le")).numpy(), np.uint16)
    outs = up.push(b) + up.finish()
    assert torch.equal(_cat(outs), _composition(torch.from_numpy(b), "bgr48le", "p010", 4))


def test_refusals(cpu_colour):
    net = StandIn()
    for fmt in ("yuv420p10le", "p010"):
        with pytest.raises(ValueError, match="even LR size"):
            VideoUpscaler(net, (7, 8), (2, 2), in_format=fmt, out_format=fmt)
        with pytest.raises(ValueError, match=r"scale \(2\.7, 2\.7\) gives H = 389, W = 486.*bgr48le output takes any scale"):
            VideoUpscaler(net, (144, 180), (2.7, 2.7), in_format="bgr48le", out_format=fmt)
        VideoUpscaler(net, (144, 180), (2.7, 2.7), in_format=fmt, out_format="bgr48le")
        up = VideoUpscaler(net, (6, 8), (2, 2), in_format=fmt, out_format=fmt)
        with pytest.raises(TypeError, match="uint16"):
            up.push(torch.zeros(9, 8, dtype=torch.uint8))
        with pytest.raises(ValueError, match=r"\[9, 8\]"):
            up.push(torch.zeros(6, 8, 3, dtype=torch.uint16))
        with pytest.raises(ValueError, match="row stride 6"):
            up.push(torch.zeros(80, dtype=torch.uint16).as_strided((9, 8), (6, 1)))
        assert up.received == 0
    up = VideoUpscaler(net, (6, 8), (2, 2), in_format="yuv420p10le", out_format="p010")
    with pytest.raises(ValueError, match="contiguous rows"):
        up.push(torch.zeros(9, 16, dtype=torch.uint16)[:, :8])
    up = VideoUpscaler(net, (6, 8), (2, 2), in_format="bgr48le", out_format="bgr48le")
    with pytest.raises(TypeError, match="uint16"):
        up.push(torch.zeros(6, 8, 3, dtype=torch.uint8))
    up = VideoUpscaler(net, (6, 8), (2, 2), in_format="bgr24", out_format="bgr48le")
    with pytest.raises(TypeError, match="uint8"):
        up.push(torch.zeros(6, 8, 3, dtype=torch.uint16))
    for a in colour.DEEP_FORMATS:
        for b in ("bgr24", "yuv420p", "nv12"):
            with pytest.raises(ValueError, match=f"deep input {a} with 8-bit output {b}"):
                VideoUpscaler(net, (6, 8), (2, 2), in_format=a, out_format=b)


# ------------------------------------------------------------------------------------------------ GPU

DEV = torch.device("cuda", 0)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,pitch", [("yuv420p10le", None), ("p010", None), ("p010", 8448)])
def test_decode_every_10bit_triple(fmt, pitch):
    """All 2^30 (Y, U, V) in 16 frames of 8192 x 8192: chroma block b of chunk c carries (U, V) = divmod(c 2^16 + b // 256, 1024) and
    its four pixels Y = 4 (b % 256) + 0..3.  Against dec10 in device integer ops."""
    N = 8192
    b = torch.arange(N // 2 * N // 2, device=DEV)
    y4 = (4 * (b % 256)).reshape(N // 2, N // 2)
    Y = torch.stack([torch.stack([y4, y4 + 1], -1), torch.stack([y4 + 2, y4 + 3], -1)], 1).reshape(1, N, N)
    up = lambda c: c.repeat_interleave(2, 1).repeat_interleave(2, 2)  # noqa: E731
    for chunk in range(16):
        uv = chunk * 65536 + b // 256
        U, V = (uv // 1024).reshape(1, N // 2, N // 2), (uv % 1024).reshape(1, N // 2, N // 2)
        x = frames10(Y, U, V, fmt, pitch)
        got = _i64(colour.yuv420_to_bgr(x, fmt))
        want = dec10(Y, up(U), up(V))
        for k in range(3):
            assert torch.equal(got[..., k], want[k]), (chunk, k)
        del x, got, want


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,pitch", [("yuv420p10le", None), ("p010", None), ("p010", 1024)])
@pytest.mark.parametrize("h,w", [(2, 2), (144, 180), (180, 318), (1080, 1920)])
def test_encode_random_and_edge_values(fmt, pitch, h, w):
    if pitch is not None and pitch < w:
        pitch = w + 64
    n = 3
    g = torch.Generator().manual_seed(h + w)
    v = torch.randint(0, 65536, (n, h, w, 3), generator=g)
    ends = torch.tensor([0, 1, 255, 256, 32767, 32768, 65279, 65534, 65535])
    v.view(-1)[:min(v.numel(), 3 * 729)] = torch.stack(torch.meshgrid(ends, ends, ends, indexing="ij"), -1).reshape(-1)[:min(v.numel(), 3 * 729)]
    bgr = _u16(v).to(DEV)
    want = enc_frames10(bgr, fmt)
    if pitch is None:
        got = colour.bgr_to_yuv420(bgr, fmt)
        assert got.is_contiguous()
    else:
        surf = _u16(torch.full((n, 3 * h // 2, pitch), 7, device=DEV))
        got = colour.bgr_to_yuv420(bgr, fmt, out=surf[:, :, :w])
        assert int((_i64(surf[:, :, w:]) != 7).sum()) == 0                 # nothing written past the width
    assert torch.equal(_i64(got), _i64(want))
    # and back: decode of random frames, rows starting on addresses 2 mod 16
    x = _clip(n, fmt, h, w, seed=w).to(DEV)
    buf = _u16(torch.zeros(x[0].numel() * n + 1, device=DEV))
    xo = buf[1:].view(n, 3 * h // 2, w)
    xo.copy_(x)
    assert torch.equal(_i64(colour.yuv420_to_bgr(xo, fmt)), _i64(dec_frames10(x, fmt)))


def _gpu_net(precision="bf16", graph=True, seed=0):
    import savsr_b200
    net = savsr_b200.SAVSR().to(DEV).eval()
    net.load_state_dict(make_state_dict(seed), strict=True)
    net.precision, net.use_graph = precision, graph
    return net


UNIT16 = torch.from_numpy(np.arange(65536, dtype=np.float32) / np.float32(65535))      # correctly rounded v / 65535


def _contract(net, x16):
    """round(clamp(forward(x'), 0, 1) * 65535) in fp32, half to even, as int64."""
    xf = UNIT16.to(DEV)[_i64(x16)].flip(-1).permute(0, 1, 4, 2, 3).contiguous()
    return (net(xf).clamp(0, 1) * 65535).round().to(torch.int64).permute(0, 2, 3, 1).flip(-1)       # RGB planes -> BGR pixels


def _windows16(b, h, w, seed):
    return _u16(torch.randint(0, 65536, (b, 7, h, w, 3), generator=torch.Generator().manual_seed(seed))).to(DEV)


@pytest.mark.gpu
@pytest.mark.parametrize("b,h,w,scale,precision,graph", [
    (2, 144, 180, (4, 4), "bf16", True),         # Vid4 at x4
    (2, 144, 180, (1.5, 4), "fp16", True),
    (2, 144, 180, (2.7, 2.7), "bf16", False),
    (2, 144, 180, (2.7, 2.7), "fp16", False),
    (2, 179, 317, (4, 4), "bf16", False),        # odd size: pad_spatial
    (2, 179, 317, (4, 4), "fp16", True),
    (1, 144, 180, (4, 4), "bf16", False),
    (1, 144, 180, (1.5, 4), "fp16", True),
])
def test_forward_bgr48_contract(b, h, w, scale, precision, graph):
    net = _gpu_net(precision, graph)
    net.set_scale(scale)
    x = _windows16(b, h, w, seed=b * 1000 + h + int(10 * scale[0]))
    with torch.no_grad():
        got = net.forward_bgr48(x)
        want = _contract(net, x)
        again = net.forward_bgr48(x)
    assert got.dtype == torch.uint16 and tuple(got.shape) == (b, *engine.get_hw(h, w, scale), 3)
    assert torch.equal(_i64(got), want), int((_i64(got) - want).abs().max())
    assert torch.equal(_i64(again), want)
    assert tuple(net.forward_bgr48(x[:0]).shape) == (0, *engine.get_hw(h, w, scale), 3)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_forward_bgr48_of_widened_8bit_frames(precision):
    """On 257 x8 the forward sees what forward_bgr_u8 sees on x8: the contract on x8 / 255, and forward_bgr_u8's image of it."""
    net = _gpu_net(precision)
    net.set_scale((4, 4))
    x8 = torch.randint(0, 256, (2, 7, 144, 180, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(3)).to(DEV)
    with torch.no_grad():
        got = _i64(net.forward_bgr48(_u16(x8.to(torch.int32) * 257)))
        u8 = torch.from_numpy(np.arange(256, dtype=np.float32) / np.float32(255)).to(DEV)
        y = net(u8[x8.long()].flip(-1).permute(0, 1, 4, 2, 3).contiguous())
        assert torch.equal(got, (y.clamp(0, 1) * 65535).round().to(torch.int64).permute(0, 2, 3, 1).flip(-1))
        assert torch.equal(net.forward_bgr_u8(x8).to(torch.int64), (y.clamp(0, 1) * 255).round().to(torch.int64).permute(0, 2, 3, 1).flip(-1))


@pytest.mark.gpu
def test_forward_bgr48_indexed_and_the_c_call():
    import ctypes as C
    net = _gpu_net()
    net.set_scale((1.5, 4))
    pool = _u16(torch.randint(0, 65536, (9, 37, 45, 3), generator=torch.Generator().manual_seed(5))).to(DEV)
    idx = torch.tensor([[0, 1, 2, 3, 4, 5, 6], [8, 8, 7, 3, 2, 0, 1]])
    gathered = pool.view(torch.int16)[idx.to(DEV)].view(torch.uint16)
    with torch.no_grad():
        want = _i64(net.forward_bgr48(gathered))
        assert torch.equal(_i64(net.forward_bgr48_indexed(pool, idx)), want)
        assert torch.equal(_i64(net.forward_bgr48_indexed(pool, idx.tolist())), want)
        pd = net._plan(2, 37, 45, DEV, "bgr48_frames", net.scale)
        pf = net._plan(2, 37, 45, DEV, "bgr_u8_frames", net.scale)
        assert pd.cplan is not None and pd.store is pf.store
        ptrs = (idx.reshape(-1) * (37 * 45 * 3 * 2) + pool.data_ptr()).tolist()
        out = _u16(torch.zeros(2, *pd.out.shape[1:], device=DEV))
        pd.forward_frames_c(ptrs, out)                     # savsr_forward_u16_frames
        torch.cuda.synchronize()
        assert torch.equal(_i64(out), want)
        lib, st = pd.lib, torch.cuda.current_stream().cuda_stream
        arr = (C.c_void_p * len(ptrs))(*ptrs)
        out.view(torch.int16).zero_()
        assert lib.savsr_forward_u8_frames(pd.cplan.handle, arr, out.data_ptr(), st) != 0
        assert b"savsr_forward_u16_frames" in lib.savsr_last_error()
        assert lib.savsr_forward_u16_frames(pf.cplan.handle, arr, out.data_ptr(), st) != 0
        assert b"savsr_forward_u8_frames" in lib.savsr_last_error()
        assert lib.savsr_forward(pd.cplan.handle, out.data_ptr(), out.data_ptr(), st) != 0
        bad = (C.c_void_p * len(ptrs))(*ptrs[:-1], None)
        assert lib.savsr_forward_u16_frames(pd.cplan.handle, bad, out.data_ptr(), st) != 0
        assert b"null" in lib.savsr_last_error()
        torch.cuda.synchronize()
        assert int(out.view(torch.int16).count_nonzero()) == 0        # the refused calls copied and launched nothing
        for b in (64, 65):                                  # one and two table-writer launches
            many = torch.arange(b * 7).reshape(b, 7) % 9
            assert torch.equal(_i64(net.forward_bgr48_indexed(pool, many)),
                               _i64(net.forward_bgr48(pool.view(torch.int16)[many.to(DEV)].view(torch.uint16))))


def _feed(clip, fmt, how):
    """The clip's frames one by one as the caller hands them: pageable host, pinned host, or device (p010 with a 512-byte pitch, as a
    decoder surface; the other formats contiguous)."""
    if how == "pageable":
        return list(clip)
    if how == "pinned":
        return list(clip.pin_memory())
    if fmt == "p010":
        T, rows, w = clip.shape
        surf = torch.zeros(T, rows, 256, dtype=torch.int16, device=DEV)
        surf[:, :, :w] = clip.view(torch.int16).to(DEV)
        return list(surf.view(torch.uint16)[:, :, :w])
    return list(clip.to(DEV))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_video_upscaler_deep_and_mixed_pairs(precision):
    import savsr_b200
    net = _gpu_net(precision)
    h, w, T, batch, scale = 144, 180, 34, (26, 8), (4, 4)
    g = torch.Generator().manual_seed(6)
    Y8 = torch.randint(16, 236, (T, h, w), dtype=torch.uint8, generator=g)
    U8, V8 = (torch.randint(16, 241, (T, h // 2, w // 2), dtype=torch.uint8, generator=g) for _ in range(2))
    Y10 = torch.randint(64, 941, (T, h, w), generator=g)
    U10, V10 = (torch.randint(64, 961, (T, h // 2, w // 2), generator=g) for _ in range(2))
    clips = {"bgr24": torch.randint(0, 256, (T, h, w, 3), dtype=torch.uint8, generator=g),
             "yuv420p": torch.cat([Y8.reshape(T, -1), U8.reshape(T, -1), V8.reshape(T, -1)], 1).reshape(T, 3 * h // 2, w),
             "nv12": torch.cat([Y8, torch.stack([U8, V8], -1).reshape(T, h // 2, w)], 1),
             "bgr48le": _u16(torch.randint(0, 65536, (T, h, w, 3), generator=g)),
             "yuv420p10le": frames10(Y10, U10, V10, "yuv420p10le"), "p010": frames10(Y10, U10, V10, "p010")}
    with torch.no_grad():
        net.set_scale(scale)
        hr = {}
        for src in ("bgr24", "yuv420p", "bgr48le", "yuv420p10le"):         # nv12 and p010 hold the planes of yuv420p and yuv420p10le
            d = dec_any(clips[src], src).to(DEV)
            hr[src] = sharding.infer_clip(lambda x: net.forward_bgr48(x.view(torch.uint16)).view(torch.int16), d.view(torch.int16),
                                          batch=batch).view(torch.uint16)
        hr["nv12"], hr["p010"] = hr["yuv420p"], hr["yuv420p10le"]
        for in_fmt, out_fmt in PAIRS:
            want = _i64(enc_any(hr[in_fmt], out_fmt)).cpu()
            up = savsr_b200.VideoUpscaler(net, (h, w), scale, batch=batch, in_format=in_fmt, out_format=out_fmt)
            for how in ("pageable", "pinned", "device"):
                up.reset()
                outs = []
                for f in _feed(clips[in_fmt], in_fmt, how):
                    outs += up.push(f)
                outs += up.finish()
                assert all(y.is_cuda and y.dtype == torch.uint16 for _, y in outs)
                assert [s for s, _ in outs] == [i for i, _ in sharding.batch_schedule(T, batch)]
                assert torch.equal(_cat(outs).cpu(), want), (in_fmt, out_fmt, how)


@pytest.mark.gpu
def test_refused_pairs_and_sizes():
    import savsr_b200
    net = _gpu_net()
    for a in colour.DEEP_FORMATS:
        for b in ("bgr24", "yuv420p", "nv12"):
            with pytest.raises(ValueError, match=f"deep input {a} with 8-bit output {b}"):
                savsr_b200.VideoUpscaler(net, (144, 180), (4, 4), in_format=a, out_format=b)
    for fmt in ("yuv420p10le", "p010"):
        with pytest.raises(ValueError, match=r"gives H = 389, W = 486"):
            savsr_b200.VideoUpscaler(net, (144, 180), (2.7, 2.7), in_format="bgr48le", out_format=fmt)
    ctx = engine.context(0)
    lib, st = ctx.lib, torch.cuda.current_stream().cuda_stream
    h, w, n = 36, 44, 2
    x = _clip(n, "p010", h, w, seed=1).to(DEV)
    out = _u16(torch.zeros(n, h, w, 3, device=DEV))
    p = x.data_ptr()
    args = [p, w, p + 2 * h * w, p + 2 * h * w + 2, w, 2, x.stride(0), 1, n, h, w, out.data_ptr(), st]
    assert lib.savsr_yuv420_10_to_bgr48(ctx.handle, *args) == 0
    torch.cuda.synchronize()
    assert torch.equal(_i64(out), _i64(dec_frames10(x, "p010")))
    out.view(torch.int16).zero_()
    for i, v, msg in [(9, h - 1, b"even"), (0, None, b"null"), (11, None, b"null"), (1, w - 2, b"y_pitch"), (4, w - 2, b"c_pitch"),
                      (5, 3, b"c_step"), (6, -1, b"frame_stride"), (7, 2, b"msb")]:
        bad = list(args)
        bad[i] = v
        assert lib.savsr_yuv420_10_to_bgr48(ctx.handle, *bad) != 0, (i, v)
        assert msg in lib.savsr_last_error(), (i, v, lib.savsr_last_error())
    eargs = [out.data_ptr(), n, h, w, p, w, p + 2 * h * w, p + 2 * h * w + 2, w, 2, x.stride(0), 1, st]
    for i, v, msg in [(2, h + 1, b"even"), (0, None, b"null"), (5, w - 1, b"y_pitch"), (11, -1, b"msb")]:
        bad = list(eargs)
        bad[i] = v
        assert lib.savsr_bgr48_to_yuv420_10(ctx.handle, *bad) != 0, (i, v)
        assert msg in lib.savsr_last_error(), (i, v, lib.savsr_last_error())
    assert lib.savsr_widen_u8_to_u16(ctx.handle, None, 1, h, w, out.data_ptr(), st) != 0
    assert lib.savsr_widen_u8_to_u16(ctx.handle, out.data_ptr(), 1, 0, w, out.data_ptr(), st) != 0
    torch.cuda.synchronize()
    assert int(out.view(torch.int16).count_nonzero()) == 0
    # widen: aligned and unaligned buffers
    for off in (0, 1):
        src = torch.randint(0, 256, (3 * h * w * 3 + off,), dtype=torch.uint8, device=DEV)[off:].view(3, h, w, 3)
        dst = _u16(torch.zeros(3, h, w, 3, device=DEV))
        colour.widen(src, dst)
        assert torch.equal(_i64(dst), src.to(torch.int64) * 257)
