"""Colour matrix and range of the YUV conversions: BT.601, BT.709 and BT.2020 (non-constant luminance), tv and pc range, at both depths
(savsr_b200.colour's colorspace / color_range, the _cs entry points of libsavsr_sm100, and VideoUpscaler's in_ / out_ pairs).

The H.273 maps are restated here in integer numpy / torch (dec, enc: common.cuh's fixed-point forms, constants restated and re-derived
from exact fractions) and checked against the real-valued maps; the kernels must equal the restatement exactly.  The default pair
("bt601", "tv") stays the cv2-exact conversion of tests/test_video_yuv.py and tests/test_video_deep.py.

CPU: the constants, the error bounds, grey neutrality, name resolution, C-call arguments against the recording fake library, and
VideoUpscaler's host logic with the conversions replaced by the restatement.  GPU: all exact with torch.equal.
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
from test_video_deep import frames10, planes10, _i64, _u16

KRKB = {"bt601": (Fraction(299, 1000), Fraction(114, 1000)), "bt709": (Fraction(2126, 10000), Fraction(722, 10000)),
        "bt2020nc": (Fraction(2627, 10000), Fraction(593, 10000))}
SHIFT = {8: (20, 20), 10: (22, 21)}          # (decode, encode)
FULL = {8: 255, 10: 65535}                   # BGR full scale of each YUV depth
# common.cuh kYuvCoeffs8 / kYuvCoeffs10: (y0, dy, dvr, dvg, dug, dub, eyr, eyg, eyb, eur, eug, eub, evr, evg, evb)
COEFFS = {
    8: {("bt601", "tv"): (16, 1220945, 1673555, -852458, -410793, 2115221, 269262, 528618, 102662, -155423, -305128, 460551, 460551, -385654, -74897),
        ("bt601", "pc"): (0, 1048576, 1470104, -748826, -360853, 1858077, 313524, 615514, 119538, -176932, -347356, 524288, 524288, -439026, -85262),
        ("bt709", "tv"): (16, 1220945, 1879825, -558796, -223607, 2215014, 191455, 644067, 65019, -105533, -355018, 460551, 460551, -418321, -42230),
        ("bt709", "pc"): (0, 1048576, 1651297, -490864, -196424, 1945738, 222927, 749942, 75707, -120138, -404150, 524288, 524288, -476214, -48074),
        ("bt2020nc", "tv"): (16, 1220945, 1760217, -682019, -196426, 2245811, 236572, 610567, 53402, -128614, -331937, 460551, 460551, -423510,
                             -37041),
        ("bt2020nc", "pc"): (0, 1048576, 1546230, -599107, -172546, 1972791, 275461, 710935, 62181, -146413, -377875, 524288, 524288, -482120,
                             -42168)},
    10: {("bt601", "tv"): (64, 313782777, 430103733, -219081799, -105573682, 543611851, 8382, 16455, 3196, -4838, -9498, 14336, 14336, -12005, -2331),
         ("bt601", "pc"): (0, 268693756, 376708646, -191883961, -92467271, 476125336, 9788, 19216, 3732, -5524, -10844, 16368, 16368, -13706, -2662),
         ("bt709", "tv"): (64, 313782777, 483115092, -143610555, -57467096, 569258550, 5960, 20049, 2024, -3285, -11051, 14336, 14336, -13022, -1315),
         ("bt709", "pc"): (0, 268693756, 423138927, -125782069, -50332863, 498588134, 6960, 23413, 2364, -3751, -12618, 16368, 16368, -14867, -1501),
         ("bt2020nc", "tv"): (64, 313782777, 452375867, -175278968, -50481394, 577173441, 7364, 19006, 1662, -4004, -10333, 14336, 14336, -13183,
                              -1153),
         ("bt2020nc", "pc"): (0, 268693756, 396215813, -153519018, -44214398, 505520433, 8600, 22195, 1941, -4571, -11797, 16368, 16368, -15052,
                              -1316)}}
NEW_PAIRS = [("bt601", "pc"), ("bt709", "tv"), ("bt709", "pc"), ("bt2020nc", "tv"), ("bt2020nc", "pc")]


def exact(cs, rng, n):
    """The real-valued maps' coefficients as Fractions: (y0, decode [dy, dvr, dvg, dug, dub], encode [eyr .. evb]) (common.cuh)."""
    kr, kb = KRKB[cs]
    kg, M, s = 1 - kr - kb, FULL[n], 1 << (n - 8)
    y0, ys, c = (16 * s, 219 * s, 224 * s) if rng == "tv" else (0, (1 << n) - 1, (1 << n) - 1)
    dec = [Fraction(M, ys), M * 2 * (1 - kr) / c, -M * 2 * kr * (1 - kr) / (kg * c), -M * 2 * kb * (1 - kb) / (kg * c), M * 2 * (1 - kb) / c]
    enc = [ys * kr / M, ys * kg / M, ys * kb / M, -c * kr / (2 * (1 - kb) * M), -c * kg / (2 * (1 - kb) * M), Fraction(c, 2 * M),
           Fraction(c, 2 * M), -c * kg / (2 * (1 - kr) * M), -c * kb / (2 * (1 - kr) * M)]
    return y0, dec, enc


def _round_away(q: Fraction) -> int:
    r = int(abs(q) + Fraction(1, 2))
    return r if q >= 0 else -r


def dec(Y, U, V, cs, rng, n):
    """(Y, U, V) -> (B, G, R): the kernels' integer form.  int64 numpy arrays or torch tensors."""
    y0, dy, dvr, dvg, dug, dub = COEFFS[n][(cs, rng)][:6]
    S, c, M = SHIFT[n][0], 1 << (n - 1), FULL[n]
    y, u, v, half = (Y - y0) * dy, U - c, V - c, 1 << (S - 1)
    return [((y + half + t) >> S).clip(0, M) for t in (dub * u, dvg * v + dug * u, dvr * v)]


def enc(R, G, B, cs, rng, n):
    """(R, G, B) -> (Y, U, V): the kernels' integer form."""
    k = COEFFS[n][(cs, rng)]
    S, half, top = SHIFT[n][1], 1 << (SHIFT[n][1] - 1), (1 << n) - 1
    off = (k[0], 1 << (n - 1), 1 << (n - 1))
    return [(o + ((a * R + b * G + d * B + half) >> S)).clip(0, top) for o, (a, b, d) in zip(off, (k[6:9], k[9:12], k[12:15]))]


def dec_real(Y, U, V, cs, rng, n):
    y0, d, _ = exact(cs, rng, n)
    dy, dvr, dvg, dug, dub = (float(x) for x in d)
    c, M = 1 << (n - 1), FULL[n]
    y, u, v = (Y - y0).astype(np.float64) * dy, (U - c).astype(np.float64), (V - c).astype(np.float64)
    return [np.clip(y + t, 0, M) for t in (dub * u, dvg * v + dug * u, dvr * v)]


def enc_real(R, G, B, cs, rng, n):
    y0, _, e = exact(cs, rng, n)
    e = [float(x) for x in e]
    R, G, B = (x.astype(np.float64) for x in (R, G, B))
    off = (y0, 1 << (n - 1), 1 << (n - 1))
    return [np.clip(o + e[3 * i] * R + e[3 * i + 1] * G + e[3 * i + 2] * B, 0, (1 << n) - 1) for i, o in enumerate(off)]


# ------------------------------------------------------------------------------------------------ frames (torch, any device)

def frames8(Y, U, V, fmt, pitch=None):
    """[n, 3h/2, w] uint8 frames of yuv420p or nv12 (with row `pitch` when given) from planes Y [n,h,w], U, V [n,h/2,w/2]."""
    n, h, w = Y.shape
    if fmt == "yuv420p":
        x = torch.cat([Y.reshape(n, -1), U.reshape(n, -1), V.reshape(n, -1)], 1).reshape(n, 3 * h // 2, w)
    else:
        x = torch.cat([Y, torch.stack([U, V], -1).reshape(n, h // 2, w)], 1)
    x = x.to(torch.uint8)
    if pitch is None or pitch == w:
        return x
    buf = torch.zeros(n, 3 * h // 2, pitch, dtype=torch.uint8, device=x.device)
    buf[:, :, :w] = x
    return buf[:, :, :w]


def planes8(x, fmt):
    x = x.to(torch.int64)
    n, rows, w = x.shape
    h = 2 * rows // 3
    if fmt == "yuv420p":
        flat = x.reshape(n, -1)
        q = h * w // 4
        return flat[:, :h * w].reshape(n, h, w), flat[:, h * w:h * w + q].reshape(n, h // 2, w // 2), flat[:, h * w + q:].reshape(n, h // 2, w // 2)
    uv = x[:, h:].reshape(n, h // 2, w // 2, 2)
    return x[:, :h], uv[..., 0], uv[..., 1]


def _up(c):
    return c.repeat_interleave(2, 1).repeat_interleave(2, 2)


def dec_frames(x, fmt, cs, rng):
    """The restatement of colour.yuv420_to_bgr for a pair of NEW_PAIRS: frames [n, 3h/2, w] -> BGR [n, h, w, 3] of the same depth."""
    deep = fmt in colour.DEEP_FORMATS
    Y, U, V = planes10(x, fmt) if deep else planes8(x, fmt)
    bgr = torch.stack(dec(Y, _up(U), _up(V), cs, rng, 10 if deep else 8), -1)
    return _u16(bgr) if deep else bgr.to(torch.uint8)


def enc_frames(bgr, fmt, cs, rng):
    deep = fmt in colour.DEEP_FORMATS
    b = _i64(bgr) if deep else bgr.to(torch.int64)
    B, G, R = b[..., 0], b[..., 1], b[..., 2]
    n = 10 if deep else 8
    Y = enc(R, G, B, cs, rng, n)[0]
    tl = lambda c: c[:, ::2, ::2]  # noqa: E731
    _, U, V = enc(tl(R), tl(G), tl(B), cs, rng, n)
    return frames10(Y, U, V, fmt) if deep else frames8(Y, U, V, fmt)


# ------------------------------------------------------------------------------------------------ CPU: the maps

def test_constants_follow_the_rule():
    for n in (8, 10):
        assert set(COEFFS[n]) == {(cs, r) for cs in KRKB for r in ("tv", "pc")}
        for (cs, rng), k in COEFFS[n].items():
            y0, d, e = exact(cs, rng, n)
            sd, se = SHIFT[n]
            assert k == (y0, *[_round_away(q * 2 ** sd) for q in d], *[_round_away(q * 2 ** se) for q in e]), (n, cs, rng)
            assert all(abs(v) < 2 ** 31 for v in k)
            if n == 8:                            # the 8-bit forms are int32 both ways: every sum before the shift
                y0, dy, dvr, dvg, dug, dub = k[:6]
                assert abs(dy) * 255 + max(abs(dvr), abs(dvg) + abs(dug), abs(dub)) * 128 + (1 << 19) < 2 ** 31
                assert all(sum(abs(x) for x in k[i:i + 3]) * 255 + (1 << 19) < 2 ** 31 for i in (6, 9, 12))


def test_every_8bit_yuv_triple_decodes_within_0_55():
    Y = np.arange(256, dtype=np.int64).reshape(-1, 1, 1)
    U = np.arange(256, dtype=np.int64).reshape(1, -1, 1)
    V = np.arange(256, dtype=np.int64).reshape(1, 1, -1)
    for cs, rng in NEW_PAIRS:
        for lo in range(0, 256, 64):
            y = Y[lo:lo + 64]
            for g, r in zip(dec(y, U, V, cs, rng, 8), dec_real(y, U, V, cs, rng, 8)):
                assert g.min() >= 0 and g.max() <= 255
                assert float(np.abs(g - r).max()) <= 0.55, (cs, rng)


def test_every_8bit_bgr_triple_encodes_within_0_55():
    R = np.arange(256, dtype=np.int64).reshape(-1, 1, 1)
    G = np.arange(256, dtype=np.int64).reshape(1, -1, 1)
    B = np.arange(256, dtype=np.int64).reshape(1, 1, -1)
    for cs, rng in NEW_PAIRS:
        for lo in range(0, 256, 64):
            r = R[lo:lo + 64]
            got, real = enc(r, G, B, cs, rng, 8), enc_real(r, G, B, cs, rng, 8)
            for ch in range(3):
                assert float(np.abs(got[ch] - real[ch]).max()) <= 0.55, (cs, rng, ch)
            if rng == "tv":
                assert got[0].min() >= 16 and got[0].max() <= 235 and min(got[1].min(), got[2].min()) >= 16 and max(got[1].max(), got[2].max()) <= 240
    # pc chroma reaches past the top code value before saturation: 128 + 127.5 for pure blue
    assert [int(c) for c in enc(np.int64(0), np.int64(0), np.int64(255), "bt709", "pc", 8)][1] == 255


def test_10bit_decode_within_0_55():
    rng_ = np.random.default_rng(1)
    U = np.repeat(np.arange(1024, dtype=np.int64), 1024)
    V = np.tile(np.arange(1024, dtype=np.int64), 1024)
    for cs, rng in NEW_PAIRS:
        y0 = COEFFS[10][(cs, rng)][0]
        for y in (0, y0, 940 if rng == "tv" else 1023, 1023, int(rng_.integers(0, 1024))):
            Y = np.full_like(U, y)
            for g, r in zip(dec(Y, U, V, cs, rng, 10), dec_real(Y, U, V, cs, rng, 10)):
                assert float(np.abs(g - r).max()) <= 0.55, (cs, rng, y)


def test_16bit_encode_within_0_55():
    rng_ = np.random.default_rng(2)
    corners = np.array([[r, g, b] for r in (0, 65535) for g in (0, 65535) for b in (0, 65535)])
    ramp = np.repeat(np.arange(0, 65536, 7), 3).reshape(-1, 3)
    px = np.concatenate([rng_.integers(0, 65536, (1 << 22, 3)), corners, ramp]).astype(np.int64)
    R, G, B = px[:, 0], px[:, 1], px[:, 2]
    for cs, rng in NEW_PAIRS:
        got, real = enc(R, G, B, cs, rng, 10), enc_real(R, G, B, cs, rng, 10)
        for ch in range(3):
            assert float(np.abs(got[ch] - real[ch]).max()) <= 0.55, (cs, rng, ch)
        k = COEFFS[10][(cs, rng)]                 # int32: every sum before the shift, offsets excluded
        for a, b, d in (k[6:9], k[9:12], k[12:15]):
            assert (max(a, 0) + max(b, 0) + max(d, 0)) * 65535 + (1 << 20) < 2 ** 31
            assert (min(a, 0) + min(b, 0) + min(d, 0)) * 65535 >= -2 ** 31


def test_grey_encodes_to_neutral_chroma():
    for n in (8, 10):
        g = np.arange(FULL[n] + 1, dtype=np.int64)
        for cs, rng in COEFFS[n]:
            _, U, V = enc(g, g, g, cs, rng, n)
            assert (U == 1 << (n - 1)).all() and (V == 1 << (n - 1)).all(), (n, cs, rng)


def test_names_and_aliases():
    for name, want in [("bt601", "bt601"), ("bt470bg", "bt601"), ("smpte170m", "bt601"), ("bt709", "bt709"), ("bt2020nc", "bt2020nc"),
                       ("bt2020", "bt2020nc")]:
        assert colour.check_colorspace(name) == want
    for name, want in [("tv", "tv"), ("limited", "tv"), ("mpeg", "tv"), ("pc", "pc"), ("full", "pc"), ("jpeg", "pc")]:
        assert colour.check_color_range(name) == want
    assert colour.COLORSPACES == {"bt601": 0, "bt709": 1, "bt2020nc": 2} and colour.COLOR_RANGES == {"tv": 0, "pc": 1}
    with pytest.raises(ValueError, match=r"unknown colorspace 'bt2020c': expected one of bt601, bt709, bt2020nc, bt470bg"):
        colour.check_colorspace("bt2020c")
    with pytest.raises(ValueError, match=r"unknown out_color_range 'studio': expected one of tv, pc, limited, mpeg, full, jpeg"):
        colour.check_color_range("studio", "out_color_range")


# ------------------------------------------------------------------------------------------------ CPU: C-call arguments

class _ClaimsCuda(torch.Tensor):
    """A CPU tensor that reports is_cuda, so the host logic runs without a device (nothing is launched)."""
    is_cuda = property(lambda self: True)


def test_c_call_arguments():
    n, h, w = 3, 6, 8
    c = lambda t: t.as_subclass(_ClaimsCuda)  # noqa: E731
    with mocked_engine() as lib:
        x8, b8 = c(torch.zeros(n, 9, w, dtype=torch.uint8)), c(torch.zeros(n, h, w, 3, dtype=torch.uint8))
        x16, b16 = c(torch.zeros(n, 9, w, dtype=torch.uint16)), c(torch.zeros(n, h, w, 3, dtype=torch.uint16))
        calls = [lambda **kw: colour.yuv420_to_bgr(x8, "nv12", out=b8, **kw), lambda **kw: colour.bgr_to_yuv420(b8, "yuv420p", out=x8, **kw),
                 lambda **kw: colour.yuv420_to_bgr(x16, "p010", out=b16, **kw),
                 lambda **kw: colour.bgr_to_yuv420(b16, "yuv420p10le", out=x16, **kw)]
        names = ["savsr_yuv420_to_bgr", "savsr_bgr_to_yuv420", "savsr_yuv420_10_to_bgr48", "savsr_bgr48_to_yuv420_10"]
        for call, name in zip(calls, names):
            lib.calls.clear()
            call()
            (n0, plain), = lib.calls
            for kw in ({"colorspace": "bt601", "color_range": "tv"}, {"colorspace": "smpte170m", "color_range": "limited"}):
                lib.calls.clear()
                call(**kw)
                assert lib.calls == [(name, plain)]               # the default pair: today's entry point, today's arguments
            for cs, rng, want in [("bt709", "tv", (1, 0)), ("bt2020", "pc", (2, 1)), ("bt601", "jpeg", (0, 1)), ("bt709", "full", (1, 1))]:
                lib.calls.clear()
                call(colorspace=cs, color_range=rng)
                (got, a), = lib.calls
                assert got == name + "_cs" and a == (*plain[:-1], *want, plain[-1]), (name, cs, rng)
            lib.calls.clear()
            with pytest.raises(ValueError, match="unknown colorspace"):
                call(colorspace="bt2020c")
            with pytest.raises(ValueError, match="unknown color_range"):
                call(color_range="studio")
            assert lib.calls == []


class CpuPlanFrames(CpuPlan):
    io = "bgr_u8_frames"


def test_plan_output_colour(monkeypatch):
    with mocked_engine() as lib:
        plan = CpuPlanFrames(make_state_dict(0), 2, 8, 10, (2, 2), store=engine.WeightStore())
        plan.out = plan.out.as_subclass(_ClaimsCuda)
        out = torch.empty(2, 3 * plan.H // 2, plan.W, dtype=torch.uint8).as_subclass(_ClaimsCuda)
        lib.calls.clear()
        plan.forward_frames_into([0x1000] * 14, out, graph=False, out_format="nv12", out_colorspace="bt709", out_color_range="tv")
        assert lib.calls[-1][0] == "savsr_bgr_to_yuv420_cs" and lib.calls[-1][1][-3:] == (1, 0, 0)
        assert sum(c[0].startswith("savsr_satu_hr") for c in lib.calls) == 1          # one HR pass, converted in place of the copy
        lib.calls.clear()
        plan.forward_frames_into([0x1000] * 14, out, graph=False, out_format="nv12")
        assert lib.calls[-1][0] == "savsr_bgr_to_yuv420"
        lib.calls.clear()
        with pytest.raises(ValueError, match="need a YUV out_format"):
            plan.forward_frames_into([0x1000] * 14, torch.empty_like(plan.out), graph=False, out_colorspace="bt709")
        with pytest.raises(ValueError, match="unknown out_colorspace"):
            plan.forward_frames_into([0x1000] * 14, out, graph=False, out_format="nv12", out_colorspace="xyz")
        assert lib.calls == []


# ------------------------------------------------------------------------------------------------ CPU: VideoUpscaler

def _cpu_dec(frames, fmt, out=None, colorspace="bt601", color_range="tv"):
    x = colour.yuv_frames(torch.as_tensor(frames), fmt)
    pair = (colour.check_colorspace(colorspace), colour.check_color_range(color_range))
    if pair == ("bt601", "tv"):
        assert fmt in ("yuv420p", "nv12")
        y = torch.stack([torch.from_numpy(cv2.cvtColor(np.ascontiguousarray(f.numpy()), cv2.COLOR_YUV2BGR_I420 if fmt == "yuv420p" else
                                                       cv2.COLOR_YUV2BGR_NV12)) for f in x])
    else:
        y = dec_frames(x, fmt, *pair)
    y = y if torch.as_tensor(frames).dim() == 3 else y[0]
    return y if out is None else out.copy_(y)


def _cpu_enc(bgr, fmt, out=None, colorspace="bt601", color_range="tv"):
    x = torch.as_tensor(bgr)
    x = x if x.dim() == 4 else x[None]
    pair = (colour.check_colorspace(colorspace), colour.check_color_range(color_range))
    if pair == ("bt601", "tv"):
        assert fmt in ("yuv420p", "nv12")
        i420 = torch.stack([torch.from_numpy(cv2.cvtColor(f.numpy(), cv2.COLOR_BGR2YUV_I420)) for f in x])
        y = i420 if fmt == "yuv420p" else frames8(*planes8(i420, "yuv420p"), "nv12")
    else:
        y = enc_frames(x, fmt, *pair)
    y = y if torch.as_tensor(bgr).dim() == 4 else y[0]
    return y if out is None else out.copy_(y)


@pytest.fixture
def cpu_colour(monkeypatch):
    seen = []

    def dec_(*a, **kw):
        seen.append(("dec", kw.get("colorspace"), kw.get("color_range")))
        return _cpu_dec(*a, **kw)

    def enc_(*a, **kw):
        seen.append(("enc", kw.get("colorspace"), kw.get("color_range")))
        return _cpu_enc(*a, **kw)
    monkeypatch.setattr(colour, "yuv420_to_bgr", dec_)
    monkeypatch.setattr(colour, "bgr_to_yuv420", enc_)
    monkeypatch.setattr(colour, "widen", lambda bgr, out: out.copy_(_u16(bgr.to(torch.int32) * 257)))
    return seen


def _net(x, full):
    """Stand-in forward on int64 BGR windows [n,7,h,w,3] -> [n,2h,2w,3], a function of every frame of the window."""
    return (_up(x[:, 3]) + _up(x.sum(1)) * 7) % (full + 1)


class StandIn:
    """CPU stand-in for a SAVSR in eval mode, with the output conversion of SAVSR._forward_bgr_u8_indexed."""
    training = False

    def __init__(self):
        self.gamma = torch.zeros(1)
        self.calls = []

    def _forward_bgr_u8_indexed(self, pool, windows, scale, out_format=None, out_colorspace="bt601", out_color_range="tv"):
        self.calls.append((out_format, out_colorspace, out_color_range))
        deep = pool.dtype == torch.uint16
        x = (_i64 if deep else lambda t: t.to(torch.int64))(pool[torch.as_tensor(windows)])
        hr = _net(x, 65535 if deep else 255)
        hr = _u16(hr) if deep else hr.to(torch.uint8)
        return hr if out_format is None else colour.bgr_to_yuv420(hr, out_format, colorspace=out_colorspace, color_range=out_color_range)


def _clip(T, fmt, h=6, w=8, seed=0):
    g = torch.Generator().manual_seed(seed)
    if fmt == "bgr24":
        return torch.randint(0, 256, (T, h, w, 3), dtype=torch.uint8, generator=g)
    top = 1024 if fmt in colour.DEEP_FORMATS else 256
    Y = torch.randint(0, top, (T, h, w), generator=g)
    U, V = (torch.randint(0, top, (T, h // 2, w // 2), generator=g) for _ in range(2))
    return frames10(Y, U, V, fmt) if fmt in colour.DEEP_FORMATS else frames8(Y, U, V, fmt)


# (in_format, in pair, out_format, out pair)
STREAMS = [("nv12", ("bt601", "tv"), "nv12", ("bt709", "tv")),
           ("yuv420p", ("bt709", "pc"), "yuv420p", ("bt709", "tv")),
           ("p010", ("bt2020nc", "tv"), "p010", ("bt2020nc", "tv")),
           ("nv12", ("bt601", "tv"), "p010", ("bt709", "tv")),
           ("bgr24", ("bt601", "tv"), "nv12", ("bt709", "tv"))]


def _kw(in_pair, out_pair):
    return dict(in_colorspace=in_pair[0], in_color_range=in_pair[1], out_colorspace=out_pair[0], out_color_range=out_pair[1])


def _composition(clip, in_fmt, in_pair, out_fmt, out_pair, batch, forward):
    """enc_out(infer_clip(forward, dec_in(frames), batch)), an 8-bit source of a deep output widened by 257."""
    bgr = clip if in_fmt == "bgr24" else _cpu_dec(clip, in_fmt, colorspace=in_pair[0], color_range=in_pair[1])
    if out_fmt in colour.DEEP_FORMATS and in_fmt not in colour.DEEP_FORMATS:
        bgr = _u16(bgr.to(torch.int32) * 257)
    hr = sharding.infer_clip(forward, bgr.view(torch.int16) if bgr.dtype == torch.uint16 else bgr, batch=batch)
    hr = hr.view(torch.uint16) if hr.dtype == torch.int16 else hr
    return _cpu_enc(hr, out_fmt, colorspace=out_pair[0], color_range=out_pair[1])


def _as_int(y):
    return _i64(y) if y.dtype == torch.uint16 else y.to(torch.int64)


@pytest.mark.parametrize("in_fmt,in_pair,out_fmt,out_pair", STREAMS)
@pytest.mark.parametrize("T", [4, 5, 13, 34, 35])
def test_stream_equals_the_composition(cpu_colour, T, in_fmt, in_pair, out_fmt, out_pair):
    batch = (26, 8)
    clip = _clip(T, in_fmt, seed=T)
    deep = out_fmt in colour.DEEP_FORMATS

    def forward(x):
        v = _i64(x.view(torch.uint16)) if x.dtype == torch.int16 else x.to(torch.int64)
        y = _net(v, 65535 if deep else 255)
        return _u16(y).view(torch.int16) if deep else y.to(torch.uint8)
    want = _as_int(_composition(clip, in_fmt, in_pair, out_fmt, out_pair, batch, forward))
    rng = random.Random(T)
    for chunks in ([1] * T, [min(rng.choice([1, 2, 3, 5, 9, 17, 40]), T) for _ in range(T)]):
        net = StandIn()
        up = VideoUpscaler(net, (6, 8), (2, 2), batch=batch, in_format=in_fmt, out_format=out_fmt, **_kw(in_pair, out_pair))
        for rep in range(2):                                  # reset() keeps the colour settings
            up.reset()
            cpu_colour.clear()
            outs, k = [], 0
            for c in chunks:
                outs += up.push(clip[k:k + c])
                k += c
                if k >= T:
                    break
            outs += up.finish()
            assert [s for s, _ in outs] == [i for i, _ in sharding.batch_schedule(T, batch)]
            assert torch.equal(torch.cat([_as_int(y) for _, y in outs]), want), (chunks, rep)
            decs = {e[1:] for e in cpu_colour if e[0] == "dec"}
            assert decs == (set() if in_fmt == "bgr24" else {(None, None) if in_pair == ("bt601", "tv") else in_pair})
            assert {e[1:] for e in cpu_colour if e[0] == "enc"} == {out_pair}
        assert {c[1:] for c in net.calls} == {out_pair}


def test_refusals(cpu_colour):
    net = StandIn()
    with pytest.raises(ValueError, match=r"in_colorspace / in_color_range \('bt709', 'tv'\) need a YUV in_format: in_format bgr24"):
        VideoUpscaler(net, (6, 8), (2, 2), in_format="bgr24", out_format="nv12", in_colorspace="bt709")
    with pytest.raises(ValueError, match=r"out_colorspace / out_color_range \('bt601', 'pc'\) need a YUV out_format: out_format bgr48le"):
        VideoUpscaler(net, (6, 8), (2, 2), in_format="p010", out_format="bgr48le", out_color_range="full")
    with pytest.raises(ValueError, match="unknown in_colorspace 'bt2020c'"):
        VideoUpscaler(net, (6, 8), (2, 2), in_format="nv12", in_colorspace="bt2020c")
    with pytest.raises(ValueError, match="unknown out_color_range 'studio'"):
        VideoUpscaler(net, (6, 8), (2, 2), out_format="nv12", out_color_range="studio")
    # aliases of the default pair are the default pair, on a packed side too
    up = VideoUpscaler(net, (6, 8), (2, 2), in_format="bgr24", out_format="bgr24", in_colorspace="bt470bg", out_color_range="limited")
    assert up.in_colour == up.out_colour == ("bt601", "tv")
    up = VideoUpscaler(net, (6, 8), (2, 2), in_format="yuv420p", out_format="p010", in_colorspace="bt2020", out_color_range="jpeg")
    assert up.in_colour == ("bt2020nc", "tv") and up.out_colour == ("bt601", "pc")


def test_module_passes_the_output_colour(monkeypatch):
    import savsr_b200
    from savsr_b200.archs import savsr_arch
    net = savsr_b200.SAVSR().eval()
    net.load_state_dict(make_state_dict(0), strict=True)
    seen = []

    class Plan(CpuPlanFrames):
        def forward_frames_into(self, ptrs, out, graph=True, out_format=None, **kw):
            seen.append((out_format, kw))

    with mocked_engine():
        monkeypatch.setattr(savsr_arch, "engine", SimpleNamespace(**{**vars(engine), "Plan": lambda p, b, h, w, s, d, io="f32", **kw:
                                                                       Plan(p, b, h, w, s, **kw)}))
        pool = torch.zeros(9, 8, 10, 3, dtype=torch.uint8).as_subclass(_ClaimsCuda)
        net._forward_bgr_u8_indexed(pool, [[0] * 7], (2, 2), "nv12")
        net._forward_bgr_u8_indexed(pool, [[0] * 7], (2, 2), "nv12", out_colorspace="bt709", out_color_range="full")
        assert seen == [("nv12", {}), ("nv12", {"out_colorspace": "bt709", "out_color_range": "pc"})]
        with pytest.raises(ValueError, match="need a YUV out_format"):
            net._forward_bgr_u8_indexed(pool, [[0] * 7], (2, 2), None, out_colorspace="bt709")


# ------------------------------------------------------------------------------------------------ GPU

DEV = torch.device("cuda", 0)


@pytest.mark.gpu
@pytest.mark.parametrize("cs,rng", NEW_PAIRS)
def test_every_8bit_triple_on_the_device(cs, rng):
    """Decode of all 2^24 (Y, U, V) as yuv420p and as pitched NV12, and encode of all 2^24 BGR triples on the top-left pixel of a 2x2
    block (four shifted frames) and as luma everywhere."""
    N = 4096
    b = torch.arange(N // 2 * N // 2, device=DEV)
    U, V = ((b // 64) // 256).reshape(1, N // 2, N // 2), ((b // 64) % 256).reshape(1, N // 2, N // 2)
    y4 = (4 * (b % 64)).reshape(N // 2, N // 2)
    Y = torch.stack([torch.stack([y4, y4 + 1], -1), torch.stack([y4 + 2, y4 + 3], -1)], 1).reshape(1, N, N)
    want = torch.stack(dec(Y, _up(U), _up(V), cs, rng, 8), -1)
    for fmt, pitch in (("yuv420p", None), ("nv12", N + 64)):
        x = frames8(Y, U, V, fmt, pitch)
        got = colour.yuv420_to_bgr(x, fmt, colorspace=cs, color_range=rng)
        assert torch.equal(got.to(torch.int64), want), (cs, rng, fmt)
    p = torch.arange(N * N, device=DEV)
    base = torch.stack([p >> 16, (p >> 8) & 255, p & 255], -1).to(torch.uint8).reshape(1, N, N, 3)
    for dy, dx in ((0, 0), (0, 1), (1, 0), (1, 1)):
        bgr = torch.roll(base, (dy, dx), (1, 2)).contiguous()
        for fmt in ("yuv420p", "nv12"):
            got = colour.bgr_to_yuv420(bgr, fmt, colorspace=cs, color_range=rng)
            assert torch.equal(got, enc_frames(bgr, fmt, cs, rng)), (cs, rng, fmt, dy, dx)


@pytest.mark.gpu
@pytest.mark.parametrize("cs,rng", NEW_PAIRS)
def test_every_10bit_triple_on_pitched_p010(cs, rng):
    """All 2^30 (Y, U, V) in 16 frames of 8192 x 8192, laid out as in tests/test_video_deep.py, on P010 with a row pitch."""
    N = 8192
    b = torch.arange(N // 2 * N // 2, device=DEV)
    y4 = (4 * (b % 256)).reshape(N // 2, N // 2)
    Y = torch.stack([torch.stack([y4, y4 + 1], -1), torch.stack([y4 + 2, y4 + 3], -1)], 1).reshape(1, N, N)
    for chunk in range(16):
        uv = chunk * 65536 + b // 256
        U, V = (uv // 1024).reshape(1, N // 2, N // 2), (uv % 1024).reshape(1, N // 2, N // 2)
        got = _i64(colour.yuv420_to_bgr(frames10(Y, U, V, "p010", 8448), "p010", colorspace=cs, color_range=rng))
        want = dec(Y, _up(U), _up(V), cs, rng, 10)
        for k in range(3):
            assert torch.equal(got[..., k], want[k]), (cs, rng, chunk, k)
        del got, want


@pytest.mark.gpu
@pytest.mark.parametrize("cs,rng", NEW_PAIRS)
@pytest.mark.parametrize("h,w", [(2, 2), (144, 180), (1080, 1920)])
def test_16bit_encode_on_the_device(cs, rng, h, w):
    n = 3
    g = torch.Generator().manual_seed(h + w)
    v = torch.randint(0, 65536, (n, h, w, 3), generator=g)
    ends = torch.tensor([0, 1, 255, 256, 32767, 32768, 65279, 65534, 65535])
    edge = torch.stack(torch.meshgrid(ends, ends, ends, indexing="ij"), -1).reshape(-1)
    v.view(-1)[:min(v.numel(), edge.numel())] = edge[:min(v.numel(), edge.numel())]
    bgr = _u16(v).to(DEV)
    for fmt, pitch in (("yuv420p10le", None), ("p010", w + 64)):
        want = _i64(enc_frames(bgr, fmt, cs, rng))
        if pitch is None:
            got = colour.bgr_to_yuv420(bgr, fmt, colorspace=cs, color_range=rng)
        else:
            surf = _u16(torch.full((n, 3 * h // 2, pitch), 7, device=DEV))
            got = colour.bgr_to_yuv420(bgr, fmt, out=surf[:, :, :w], colorspace=cs, color_range=rng)
            assert int((_i64(surf[:, :, w:]) != 7).sum()) == 0
        assert torch.equal(_i64(got), want), (cs, rng, fmt)


@pytest.mark.gpu
def test_cs_entry_points_with_the_default_pair_are_the_plain_ones():
    ctx = engine.context(0)
    lib, st = ctx.lib, torch.cuda.current_stream().cuda_stream
    n, h, w = 2, 36, 44
    g = torch.Generator().manual_seed(9)
    x8 = torch.randint(0, 256, (n, 3 * h // 2, w), dtype=torch.uint8, generator=g).to(DEV)
    x16 = _u16(torch.randint(0, 1024, (n, 3 * h // 2, w), generator=g) << 6).to(DEV)
    b8 = torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, generator=g).to(DEV)
    b16 = _u16(torch.randint(0, 65536, (n, h, w, 3), generator=g)).to(DEV)

    def run(fn, src, dst, args_of):
        dst.view(torch.int16 if dst.dtype == torch.uint16 else torch.uint8).zero_()
        assert fn(ctx.handle, *args_of(src, dst)) == 0
        torch.cuda.synchronize()
        return dst.clone()
    p8 = lambda x: (x.data_ptr(), w, x.data_ptr() + h * w, x.data_ptr() + h * w + 1, w, 2, x.stride(0))  # noqa: E731  nv12
    p16 = lambda x: (x.data_ptr(), w, x.data_ptr() + 2 * h * w, x.data_ptr() + 2 * h * w + 2, w, 2, x.stride(0))  # noqa: E731  p010
    cases = [("savsr_yuv420_to_bgr", x8, torch.empty_like(b8), lambda s, d, *c: (*p8(s), n, h, w, d.data_ptr(), *c, st)),
             ("savsr_bgr_to_yuv420", b8, torch.empty_like(x8), lambda s, d, *c: (s.data_ptr(), n, h, w, *p8(d), *c, st)),
             ("savsr_yuv420_10_to_bgr48", x16, _u16(torch.zeros(n, h, w, 3, device=DEV)),
              lambda s, d, *c: (*p16(s), 1, n, h, w, d.data_ptr(), *c, st)),
             ("savsr_bgr48_to_yuv420_10", b16, _u16(torch.zeros(n, 3 * h // 2, w, device=DEV)),
              lambda s, d, *c: (s.data_ptr(), n, h, w, *p16(d), 1, *c, st))]
    for name, src, dst, args in cases:
        plain = run(getattr(lib, name), src, dst, lambda s, d: args(s, d))
        cs = run(getattr(lib, name + "_cs"), src, dst, lambda s, d: args(s, d, 0, 0))
        assert torch.equal(plain.view(torch.uint8), cs.view(torch.uint8)), name
        assert int(plain.view(torch.uint8).count_nonzero()) > 0
        other = run(getattr(lib, name + "_cs"), src, dst, lambda s, d: args(s, d, 1, 0))
        assert not torch.equal(other.view(torch.uint8), plain.view(torch.uint8)), name
        dst.view(torch.uint8).fill_(0)
        for bad, msg in (((3, 0), b"unknown colorspace 3"), ((-1, 0), b"unknown colorspace -1"), ((0, 2), b"unknown color range 2")):
            assert getattr(lib, name + "_cs")(ctx.handle, *args(src, dst, *bad)) != 0
            assert msg in lib.savsr_last_error() and (name + "_cs").encode() in lib.savsr_last_error()
        torch.cuda.synchronize()
        assert int(dst.view(torch.uint8).count_nonzero()) == 0                # refused before any launch


def _gpu_net(precision):
    import savsr_b200
    net = savsr_b200.SAVSR().to(DEV).eval()
    net.load_state_dict(make_state_dict(0), strict=True)
    net.precision = precision
    return net


def _gpu_dec(x, fmt, pair):
    return colour.yuv420_to_bgr(x, fmt, colorspace=pair[0], color_range=pair[1])


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "fp16"])
@pytest.mark.parametrize("scale", [(4, 4), (1.5, 4)])
def test_video_upscaler_colour_pairs(precision, scale):
    import savsr_b200
    net = _gpu_net(precision)
    h, w, T, batch = 144, 180, 13, (8, 4)
    g = torch.Generator().manual_seed(11)
    Y8 = torch.randint(0, 256, (T, h, w), generator=g)
    U8, V8 = (torch.randint(0, 256, (T, h // 2, w // 2), generator=g) for _ in range(2))
    Y10 = torch.randint(0, 1024, (T, h, w), generator=g)
    U10, V10 = (torch.randint(0, 1024, (T, h // 2, w // 2), generator=g) for _ in range(2))
    clips = {"nv12": frames8(Y8, U8, V8, "nv12"), "yuv420p": frames8(Y8, U8, V8, "yuv420p"), "p010": frames10(Y10, U10, V10, "p010"),
             "bgr24": torch.randint(0, 256, (T, h, w, 3), dtype=torch.uint8, generator=g)}
    net.set_scale(scale)
    deep16 = lambda x: net.forward_bgr48(x.view(torch.uint16)).view(torch.int16)  # noqa: E731
    with torch.no_grad():
        for in_fmt, in_pair, out_fmt, out_pair in STREAMS:
            src = clips[in_fmt].to(DEV)
            bgr = src if in_fmt == "bgr24" else _gpu_dec(src, in_fmt, in_pair)
            if out_fmt in colour.DEEP_FORMATS:
                if bgr.dtype == torch.uint8:
                    wide = _u16(torch.zeros(bgr.shape, device=DEV))
                    bgr = colour.widen(bgr, wide)
                hr = sharding.infer_clip(deep16, bgr.view(torch.int16), batch=batch).view(torch.uint16)
            else:
                hr = sharding.infer_clip(net.forward_bgr_u8, bgr, batch=batch)
            want = colour.bgr_to_yuv420(hr, out_fmt, colorspace=out_pair[0], color_range=out_pair[1]).view(torch.uint8)
            up = savsr_b200.VideoUpscaler(net, (h, w), scale, batch=batch, in_format=in_fmt, out_format=out_fmt, **_kw(in_pair, out_pair))
            for feed in (list(clips[in_fmt]), list(src)):              # host frames and device frames
                up.reset()
                outs = []
                for f in feed:
                    outs += up.push(f)
                outs += up.finish()
                got = torch.cat([y for _, y in outs]).view(torch.uint8)
                assert torch.equal(got, want), (precision, scale, in_fmt, in_pair, out_fmt, out_pair)
            # and the new conversions really differ from the default pair on this clip
            default = colour.bgr_to_yuv420(hr, out_fmt).view(torch.uint8)
            assert not torch.equal(default, want)
