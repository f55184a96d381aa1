"""Scene cuts in the streaming upscaler: the window fold (sharding.scene_window_indices), cuts in infer_clip, the integer cut score
(savsr_b200.scenes, csrc/scenes.cu) and VideoUpscaler(scene_threshold=..., push(new_scene=...)).

CPU: the fold against frame_window_indices, the window-index cache, the threshold bound against exact fractions, the recorded launch
list of a stream against the recording fake library (no cut: today's list; marked cuts: the pointer writer with the host fold; detection:
one score launch per frame and the scene table writer, with no host synchronise), the stream against infer_clip(cuts=...) with a CPU
stand-in for the forward, and the refusals.
GPU, all exact: the score kernel against NumPy, the scene table writer against the host fold for every cut pattern of 12 frames, and
streams of a real net against the composition enc(infer_clip(forward, dec(frames), batch, cuts)).
"""
import ctypes as C
import math
import random
from fractions import Fraction
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from fake_lib import CpuPlan, mocked_engine
from oracle.state_dict_fixture import make_state_dict
from savsr_b200 import _capi as K
from savsr_b200 import colour, engine, scenes, sharding
from savsr_b200.videostream import VideoUpscaler


# ------------------------------------------------------------------------------------------------ CPU

def test_fold_is_the_reference_reflection_for_shots_of_4_or_more():
    for L in range(4, 41):
        for start in (0, 7):
            for c in range(start, start + L):
                got = sharding.scene_window_indices(c, start, start + L)
                assert got == [start + i for i in sharding.frame_window_indices(c - start, L)], (L, start, c)


def test_fold_stays_inside_short_shots():
    for L in (1, 2, 3):
        for c in range(10, 10 + L):
            got = sharding.scene_window_indices(c, 10, 10 + L)
            assert all(10 <= i < 10 + L for i in got) and got[3] == c, (L, c, got)
    assert sharding.scene_window_indices(5, 5, 6) == [5] * 7
    assert sharding.scene_window_indices(0, 0, 2) == [1, 0, 1, 0, 1, 0, 1]
    assert sharding.scene_window_indices(1, 0, 3) == [2, 1, 0, 1, 2, 1, 0]
    with pytest.raises(ValueError):
        sharding.frame_window_indices(0, 3)                # unchanged: a clip of 3 frames is refused


def test_infer_clip_without_cuts_gathers_as_before_and_the_cache_keys_the_cuts():
    sharding._WINDOW_INDEX_CACHE.clear()
    clip = torch.arange(20).view(20, 1)
    seen = []

    def net(x):
        seen.append(x[..., 0].tolist())
        return x[:, 3]
    sharding.infer_clip(net, clip, batch=8)
    assert seen == [[sharding.frame_window_indices(c, 20) for c in range(i, j)] for i, j in sharding.batch_schedule(20, 8)]
    assert all(len(k) == 5 for k in sharding._WINDOW_INDEX_CACHE)       # the key of a clip without cuts is the one it always was
    n = len(sharding._WINDOW_INDEX_CACHE)
    for cuts in ([5], [5, 6], [12]):
        seen.clear()
        sharding.infer_clip(net, clip, batch=8, cuts=cuts)
        assert seen == [[sharding.clip_window_indices(c, 20, cuts) for c in range(i, j)] for i, j in sharding.batch_schedule(20, 8)]
    assert len(sharding._WINDOW_INDEX_CACHE) == n + 3 * 3
    assert not torch.equal(sharding.gather_windows(clip, [4], cuts=[5]), sharding.gather_windows(clip, [4], cuts=[6]))
    assert torch.equal(sharding.gather_windows(clip, range(20), cuts=[]), sharding.gather_windows(clip, range(20)))
    for bad in ([5, 5], [6, 5], [20], [-1]):
        with pytest.raises(ValueError, match="cuts must be sorted"):
            sharding.gather_windows(clip, [0], cuts=bad)
    with pytest.raises(ValueError, match="too short"):
        sharding.gather_windows(clip[:3], [0], cuts=[1])


def test_bound_is_the_exact_ceiling():
    for tau in (10, 10.0, 0.1, 1 / 3, 2 / 3, 0.3, 7.7, 12.345, 99.99, 100, 1e-9, math.nextafter(10.0, 0.0)):
        for h, w, maxval in ((270, 480, 255), (37, 45, 65535), (1, 1, 255)):
            want = Fraction(tau) * 3 * h * w * maxval / 100
            b = scenes.score_bound(tau, h, w, maxval)
            assert b == math.ceil(want) and b - 1 < want <= b, (tau, h, w)
    assert scenes.score_bound(10, 270, 480, 255) == 3 * 270 * 480 * 255 // 10
    assert scenes.score_bound(0.1, 2, 2, 255) == math.ceil(Fraction(0.1) * 3060 / 100) == 4   # 0.1's float is above 1/10


def test_reference_scores_depth_invariance():
    g = np.random.default_rng(0)
    x = g.integers(0, 256, (9, 5, 7, 3)).astype(np.uint8)
    x[4:] = x[3]                                            # still frames: SAD 0
    s8, sc8, c8 = scenes.reference_scores(x, 10)
    s16, sc16, c16 = scenes.reference_scores(x.astype(np.uint16) * 257, 10)
    assert (s16 == 257 * s8).all() and np.allclose(sc8, sc16) and (c8 == c16).all()
    assert s8[0] == 0 and not c8[0] and (s8[5:] == 0).all()


class _ClaimsCuda(torch.Tensor):
    """A CPU tensor that reports is_cuda, so the module's host logic runs without a device (nothing is launched)."""
    is_cuda = property(lambda self: True)


class CpuPlanFrames(CpuPlan):
    io = "bgr_u8_frames"


def _cpu_net(monkeypatch):
    """A real SAVSR whose plans are CPU plans on the recording fake library, eager (no graph), its device check relaxed."""
    import savsr_b200
    from savsr_b200.archs import savsr_arch
    net = savsr_b200.SAVSR().eval()
    net.load_state_dict(make_state_dict(0), strict=True)
    net.use_graph = False
    monkeypatch.setattr(net, "_check_device", lambda x: None)
    monkeypatch.setattr(savsr_arch, "engine", SimpleNamespace(**{**vars(engine), "Plan": lambda p, b, h, w, s, d, io="f32", **kw:
                                                                   CpuPlanFrames(p, b, h, w, s, **kw)}))
    return net


def _frames(T, h=8, w=10, seed=0):
    return torch.randint(0, 256, (T, h, w, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(seed))


def _run_stream(up, clip, marks=(), chunk=1):
    """Push `clip` `chunk` frames at a time, with new_scene on the pushes that begin at a frame of `marks`; returns the outputs."""
    outs, T, k = [], clip.shape[0], 0
    starts = sorted(set(range(0, T, chunk)) | set(marks))
    for a, b in zip(starts, starts[1:] + [T]):
        outs += up.push(clip[a:b], new_scene=a in marks)
    return outs + up.finish()


def _split(calls):
    """The recorded calls grouped per forward: [(table writer call, names of the plan's launches), ...] and the other calls."""
    fwd, other, cur = [], [], None
    for name, args in calls:
        if name in ("savsr_write_frame_table", "savsr_write_scene_frame_table"):
            cur = ((name, args), [])
            fwd.append(cur)
        elif name.startswith("savsr_scene_score"):
            other.append((name, args))
        elif cur is not None:
            cur[1].append(name)
        else:
            other.append((name, args))
    return fwd, other


def _pointer_windows(args, ring, R):
    fb = ring[0].numel() * ring.element_size()
    ptrs = [args[2][k] for k in range(args[3])]
    return [[(p - ring.data_ptr()) // fb for p in ptrs[7 * n:7 * n + 7]] for n in range(len(ptrs) // 7)]


@pytest.mark.parametrize("batch", [4, (26, 8)])
def test_launch_lists_of_a_stream(monkeypatch, batch):
    net = _cpu_net(monkeypatch)
    T, marks = 23, (6, 7, 15)
    clip = _frames(T)
    with mocked_engine() as lib:
        # today's list: one forward per batch of the schedule, windows of frame_window_indices, through _forward_bgr_u8_indexed
        up = VideoUpscaler(net, (8, 10), (2, 2), batch=batch)
        R = up.capacity
        ring = up.ring.as_subclass(_ClaimsCuda)
        for _ in range(2):                                    # the second pass: every plan is built (its build-time calls are not launches)
            lib.calls.clear()
            for i, j in sharding.batch_schedule(T, batch):
                net._forward_bgr_u8_indexed(ring, [[f % R for f in sharding.frame_window_indices(c, T)] for c in range(i, j)], up.scale)
        today = [(a[0], [w for w in _pointer_windows(a[1], ring, R)], names) for a, names in _split(lib.calls)[0]]

        def stream(marks, **kw):
            up = VideoUpscaler(net, (8, 10), (2, 2), batch=batch, **kw)
            up.ring = up.ring.as_subclass(_ClaimsCuda)
            if up.detector is not None:
                up.detector.ring = up.ring
            lib.calls.clear()
            _run_stream(up, clip, marks, chunk=3)
            return up, _split(lib.calls)

        up, (fwd, other) = stream(())
        assert other == [] and [(a[0], _pointer_windows(a[1], up.ring, R), names) for a, names in fwd] == \
            [(n, [[f for f in w] for w in ws], names) for n, ws, names in today]
        assert up.scene_cuts() == []

        up, (fwd, other) = stream(marks)                      # marked cuts, no detection: the pointer writer with the host fold
        assert other == [] and [a[0] for a, _ in fwd] == ["savsr_write_frame_table"] * len(fwd)
        assert [names for _, names in fwd] == [names for _, _, names in today]
        want = [[[f % R for f in sharding.clip_window_indices(c, T, list(marks))] for c in range(i, j)]
                for i, j in sharding.batch_schedule(T, batch)]
        assert [_pointer_windows(a[1], up.ring, R) for a, _ in fwd] == want
        assert up.scene_cuts() == list(marks)

        def no_sync(*a, **k):
            raise AssertionError("push / finish synchronised with the device")
        monkeypatch.setattr(torch.cuda, "synchronize", no_sync)
        monkeypatch.setattr(torch.cuda.Event, "synchronize", no_sync)
        up, (fwd, other) = stream(marks, scene_threshold=10)  # detection: one score per frame, the scene table writer
        assert [n for n, _ in other] == ["savsr_scene_score_u8"] * T
        assert [a[5] for _, a in other] == list(range(T))                       # t
        assert [a[6] for _, a in other] == [int(t in marks) for t in range(T)]  # marked
        assert {a[7] for _, a in other} == {scenes.score_bound(10, 8, 10, 255)}
        assert all(a[1] == up.ring.data_ptr() and a[2] == R and a[8] == up.detector.cut.data_ptr() for _, a in other)
        assert [a[0] for a, _ in fwd] == ["savsr_write_scene_frame_table"] * len(fwd)
        assert [names for _, names in fwd] == [names for _, _, names in today]
        sched = sharding.batch_schedule(T, batch)
        # (ctx, table, ring, frame bytes, R, cut, first, count, received, finished, stream)
        got = [(a[1][2], a[1][3], a[1][4], a[1][6], a[1][7], a[1][8], a[1][9]) for a, _ in fwd]
        assert [g[0] for g in got] == [up.ring.data_ptr()] * len(sched) and {g[1:3] for g in got} == {(8 * 10 * 3, R)}
        assert all(a[1][5] == up.detector.cut.data_ptr() for a, _ in fwd)
        assert [(g[3], g[4]) for g in got] == [(i, j - i) for i, j in sched]
        assert got[-1][5] == T and got[-1][6] == 1
        assert all(g[5] >= g[3] + g[4] + 3 for g in got if not g[6])            # before the end: whole windows received


class StandIn:
    """CPU stand-in for a SAVSR in eval mode: the frame numbers of every window it is given (pixel (0, 0) carries them)."""
    training = False

    def __init__(self):
        self.gamma = torch.zeros(1)
        self.windows = []

    def _forward_bgr_u8_indexed(self, pool, windows, scale):
        x = pool[torch.as_tensor(windows)]
        self.windows.append(x[..., 0, 0, 0].long().tolist())
        return x[:, 3].repeat_interleave(2, 1).repeat_interleave(2, 2) + x.sum(1, dtype=torch.uint8).repeat_interleave(2, 1).repeat_interleave(2, 2)


@pytest.mark.parametrize("batch", [5, (26, 8)])
@pytest.mark.parametrize("T", [4, 9, 40])
def test_marked_stream_equals_infer_clip_with_cuts(T, batch):
    clip = _frames(T, 6, 8, seed=T)
    clip[:, 0, 0, 0] = torch.arange(T)
    rng = random.Random(T)
    for _ in range(4):
        marks = sorted(rng.sample(range(1, T), rng.randint(0, min(T - 1, 6))))
        seen = []

        def net(x):
            seen.append(x[..., 0, 0, 0].long().tolist())
            return x[:, 3].repeat_interleave(2, 1).repeat_interleave(2, 2) + x.sum(1, dtype=torch.uint8).repeat_interleave(2, 1).repeat_interleave(2, 2)
        want = sharding.infer_clip(net, clip, batch=batch, cuts=marks)
        for chunk in (1, 3):
            s = StandIn()
            up = VideoUpscaler(s, (6, 8), (2, 2), batch=batch)
            outs = _run_stream(up, clip, marks, chunk)
            assert s.windows == seen and torch.equal(torch.cat([y for _, y in outs]), want), (marks, chunk)
            assert up.scene_cuts() == marks
            up.reset()
            assert up.scene_cuts() == []


def test_refusals():
    s = StandIn()
    for bad in (0, -1, 100.5, float("nan"), float("inf"), "ten", [], 1e300):
        with pytest.raises(ValueError, match="scene_threshold"):
            VideoUpscaler(s, (6, 8), (2, 2), scene_threshold=bad)
    up = VideoUpscaler(s, (6, 8), (2, 2), batch=4)
    with pytest.raises(ValueError, match="new_scene"):
        up.push(torch.zeros(0, 6, 8, 3, dtype=torch.uint8), new_scene=True)
    assert up.push(torch.zeros(0, 6, 8, 3, dtype=torch.uint8)) == []
    up.push(_frames(3, 6, 8), new_scene=True)
    up.push(_frames(1, 6, 8), new_scene=True)
    assert up.scene_cuts() == [3]
    up.reset()
    up.push(_frames(2, 6, 8))
    up.push(_frames(1, 6, 8), new_scene=True)
    with pytest.raises(ValueError, match="too short"):     # a whole stream of 3 frames is still refused, cuts or not
        up.finish()
    assert scenes.check_threshold(100) == 100.0 and scenes.check_threshold(1e-6) == 1e-6


def test_c_writer_refusals_before_any_launch():
    """The argument checks of the C entry points run before any launch (they need no device: the checks come first)."""
    lib = K.load()
    cut = (C.c_uint8 * 8)()
    tab = (C.c_void_p * 70)()
    ring = (C.c_uint8 * 64)()
    sad, scratch = (C.c_ulonglong * 8)(), (C.c_ulonglong * 4)()
    ctx = C.c_void_p(1)   # never dereferenced: every call below is refused first
    cases = [
        (lambda: lib.savsr_write_scene_frame_table(ctx, tab, ring, 10, 6, cut, 0, 1, 8, 1, None), b"R = 6"),
        (lambda: lib.savsr_write_scene_frame_table(ctx, None, ring, 10, 8, cut, 0, 1, 8, 1, None), b"null"),
        (lambda: lib.savsr_write_scene_frame_table(ctx, tab, ring, 10, 8, None, 0, 1, 8, 1, None), b"null"),
        (lambda: lib.savsr_write_scene_frame_table(ctx, tab, ring, 10, 8, cut, 5, 4, 8, 1, None), b"reaches past the 8 received"),
        (lambda: lib.savsr_write_scene_frame_table(ctx, tab, ring, 10, 8, cut, 3, 2, 7, 0, None), b"not known"),
        (lambda: lib.savsr_write_scene_frame_table(ctx, tab, ring, 10, 8, cut, 0, 0, 8, 1, None), b"count = 0"),
        (lambda: lib.savsr_write_scene_frame_table(ctx, tab, ring, 10, 8, cut, 10, 2, 20, 0, None), b"more than the ring"),
        (lambda: lib.savsr_scene_score_u8(ctx, ring, 8, 2, 2, 0, 0, 0, cut, sad, scratch, None), b"bound = 0"),
        (lambda: lib.savsr_scene_score_u16(ctx, ring, 8, 2, 2, 0, 0, -5, cut, sad, scratch, None), b"bound = -5"),
        (lambda: lib.savsr_scene_score_u8(ctx, ring, 5, 2, 2, 0, 0, 10, cut, sad, scratch, None), b"R = 5"),
        (lambda: lib.savsr_scene_score_u8(ctx, ring, 8, 2, 2, 0, 0, 10, cut, sad, None, None), b"null"),
        (lambda: lib.savsr_scene_score_u8(ctx, None, 8, 2, 2, 0, 0, 10, cut, sad, scratch, None), b"null"),
    ]
    for call, msg in cases:
        assert call() != 0
        assert msg in lib.savsr_last_error(), (msg, lib.savsr_last_error())


# ------------------------------------------------------------------------------------------------ GPU

DEV = torch.device("cuda", 0)


def _gpu_net(precision="bf16", seed=0):
    import savsr_b200
    net = savsr_b200.SAVSR().to(DEV).eval()
    net.load_state_dict(make_state_dict(seed), strict=True)
    net.precision = precision
    return net


def _u16(x):
    x = x.to(torch.int32)
    return (x - 65536 * (x >= 32768)).to(torch.int16).view(torch.uint16)


def _i64(x):
    return x.view(torch.int16).to(torch.int64) & 0xFFFF if x.dtype == torch.uint16 else x.to(torch.int64)


def _score_all(frames, threshold, R=None, marks=()):
    """Score frames [T, h, w, 3] (CUDA, uint8 / uint16) through a ring of R slots; returns (SAD [T], cut [T]) read after each frame."""
    T = frames.shape[0]
    R = R or max(T, 7)
    ring = torch.zeros((R, *frames.shape[1:]), dtype=frames.dtype, device=DEV)
    det = scenes.Detector(ring, threshold)
    sad, cut = [], []
    for t in range(T):
        ring[t % R].copy_(frames[t])
        det.score(t, t in marks)
        sad.append(int(det.sad[t % R]))
        cut.append(bool(det.cut[t % R]))
    return np.array(sad, dtype=np.uint64), np.array(cut)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.uint8, torch.uint16])
@pytest.mark.parametrize("h,w", [(270, 480), (37, 45)])
def test_score_kernel_equals_numpy(dtype, h, w):
    g = torch.Generator().manual_seed(h + w)
    top = 256 if dtype == torch.uint8 else 65536
    base = torch.randint(0, top, (h, w, 3), generator=g)
    fr = [base]
    for t in range(1, 12):                                   # small drifts, a few jumps, a still frame, a flash
        if t in (4, 9):
            fr.append(torch.randint(0, top, (h, w, 3), generator=g))
        elif t == 6:
            fr.append(fr[-1].clone())
        else:
            fr.append((fr[-1] + torch.randint(-top // 50, top // 50 + 1, (h, w, 3), generator=g)).clamp(0, top - 1))
    x = torch.stack(fr)
    x = x.to(torch.uint8) if dtype == torch.uint8 else _u16(x)
    for tau, R in ((10, 7), (3.3, 12), (0.5, 32)):
        want_sad, _, want_cut = scenes.reference_scores(x.numpy(), tau)
        sad, cut = _score_all(x.to(DEV), tau, R=R, marks=(7,))
        want_cut[7] = True
        assert (sad == want_sad).all(), (tau, sad, want_sad)
        assert (cut == want_cut).all(), (tau, cut, want_cut)
    assert want_cut[4] and not want_cut[6]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.uint8, torch.uint16])
def test_score_decision_at_the_bound(dtype):
    """m_t exactly on, one below and one above the bound (100 m_t on, below and above tau * 3hw * maxval) pins the >=."""
    h, w = 33, 41
    maxval = 255 if dtype == torch.uint8 else 65535
    lib = engine.context(0).lib
    for S in (1, 777, 3 * h * w * 9 - 4):
        a = torch.zeros(h * w * 3, dtype=torch.int64)
        k, rest = divmod(S, 9)
        a[:k] = 9
        a[k] = rest
        x = torch.stack([torch.zeros_like(a), a]).view(2, h, w, 3)     # SAD_1 = S, m_1 = S
        x = (x.to(torch.uint8) if dtype == torch.uint8 else _u16(x * (maxval // 255)))
        m = S * (maxval // 255)
        for bound, fires in ((m, True), (m + 1, False), (m - 1, True)):
            if bound == 0:                                     # refused: a threshold is positive
                continue
            ring = torch.zeros(7, h, w, 3, dtype=dtype, device=DEV)
            ring[:2] = x.to(DEV)
            cut = torch.zeros(7, dtype=torch.uint8, device=DEV)
            sad = torch.zeros(7, dtype=torch.int64, device=DEV)
            scratch = torch.zeros(K.SCENE_SCRATCH_WORDS, dtype=torch.int64, device=DEV)
            fn = lib.savsr_scene_score_u16 if dtype == torch.uint16 else lib.savsr_scene_score_u8
            st = torch.cuda.current_stream().cuda_stream
            for t in (0, 1):
                K.check(fn(engine.context(0).handle, ring.data_ptr(), 7, h, w, t, 0, bound, cut.data_ptr(), sad.data_ptr(), scratch.data_ptr(), st))
            assert int(sad[1]) == m and bool(cut[1]) == fires and int(cut[0]) == 0, (S, bound)
            assert int(scratch[0]) == 0                            # the ticket counter is left ready for the next call


@pytest.mark.gpu
def test_scene_writer_equals_the_host_fold_for_every_cut_pattern():
    ctx = engine.context(0)
    lib, st = ctx.lib, torch.cuda.current_stream().cuda_stream
    N, fb = 12, 48
    pats = np.arange(1 << (N - 1))
    # host fold of every pattern: win[p, n, c] = the window of frame c among n frames, cuts = the pattern's frames below n
    win = np.zeros((len(pats), N + 1, N, 7), dtype=np.int64)
    for p in pats:
        for n in range(1, N + 1):
            cuts = [f for f in range(1, n) if p >> (f - 1) & 1]
            for c in range(n):
                win[p, n, c] = sharding.clip_window_indices(c, n, cuts)
    for R in (7, 32):
        ring = torch.empty(R * fb, dtype=torch.uint8, device=DEV)
        positions = [(n, finished, first, count) for n in range(1, N + 1) for finished in (0, 1) for first in range(n)
                     for count in range(1, min(n - first, R - 6) + 1)
                     if (finished or first + count + 2 < n) and n - max(first - 3, 0) <= R]
        # per (pattern, received n) the flags a ring of R slots holds: slot f % R <- the flag of frame f, for the last R frames
        flags = np.zeros((len(pats), N + 1, R), dtype=np.uint8)
        for n in range(1, N + 1):
            for f in range(max(1, n - R), n):
                flags[:, n, f % R] = (pats >> (f - 1)) & 1
        flags_d = torch.from_numpy(flags).to(DEV)
        fp = flags_d.data_ptr()
        total = sum(7 * q[3] for q in positions) * len(pats)
        table = torch.zeros(total, dtype=torch.int64, device=DEV)
        tp, base = table.data_ptr(), ring.data_ptr()
        expect, off = [], 0
        for n, finished, first, count in positions:
            for p in range(len(pats)):
                K.check(lib.savsr_write_scene_frame_table(ctx.handle, tp + 8 * off, base, fb, R, fp + (p * (N + 1) + n) * R, first, count, n,
                                                          finished, st))
                off += 7 * count
            expect.append((base + fb * (win[:, n, first:first + count] % R)).reshape(-1))
        got = table.cpu().numpy()
        expect = np.concatenate(expect)
        bad = np.nonzero(got != expect)[0]
        assert bad.size == 0, (R, bad[:10], got[bad[:10]], expect[bad[:10]])


def _texture(seed, h, w, maxval):
    """A smooth random texture (a 12 x 12 grid of values, upsampled bilinearly): a shift of one pixel changes it little."""
    g = torch.Generator().manual_seed(seed)
    grid = torch.rand(1, 3, 12, 12, generator=g)
    big = torch.nn.functional.interpolate(grid, size=(h, w), mode="bilinear", align_corners=False)[0].permute(1, 2, 0)
    return (big * maxval).round()


def _multishot(lengths, h, w, maxval, seed=0):
    """Frames [T, h, w, 3] (int64 values in [0, maxval]): one drifting crop of an unrelated texture per shot; returns (frames, cut frames)."""
    frames, cuts, k = [], [], 0
    for s, L in enumerate(lengths):
        tex = _texture(seed * 100 + s, h + 64, w + 64, maxval)
        for t in range(L):
            frames.append(tex[t:t + h, t:t + w])
        if s:
            cuts.append(k)
        k += L
    return torch.stack(frames).to(torch.int64), cuts


SHOTS = [30, 2, 5, 1, 3, 30]          # cuts at 30, 32, 37, 38, 41; the one that ends the 1-frame shot (38) is not detected: it is marked


def _source(fmt, bgr8):
    """The multi-shot clip in `fmt` on the device, from 8-bit BGR values [T, h, w, 3]."""
    x = bgr8.to(DEV)
    if fmt == "bgr24":
        return x.to(torch.uint8)
    if fmt == "p010":
        return colour.bgr_to_yuv420(_u16(x * 257), "p010")
    return colour.bgr_to_yuv420(x.to(torch.uint8), fmt)


def _decoded(fmt, src, deep_out):
    bgr = src if fmt == "bgr24" else colour.yuv420_to_bgr(src, fmt)
    if deep_out and bgr.dtype == torch.uint8:
        bgr = colour.widen(bgr, out=torch.empty(bgr.shape, dtype=torch.uint16, device=DEV))
    return bgr


def _composition(net, bgr, out_fmt, batch, cuts):
    if bgr.dtype == torch.uint16:
        deep = lambda x: net.forward_bgr48(x.view(torch.uint16)).view(torch.int16)  # noqa: E731
        hr = sharding.infer_clip(deep, bgr.view(torch.int16), batch=batch, cuts=cuts).view(torch.uint16)
    else:
        hr = sharding.infer_clip(net.forward_bgr_u8, bgr, batch=batch, cuts=cuts)
    return hr if out_fmt in ("bgr24", "bgr48le") else colour.bgr_to_yuv420(hr, out_fmt)


def _stream(net, src, in_fmt, out_fmt, scale, batch, marks, **kw):
    h, w = (src.shape[1] * 2 // 3, src.shape[2]) if in_fmt in colour.YUV_FORMATS else src.shape[1:3]
    up = VideoUpscaler(net, (h, w), scale, batch=batch, in_format=in_fmt, out_format=out_fmt, **kw)
    outs, starts = [], sorted({0, *marks})
    T = src.shape[0]
    for a, b in zip(starts, starts[1:] + [T]):
        for k in range(a, b, 4):
            outs += up.push(src[k:min(k + 4, b)], new_scene=k == a and a in marks)
    outs += up.finish()
    return up, outs


@pytest.mark.gpu
@pytest.mark.parametrize("in_fmt,out_fmt,precision,scale,batch,detect", [
    ("bgr24", "bgr24", "bf16", (4, 4), (26, 8), True),
    ("nv12", "nv12", "fp16", (1.5, 4), 5, True),
    ("p010", "p010", "bf16", (1.5, 4), (26, 8), True),
    ("nv12", "p010", "bf16", (4, 4), 5, True),
    ("bgr24", "nv12", "fp16", (4, 4), (26, 8), False),       # marked cuts only
])
def test_stream_with_cuts_equals_the_composition(in_fmt, out_fmt, precision, scale, batch, detect):
    h, w = 64, 96
    vals, true_cuts = _multishot(SHOTS, h, w, 255)
    flash_end = true_cuts[3]                                 # the frame after the 1-frame shot
    assert flash_end == true_cuts[2] + 1
    net = _gpu_net(precision)
    src = _source(in_fmt, vals)
    deep_out = out_fmt in colour.DEEP_FORMATS
    bgr = _decoded(in_fmt, src, deep_out)
    marks = [flash_end] if detect else list(true_cuts)
    with torch.no_grad():
        up, outs = _stream(net, src, in_fmt, out_fmt, scale, batch, marks, **({"scene_threshold": 10} if detect else {}))
        cuts = up.scene_cuts()
        assert cuts == true_cuts, (cuts, true_cuts)
        if detect:
            _, _, ref = scenes.reference_scores(bgr.cpu().numpy(), 10)
            assert sorted(set(np.nonzero(ref)[0].tolist()) | {flash_end}) == true_cuts
            assert not ref[flash_end]                        # not detected by design: its SAD and the one before it cancel
        net.set_scale(scale)
        want = _composition(net, bgr, out_fmt, batch, cuts)
    assert [s for s, _ in outs] == [i for i, _ in sharding.batch_schedule(bgr.shape[0], batch)]
    got = torch.cat([y for _, y in outs])
    assert torch.equal(_i64(got), _i64(want))


@pytest.mark.gpu
def test_depth_invariance_of_the_cuts():
    vals, true_cuts = _multishot(SHOTS, 48, 64, 255, seed=3)
    net = _gpu_net()
    src = _source("nv12", vals)
    with torch.no_grad():
        up8, _ = _stream(net, src, "nv12", "nv12", (2, 2), (26, 8), (), scene_threshold=10)
        up16, _ = _stream(net, src, "nv12", "p010", (2, 2), (26, 8), (), scene_threshold=10)
        assert up16.ring.dtype == torch.uint16 and up8.ring.dtype == torch.uint8
        assert up8.scene_cuts() == up16.scene_cuts() == [c for c in true_cuts if c != true_cuts[3]]
        c8 = _stream(net, src, "nv12", "nv12", (2, 2), 8, (), scene_threshold=2.5)[0].scene_cuts()
        c16 = _stream(net, src, "nv12", "p010", (2, 2), 8, (), scene_threshold=2.5)[0].scene_cuts()
        assert c8 == c16


@pytest.mark.gpu
def test_one_shot_video_is_unchanged():
    T, h, w, batch = 34, 144, 180, (26, 8)                     # the Vid4 clip's shape, at x4
    vals, _ = _multishot([T], h, w, 255, seed=7)
    clip = vals.to(torch.uint8).to(DEV)
    _, score, _ = scenes.reference_scores(clip.cpu().numpy())
    tau = min(100.0, float(score.max()) + 1.0)
    assert tau < 100
    net = _gpu_net()
    with torch.no_grad():
        off, a = _stream(net, clip, "bgr24", "bgr24", (4, 4), batch, ())
        on, b = _stream(net, clip, "bgr24", "bgr24", (4, 4), batch, (), scene_threshold=tau)
        net.set_scale((4, 4))
        today = sharding.infer_clip(net.forward_bgr_u8, clip, batch=batch)
    assert on.scene_cuts() == [] and off.scene_cuts() == []
    assert torch.equal(torch.cat([y for _, y in b]), torch.cat([y for _, y in a]))
    assert torch.equal(torch.cat([y for _, y in a]), today)


@pytest.mark.gpu
def test_memory_does_not_grow_with_the_length_with_detection_on():
    import savsr_b200
    net = _gpu_net()
    h, w = 24, 32
    up = savsr_b200.VideoUpscaler(net, (h, w), (2, 2), batch=4, scene_threshold=10)
    vals, _ = _multishot([3, 5], h, w, 255, seed=4)
    frames = vals.to(torch.uint8)

    def run(T):
        up.reset()
        for k in range(T):
            for _, hr in up.push(frames[k % 8], new_scene=k % 50 == 49):
                del hr
        for _, hr in up.finish():
            del hr
        torch.cuda.synchronize()

    with torch.no_grad():
        run(100)
        torch.cuda.reset_peak_memory_stats(DEV)
        run(500)
        peak500 = torch.cuda.max_memory_allocated(DEV)
        torch.cuda.reset_peak_memory_stats(DEV)
        run(2000)
        peak2000 = torch.cuda.max_memory_allocated(DEV)
        assert len(up.scene_cuts()) > 2000 // 8
    assert peak2000 <= peak500, (peak500, peak2000)
