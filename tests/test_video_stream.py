"""Streaming 8-bit video: frames read in place through a frame table (engine.Plan(io="bgr_u8_frames"), savsr_forward_u8_frames,
SAVSR.forward_bgr_u8_indexed) and the frame-in / frame-out driver savsr_b200.VideoUpscaler.

CPU: the launch list against the recording fake library, the plan cache, the refusals of forward_bgr_u8_indexed, and the driver's
host logic with a CPU stand-in for the forward: its windows and batch partition are those of infer_clip / batch_schedule.
GPU, all exact:  forward_bgr_u8_indexed(pool, idx) == forward_bgr_u8(pool[idx]),  savsr_forward_u8_frames == savsr_forward_u8, and
VideoUpscaler == infer_clip(net.forward_bgr_u8, clip, batch=...).
"""
import random
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from fake_lib import CpuPlan, mocked_engine
from oracle.state_dict_fixture import make_state_dict
from savsr_b200 import engine, sharding
from savsr_b200.videostream import VideoUpscaler


# ------------------------------------------------------------------------------------------------ CPU

class CpuPlanU8(CpuPlan):
    io = "bgr_u8"


class CpuPlanFrames(CpuPlan):
    io = "bgr_u8_frames"


@pytest.fixture(scope="module")
def sd():
    return make_state_dict(0)


def _record(cls, sd, store, b=2, h=13, w=15, scale=(1.5, 4)):
    with mocked_engine() as lib:
        plan = cls(sd, b, h, w, scale, store=store)
        for op in plan.ops:
            assert op(0) == 0
        return plan, list(lib.calls)


def test_frames_plan_swaps_only_the_first_and_last_launch(sd):
    store = engine.WeightStore()
    _record(CpuPlanU8, sd, store)                      # fills the store: the plans below record launches only
    n_keys = len(store.cache)
    p8, c8 = _record(CpuPlanU8, sd, store)
    pf, cf = _record(CpuPlanFrames, sd, store)
    assert len(store.cache) == n_keys                  # every derived weight came from the shared store
    n8, nf = [c[0] for c in c8], [c[0] for c in cf]
    assert len(n8) == len(nf) and len(p8.ops) == len(pf.ops) and p8.n_launches == pf.n_launches
    diff = [(a, b) for a, b in zip(n8, nf) if a != b]
    assert diff == [("savsr_pack_frames_u8", "savsr_pack_frames_u8_table"), ("savsr_satu_hr_u8", "savsr_satu_hr_u8_table")]
    run = cf[-len(pf.ops):]                            # the calls of the launch list (one per op), after the build-time calls
    assert run[0][0] == "savsr_pack_frames_u8_table" and run[-1][0] == "savsr_satu_hr_u8_table"
    for a, b in zip(c8, cf):                           # the launches between them: same scalar arguments
        assert len(a[1]) == len(b[1])
        assert [v for v in a[1] if isinstance(v, (float, str))] == [v for v in b[1] if isinstance(v, (float, str))]
    table = pf.frame_table.data_ptr()
    assert run[0][1][2] == table and run[0][1][3:7] == (7, 13, 15, 1)
    assert run[-1][1][14] == table and run[-1][1][17] == pf.out.data_ptr()
    assert pf.x_in is None                              # no input staging: the frames are read in place
    assert pf.frame_table.dtype == torch.int64 and tuple(pf.frame_table.shape) == (2 * 7,)
    assert pf.out.dtype == torch.uint8 and tuple(pf.out.shape) == (2, *engine.get_hw(13, 15, (1.5, 4)), 3)
    assert pf.nbytes < p8.nbytes
    with pytest.raises(ValueError, match="forward_frames_into"):
        pf.forward_into(torch.zeros(2, 7, 13, 15, 3, dtype=torch.uint8), torch.empty_like(pf.out))
    with pytest.raises(ValueError, match="bgr_u8_frames"):
        p8.forward_frames_into([0] * 14, torch.empty_like(p8.out))


def test_frames_table_writer_gets_every_pointer(sd):
    pf, _ = _record(CpuPlanFrames, sd, engine.WeightStore(), b=3)
    lib = pf.lib
    lib.calls.clear()
    with mocked_engine():
        ptrs = [0x1000 * (k + 1) for k in range(21)]
        pf.write_frame_table(ptrs)
        (name, args), = lib.calls
        assert name == "savsr_write_frame_table" and args[1] == pf.frame_table.data_ptr() and args[3] == 21
        assert [args[2][k] for k in range(21)] == ptrs
        with pytest.raises(ValueError, match="21 frame pointers"):
            pf.write_frame_table(ptrs[:-1])


class _ClaimsCuda(torch.Tensor):
    """A CPU tensor that reports is_cuda, so the module's host logic runs without a device (nothing is launched)."""
    is_cuda = property(lambda self: True)


def _cpu_net():
    import savsr_b200
    net = savsr_b200.SAVSR().eval()
    net.load_state_dict(make_state_dict(0), strict=True)
    net.set_scale((2, 2))
    return net


def test_plan_cache_keys_the_frames_mode(monkeypatch):
    net = _cpu_net()
    built = []

    def fake_plan(params, b, h, w, s, device, io="f32", **kw):
        built.append(io)
        cls = {"f32": CpuPlan, "bgr_u8": CpuPlanU8, "bgr_u8_frames": CpuPlanFrames}[io]
        return cls(params, b, h, w, s, **kw)
    from savsr_b200.archs import savsr_arch
    with mocked_engine():
        monkeypatch.setattr(savsr_arch, "engine", SimpleNamespace(**{**vars(engine), "Plan": fake_plan}))
        x8 = torch.zeros(1, 7, 8, 10, 3, dtype=torch.uint8).as_subclass(_ClaimsCuda)
        a = net.plan_for(x8, io="bgr_u8")
        b = net._plan(1, 8, 10, x8.device, "bgr_u8_frames", net.scale)
        assert built == ["bgr_u8", "bgr_u8_frames"] and a is not b and a.store is b.store
        assert net._plan(1, 8, 10, x8.device, "bgr_u8_frames", net.scale) is b and len(built) == 2
        assert sorted(k[9] for k in net._plans) == ["bgr_u8", "bgr_u8_frames"]
        c = net._plan(1, 8, 10, x8.device, "bgr_u8_frames", (4, 4))          # the scale is part of the key
        assert c is not b and len(built) == 3


def test_forward_bgr_u8_indexed_refusals():
    net = _cpu_net()
    pool = torch.zeros(5, 8, 10, 3, dtype=torch.uint8).as_subclass(_ClaimsCuda)
    idx = [[0, 1, 2, 3, 4, 4, 4]]
    with pytest.raises(TypeError, match="uint8"):
        net.forward_bgr_u8_indexed(pool.float(), idx)
    with pytest.raises(ValueError, match=r"\[N, h, w, 3\]"):
        net.forward_bgr_u8_indexed(torch.zeros(5, 3, 8, 10, dtype=torch.uint8).as_subclass(_ClaimsCuda), idx)
    with pytest.raises(ValueError, match=r"\[N, h, w, 3\]"):
        net.forward_bgr_u8_indexed(pool[0], idx)
    with pytest.raises(ValueError, match="contiguous"):
        net.forward_bgr_u8_indexed(torch.zeros(5, 10, 8, 3, dtype=torch.uint8).transpose(1, 2).as_subclass(_ClaimsCuda), idx)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        net.forward_bgr_u8_indexed(torch.zeros(5, 8, 10, 3, dtype=torch.uint8), idx)
    with pytest.raises(ValueError, match=r"\[b, 7\]"):
        net.forward_bgr_u8_indexed(pool, [[0, 1, 2, 3, 4, 4]])
    with pytest.raises(TypeError, match="integer"):
        net.forward_bgr_u8_indexed(pool, torch.zeros(1, 7))
    with pytest.raises(IndexError, match="5 frames"):
        net.forward_bgr_u8_indexed(pool, [[0, 1, 2, 3, 4, 5, 4]])
    with pytest.raises(IndexError, match="-1"):
        net.forward_bgr_u8_indexed(pool, torch.tensor([[0, 1, 2, -1, 4, 4, 4]]))
    y = net.forward_bgr_u8_indexed(pool, torch.zeros(0, 7, dtype=torch.int32), scale=(2.7, 4))
    H, W = engine.get_hw(8, 10, (2.7, 4))
    assert tuple(y.shape) == (0, H, W, 3) and y.dtype == torch.uint8 and not net._plans
    assert tuple(net.forward_bgr_u8_indexed(pool, []).shape) == (0, H, W, 3)
    net.train()
    with pytest.raises(RuntimeError, match="inference only"):
        net.forward_bgr_u8_indexed(pool, idx)


def _frame_id(frames: torch.Tensor) -> torch.Tensor:
    """The frame number the test clips carry in pixel (0, 0), channels 0 and 1."""
    return frames[..., 0, 0, 0].long() + 256 * frames[..., 0, 0, 1].long()


def _u8_net(x):
    """Stand-in for forward_bgr_u8: uint8 [n,7,h,w,3] -> uint8 [n,2h,2w,3], a function of every frame of the window."""
    c = x[:, 3].repeat_interleave(2, 1).repeat_interleave(2, 2)
    return (c.int() + x.int().sum(1).repeat_interleave(2, 1).repeat_interleave(2, 2) * 7).to(torch.uint8)


class StandIn:
    """CPU stand-in for a SAVSR in eval mode: records the windows (as frame numbers) and the scale of every forward."""
    training = False

    def __init__(self):
        self.gamma = torch.zeros(1)
        self.windows, self.scales = [], []

    def _forward_bgr_u8_indexed(self, pool, windows, scale):
        x = pool[torch.as_tensor(windows)]               # read at call time: a slot rewritten too early shows here
        self.windows.append(_frame_id(x).tolist())
        self.scales.append(scale)
        return _u8_net(x)


def _clip(T, h=6, w=8, seed=0):
    clip = torch.randint(0, 256, (T, h, w, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(seed))
    clip[:, 0, 0, 0] = torch.arange(T) % 256
    clip[:, 0, 0, 1] = torch.arange(T) // 256
    return clip


def _clip_reference(clip, batch):
    """What infer_clip does on the whole clip: the windows of every forward, in order, and the frames it returns."""
    seen = []

    def net(x):
        seen.append(_frame_id(x).tolist())
        return _u8_net(x)
    return seen, sharding.infer_clip(net, clip, batch=batch)


def _stream(up, clip, chunks):
    outs, k = [], 0
    for n in chunks:
        outs += up.push(clip[k:k + n])
        k += n
    assert k == clip.shape[0]
    outs += up.finish()
    return outs


def _chunkings(T, rng):
    yield [1] * T
    sizes = []
    while sum(sizes) < T:
        sizes.append(min(rng.choice([1, 2, 3, 5, 9, 17, 40]), T - sum(sizes)))
    yield sizes


@pytest.mark.parametrize("batch", [17, (26, 8)])
@pytest.mark.parametrize("T", [4, 5, 7, 8, 13, 34, 35, 100])
def test_stream_matches_infer_clip(T, batch):
    clip = _clip(T, seed=T)
    want_windows, want = _clip_reference(clip, batch)
    assert [len(w) for w in want_windows] == [j - i for i, j in sharding.batch_schedule(T, batch)]
    rng = random.Random(T)
    for chunks in _chunkings(T, rng):
        net = StandIn()
        up = VideoUpscaler(net, (6, 8), (2, 2), batch=batch)
        outs = _stream(up, clip, chunks)
        assert net.windows == want_windows                              # the same windows, in the same batch partition
        assert [s for s, _ in outs] == [i for i, _ in sharding.batch_schedule(T, batch)]
        assert torch.equal(torch.cat([y for _, y in outs]), want)
        assert up.capacity == max([batch] if isinstance(batch, int) else batch) + 6 and up.ring.shape[0] == up.capacity


def test_batches_run_as_soon_as_their_last_frame_arrives():
    net = StandIn()
    up = VideoUpscaler(net, (6, 8), (2, 2), batch=(5, 3))
    clip = _clip(20)
    ready = {k: [s for s, _ in up.push(clip[k])] for k in range(20)}
    assert {k: v for k, v in ready.items() if v} == {7: [0], 10: [5], 13: [8], 16: [11], 19: [14]}   # batch [i, j) after frame j + 2
    assert [s for s, _ in up.finish()] == [17]


def test_ring_capacity_does_not_depend_on_the_length():
    caps = set()
    for T in (8, 100, 1000):
        up = VideoUpscaler(StandIn(), (6, 8), (2, 2), batch=(26, 8))
        _stream(up, _clip(T), [1] * T)
        caps.add(tuple(up.ring.shape))
    assert caps == {(32, 6, 8, 3)}


def test_reset_reuses_the_ring_and_a_later_set_scale_does_not_reach_the_stream():
    net = StandIn()
    up = VideoUpscaler(net, (6, 8), (4, 3), batch=4)
    ring = up.ring
    a, b = _clip(9, seed=1), _clip(12, seed=2)
    for clip in (a, b):
        _, want = _clip_reference(clip, 4)
        assert torch.equal(torch.cat([y for _, y in _stream(up, clip, [1] * clip.shape[0])]), want)
        up.reset()
    assert up.ring is ring and set(net.scales) == {(4.0, 3.0)}


def test_refusals():
    net = StandIn()
    up = VideoUpscaler(net, (6, 8), (2, 2), batch=4)
    for T in (0, 1, 2, 3):
        up.reset()
        for k in range(T):
            assert up.push(_clip(T)[k]) == []
        with pytest.raises(ValueError, match="too short"):
            up.finish()
    up.reset()
    with pytest.raises(ValueError, match=r"\[6, 8, 3\]"):
        up.push(torch.zeros(6, 9, 3, dtype=torch.uint8))
    with pytest.raises(ValueError, match=r"\[6, 8, 3\]"):
        up.push(torch.zeros(2, 6, 8, 4, dtype=torch.uint8))
    with pytest.raises(TypeError, match="uint8"):
        up.push(torch.zeros(6, 8, 3))
    up.push(np.zeros((4, 6, 8, 3), dtype=np.uint8))       # numpy frames from a decoder are taken as they are
    up.finish()
    with pytest.raises(RuntimeError, match="after finish"):
        up.push(_clip(1)[0])
    with pytest.raises(RuntimeError, match="already called"):
        up.finish()
    up.reset()
    net.training = True
    with pytest.raises(RuntimeError, match="train mode"):
        up.push(_clip(1)[0])
    with pytest.raises(RuntimeError, match="inference only"):
        VideoUpscaler(net, (6, 8), (2, 2))
    net.training = False
    with pytest.raises(ValueError, match="positive"):
        VideoUpscaler(net, (6, 8), (2, 2), batch=(4, 0))


# ------------------------------------------------------------------------------------------------ GPU

DEV = torch.device("cuda", 0)


def _gpu_net(precision="bf16", graph=True, seed=0):
    import savsr_b200
    net = savsr_b200.SAVSR().to(DEV).eval()
    net.load_state_dict(make_state_dict(seed), strict=True)
    net.precision, net.use_graph = precision, graph
    return net


def _pool(n, h, w, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, generator=g).to(DEV)


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
def test_forward_bgr_u8_indexed_is_forward_bgr_u8_of_the_gathered_windows(b, h, w, scale, precision, graph):
    net = _gpu_net(precision, graph)
    net.set_scale(scale)
    pool = _pool(11, h, w, seed=b * 100 + h + int(10 * scale[0]))
    rng = np.random.default_rng(b + h)
    windows = [list(range(3, 10)), list(range(9, 2, -1)), [5] * 7, [0, 10, 2, 7, 7, 1, 4]][:b]   # in order, reversed, repeated, scattered
    if b == 1:
        windows = [rng.integers(0, 11, 7).tolist()]
    idx = torch.tensor(windows)
    with torch.no_grad():
        want = net.forward_bgr_u8(pool[idx.to(DEV)])
        got = net.forward_bgr_u8_indexed(pool, idx)
        again = net.forward_bgr_u8_indexed(pool, windows)            # a second call replays the cached plan, host list this time
    assert got.dtype == torch.uint8 and tuple(got.shape) == (b, *engine.get_hw(h, w, scale), 3)
    assert torch.equal(got, want), int((got.int() - want.int()).abs().max())
    assert torch.equal(again, want)


@pytest.mark.gpu
def test_forward_u8_frames_c_and_mismatched_calls():
    import ctypes as C
    net = _gpu_net()
    net.set_scale((1.5, 4))
    pool = _pool(9, 37, 45, seed=5)
    idx = torch.tensor([[0, 1, 2, 3, 4, 5, 6], [8, 8, 7, 3, 2, 0, 1]])
    xu8 = pool[idx.to(DEV)].contiguous()
    with torch.no_grad():
        want = net.forward_bgr_u8(xu8)
        p8 = net.plan_for(xu8, io="bgr_u8")
        pf = net._plan(2, 37, 45, DEV, "bgr_u8_frames", net.scale)
        assert p8.cplan is not None and pf.cplan is not None
        ptrs = (idx.reshape(-1) * (37 * 45 * 3) + pool.data_ptr()).tolist()
        out8, outf = torch.zeros_like(want), torch.zeros_like(want)
        p8.forward_c(xu8, out8)                           # savsr_forward_u8
        pf.forward_frames_c(ptrs, outf)                   # savsr_forward_u8_frames
        torch.cuda.synchronize()
        assert torch.equal(out8, want) and torch.equal(outf, want)
        lib, st = pf.lib, torch.cuda.current_stream().cuda_stream
        arr = (C.c_void_p * len(ptrs))(*ptrs)
        outf.zero_()
        assert lib.savsr_forward_u8(pf.cplan.handle, xu8.data_ptr(), outf.data_ptr(), st) != 0
        assert b"savsr_forward_u8_frames" in lib.savsr_last_error()
        assert lib.savsr_forward(pf.cplan.handle, xu8.data_ptr(), outf.data_ptr(), st) != 0
        assert lib.savsr_forward_u8_frames(p8.cplan.handle, arr, outf.data_ptr(), st) != 0
        assert b"savsr_forward_u8" in lib.savsr_last_error()
        bad = (C.c_void_p * len(ptrs))(*ptrs[:-1], None)
        assert lib.savsr_forward_u8_frames(pf.cplan.handle, bad, outf.data_ptr(), st) != 0
        assert b"null" in lib.savsr_last_error()
        torch.cuda.synchronize()
        assert int(outf.count_nonzero()) == 0             # the refused calls copied and launched nothing
        # more than one writer launch: 64 windows = 448 pointers fill one launch exactly, 65 need two
        for b in (64, 65):
            many = torch.arange(b * 7).reshape(b, 7) % 9
            assert torch.equal(net.forward_bgr_u8_indexed(pool, many), net.forward_bgr_u8(pool[many.to(DEV)]))


def _reference_clip(net, clip, batch):
    with torch.no_grad():
        return sharding.infer_clip(net.forward_bgr_u8, clip.to(DEV), batch=batch)


@pytest.mark.gpu
@pytest.mark.parametrize("T", [4, 7, 34, 35])
def test_video_upscaler_equals_infer_clip(T):
    import savsr_b200
    net = _gpu_net()
    h, w, batch = 36, 44, (26, 8)
    clip = torch.randint(0, 256, (T, h, w, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(T))
    net.set_scale((4, 4))
    want = _reference_clip(net, clip, batch)
    net.set_scale((2, 2))                                     # the stream keeps the scale it was built with
    up = savsr_b200.VideoUpscaler(net, (h, w), (4, 4), batch=batch)
    pinned = clip.pin_memory()
    feeds = {
        "pageable": lambda k: clip[k],
        "pinned": lambda k: pinned[k],
        "cuda_chunks": None,
    }
    with torch.no_grad():
        for name, feed in feeds.items():
            up.reset()
            outs = []
            if feed is None:
                dev_clip = clip.to(DEV)
                for k in range(0, T, 5):
                    outs += up.push(dev_clip[k:k + 5])
            else:
                buf = torch.empty(h, w, 3, dtype=torch.uint8)
                for k in range(T):
                    buf.copy_(feed(k))
                    outs += up.push(buf)
                    buf.fill_(255 - k % 256)                  # the caller overwrites its buffer right after push
            outs += up.finish()
            got = torch.cat([y for _, y in outs])
            assert [s for s, _ in outs] == [i for i, _ in sharding.batch_schedule(T, batch)], name
            assert torch.equal(got, want), name
    assert net.scale == (2, 2)


@pytest.mark.gpu
def test_video_upscaler_memory_does_not_grow_with_the_length():
    import savsr_b200
    net = _gpu_net()
    h, w = 24, 32
    up = savsr_b200.VideoUpscaler(net, (h, w), (2, 2), batch=4)
    gen = torch.Generator().manual_seed(4)
    frames = torch.randint(0, 256, (8, h, w, 3), dtype=torch.uint8, generator=gen)

    def run(T):
        up.reset()
        for k in range(T):
            for _, hr in up.push(frames[k % 8]):
                del hr
        for _, hr in up.finish():
            del hr
        torch.cuda.synchronize()

    with torch.no_grad():
        run(100)                                           # builds the plan and the ring's staging buffers
        torch.cuda.reset_peak_memory_stats(DEV)
        run(100)
        peak100 = torch.cuda.max_memory_allocated(DEV)
        torch.cuda.reset_peak_memory_stats(DEV)
        run(400)
        peak400 = torch.cuda.max_memory_allocated(DEV)
    assert peak400 <= peak100, (peak100, peak400)
