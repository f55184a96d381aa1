"""8-bit video I/O (SAVSR.forward_bgr_u8, engine.Plan(io="bgr_u8"), savsr_forward_u8).

CPU: the plan's launch list and staging buffers against the recording fake library, the plan cache, input validation, the u / 255
conversion the kernels use, and the clip driver carrying uint8 frames over two gloo ranks.
GPU: the contract, bit for bit:  forward_bgr_u8(xu8) == tensor2img(forward(xf)),  xf[n,f,c,y,x] = float32(xu8[n,f,y,x,2-c]) / 255
correctly rounded (the reference's img.astype(np.float32) / 255.).
"""
import os
from fractions import Fraction
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from fake_lib import CpuPlan, mocked_engine
from oracle.state_dict_fixture import make_state_dict
from savsr_b200 import engine, sharding

UNIT = np.arange(256, dtype=np.float32) / np.float32(255)      # the reference's conversion of every 8-bit value


def to_f32_windows(xu8: torch.Tensor) -> torch.Tensor:
    """uint8 [b,7,h,w,3] BGR -> fp32 [b,7,3,h,w] RGB through the 256-entry table (an exact gather, no division on the device)."""
    table = torch.from_numpy(UNIT).to(xu8.device)
    return table[xu8.long()].flip(-1).permute(0, 1, 4, 2, 3).contiguous()


# ------------------------------------------------------------------------------------------------ CPU

class CpuPlanU8(CpuPlan):
    io = "bgr_u8"


def _record(cls, sd, b=2, h=13, w=15, scale=(1.5, 4)):
    with mocked_engine() as lib:
        plan = cls(sd, b, h, w, scale)
        for op in plan.ops:
            assert op(0) == 0
        return plan, list(lib.calls)


@pytest.fixture(scope="module")
def sd():
    return make_state_dict(0)


def test_u8_plan_swaps_only_the_first_and_last_launch(sd):
    p32, c32 = _record(CpuPlan, sd)
    p8, c8 = _record(CpuPlanU8, sd)
    n32, n8 = [c[0] for c in c32], [c[0] for c in c8]
    assert len(n32) == len(n8) and len(p32.ops) == len(p8.ops) and p32.n_launches == p8.n_launches
    diff = [(a, b) for a, b in zip(n32, n8) if a != b]
    assert diff == [("savsr_pack_frames", "savsr_pack_frames_u8"), ("savsr_satu_hr", "savsr_satu_hr_u8")]
    assert "savsr_pack_frames" not in n8 and "savsr_satu_hr" not in n8
    for a, b in zip(c32, c8):                         # same launches with the same scalar arguments in between
        assert len(a[1]) == len(b[1])
        assert [v for v in a[1] if isinstance(v, (float, str))] == [v for v in b[1] if isinstance(v, (float, str))]
    pack = next(args for name, args in c8 if name == "savsr_pack_frames_u8")
    hr = next(args for name, args in c8 if name == "savsr_satu_hr_u8")
    assert pack[2] == p8.x_in.data_ptr() and pack[3:7] == (7, 13, 15, 1)
    assert hr[14] == p8.x_in.data_ptr() and hr[17] == p8.out.data_ptr()
    assert [m[0] for m in p32.op_meta] == [m[0] for m in p8.op_meta]


def test_u8_staging_buffers(sd):
    p8, _ = _record(CpuPlanU8, sd, b=3, h=13, w=15, scale=(2.7, 2.7))
    assert p8.x_in.dtype == torch.uint8 and tuple(p8.x_in.shape) == (3, 7, 13, 15, 3)
    assert p8.out.dtype == torch.uint8 and tuple(p8.out.shape) == (3, 35, 40, 3)
    p32, _ = _record(CpuPlan, sd, b=3, h=13, w=15, scale=(2.7, 2.7))
    assert p32.x_in.dtype == torch.float32 and tuple(p32.x_in.shape) == (3, 7, 3, 13, 15)
    assert tuple(p32.out.shape) == (3, 3, 35, 40)
    with pytest.raises(ValueError, match="io must be one of"):
        engine.Plan(sd, 1, 8, 8, 2, torch.device("cuda", 0), io="rgb_u8")


class _ClaimsCuda(torch.Tensor):
    """A CPU tensor that reports is_cuda, so the module's host logic runs without a device (nothing is launched)."""
    is_cuda = property(lambda self: True)


def _cpu_net():
    import savsr_b200
    net = savsr_b200.SAVSR().eval()
    net.load_state_dict(make_state_dict(0), strict=True)
    net.set_scale((2, 2))
    return net


def test_plan_cache_keys_the_io_mode_and_shares_weights(monkeypatch):
    net = _cpu_net()
    built = []

    def fake_plan(params, b, h, w, s, device, io="f32", **kw):
        built.append(io)
        cls = CpuPlanU8 if io == "bgr_u8" else CpuPlan
        return cls(params, b, h, w, s, **kw)
    from savsr_b200.archs import savsr_arch
    with mocked_engine():
        monkeypatch.setattr(savsr_arch, "engine", SimpleNamespace(**{**vars(engine), "Plan": fake_plan}))
        x32 = torch.zeros(1, 7, 3, 8, 10).as_subclass(_ClaimsCuda)
        x8 = torch.zeros(1, 7, 8, 10, 3, dtype=torch.uint8).as_subclass(_ClaimsCuda)
        a, b = net.plan_for(x32), net.plan_for(x8, io="bgr_u8")
        assert built == ["f32", "bgr_u8"] and a is not b
        assert a.io == "f32" and b.io == "bgr_u8" and a.store is b.store
        assert net.plan_for(x8, io="bgr_u8") is b and net.plan_for(x32) is a and len(built) == 2
        assert sorted(k[9] for k in net._plans) == ["bgr_u8", "f32"]


def test_forward_bgr_u8_validates_its_input():
    net = _cpu_net()
    good = torch.zeros(1, 7, 8, 10, 3, dtype=torch.uint8)
    with pytest.raises(TypeError, match="uint8"):
        net.forward_bgr_u8(good.float())
    with pytest.raises(ValueError, match=r"\[b, 7, h, w, 3\]"):
        net.forward_bgr_u8(torch.zeros(1, 7, 3, 8, 10, dtype=torch.uint8))          # the fp32 forward's layout
    with pytest.raises(ValueError):
        net.forward_bgr_u8(torch.zeros(7, 8, 10, 3, dtype=torch.uint8))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        net.forward_bgr_u8(good)
    net.train()
    with pytest.raises(RuntimeError, match="inference only"):
        net.forward_bgr_u8(good.as_subclass(_ClaimsCuda))


def test_forward_bgr_u8_empty_batch():
    net = _cpu_net()
    y = net.forward_bgr_u8(torch.zeros(0, 7, 9, 10, 3, dtype=torch.uint8).as_subclass(_ClaimsCuda), scale=(2.7, 4))
    assert tuple(y.shape) == (0, 24, 40, 3) and y.dtype == torch.uint8 and not net._plans


def _rn32(q: Fraction) -> np.float32:
    return np.float32(float(q))      # Fraction -> float64 is correctly rounded; no value below sits on a float32 tie


def test_u8_to_unit_is_the_correctly_rounded_quotient():
    """The kernels' u8_to_unit (common.cuh): q = u * RN(1/255), then q + fma(-q, 255, u) * RN(1/255), each step rounded once.
    Emulated here in exact arithmetic for all 256 values against numpy's float32 division."""
    r = np.float32(1) / np.float32(255)
    plain_wrong = 0
    for u in range(256):
        q = np.float32(np.float32(u) * r)
        plain_wrong += int(q != UNIT[u])
        rem = _rn32(Fraction(u) - Fraction(float(q)) * 255)
        assert Fraction(float(rem)) == Fraction(u) - Fraction(float(q)) * 255          # the remainder is exact
        got = _rn32(Fraction(float(rem)) * Fraction(float(r)) + Fraction(float(q)))
        assert got == UNIT[u], (u, got, UNIT[u])
    assert plain_wrong > 0                       # so the correction step is needed


def _u8_net(x):
    """Stand-in for forward_bgr_u8: uint8 [n,7,h,w,3] -> uint8 [n,2h,2w,3], a function of the centre frame and the window's frames."""
    c = x[:, 3].repeat_interleave(2, 1).repeat_interleave(2, 2)
    return (c.int() + x[:, 0, :1, :1].int() * 3).to(torch.uint8)


def test_infer_clip_carries_uint8_frames():
    clip = torch.randint(0, 256, (11, 6, 8, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(3))
    full = sharding.infer_clip(_u8_net, clip, batch=11)
    assert full.dtype == torch.uint8 and tuple(full.shape) == (11, 12, 16, 3)
    for b in (1, 4, (7, 3)):
        assert torch.equal(sharding.infer_clip(_u8_net, clip, batch=b), full)
    out = torch.empty(11, 12, 16, 3, dtype=torch.uint8)
    assert sharding.infer_clip(_u8_net, clip, batch=(8, 2), out=out) is out and torch.equal(out, full)


def _worker(rank, world, port, n_frames, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        clip = torch.randint(0, 256, (n_frames, 6, 8, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(7))
        ref = sharding.infer_clip(_u8_net, clip, batch=3)
        ok = True
        for contiguous in (False, True):
            mine = sharding.shard_frames(n_frames, rank, world, contiguous)
            local = sharding.infer_clip(_u8_net, clip, frames=mine, batch=2) if mine else torch.empty(0, 12, 16, 3, dtype=torch.uint8)
            full = sharding.gather_outputs(local, n_frames, rank, world, dst=0, contiguous=contiguous)
            ok &= (full is None) if rank != 0 else bool(full.dtype == torch.uint8 and torch.equal(full, ref))
            work, finish = sharding.gather_outputs(local, n_frames, rank, world, dst=None, contiguous=contiguous, async_op=True)
            work.wait()
            got = finish()
            ok &= bool(got.dtype == torch.uint8 and torch.equal(got, ref))
        ret[rank] = ok
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("n_frames", [5, 8])
def test_two_rank_uint8_frames(n_frames):
    world = 2
    ret = mp.Manager().dict()
    port = 31500 + (os.getpid() % 2000) + n_frames
    mp.spawn(_worker, args=(world, port, n_frames, ret), nprocs=world, join=True)
    assert dict(ret) == {0: True, 1: True}


# ------------------------------------------------------------------------------------------------ GPU

DEV = torch.device("cuda", 0)


def _gpu_net(precision="bf16", graph=True, seed=0):
    import savsr_b200
    net = savsr_b200.SAVSR().to(DEV).eval()
    net.load_state_dict(make_state_dict(seed), strict=True)
    net.precision, net.use_graph = precision, graph
    return net


def _windows(b, h, w, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 256, (b, 7, h, w, 3), dtype=torch.uint8, generator=g).to(DEV)


def _reference(net, xu8):
    from savsr_b200 import postproc
    img, _ = postproc.tensor2img_psnr(net(to_f32_windows(xu8)))
    return img


@pytest.mark.gpu
@pytest.mark.parametrize("b,h,w,scale,precision,graph", [
    (2, 144, 180, (4, 4), "bf16", True),         # Vid4 at x4
    (2, 144, 180, (1.5, 4), "fp16", True),
    (2, 144, 180, (2.7, 2.7), "bf16", False),    # W = 486: W * 3 = 1458 is not a multiple of 4
    (2, 144, 180, (2.7, 2.7), "fp16", False),
    (2, 179, 317, (4, 4), "bf16", False),        # odd size: pad_spatial
    (2, 179, 317, (4, 4), "fp16", True),
    (1, 144, 180, (4, 4), "bf16", False),
    (1, 144, 180, (1.5, 4), "fp16", True),
])
def test_forward_bgr_u8_is_tensor2img_of_forward(b, h, w, scale, precision, graph):
    net = _gpu_net(precision, graph)
    net.set_scale(scale)
    xu8 = _windows(b, h, w, seed=b * 1000 + h + int(10 * scale[0]))
    with torch.no_grad():
        got = net.forward_bgr_u8(xu8)
        want = _reference(net, xu8)
        again = net.forward_bgr_u8(xu8)                  # a second call replays the cached plan (graph or eager)
    H, W = engine.get_hw(h, w, scale)
    assert got.dtype == torch.uint8 and tuple(got.shape) == (b, H, W, 3)
    assert torch.equal(got, want), int((got.int() - want.int()).abs().max())
    assert torch.equal(again, got)
    assert tuple(net.forward_bgr_u8(xu8[:0]).shape) == (0, H, W, 3)


@pytest.mark.gpu
def test_forward_c_u8_and_mismatched_calls():
    from savsr_b200 import _capi as K
    net = _gpu_net()
    net.set_scale((1.5, 4))
    xu8 = _windows(2, 37, 45, seed=5)
    with torch.no_grad():
        want = net.forward_bgr_u8(xu8)
        p8 = net.plan_for(xu8, io="bgr_u8")
        p32 = net.plan_for(to_f32_windows(xu8))
        assert p8.cplan is not None and p32.cplan is not None
        out = torch.zeros_like(want)
        p8.forward_c(xu8.contiguous(), out)              # one C call: savsr_forward_u8
        torch.cuda.synchronize()
        assert torch.equal(out, want)
        with pytest.raises(ValueError, match="uint8"):
            p8.forward_c(to_f32_windows(xu8), torch.empty(p32.out.shape, device=DEV))
        lib, st = p8.lib, torch.cuda.current_stream().cuda_stream
        out.zero_()
        assert lib.savsr_forward(p8.cplan.handle, xu8.data_ptr(), out.data_ptr(), st) != 0
        assert b"savsr_forward_u8" in lib.savsr_last_error()
        x32, y32 = to_f32_windows(xu8), torch.empty(p32.out.shape, device=DEV)
        assert lib.savsr_forward_u8(p32.cplan.handle, x32.data_ptr(), y32.data_ptr(), st) != 0
        assert b"fp32" in lib.savsr_last_error()
        torch.cuda.synchronize()
        assert int(out.count_nonzero()) == 0             # the refused call copied and launched nothing


@pytest.mark.gpu
def test_infer_clip_u8_into_pinned_host_buffer():
    from savsr_b200 import postproc
    net = _gpu_net()
    net.set_scale((4, 4))
    T, h, w = 34, 144, 180
    clip = torch.randint(0, 256, (T, h, w, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(9)).pin_memory()
    out = torch.empty(T, 4 * h, 4 * w, 3, dtype=torch.uint8).pin_memory()
    with torch.no_grad():
        dev_clip = clip.to(DEV, non_blocking=True)
        res = sharding.infer_clip(net.forward_bgr_u8, dev_clip, batch=(26, 8), out=out)
        torch.cuda.synchronize()
        assert res is out
        clip32 = to_f32_windows(dev_clip.unsqueeze(0))[0]                     # [T, 3, h, w]
        want = sharding.infer_clip(lambda x: postproc.tensor2img_psnr(net(x))[0], clip32, batch=(26, 8))
    assert torch.equal(out, want.cpu())


@pytest.mark.gpu
def test_u8_and_f32_plans_of_one_shape_alternate():
    from savsr_b200 import postproc
    net = _gpu_net()
    net.set_scale((2, 2))
    xa, xb = _windows(2, 40, 52, seed=11), _windows(2, 40, 52, seed=12)
    with torch.no_grad():
        ref32 = {k: net(to_f32_windows(x)).clone() for k, x in (("a", xa), ("b", xb))}
        ref8 = {k: postproc.tensor2img_psnr(v)[0] for k, v in ref32.items()}
        for k, x in (("a", xa), ("b", xb), ("a", xa), ("b", xb)):
            assert torch.equal(net.forward_bgr_u8(x), ref8[k])
            assert torch.equal(net(to_f32_windows(x)), ref32[k])
    assert sorted(key[9] for key in net._plans) == ["bgr_u8", "f32"]
    stores = {id(p.store) for p in net._plans.values()}
    assert len(stores) == 1
