"""NativeTrainer under the reference's training recipe: learning-rate schedules (also under CUDA-graph replay), Adam state in
torch.optim.Adam's state_dict layout (save / resume, and moving between the module path's torch.optim.Adam and the native step in both
directions), and the EMA network as a full 791-key state_dict.  CPU: host logic against the recording fake of the C library.
GPU: the device-lr Adam kernel, graph replay following the lr, resume and interop against uninterrupted runs."""
import contextlib
import copy
import io
import math
import re
import warnings

import pytest
import torch

from fake_lib import mocked_engine


# ---------------------------------------------------------------------------------------------------- the reference's schedule
class CosineAnnealingRestartLR(torch.optim.lr_scheduler._LRScheduler):
    """BasicSR's cosine annealing with restarts (basicsr/models/lr_scheduler.py), as the reference's train YAML uses it."""

    def __init__(self, optimizer, periods, restart_weights=(1,), eta_min=0, last_epoch=-1):
        self.periods, self.restart_weights, self.eta_min = list(periods), list(restart_weights), eta_min
        self.cumulative_period = [sum(self.periods[0:i + 1]) for i in range(len(self.periods))]
        super().__init__(optimizer, last_epoch)

    def get_lr(self):
        idx = next(i for i, p in enumerate(self.cumulative_period) if self.last_epoch <= p)
        weight = self.restart_weights[idx]
        restart = 0 if idx == 0 else self.cumulative_period[idx - 1]
        period = self.periods[idx]
        return [self.eta_min + weight * 0.5 * (base - self.eta_min) * (1 + math.cos(math.pi * ((self.last_epoch - restart) / period)))
                for base in self.base_lrs]


def update_learning_rate(optimizer, schedulers, current_iter, warmup_iter=-1):
    """BasicSR's BaseModel.update_learning_rate: scheduler steps from the second iteration on, linear warm-up written into the groups."""
    if current_iter > 1:
        for s in schedulers:
            s.step()
    if current_iter < warmup_iter:
        for g in optimizer.param_groups:
            g["lr"] = g["initial_lr"] / warmup_iter * current_iter


# ---------------------------------------------------------------------------------------------------- CPU: recording fake library
@contextlib.contextmanager
def mocked_trainer():
    """The fake library plus what NativeTrainer needs to build on CPU tensors (as in test_trainplan_host_logic.py)."""
    from savsr_b200 import trainplan as TP
    import savsr_b200.autograd as A
    import torch.nn.functional as F
    with mocked_engine() as lib:
        saved = (TP.context, TP._require_cuda, A.sta_lrelu)
        TP.context = lambda idx: __import__("savsr_b200.engine", fromlist=["context"]).context(idx)
        TP._require_cuda = lambda dev: None

        def sta_lrelu_torch(x, kpre, slope=0.1):
            b, c, h, w = x.shape
            kern = F.leaky_relu(kpre, slope).view(b, c, 25, h * w)
            return (F.unfold(F.pad(x, (2, 2, 2, 2), mode="replicate"), 5).view(b, c, 25, h * w) * kern).sum(2).view(b, c, h, w)
        A.sta_lrelu = sta_lrelu_torch
        try:
            yield lib
        finally:
            TP.context, TP._require_cuda, A.sta_lrelu = saved


def _net(seed=0):
    import savsr_b200
    torch.manual_seed(seed)
    return savsr_b200.SAVSR()


def _torch_adam_state(net, steps=1, seed=1):
    """torch.optim.Adam(lr 2e-4, betas 0.9 / 0.99) after `steps` steps on random gradients: (optimizer, state_dict)."""
    opt = torch.optim.Adam(net.parameters(), lr=2e-4, betas=(0.9, 0.99))
    g = torch.Generator().manual_seed(seed)
    for _ in range(steps):
        for p in net.parameters():
            p.grad = torch.randn(p.shape, generator=g) * 1e-3
        opt.step()
    return opt, opt.state_dict()


def test_state_dict_has_torch_adams_format():
    from savsr_b200 import trainplan as TP
    net, ref_net = _net(), _net()
    _, ref = _torch_adam_state(ref_net, steps=1)
    with mocked_trainer():
        tr = TP.NativeTrainer(net, lr=2e-4, betas=(0.9, 0.99), use_graph=False)
        assert tr.optimizer.state_dict()["state"] == {}                 # like torch.optim.Adam before its first step
        tr.optimizer.step()
    sd = tr.optimizer.state_dict()
    assert len(sd["param_groups"]) == 1 and len(ref["param_groups"]) == 1
    g, rg = sd["param_groups"][0], ref["param_groups"][0]
    assert list(g) == list(rg)
    assert g["params"] == rg["params"] == list(range(707))
    assert {k: v for k, v in g.items() if k != "params"} == {k: v for k, v in rg.items() if k != "params"}
    assert list(sd["state"]) == list(ref["state"])
    for i, rs in ref["state"].items():
        s = sd["state"][i]
        assert list(s) == list(rs) == ["step", "exp_avg", "exp_avg_sq"]
        for k in s:
            assert s[k].shape == rs[k].shape and s[k].dtype == rs[k].dtype, (i, k)
        assert float(s["step"]) == float(rs["step"]) == 1.0 and s["step"].device == rs["step"].device
    assert not tr.optimizer.state                                    # the per-parameter entries exist in the returned dict only


def test_torch_adam_state_round_trips_exactly():
    from savsr_b200 import trainplan as TP
    ref_net = _net()
    _, ref = _torch_adam_state(ref_net, steps=3)
    with mocked_trainer():
        tr = TP.NativeTrainer(_net(), use_graph=False)
        tr.optimizer.load_state_dict(ref)
    assert float(tr.flat.step_t) == 3.0 and tr.lr == 2e-4 and tr.betas == (0.9, 0.99)
    back = torch.optim.Adam(_net(2).parameters(), lr=1.0)
    back.load_state_dict(tr.optimizer.state_dict())
    out = back.state_dict()
    assert out["param_groups"][0]["lr"] == 2e-4
    for i, rs in ref["state"].items():
        s = out["state"][i]
        assert float(s["step"]) == float(rs["step"])
        assert torch.equal(s["exp_avg"], rs["exp_avg"]) and torch.equal(s["exp_avg_sq"], rs["exp_avg_sq"]), i


def _refusal_cases():
    def two_groups(sd):
        sd["param_groups"].append(dict(sd["param_groups"][0], params=[]))

    def fewer_params(sd):
        sd["param_groups"][0]["params"].pop()

    def wrong_shape(sd):
        sd["state"][5]["exp_avg"] = sd["state"][5]["exp_avg"].flatten()[:3].clone()

    def uneven_steps(sd):
        sd["state"][7]["step"] = torch.tensor(9.0)

    def weight_decay(sd):
        sd["param_groups"][0]["weight_decay"] = 1e-4

    def amsgrad(sd):
        sd["param_groups"][0]["amsgrad"] = True

    def maximize(sd):
        sd["param_groups"][0]["maximize"] = True
    return [two_groups, fewer_params, wrong_shape, uneven_steps, weight_decay, amsgrad, maximize]


@pytest.fixture(scope="module")
def adam_state():
    return _torch_adam_state(_net(), steps=2)[1]


@pytest.mark.parametrize("mutate", _refusal_cases(), ids=lambda f: f.__name__)
def test_load_state_dict_refuses_what_the_kernel_cannot_continue(adam_state, mutate):
    from savsr_b200 import trainplan as TP
    sd = copy.deepcopy(adam_state)
    mutate(sd)
    with mocked_trainer():
        tr = TP.NativeTrainer(_net(), use_graph=False)
        with pytest.raises(ValueError):
            tr.optimizer.load_state_dict(sd)


def test_ema_state_dict_is_the_full_network_state():
    import savsr_b200
    from savsr_b200 import trainplan as TP
    net = _net()
    keys = list(net.state_dict())
    assert len(keys) == 791
    with mocked_trainer():
        tr = TP.NativeTrainer(net, use_graph=False)
    sd = tr.ema_state_dict()
    assert list(sd) == keys
    for n in tr.flat.P:
        assert sd[n].data_ptr() == tr.flat.ema_view(n).data_ptr()
    fresh = savsr_b200.SAVSR()
    fresh.load_state_dict(sd, strict=True)
    # buffers: those of the network when the EMA was initialised, not the ones train-mode BatchNorm updates later (BasicSR's model_ema)
    rm = next(k for k in keys if k.endswith("running_mean"))
    before = sd[rm].clone()
    net.state_dict()[rm].add_(1.0)
    assert torch.equal(tr.ema_state_dict()[rm], before)
    # load_ema_state_dict: the reverse, strict
    other = _net(3).state_dict()
    tr.load_ema_state_dict(other)
    back = tr.ema_state_dict()
    assert all(torch.equal(back[k], other[k]) for k in keys)
    with pytest.raises(ValueError):
        tr.load_ema_state_dict({k: v for k, v in other.items() if k != rm})
    with pytest.raises(ValueError):
        tr.load_ema_state_dict(dict(other, extra=torch.zeros(1)))


def test_schedule_reaches_the_eager_launch():
    """Warm-up + BasicSR's cosine schedule on tr.optimizer; the lr of every savsr_adam_ema launch is the group's lr of that step, and
    torch's scheduler sees the optimizer step (no 'lr_scheduler.step() before optimizer.step()' warning)."""
    from savsr_b200 import trainplan as TP
    net = _net()
    with mocked_trainer() as lib:
        tr = TP.NativeTrainer(net, lr=2e-4, use_graph=False)
        sched = CosineAnnealingRestartLR(tr.optimizer, periods=[6], eta_min=1e-7)
        lq, gt = torch.rand(2, 7, 3, 16, 24), torch.rand(2, 3, 32, 48)
        tr.plan_for(lq, (2, 2))
        want, got = [], []
        with warnings.catch_warnings(record=True) as caught:
            warnings.simplefilter("always")
            for it in range(1, 7):
                update_learning_rate(tr.optimizer, [sched], it, warmup_iter=3)
                want.append(tr.optimizer.param_groups[0]["lr"])
                lib.calls.clear()
                tr.step(lq, gt, (2, 2))
                adam = [args for name, args in lib.calls if name == "savsr_adam_ema"]
                assert len(adam) == 1 and not any(name == "savsr_adam_ema_dev" for name, _ in lib.calls)
                got.append(adam[0][7])
    assert not [w for w in caught if "lr_scheduler.step()" in str(w.message)]
    assert got == want
    assert len(set(want)) == 6 and want[0] == pytest.approx(2e-4 / 3) and tr.lr == want[-1]
    assert float(tr.flat.step_t) == 6.0


def test_graph_mode_writes_the_device_lr_only_when_it_changes(monkeypatch):
    """With use_graph the optimizer launch is captured once (savsr_adam_ema_dev, reading the device lr); a constant lr writes nothing
    per step, a new lr one fill before the replay, new betas a new capture."""
    from savsr_b200 import trainplan as TP
    replays = []

    class FakeGraph:
        def replay(self):
            replays.append(self)
    monkeypatch.setattr(torch.cuda, "CUDAGraph", FakeGraph)
    monkeypatch.setattr(torch.cuda, "graph", lambda g, stream=None: contextlib.nullcontext())
    with mocked_trainer() as lib:
        tr = TP.NativeTrainer(_net(), lr=2e-4, use_graph=True)
        opt = tr.optimizer
        v0 = opt.lr_dev._version
        for _ in range(3):
            opt.step()
        names = [n for n, _ in lib.calls]
        assert names == ["savsr_adam_ema_dev"] and len(replays) == 3 and opt.lr_dev._version == v0
        assert lib.calls[0][1][7] == opt.lr_dev.data_ptr()
        tr.lr = 1e-4
        opt.step()
        opt.step()
        assert opt.lr_dev._version == v0 + 1 and float(opt.lr_dev) == pytest.approx(1e-4) and len(lib.calls) == 1
        opt.param_groups[0]["betas"] = (0.8, 0.99)
        opt.step()
        assert [n for n, _ in lib.calls] == ["savsr_adam_ema_dev"] * 2 and lib.calls[1][1][8] == pytest.approx(0.8)
        tr.use_graph = False
        opt.step()
        assert lib.calls[-1][0] == "savsr_adam_ema" and lib.calls[-1][1][7] == 1e-4


def test_training_state_and_resume_follow_basicsr():
    from savsr_b200 import trainplan as TP
    with mocked_trainer():
        tr = TP.NativeTrainer(_net(), use_graph=False)
        sched = CosineAnnealingRestartLR(tr.optimizer, periods=[10], eta_min=1e-7)
        for _ in range(2):
            tr.optimizer.step()
            sched.step()
        state = tr.training_state(iter=2, epoch=0, schedulers=[sched])
        assert set(state) == {"epoch", "iter", "optimizers", "schedulers"} and len(state["optimizers"]) == 1
        buf = io.BytesIO()
        torch.save(state, buf)
        buf.seek(0)
        state = torch.load(buf)
        tr2 = TP.NativeTrainer(_net(1), use_graph=False)
        sched2 = CosineAnnealingRestartLR(tr2.optimizer, periods=[10], eta_min=1e-7)
        assert tr2.resume(state, [sched2]) == (0, 2)
        with pytest.raises(ValueError):
            tr2.resume(state, [])
    assert float(tr2.flat.step_t) == 2.0 and tr2.lr == tr.lr and sched2.last_epoch == sched.last_epoch
    assert tr2.optimizer.param_groups[0]["initial_lr"] == 2e-4
    assert torch.equal(tr2.flat.m, tr.flat.m) and torch.equal(tr2.flat.v, tr.flat.v)


# ---------------------------------------------------------------------------------------------------- GPU (B200)
DEV = torch.device("cuda", 0)
SCALE = (2, 2)
B, H, W = 2, 16, 20


def _batch(i):
    g = torch.Generator().manual_seed(1000 + i)
    return torch.rand(B, 7, 3, H, W, generator=g).to(DEV), torch.rand(B, 3, 2 * H, 2 * W, generator=g).to(DEV)


def _gpu_net(sd=None):
    import savsr_b200
    torch.manual_seed(0)
    net = savsr_b200.SAVSR().to(DEV)
    if sd is not None:
        net.load_state_dict(sd, strict=True)
    net.train()
    return net


def _flat_params(net):
    return {n: p.detach().clone() for n, p in net.named_parameters()}


def _native_moments(tr):
    return {n: tr.flat.view(tr.flat.m, n).detach().clone() for n in tr.flat.P}


def _torch_moments(net, opt):
    return {n: opt.state[p]["exp_avg"].detach().clone() for n, p in net.named_parameters()}


# Parameters whose true gradient is zero or ill-conditioned at a batch of two (gpu_checks._grad_report): everything upstream of
# ScaleAttention's train-mode BatchNorm over a batch of two 1x1 maps, whose output is +-1 whatever its input (scale_routing, attention.fc),
# and the conv biases right in front of the mask net's train-mode BatchNorms.  Their per-tensor error compares rounding noise with rounding noise.
ILL_CONDITIONED = re.compile(r"\.scale_routing\.|\.attention\.fc\.weight$|\.mask\.(0|4|7|11)\.bias$")


def _rel(a, b, keys):
    """Cosine of the concatenated tensors and the worst per-tensor |a - b| / max(|b|, 1 % of the largest |b| tensor norm) with its name:
    the training parity measure of DESIGN section 9."""
    va = torch.cat([a[n].double().flatten() for n in keys])
    vb = torch.cat([b[n].double().flatten() for n in keys])
    cos = float(va @ vb / (va.norm() * vb.norm()))
    floor = 0.01 * max(float(b[n].double().norm()) for n in keys)
    worst = max((float((a[n].double() - b[n].double()).norm()) / max(float(b[n].double().norm()), floor), n) for n in keys)
    return cos, worst


def _assert_parity(params_a, params_b, m_a, m_b, base, what):
    """Two runs continued from the same saved state `base` (parameters at the split).  Weight gradients use fp32 atomics, so the runs
    are not bit-equal.  Asserted at the bounds of DESIGN section 9 (cosine >= 0.9999, worst tensor <= 5 %) over the well-conditioned
    tensors: the cosine of the parameter updates, and per tensor the Adam first moment (the running mean of the gradients each run saw
    along its own trajectory).  Reported only: the per-tensor error of the updates (Adam divides every element by its own gradient
    history, so an element whose gradient is at the noise level of the atomics moves by about +-lr in either run, whatever its sign)
    and everything about the ill-conditioned tensors."""
    keys = list(base)
    good = [n for n in keys if not ILL_CONDITIONED.search(n)]
    assert 0 < len(keys) - len(good) < 100, len(keys) - len(good)
    upd_a = {n: params_a[n] - base[n] for n in keys}
    upd_b = {n: params_b[n] - base[n] for n in keys}
    cos_u, worst_u = _rel(upd_a, upd_b, good)
    cos_m, worst_m = _rel(m_a, m_b, good)
    cos_all, worst_ill = _rel(m_a, m_b, keys)[0], _rel(m_a, m_b, [n for n in keys if n not in good])[1]
    print(f"{what}: well-conditioned tensors ({len(good)}): parameter updates cosine {cos_u:.7f}, worst tensor {100 * worst_u[0]:.2f} % "
          f"({worst_u[1]}); Adam first moment cosine {cos_m:.7f}, worst tensor {100 * worst_m[0]:.2f} % ({worst_m[1]}).  All tensors: "
          f"Adam first moment cosine {cos_all:.7f}; ill-conditioned worst {100 * worst_ill[0]:.1f} % ({worst_ill[1]})")
    assert cos_u >= 0.9999 and cos_m >= 0.9999 and worst_m[0] <= 0.05, (what, cos_u, cos_m, worst_m)


@pytest.mark.gpu
def test_adam_ema_dev_kernel_matches_host_lr_and_torch_adam():
    from savsr_b200 import _capi as K
    from savsr_b200.engine import context
    lib, ctx = K.load(), context(0)
    st = torch.cuda.current_stream(DEV).cuda_stream
    n = 100003
    g = torch.Generator().manual_seed(7)
    p0 = torch.randn(n, generator=g).to(DEV)
    host = [p0.clone(), torch.zeros(n, device=DEV), torch.zeros(n, device=DEV), p0.clone()]
    dev = [t.clone() for t in host]
    step_h, step_d = torch.zeros(1, device=DEV), torch.zeros(1, device=DEV)
    lr_dev = torch.zeros(1, device=DEV)
    rp = p0.clone().requires_grad_(True)
    opt = torch.optim.Adam([rp], lr=2e-4, betas=(0.9, 0.99), eps=1e-8)
    rema = p0.clone()
    lrs = [2e-4, 1.5e-4, 3e-4, 1e-5, 0.0, 7e-5]
    for lr in lrs:
        grad = torch.randn(n, generator=g).to(DEV) * 1e-3
        lr_dev.fill_(lr)
        step_h.add_(1.0)
        step_d.add_(1.0)
        K.check(lib.savsr_adam_ema(ctx.handle, *(t.data_ptr() for t in host[:1]), grad.data_ptr(), *(t.data_ptr() for t in host[1:]), n, lr,
                                   0.9, 0.99, 1e-8, step_h.data_ptr(), 0.999, 1.0, st))
        K.check(lib.savsr_adam_ema_dev(ctx.handle, *(t.data_ptr() for t in dev[:1]), grad.data_ptr(), *(t.data_ptr() for t in dev[1:]), n,
                                       lr_dev.data_ptr(), 0.9, 0.99, 1e-8, step_d.data_ptr(), 0.999, 1.0, st))
        opt.param_groups[0]["lr"] = lr
        rp.grad = grad.clone()
        opt.step()
        rema.mul_(0.999).add_(rp.detach(), alpha=0.001)
        torch.cuda.synchronize()
        for a, b in zip(host, dev):
            assert torch.equal(a, b), f"savsr_adam_ema_dev differs from savsr_adam_ema at lr {lr}"
    e_p = float((dev[0] - rp.detach()).abs().max())
    e_ema = float((dev[3] - rema).abs().max())
    print(f"6 steps, lr {lrs}: param max abs {e_p:.3e}, EMA max abs {e_ema:.3e}")
    assert e_p < 2e-6 and e_ema < 2e-6, (e_p, e_ema)


@pytest.mark.gpu
def test_graph_replay_follows_the_lr():
    from savsr_b200 import trainplan as TP
    tr = TP.NativeTrainer(_gpu_net(), use_graph=True)
    for i in range(2):
        tr.step(*_batch(i), SCALE)
    tr.lr = 0.0
    torch.cuda.synchronize()
    p, ema = tr.flat.p.clone(), tr.flat.ema.clone()
    tr.step(*_batch(2), SCALE)
    torch.cuda.synchronize()
    assert torch.equal(tr.flat.p, p), "a replayed step at lr 0 changed the parameters"
    assert not torch.equal(tr.flat.ema, ema), "the EMA did not move"
    tr.lr = 2e-4
    tr.step(*_batch(3), SCALE)
    torch.cuda.synchronize()
    assert not torch.equal(tr.flat.p, p)


def _roundtrip(obj):
    buf = io.BytesIO()
    torch.save(obj, buf)
    buf.seek(0)
    return torch.load(buf, map_location=lambda s, loc: s.cuda(0))


def _native_steps(tr, sched, its):
    for it in its:
        update_learning_rate(tr.optimizer, [sched], it)
        tr.step(*_batch(it), SCALE)
    torch.cuda.synchronize()


def _native_from(ckpt, state, use_graph):
    """A fresh net + NativeTrainer + scheduler resumed from a checkpoint: {'params', 'params_ema'} and a training_state."""
    from savsr_b200 import trainplan as TP
    net = _gpu_net(ckpt["params"])
    tr = TP.NativeTrainer(net, use_graph=use_graph)
    sched = CosineAnnealingRestartLR(tr.optimizer, periods=[8], eta_min=1e-7)
    assert tr.resume(state, [sched]) == (state["epoch"], state["iter"])
    if "params_ema" in ckpt:
        tr.load_ema_state_dict(ckpt["params_ema"])
    return net, tr, sched


def _native_start(steps, use_graph=True):
    """A native run of `steps` scheduled steps from the default initialisation, and its checkpoint (through torch.save / torch.load)."""
    from savsr_b200 import trainplan as TP
    net = _gpu_net()
    tr = TP.NativeTrainer(net, use_graph=use_graph)
    sched = CosineAnnealingRestartLR(tr.optimizer, periods=[8], eta_min=1e-7)
    _native_steps(tr, sched, range(1, steps + 1))
    ckpt = _roundtrip({"params": net.state_dict(), "params_ema": tr.ema_state_dict()})
    state = _roundtrip(tr.training_state(iter=steps, epoch=0, schedulers=[sched]))
    return net, tr, sched, ckpt, state


@pytest.mark.gpu
def test_cosine_schedule_graph_and_eager_agree():
    """The same 4 scheduled steps (a different lr each) replayed as CUDA graphs and issued eagerly, both from one saved state."""
    net0, _, _, ckpt, state = _native_start(3)
    base = _flat_params(net0)
    runs = {}
    for use_graph in (True, False):
        net, tr, sched = _native_from(ckpt, state, use_graph)
        lrs = []
        for it in range(4, 8):
            update_learning_rate(tr.optimizer, [sched], it)
            lrs.append(tr.lr)
            tr.step(*_batch(it), SCALE)
        torch.cuda.synchronize()
        runs[use_graph] = (_flat_params(net), _native_moments(tr), lrs)
    assert runs[True][2] == runs[False][2] and len(set(runs[True][2])) == 4
    _assert_parity(runs[True][0], runs[False][0], runs[True][1], runs[False][1], base, "cosine schedule, 4 steps, graph vs eager")


@pytest.mark.gpu
def test_resume_is_exact_at_load_and_continues_like_an_uninterrupted_run():
    net_a, tr_a, s_a, ckpt, state = _native_start(3)
    base = _flat_params(net_a)
    net_c, tr_c, s_c = _native_from(ckpt, state, use_graph=True)
    fa, fc = tr_a.flat, tr_c.flat
    for n in fa.P:
        for buf_a, buf_c in ((fa.p, fc.p), (fa.m, fc.m), (fa.v, fc.v), (fa.ema, fc.ema)):
            assert torch.equal(fa.view(buf_a, n), fc.view(buf_c, n)), n
    assert torch.equal(fa.step_t, fc.step_t) and tr_c.lr == tr_a.lr
    ema_sd = tr_c.ema_state_dict()
    assert list(ema_sd) == list(ckpt["params_ema"]) and all(torch.equal(ema_sd[k], v) for k, v in ckpt["params_ema"].items())
    _native_steps(tr_a, s_a, range(4, 7))                             # the uninterrupted run goes on
    _native_steps(tr_c, s_c, range(4, 7))
    assert tr_c.lr == tr_a.lr and float(fc.step_t) == float(fa.step_t) == 6.0
    _assert_parity(_flat_params(net_c), _flat_params(net_a), _native_moments(tr_c), _native_moments(tr_a), base,
                   "resumed after 3 steps vs uninterrupted, 3 more steps")


def _module_steps(net, opt, sched, its):
    from savsr_b200 import train as T
    net.set_scale(SCALE)
    for it in its:
        update_learning_rate(opt, [sched], it)
        opt.zero_grad(set_to_none=True)
        lq, gt = _batch(it)
        T.charbonnier(net(lq), gt).backward()
        opt.step()
    torch.cuda.synchronize()


def _module_opt(net):
    opt = torch.optim.Adam(net.parameters(), lr=2e-4, betas=(0.9, 0.99))
    return opt, CosineAnnealingRestartLR(opt, periods=[8], eta_min=1e-7)


@pytest.mark.gpu
def test_module_path_adam_state_continues_in_the_native_trainer():
    net = _gpu_net()
    opt, sched = _module_opt(net)
    _module_steps(net, opt, sched, range(1, 4))
    base = _flat_params(net)
    ckpt = _roundtrip({"params": net.state_dict()})
    state = _roundtrip({"optimizers": [opt.state_dict()], "schedulers": [sched.state_dict()], "epoch": 0, "iter": 3})
    _module_steps(net, opt, sched, range(4, 7))                       # the module path goes on
    net_n, tr, s_n = _native_from(ckpt, state, use_graph=True)
    assert float(tr.flat.step_t) == 3.0
    _native_steps(tr, s_n, range(4, 7))
    assert tr.lr == opt.param_groups[0]["lr"]
    _assert_parity(_flat_params(net_n), _flat_params(net), _native_moments(tr), _torch_moments(net, opt), base,
                   "module path 3 steps -> NativeTrainer 3 steps vs module path 6")


@pytest.mark.gpu
def test_native_trainer_adam_state_continues_in_the_module_path():
    net, tr, sched, ckpt, state = _native_start(3)
    base = _flat_params(net)
    _native_steps(tr, sched, range(4, 7))                             # the native step goes on
    net_m = _gpu_net(ckpt["params"])
    opt, s_m = _module_opt(net_m)
    opt.load_state_dict(state["optimizers"][0])
    s_m.load_state_dict(state["schedulers"][0])
    assert all(float(s["step"]) == 3.0 for s in opt.state_dict()["state"].values())
    _module_steps(net_m, opt, s_m, range(4, 7))
    assert tr.lr == opt.param_groups[0]["lr"]
    _assert_parity(_flat_params(net_m), _flat_params(net), _torch_moments(net_m, opt), _native_moments(tr), base,
                   "NativeTrainer 3 steps -> module path 3 steps vs NativeTrainer 6")
