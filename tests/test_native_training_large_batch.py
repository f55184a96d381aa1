"""The native training step at up to 32 samples per GPU (trainplan.MAX_NATIVE_BATCH), which covers the reference's training YAML
(16 crops of 60 x 60 per GPU).  CPU: which path the module and the plan choose at each batch size, checked against the recording fake
of the C library.  GPU: gradients against the fp32 oracle at remainder / ceiling batches and at the YAML shape, and the module path
driven the way the reference's training loop drives it."""
import numpy as np
import pytest
import torch
from types import SimpleNamespace

from fake_lib import mocked_engine

ATTN_CALLS = ("savsr_osa_prologue_train", "savsr_osa_fold_backward", "savsr_ca_backward")


def _flat_grad(net):
    return torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).flatten() for p in net.parameters()]).double()


def _fake_cuda(*shape):
    """Quacks like a CUDA tensor for ModuleTraining.supports (the check only looks at the device and the shape)."""
    return SimpleNamespace(is_cuda=True, shape=shape, dim=lambda: len(shape))


@pytest.mark.parametrize("shape,ok", [((16, 7, 3, 60, 60), True), ((32, 7, 3, 60, 60), True), ((1, 7, 3, 16, 24), True),
                                      ((33, 7, 3, 60, 60), False), ((16, 7, 3, 61, 60), False), ((16, 7, 3, 60, 59), False),
                                      ((16, 5, 3, 60, 60), False)],
                         ids=["b16_yaml", "b32_ceiling", "b1", "b33", "odd_h", "odd_w", "t5"])
def test_module_takes_the_native_path_up_to_32_samples(shape, ok):
    from savsr_b200 import trainplan as TP
    assert TP.MAX_NATIVE_BATCH == 32
    assert TP.ModuleTraining.supports(_fake_cuda(*shape)) is ok


@pytest.fixture(scope="module")
def recorded_batches():
    """One NativeTrainer step at b = 16 and b = 33 (16 x 24, x2) against the fake library, plus the b = 2 plan of the same size."""
    import savsr_b200
    from savsr_b200 import trainplan as TP
    torch.manual_seed(0)
    net = savsr_b200.SAVSR()
    out = {}
    with mocked_engine() as lib:
        import savsr_b200.autograd as A
        import torch.nn.functional as F
        saved = (TP.context, TP._require_cuda, A.sta_lrelu)
        TP.context = lambda idx: __import__("savsr_b200.engine", fromlist=["context"]).context(idx)
        TP._require_cuda = lambda dev: None

        def sta_lrelu_torch(x, kpre, slope=0.1):           # the ATen formulation of the fused op (no kernel runs in this test)
            b, c, h, w = x.shape
            kern = F.leaky_relu(kpre, slope).view(b, c, 25, h * w)
            return (F.unfold(F.pad(x, (2, 2, 2, 2), mode="replicate"), 5).view(b, c, 25, h * w) * kern).sum(2).view(b, c, h, w)
        A.sta_lrelu = sta_lrelu_torch
        try:
            tr = TP.NativeTrainer(net, use_graph=False)
            out[2] = (tr.plan_for(torch.rand(2, 7, 3, 16, 24), (2, 2)), None)
            for b in (16, 33):
                lq = torch.rand(b, 7, 3, 16, 24)
                gt = torch.rand(b, 3, 32, 48)
                plan = tr.plan_for(lq, (2, 2))
                lib.calls.clear()
                tr.step(lq, gt, (2, 2))
                out[b] = (plan, list(lib.calls))
                tr.plans.clear()                               # (drop the plan: its arenas are large on the host)
        finally:
            TP.context, TP._require_cuda, A.sta_lrelu = saved
    return out


def test_b16_step_runs_the_native_attention_kernels(recorded_batches):
    plan, calls = recorded_batches[16]
    names = [c[0] for c in calls]
    # l1 5 iterations x 3 blocks (both directions per launch), l2 2, adapt 4
    for name, arg in (("savsr_osa_prologue_train", 4), ("savsr_osa_fold_backward", 5)):
        batches = [args[arg] for n, args in calls if n == name]
        assert len(batches) == 15 + 2 + 4 and set(batches) == {16}, (name, batches)
    assert names.count("savsr_ca_backward") == 32
    assert set(args[4] for n, args in calls if n == "savsr_ca_backward") == {16}
    islands = {k for k in plan.kinds.values() if "island_osa" in k or "island_ca" in k}
    assert not islands, islands
    assert plan.native_attn


def test_slot_counts_do_not_depend_on_the_batch(recorded_batches):
    p2, p16 = recorded_batches[2][0], recorded_batches[16][0]
    assert (p16.n_slots, p16.n_tslots) == (p2.n_slots, p2.n_tslots)


def test_b33_step_keeps_the_attention_islands(recorded_batches):
    plan, calls = recorded_batches[33]
    names = {c[0] for c in calls}
    assert not names & set(ATTN_CALLS), names & set(ATTN_CALLS)
    assert not plan.native_attn
    kinds = set(plan.kinds.values())
    assert any("island_osa" in k for k in kinds) and any("island_ca" in k for k in kinds), kinds


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def G():
    import gpu_checks
    return gpu_checks


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(b=13, scale=(1.5, 4), seed=1), dict(b=32, scale=(2, 2), seed=2)], ids=["b13_x1.5x4", "b32_x2"])
def test_remainder_and_ceiling_batches_match_the_oracle(G, kw):
    """b = 13 runs the unfold kernel's four-sample loop with a remainder of one and the 16-sample matvec bucket; b = 32 is the ceiling
    (largest shared-memory footprint, the 32-sample matvec bucket).  Oracle in fp32 on the GPU, the 16 x 20 bounds of 10 % / 0.999."""
    info = G.check_trainplan(h=16, w=20, oracle_device="cuda", **kw)
    print({k: info[k] for k in ("loss", "ref_loss", "cos", "median", "worst")})


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(scale=(4, 4)), dict(scale=(1.5, 4)), dict(scale=(4, 4), steps=2, graph=True)],
                         ids=["x4", "x1.5x4", "x4_graph_steps"])
def test_native_training_plan_at_the_yaml_shape(G, kw):
    """The reference's training YAML per GPU: 16 x 7 x 3 x 60 x 60 (lq_size 60, batch_size_per_gpu 16).  Every parameter gradient against
    the oracle's fp32 autograd on the GPU (TF32 off) with the cfg-5 bounds of 5 % worst tensor and cosine 0.9999.  The graph case then
    replays two steps of this scale interleaved with a second scale that shares the arenas, and the loss of both decreases."""
    info = G.check_trainplan(b=16, h=60, w=60, seed=3, oracle_device="cuda", tol_worst=0.05, tol_cos=0.9999, **kw)
    print({k: info[k] for k in ("loss", "ref_loss", "cos", "median", "worst", "slots", "tslots") + (("losses", "losses_second_scale") if "steps" in kw else ())})


@pytest.mark.gpu
def test_module_path_at_the_yaml_shape(G):
    """SAVSR in train mode under the reference's own loop (net(lq), Charbonnier, backward, torch.optim.Adam) at 16 x 60 x 60: it takes the
    native launch list, captures its graphs by the second step, and its step-0 gradient equals NativeTrainer's on the same input and weights
    up to the ordering of fp32 atomics (both run the same launch list)."""
    import savsr_b200
    from oracle.state_dict_fixture import make_input, make_state_dict
    from savsr_b200 import train as T
    from savsr_b200 import trainplan as TP
    dev = G.DEV
    scale = (4, 4)
    sd = make_state_dict(3)
    x = make_input(16, 60, 60, 1237).to(dev)
    gt = torch.rand(16, 3, 240, 240, generator=torch.Generator().manual_seed(5)).to(dev)

    ref_net = savsr_b200.SAVSR().to(dev)
    ref_net.load_state_dict(sd, strict=True)
    ref_net.set_scale(scale); ref_net.train()
    tr = TP.NativeTrainer(ref_net, use_graph=False)
    plan = tr.plan_for(x, scale)
    plan.x_in.copy_(x); plan.gt.copy_(gt)
    ref_loss = float(tr._fwd_bwd(plan))
    ref_flat = _flat_grad(ref_net)
    del tr, plan, ref_net
    torch.cuda.empty_cache()

    net = savsr_b200.SAVSR().to(dev)
    net.load_state_dict(sd, strict=True)
    net.set_scale(scale); net.train()
    opt = torch.optim.Adam(net.parameters(), lr=2e-4, betas=(0.9, 0.99))
    losses = []
    for step in range(3):
        opt.zero_grad(set_to_none=True)
        loss = T.charbonnier(net(x), gt)
        loss.backward()
        if step == 0:
            flat = _flat_grad(net)
        opt.step()
        losses.append(float(loss))
        state = net.__dict__.get("_train_state")
        assert state is not None, "the module took the stage-A tape, not the native launch list"
        if step == 1:
            (mplan,) = state.plans.values()
            assert mplan.g_fwd is not None and mplan.g_bwd is not None, "graphs not captured by the second step"
    cos = float(torch.dot(flat, ref_flat) / (flat.norm() * ref_flat.norm()))
    info = dict(loss0=losses[0], native_trainer_loss=ref_loss, cos=cos, losses=losses)
    print(info)
    assert abs(losses[0] - ref_loss) <= 1e-5 * abs(ref_loss), info
    assert np.isfinite(cos) and cos >= 0.9999, info
    assert all(np.isfinite(l) for l in losses) and losses[-1] < losses[0], info
