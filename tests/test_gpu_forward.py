"""-m gpu: the whole SAVSR forward through the drop-in module (C ABI underneath) against the golden vectors of the
reference, the CPU oracle, and size-independent properties at the BASELINE shapes."""
import glob
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = sorted(p for p in glob.glob(os.path.join(GOLDEN, "*.npz"))
               if "fingerprint" not in p and "metrics" not in p and "_kat" not in p and not os.path.basename(p).startswith("train_"))
TRAIN_CASES = sorted(glob.glob(os.path.join(GOLDEN, "train_*.npz")))

# Tolerances, straight from the north star:
#   * bf16 operand path (fp32 accumulate): <= 0.05 dB PSNR delta (test_psnr_delta_gate); max-abs is reported and asserted
#     with the margin that bf16 rounding of ~150 stacked layers needs (measured 1.0-1.5e-3).
#   * high-precision path (fp16 operands, 10-bit mantissa, fp32 accumulate; same kernels, same speed): the fp32 criterion
#     max-abs <= 1e-3 against the fp32 reference (measured 1.2e-4).
MAX_ABS_TOL = 4e-3
STAGE_REL_TOL = 0.03
FP32_CRITERION = 1e-3
TOL = {"bf16": (MAX_ABS_TOL, STAGE_REL_TOL), "fp16": (FP32_CRITERION, 0.005)}


@pytest.fixture(scope="module")
def G():
    import gpu_checks
    return gpu_checks


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p)[:-4] for p in CASES])
@pytest.mark.parametrize("impl,precision", [("halo", "bf16"), ("tap", "bf16"), ("halo", "fp16")])
def test_forward_matches_reference_golden(G, path, impl, precision):
    from oracle.state_dict_fixture import make_input, make_state_dict
    g = np.load(path)
    b, h, w = int(g["b"]), int(g["h"]), int(g["w"])
    scale = tuple(float(s) if float(s) != int(s) else int(s) for s in g["scale"])
    y, taps, plan = G.run_forward(make_state_dict(int(g["sd_seed"])), make_input(b, h, w, int(g["in_seed"])), scale, impl=impl, taps=G.TAPS,
                                  precision=precision)
    max_abs_tol, stage_tol = TOL[precision]
    ref = torch.from_numpy(g["out"])
    assert y.shape == ref.shape
    assert float((y - ref).abs().max()) < max_abs_tol
    for key in ("f2p_last", "p2f_last", "align", "rg0", "rg3"):
        t = taps[key][..., :h, :w].contiguous().flatten()
        idx = torch.linspace(0, t.numel() - 1, steps=min(257, t.numel())).long()
        if tuple(g[f"probe.{key}.shape"]) != tuple(taps[key][..., :h, :w].shape):
            continue                          # padded sizes: the golden probe was taken on the padded map
        samp = torch.from_numpy(g[f"probe.{key}.sample"])
        assert float((t[idx] - samp).abs().max()) < stage_tol * float(g[f"probe.{key}.absmax"]), key
    # the SATU + tail branch on its own (the output is dominated by the bilinear skip): y - skip against the reference's tail probe
    x = make_input(b, h, w, int(g["in_seed"]))
    skip = torch.nn.functional.interpolate(x[:, 3], size=tuple(y.shape[-2:]), mode="bilinear", align_corners=False)
    t = (y - skip).contiguous().flatten()
    assert tuple(g["probe.tail.shape"]) == tuple(y.shape)
    idx = torch.linspace(0, t.numel() - 1, steps=min(257, t.numel())).long()
    assert float((t[idx] - torch.from_numpy(g["probe.tail.sample"])).abs().max()) < stage_tol * float(g["probe.tail.absmax"]), "tail"


@pytest.mark.parametrize("kw", [dict(b=1, h=16, w=20, scale=(2, 2)), dict(b=2, h=13, w=15, scale=(1.5, 4), sd_seed=1, in_seed=1236),
                                dict(b=1, h=31, w=31, scale=(3, 3), sd_seed=2), dict(b=3, h=20, w=36, scale=(2.7, 2.7), sd_seed=1),
                                dict(b=1, h=8, w=8, scale=(4, 4)), dict(b=1, h=2, w=3, scale=(1.1, 1.1))])
def test_forward_vs_oracle_with_stage_errors(G, kw):
    info = G.check_forward(impl="halo", tol=MAX_ABS_TOL, stage_tol=STAGE_REL_TOL, **kw)
    assert info["psnr_vs_oracle"] > 55.0


@pytest.mark.parametrize("seed", range(6))
def test_forward_random_shapes_and_scales(G, seed):
    """Edge sweep: random odd / tiny frame sizes, batch sizes and asymmetric non-integer scales (up to x8) vs the oracle."""
    import random
    rnd = random.Random(1000 + seed)
    h, w = rnd.randint(5, 37), rnd.randint(5, 41)
    scale = (rnd.choice([1.1, 1.5, 2, 2.3, 3, 3.9, 4, 6.25, 8]), rnd.choice([1.2, 1.7, 2, 2.7, 3.5, 4, 5.1, 7.3]))
    info = G.check_forward(b=rnd.randint(1, 3), h=h, w=w, scale=scale, sd_seed=seed % 3, in_seed=77 + seed, impl="halo", graph=bool(seed & 1),
                           tol=TOL["bf16"][0], stage_tol=TOL["bf16"][1])
    assert info["psnr_vs_oracle"] > 55.0, info


def test_fp16_path_meets_the_fp32_criterion_with_stage_errors(G):
    for kw in (dict(b=1, h=16, w=20, scale=(2, 2)), dict(b=2, h=13, w=15, scale=(1.5, 4), sd_seed=1, in_seed=1236),
               dict(b=1, h=31, w=31, scale=(3, 3), sd_seed=2)):
        info = G.check_forward(impl="halo", precision="fp16", tol=FP32_CRITERION, stage_tol=0.005, **kw)
        assert info["psnr_vs_oracle"] > 65.0


def test_psnr_delta_gate_bf16_path(G):
    """North-star gate on a Vid4-SHAPED clip (144x180 LR -> 576x720 HR, x4, three output frames of a 9-frame clip):
    PSNR_Y(oracle, GT) - PSNR_Y(ours, GT) <= 0.05 dB with the reference's own metric chain (SURVEY.md 8d)."""
    import torch.nn.functional as F
    from oracle import savsr_oracle as O
    from oracle.state_dict_fixture import make_state_dict
    from savsr_b200 import sharding
    torch.manual_seed(3)
    torch.set_num_threads(os.cpu_count() or 1)
    scale, h, w = (4, 4), 144, 180
    gt = torch.rand(9, 3, 18, 23)
    gt = F.interpolate(gt, size=(h * 4, w * 4), mode="bicubic", align_corners=False).clamp(0, 1)       # smooth synthetic HR clip
    lr = F.interpolate(gt, size=(h, w), mode="bicubic", align_corners=False, antialias=True).clamp(0, 1)
    sd = make_state_dict(0)
    frames = [3, 4, 5]
    win = sharding.gather_windows(lr, frames)
    with torch.no_grad():
        y_ref = O.forward(sd, win, scale)
    for precision in ("bf16", "fp16"):
        y, _, _ = G.run_forward(sd, win, scale, impl="halo", graph=True, precision=precision)
        p_ref = O.psnr_y(y_ref, gt[frames]); p_new = O.psnr_y(y, gt[frames])
        assert abs(p_ref - p_new) <= 0.05, (precision, p_ref, p_new)
        assert O.psnr_y(y, y_ref) > 55.0
        if precision == "fp16":
            assert float((y - y_ref).abs().max()) < FP32_CRITERION


def test_determinism_graph_and_batch_invariance(G):
    """Size-independent properties: run-to-run bit-exact, CUDA graph == eager, batched == per-sample (SURVEY.md section 4)."""
    from oracle.state_dict_fixture import make_input, make_state_dict
    sd = make_state_dict(1)
    x = make_input(3, 22, 26, 77)
    y1, _, _ = G.run_forward(sd, x, (2.7, 2.7), impl="halo", graph=False)
    y2, _, _ = G.run_forward(sd, x, (2.7, 2.7), impl="halo", graph=True)
    y3, _, _ = G.run_forward(sd, x, (2.7, 2.7), impl="halo", graph=True)
    assert torch.equal(y1, y2) and torch.equal(y2, y3)
    singles = torch.cat([G.run_forward(sd, x[i:i + 1], (2.7, 2.7), impl="halo")[0] for i in range(3)])
    assert torch.equal(singles, y1)            # eval-mode windows are independent: batching is numerically free
    yt, _, _ = G.run_forward(sd, x, (2.7, 2.7), impl="tap")
    assert float((yt - y1).abs().max()) < 1e-5  # the two A-fetch modes feed identical operands to the tensor core


@pytest.mark.parametrize("scale", [(4, 4), (1.5, 4), (2.7, 2.7)])
@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_vid4_shape_against_oracle(G, scale, precision):
    """BASELINE configs 2-3 at full size (one 144x180 window; the CPU oracle needs about a second per frame)."""
    from oracle import savsr_oracle as O
    from oracle.state_dict_fixture import make_input, make_state_dict
    sd = make_state_dict(0)
    x = make_input(1, 144, 180, 1234)
    y, _, plan = G.run_forward(sd, x, scale, impl="halo", graph=True, precision=precision)
    torch.set_num_threads(os.cpu_count() or 1)
    with torch.no_grad():
        y_ref = O.forward(sd, x, scale)
    assert tuple(y.shape) == (1, 3) + O.get_hw(144, 180, scale)
    assert float((y - y_ref).abs().max()) < TOL[precision][0]
    assert O.psnr_y(y, y_ref) > (55.0 if precision == "bf16" else 65.0)
    # bit-exact sampling indices at this shape (north star): cell / corner / R vectors vs the numpy oracle
    H, W = O.get_hw(144, 180, scale)
    assert np.array_equal(plan.cell_y.cpu().numpy(), O.satu_cell(H, scale[0]))
    assert np.array_equal(plan.cell_x.cpu().numpy(), O.satu_cell(W, scale[1]))
    assert np.array_equal(plan.corner_y.cpu().numpy(), O.satu_base_corner(H, 144, scale[0]))
    assert np.array_equal(plan.corner_x.cpu().numpy(), O.satu_base_corner(W, 180, scale[1]))
    assert np.array_equal(plan.rel_y.cpu().numpy().view(np.uint32), O.satu_rel_coord(H, scale[0]).view(np.uint32))
    assert np.array_equal(plan.rel_x.cpu().numpy().view(np.uint32), O.satu_rel_coord(W, scale[1]).view(np.uint32))


@pytest.mark.parametrize("name,b,h,w,scale", [("udm10_x4", 1, 180, 318, (4, 4)), ("cfg1_x2", 1, 64, 64, (2, 2)),
                                                ("udm10_x4_b2_odd_tail", 2, 179, 317, (4, 4))])
@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_baseline_shapes_against_oracle(G, name, b, h, w, scale, precision):
    """BASELINE config 4 (UDM10 shape: 23 x 12 = 276 tiles per image, another chunking of the persistent loop) and config 1
    (64x64, x2) at full size, whole forward + stage taps vs the CPU oracle; the odd-size case exercises pad_spatial there."""
    torch.set_num_threads(os.cpu_count() or 1)
    info = G.check_forward(b=b, h=h, w=w, scale=scale, sd_seed=0, in_seed=1234, impl="halo", graph=True, tol=TOL[precision][0],
                           stage_tol=TOL[precision][1], precision=precision)
    assert info["psnr_vs_oracle"] > (55.0 if precision == "bf16" else 65.0), info


@pytest.mark.parametrize("block", ["residual_group", "window_unit_l1", "osadapt"])
@pytest.mark.parametrize("precision,tol,median", [("fp16", 0.04, 0.012), ("bf16", 0.08, 0.03)])
def test_train_mode_gradients_match_the_oracle(G, block, precision, tol, median):
    """Row f1 stage A: gradients of one ResidualGroup, one WindowUnit_l1 (three OSA-Convs inside) and one OSAdapt (train-mode
    BatchNorm in the mask net) at 16x20, b = 2 against fp32 CPU autograd on the oracle, relative L2 error per parameter tensor.
    Every activation and every incoming gradient is rounded to the 16-bit operand format on its way into the tensor core, and a
    rounding that flips the sign of a pre-activation flips a ReLU mask: with fp16 operands (2^-11) every tensor agrees to 4 %
    (measured: worst 2.4-3.2 %, median 0.1-0.8 %), with bf16 operands (2^-9) to 8 % (measured: worst 5-6 % in the 17-conv-deep
    ResidualGroup and the three-OSA WindowUnit, median 0.3-2.4 %).  See gpu_checks._grad_report for the error definition."""
    G.set_precision(precision)
    try:
        info = G.check_train_block(block, tol=tol)
    finally:
        G.set_precision("bf16")
    assert info["median"] < median, info


@pytest.mark.parametrize("native_module", [True, False], ids=["native_launch_list", "stage_a_aten_tape"])
def test_training_step_whole_net(G, native_module):
    """The reference's optimisation step as ITS code runs it (sr_model.py:101-128): `net.train(); out = net(lq)`, the caller's Charbonnier
    loss, `backward()`, torch.optim.Adam, EMA -- on the module.  By default the module's train-mode forward is the native launch list behind
    one autograd node (per-tensor gradient parity vs the oracle asserted); the ATen-tape path of stage A stays selectable."""
    info = G.check_train_step(native_module=native_module)
    print(info)
    assert info["losses"][-1] < info["losses"][0]


def test_second_device_in_one_process(G):
    """Advisor finding (round 1): kernel attributes are per device and launches must follow the module's device, not the caller's
    current device.  One process, module on cuda:1 while cuda:0 is current; result must equal the cuda:0 result bit for bit."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs in one process")
    import savsr_b200
    from oracle.state_dict_fixture import make_input, make_state_dict
    sd = make_state_dict(1)
    x = make_input(2, 18, 22, 5)
    outs = []
    for dev in ("cuda:0", "cuda:1"):
        net = savsr_b200.SAVSR().to(dev)
        net.load_state_dict(sd, strict=True)
        net.eval(); net.set_scale((2.7, 1.5))
        torch.cuda.set_device(0)                                   # the caller's current device stays cuda:0 throughout
        with torch.no_grad():
            y = net(x.to(dev))
            y2 = net(x.flip(0).to(dev))                            # second call, other input: a real CUDA-graph replay on that device
            net.use_graph = False
            y3 = net(x.flip(0).to(dev))                            # the same eagerly
        assert y.device == torch.device(dev) and torch.equal(y2, y3) and not torch.equal(y, y2)
        assert torch.equal(y2.flip(0), y)                          # windows are independent: flipping the batch flips the result
        assert torch.cuda.current_device() == 0
        outs.append(y.cpu())
    assert torch.equal(outs[0], outs[1])


def test_module_api_errors(G):
    import savsr_b200
    net = savsr_b200.SAVSR().cuda()
    net.eval()
    with pytest.raises(ValueError):
        net(torch.zeros(1, 7, 3, 1, 8, device="cuda"))
    net.set_scale(2)
    y = net(torch.rand(1, 7, 3, 8, 10, device="cuda"))
    assert tuple(y.shape) == (1, 3, 16, 20) and y.dtype == torch.float32
    y0 = net(torch.rand(0, 7, 3, 8, 10, device="cuda"))            # an empty batch (a rank that owns no frame): empty result, no launch
    assert tuple(y0.shape) == (0, 3, 16, 20) and y0.dtype == torch.float32
    with pytest.raises(ValueError):
        net(torch.zeros(1, 5, 3, 8, 10, device="cuda"))            # not a 7-frame window
    with pytest.raises(RuntimeError):
        net(torch.zeros(1, 7, 3, 8, 10))                           # CPU tensors are refused: there is no CPU path


@pytest.mark.gpu
@pytest.mark.parametrize("kw", [dict(), dict(scale=(1.5, 4), seed=1, b=3, h=12, w=24), dict(native_attn=False, native_mask=False),
                                dict(scale=(2.7, 2.7), seed=2, b=1, h=8, w=72)],
                         ids=["x2", "x1.5x4_b3", "aten_attention_and_mask_islands", "x2.7_w72"])
def test_native_training_plan_gradients_match_the_oracle(G, kw):
    """Row f1 stage B: the static forward + backward launch list (savsr_b200.trainplan) against fp32 CPU autograd through the oracle on
    the WHOLE net: loss to 2e-3, every parameter tensor's gradient within 10 % of max(|r|, 1 % of the largest tensor gradient)
    (measured worst 4.5 %, median 0.07 %), cosine of the flat gradient > 0.999.  Gradients are stored in bf16 between layers."""
    info = G.check_trainplan(**kw)
    print(info)


@pytest.mark.gpu
@pytest.mark.parametrize("scale", [(4, 4), (1.5, 4)], ids=["x4", "x1.5x4"])
def test_native_training_plan_at_the_cfg5_batch(G, scale):
    """BASELINE config 5 at its full size (4 x 7 x 3 x 64 x 64 Vimeo90K crops): loss and every parameter gradient of the native step against
    the oracle's fp32 autograd evaluated on the GPU (TF32 off).  With 16 384 pixels per sample the batch statistics and the pixel sums are
    well conditioned: measured worst tensor 1.1 %, median 0.04 %, cosine 0.999994 -- bounds 5 % / 0.9999 (the 16 x 20 CPU-oracle cases keep 10 %)."""
    info = G.check_trainplan(b=4, h=64, w=64, scale=scale, seed=3, oracle_device="cuda", tol_worst=0.05, tol_cos=0.9999)
    print({k: info[k] for k in ("loss", "ref_loss", "cos", "median", "worst")})


@pytest.mark.gpu
@pytest.mark.parametrize("path", TRAIN_CASES, ids=[os.path.basename(p)[:-4] for p in TRAIN_CASES])
def test_training_step_matches_reference_golden(G, path):
    """Row f1 against the reference itself (not through the oracle): tests/golden/train_*.npz hold the loss and the gradients of the
    unmodified reference in train() mode."""
    info = G.check_train_golden(path)
    print(info)
    if "b2_12x14" in path:
        assert info["native"], "an even-sized batch must take the native launch list"


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True], ids=["eager", "cuda_graph"])
def test_native_training_steps_reduce_the_loss(G, graph):
    """Pack -> forward -> backward -> Adam + EMA for a few steps on a fixed batch, eagerly and as replayed CUDA graphs."""
    info = G.check_trainplan(steps=4, graph=graph)
    print(info["losses"])


@pytest.mark.gpu
def test_forward_as_one_c_call(G):
    """SURVEY section 8b: `savsr_forward(plan, x, out, stream)` -- the recorded launch list of the plan replayed by one C call."""
    print(G.check_c_plan())


@pytest.mark.gpu
def test_fp16_path_refuses_to_saturate(G):
    """The criterion-meeting fp16 path has 65504 of range: SAVSR.forward measures the headroom once per plan and raises below 4x."""
    print(G.check_fp16_range_guard())
