#!/usr/bin/env python
"""SAVSR forward hot-path benchmark (contract: see task brief / DESIGN.md section "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload vid4_x4] [--batch B] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A "step" = super-resolving one synthetic Vid4-shaped clip (34 frames, 144x180 LR -> 576x720 HR at x4; every output frame is
an independent 7-frame window, lbasicsr/models/video_base_model.py:50-59), in batches of `--batch` windows.  With N GPUs every
rank processes its own clip (frames shard with no data-path collective; weak scaling).  Rank 0 prints ONE JSON line:

  value         HR Mpix/s, whole job, windows already resident in HBM when the timed region starts
  e2e           same metric through the public API (savsr_b200.sharding.infer_clip on the savsr_b200.SAVSR module) with the
                LR clip in pinned HOST memory and the HR result copied back to pinned host memory every step
  roofline      dominant kernel (tcgen05 implicit-GEMM 3x3 conv, N = 64): ALGORITHMIC FLOPs (reference channel counts, no zero
                padding) / CUDA-event time of those launches, measured live in an eager pass, against the measured bf16 peak
  roofline_osa  the same for the OSA-Conv launches alone (per-sample folded weights; north star: >= 60 % of the tensor peak)
  roofline_satu SATU chain (kernel_conv+sta, HR gather/experts/fusion/tail): compulsory bytes / time vs the HBM peak AND
                FLOPs / time vs the tensor peak (SATU is compute-bound under the compulsory byte count, SURVEY.md D7)
  fp16          the same resident measurement with fp16 operands (the path that meets the <= 1e-3 fp32 criterion)
  latency_b1    one window per call through SAVSR.forward (what lbasicsr/test.py does), VSR_runtime_test protocol
  gpu_reference the reference's own PyTorch/cuDNN path on THIS GPU (cudnn.benchmark, TF32 on/off), b = 1 and b = batch
  cfg4_strong   BASELINE config 4: 10 UDM10-shaped clips x 32 frames (320 frames, 180x318 -> 720x1272), FIXED work sharded
                rank-strided over the N ranks (strong scaling), with the reference's metric reduction (dist.reduce of
                [n_frames, n_metrics]) and, second figure, the gather of all HR frames to rank 0 inside the timed region
  cpu_baseline  the reference's CPU path on the host cores, bounded sample
  pipeline      (informational) the reference's whole test loop minus the PNG codec through savsr_b200.datapath.evaluate_clip

--impl reference times the reference's own CPU implementation of the path (the unmodified reference installed under
baseline/_ref when present, else the pinned oracle port) on this arm's workload / metric, rank 0 only.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {  # name: (frames, h, w, scale)
    "vid4_x4": (34, 144, 180, (4, 4)),
    "vid4_x1.5x4": (34, 144, 180, (1.5, 4)),
    "vid4_x2.7": (34, 144, 180, (2.7, 2.7)),
    "udm10_x4": (32, 180, 318, (4, 4)),
    "cfg1_x2": (7, 64, 64, (2, 2)),
}
YAML_KWARGS = dict(num_in_ch=3, num_feat=64, num_frame=7, slid_win=3, fusion_win=5, interval=0, w1_num_block=4, w2_num_block=2,
                   n_resgroups=4, n_resblocks=8, center_frame_idx=None)     # options/test/SAVSR/test_SAVSR_Vid4_asBI.yml:830-842
SATU_KINDS = ("satu_kconv_sta", "satu_fused", "satu_hr", "satu_tail")


def hw_out(h, w, scale):
    return round(h * scale[0]), round(w * scale[1])          # savsr_arch.py:745-751 (python round)


def flops_per_frame(h, w, H, W):
    """BASELINE.md section 3: F = 2 * [22 888 128 hp wp + 104 000 h w + 19 904 H W]."""
    hp, wp = h + (h & 1), w + (w & 1)
    return 2.0 * (22888128.0 * hp * wp + 104000.0 * h * w + 19904.0 * H * W)


def satu_flops_per_frame(h, w, H, W):
    """SURVEY.md 8d: kernel_conv 102 400 + sta_conv 1 600 MAC per LR px; body + heads + expert mix + fusion 18 176 and tail 1 728 per HR px."""
    return 2.0 * (104000.0 * h * w + 19904.0 * H * W)


def satu_compulsory_bytes(h, w, H, W):
    """SURVEY.md 8d: B_SATU = 4 (64 hw [x] + 64 hw [st_feat] + 3 hw [x_center] + 3 HW [out]) per frame (+0.49 MB of parameters per launch)."""
    return 4.0 * (2 * 64 * h * w + 3 * h * w + 3 * H * W)


def workload_config(name, world):
    """The `config` object both arms print (identical keys and values, so the driver's same_config check holds)."""
    frames, h, w, scale = WORKLOADS[name]
    H, W = hw_out(h, w, scale)
    return {"workload": name, "frames_per_clip": frames, "clips": world, "lr": [h, w], "hr": [H, W], "scale": list(scale),
            "weights": "random init (seed 0)", "parallelism": f"frame-sharded x{world}, no data-path collective",
            # timing rule "flush L2 or use inputs larger than L2": the latter (GPU arm; the CPU arm carries the same text so the objects stay equal)
            "l2": "no explicit flush: the per-step working set (16-bit activation arenas, several GB per clip) exceeds the 126 MB L2"}


DUMP_BYTES = 64 * 10 ** 6


def write_outputs(dirname, arrays):
    """--dump-outputs: write each tensor as float32 `dirname/<name>.npy`, at most DUMP_BYTES in all, so that two builds run with the
    same arguments can be compared output for output.  A tensor larger than its share of the budget is cut to a fixed sample of its
    rows along dim 0 (torch.randperm with seed 0, kept in ascending order)."""
    os.makedirs(dirname, exist_ok=True)
    import numpy as np
    share = DUMP_BYTES // len(arrays) - 4096                       # room for the .npy header
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() * 4 > share:
            keep = share // (t[0].numel() * 4)
            if keep == 0:
                raise ValueError(f"--dump-outputs: one row of {name} {tuple(t.shape)} is larger than its {share}-byte share")
            rows = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
            t = t[rows.to(t.device)]
        np.save(os.path.join(dirname, f"{name}.npy"), t.cpu().numpy())


class ClockSampler(threading.Thread):
    """SM clock / power / throttle reasons sampled while the timed region runs: NVML every 20 ms when `pynvml` imports,
    else one nvidia-smi call per 200 ms."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()   # rows: (sm MHz, max MHz, watts, {reasons})
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices; CUDA_VISIBLE_DEVICES may remap torch's index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n, h = self.nvml, self.handle
        sm = n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM)
        watts = n.nvmlDeviceGetPowerUsage(h) / 1e3
        try:
            mask = n.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        self.rows.append((float(sm), float(mx), watts, {name for name, bit in self.BITS if mask & bit}))

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        if out:
            r = [c.strip() for c in out.split(",")]
            names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
            self.rows.append((float(r[0]), float(r[1]), float(r[2]), {nm for nm, v in zip(names, r[3:7]) if v.lower().startswith("active")}))

    def run(self):
        while not self._stop_evt.is_set():
            try:
                if self.nvml is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            self._stop_evt.wait(0.02 if self.nvml is not None else 0.2)

    def stop(self) -> dict:
        self._stop_evt.set()
        self.join(timeout=6)
        sm = [r[0] for r in self.rows]
        reasons = set().union(*[r[3] for r in self.rows]) if self.rows else set()
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=max(r[1] for r in self.rows) if self.rows else None,
                    reasons=sorted(reasons), samples=len(sm), power_w_avg=round(statistics.median(r[2] for r in self.rows), 1) if self.rows else None,
                    source="nvml" if self.nvml is not None else "nvidia-smi")


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(bf16_sustained=d.get("bf16_tflops_sustained", 1418.2), bf16_burst=d.get("bf16_tflops", 1675.7),
                    hbm_gbs=d.get("hbm_gbs", 6543.7), source="measured")
    return dict(bf16_sustained=1400.0, bf16_burst=1590.0, hbm_gbs=6650.0, source="fallback")


# ------------------------------------------------------------------------------------------------ the reference itself
def load_reference(state_dict=None, device="cpu"):
    """The UNMODIFIED reference arch (lbasicsr/archs/savsr_arch.py) from baseline/_ref -- the offline install of /root/reference
    (`pip install --no-index --no-deps --target baseline/_ref`, git-ignored, travels to the GPU box).  Returns (module, "reference"),
    or (None, reason) when it is not installed / not importable."""
    ref_root = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_root, "lbasicsr")):
        return None, "baseline/_ref not installed"
    try:
        if ref_root not in sys.path:
            sys.path.insert(0, ref_root)
        import logging
        logging.disable(logging.INFO)
        from lbasicsr.archs import build_network               # lbasicsr/archs/__init__.py:19-28
        torch.manual_seed(0)
        ref = build_network(dict(type="SAVSR", **YAML_KWARGS)).eval()
        logging.disable(logging.NOTSET)
        if state_dict is not None:
            ref.load_state_dict({k: v.detach().cpu() for k, v in state_dict.items()}, strict=True)
        return ref.to(device), "reference"
    except Exception as e:  # noqa: BLE001 -- any import problem of the optional tree just selects the port
        return None, f"baseline/_ref not importable: {type(e).__name__}: {e}"


def cpu_reference_time(sd_cpu, frames, h, w, scale, threads=None):
    """Time the reference's CPU path on `frames` windows: the real reference when baseline/_ref is importable (kind
    "reference"), else the oracle port.  Returns (HR Mpix/s, seconds, threads, kind, output of the last window)."""
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    H, W = hw_out(h, w, scale)
    x = torch.rand(1, 7, 3, h, w, generator=torch.Generator().manual_seed(1234))
    ref, kind = load_reference(sd_cpu)
    if ref is not None:
        ref.set_scale(tuple(scale))
        run = lambda inp: ref(inp)                  # noqa: E731
    else:
        from oracle import savsr_oracle as O           # only the CPU-baseline legs of bench.py may touch oracle/
        kind = "port"
        run = lambda inp: O.forward(sd_cpu, inp, scale)   # noqa: E731
    with torch.no_grad():
        run(x[:, :, :, : min(h, 32), : min(w, 32)].contiguous())    # warm-up (thread pool, oneDNN primitives)
        t0 = time.perf_counter()
        for _ in range(frames):
            y = run(x)
        dt = time.perf_counter() - t0
    return frames * H * W / dt / 1e6, dt, threads, kind, y


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path on the host cores, rank 0 only."""
    if rank != 0:
        return
    import savsr_b200
    frames, h, w, scale = WORKLOADS[args.workload]
    torch.manual_seed(0)
    sd = {k: v.detach().clone() for k, v in savsr_b200.SAVSR().state_dict().items()}
    H, W = hw_out(h, w, scale)
    per_step = 1                                     # bounded sample: one output frame (one 7-frame window) per step
    for _ in range(min(args.warmup, 1)):
        cpu_reference_time(sd, 1, h, w, scale)
    t_total, n, kind, threads = 0.0, 0, "port", 1
    for _ in range(args.steps):
        _, dt, threads, kind, y = cpu_reference_time(sd, per_step, h, w, scale)
        t_total += dt; n += per_step
    if args.dump_outputs:
        write_outputs(args.dump_outputs, {"hr": y})
    val = n * H * W / t_total / 1e6
    what = ("the unmodified reference (baseline/_ref, lbasicsr/archs/savsr_arch.py) on CPU" if kind == "reference"
            else "oracle port of lbasicsr/archs/savsr_arch.py (pinned to the reference by tests/golden)")
    sample = f"{per_step} output frame(s) of the {args.workload} clip per step ({h}x{w} LR -> {H}x{W}), fp32, {threads} threads; {what}"
    print(json.dumps({
        "impl": "reference", "metric": "hr_mpix_per_s", "value": round(val, 5), "unit": "HR Mpix/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * t_total / args.steps, 2), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, args.gpus),
        "cpu_baseline": {"value": round(val, 5), "unit": "HR Mpix/s", "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": round(val, 5), "unit": "HR Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------------------------------ GPU-side reference
def vsr_runtime(fn, warm, reps):
    """lbasicsr/metrics/runtime.py:36-66: warm-up, then per repetition an event pair + synchronize, mean ms (fewer repetitions
    than the reference's 100 / 300 so that the default bench run stays short; stated in the output)."""
    with torch.no_grad():
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
    return sum(ts) / len(ts)


def gpu_reference(net, dev, h, w, scale, B):
    """The reference's own path on this GPU: the unmodified reference module (baseline/_ref) -- else the oracle port -- on CUDA
    with cudnn.benchmark = True (lbasicsr/test.py:15), TF32 convs on (PyTorch default = what the reference runs) and off."""
    H, W = hw_out(h, w, scale)
    sd = net.state_dict()
    ref, kind = load_reference(sd, dev)
    if ref is not None:
        ref.set_scale(tuple(scale))
        fwd = lambda x: ref(x)                       # noqa: E731
    else:
        from oracle import savsr_oracle as O            # device-aware restatement: the same ATen / cuDNN calls
        note = kind
        kind = "port"
        sd_dev = {k: v.detach().to(dev) for k, v in sd.items()}
        fwd = lambda x: O.forward(sd_dev, x, scale)  # noqa: E731
    out = {"kind": kind, "protocol": "VSR_runtime_test (lbasicsr/metrics/runtime.py:36-66) with 10 warm-up + 30 repetitions at b=1, "
                                     "2 + 3 at the batched size; cudnn.benchmark=True", "lr": [h, w], "hr": [H, W]}
    if ref is None:
        out["note"] = note
    saved = (torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32)
    torch.backends.cudnn.benchmark = True
    x1 = torch.rand(1, 7, 3, h, w, device=dev, generator=torch.Generator(device=dev).manual_seed(1234))
    xb = torch.rand(B, 7, 3, h, w, device=dev, generator=torch.Generator(device=dev).manual_seed(1235))
    try:
        for tf32 in (True, False):
            torch.backends.cudnn.allow_tf32 = tf32
            tag = "tf32" if tf32 else "fp32"
            ms1 = vsr_runtime(lambda: fwd(x1), 10, 30)
            out[f"b1_{tag}_ms"] = round(ms1, 3)
            out[f"b1_{tag}_hr_mpix_s"] = round(H * W / ms1 / 1e3, 2)
            try:
                msb = vsr_runtime(lambda: fwd(xb), 2, 3)
                out[f"b{B}_{tag}_ms"] = round(msb, 3)
                out[f"b{B}_{tag}_hr_mpix_s"] = round(B * H * W / msb / 1e3, 2)
            except torch.OutOfMemoryError as e:
                out[f"b{B}_{tag}_error"] = f"OOM: {str(e)[:80]}"
                torch.cuda.empty_cache()
        # parity against the reference's own GPU arithmetic with TF32 off (informational; the gate is the CPU oracle)
        torch.backends.cudnn.allow_tf32 = False
        with torch.no_grad():
            net.set_scale(scale)
            y_ref = fwd(x1)
            out["max_abs_ours_vs_gpu_reference_fp32"] = float((net(x1) - y_ref).abs().max())
    finally:
        torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32 = saved
        del ref
        torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------ BASELINE config 4, strong scaling
def run_cfg4(net, dev, rank, world, timed, steps=2, warmup=1, B=None):
    """10 UDM10-shaped clips x 32 frames at x4, FIXED total work, sharded rank-strided over the ranks exactly like the
    reference's loop (video_base_model.py:50: `for idx in range(rank, len(dataset), world_size)`), metrics on the device and
    the reference's reduction (`dist.reduce` of [n_frames, n_metrics], video_base_model.py:106-113) inside the timed region."""
    import torch.distributed as dist
    from savsr_b200 import postproc, sharding
    clips, T, h, w, scale = 10, 32, 180, 318, (4, 4)
    H, W = hw_out(h, w, scale)
    n_frames = clips * T
    mine = sharding.shard_frames(n_frames, rank, world)
    if B is None:
        # windows per forward: the largest of 40 / 16 / 8 that divides the shard (every launch has a fixed cost of a few microseconds, so
        # larger batches amortise it: +2.7 % from 17 to 34 Vid4 windows; 40 UDM10 windows = 11 GB of arena)
        B = next(b for b in (40, 16, 8) if len(mine) % b == 0)
    net.set_scale(scale)
    lr_all = torch.rand(n_frames, 3, h, w, generator=torch.Generator().manual_seed(4321)).to(dev)     # identical on every rank
    # 7-frame window of dataset item idx = frames of ITS clip with reflection padding at the clip ends (data_util.py:63-112)
    widx = torch.tensor([[(i // T) * T + t for t in sharding.frame_window_indices(i % T, T)] for i in mine], device=dev)
    gt = torch.rand(B, 3, H, W, device=dev, generator=torch.Generator(device=dev).manual_seed(99))   # synthetic ground truth, reused per batch
    local_out = torch.empty(len(mine), 3, H, W, device=dev)
    full_out = torch.empty(n_frames, 3, H, W, device=dev) if rank == 0 else None
    batches = [(a, min(a + B, len(mine))) for a in range(0, len(mine), B)]
    with torch.no_grad():
        plans = {b - a: net.plan_for(lr_all[widx[a:b].reshape(-1)].view(b - a, 7, 3, h, w)) for a, b in batches}
        for p in plans.values():
            p.capture()
    if len(mine) * world != n_frames or len(mine) % B:
        raise RuntimeError("cfg4: 320 frames must divide evenly over the ranks and into batches (1/2/4/8 ranks do)")
    n_local = len(mine)
    # rank 0 receives every batch of every rank into its own buffer (no reuse hazards), then assembles clip order:
    # global frame = rank + world * local index, i.e. full_out viewed as [n_local, world, ...]
    recv = torch.empty(len(batches), world, B, 3, H, W, device=dev) if (rank == 0 and world > 1) else None
    state = {}

    def step(gather):
        rows, works = [], []
        with torch.no_grad():
            for j, (a, b) in enumerate(batches):
                win = lr_all[widx[a:b].reshape(-1)].view(b - a, 7, 3, h, w)
                plans[b - a].forward_into(win, local_out[a:b])
                _, psnr = postproc.tensor2img_psnr(local_out[a:b], gt[:b - a], want_image=False)
                ssim = postproc.ssim_y(local_out[a:b], gt[:b - a])
                rows.append(torch.stack([psnr, ssim], 1).float())
                if gather and world > 1:      # this batch's frames travel to rank 0 while the next batch computes (NCCL's own stream)
                    works.append(dist.gather(local_out[a:b], list(recv[j].unbind(0)) if rank == 0 else None, dst=0, async_op=True))
                elif gather:
                    full_out[a:b].copy_(local_out[a:b], non_blocking=True)
            state["metrics"] = sharding.reduce_metrics(torch.cat(rows), mine, n_frames) if world > 1 else torch.cat(rows)
            for wk in works:
                wk.wait()
            if works and rank == 0:
                fo = full_out.view(n_local, world, 3, H, W)
                for j, (a, b) in enumerate(batches):
                    fo[a:b].copy_(recv[j].transpose(0, 1), non_blocking=True)
        torch.cuda.current_stream().synchronize()

    res = {}
    for gather in (False, True):
        for _ in range(warmup):
            step(gather)
        ms = timed(lambda: step(gather), steps)
        res["gather" if gather else "reduce"] = ms / steps
    mpix = n_frames * H * W / 1e6
    out = {"workload": "udm10_x4_10clips", "scaling": "strong", "frames": n_frames, "clips": clips, "lr": [h, w], "hr": [H, W],
           "scale": list(scale), "windows_per_forward": B, "frames_per_rank": len(mine), "steps": steps, "warmup": warmup,
           "sharding": "rank-strided frames (video_base_model.py:50), no data-path collective",
           "value": round(mpix / (res["reduce"] / 1e3), 2), "unit": "HR Mpix/s", "ms_per_step": round(res["reduce"], 3),
           "frames_per_s": round(n_frames / (res["reduce"] / 1e3), 2),
           "collective": f"dist.reduce of a [{n_frames}, 2] fp32 metric tensor to rank 0 ({n_frames * 2 * 4} bytes), inside the timed region",
           "with_gather": {"value": round(mpix / (res["gather"] / 1e3), 2), "unit": "HR Mpix/s", "ms_per_step": round(res["gather"], 3),
                           "collective": "dist.gather of every batch's HR frames to rank 0, asynchronous (overlaps the next batch), "
                                         "plus one strided copy per batch on rank 0",
                           "bytes_into_rank0": (world - 1) * n_local * 3 * H * W * 4,
                           "exposed_ms": round(res["gather"] - res["reduce"], 3)},
           "includes": "window gather, forward (CUDA graph), device tensor2img + PSNR-Y + SSIM-Y against a synthetic ground truth, the reduction"}
    if rank == 0 and world > 1:
        out["metrics_checksum"] = float(state["metrics"].double().sum())
    del plans
    net.release_plans()
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------ BASELINE config 5: training step
TRAIN_SCALES = [(2, 2), (3, 3), (4, 4), (1.5, 4), (2.7, 2.7), (1.1, 1.1), (3.5, 2), (4, 1.5)]    # a slice of the 60-entry list of vimeo90k_dataset.py:178-202


def run_train(args, rank, world, local_rank):
    """`--workload train_cfg5`: the optimisation step of lbasicsr/models/sr_model.py:101-128 on synthetic Vimeo90K-shaped batches
    (7 x 3 x 64 x 64 LR crops, 4 per GPU, one scale per step, data-parallel over the ranks with DistributedDataParallel / NCCL).
    Row f1 is staged: the 3x3 convolutions (forward, dgrad, wgrad) run on the tcgen05 kernels, the glue on ATen; the same step of
    the unmodified reference (cuDNN) is timed beside it when baseline/_ref is installed."""
    import torch.distributed as dist
    import savsr_b200
    from savsr_b200 import train as T
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    per_gpu, h, w = 4, 64, 64
    torch.manual_seed(0)
    net = savsr_b200.SAVSR().to(dev)
    native = args.train_engine == "native"
    torch.backends.cudnn.benchmark = os.environ.get("SAVSR_BENCH_CUDNN_BENCHMARK", "1") != "0"      # lbasicsr/train.py sets it; the ATen island's convs use it
    if native:
        # stage B: the static launch list of savsr_b200/trainplan.py (arena-resident forward / dgrad / batched wgrad, native attention
        # backward, flat Adam + EMA), one CUDA graph per scale; data parallelism = one NCCL all-reduce of the flat gradient buffer
        from savsr_b200 import trainplan as TP
        graph = not args.no_train_graph
        tr = TP.NativeTrainer(net, use_graph=graph, world_size=world)
    else:
        net.native_training = False                             # stage A: the ATen tape with the 3x3 convolutions on tcgen05 (savsr_b200/train.py)
        model = torch.nn.parallel.DistributedDataParallel(net, device_ids=[local_rank]) if world > 1 else net
        graph = world == 1 and not args.no_train_graph          # one CUDA graph per scale for the whole step (single process)
        tr = T.Trainer(model, use_graph=graph)
    gen = torch.Generator().manual_seed(100 + rank)
    lq_host = torch.rand(per_gpu, 7, 3, h, w, generator=gen).pin_memory()
    gts = {s: torch.rand(per_gpu, 3, *hw_out(h, w, s), generator=gen).pin_memory() for s in TRAIN_SCALES}

    def step(i):
        s = TRAIN_SCALES[i % len(TRAIN_SCALES)]
        loss = tr.step(lq_host.to(dev, non_blocking=True), gts[s].to(dev, non_blocking=True), s)
        return loss

    def timed_steps(fn, n):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        last = None
        for i in range(n):
            last = fn(i)
        e1.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), float(last)

    for i in range(max(max(args.warmup, 2), len(TRAIN_SCALES) if graph else 0)):      # with graphs: capture every scale before timing
        step(i)
    sampler = ClockSampler(local_rank); sampler.start()
    ms, loss = timed_steps(step, args.steps)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, {"loss": torch.tensor([loss]), "params": torch.cat([p.detach().flatten() for p in net.parameters()])})
    # the same step as the reference's loop sees it (sr_model.py:101-128 + the logger reading l_pix): batches from pinned host memory
    # (already the case above) and the loss value read back by the host EVERY step, which serialises host and device
    ms_e2e, _ = timed_steps(lambda i: float(step(i)), args.steps)
    line = {"metric": "train_samples_per_s", "value": round(per_gpu * world * args.steps / (ms / 1e3), 2), "unit": "samples/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 2), "ms_per_step": round(ms / args.steps, 2), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16 conv operands, fp32 master weights / accumulation", "data": "synthetic",
            "config": {"workload": "train_cfg5", "per_gpu_batch": per_gpu, "global_batch": per_gpu * world, "lr_crop": [h, w], "frames": 7,
                       "scales": [list(s) for s in TRAIN_SCALES], "optimizer": "Adam 2e-4 (0.9, 0.99), Charbonnier, EMA 0.999",
                       "l2": "no explicit flush: a step touches the plan's arenas (5.5 GB) and 300 MB of parameter / optimizer state, far beyond the 126 MB L2",
                       "parallelism": f"DistributedDataParallel x{world} (NCCL gradient all-reduce, 75.6 MB fp32)" if world > 1 else "single GPU"},
            "last_loss": round(loss, 5), "cuda_graph_per_scale": bool(graph), "engine": args.train_engine, "clocks": clocks,
            "e2e": {"value": round(per_gpu * world * args.steps / (ms_e2e / 1e3), 2), "unit": "samples/s", "ms_per_step": round(ms_e2e / args.steps, 2),
                    "h2d_bytes_per_step": int(lq_host.numel() * 4 + sum(g.numel() for g in gts.values()) * 4 // len(gts)), "d2h_bytes_per_step": 4,
                    "api": "NativeTrainer.step(lq, gt, scale) on pinned host batches, float(loss) read by the host every step"
                           if native else "train.Trainer.step(lq, gt, scale) on pinned host batches, float(loss) read by the host every step",
                    "note": "`value` feeds the same pinned host batches but reads the loss once at the end (the host runs ahead of the device)"}}
    # algorithmic work of a step: forward FLOPs of SURVEY 8d per sample, x3 for forward + data gradient + weight gradient (SURVEY 8d's own estimate)
    step_flops = sum(3.0 * flops_per_frame(h, w, *hw_out(h, w, TRAIN_SCALES[i % len(TRAIN_SCALES)])) * per_gpu * world for i in range(args.steps))
    line["algorithmic_tflops"] = round(step_flops / (ms / 1e3) / 1e12, 1)
    line["algorithmic_tflop_per_step"] = round(step_flops / args.steps / 1e12, 3)
    line["note_small_shapes"] = ("4 x 64 x 64 crops are 128 output tiles per convolution: one to six tiles per CTA on 148 SMs, ~1 400 launches of a few "
                                 "microseconds each -- the step is launch-latency bound, not tensor bound (DESIGN.md section 9)")
    if native:
        plan = next(iter(tr.plans.values()))
        line["config"]["parallelism"] = (f"data parallel x{world}: one NCCL all-reduce of the flat fp32 gradient buffer ({tr.flat.n * 4 / 1e6:.1f} MB) per step"
                                         if world > 1 else "single GPU")
        line["stage"] = ("f1 stage B: static forward + backward launch list on the 16-bit NHWC arena (savsr_b200/trainplan.py): every trunk convolution "
                         "forward / dgrad / batched wgrad on tcgen05 with no layout conversion in between, OSA-Conv attention (train-mode BatchNorm) and "
                         "channel attention forward + backward native, OSAdapt mask net (train-mode BatchNorm) native, table-driven weight packing, flat Adam + EMA; "
                         "ATen island: SATU HR side + tail + loss")
        line["gpu_launches"] = args.steps * (plan.launches["fwd"] + plan.launches["bwd"])       # native launches + the island's estimate, timed region
        line["plan"] = {"launches_native_estimate": plan.launches, "arena_slots": plan.n_slots, "t_slots": plan.n_tslots, "plan_gb": round(plan.nbytes / 2 ** 30, 2)}
    else:
        line["stage"] = ("f1 stage A: 3x3 convs (fwd / dgrad / wgrad, 98 % of the FLOPs) on tcgen05 through savsr_b200.autograd.conv3x3, each call "
                         "still converting NCHW fp32 <-> the NHWC 16-bit arena; glue ops on ATen")
    if world == 1 and not args.no_extras:
        ref, kind = load_reference(net.state_dict(), dev)
        if ref is not None:
            ref.train()
            opt = torch.optim.Adam(ref.parameters(), lr=2e-4, betas=(0.9, 0.99))
            saved = torch.backends.cudnn.benchmark
            torch.backends.cudnn.benchmark = True

            def ref_step(i):
                s = TRAIN_SCALES[i % len(TRAIN_SCALES)]
                ref.set_scale(s)
                opt.zero_grad(set_to_none=True)
                out = ref(lq_host.to(dev, non_blocking=True))
                l = T.charbonnier(out, gts[s].to(dev, non_blocking=True))
                l.backward()
                opt.step()
                return l.detach()
            for i in range(len(TRAIN_SCALES)):
                ref_step(i)                                   # cudnn.benchmark autotunes per shape
            rms, rloss = timed_steps(ref_step, args.steps)
            torch.backends.cudnn.benchmark = saved
            line["gpu_reference"] = {"kind": kind, "ms_per_step": round(rms / args.steps, 2), "samples_per_s": round(per_gpu * args.steps / (rms / 1e3), 2),
                                     "what": "the unmodified reference module in train mode on this GPU (cuDNN TF32 fprop / dgrad / wgrad, cudnn.benchmark), same step"}
        else:
            line["gpu_reference"] = {"unavailable": kind}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps of the headline, e2e, streamed, pipeline, other_scales and train_cfg5 "
                    "measurements; cfg4_strong (2 steps), latency_b1 and gpu_reference (their own repetition counts) state theirs in the output")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="vid4_x4", choices=sorted(WORKLOADS) + ["train_cfg5"])
    ap.add_argument("--batch", type=int, default=34, help="windows per forward (resident measurement; 34 = the whole Vid4-shaped clip)")
    ap.add_argument("--e2e-batches", default="26,8", help="batch schedule of the host-buffer (e2e) leg: a large forward, then a short one whose "
                    "device-to-host copy is the only one that cannot overlap compute")
    ap.add_argument("--conv-impl", default=os.environ.get("SAVSR_CONV_IMPL", "halo"), choices=["halo", "tap"])
    ap.add_argument("--precision", default=os.environ.get("SAVSR_PRECISION", "bf16"), choices=["bf16", "fp16"],
                    help="16-bit operand format (fp32 accumulate): bf16 = throughput path, fp16 = <=1e-3 max-abs path, same speed")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip fp16 / latency / gpu_reference / cfg4 legs (profiling runs)")
    ap.add_argument("--no-cfg4", action="store_true")
    ap.add_argument("--train-engine", default="native", choices=["native", "autograd"],
                    help="train_cfg5: native = savsr_b200.trainplan (static launch list, stage B); autograd = savsr_b200.train.Trainer (stage A)")
    ap.add_argument("--no-train-graph", action="store_true", help="train_cfg5: issue the step eagerly instead of replaying one CUDA graph per scale")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the timed path computed in its last step as "
                    "DIR/<name>.npy (float32, at most 64 MB in all; rank 0's arrays): hr = the HR frames (a fixed sample of them when the clip "
                    "is larger), or for train_cfg5 loss and params (a fixed sample of the updated parameters; its weight gradients are summed "
                    "with fp32 atomics, so two runs agree to rounding amplified by Adam, about lr per step, not bit for bit).  For comparing two builds of "
                    "one arm: --impl reference writes the output of its single timed window (input seed 1234), not frames of our arm's clip "
                    "(seed 1234 + rank)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        if args.workload == "train_cfg5":
            raise SystemExit("--impl reference is defined for the inference workloads (the metric of BASELINE.json)")
        run_reference(args, rank, world)
        return
    if args.workload == "train_cfg5":
        if not torch.cuda.is_available():
            raise SystemExit("bench.py --workload train_cfg5 needs a CUDA device (sm_100a); there is no CPU fallback")
        run_train(args, rank, world, local_rank)
        return

    import torch.distributed as dist
    import savsr_b200
    from savsr_b200 import sharding

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (sm_100a); there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, f"launched with WORLD_SIZE={world} but --gpus {args.gpus}"

    frames, h, w, scale = WORKLOADS[args.workload]
    H, W = savsr_b200.get_HW(h, w, scale)
    torch.manual_seed(0)                                   # random-init weights of the shipped architecture
    net = savsr_b200.SAVSR().to(dev).eval()
    net.conv_impl = args.conv_impl
    net.precision = args.precision
    net.set_scale(scale)
    B = min(args.batch, frames)
    e2e_batches = tuple(min(int(b), frames) for b in args.e2e_batches.split(","))

    # synthetic clip (one per rank), U[0,1) fp32; pinned host copy for the e2e leg
    gen = torch.Generator().manual_seed(1234 + rank)
    clip_host = torch.rand(frames, 3, h, w, generator=gen).pin_memory()
    out_host = torch.empty(frames, 3, H, W).pin_memory()
    windows = sharding.gather_windows(clip_host.to(dev), list(range(frames)))   # [frames, 7, 3, h, w] resident in HBM
    out_dev = torch.empty(frames, 3, H, W, device=dev)
    batches = [(i, min(i + B, frames)) for i in range(0, frames, B)]

    def build_plans():
        plans = {}
        with torch.no_grad():
            for (a, b) in batches:
                if b - a not in plans:
                    plan = net.plan_for(windows[a:b])
                    plan.x_in.copy_(windows[a:b]); plan.capture()
                    plans[b - a] = plan
        return plans
    plans = build_plans()
    launches_per_step = sum(plans[b - a].n_launches for a, b in batches)

    def step_resident():
        for (a, b) in batches:
            p = plans[b - a]
            p.x_in.copy_(windows[a:b], non_blocking=True)
            p.run_graph()
            out_dev[a:b].copy_(p.out, non_blocking=True)

    def step_e2e():
        # public API, host buffers: H2D of the LR clip, window gather + forward per batch, D2H of the HR frames
        clip = clip_host.to(dev, non_blocking=True)
        with torch.no_grad():
            sharding.infer_clip(net, clip, batch=e2e_batches, out=out_host)      # D2H of batch i overlaps the forward of batch i+1
        torch.cuda.current_stream().synchronize()

    # the same through-the-API measurement for a STREAM of clips: no host synchronisation per clip, two host output buffers in rotation, one
    # copy stream; every clip's H2D and D2H still happen inside the timed region, the last clip's copy is waited for before the clock stops
    out_host2 = torch.empty(frames, 3, H, W).pin_memory()
    pipe_state = {"i": 0, "copy": torch.cuda.Stream(dev)}

    def step_e2e_stream():
        clip = clip_host.to(dev, non_blocking=True)
        buf = out_host if pipe_state["i"] % 2 == 0 else out_host2
        pipe_state["i"] += 1
        with torch.no_grad():
            sharding.infer_clip(net, clip, batch=B, out=buf, copy_stream=pipe_state["copy"], join=False)

    # reference test loop on the device (rows f2 + f3): uint8 ground-truth frames in pinned host memory -> LR synthesis ->
    # windows -> net -> uint8 BGR images + PSNR-Y + SSIM-Y back in host memory (PNG decode / encode stay outside)
    from savsr_b200 import datapath
    pipeline_ok = datapath.as_mod_crop_size(H, W, scale) == (H, W) and datapath.lr_size(H, W, scale) == (h, w)
    if pipeline_ok:
        gt_u8_host = torch.randint(0, 256, (frames, H, W, 3), dtype=torch.uint8, generator=gen).pin_memory()
        img_host = torch.empty(frames, H, W, 3, dtype=torch.uint8).pin_memory()
        met_host = torch.empty(2, frames, dtype=torch.float64).pin_memory()

    def step_pipeline():
        gt_u8 = gt_u8_host.to(dev, non_blocking=True)
        with torch.no_grad():
            res = datapath.evaluate_clip(net, gt_u8, scale, batch=B)
        img_host.copy_(res["images"], non_blocking=True)
        met_host[0].copy_(res["psnr_y"], non_blocking=True)
        met_host[1].copy_(res["ssim_y"], non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    for _ in range(max(args.warmup, 3)):
        step_resident()
    sampler = ClockSampler(local_rank); sampler.start()
    ms_total = timed(step_resident, args.steps)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, {"hr": out_dev})
    for _ in range(2):
        step_e2e()
    ms_e2e = timed(step_e2e, args.steps)
    for _ in range(2):
        step_e2e_stream()
    torch.cuda.synchronize()

    def stream_steps():
        for _ in range(args.steps):
            step_e2e_stream()
        pipe_state["copy"].synchronize()
    ms_e2e_stream = timed(stream_steps, 1)
    ms_pipe = None
    if pipeline_ok:
        for _ in range(2):
            step_pipeline()
        ms_pipe = timed(step_pipeline, args.steps)

    mpix_step = frames * H * W / 1e6 * world
    value = mpix_step * args.steps / (ms_total / 1e3)
    e2e = mpix_step * args.steps / (ms_e2e / 1e3)

    # ---- rooflines, measured live (eager pass with a CUDA-event pair around every op on the launching stream)
    peaks = measured_peaks()
    big = plans[max(plans)]
    big.run_profiled()
    prof = big.run_profiled(detail=True)
    total_ms = sum(d["ms"] for d in prof.values())
    per_kind = {}
    for k, d in prof.items():
        e = per_kind.setdefault(k.split(":")[0], dict(ms=0.0, flops=0.0, launches=0))
        e["ms"] += d["ms"]; e["flops"] += d["flops"]; e["launches"] += d["launches"]
    conv = per_kind.get("conv3x3_n64", dict(ms=0.0, flops=0.0, launches=0))
    achieved = conv["flops"] / (conv["ms"] * 1e-3) / 1e12 if conv["ms"] else 0.0        # reproducible by hand from per_kind_ms
    # Cross-check: all conv launches of the forward replayed back to back as their own CUDA graph between one event pair (no lighter kernels in
    # between: the most power-hungry arrangement, so the clocks sit lowest; the per-op number above has the forward's own mix).
    conv_g = big.time_ops_graph(lambda kind, detail: kind == "conv3x3_n64")
    achieved_graph = conv_g["flops"] / (conv_g["ms"] * 1e-3) / 1e12 if conv_g["ms"] else 0.0
    osa_g = big.time_ops_graph(lambda kind, detail: kind == "conv3x3_n64" and detail.endswith("osa"))

    def traffic_of(fname):
        tpath = os.path.join(ROOT, "profiles", fname)
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            return tj.get("dram_bytes_per_launch"), f"ncu --set full, one launch: {tj.get('launch')} ({tj.get('source')})"
        return None, None
    traffic, traffic_note = traffic_of("conv_traffic.json")
    roofline = {"bound": "tensor", "kernel": "conv_igemm_bigk_kernel (tcgen05 implicit-GEMM 3x3 conv, N = 64; all launches of one forward)",
                "achieved": round(achieved, 1), "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                "frac": round(achieved / peaks["bf16_sustained"], 4), "peak_source": peaks["source"] + " bf16 sustained",
                "frac_of_burst_peak": round(achieved / peaks["bf16_burst"], 4),
                "flops_counted": "algorithmic: 2 * px * 64 * 9 * Ci per conv and sample with the reference's Ci (3 / 6 for the first layer, not the "
                                 "64 of the zero-expanded filters)",
                "algorithmic_tflop_per_forward": round(conv["flops"] / 1e12, 3),
                "traffic": traffic, "traffic_note": traffic_note, "share_of_step": round(conv["ms"] / total_ms, 3) if total_ms else None,
                "launches": conv["launches"], "avg_launch_us": round(1e3 * conv["ms"] / max(conv["launches"], 1), 1),
                "method": "eager forward of %d windows with a CUDA-event pair around every op on the launching stream; achieved = algorithmic FLOPs of "
                          "the N = 64 3x3 conv launches / their summed time (per_kind_ms.conv3x3_n64)" % big.B,
                "back_to_back_graph": {"achieved": round(achieved_graph, 1), "frac": round(achieved_graph / peaks["bf16_sustained"], 4),
                                       "conv_ms": round(conv_g["ms"], 3),
                                       "note": "the same launches replayed as one CUDA graph of convolutions only (Plan.time_ops_graph), one event pair"},
                "per_kind_ms": {k: round(v["ms"], 3) for k, v in sorted(per_kind.items(), key=lambda kv: -kv[1]["ms"])},
                "per_conv_shape": {k: {"ms": round(d["ms"], 3), "tflops": round(d["flops"] / (d["ms"] * 1e-3) / 1e12, 1), "launches": d["launches"]}
                                   for k, d in sorted(prof.items()) if k.startswith("conv3x3_n64") and d["ms"] > 0}}
    osa = [d for k, d in prof.items() if k.startswith("conv3x3_n64") and k.endswith("osa")]
    osa_ms, osa_fl, osa_n = sum(d["ms"] for d in osa), sum(d["flops"] for d in osa), sum(d["launches"] for d in osa)
    osa_ms_graph = osa_g["ms"]                                                         # the OSA-Conv launches as their own CUDA graph (cross-check)
    pro = per_kind.get("osa_prologue", dict(ms=0.0))
    roofline_osa = {"bound": "tensor", "kernel": "OSA-Conv launches only (per-sample folded weights, savsr_arch.py:139-172)",
                    "achieved": round(osa_fl / (osa_ms * 1e-3) / 1e12, 1) if osa_ms else None, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                    "frac": round(osa_fl / (osa_ms * 1e-3) / 1e12 / peaks["bf16_sustained"], 4) if osa_ms else None,
                    "frac_of_burst_peak": round(osa_fl / (osa_ms * 1e-3) / 1e12 / peaks["bf16_burst"], 4) if osa_ms else None,
                    "launches": osa_n, "conv_ms": round(osa_ms, 3), "conv_ms_back_to_back_graph": round(osa_ms_graph, 3), "prologue_ms": round(pro["ms"], 3),
                    "frac_including_prologue": round(osa_fl / ((osa_ms + pro["ms"]) * 1e-3) / 1e12 / peaks["bf16_sustained"], 4) if osa_ms else None}
    nb = big.B
    satu_ms = sum(per_kind[k]["ms"] for k in SATU_KINDS if k in per_kind)
    satu_bytes = satu_compulsory_bytes(h, w, H, W) * nb + 0.49e6
    satu_fl = satu_flops_per_frame(h, w, H, W) * nb
    extra = getattr(big, "satu_extra_bytes_per_sample", None)
    s_traffic, s_note = traffic_of("satu_traffic.json")
    roofline_satu = {"bound": "hbm", "kernels": [k for k in SATU_KINDS if k in per_kind],
                     "ms_per_launch_set": round(satu_ms, 3), "us_per_frame": round(1e3 * satu_ms / nb, 2),
                     "achieved": round(satu_bytes / (satu_ms * 1e-3) / 1e9, 1) if satu_ms else None, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                     "frac": round(satu_bytes / (satu_ms * 1e-3) / 1e9 / peaks["hbm_gbs"], 4) if satu_ms else None,
                     "compulsory_bytes_per_frame": satu_compulsory_bytes(h, w, H, W),
                     "declared_extra_bytes_per_frame": extra,
                     "compute": {"achieved": round(satu_fl / (satu_ms * 1e-3) / 1e12, 1) if satu_ms else None, "peak": peaks["bf16_sustained"],
                                 "unit": "TFLOP/s", "frac": round(satu_fl / (satu_ms * 1e-3) / 1e12 / peaks["bf16_sustained"], 4) if satu_ms else None},
                     "traffic": s_traffic, "traffic_note": s_note,
                     "caveat": "SATU carries ~1 180 FLOP per compulsory byte, so under this byte count it is compute-bound: 70 % of HBM would "
                               "mean ~4 us/frame (SURVEY.md D7); both fractions are printed"}
    whole = flops_per_frame(h, w, H, W) * frames * world * args.steps / (ms_total / 1e3) / 1e12

    cfg = workload_config(args.workload, world)
    line = {
        "metric": "hr_mpix_per_s", "value": round(value, 2), "unit": "HR Mpix/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": round(ms_total / args.steps, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
        "config": cfg,
        "run": {"windows_per_forward": B, "conv_impl": args.conv_impl,
                "l2": "per-step working set (activation arenas, several GB) exceeds the 126 MB L2; no explicit flush"},
        "frames_per_s": round(frames * world * args.steps / (ms_total / 1e3), 2),
        "whole_forward_tflops": round(whole, 1),
        "e2e": {"value": round(e2e, 2), "unit": "HR Mpix/s", "ms_per_step": round(ms_e2e / args.steps, 3),
                "h2d_bytes_per_step": clip_host.numel() * 4, "d2h_bytes_per_step": out_host.numel() * 4,
                "api": "savsr_b200.sharding.infer_clip(savsr_b200.SAVSR, clip, batch=%s)" % (list(e2e_batches),),
                "batches": list(e2e_batches),
                "note": "synchronous: the host waits for every clip's frames before it submits the next clip",
                "streamed": {"value": round(mpix_step * args.steps / (ms_e2e_stream / 1e3), 2), "unit": "HR Mpix/s", "ms_per_step": round(ms_e2e_stream / args.steps, 3),
                             "what": "the same API on a stream of clips (infer_clip(..., batch=%d, copy_stream=s, join=False)): two pinned output buffers in rotation, no "
                                     "host synchronisation per clip, the clock stops when the last clip's frames are in host memory" % B}},
        "pipeline": None if ms_pipe is None else {
            "value": round(mpix_step * args.steps / (ms_pipe / 1e3), 2), "unit": "HR Mpix/s", "ms_per_step": round(ms_pipe / args.steps, 3),
            "h2d_bytes_per_step": frames * H * W * 3, "d2h_bytes_per_step": frames * H * W * 3 + 16 * frames,
            "api": "savsr_b200.datapath.evaluate_clip(net, uint8 GT frames, scale)",
            "what": "the reference test loop minus the PNG codec: uint8 GT frames in pinned host memory -> as_mod_crop + antialiased "
                    "bicubic LR synthesis -> windows -> net -> uint8 BGR images, PSNR-Y and SSIM-Y back in host memory"},
        "gpu_launches": launches_per_step * args.steps * world,
        "clocks": clocks,
        "roofline": roofline,
        "roofline_osa": roofline_osa,
        "roofline_satu": roofline_satu,
    }

    extras = not args.no_extras
    if extras and world == 1:
        # ---- the fp16-operand path (meets the fp32 criterion), same resident measurement
        other = "fp16" if args.precision == "bf16" else "bf16"
        net.precision = other
        plans_main, plans = plans, None
        plans = build_plans()
        for _ in range(3):
            step_resident()
        ms_o = timed(step_resident, args.steps)
        line[other] = {"value": round(mpix_step * args.steps / (ms_o / 1e3), 2), "unit": "HR Mpix/s", "ms_per_step": round(ms_o / args.steps, 3),
                       "dtype": other, "note": "same kernels, 16-bit operands in the other format, fp32 accumulate; fp16 meets max-abs <= 1e-3 "
                                               "against the fp32 reference (tests/test_gpu_forward.py)"}
        net.precision = args.precision
        plans = plans_main
        # ---- BASELINE configs[2]: the asymmetric and the non-integer scale on the same clip (the trunk is scale independent: frames/s stays,
        #      HR Mpix/s follows the scale product; SATU's index path is bit-exact at these scales: tests/test_gpu_kernels.py)
        if args.workload == "vid4_x4":
            line["other_scales"] = {}
            for tag, s2 in (("x1.5x4", (1.5, 4)), ("x2.7", (2.7, 2.7))):
                net.set_scale(s2)
                H2, W2 = savsr_b200.get_HW(h, w, s2)
                with torch.no_grad():
                    p2 = net.plan_for(windows[:B])
                    p2.x_in.copy_(windows[:B]); p2.capture()
                for _ in range(3):
                    p2.run_graph()
                ms2 = timed(p2.run_graph, args.steps)
                line["other_scales"][tag] = {"scale": list(s2), "hr": [H2, W2], "value": round(B * H2 * W2 * args.steps / (ms2 / 1e3) / 1e6, 2), "unit": "HR Mpix/s",
                                             "frames_per_s": round(B * args.steps / (ms2 / 1e3), 2), "ms_per_forward": round(ms2 / args.steps, 3),
                                             "windows_per_forward": B}
                p2 = None
        # ---- one window per call through the module (what lbasicsr/test.py does, video_base_model.py:50-59)
        net.set_scale(scale)
        x1 = windows[:1].clone()
        with torch.no_grad():
            net(x1)
            first_build = net.last_plan_build_ms
            s2 = (scale[0] - 0.1, scale[1] - 0.1)
            net.set_scale(s2); net(x1)
            next_build = net.last_plan_build_ms
            net.set_scale(scale)
        ms_b1 = vsr_runtime(lambda: net(x1), 10, 30)
        line["latency_b1"] = {"ms": round(ms_b1, 3), "hr_mpix_s": round(H * W / ms_b1 / 1e3, 2), "api": "SAVSR.forward(x[1,7,3,h,w]) incl. plan lookup, "
                              "input staging, CUDA-graph replay and a fresh output tensor", "protocol": "10 warm-up + 30 repetitions, event pair + synchronize each",
                              "plan_build_ms": {"first_plan_b1": round(first_build, 1), "next_scale_b1": round(next_build, 1),
                                                "note": "packed weights / folded BN are shared across plans of one weights version"}}
        try:
            line["gpu_reference"] = gpu_reference(net, dev, h, w, scale, B)
            g = line["gpu_reference"]
            if f"b{B}_tf32_hr_mpix_s" in g:
                g["speedup_resident_vs_tf32_batched"] = round(value / g[f"b{B}_tf32_hr_mpix_s"], 2)
            g["speedup_b1_vs_tf32"] = round(g["b1_tf32_ms"] / ms_b1, 2)
        except Exception as e:  # noqa: BLE001
            line["gpu_reference"] = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
    if extras and not args.no_cfg4:
        plans = None
        big = None
        net.release_plans()
        torch.cuda.empty_cache()
        try:
            line["cfg4_strong"] = run_cfg4(net, dev, rank, world, timed)
        except Exception as e:  # noqa: BLE001
            line["cfg4_strong"] = {"error": f"{type(e).__name__}: {str(e)[:300]}"}

    if rank == 0 and not args.no_cpu_baseline and world == 1:
        sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
        n_cpu = 3
        val, dt, threads, kind, _ = cpu_reference_time(sd, n_cpu, h, w, scale)
        line["cpu_baseline"] = {"value": round(val, 5), "unit": "HR Mpix/s", "cores": threads, "kind": kind,
                                "sample": f"{n_cpu} output frames of the same clip shape ({h}x{w} -> {H}x{W}), fp32, {dt:.1f} s; "
                                          + ("the unmodified reference (baseline/_ref)" if kind == "reference" else "oracle port")}
    elif rank == 0:
        line["cpu_baseline"] = None
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
