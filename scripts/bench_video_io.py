"""8-bit video I/O against the fp32 path on the Vid4-shaped clip (34 frames, 144x180 -> 576x720 at x4), bf16, random-init weights
(seed 0), a seeded uint8 clip.  Three arms in one process, every shape warmed up first, timed alternately:

  f32          pinned fp32 clip -> infer_clip(net, ..., batch=(26, 8), out=pinned fp32): what bench.py's e2e leg does
  f32_then_u8  the same windows through net, then postproc.tensor2img_psnr per batch, then a uint8 device-to-host copy: the best a
               caller could do before forward_bgr_u8
  u8           pinned uint8 clip -> infer_clip(net.forward_bgr_u8, ..., batch=(26, 8), out=pinned uint8)

Each arm is timed twice: from/to pinned host buffers (host clock around --steps clips, ending in a device synchronise) and
HBM-resident (clip on the device, results left there).  Also: satu_hr / pack_frames device ms of both I/O modes from
Plan.run_profiled(), the bytes each arm moves (computed from the shapes), the card's name and power limit, and a byte-for-byte
comparison of the f32_then_u8 and u8 outputs.  Writes the JSON to --out (default profiles/r03_video_u8_io.json) and prints it.
Usage: python scripts/bench_video_io.py --steps 20 --rounds 3
"""
import argparse
import json
import os
import statistics
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from scripts.bench_train_shape import gpu_identity  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="clips per timed window")
    ap.add_argument("--rounds", type=int, default=3, help="alternating rounds over the arms")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_video_u8_io.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_video_io.py measures on a CUDA device; none found")
    import savsr_b200
    from savsr_b200 import postproc, sharding

    dev = torch.device("cuda", 0)
    T, h, w, scale, sched = 34, 144, 180, (4, 4), (26, 8)
    H, W = 4 * h, 4 * w
    torch.manual_seed(0)
    net = savsr_b200.SAVSR().to(dev).eval()
    net.set_scale(scale)
    net.precision = "bf16"
    gen = torch.Generator().manual_seed(1)
    clip_u8_host = torch.randint(0, 256, (T, h, w, 3), dtype=torch.uint8, generator=gen).pin_memory()
    table = torch.from_numpy(np.arange(256, dtype=np.float32) / np.float32(255))          # the reference's u / 255
    clip_f32_host = table[clip_u8_host.long()].flip(-1).permute(0, 3, 1, 2).contiguous().pin_memory()
    out_f32_host = torch.empty(T, 3, H, W).pin_memory()
    out_u8_host = torch.empty(T, H, W, 3, dtype=torch.uint8).pin_memory()
    out_u8_host2 = torch.empty(T, H, W, 3, dtype=torch.uint8).pin_memory()
    clip_u8_dev, clip_f32_dev = clip_u8_host.to(dev), clip_f32_host.to(dev)

    def to_img(x):
        return postproc.tensor2img_psnr(net(x))[0]

    def arm_f32(host):
        clip = clip_f32_host.to(dev, non_blocking=True) if host else clip_f32_dev
        return sharding.infer_clip(net, clip, batch=sched, out=out_f32_host if host else None)

    def arm_f32_then_u8(host):
        clip = clip_f32_host.to(dev, non_blocking=True) if host else clip_f32_dev
        return sharding.infer_clip(to_img, clip, batch=sched, out=out_u8_host2 if host else None)

    def arm_u8(host):
        clip = clip_u8_host.to(dev, non_blocking=True) if host else clip_u8_dev
        return sharding.infer_clip(net.forward_bgr_u8, clip, batch=sched, out=out_u8_host if host else None)

    arms = {"f32": arm_f32, "f32_then_u8": arm_f32_then_u8, "u8": arm_u8}
    with torch.no_grad():
        for fn in arms.values():                         # builds and captures every plan of both modes, both batch sizes
            for host in (True, False):
                fn(host); fn(host)
        torch.cuda.synchronize()
        identical_dev = bool(torch.equal(arm_f32_then_u8(False), arm_u8(False)))
        arm_f32_then_u8(True); arm_u8(True)
        torch.cuda.synchronize()
        identical_host = bool(torch.equal(out_u8_host, out_u8_host2))
        assert identical_dev and identical_host, "forward_bgr_u8 differs from tensor2img of the fp32 forward"

        ms = {f"{k}_{m}": [] for k in arms for m in ("host", "resident")}
        for _ in range(args.rounds):
            for name, fn in arms.items():
                for host in (True, False):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    for _ in range(args.steps):
                        fn(host)
                    torch.cuda.synchronize()
                    ms[f"{name}_{'host' if host else 'resident'}"].append(1e3 * (time.perf_counter() - t0) / args.steps)

        kernels = {}
        for io in ("f32", "bgr_u8"):
            for b in sched:
                x = sharding.gather_windows(clip_u8_dev if io == "bgr_u8" else clip_f32_dev, range(b))
                plan = net.plan_for(x, io=io)
                plan.run_profiled()                                                      # warm
                runs = [plan.run_profiled() for _ in range(5)]
                kernels[f"{io}_b{b}"] = {k: round(statistics.median(r[k]["ms"] for r in runs), 4) for k in ("satu_hr", "pack_frames")}

    mpix = T * H * W / 1e6
    res = {k: {"ms_per_clip_median": round(statistics.median(v), 3), "ms_per_clip_all": [round(x, 3) for x in v],
               "hr_mpix_per_s": round(mpix / (statistics.median(v) / 1e3), 1)} for k, v in ms.items()}
    lr_px, hr_px, win_px = T * h * w * 3, T * H * W * 3, T * 7 * h * w * 3
    bytes_moved = {
        "f32": {"h2d": 4 * lr_px, "windows_hbm": 4 * win_px, "satu_hr_store": 4 * hr_px, "d2h": 4 * hr_px},
        "f32_then_u8": {"h2d": 4 * lr_px, "windows_hbm": 4 * win_px, "satu_hr_store": 4 * hr_px, "tensor2img_read": 4 * hr_px,
                        "tensor2img_write": hr_px, "d2h": hr_px},
        "u8": {"h2d": lr_px, "windows_hbm": win_px, "satu_hr_store": hr_px, "d2h": hr_px},
    }
    out = {"gpu": gpu_identity(0), "clip": {"frames": T, "lr": [h, w], "hr": [H, W], "scale": scale, "batch_schedule": sched,
                                           "precision": "bf16", "weights": "random init, torch.manual_seed(0)"},
           "steps": args.steps, "rounds": args.rounds, "u8_equals_f32_then_u8": identical_dev and identical_host,
           "arms": res, "kernel_ms_run_profiled": kernels, "bytes_per_clip": bytes_moved}
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
