"""Streaming 8-bit video (savsr_b200.VideoUpscaler) against the whole-clip driver, bf16, random-init weights (seed 0), seeded uint8
frames.  Vid4-shaped clip (34 frames, 144x180 -> 576x720 at x4, batch schedule (26, 8)); every shape warmed up first; three arms
timed alternately, host clock around --steps clips ending in a device synchronise:

  resident  infer_clip(net.forward_bgr_u8, clip on the device, batch=(26, 8)), results left on the device
  pinned    pinned uint8 clip -> infer_clip(net.forward_bgr_u8, ..., out=pinned uint8): bench_video_io.py's u8 arm
  stream    VideoUpscaler fed one frame at a time from pinned host memory; the caller copies each returned batch to pinned host
            memory on a side stream

The stream's output is checked byte for byte against infer_clip's.  Long-stream arm: --long-frames frames (default 2 000) at
270x480 -> 1080x1920 (x4), batch 26, fed one frame at a time from pinned host memory (a cycle of 32 distinct frames), outputs left on
the device: HR Mpix/s, and torch.cuda.max_memory_allocated after 500 frames and after the last one.  Also the card's name and power
limit, read in the same run.  Writes the JSON to --out (default profiles/r03_video_stream.json) and prints it.
Usage: python scripts/bench_video_stream.py --steps 20 --rounds 3
"""
import argparse
import json
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from scripts.bench_train_shape import gpu_identity  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="clips per timed window")
    ap.add_argument("--rounds", type=int, default=3, help="alternating rounds over the arms")
    ap.add_argument("--long-frames", type=int, default=2000, help="frames of the long stream")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_video_stream.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_video_stream.py measures on a CUDA device; none found")
    import savsr_b200
    from savsr_b200 import sharding

    dev = torch.device("cuda", 0)
    T, h, w, scale, sched = 34, 144, 180, (4, 4), (26, 8)
    H, W = 4 * h, 4 * w
    torch.manual_seed(0)
    net = savsr_b200.SAVSR().to(dev).eval()
    net.set_scale(scale)
    net.precision = "bf16"
    gen = torch.Generator().manual_seed(1)
    clip_host = torch.randint(0, 256, (T, h, w, 3), dtype=torch.uint8, generator=gen).pin_memory()
    clip_dev = clip_host.to(dev)
    out_clip = torch.empty(T, H, W, 3, dtype=torch.uint8).pin_memory()
    out_stream = torch.empty(T, H, W, 3, dtype=torch.uint8).pin_memory()
    copy_stream = torch.cuda.Stream(dev)
    up = savsr_b200.VideoUpscaler(net, (h, w), scale, batch=sched)

    def arm_resident():
        return sharding.infer_clip(net.forward_bgr_u8, clip_dev, batch=sched)

    def arm_pinned():
        return sharding.infer_clip(net.forward_bgr_u8, clip_host.to(dev, non_blocking=True), batch=sched, out=out_clip)

    def arm_stream():
        up.reset()
        cur = torch.cuda.current_stream(dev)

        def take(batches):
            for s, hr in batches:
                copy_stream.wait_stream(cur)
                with torch.cuda.stream(copy_stream):
                    out_stream[s:s + hr.shape[0]].copy_(hr, non_blocking=True)
                hr.record_stream(copy_stream)
        for k in range(T):
            take(up.push(clip_host[k]))
        take(up.finish())
        cur.wait_stream(copy_stream)
        return out_stream

    arms = {"resident": arm_resident, "pinned": arm_pinned, "stream": arm_stream}
    with torch.no_grad():
        for fn in arms.values():                         # builds and captures the plans of both I/O modes, both batch sizes
            fn(); fn()
        torch.cuda.synchronize()
        want = arm_resident().cpu()
        arm_stream()
        torch.cuda.synchronize()
        identical = bool(torch.equal(out_stream, want))
        assert identical, "VideoUpscaler differs from infer_clip(net.forward_bgr_u8)"

        ms = {k: [] for k in arms}
        for _ in range(args.rounds):
            for name, fn in arms.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(args.steps):
                    fn()
                torch.cuda.synchronize()
                ms[name].append(1e3 * (time.perf_counter() - t0) / args.steps)

        # ---- long stream
        lh, lw, lb, n_long = 270, 480, 26, args.long_frames
        LH, LW = 4 * lh, 4 * lw
        src = torch.randint(0, 256, (32, lh, lw, 3), dtype=torch.uint8, generator=gen).pin_memory()
        long_up = savsr_b200.VideoUpscaler(net, (lh, lw), scale, batch=lb)

        def long_stream(n, mark=None):
            long_up.reset()
            peak_at_mark = None
            for k in range(n):
                for _, hr in long_up.push(src[k % 32]):
                    del hr
                if mark is not None and k + 1 == mark:
                    peak_at_mark = torch.cuda.max_memory_allocated(dev)
            for _, hr in long_up.finish():
                del hr
            return peak_at_mark

        long_stream(lb + (n_long % lb or lb))            # warm-up: the plans of the full batch and of the stream's last batch
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(dev)
        t0 = time.perf_counter()
        peak_500 = long_stream(n_long, mark=500)
        torch.cuda.synchronize()
        long_s = time.perf_counter() - t0
        peak_end = torch.cuda.max_memory_allocated(dev)

    mpix = T * H * W / 1e6
    res = {k: {"ms_per_clip_median": round(statistics.median(v), 3), "ms_per_clip_all": [round(x, 3) for x in v],
               "hr_mpix_per_s": round(mpix / (statistics.median(v) / 1e3), 1)} for k, v in ms.items()}
    lr_px, win_px = T * h * w * 3, T * 7 * h * w * 3
    out = {"gpu": gpu_identity(0),
           "clip": {"frames": T, "lr": [h, w], "hr": [H, W], "scale": scale, "batch_schedule": sched, "precision": "bf16",
                    "weights": "random init, torch.manual_seed(0)"},
           "steps": args.steps, "rounds": args.rounds, "stream_equals_infer_clip": identical, "arms": res,
           "input_bytes_per_clip": {"frames": lr_px, "windows_gathered_by_infer_clip": win_px},
           "stream_ring": {"frames": up.capacity, "bytes": up.ring.numel()},
           "long_stream": {"frames": n_long, "lr": [lh, lw], "hr": [LH, LW], "batch": lb, "feed": "one pinned host frame per push",
                           "outputs": "left on the device", "seconds": round(long_s, 3),
                           "hr_mpix_per_s": round(n_long * LH * LW / 1e6 / long_s, 1),
                           "ring_frames": long_up.capacity, "ring_bytes": long_up.ring.numel(),
                           "max_memory_allocated_after_500": peak_500, "max_memory_allocated_after_all": peak_end}}
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
