"""YUV 4:2:0 video through savsr_b200.VideoUpscaler: colour conversion on the host (today's way) against the device kernels, bf16,
random-init weights (seed 0), seeded frames.  Three arms, timed alternately in one process, host clock around whole streams ending in a
device synchronise, median of --rounds:

  host_cv2     a yuv420p host source: cv2 YUV->BGR per frame on the host, a bgr24 VideoUpscaler, each HR batch copied to pinned host
               memory, cv2 BGR->I420 per frame on the host (a batch is converted while the next one runs on the device)
  yuv420p      yuv420p -> yuv420p VideoUpscaler from the same pageable host frames; each HR batch copied to pinned host memory
  nv12_device  NV12 device frames with a 256-byte-aligned row pitch (a decoder's surfaces) -> NV12 device output, left on the device

Workloads: the Vid4 clip shape (34 frames, 144x180 -> 576x720 at x4, batch schedule (26, 8)), --steps clips per timed window; and the
270x480 -> 1080x1920 stream at x4, batch 26, --long-frames frames (a cycle of 32 distinct frames).  The arms' outputs are checked byte
for byte against each other on the Vid4 clip.  Also each conversion kernel on its own with CUDA events (decode at LR 270x480, encode at
HR 1080x1920, one frame and 26 frames per launch, replayed as a CUDA graph), cycling over buffers larger than the 126 MB L2, as bytes moved over time.  The card's
name and power limit are read in the same run.  Writes --out (default profiles/r03_video_yuv.json) and prints it.
Usage: python scripts/bench_video_yuv.py --steps 10 --rounds 3 --long-frames 520
"""
import argparse
import json
import os
import statistics
import sys
import time

import cv2
import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from scripts.bench_train_shape import gpu_identity  # noqa: E402

HBM_TBPS = 7.7      # NVIDIA HGX B200 data sheet, per GPU


class HostSink:
    """HR batches -> pinned host memory (double-buffered by batch), then optionally cv2 BGR -> I420 on the host, into dest[frame % len]."""

    def __init__(self, dev, max_batch, frame_shape, dest, convert):
        self.dev, self.dest, self.convert = dev, dest, convert
        self.bufs = [torch.empty((max_batch, *frame_shape), dtype=torch.uint8).pin_memory() for _ in range(2)]
        self.events = [torch.cuda.Event(), torch.cuda.Event()]
        self.pending = [None, None]
        self.k = 0

    def _drain(self, slot):
        if self.pending[slot] is None:
            return
        start, m = self.pending[slot]
        self.events[slot].synchronize()
        for i in range(m):
            f = self.bufs[slot][i].numpy()
            d = self.dest[(start + i) % len(self.dest)]
            if self.convert:
                cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420, dst=d)
            else:
                d[...] = f
        self.pending[slot] = None

    def take(self, batches):
        for start, hr in batches:
            slot = self.k % 2
            self._drain(slot)                     # the batch that used this buffer two batches ago
            self.bufs[slot][:hr.shape[0]].copy_(hr, non_blocking=True)
            self.events[slot].record(torch.cuda.current_stream(self.dev))
            self.pending[slot] = (start, hr.shape[0])
            self.k += 1
            self._drain(1 - slot)                 # the previous batch, while this one's copy and the next forward run

    def finish(self):
        self._drain(self.k % 2)
        self._drain(1 - self.k % 2)


def make_arms(savsr_b200, net, dev, h, w, scale, sched, yuv_host, nv12_dev, n_frames, dests):
    H, W = round(h * scale[0]), round(w * scale[1])
    mb = sched if isinstance(sched, int) else max(sched)
    ups = {"host_cv2": savsr_b200.VideoUpscaler(net, (h, w), scale, batch=sched),
           "yuv420p": savsr_b200.VideoUpscaler(net, (h, w), scale, batch=sched, in_format="yuv420p", out_format="yuv420p"),
           "nv12_device": savsr_b200.VideoUpscaler(net, (h, w), scale, batch=sched, in_format="nv12", out_format="nv12")}
    sinks = {"host_cv2": HostSink(dev, mb, (H, W, 3), dests["host_cv2"], convert=True),
             "yuv420p": HostSink(dev, mb, (3 * H // 2, W), dests["yuv420p"], convert=False)}
    src = yuv_host.numpy()
    S = len(src)

    def host_cv2():
        up = ups["host_cv2"]
        up.reset()
        sink = sinks["host_cv2"]
        for k in range(n_frames):
            sink.take(up.push(cv2.cvtColor(src[k % S], cv2.COLOR_YUV2BGR_I420)))
        sink.take(up.finish())
        sink.finish()

    def yuv420p():
        up = ups["yuv420p"]
        up.reset()
        sink = sinks["yuv420p"]
        for k in range(n_frames):
            sink.take(up.push(yuv_host[k % S]))
        sink.take(up.finish())
        sink.finish()

    def nv12_device():
        up = ups["nv12_device"]
        up.reset()
        outs = []
        for k in range(n_frames):
            outs += up.push(nv12_dev[k % S])
        outs += up.finish()
        dests["nv12_device"] = outs               # left on the device (an encoder taking device surfaces reads them there)

    return {"host_cv2": host_cv2, "yuv420p": yuv420p, "nv12_device": nv12_device}


def time_arms(arms, rounds, reps):
    ms = {k: [] for k in arms}
    for _ in range(rounds):
        for name, fn in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(reps):
                fn()
            torch.cuda.synchronize()
            ms[name].append(1e3 * (time.perf_counter() - t0) / reps)
    return ms


def kernel_times(colour, dev, reps=200):
    """Per-launch device time of each conversion kernel: `reps` launches in one CUDA graph, cycling over buffers of > 256 MB so each
    launch reads from HBM, not L2."""
    res = {}
    for name, (h, w, n, fmt, direction) in {
            "decode_yuv420p_lr_270x480_n1": (270, 480, 1, "yuv420p", "dec"),
            "decode_nv12_lr_270x480_n1": (270, 480, 1, "nv12", "dec"),
            "decode_yuv420p_lr_270x480_n26": (270, 480, 26, "yuv420p", "dec"),
            "encode_yuv420p_hr_1080x1920_n1": (1080, 1920, 1, "yuv420p", "enc"),
            "encode_nv12_hr_1080x1920_n1": (1080, 1920, 1, "nv12", "enc"),
            "encode_yuv420p_hr_1080x1920_n26": (1080, 1920, 26, "yuv420p", "enc")}.items():
        yuv_b, bgr_b = n * 3 * h * w // 2, n * 3 * h * w
        copies = max(2, -(-(256 << 20) // (yuv_b + bgr_b)))
        yuv = torch.randint(0, 256, (copies, n, 3 * h // 2, w), dtype=torch.uint8, device=dev)
        bgr = torch.randint(0, 256, (copies, n, h, w, 3), dtype=torch.uint8, device=dev)
        run = (lambda i: colour.yuv420_to_bgr(yuv[i], fmt, out=bgr[i])) if direction == "dec" else \
              (lambda i: colour.bgr_to_yuv420(bgr[i], fmt, out=yuv[i]))
        run(0)
        torch.cuda.synchronize(dev)
        g = torch.cuda.CUDAGraph()               # replayed as a graph, so the host's launch rate does not bound the kernels
        with torch.cuda.graph(g):
            for i in range(reps):
                run(i % copies)
        g.replay()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize(dev)
        us = 1e3 * e0.elapsed_time(e1) / reps
        moved = yuv_b + bgr_b
        res[name] = {"us_per_launch": round(us, 2), "bytes_moved": moved, "gb_per_s": round(moved / us / 1e3, 1),
                     "share_of_hbm_data_sheet": round(moved / us / 1e6 / HBM_TBPS, 3), "buffers_cycled": copies}
        del yuv, bgr
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10, help="Vid4 clips per timed window")
    ap.add_argument("--rounds", type=int, default=3, help="alternating rounds over the arms")
    ap.add_argument("--long-frames", type=int, default=520, help="frames of the 1080p-output stream")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_video_yuv.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_video_yuv.py measures on a CUDA device; none found")
    import savsr_b200
    from savsr_b200 import colour

    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    net = savsr_b200.SAVSR().to(dev).eval()
    net.precision = "bf16"
    gen = torch.Generator().manual_seed(1)
    out = {"gpu": gpu_identity(0), "precision": "bf16", "weights": "random init, torch.manual_seed(0)", "rounds": args.rounds}

    def sources(T, h, w, pitch):
        yuv = torch.randint(0, 256, (T, 3 * h // 2, w), dtype=torch.uint8, generator=gen)
        nv = yuv.clone()
        uv = yuv.reshape(T, -1)[:, h * w:].reshape(T, 2, h // 2, w // 2)      # the U plane, then the V plane
        nv[:, h:] = torch.stack([uv[:, 0], uv[:, 1]], -1).reshape(T, h // 2, w)
        surf = torch.zeros(T, 3 * h // 2, pitch, dtype=torch.uint8, device=dev)
        surf[:, :, :w] = nv.to(dev)
        return yuv, surf[:, :, :w]

    with torch.no_grad():
        # ---- Vid4 clip
        T, h, w, scale, sched = 34, 144, 180, (4, 4), (26, 8)
        H, W = 4 * h, 4 * w
        yuv_host, nv12_dev = sources(T, h, w, 256)
        dests = {"host_cv2": np.zeros((T, 3 * H // 2, W), np.uint8), "yuv420p": np.zeros((T, 3 * H // 2, W), np.uint8)}
        arms = make_arms(savsr_b200, net, dev, h, w, scale, sched, yuv_host, nv12_dev, T, dests)
        for fn in arms.values():
            fn(); fn()
        want = dests["host_cv2"]
        nv_want = want.copy()
        uv = want.reshape(T, -1)[:, H * W:].reshape(T, 2, H // 2, W // 2)
        nv_want[:, H:] = np.stack([uv[:, 0], uv[:, 1]], -1).reshape(T, H // 2, W)
        identical = {"yuv420p": bool(np.array_equal(dests["yuv420p"], want)),
                     "nv12_device": bool(np.array_equal(torch.cat([y for _, y in dests["nv12_device"]]).cpu().numpy(), nv_want))}
        assert all(identical.values()), identical
        ms = time_arms(arms, args.rounds, args.steps)
        mpix = T * H * W / 1e6
        out["vid4"] = {"frames": T, "lr": [h, w], "hr": [H, W], "scale": scale, "batch_schedule": sched, "clips_per_window": args.steps,
                       "outputs_identical_to_host_cv2": identical,
                       "arms": {k: {"ms_per_clip_median": round(statistics.median(v), 3), "ms_per_clip_all": [round(x, 3) for x in v],
                                    "hr_mpix_per_s": round(mpix / (statistics.median(v) / 1e3), 1)} for k, v in ms.items()}}
        del arms, dests

        # ---- 270x480 -> 1080x1920 stream
        h, w, lb, n = 270, 480, 26, args.long_frames
        H, W = 4 * h, 4 * w
        yuv_host, nv12_dev = sources(32, h, w, 512)
        dests = {"host_cv2": np.zeros((2 * lb, 3 * H // 2, W), np.uint8), "yuv420p": np.zeros((2 * lb, 3 * H // 2, W), np.uint8)}
        arms = make_arms(savsr_b200, net, dev, h, w, scale, lb, yuv_host, nv12_dev, n, dests)
        warm = make_arms(savsr_b200, net, dev, h, w, scale, lb, yuv_host, nv12_dev, lb + (n % lb or lb), dests)
        for fn in warm.values():                  # the plans of the full batch and of the stream's last batch
            fn()
        ms = time_arms(arms, args.rounds, 1)
        out["long_stream"] = {"frames": n, "lr": [h, w], "hr": [H, W], "scale": scale, "batch": lb, "nv12_pitch": 512,
                              "arms": {k: {"seconds_median": round(statistics.median(v) / 1e3, 3), "seconds_all": [round(x / 1e3, 3) for x in v],
                                           "hr_mpix_per_s": round(n * H * W / 1e6 / (statistics.median(v) / 1e3), 1),
                                           "frames_per_s": round(n / (statistics.median(v) / 1e3), 1)} for k, v in ms.items()}}
        del arms, warm, dests

        out["kernels"] = kernel_times(colour, dev)
        out["hbm_data_sheet_tb_per_s"] = HBM_TBPS
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
