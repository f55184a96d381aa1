"""YUV 4:2:2 in the streaming upscaler: the 4:2:2 conversion kernels next to their 4:2:0 twins, and whole streams with 4:2:2 frames
in and out against the NV12 baseline.  bf16, random-init weights (seed 0), seeded frames, the default colour pair (bt601, tv).

Kernels: each conversion on its own with CUDA events (replayed as a CUDA graph, cycling over buffers larger than the 126 MB L2), decode
270x480 and encode 1080x1920, each at n = 1 and n = 26, for every 4:2:2 format and the 4:2:0 formats (yuv420p, nv12, yuv420p10le,
p010), timed alternately; median of --rounds.  Bytes moved from the shapes, over time, against the 7.7 TB/s data-sheet HBM bandwidth.

Streams: savsr_b200.VideoUpscaler, host clock around whole streams ending in a device synchronise, arms timed alternately, median of
--rounds, at two shapes: the Vid4 clip shape (34 frames, 144x180 -> 576x720 at x4, batch schedule (26, 8), --steps clips per window)
and 34 frames of 270x480 -> 1080x1920 at x4 with the same schedule (--hd-steps clips per window):

  nv12            NV12 device frames (rows 256-byte aligned) -> NV12 device frames (the baseline)
  nv16            NV16 device frames (rows 256-byte aligned) -> NV16 device frames
  p210            P210 device frames (rows 512-byte aligned) -> P210 device frames
  yuv422p10le     yuv422p10le pageable host frames -> yuv422p10le frames copied into pinned host memory
  uyvy422_to_nv16 UYVY pageable host frames (a capture device) -> NV16 device frames

Every arm's output is checked against enc(infer_clip(forward, dec(frames), batch)) and the result recorded.  The card's name and
power limit are read in the same run.  Writes --out (default profiles/r03_video_422.json) and prints it.
Usage: python scripts/bench_video_422.py --steps 10 --hd-steps 2 --rounds 5
"""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from scripts.bench_train_shape import gpu_identity  # noqa: E402
from scripts.bench_video_deep import _u16  # noqa: E402
from scripts.bench_video_yuv import HBM_TBPS, time_arms  # noqa: E402

KERNEL_FORMATS = ("yuv420p", "nv12", "yuv420p10le", "p010", "yuv422p", "nv16", "yuyv422", "uyvy422", "yuv422p10le", "p210")
ARMS = {"nv12": ("nv12", 256, "device", "nv12", "device"), "nv16": ("nv16", 256, "device", "nv16", "device"),
        "p210": ("p210", 256, "device", "p210", "device"), "yuv422p10le": ("yuv422p10le", None, "host", "yuv422p10le", "host"),
        "uyvy422_to_nv16": ("uyvy422", None, "host", "nv16", "device")}


def _random(colour, fmt, n, rows, cols, dev, gen):
    if fmt in colour.DEEP_FORMATS:
        return _u16(torch.randint(0, 1024, (n, rows, cols), generator=gen) << (6 if fmt in ("p010", "p210") else 0)).to(dev)
    return torch.randint(0, 256, (n, rows, cols), dtype=torch.uint8, generator=gen).to(dev)


def kernel_times(colour, dev, rounds, reps=200):
    res = {}
    gen = torch.Generator().manual_seed(3)
    for shape, (h, w, n, direction) in {"decode_lr_270x480_n1": (270, 480, 1, "dec"), "decode_lr_270x480_n26": (270, 480, 26, "dec"),
                                         "encode_hr_1080x1920_n1": (1080, 1920, 1, "enc"),
                                         "encode_hr_1080x1920_n26": (1080, 1920, 26, "enc")}.items():
        graphs, moved, bufs = {}, {}, []
        for fmt in KERNEL_FORMATS:
            deep = fmt in colour.DEEP_FORMATS
            e = 2 if deep else 1
            rows, cols = colour.yuv_shape(h, w, fmt)
            yuv_b, bgr_b = n * rows * cols * e, n * h * w * 3 * e
            copies = max(2, -(-(256 << 20) // (yuv_b + bgr_b)))
            yuv = _random(colour, fmt, copies * n, rows, cols, dev, gen).view(copies, n, rows, cols)
            bgr = (_u16(torch.randint(0, 65536, (copies, n, h, w, 3), device=dev)) if deep else
                   torch.randint(0, 256, (copies, n, h, w, 3), dtype=torch.uint8, device=dev))
            bufs.append((yuv, bgr))
            run = (lambda i, yuv=yuv, bgr=bgr, fmt=fmt: colour.yuv_to_bgr(yuv[i], fmt, out=bgr[i])) if direction == "dec" else \
                  (lambda i, yuv=yuv, bgr=bgr, fmt=fmt: colour.bgr_to_yuv(bgr[i], fmt, out=yuv[i]))
            run(0)
            torch.cuda.synchronize(dev)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for i in range(reps):
                    run(i % copies)
            g.replay()                               # warm-up
            graphs[fmt], moved[fmt] = g, (yuv_b + bgr_b, copies)
        torch.cuda.synchronize(dev)
        us = {k: [] for k in graphs}
        for _ in range(rounds):
            for k, g in graphs.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                g.replay()
                e1.record()
                torch.cuda.synchronize(dev)
                us[k].append(1e3 * e0.elapsed_time(e1) / reps)
        twin = {"yuv422p": "yuv420p", "nv16": "nv12", "yuyv422": "nv12", "uyvy422": "nv12", "yuv422p10le": "yuv420p10le", "p210": "p010"}
        res[shape] = {}
        for k, v in us.items():
            med = statistics.median(v)
            b, copies = moved[k]
            r = {"bytes_moved": b, "buffers_cycled": copies, "us_per_launch": round(med, 2), "us_all": [round(x, 2) for x in v],
                 "gb_per_s": round(b / med / 1e3, 1), "share_of_hbm_data_sheet": round(b / med / 1e6 / HBM_TBPS, 3)}
            if k in twin:
                r["vs_420_twin"] = {"twin": twin[k], "ratio": round(med / statistics.median(us[twin[k]]), 4)}
            res[shape][k] = r
        del graphs, bufs
    return res


def stream_arms(savsr_b200, colour, sharding, net, dev, T, h, w, scale, sched, gen):
    """(arms, check): the arms of ARMS at LR h x w, and a function that returns, per arm, whether its last output equals the
    composition."""
    srcs, ups, keep, sinks = {}, {}, {}, {}
    H, W = round(h * scale[0]), round(w * scale[1])
    for name, (fi, pitch, where, fo, out_where) in ARMS.items():
        rows, cols = colour.yuv_shape(h, w, fi)
        x = _random(colour, fi, T, rows, cols, "cpu", gen)
        if where == "device":
            x = x.to(dev)
            if pitch:                                # rows start every `pitch` samples, like a decoder surface's
                x = torch.empty(T, rows, -(-cols // pitch) * pitch, dtype=x.dtype, device=dev)[:, :, :cols].copy_(x)
        srcs[name] = x
        ups[name] = savsr_b200.VideoUpscaler(net, (h, w), scale, batch=sched, in_format=fi, out_format=fo)
        if out_where == "host":
            sinks[name] = torch.empty((T, *colour.yuv_shape(H, W, fo)), dtype=colour.dtype_of(fo)).pin_memory()

    def arm(name):
        def run():
            up, src = ups[name], srcs[name]
            up.reset()
            outs = []
            for k in range(T + 1):
                ready = up.push(src[k]) if k < T else up.finish()
                if name in sinks:                    # each batch into pinned host memory as it comes, in stream order
                    for start, y in ready:
                        sinks[name][start:start + y.shape[0]].copy_(y, non_blocking=True)
                outs += ready
            keep[name] = outs
        return run

    def check():
        i64 = lambda t: t.view(torch.int16).to(torch.int64) & 0xFFFF if t.dtype == torch.uint16 else t.to(torch.int64)  # noqa: E731
        net.set_scale(scale)
        deep = lambda x: net.forward_bgr48(x.view(torch.uint16)).view(torch.int16)  # noqa: E731
        torch.cuda.synchronize(dev)
        same = {}
        for name, (fi, _, _, fo, _) in ARMS.items():
            bgr = colour.yuv_to_bgr(srcs[name].to(dev), fi)
            if fo in colour.DEEP_FORMATS:
                if bgr.dtype == torch.uint8:
                    bgr = colour.widen(bgr, torch.empty(bgr.shape, dtype=torch.uint16, device=dev))
                hr = sharding.infer_clip(deep, bgr.view(torch.int16), batch=sched).view(torch.uint16)
            else:
                hr = sharding.infer_clip(net.forward_bgr_u8, bgr, batch=sched)
            want = i64(colour.bgr_to_yuv(hr, fo))
            got = sinks[name].to(dev) if name in sinks else torch.cat([y for _, y in keep[name]])
            same[name] = bool(torch.equal(i64(got), want))
        return same
    return {k: arm(k) for k in ARMS}, check


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10, help="Vid4 clips per timed window")
    ap.add_argument("--hd-steps", type=int, default=2, help="270x480 -> 1080x1920 clips per timed window")
    ap.add_argument("--rounds", type=int, default=5, help="alternating rounds over the arms and the kernels")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_video_422.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_video_422.py measures on a CUDA device; none found")
    import savsr_b200
    from savsr_b200 import colour, sharding

    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    net = savsr_b200.SAVSR().to(dev).eval()
    net.precision = "bf16"
    gen = torch.Generator().manual_seed(1)
    out = {"gpu": gpu_identity(0), "precision": "bf16", "weights": "random init, torch.manual_seed(0)", "rounds": args.rounds,
           "colour_pair": ["bt601", "tv"],
           "arms_spec": {k: {"in": v[0], "in_row_align_samples": v[1], "in_memory": v[2], "out": v[3], "out_memory": v[4]} for k, v in ARMS.items()}}
    with torch.no_grad():
        for key, (T, h, w, steps) in {"vid4": (34, 144, 180, args.steps), "hd_270x480": (34, 270, 480, args.hd_steps)}.items():
            scale, sched = (4, 4), (26, 8)
            arms, check = stream_arms(savsr_b200, colour, sharding, net, dev, T, h, w, scale, sched, gen)
            for fn in arms.values():                 # every shape and plan warmed up
                fn(); fn()
            identical = check()
            assert all(identical.values()), identical
            ms = time_arms(arms, args.rounds, steps)
            mpix = T * 4 * h * 4 * w / 1e6
            base = statistics.median(ms["nv12"])
            out[key] = {"frames": T, "lr": [h, w], "hr": [4 * h, 4 * w], "scale": scale, "batch_schedule": sched, "clips_per_window": steps,
                        "outputs_equal_to_the_composition": identical,
                        "arms": {k: {"ms_per_clip_median": round(statistics.median(v), 3), "ms_per_clip_all": [round(x, 3) for x in v],
                                     "vs_nv12": round(statistics.median(v) / base, 4),
                                     "hr_mpix_per_s": round(mpix / (statistics.median(v) / 1e3), 1)} for k, v in ms.items()}}
            del arms, check
            torch.cuda.empty_cache()
        out["kernels"] = kernel_times(colour, dev, args.rounds)
        out["hbm_data_sheet_tb_per_s"] = HBM_TBPS
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
