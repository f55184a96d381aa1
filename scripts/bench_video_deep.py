"""Deep video through savsr_b200.VideoUpscaler against the 8-bit path, bf16, random-init weights (seed 0), seeded frames.  Four arms,
timed alternately in one process, host clock around whole streams ending in a device synchronise, median of --rounds:

  nv12            NV12 device frames with a 256-byte row pitch -> NV12 device output (the 8-bit baseline)
  p010            P010 device frames with a 256-byte row pitch -> P010 device output
  yuv420p10le     yuv420p10le pageable host frames -> yuv420p10le, each HR batch copied to pinned host memory
  nv12_to_p010    the NV12 device frames -> P010 device output (an 8-bit source, widened into a 16-bit ring)

Workloads: the Vid4 clip shape (34 frames, 144x180 -> 576x720 at x4, batch schedule (26, 8)), --steps clips per timed window; and the
270x480 -> 1080x1920 stream at x4, batch 26, --long-frames frames (a cycle of 32 distinct frames).  The arms' Vid4 outputs are checked
against enc(infer_clip(net.forward_bgr48, dec(frames), batch)) (dec of the 8-bit source widened by 257), and the nv12 arm against
infer_clip(net.forward_bgr_u8, ...).  Also each deep conversion kernel on its own with CUDA events (replayed as a CUDA graph, cycling over
buffers larger than the 126 MB L2), as bytes moved over time against the 7.7 TB/s data-sheet HBM bandwidth.  The card's name and power
limit are read in the same run.  Writes --out (default profiles/r03_video_deep.json) and prints it.
Usage: python scripts/bench_video_deep.py --steps 10 --rounds 3 --long-frames 520
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
from scripts.bench_video_yuv import HBM_TBPS, time_arms  # noqa: E402


def _u16(x):
    x = x.to(torch.int32)
    return (x - 65536 * (x >= 32768)).to(torch.int16).view(torch.uint16)


def sources(gen, dev, T, h, w, pitch):
    """(nv12 device frames, p010 device frames, yuv420p10le host frames) of T random frames; the device ones with a row pitch."""
    def pitched(x):
        vt = torch.uint8 if x.dtype == torch.uint8 else torch.int16
        surf = torch.zeros(T, 3 * h // 2, pitch, dtype=vt, device=dev)
        surf[:, :, :w] = x.view(vt).to(dev)
        return surf.view(x.dtype)[:, :, :w]
    Y, U, V = (torch.randint(16, 236, (T, h, w), generator=gen),) + tuple(torch.randint(16, 241, (T, h // 2, w // 2), generator=gen) for _ in range(2))
    nv12 = torch.cat([Y, torch.stack([U, V], -1).reshape(T, h // 2, w)], 1).to(torch.uint8)
    Y, U, V = (torch.randint(64, 941, (T, h, w), generator=gen),) + tuple(torch.randint(64, 961, (T, h // 2, w // 2), generator=gen) for _ in range(2))
    p010 = _u16(torch.cat([Y, torch.stack([U, V], -1).reshape(T, h // 2, w)], 1) << 6)
    le = _u16(torch.cat([Y.reshape(T, -1), U.reshape(T, -1), V.reshape(T, -1)], 1).reshape(T, 3 * h // 2, w))
    return pitched(nv12), pitched(p010), le


class HostSink:
    """HR batches -> pinned host memory, double-buffered by batch (the copy of one overlaps the next forward)."""

    def __init__(self, dev, max_batch, frame_shape, dtype):
        self.dev = dev
        self.bufs = [torch.empty((max_batch, *frame_shape), dtype=dtype).pin_memory() for _ in range(2)]
        self.k = 0

    def take(self, batches):
        for _, hr in batches:
            self.bufs[self.k % 2][:hr.shape[0]].copy_(hr, non_blocking=True)
            self.k += 1


def make_arms(savsr_b200, net, dev, h, w, scale, sched, nv12, p010, le, n_frames, keep):
    H, W = round(h * scale[0]), round(w * scale[1])
    mb = sched if isinstance(sched, int) else max(sched)
    ups = {"nv12": savsr_b200.VideoUpscaler(net, (h, w), scale, batch=sched, in_format="nv12", out_format="nv12"),
           "p010": savsr_b200.VideoUpscaler(net, (h, w), scale, batch=sched, in_format="p010", out_format="p010"),
           "yuv420p10le": savsr_b200.VideoUpscaler(net, (h, w), scale, batch=sched, in_format="yuv420p10le", out_format="yuv420p10le"),
           "nv12_to_p010": savsr_b200.VideoUpscaler(net, (h, w), scale, batch=sched, in_format="nv12", out_format="p010")}
    srcs = {"nv12": nv12, "p010": p010, "yuv420p10le": le, "nv12_to_p010": nv12}
    sink = HostSink(dev, mb, (3 * H // 2, W), torch.uint16)
    S = nv12.shape[0]

    def arm(name):
        def run():
            up, src = ups[name], srcs[name]
            up.reset()
            outs = []
            for k in range(n_frames):
                b = up.push(src[k % S])
                sink.take(b) if name == "yuv420p10le" else outs.extend(b)
            b = up.finish()
            sink.take(b) if name == "yuv420p10le" else outs.extend(b)
            if keep is not None and name != "yuv420p10le":
                keep[name] = outs
        return run
    return {k: arm(k) for k in ups}


def kernel_times(colour, dev, reps=200):
    res = {}
    for name, (h, w, n, fmt, direction) in {
            "decode_p010_lr_270x480_n1": (270, 480, 1, "p010", "dec"),
            "decode_yuv420p10le_lr_270x480_n26": (270, 480, 26, "yuv420p10le", "dec"),
            "encode_p010_hr_1080x1920_n1": (1080, 1920, 1, "p010", "enc"),
            "encode_yuv420p10le_hr_1080x1920_n26": (1080, 1920, 26, "yuv420p10le", "enc"),
            "widen_u8_to_u16_lr_270x480_n1": (270, 480, 1, None, "widen")}.items():
        yuv_b, bgr_b = n * 3 * h * w, n * 6 * h * w
        if direction == "widen":
            yuv_b = n * 3 * h * w                  # the uint8 source
        copies = max(2, -(-(256 << 20) // (yuv_b + bgr_b)))
        bgr = _u16(torch.randint(0, 65536, (copies, n, h, w, 3), device=dev))
        if direction == "widen":
            src = torch.randint(0, 256, (copies, n, h, w, 3), dtype=torch.uint8, device=dev)
            run = lambda i: colour.widen(src[i], out=bgr[i])  # noqa: E731
        else:
            yuv = _u16(torch.randint(0, 1024, (copies, n, 3 * h // 2, w), device=dev) << (6 if fmt == "p010" else 0))
            run = (lambda i: colour.yuv420_to_bgr(yuv[i], fmt, out=bgr[i])) if direction == "dec" else \
                  (lambda i: colour.bgr_to_yuv420(bgr[i], fmt, out=yuv[i]))
        run(0)
        torch.cuda.synchronize(dev)
        g = torch.cuda.CUDAGraph()
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
        del bgr, g
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10, help="Vid4 clips per timed window")
    ap.add_argument("--rounds", type=int, default=3, help="alternating rounds over the arms")
    ap.add_argument("--long-frames", type=int, default=520, help="frames of the 1080p-output stream")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_video_deep.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_video_deep.py measures on a CUDA device; none found")
    import savsr_b200
    from savsr_b200 import colour, sharding

    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    net = savsr_b200.SAVSR().to(dev).eval()
    net.precision = "bf16"
    gen = torch.Generator().manual_seed(1)
    out = {"gpu": gpu_identity(0), "precision": "bf16", "weights": "random init, torch.manual_seed(0)", "rounds": args.rounds}
    i64 = lambda t: t.view(torch.int16).to(torch.int64) & 0xFFFF  # noqa: E731

    with torch.no_grad():
        # ---- Vid4 clip
        T, h, w, scale, sched = 34, 144, 180, (4, 4), (26, 8)
        H, W = 4 * h, 4 * w
        nv12, p010, le = sources(gen, dev, T, h, w, 256)
        keep = {}
        arms = make_arms(savsr_b200, net, dev, h, w, scale, sched, nv12, p010, le, T, keep)
        for fn in arms.values():
            fn(); fn()
        net.set_scale(scale)
        deep = lambda x: net.forward_bgr48(x.view(torch.uint16)).view(torch.int16)  # noqa: E731
        cat = lambda outs: torch.cat([y for _, y in outs])  # noqa: E731
        bgr8 = colour.yuv420_to_bgr(nv12, "nv12")
        want8 = colour.bgr_to_yuv420(sharding.infer_clip(net.forward_bgr_u8, bgr8, batch=sched), "nv12")
        wide = torch.empty(bgr8.shape, dtype=torch.uint16, device=dev)
        colour.widen(bgr8, out=wide)
        want_wide = colour.bgr_to_yuv420(sharding.infer_clip(deep, wide.view(torch.int16), batch=sched).view(torch.uint16), "p010")
        hr10 = sharding.infer_clip(deep, colour.yuv420_to_bgr(p010, "p010").view(torch.int16), batch=sched).view(torch.uint16)
        identical = {"nv12": bool(torch.equal(cat(keep["nv12"]), want8)),
                     "p010": bool(torch.equal(i64(cat(keep["p010"])), i64(colour.bgr_to_yuv420(hr10, "p010")))),
                     "nv12_to_p010": bool(torch.equal(i64(cat(keep["nv12_to_p010"])), i64(want_wide)))}
        up = savsr_b200.VideoUpscaler(net, (h, w), scale, batch=sched, in_format="yuv420p10le", out_format="yuv420p10le")
        got = cat([b for k in range(T) for b in up.push(le[k])] + up.finish())
        identical["yuv420p10le"] = bool(torch.equal(i64(got), i64(colour.bgr_to_yuv420(hr10, "yuv420p10le"))))
        assert all(identical.values()), identical
        ms = time_arms(arms, args.rounds, args.steps)
        mpix = T * H * W / 1e6
        base = statistics.median(ms["nv12"])
        out["vid4"] = {"frames": T, "lr": [h, w], "hr": [H, W], "scale": scale, "batch_schedule": sched, "clips_per_window": args.steps,
                       "pitch_bytes": 256, "outputs_equal_to_the_composition": identical,
                       "arms": {k: {"ms_per_clip_median": round(statistics.median(v), 3), "ms_per_clip_all": [round(x, 3) for x in v],
                                    "vs_nv12": round(statistics.median(v) / base, 4),
                                    "hr_mpix_per_s": round(mpix / (statistics.median(v) / 1e3), 1)} for k, v in ms.items()}}
        del arms

        # ---- 270x480 -> 1080x1920 stream
        h, w, lb, n = 270, 480, 26, args.long_frames
        H, W = 4 * h, 4 * w
        nv12, p010, le = sources(gen, dev, 32, h, w, 512)
        arms = make_arms(savsr_b200, net, dev, h, w, scale, lb, nv12, p010, le, n, None)
        warm = make_arms(savsr_b200, net, dev, h, w, scale, lb, nv12, p010, le, lb + (n % lb or lb), None)
        for fn in warm.values():
            fn()
        ms = time_arms(arms, args.rounds, 1)
        base = statistics.median(ms["nv12"])
        out["long_stream"] = {"frames": n, "lr": [h, w], "hr": [H, W], "scale": scale, "batch": lb, "pitch_bytes": 512,
                              "arms": {k: {"seconds_median": round(statistics.median(v) / 1e3, 3), "seconds_all": [round(x / 1e3, 3) for x in v],
                                           "vs_nv12": round(statistics.median(v) / base, 4),
                                           "frames_per_s": round(n / (statistics.median(v) / 1e3), 1)} for k, v in ms.items()}}
        del arms, warm

        out["kernels"] = kernel_times(colour, dev)
        out["hbm_data_sheet_tb_per_s"] = HBM_TBPS
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
