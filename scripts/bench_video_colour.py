"""Colour matrix and range of the streaming upscaler: the H.273 conversions (BT.709, BT.2020, pc range) against the default cv2-exact
BT.601 tv-range ones, bf16, random-init weights (seed 0), seeded frames.

Kernels: each conversion on its own with CUDA events (replayed as a CUDA graph, cycling over buffers larger than the 126 MB L2), for
every (colorspace, range) pair next to ("bt601", "tv") in the same run, at the shapes of profiles/r03_video_yuv.json and
r03_video_deep.json: decode 270x480 at n = 1 (nv12 / p010) and n = 26 (yuv420p / yuv420p10le), encode 1080x1920 at the same n and
formats, 8- and 10-bit.  Bytes moved over time, against the 7.7 TB/s data-sheet HBM bandwidth.  Each pair's median over --rounds
alternating rounds.

Streams: the Vid4 clip shape (34 frames, 144x180 -> 576x720 at x4, batch schedule (26, 8)) through savsr_b200.VideoUpscaler, device
frames in, device frames out, host clock around whole streams ending in a device synchronise, arms timed alternately, median of
--rounds, --steps clips per timed window:

  nv12_bt601          NV12 bt601 tv -> NV12 bt601 tv (the baseline)
  nv12_bt601_to_bt709 NV12 bt601 tv -> NV12 bt709 tv (SD to HD)
  p010_bt2020         P010 bt2020nc tv -> P010 bt2020nc tv
  yuv420p_pc_to_tv    yuv420p bt709 pc -> yuv420p bt709 tv

Every arm's output is checked against enc_out(infer_clip(forward, dec_in(frames), batch)).  The card's name and power limit are read
in the same run.  Writes --out (default profiles/r03_video_colour.json) and prints it.
Usage: python scripts/bench_video_colour.py --steps 10 --rounds 5
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
from scripts.bench_video_deep import _u16, sources  # noqa: E402
from scripts.bench_video_yuv import HBM_TBPS, time_arms  # noqa: E402

PAIRS = [("bt601", "tv"), ("bt601", "pc"), ("bt709", "tv"), ("bt709", "pc"), ("bt2020nc", "tv"), ("bt2020nc", "pc")]
# (in_format, in pair, out_format, out pair)
ARMS = {"nv12_bt601": ("nv12", ("bt601", "tv"), "nv12", ("bt601", "tv")),
        "nv12_bt601_to_bt709": ("nv12", ("bt601", "tv"), "nv12", ("bt709", "tv")),
        "p010_bt2020": ("p010", ("bt2020nc", "tv"), "p010", ("bt2020nc", "tv")),
        "yuv420p_pc_to_tv": ("yuv420p", ("bt709", "pc"), "yuv420p", ("bt709", "tv"))}


def kernel_times(colour, dev, rounds, reps=200):
    res = {}
    for shape, (h, w, n, direction, fmts) in {
            "decode_lr_270x480_n1": (270, 480, 1, "dec", ("nv12", "p010")),
            "decode_lr_270x480_n26": (270, 480, 26, "dec", ("yuv420p", "yuv420p10le")),
            "encode_hr_1080x1920_n1": (1080, 1920, 1, "enc", ("nv12", "p010")),
            "encode_hr_1080x1920_n26": (1080, 1920, 26, "enc", ("yuv420p", "yuv420p10le"))}.items():
        for fmt in fmts:
            deep = fmt in colour.DEEP_FORMATS
            e = 2 if deep else 1
            yuv_b, bgr_b = n * 3 * h * w // 2 * e, n * 3 * h * w * e
            copies = max(2, -(-(256 << 20) // (yuv_b + bgr_b)))
            if deep:
                bgr = _u16(torch.randint(0, 65536, (copies, n, h, w, 3), device=dev))
                yuv = _u16(torch.randint(0, 1024, (copies, n, 3 * h // 2, w), device=dev) << (6 if fmt == "p010" else 0))
            else:
                bgr = torch.randint(0, 256, (copies, n, h, w, 3), dtype=torch.uint8, device=dev)
                yuv = torch.randint(0, 256, (copies, n, 3 * h // 2, w), dtype=torch.uint8, device=dev)
            graphs = {}
            for cs, rng in PAIRS:
                kw = dict(colorspace=cs, color_range=rng)
                run = (lambda i, kw=kw: colour.yuv420_to_bgr(yuv[i], fmt, out=bgr[i], **kw)) if direction == "dec" else \
                      (lambda i, kw=kw: colour.bgr_to_yuv420(bgr[i], fmt, out=yuv[i], **kw))
                run(0)
                torch.cuda.synchronize(dev)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    for i in range(reps):
                        run(i % copies)
                g.replay()
                graphs[f"{cs}_{rng}"] = g
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
            moved = yuv_b + bgr_b
            base = statistics.median(us["bt601_tv"])
            res[f"{shape}_{fmt}"] = {
                "bytes_moved": moved, "buffers_cycled": copies,
                "pairs": {k: {"us_per_launch": round(statistics.median(v), 2), "us_all": [round(x, 2) for x in v],
                              "gb_per_s": round(moved / statistics.median(v) / 1e3, 1),
                              "share_of_hbm_data_sheet": round(moved / statistics.median(v) / 1e6 / HBM_TBPS, 3),
                              "vs_bt601_tv": round(statistics.median(v) / base, 4)} for k, v in us.items()}}
            del bgr, yuv, graphs
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10, help="Vid4 clips per timed window")
    ap.add_argument("--rounds", type=int, default=5, help="alternating rounds over the arms and the kernel pairs")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_video_colour.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_video_colour.py measures on a CUDA device; none found")
    import savsr_b200
    from savsr_b200 import colour, sharding

    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    net = savsr_b200.SAVSR().to(dev).eval()
    net.precision = "bf16"
    gen = torch.Generator().manual_seed(1)
    out = {"gpu": gpu_identity(0), "precision": "bf16", "weights": "random init, torch.manual_seed(0)", "rounds": args.rounds}
    i64 = lambda t: t.view(torch.int16).to(torch.int64) & 0xFFFF if t.dtype == torch.uint16 else t.to(torch.int64)  # noqa: E731

    with torch.no_grad():
        T, h, w, scale, sched = 34, 144, 180, (4, 4), (26, 8)
        H, W = 4 * h, 4 * w
        nv12, p010, _ = sources(gen, dev, T, h, w, 256)
        g = torch.Generator().manual_seed(2)
        Y, U, V = (torch.randint(0, 256, (T, h, w), generator=g),) + tuple(torch.randint(0, 256, (T, h // 2, w // 2), generator=g) for _ in range(2))
        yuv420p = torch.cat([Y.reshape(T, -1), U.reshape(T, -1), V.reshape(T, -1)], 1).reshape(T, 3 * h // 2, w).to(torch.uint8).to(dev)
        srcs = {"nv12": nv12, "p010": p010, "yuv420p": yuv420p}
        ups, keep = {}, {}
        for name, (fi, pi, fo, po) in ARMS.items():
            ups[name] = savsr_b200.VideoUpscaler(net, (h, w), scale, batch=sched, in_format=fi, out_format=fo, in_colorspace=pi[0],
                                                 in_color_range=pi[1], out_colorspace=po[0], out_color_range=po[1])

        def arm(name):
            def run():
                up, src = ups[name], srcs[ARMS[name][0]]
                up.reset()
                outs = []
                for k in range(T):
                    outs += up.push(src[k])
                keep[name] = outs + up.finish()
            return run
        arms = {k: arm(k) for k in ARMS}
        for fn in arms.values():
            fn(); fn()
        net.set_scale(scale)
        deep = lambda x: net.forward_bgr48(x.view(torch.uint16)).view(torch.int16)  # noqa: E731
        identical = {}
        for name, (fi, pi, fo, po) in ARMS.items():
            bgr = colour.yuv420_to_bgr(srcs[fi], fi, colorspace=pi[0], color_range=pi[1])
            if bgr.dtype == torch.uint16:
                hr = sharding.infer_clip(deep, bgr.view(torch.int16), batch=sched).view(torch.uint16)
            else:
                hr = sharding.infer_clip(net.forward_bgr_u8, bgr, batch=sched)
            want = colour.bgr_to_yuv420(hr, fo, colorspace=po[0], color_range=po[1])
            identical[name] = bool(torch.equal(i64(torch.cat([y for _, y in keep[name]])), i64(want)))
        assert all(identical.values()), identical
        ms = time_arms(arms, args.rounds, args.steps)
        mpix = T * H * W / 1e6
        base = statistics.median(ms["nv12_bt601"])
        out["vid4"] = {"frames": T, "lr": [h, w], "hr": [H, W], "scale": scale, "batch_schedule": sched, "clips_per_window": args.steps,
                       "device_frames": True, "pitch_bytes": {"nv12": 256, "p010": 256, "yuv420p": w},
                       "arms_spec": {k: {"in": [v[0], *v[1]], "out": [v[2], *v[3]]} for k, v in ARMS.items()},
                       "outputs_equal_to_the_composition": identical,
                       "arms": {k: {"ms_per_clip_median": round(statistics.median(v), 3), "ms_per_clip_all": [round(x, 3) for x in v],
                                    "vs_nv12_bt601": round(statistics.median(v) / base, 4),
                                    "hr_mpix_per_s": round(mpix / (statistics.median(v) / 1e3), 1)} for k, v in ms.items()}}
        del arms, ups, keep

        out["kernels"] = kernel_times(colour, dev, args.rounds)
        out["hbm_data_sheet_tb_per_s"] = HBM_TBPS
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
