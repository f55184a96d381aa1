"""Scene cuts in the streaming upscaler: what scoring every frame on the device and folding the windows at cuts costs, bf16, random-init
weights (seed 0), seeded synthetic frames (drifting crops of smooth random textures, one texture per shot).

Streams, uint8 BGR device frames in and out through savsr_b200.VideoUpscaler, host clock around whole streams ending in a device
synchronise, arms timed alternately, median and range of --rounds, --steps streams per timed window:

  off             no scene_threshold, one shot (the baseline)
  on_no_cut       scene_threshold above every score of the clip: every frame is scored, no cut fires
  on_multishot    scene_threshold 10 over a multi-shot clip of the same length (cuts detected; the cut after a 1-frame shot marked)
  marked          no scene_threshold, the multi-shot clip with every cut marked by push(new_scene=True)

at two shapes: the Vid4 clip (34 frames, 144x180 -> 576x720 at x4, batch schedule (26, 8)) and 270x480 -> 1080x1920 at x4, batch 26.
Every arm's output is checked against infer_clip(net.forward_bgr_u8, clip, batch, cuts=up.scene_cuts()).

Kernels (CUDA events around a CUDA graph of one launch per ring slot, the ring larger than the 126 MB L2): savsr_scene_score_u8 / _u16 at
144x180 and 270x480, one frame per launch; bytes read per launch (two frames; the previous launch read one of them) against the 7.7 TB/s
data-sheet bandwidth.  savsr_write_scene_frame_table at batch 26 next to savsr_write_frame_table.  The card's name and power limit are
read in the same run.  Writes --out (default profiles/r03_video_scenes.json) and prints it.
Usage: python scripts/bench_video_scenes.py --steps 5 --rounds 5
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


def texture_clip(lengths, h, w, seed):
    """uint8 BGR [sum(lengths), h, w, 3]: per shot, a crop drifting one pixel per frame over its own smooth random texture."""
    frames = []
    for s, L in enumerate(lengths):
        g = torch.Generator().manual_seed(seed * 1000 + s)
        grid = torch.rand(1, 3, 12, 12, generator=g)
        tex = torch.nn.functional.interpolate(grid, size=(h + L, w + L), mode="bilinear", align_corners=False)[0].permute(1, 2, 0)
        frames += [(tex[t:t + h, t:t + w] * 255).round() for t in range(L)]
    return torch.stack(frames).to(torch.uint8)


def event_us(fn, reps_in_graph, rounds):
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    g.replay()
    torch.cuda.synchronize()
    us = []
    for _ in range(rounds):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        us.append(1e3 * e0.elapsed_time(e1) / reps_in_graph)
    return us


def summary(v, digits=3):
    return {"median": round(statistics.median(v), digits), "min": round(min(v), digits), "max": round(max(v), digits),
            "all": [round(x, digits) for x in v]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5, help="Vid4 streams per timed window (the 1080p stream runs max(1, steps // 5))")
    ap.add_argument("--rounds", type=int, default=5, help="alternating rounds over the arms")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_video_scenes.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_video_scenes.py measures on a CUDA device; none found")
    import savsr_b200
    from savsr_b200 import engine, scenes, sharding

    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    net = savsr_b200.SAVSR().to(dev).eval()
    net.precision = "bf16"
    out = {"gpu": gpu_identity(0), "precision": "bf16", "weights": "random init, torch.manual_seed(0)", "rounds": args.rounds}

    with torch.no_grad():
        for name, (T, h, w, sched, shots, steps) in {
                "vid4_x4": (34, 144, 180, (26, 8), [8, 5, 1, 12, 8], args.steps),
                "lr270x480_to_1080x1920": (52, 270, 480, 26, [10, 1, 6, 2, 20, 13], max(1, args.steps // 5))}.items():
            one = texture_clip([T], h, w, seed=1).to(dev)
            multi = texture_clip(shots, h, w, seed=2).to(dev)
            cuts_true = [sum(shots[:k]) for k in range(1, len(shots))]
            flash_end = [c for k, c in enumerate(cuts_true) if shots[k] == 1]      # the cut after a 1-frame shot: marked
            _, score, _ = scenes.reference_scores(one.cpu().numpy())
            tau_none = min(100.0, float(score.max()) * 1.5 + 0.5)
            spec = {"off": (one, {}, []), "on_no_cut": (one, {"scene_threshold": tau_none}, []),
                    "on_multishot": (multi, {"scene_threshold": 10}, flash_end), "marked": (multi, {}, cuts_true)}
            ups = {k: savsr_b200.VideoUpscaler(net, (h, w), (4, 4), batch=sched, **kw) for k, (_, kw, _) in spec.items()}
            keep = {}

            def arm(k):
                def run():
                    clip, _, marks = spec[k]
                    up = ups[k]
                    up.reset()
                    outs = []
                    for t in range(T):
                        outs += up.push(clip[t], new_scene=t in marks)
                    keep[k] = outs + up.finish()
                return run
            arms = {k: arm(k) for k in spec}
            for fn in arms.values():
                fn(); fn()
            net.set_scale((4, 4))
            identical, cuts = {}, {}
            for k, (clip, _, _) in spec.items():
                cuts[k] = ups[k].scene_cuts()
                want = sharding.infer_clip(net.forward_bgr_u8, clip, batch=sched, cuts=cuts[k] or None)
                identical[k] = bool(torch.equal(torch.cat([y for _, y in keep[k]]), want))
            assert all(identical.values()), identical
            assert cuts["off"] == cuts["on_no_cut"] == [] and cuts["on_multishot"] == cuts["marked"] == cuts_true, cuts
            ms = time_arms(arms, args.rounds, steps)
            base = statistics.median(ms["off"])
            out[name] = {"frames": T, "lr": [h, w], "hr": [4 * h, 4 * w], "scale": [4, 4], "batch_schedule": sched, "streams_per_window": steps,
                         "shots_multishot": shots, "cuts_true": cuts_true, "cuts_found": cuts, "threshold_on_no_cut": tau_none,
                         "threshold_multishot": 10, "outputs_equal_to_the_composition": identical,
                         "arms": {k: {"ms_per_stream": summary(v), "vs_off": round(statistics.median(v) / base, 4)} for k, v in ms.items()}}
            del ups, keep, arms

        kern = {}
        ctx = engine.context(0)
        for h, w in ((144, 180), (270, 480)):
            for dt in (torch.uint8, torch.uint16):
                fbytes = 3 * h * w * (2 if dt == torch.uint16 else 1)
                R = -(-(256 << 20) // fbytes)
                ring = torch.randint(0, 256, (R, h, w, 3), dtype=torch.int32, device=dev).to(dt)
                det = scenes.Detector(ring, 10)

                def run(det=det, R=R):
                    for t in range(1, R + 1):
                        det.score(t, False)
                us = event_us(run, R, args.rounds)
                med = statistics.median(us)
                kern[f"scene_score_{'u16' if dt == torch.uint16 else 'u8'}_{h}x{w}"] = {
                    "us_per_launch": summary(us, 2), "ring_frames": R, "ring_bytes": R * fbytes, "bytes_read_per_launch": 2 * fbytes,
                    "gb_per_s": round(2 * fbytes / med / 1e3, 1), "share_of_hbm_data_sheet": round(2 * fbytes / med / 1e6 / HBM_TBPS, 4),
                    "new_bytes_per_launch": fbytes}
                del ring, det
        B, h, w = 26, 270, 480
        plan = net._plan(B, h, w, dev, "bgr_u8_frames", (4, 4))
        ring = torch.zeros(B + 6, h, w, 3, dtype=torch.uint8, device=dev)
        cut = torch.zeros(B + 6, dtype=torch.uint8, device=dev)
        ptrs = [ring.data_ptr() + 3 * h * w * (k % (B + 6)) for k in range(7 * B)]
        reps = 500
        kern["write_scene_frame_table_b26"] = {"us_per_launch": summary(event_us(
            lambda: [plan.write_scene_frame_table(ring, cut, 3, B + 6, False) for _ in range(reps)], reps, args.rounds), 2)}
        kern["write_frame_table_b26"] = {"us_per_launch": summary(event_us(
            lambda: [plan.write_frame_table(ptrs) for _ in range(reps)], reps, args.rounds), 2)}
        out["kernels"] = kern
        out["hbm_data_sheet_tb_per_s"] = HBM_TBPS
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
