"""Frame-in / frame-out upscaling of decoded 8-bit or deep (10- and 16-bit) video of any length.

``VideoUpscaler`` takes frames as a decoder produces them and returns HR frames in order, with the same windows, reflection and
batch partition as ``sharding.infer_clip(net.forward_bgr_u8, clip, batch=...)`` on the whole clip, so its output is byte-identical to
that call.  Frames are uploaded once into a device ring and read in place by ``SAVSR.forward_bgr_u8_indexed``; the ring's size depends
on the largest batch of the schedule, not on the length of the video.  Frames may come and go as packed BGR, as YUV 4:2:0 (yuv420p,
NV12) or as YUV 4:2:2 (yuv422p, NV16, YUYV, UYVY: savsr_b200.colour), converted on the device on their way into the ring and out of
the forward's output buffer, each side with its own colour matrix and range (BT.601, BT.709, BT.2020; tv or pc).  Deep video (bgr48le,
yuv420p10le, P010, yuv422p10le, P210) streams through a ring of uint16 frames and ``SAVSR.forward_bgr48_indexed``.  Scene cuts, marked by the caller or detected on the device
(savsr_b200.scenes), fold each window into its own shot, so that no output frame is made of two shots.
"""
from __future__ import annotations

import contextlib
from typing import List, Optional, Tuple

import torch

from . import colour, engine, scenes, sharding


class VideoUpscaler:
    """Stream uint8 frames through `net` (a SAVSR in eval mode)::

        up = VideoUpscaler(net, lr_size=(h, w), scale=(4, 4), batch=(26, 8))
        for frame in decoder:                  # uint8 [h, w, 3] or [n, h, w, 3]; host (pageable or pinned) or CUDA
            for start, hr in up.push(frame):   # hr: fresh uint8 CUDA [m, H, W, 3], frames start .. start + m - 1, in order
                encode(hr)
        for start, hr in up.finish():          # the last windows, reflected about the now-known last frame
            encode(hr)

    Forwards follow ``sharding.batch_schedule(T, batch)``: batch [i, j) runs as soon as frame j + 2 has arrived (its windows then need
    no reflection at the end), and the batches whose windows reach past the last frame run in ``finish()``.  `scale` is fixed for the
    stream; a later ``net.set_scale`` does not change it.

    `in_format` and `out_format` name the frames' layout with ffmpeg's pix_fmt names (savsr_b200.colour): "bgr24" (the default,
    [h, w, 3]), "yuv420p" or "nv12" (one uint8 [3h/2, w] array per frame, [n, 3h/2, w] for several; an NV12 frame may have a row pitch,
    like a decoder surface viewed as a tensor).  YUV input is converted to BGR on its way into the ring and YUV output from the forward's
    output buffer, exactly as cv2.cvtColor converts (COLOR_YUV2BGR_I420 / _NV12, COLOR_BGR2YUV_I420), so the output is
    enc(infer_clip(net.forward_bgr_u8, dec(frames), batch=...)).  YUV needs even sizes: even h and w for YUV input, an even HR size
    for YUV output (bgr24 output takes any scale).

    Deep formats: "bgr48le" (uint16 [h, w, 3]), "yuv420p10le" and "p010" (one uint16 [3h/2, w] array per frame; a P010 frame may have
    a row pitch).  When either side is deep the ring holds uint16 BGR frames and the forward is net.forward_bgr48: 8-bit input is
    decoded as above and widened by 257 on its way into the ring, so it enters the network exactly as the 8-bit path feeds it, and the
    output is enc(infer_clip(net.forward_bgr48, dec(frames), batch=...)) with dec of an 8-bit source widened.  An 8-bit source gets
    deep output this way, without 8-bit banding; deep input with 8-bit output is refused.

    4:2:2 formats (savsr_b200.colour): "yuv422p", "nv16" (uint8 [2h, w]), "yuyv422", "uyvy422" (uint8 [h, 2w]), "yuv422p10le" and
    "p210" (uint16 [2h, w]); all but yuv422p and yuv422p10le may have a row pitch.  They need an even width only: an even LR width for
    4:2:2 input, an even HR width (any HR height) for 4:2:2 output.  Decoding gives both pixels of a horizontal pair the pair's chroma,
    encoding takes it from the pair's left pixel; either side may be 4:2:0 or 4:2:2 independently of the other.

    Colour: YUV input is decoded with the matrix `in_colorspace` and the range `in_color_range`, YUV output encoded with
    `out_colorspace` and `out_color_range` (ffmpeg's -colorspace / -color_range names: "bt601", "bt709", "bt2020nc"; "tv", "pc";
    savsr_b200.colour).  The default ("bt601", "tv") is the cv2-exact conversion above; the other pairs use the H.273 map.  An SD
    source upscaled to HD is ``in_colorspace="bt601", out_colorspace="bt709"``, so the output carries HD's usual tag.  dec and enc of
    the compositions above are then the conversions of these pairs (an 8-bit source for a 16-bit ring is decoded with the input pair,
    then widened).  A packed BGR side has nothing to convert and takes only the defaults.  No transfer function is applied: BT.2020
    frames are converted as code values.

    Ownership: the caller may overwrite or free what it passed to ``push`` as soon as ``push`` returns.  Host frames are staged through
    the upscaler's own pinned buffers (a staging slot is reused only after the event of its upload); CUDA frames are copied in stream
    order on the current stream.  Everything runs on the current stream of the net's device, so a ring slot is rewritten only after
    every forward enqueued before that has read it.

    Scene cuts: ``push(frames, new_scene=True)`` marks the first of those frames as the start of a shot (from an edit list, or the
    encoder's own detector), and with `scene_threshold` set (percent, in (0, 100]) every pushed frame is also scored on the device
    against the one before it, after any YUV decode or widening (savsr_b200.scenes: ffmpeg scdet's rule in exact integers), and starts a
    shot when its score reaches the threshold.  Each window is then folded into its own shot (sharding.scene_window_indices, the
    reference's reflection at a clip's ends applied at every cut), and the output is enc(infer_clip(net..., dec(frames), batch=...,
    cuts=up.scene_cuts())) with the same batches as without cuts.  About 10, scdet's default, is a starting point for the threshold; it
    has not been tuned on real footage.  A cut that ends a 1-frame shot (a flash) is not detected by design: mark it.  Detected cuts are
    resolved on the device when the frame table is written, so push and finish never wait for a score; without a threshold, marked
    cuts are resolved on the host into the usual frame pointers, and with no cut marked the launches are exactly those of a stream
    without cuts.  Fades and dissolves are not detected."""

    def __init__(self, net, lr_size: Tuple[int, int], scale, batch=1, num_frames: int = 7, in_format: str = "bgr24",
                 out_format: str = "bgr24", in_colorspace: str = "bt601", in_color_range: str = "tv", out_colorspace: str = "bt601",
                 out_color_range: str = "tv", scene_threshold=None):
        if net.training:
            raise RuntimeError("VideoUpscaler is inference only: call net.eval() first")
        h, w = (int(v) for v in lr_size)
        if h < 2 or w < 2:
            raise ValueError(f"LR frames must be at least 2x2, got {h}x{w}")
        sizes = [int(batch)] if isinstance(batch, int) else [int(b) for b in batch]
        sharding.batch_schedule(1, batch)                      # refuses empty or non-positive schedules
        self.net, self.h, self.w, self.batch, self.sizes = net, h, w, batch, sizes
        self.num_frames, self.pad = num_frames, num_frames // 2
        self.scale = engine.normalize_scale(scale)
        self.in_format = colour.check_format(in_format, "in_format")
        self.out_format = colour.check_format(out_format, "out_format")
        deep_in, deep_out = in_format in colour.DEEP_FORMATS, out_format in colour.DEEP_FORMATS
        if deep_in and not deep_out:
            raise ValueError(f"deep input {in_format} with 8-bit output {out_format} is not supported: choose an output of "
                             f"{', '.join(colour.DEEP_FORMATS)}")
        self.in_colour = (colour.check_colorspace(in_colorspace, "in_colorspace"), colour.check_color_range(in_color_range, "in_color_range"))
        self.out_colour = (colour.check_colorspace(out_colorspace, "out_colorspace"),
                           colour.check_color_range(out_color_range, "out_color_range"))
        for side, fmt, pair in (("in", in_format, self.in_colour), ("out", out_format, self.out_colour)):
            if fmt not in colour.YUV_FORMATS and pair != ("bt601", "tv"):
                raise ValueError(f"{side}_colorspace / {side}_color_range {pair} need a YUV {side}_format: {side}_format {fmt} is packed "
                                 f"BGR and is not converted")
        need = colour._uneven(in_format, h, w)
        if need:
            raise ValueError(f"{in_format} input needs an even LR {need}, got {h}x{w}")
        H, W = engine.get_hw(h, w, self.scale)
        need = colour._uneven(out_format, H, W)
        if need:
            gives = f"H = {H}, W = {W}" if need == "size" else f"W = {W}"
            raise ValueError(f"{out_format} output needs an even HR {need}: {h}x{w} at scale {self.scale} gives {gives}; "
                             f"{colour.bgr_format(out_format)} output takes any scale")
        if scene_threshold is not None:
            scenes.check_threshold(scene_threshold)
        self.device = net.gamma.device
        # Until batch [i, j) has run, the ring holds frames i - pad .. j - 1 + pad, the ones its windows read, and nothing newer.
        self.capacity = max(sizes) + 2 * self.pad
        self.ring = torch.empty(self.capacity, h, w, 3, dtype=torch.uint16 if deep_out else torch.uint8, device=self.device)
        self._widen = deep_out and not deep_in                  # 8-bit frames into a 16-bit ring: decoded to uint8 BGR, then x 257
        self._staging: Optional[torch.Tensor] = None           # pinned twin of the ring for host frames (YUV-sized for YUV input), on first use
        self._yuv_dev: Optional[torch.Tensor] = None           # device staging of one host YUV frame, converted from there into the ring
        self._bgr8_dev: Optional[torch.Tensor] = None          # one uint8 BGR frame on its way into a 16-bit ring, widened from there
        self._uploaded: List[Optional[torch.cuda.Event]] = [None] * self.capacity
        # scene detection: per-slot cut flags and SADs beside the ring (sized by it), and a host log of each frame's flag, copied
        # back asynchronously for scene_cuts() in chunks of pinned memory that are reused by the next video
        self.detector = None if scene_threshold is None else scenes.Detector(self.ring, scene_threshold)
        self._cut_log: List[torch.Tensor] = []
        self.reset()

    def reset(self) -> None:
        """Start the next video of the same frame size: the ring, the staging buffers and the module's cached plans are reused."""
        self.received = 0          # frames pushed
        self.done = 0              # frames whose HR output has been returned (start of the next batch)
        self.batches = 0           # forwards run
        self.finished = False
        self._marked: List[int] = []   # frames > 0 marked with push(..., new_scene=True)

    def push(self, frames, new_scene: bool = False) -> List[Tuple[int, torch.Tensor]]:
        """Append frames in `in_format` (uint8, uint16 for the deep formats): BGR [h, w, 3] or [n, h, w, 3], YUV one
        colour.yuv_shape(h, w, in_format) array per frame or [n, ...] (torch or numpy, host or CUDA).  Returns the batches that became
        ready, as (index of the first frame, [m, H, W, 3], or [m, *colour.yuv_shape(H, W, out_format)] in a YUV out_format, of
        out_format's sample type) in frame order; often none.  `new_scene`: the first of these
        frames starts a new shot (the first frame of a video always does)."""
        if self.finished:
            raise RuntimeError("push() after finish(): call reset() to start the next video")
        self._check_net()
        x = self._frames(frames)
        if new_scene and x.shape[0] == 0:
            raise ValueError("push(new_scene=True) needs at least one frame: new_scene marks the first frame of the push")
        if new_scene and self.received > 0:
            self._marked.append(self.received)
        out = []
        with self._on_device():
            for k, f in enumerate(x):
                self._upload(f)
                if self.detector is not None:
                    self._score(self.received, bool(new_scene) and k == 0)
                self.received += 1
                while True:
                    i, j = self._next_batch()
                    if j + self.pad > self.received:       # frame j - 1 + pad, the last one its windows read, has not arrived
                        break
                    out.append(self._forward(i, j))
        return out

    def finish(self) -> List[Tuple[int, torch.Tensor]]:
        """The video has ended: run the remaining windows, reflected about the last frame pushed."""
        if self.finished:
            raise RuntimeError("finish() was already called: call reset() to start the next video")
        self._check_net()
        sharding.frame_window_indices(0, self.received, self.num_frames)      # too short for reflection padding: ValueError
        self.finished = True
        out = []
        with self._on_device():
            while self.done < self.received:
                i, j = self._next_batch()
                out.append(self._forward(i, min(j, self.received)))
        return out

    def scene_cuts(self) -> List[int]:
        """The sorted frames that started a new shot so far, marked or detected (frame 0 is not listed).  With detection on this waits
        for the scores of the pushed frames: it synchronises with the device's current stream."""
        if self.detector is None:
            return list(self._marked)
        with self._on_device():
            if self.device.type == "cuda":
                torch.cuda.current_stream(self.device).synchronize()
        n = self.received
        flags = torch.cat(self._cut_log)[:n] if n else torch.zeros(0, dtype=torch.uint8)
        return [int(f) for f in torch.nonzero(flags[1:]).flatten().add(1)]

    # ------------------------------------------------------------------ internals
    _LOG_CHUNK = 4096

    def _score(self, t: int, marked: bool) -> None:
        """Score frame t on the device (after its upload, in stream order) and queue the copy of its flag into the host log."""
        self.detector.score(t, marked)
        k, r = divmod(t, self._LOG_CHUNK)
        if k == len(self._cut_log):
            self._cut_log.append(torch.zeros(self._LOG_CHUNK, dtype=torch.uint8, pin_memory=self.device.type == "cuda"))
        self._cut_log[k][r:r + 1].copy_(self.detector.cut[t % self.capacity:t % self.capacity + 1], non_blocking=True)

    def _check_net(self) -> None:
        if self.net.training:
            raise RuntimeError("VideoUpscaler is inference only: the net was put in train mode")

    def _on_device(self):
        return torch.cuda.device(self.device) if self.device.type == "cuda" else contextlib.nullcontext()

    def _frames(self, frames) -> torch.Tensor:
        x = frames if isinstance(frames, torch.Tensor) else torch.as_tensor(frames)
        if self.in_format in colour.YUV_FORMATS:
            x = colour.yuv_frames(x, self.in_format, self.h, self.w)      # dtype, shape, row pitch and column stride
        else:
            dt = colour.dtype_of(self.in_format)
            tn = str(dt).replace("torch.", "")
            if x.dtype != dt:
                raise TypeError(f"VideoUpscaler takes {tn} BGR frames for {self.in_format}, got {x.dtype}")
            if x.dim() == 3:
                x = x.unsqueeze(0)
            if x.dim() != 4 or tuple(x.shape[1:]) != (self.h, self.w, 3):
                raise ValueError(f"expected {tn} BGR frames [{self.h}, {self.w}, 3] or [n, {self.h}, {self.w}, 3], got {tuple(x.shape)}")
        if x.device.type != "cpu" and x.device != self.device:
            raise ValueError(f"frames on {x.device}, the net on {self.device}")
        return x

    def _upload(self, frame: torch.Tensor) -> None:
        s = self.received % self.capacity
        yuv, ring = self.in_format in colour.YUV_FORMATS, self.ring[s]
        # where the frame's BGR goes: the ring slot, or for an 8-bit frame into a 16-bit ring one uint8 scratch frame widened from there
        # (one buffer is enough: its next use follows this frame's widening in stream order)
        if self._widen and self._bgr8_dev is None:
            self._bgr8_dev = torch.empty(self.h, self.w, 3, dtype=torch.uint8, device=self.device)
        bgr = self._bgr8_dev if self._widen else ring
        if frame.device.type == "cpu" and self.device.type == "cuda":
            if self._staging is None:
                self._staging = torch.empty((self.capacity, *frame.shape), dtype=frame.dtype, pin_memory=True)
                if yuv:     # one buffer is enough: its next upload follows this frame's conversion in stream order
                    self._yuv_dev = torch.empty(frame.shape, dtype=frame.dtype, device=self.device)
            ev = self._uploaded[s]
            if ev is None:
                ev = self._uploaded[s] = torch.cuda.Event()
            else:
                ev.synchronize()                 # the previous upload from this staging slot has been read
            self._staging[s].copy_(frame)
            frame = self._yuv_dev if yuv else bgr
            frame.copy_(self._staging[s], non_blocking=True)
            ev.record(torch.cuda.current_stream(self.device))
        if yuv:                                  # CUDA frames, pitched ones too, are read in place
            colour.yuv_to_bgr(frame, self.in_format, out=bgr, **self._colour_kw(self.in_colour, "colorspace", "color_range"))
        elif frame is not bgr:
            if self._widen and frame.is_contiguous():
                bgr = frame                      # a CUDA frame is widened where it is
            else:
                bgr.copy_(frame, non_blocking=True)
        if self._widen:
            colour.widen(bgr, out=ring)

    @staticmethod
    def _colour_kw(pair: Tuple[str, str], cs_key: str, range_key: str) -> dict:
        """Keyword arguments of a conversion with colour `pair`: none for the default pair, whose calls stay exactly as they were."""
        return {} if pair == ("bt601", "tv") else {cs_key: pair[0], range_key: pair[1]}

    def _next_batch(self) -> Tuple[int, int]:
        b = self.sizes[min(self.batches, len(self.sizes) - 1)]
        return self.done, self.done + b

    def _forward(self, i: int, j: int) -> Tuple[int, torch.Tensor]:
        R = self.capacity
        yuv_out = {} if self.out_format == colour.bgr_format(self.out_format) else \
            {"out_format": self.out_format, **self._colour_kw(self.out_colour, "out_colorspace", "out_color_range")}
        if self.detector is not None:          # the cuts are on the device: the table is written there
            hr = self.net._forward_ring_scenes(self.ring, self.detector.cut, i, j - i, self.received, self.finished, self.scale, **yuv_out)
        else:
            # marked cuts only: folded on the host into the pointers (before the end, the windows lie inside the received frames, so
            # `received` stands in for the end of the last shot)
            cuts = self._marked if self._marked else None
            windows = [[f % R for f in sharding.clip_window_indices(c, self.received, cuts, self.num_frames)] for c in range(i, j)]
            hr = self.net._forward_bgr_u8_indexed(self.ring, windows, self.scale, **yuv_out)
        self.done, self.batches = j, self.batches + 1
        return i, hr
