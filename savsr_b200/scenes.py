"""Scene cuts of a streamed video: the integer cut score, its threshold bound, and the device launches that score ring frames.

A frame t >= 1 starts a new shot when 100 m_t >= tau * 3hw * maxval, i.e. m_t >= ceil(tau * 3hw * maxval / 100), where SAD_t = sum |frame_t - frame_{t-1}| over all
3hw BGR samples (SAD_0 = 0), m_t = min(SAD_t, |SAD_t - SAD_{t-1}|) (ffmpeg scdet's rule on the mean absolute frame difference), tau the
threshold in percent and maxval the full scale of the samples (255 or 65535).  The score of frame t is 100 m_t / (3hw maxval).
Everything is an integer, so the kernel (csrc/scenes.cu), reference_scores below and the 8- and 16-bit rings agree exactly; an 8-bit
frame widened by 257 gets the decisions of the 8-bit frame.  Windows are then folded into their shots (sharding.scene_window_indices).
"""
from __future__ import annotations

import math
from fractions import Fraction
from typing import Tuple

import numpy as np
import torch

from . import _capi as K, engine

MAXVAL = {torch.uint8: 255, torch.uint16: 65535}


def check_threshold(threshold) -> float:
    """`threshold` as a float in (0, 100] (percent of full scale), else a ValueError naming scene_threshold."""
    try:
        t = float(threshold)
    except (TypeError, ValueError):
        raise ValueError(f"scene_threshold must be a number in (0, 100], got {threshold!r}") from None
    if not math.isfinite(t) or not 0.0 < t <= 100.0:
        raise ValueError(f"scene_threshold must be finite and in (0, 100], got {threshold!r}")
    return t


def score_bound(threshold, h: int, w: int, maxval: int) -> int:
    """ceil(threshold * 3hw * maxval / 100) with the exact value of the float `threshold`: frame t is a cut when m_t >= this, which is
    100 m_t >= threshold * 3hw * maxval exactly (m_t is an integer)."""
    t = check_threshold(threshold)
    return math.ceil(Fraction(t) * 3 * h * w * maxval / 100)


def reference_scores(frames, threshold=None) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """NumPy reference on BGR frames [T, h, w, 3] (uint8 or uint16): (SAD uint64 [T], score float64 [T], cut bool [T]).  cut is all
    False without a threshold; SAD[0] = 0 and frame 0 is never a cut."""
    x = np.asarray(frames)
    maxval = 65535 if x.dtype == np.uint16 else 255
    T, n = x.shape[0], int(np.prod(x.shape[1:]))
    sad = np.zeros(T, dtype=np.uint64)
    if T > 1:
        d = np.abs(x[1:].astype(np.int64) - x[:-1].astype(np.int64)).reshape(T - 1, -1)
        sad[1:] = d.sum(1).astype(np.uint64)
    prev = np.concatenate([[0], sad[:-1].astype(np.int64)]) if T else np.zeros(0, np.int64)
    m = np.minimum(sad.astype(np.int64), np.abs(sad.astype(np.int64) - prev))
    m[:1] = 0
    score = 100.0 * m / (n * maxval)
    cut = np.zeros(T, dtype=bool)
    if threshold is not None:
        bound = score_bound(threshold, x.shape[1], x.shape[2], maxval)
        cut = m >= bound
        cut[:1] = False
    return sad, score, cut


class Detector:
    """The device state of one stream's detector: per-slot cut flags (uint8 [R]) and SADs (int64 [R]) beside a ring of R frames, and the
    scoring launch's scratch.  Sized by the ring, never by the length of the video."""

    def __init__(self, ring: torch.Tensor, threshold):
        if ring.dtype not in MAXVAL or ring.dim() != 4 or ring.shape[3] != 3 or not ring.is_contiguous():
            raise ValueError(f"the ring must be a contiguous uint8 or uint16 BGR tensor [R, h, w, 3], got {ring.dtype} {tuple(ring.shape)}")
        self.ring = ring
        self.R, self.h, self.w = ring.shape[0], ring.shape[1], ring.shape[2]
        self.threshold = check_threshold(threshold)
        self.bound = score_bound(self.threshold, self.h, self.w, MAXVAL[ring.dtype])
        dev = ring.device
        self.cut = torch.zeros(self.R, dtype=torch.uint8, device=dev)
        self.sad = torch.zeros(self.R, dtype=torch.int64, device=dev)
        self.scratch = torch.zeros(K.SCENE_SCRATCH_WORDS, dtype=torch.int64, device=dev)

    def score(self, t: int, marked: bool) -> None:
        """Enqueue the score of frame t (already in slot t % R) on the device's current stream: one launch, nothing waits."""
        dev = self.ring.device
        ctx = engine.context(dev.index if dev.index is not None else 0)
        fn = ctx.lib.savsr_scene_score_u16 if self.ring.dtype == torch.uint16 else ctx.lib.savsr_scene_score_u8
        with torch.cuda.device(dev):
            K.check(fn(ctx.handle, self.ring.data_ptr(), self.R, self.h, self.w, int(t), int(bool(marked)), self.bound, self.cut.data_ptr(),
                       self.sad.data_ptr(), self.scratch.data_ptr(), torch.cuda.current_stream(dev).cuda_stream))
