"""Clip-level driver: window gather, frame sharding across ranks, batched inference.

Every output frame of a clip is an independent forward over its own 7-frame LR window (the reference's
hot loop, lbasicsr/models/video_base_model.py:50-59, is ``for idx in range(rank, len(dataset),
world_size)``).  So multi-GPU inference shards *frames* across ranks with no collective on the data
path; only the optional gather of results uses ``torch.distributed`` (NCCL on GPUs, gloo in CPU tests).
"""
from __future__ import annotations

import bisect
from typing import Callable, List, Optional, Sequence

import torch


def frame_window_indices(crt_idx: int, n_frames: int, num_frames: int = 7) -> List[int]:
    """Reflection-padded window around `crt_idx` (lbasicsr/data/data_util.py:63-112, padding='reflection')."""
    if num_frames % 2 != 1:
        raise ValueError("num_frames should be an odd number.")
    last = n_frames - 1
    pad = num_frames // 2
    if n_frames <= pad:     # the reflected index -i (or 2 * last - i) would leave the clip; the reference raises IndexError here
        raise ValueError(f"a clip of {n_frames} frames is too short for reflection padding of a {num_frames}-frame window")
    out = []
    for i in range(crt_idx - pad, crt_idx + pad + 1):
        if i < 0:
            i = -i
        elif i > last:
            i = 2 * last - i
        out.append(i)
    return out


def scene_window_indices(c: int, start: int, stop: int, num_frames: int = 7) -> List[int]:
    """Window of frame `c` inside the shot [start, stop): each index c + o, |o| <= num_frames // 2, folded into the shot.  A shot of one
    frame repeats it; otherwise the index is reflected at the shot's ends, as often as it takes (period 2 (L - 1)).  For a shot of
    num_frames // 2 + 1 frames or more this is exactly frame_window_indices(c - start, L) + start, the reference's padding at a clip's
    ends, applied at every cut; shorter shots, which a clip cannot be, get the repeated fold."""
    if num_frames % 2 != 1:
        raise ValueError("num_frames should be an odd number.")
    L = stop - start
    if L < 1 or not (start <= c < stop):
        raise ValueError(f"frame {c} is not inside the shot [{start}, {stop})")
    pad = num_frames // 2
    if L == 1:
        return [start] * num_frames
    period = 2 * (L - 1)
    out = []
    for i in range(c - pad, c + pad + 1):
        r = (i - start) % period
        if r >= L:
            r = period - r
        out.append(start + r)
    return out


def check_cuts(cuts: Sequence[int], n_frames: int) -> tuple:
    """`cuts` as a tuple of ints: sorted, distinct frame indices in [0, n_frames), each the first frame of a shot."""
    out = tuple(int(f) for f in cuts)
    if any(b <= a for a, b in zip(out, out[1:])) or (out and (out[0] < 0 or out[-1] >= n_frames)):
        raise ValueError(f"cuts must be sorted, distinct frame indices in [0, {n_frames}), got {list(out)}")
    return out


def clip_window_indices(c: int, n_frames: int, cuts: Optional[Sequence[int]] = None, num_frames: int = 7) -> List[int]:
    """Window of frame `c` of a clip of `n_frames` frames: frame_window_indices with `cuts` None, else the window folded into the shot of
    `c` (scene_window_indices), where a shot starts at frame 0 and at every frame of the sorted `cuts`."""
    if cuts is None:
        return frame_window_indices(c, n_frames, num_frames)
    k = bisect.bisect_right(cuts, c)
    start = cuts[k - 1] if k > 0 else 0
    stop = cuts[k] if k < len(cuts) else n_frames
    return scene_window_indices(c, start, stop, num_frames)


def shard_frames(n_frames: int, rank: int, world_size: int, contiguous: bool = False) -> List[int]:
    """Frames of a clip owned by `rank`.  Default = the reference's rank-strided loop
    (video_base_model.py:50); `contiguous` gives equal contiguous chunks instead."""
    if not (0 <= rank < world_size):
        raise ValueError(f"rank {rank} outside world of size {world_size}")
    if contiguous:
        per = (n_frames + world_size - 1) // world_size
        return list(range(min(rank * per, n_frames), min((rank + 1) * per, n_frames)))
    return list(range(rank, n_frames, world_size))


_WINDOW_INDEX_CACHE: "dict[tuple, torch.Tensor]" = {}


def _window_index(T: int, frames: Sequence[int], num_frames: int, device: torch.device, cuts: Optional[tuple] = None) -> torch.Tensor:
    """Flat gather index of the windows of `frames`, resident on `device`.  Cached: building it per call costs a host-to-device copy from
    pageable memory, which blocks the host until the stream has drained -- between two batches of a clip that is an idle GPU.
    `cuts` (checked, a tuple) is part of the key, so clips of one length with different cuts get their own index."""
    key = (T, tuple(int(f) for f in frames), num_frames, device.type, device.index) + (() if cuts is None else (cuts,))
    idx = _WINDOW_INDEX_CACHE.get(key)
    if idx is None:
        if len(_WINDOW_INDEX_CACHE) >= 256:
            _WINDOW_INDEX_CACHE.clear()
        if cuts is not None and T <= num_frames // 2:      # the refusal of a whole clip this short stays, with or without cuts
            frame_window_indices(0, T, num_frames)
        idx = torch.tensor([clip_window_indices(f, T, cuts, num_frames) for f in key[1]], dtype=torch.long).reshape(-1).to(device)
        _WINDOW_INDEX_CACHE[key] = idx
    return idx


def gather_windows(clip: torch.Tensor, frames: Sequence[int], num_frames: int = 7, cuts: Optional[Sequence[int]] = None) -> torch.Tensor:
    """clip [T, ...] -> windows [len(frames), num_frames, ...] (temporal halo = duplicated input): fp32 [T, 3, h, w] planes for
    SAVSR.forward, or uint8 [T, h, w, 3] BGR frames for SAVSR.forward_bgr_u8.  `cuts`: sorted frame indices that each start a new
    shot; every window is then folded into its own shot (scene_window_indices) instead of mixing frames of two shots."""
    c = None if cuts is None else check_cuts(cuts, clip.shape[0])
    idx = _window_index(clip.shape[0], frames, num_frames, clip.device, c)
    return clip.index_select(0, idx).reshape(len(frames), num_frames, *clip.shape[1:])


def batch_schedule(n: int, batch) -> list:
    """[(start, stop), ...] covering n frames.  `batch` is an int (equal batches, the last one ragged) or a sequence of batch
    sizes used in order (the last entry repeats): e.g. (26, 8) runs one large forward and a short final one, so that the
    device-to-host copy that cannot overlap anything -- the last batch's -- is small."""
    sizes = [int(batch)] if isinstance(batch, int) else [int(b) for b in batch]
    if not sizes or min(sizes) < 1:
        raise ValueError(f"batch sizes must be positive, got {batch!r}")
    out, i, k = [], 0, 0
    while i < n:
        b = sizes[min(k, len(sizes) - 1)]
        out.append((i, min(i + b, n)))
        i += b
        k += 1
    return out


def infer_clip(net: Callable[[torch.Tensor], torch.Tensor], clip: torch.Tensor, frames: Optional[Sequence[int]] = None,
               batch=1, num_frames: int = 7, out: Optional[torch.Tensor] = None, copy_stream: Optional["torch.cuda.Stream"] = None,
               join: bool = True, cuts: Optional[Sequence[int]] = None) -> torch.Tensor:
    """Run `net` on the windows of `frames` (default: all), `batch` windows per forward (int or a schedule, see batch_schedule).
    Returns [len(frames), ...] of whatever `net` returns per window: [n, 3, H, W] fp32 for SAVSR (clip [T, 3, h, w] fp32), or
    [n, H, W, 3] uint8 BGR for SAVSR.forward_bgr_u8 (clip [T, h, w, 3] uint8).  The last, ragged batch is run at its own size.
    If `out` (e.g. a pinned host tensor) is given, each batch is copied into it on a side stream while the next
    batch computes, and `out` is returned once all copies are enqueued behind the current stream.
    `cuts`: sorted frame indices of the clip that each start a new shot (a scene cut); each window is folded into its own shot
    (scene_window_indices), so no output frame is made of two shots.  None (the default) is one shot, reflected at the clip's ends.
    `copy_stream` / `join=False`: for a stream of clips -- the caller owns ONE copy stream, the compute stream does not wait for the copies
    (the next clip's forwards overlap this clip's last copy), and the caller synchronises the copy stream before reading `out`."""
    frames = list(range(clip.shape[0])) if frames is None else list(frames)
    if copy_stream is None:
        copy_stream = torch.cuda.Stream(clip.device) if (out is not None and clip.is_cuda) else None
    outs = []
    for i, j in batch_schedule(len(frames), batch):
        chunk = frames[i:j]
        y = net(gather_windows(clip, chunk, num_frames) if cuts is None else gather_windows(clip, chunk, num_frames, cuts))
        if out is None:
            outs.append(y)
        elif copy_stream is None:
            out[i:i + len(chunk)].copy_(y)
        else:
            copy_stream.wait_stream(torch.cuda.current_stream(clip.device))
            with torch.cuda.stream(copy_stream):
                out[i:i + len(chunk)].copy_(y, non_blocking=True)
            y.record_stream(copy_stream)
    if out is not None:
        if copy_stream is not None and join:
            torch.cuda.current_stream(clip.device).wait_stream(copy_stream)
        return out
    if not outs:
        return torch.empty(0)
    return torch.cat(outs, 0)


def gather_outputs(local: torch.Tensor, n_frames: int, rank: int, world_size: int, dst: Optional[int] = 0,
                   contiguous: bool = False, group=None, out: Optional[torch.Tensor] = None,
                   async_op: bool = False):
    """Collect per-rank results [n_local, ...] of any dtype (frames owned per `shard_frames(n_frames, rank, world_size, contiguous)`) into
    clip order [n_frames, ...].  One pre-sized collective, no pickled metadata: every rank derives every other rank's frame
    list from the same deterministic `shard_frames`, so only payload travels.

    dst = r   : `dist.gather` to rank r (what writing the frames / logging needs; 1/world of an all-gather's traffic);
                returns the assembled tensor on rank r and None elsewhere.
    dst = None: `dist.all_gather_into_tensor`, every rank gets the clip.
    Ragged shards are padded to the longest one (at most one frame per rank).
    `async_op`: returns (work, finish) -- call finish() after work.wait() to obtain the result (lets the transfer of batch i
    overlap the forward of batch i+1)."""
    import torch.distributed as dist
    lists = [shard_frames(n_frames, r, world_size, contiguous) for r in range(world_size)]
    longest = max(len(l) for l in lists)
    shape = list(local.shape[1:])
    if local.shape[0] != len(lists[rank]):
        raise ValueError(f"rank {rank} owns {len(lists[rank])} frames but passed {local.shape[0]}")
    send = local
    if local.shape[0] != longest:
        send = torch.zeros([longest] + shape, dtype=local.dtype, device=local.device)
        send[:local.shape[0]] = local
    send = send.contiguous()
    recv = None
    if dst is None:
        recv = torch.empty([world_size * longest] + shape, dtype=local.dtype, device=local.device)
        work = dist.all_gather_into_tensor(recv, send, group=group, async_op=True)
    else:
        if rank == dst:
            recv = torch.empty([world_size * longest] + shape, dtype=local.dtype, device=local.device)
        work = dist.gather(send, list(recv.view([world_size, longest] + shape).unbind(0)) if rank == dst else None, dst=dst,
                           group=group, async_op=True)

    def finish() -> Optional[torch.Tensor]:
        if recv is None:
            return None
        res = out if out is not None else torch.empty([n_frames] + shape, dtype=local.dtype, device=local.device)
        blocks = recv.view([world_size, longest] + shape)
        for r, fl in enumerate(lists):
            if not fl:
                continue
            if contiguous:
                res[fl[0]:fl[0] + len(fl)] = blocks[r, :len(fl)]
            else:
                res[r::world_size][:len(fl)] = blocks[r, :len(fl)]          # rank-strided shard = strided slice of the clip
        return res

    if async_op:
        return work, finish
    work.wait()
    return finish()


def reduce_metrics(local_rows: torch.Tensor, frames: Sequence[int], n_frames: int, dst: int = 0, group=None) -> torch.Tensor:
    """The reference's own reduction (lbasicsr/models/video_base_model.py:36-37, 106-113): every rank fills its rows of a
    zero [n_frames, n_metrics] tensor, then `dist.reduce(..., dst=0)` sums them.  Returns the tensor (complete on `dst`)."""
    import torch.distributed as dist
    full = torch.zeros(n_frames, local_rows.shape[1], dtype=local_rows.dtype, device=local_rows.device)
    if len(frames):
        full[torch.as_tensor(list(frames), device=local_rows.device)] = local_rows
    dist.reduce(full, dst=dst, group=group)
    return full
